// integrator.cu — K1: fused multi-step kinetic-Langevin (Euler–Maruyama) integrator.
//
// Replaces utils/sampling_utils.py:6-52 (update_step + the vmapped lax.scan).  One thread owns one
// particle for the whole trajectory: (q,p) stay in registers across all S+1 steps, the noise is
// drawn in registers from Philox4x32-10 (or read from an injected tensor for parity runs), the
// drift functor is inlined, and the only HBM traffic is the initial state read, the emitted
// trajectory samples and the final state — 2d*4 bytes per emitted particle-step.
#include "common.cuh"
#include "drift.cuh"
#include "integrator_args.cuh"
#include "philox.cuh"

#include <stdlib.h>

namespace pdeip {


template <int DP>
__device__ __forceinline__ void emit_state(float* __restrict__ base, int layout, int64_t n, int64_t n_total,
                                           int d, int C, int s_e, int s_emit, const float (&q)[DP],
                                           const float (&p)[DP]) {
  if (layout == PDEIP_TRAJ_BLOCK128) {  // [S_emit][N/128][C][128]
    float* o = base + (((int64_t)s_e * (n_total >> 7) + (n >> 7)) * C) * 128 + (n & 127);
#pragma unroll
    for (int i = 0; i < DP; ++i)
      if (i < d) {
        __stcs(o + i * 128, q[i]);
        __stcs(o + (d + i) * 128, p[i]);
      }
    return;
  }
  if (layout == PDEIP_TRAJ_TIME_SOA) {  // [2d][S_emit][N]: component planes, each plane time-major
    float* o = base + (int64_t)s_e * n_total + n;
    const int64_t plane = (int64_t)s_emit * n_total;
#pragma unroll
    for (int i = 0; i < DP; ++i)
      if (i < d) {
        __stcs(o + (int64_t)i * plane, q[i]);
        __stcs(o + (int64_t)(d + i) * plane, p[i]);
      }
    return;
  }
  float* o = (layout == PDEIP_TRAJ_PARTICLE_MAJOR) ? base + (n * s_emit + s_e) * C
                                                    : base + ((int64_t)s_e * n_total + n) * C;
  if (DP % 4 == 0 && d == DP) {
#pragma unroll
    for (int i4 = 0; i4 < DP / 4; ++i4) {
      __stcs(reinterpret_cast<float4*>(o) + i4, make_float4(q[4 * i4], q[4 * i4 + 1], q[4 * i4 + 2], q[4 * i4 + 3]));
      __stcs(reinterpret_cast<float4*>(o + d) + i4,
             make_float4(p[4 * i4], p[4 * i4 + 1], p[4 * i4 + 2], p[4 * i4 + 3]));
    }
  } else {
#pragma unroll
    for (int i = 0; i < DP; ++i)
      if (i < d) {
        o[i] = q[i];
        o[d + i] = p[i];
      }
  }
}

// grad U(x) of sample s_e -> components [2d, 3d) of its slot (row width C = 3d)
template <int DP>
__device__ __forceinline__ void emit_drift_vals(float* __restrict__ base, int layout, int64_t n, int64_t n_total,
                                                int d, int C, int s_e, int s_emit, const float (&g)[DP]) {
  if (layout == PDEIP_TRAJ_BLOCK128) {
    float* o = base + (((int64_t)s_e * (n_total >> 7) + (n >> 7)) * C) * 128 + (n & 127);
#pragma unroll
    for (int i = 0; i < DP; ++i)
      if (i < d) __stcs(o + (2 * d + i) * 128, g[i]);
    return;
  }
  if (layout == PDEIP_TRAJ_TIME_SOA) {
    float* o = base + (int64_t)s_e * n_total + n;
    const int64_t plane = (int64_t)s_emit * n_total;
#pragma unroll
    for (int i = 0; i < DP; ++i)
      if (i < d) __stcs(o + (int64_t)(2 * d + i) * plane, g[i]);
    return;
  }
  float* o = (layout == PDEIP_TRAJ_PARTICLE_MAJOR) ? base + (n * s_emit + s_e) * C + 2 * d
                                                    : base + ((int64_t)s_e * n_total + n) * C + 2 * d;
  if (DP % 4 == 0 && d == DP) {
#pragma unroll
    for (int i4 = 0; i4 < DP / 4; ++i4)
      __stcs(reinterpret_cast<float4*>(o) + i4, make_float4(g[4 * i4], g[4 * i4 + 1], g[4 * i4 + 2], g[4 * i4 + 3]));
  } else {
#pragma unroll
    for (int i = 0; i < DP; ++i)
      if (i < d) o[i] = g[i];
  }
}

// v[0, d) -> components [col0, col0 + d) of sample s_e (row width C) in any trajectory layout (overdamped K1-OD)
template <int DP>
__device__ __forceinline__ void emit_cols(float* __restrict__ base, int layout, int64_t n, int64_t n_total, int d,
                                          int C, int col0, int s_e, int s_emit, const float (&v)[DP]) {
  if (layout == PDEIP_TRAJ_BLOCK128) {
    float* o = base + (((int64_t)s_e * (n_total >> 7) + (n >> 7)) * C + col0) * 128 + (n & 127);
#pragma unroll
    for (int i = 0; i < DP; ++i)
      if (i < d) __stcs(o + i * 128, v[i]);
    return;
  }
  if (layout == PDEIP_TRAJ_TIME_SOA) {
    const int64_t plane = (int64_t)s_emit * n_total;
    float* o = base + (int64_t)col0 * plane + (int64_t)s_e * n_total + n;
#pragma unroll
    for (int i = 0; i < DP; ++i)
      if (i < d) __stcs(o + (int64_t)i * plane, v[i]);
    return;
  }
  float* o = (layout == PDEIP_TRAJ_PARTICLE_MAJOR) ? base + (n * s_emit + s_e) * C + col0
                                                    : base + ((int64_t)s_e * n_total + n) * C + col0;
#pragma unroll
  for (int i = 0; i < DP; ++i)
    if (i < d) __stcs(o + i, v[i]);
}

// drift kinds of the hypothesis models (pdeip_kl_integrate_model), internal to this file
constexpr int kDriftAffine = 100;  // quadratic model: grad V = (K + K^T) y + b, params = [K (d*d), b (d)]
constexpr int kDriftMlp = 101;     // MLP model: grad V_theta, params = the flat MLP buffer (hidden width 32)

// LHMAX: hidden layers the per-thread MLP state is sized for (kDriftMlp only).
// OD: overdamped dynamics (pdeip_overdamped_integrate*): the state is x alone, x' = x - h grad U(x) + sqrt(2h) xi, on
// the UNIFORM schedule; an emitted sample is [x] or [x, grad U(x)].  OD = false is the kinetic K1 step.
template <int DP, int DRIFT, int LHMAX = 0, bool OD = false>
__global__ void __launch_bounds__(128) kl_integrate_kernel(const IntegrateArgs a) {
  extern __shared__ __align__(16) float smem[];
  // stage the drift parameters (zero-padded to DP) in shared memory
  float* A_s = smem;           // LINEAR / MEANFIELD: [DP][DP] (+ [DP] shift)
  float* shift_s = nullptr;
  constexpr bool kTable = DRIFT == PDEIP_DRIFT_MEANFIELD_TABLE;  // grad U = A x - (A xbar_s), row s of the table per step
  if constexpr (DRIFT == PDEIP_DRIFT_LINEAR || DRIFT == PDEIP_DRIFT_MEANFIELD || kTable) {
    load_padded<DP>(A_s, a.drift_params, a.d, a.d, threadIdx.x, blockDim.x);
    // rows >= d must be zero too
    for (int idx = a.d * DP + threadIdx.x; idx < DP * DP; idx += blockDim.x) A_s[idx] = 0.0f;
    if constexpr (DRIFT == PDEIP_DRIFT_MEANFIELD) {
      shift_s = smem + DP * DP;
      for (int i = threadIdx.x; i < DP; i += blockDim.x)
        shift_s[i] = i < a.d ? a.drift_params[a.d * a.d + i] : 0.0f;
    }
  } else if constexpr (DRIFT == PDEIP_DRIFT_GMM) {
    load_padded<DP>(smem, a.drift_params, a.n_gaussian, a.d, threadIdx.x, blockDim.x);
  } else if constexpr (DRIFT == kDriftAffine) {  // M = K + K^T [DP][DP], then b [DP], zero padded
    shift_s = smem + DP * DP;
    const float* K = a.drift_params;
    for (int idx = threadIdx.x; idx < DP * DP; idx += blockDim.x) {
      const int i = idx / DP, k = idx - i * DP;
      A_s[idx] = (i < a.d && k < a.d) ? K[i * a.d + k] + K[k * a.d + i] : 0.0f;
    }
    for (int i = threadIdx.x; i < DP; i += blockDim.x) shift_s[i] = i < a.d ? K[a.d * a.d + i] : 0.0f;
  } else if constexpr (DRIFT == kDriftMlp) {
    const int P = MlpShape<32>{a.d, a.layers}.num_params();
    for (int i = threadIdx.x; i < P; i += blockDim.x) smem[i] = a.drift_params[i];
  }
  __syncthreads();
  const MlpShape<32> mlp_shape{a.d, a.layers};

  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= a.n) return;
  const int d = a.d;
  const uint64_t pid = a.particle_offset + (uint64_t)n;

  float q[DP], p[DP];
#pragma unroll
  for (int i = 0; i < DP; ++i) {
    if constexpr (OD) {
      q[i] = (i < d) ? a.z0[elem_index(a.state_layout, n, i, a.n, d)] : 0.0f;
    } else {
      q[i] = (i < d) ? a.z0[elem_index(a.state_layout, n, i, a.n, 2 * d)] : 0.0f;
      p[i] = (i < d) ? a.z0[elem_index(a.state_layout, n, d + i, a.n, 2 * d)] : 0.0f;
    }
  }

  const bool ref_sched = (a.schedule == PDEIP_SCHEDULE_REFERENCE);
  float t0 = 0.0f;
  if (ref_sched) {
    // mean-field table: a common time grid (tau0 == 0) unless the caller injects tau0
    t0 = a.tau0 ? a.tau0[n] : (kTable ? 0.0f : philox_uniform01(a.seed, pid, kTagTau0) * a.dt);  // sampling_utils.py:32
  }
  const int total_steps = ref_sched ? a.n_steps + 1 : a.n_steps;
  const int n_draws = total_steps;
  const int C = OD ? (a.emit_drift ? 2 * d : d) : (a.emit_drift ? 3 * d : 2 * d);  // floats per emitted sample

  for (int s = 0; s < total_steps; ++s) {
    float h = a.dt;
    if (ref_sched) {
      if (s == 0) h = t0;                        // sampling_utils.py:33
      else if (s == a.n_steps) h = a.dt - t0;    // sampling_utils.py:45-46
    }
    // drift
    float g[DP];
    if constexpr (DRIFT == PDEIP_DRIFT_GMM) {
      gmm_grad_thread<DP>(q, smem, a.n_gaussian, a.inv_sigma2, g);
    } else if constexpr (DRIFT == kDriftAffine) {
      affine_grad_thread<DP>(q, A_s, shift_s, g);
    } else if constexpr (DRIFT == kDriftMlp) {
      mlp_grad_thread<DP, LHMAX>(q, mlp_shape, smem, g);
    } else if constexpr (DRIFT == PDEIP_DRIFT_LINEAR || DRIFT == PDEIP_DRIFT_MEANFIELD || kTable) {
      linear_grad_thread<DP>(q, A_s, shift_s, g);
      if constexpr (kTable) {
        const float* row = a.drift_params + d * d + (int64_t)s * d;
#pragma unroll
        for (int i = 0; i < DP; ++i)
          if (i < d) g[i] -= __ldg(row + i);
      }
    } else {
#pragma unroll
      for (int i = 0; i < DP; ++i) g[i] = 0.0f;
    }
    // the drift just evaluated is grad U at the state emitted as sample s-1
    if (a.emit_drift && a.traj && s >= 1 && ((s - 1) % a.emit_every) == a.emit_offset) {
      if constexpr (OD) emit_cols<DP>(a.traj, a.traj_layout, n, a.n, d, C, d, (s - 1) / a.emit_every, a.s_emit, g);
      else emit_drift_vals<DP>(a.traj, a.traj_layout, n, a.n, d, C, (s - 1) / a.emit_every, a.s_emit, g);
    }
    // noise
    float xi[DP];
    if (a.noise) {
      const float* nz = a.noise + (n * n_draws + s) * d;
#pragma unroll
      for (int i = 0; i < DP; ++i) xi[i] = (i < d) ? nz[i] : 0.0f;
    } else {
#pragma unroll
      for (int j = 0; j < (DP + 3) / 4; ++j) {
        float r4[4];
        philox_normal4(a.seed, pid, a.step_offset + (uint32_t)s, (uint32_t)j, r4);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (4 * j + k < DP) xi[4 * j + k] = (4 * j + k < d) ? r4[k] : 0.0f;
      }
    }
    // p' = p - h g + sqrt(h) sqrt(2) xi - gamma p h ;  q' = q + h p'     (sampling_utils.py:14-20)
    const float sq = sqrtf(h) * 1.41421356237309515f;
#pragma unroll
    for (int i = 0; i < DP; ++i) {
      if constexpr (OD) {  // x' = x - h grad U(x) + sqrt(h) sqrt(2) xi
        q[i] = q[i] - h * g[i] + sq * xi[i];
      } else {
        const float pn = p[i] - h * g[i] + sq * xi[i] - a.gamma * p[i] * h;
        p[i] = pn;
        q[i] = q[i] + h * pn;
      }
    }
    // emission: REFERENCE schedule emits samples 0..S-1 (the last step only feeds z_last);
    // UNIFORM schedule emits every state.
    const bool is_sample = ref_sched ? (s < a.n_steps) : true;
    if (a.traj && is_sample && (s % a.emit_every) == a.emit_offset) {
      if constexpr (OD) emit_cols<DP>(a.traj, a.traj_layout, n, a.n, d, C, 0, s / a.emit_every, a.s_emit, q);
      else emit_state<DP>(a.traj, a.traj_layout, n, a.n, d, C, s / a.emit_every, a.s_emit, q, p);
    }
  }
  if (a.emit_drift && a.traj && !ref_sched && ((total_steps - 1) % a.emit_every) == a.emit_offset) {
    // UNIFORM schedule: the last emitted sample has no following step; evaluate its drift once more
    float g[DP];
    if constexpr (DRIFT == PDEIP_DRIFT_GMM) {
      gmm_grad_thread<DP>(q, smem, a.n_gaussian, a.inv_sigma2, g);
    } else if constexpr (DRIFT == kDriftAffine) {
      affine_grad_thread<DP>(q, A_s, shift_s, g);
    } else if constexpr (DRIFT == kDriftMlp) {
      mlp_grad_thread<DP, LHMAX>(q, mlp_shape, smem, g);
    } else if constexpr (DRIFT == PDEIP_DRIFT_LINEAR || DRIFT == PDEIP_DRIFT_MEANFIELD || kTable) {
      linear_grad_thread<DP>(q, A_s, shift_s, g);
    } else {
#pragma unroll
      for (int i = 0; i < DP; ++i) g[i] = 0.0f;
    }
    if constexpr (OD) emit_cols<DP>(a.traj, a.traj_layout, n, a.n, d, C, d, (total_steps - 1) / a.emit_every, a.s_emit, g);
    else emit_drift_vals<DP>(a.traj, a.traj_layout, n, a.n, d, C, (total_steps - 1) / a.emit_every, a.s_emit, g);
  }
  if (a.z_last) {
#pragma unroll
    for (int i = 0; i < DP; ++i)
      if (i < d) {
        if constexpr (OD) {
          a.z_last[elem_index(a.state_layout, n, i, a.n, d)] = q[i];
        } else {
          a.z_last[elem_index(a.state_layout, n, i, a.n, 2 * d)] = q[i];
          a.z_last[elem_index(a.state_layout, n, d + i, a.n, 2 * d)] = p[i];
        }
      }
  }
  if (a.tau && ref_sched) {
    for (int s = 0; s < a.n_steps; ++s) a.tau[n * a.n_steps + s] = t0 + (float)s * a.dt;  // :48
  }
}

// ------------------------------------------------------------------------------------------------------------
// Production configuration of K1 (pipeline.HotPath): in-register Philox noise, per-particle tau0, every sample
// emitted as [x, v, grad U(x)] into the [3d][S][N] SoA trajectory, d == DP.  Same arithmetic as the generic kernel
// above up to rounding: the GMM drift is a branch-free tiled online softmax (8 centres per tile, one rescale per
// tile) on MUFU ex2, and every d-wide loop runs on packed fp32x2 instructions (FFMA2: half the issue slots).
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

constexpr int kGmmTile = 8;  // centres per softmax tile (4 at d = 32: register pressure); the centre table is padded to a
                             // multiple of 8 with far-away rows

// mus_s: smem [Kpad][DP]; c2 = -0.5 * inv_sigma2 * log2(e).  g = (x - sum_k softmax_k mu_k) * inv_sigma2
template <int DP>
__device__ __forceinline__ void gmm_grad_fast(const float2 (&x)[DP / 2], const float* __restrict__ mus_s, int k_pad, float c2,
                                              float inv_sigma2, float2 (&g)[DP / 2]) {
  float m = -INFINITY, se = 0.f;
  float2 acc[DP / 2];
#pragma unroll
  for (int i = 0; i < DP / 2; ++i) acc[i] = make_float2(0.f, 0.f);
  const float2 neg1 = make_float2(-1.f, -1.f);
  constexpr int TK = DP >= 32 ? 4 : kGmmTile;
#pragma unroll 1
  for (int k0 = 0; k0 < k_pad; k0 += TK) {
    float al[TK];
#pragma unroll
    for (int kk = 0; kk < TK; ++kk) {
      const float4* mu4 = reinterpret_cast<const float4*>(mus_s + (k0 + kk) * DP);
      float2 s2 = make_float2(0.f, 0.f);
#pragma unroll
      for (int i4 = 0; i4 < DP / 4; ++i4) {
        const float4 t = mu4[i4];
        const float2 r0 = __ffma2_rn(make_float2(t.x, t.y), neg1, x[2 * i4]);
        const float2 r1 = __ffma2_rn(make_float2(t.z, t.w), neg1, x[2 * i4 + 1]);
        s2 = __ffma2_rn(r0, r0, s2);
        s2 = __ffma2_rn(r1, r1, s2);
      }
      al[kk] = c2 * (s2.x + s2.y);  // log2 of the unnormalised weight
    }
    float tm = al[0];
#pragma unroll
    for (int kk = 1; kk < TK; ++kk) tm = fmaxf(tm, al[kk]);
    const float mn = fmaxf(m, tm);
    const float sc = ex2_approx(m - mn);  // m = -inf on the first tile: ex2(-inf) = 0 and acc, se are 0 anyway
    m = mn;
    se *= sc;
    const float2 sc2 = make_float2(sc, sc);
#pragma unroll
    for (int i = 0; i < DP / 2; ++i) acc[i] = __fmul2_rn(acc[i], sc2);
#pragma unroll
    for (int kk = 0; kk < TK; ++kk) {
      const float e = ex2_approx(al[kk] - m);
      se += e;
      const float2 e2 = make_float2(e, e);
      const float4* mu4 = reinterpret_cast<const float4*>(mus_s + (k0 + kk) * DP);
#pragma unroll
      for (int i4 = 0; i4 < DP / 4; ++i4) {
        const float4 t = mu4[i4];
        acc[2 * i4] = __ffma2_rn(e2, make_float2(t.x, t.y), acc[2 * i4]);
        acc[2 * i4 + 1] = __ffma2_rn(e2, make_float2(t.z, t.w), acc[2 * i4 + 1]);
      }
    }
  }
  const float ninv = -1.f / se;
  const float2 ninv2 = make_float2(ninv, ninv), is2 = make_float2(inv_sigma2, inv_sigma2);
#pragma unroll
  for (int i = 0; i < DP / 2; ++i) g[i] = __fmul2_rn(__ffma2_rn(acc[i], ninv2, x[i]), is2);
}

// AT_s: smem [DP][DP], AT_s[k][i] = A[i][k];  g = A x
template <int DP>
__device__ __forceinline__ void linear_grad_fast(const float2 (&x)[DP / 2], const float* __restrict__ AT_s, float2 (&g)[DP / 2]) {
#pragma unroll
  for (int i = 0; i < DP / 2; ++i) g[i] = make_float2(0.f, 0.f);
#pragma unroll
  for (int k = 0; k < DP; ++k) {
    const float xk = (k & 1) ? x[k >> 1].y : x[k >> 1].x;
    const float2 xk2 = make_float2(xk, xk);
    const float4* row = reinterpret_cast<const float4*>(AT_s + k * DP);
#pragma unroll
    for (int i4 = 0; i4 < DP / 4; ++i4) {
      const float4 t = row[i4];
      g[2 * i4] = __ffma2_rn(make_float2(t.x, t.y), xk2, g[2 * i4]);
      g[2 * i4 + 1] = __ffma2_rn(make_float2(t.z, t.w), xk2, g[2 * i4 + 1]);
    }
  }
}

#ifndef PDEIP_FAST_MINB
#define PDEIP_FAST_MINB 4
#endif
// BLK: trajectory in PDEIP_TRAJ_BLOCK128 (every store of a step is base + immediate) instead of PDEIP_TRAJ_TIME_SOA
template <int DP, int DRIFT, bool BLK>
__global__ void __launch_bounds__(128, DP >= 32 ? 2 : PDEIP_FAST_MINB) kl_integrate_fast_kernel(const IntegrateArgs a, int k_pad) {
  static_assert(DP % 4 == 0, "packed path needs d % 4 == 0");
  extern __shared__ __align__(16) float smem[];
  if constexpr (DRIFT == PDEIP_DRIFT_GMM) {
    for (int idx = threadIdx.x; idx < k_pad * DP; idx += blockDim.x) {
      const int r = idx / DP;
      smem[idx] = r < a.n_gaussian ? a.drift_params[idx] : 1.0e18f;  // padding rows: weight exactly 0
    }
  } else {
    for (int idx = threadIdx.x; idx < DP * DP; idx += blockDim.x) {
      const int k = idx / DP, i = idx - k * DP;
      smem[idx] = a.drift_params[i * DP + k];
    }
  }
  __syncthreads();
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= a.n) return;
  const uint64_t pid = a.particle_offset + (uint64_t)n;
  float2 q[DP / 2], p[DP / 2];
  {
    const float4* z4 = reinterpret_cast<const float4*>(a.z0 + n * (2 * DP));
#pragma unroll
    for (int i4 = 0; i4 < DP / 4; ++i4) {
      const float4 tq = z4[i4], tp = z4[DP / 4 + i4];
      q[2 * i4] = make_float2(tq.x, tq.y); q[2 * i4 + 1] = make_float2(tq.z, tq.w);
      p[2 * i4] = make_float2(tp.x, tp.y); p[2 * i4 + 1] = make_float2(tp.z, tp.w);
    }
  }
  constexpr bool kTable = DRIFT == PDEIP_DRIFT_MEANFIELD_TABLE;  // common time grid: tau0 == 0
  const float t0 = kTable ? 0.f : philox_uniform01(a.seed, pid, kTagTau0) * a.dt;  // sampling_utils.py:32
  const float c2 = -0.5f * a.inv_sigma2 * 1.4426950408889634f;
  const int S = a.n_steps;
  // BLK: element (sample s, block b, component c, lane l) at ((s B + b) 3d + c) 128 + l ; else c S N + s N + n
  const int64_t plane = BLK ? 128 : (int64_t)S * a.n;                             // floats between components
  const int64_t sstride = BLK ? (int64_t)gridDim.x * (3 * DP * 128) : a.n;        // floats between samples
  float* o = BLK ? a.traj + ((int64_t)blockIdx.x * (3 * DP) * 128 + threadIdx.x) : a.traj + n;  // sample 0, comp 0
#pragma unroll 1
  for (int s = 0; s <= S; ++s) {
    const float h = (s == 0) ? t0 : ((s == S) ? a.dt - t0 : a.dt);  // sampling_utils.py:33,45-46
    float2 g[DP / 2];
    if constexpr (DRIFT == PDEIP_DRIFT_GMM) gmm_grad_fast<DP>(q, smem, k_pad, c2, a.inv_sigma2, g);
    else linear_grad_fast<DP>(q, smem, g);
    if constexpr (kTable) {  // grad U = A (x - xbar_s): row s of the (A xbar) table (warp-uniform address)
      const float2* row = reinterpret_cast<const float2*>(a.drift_params + DP * DP + (int64_t)s * DP);
      const float2 neg1 = make_float2(-1.f, -1.f);
#pragma unroll
      for (int i = 0; i < DP / 2; ++i) g[i] = __ffma2_rn(__ldg(row + i), neg1, g[i]);
    }
    if (s >= 1) {  // grad U at the state emitted as sample s - 1
      float* og = o - sstride + 2 * DP * plane;
#pragma unroll
      for (int i = 0; i < DP / 2; ++i) {
        if constexpr (BLK) {
          __stcs(og + (2 * i) * 128, g[i].x);
          __stcs(og + (2 * i + 1) * 128, g[i].y);
        } else {
          __stcs(og + (int64_t)(2 * i) * plane, g[i].x);
          __stcs(og + (int64_t)(2 * i + 1) * plane, g[i].y);
        }
      }
    }
    // p' = p - h g + sqrt(2 h) xi - gamma h p ;  q' = q + h p'     (sampling_utils.py:14-20)
    const float sq = sqrtf(h) * 1.41421356237309515f;
    const float2 sq2 = make_float2(sq, sq), nh2 = make_float2(-h, -h), h2 = make_float2(h, h);
    const float dmp = 1.f - a.gamma * h;
    const float2 dmp2 = make_float2(dmp, dmp);
#pragma unroll
    for (int j = 0; j < DP / 4; ++j) {
      float r4[4];
      philox_normal4_rk(a.rk, pid, a.step_offset + (uint32_t)s, (uint32_t)j, r4);
      const float2 xa = make_float2(r4[0], r4[1]), xb = make_float2(r4[2], r4[3]);
      // same association as the generic kernel up to the fused damping factor (1 - gamma h)
      float2 pa = __ffma2_rn(nh2, g[2 * j], __fmul2_rn(p[2 * j], dmp2));
      float2 pb = __ffma2_rn(nh2, g[2 * j + 1], __fmul2_rn(p[2 * j + 1], dmp2));
      pa = __ffma2_rn(sq2, xa, pa);
      pb = __ffma2_rn(sq2, xb, pb);
      p[2 * j] = pa; p[2 * j + 1] = pb;
      q[2 * j] = __ffma2_rn(h2, pa, q[2 * j]);
      q[2 * j + 1] = __ffma2_rn(h2, pb, q[2 * j + 1]);
    }
    if (s < S) {
#pragma unroll
      for (int i = 0; i < DP / 2; ++i) {
        if constexpr (BLK) {
          __stcs(o + (2 * i) * 128, q[i].x);
          __stcs(o + (2 * i + 1) * 128, q[i].y);
          __stcs(o + (DP + 2 * i) * 128, p[i].x);
          __stcs(o + (DP + 2 * i + 1) * 128, p[i].y);
        } else {
          __stcs(o + (int64_t)(2 * i) * plane, q[i].x);
          __stcs(o + (int64_t)(2 * i + 1) * plane, q[i].y);
          __stcs(o + (int64_t)(DP + 2 * i) * plane, p[i].x);
          __stcs(o + (int64_t)(DP + 2 * i + 1) * plane, p[i].y);
        }
      }
      o += sstride;
    }
  }
  {
    float4* zl = reinterpret_cast<float4*>(a.z_last + n * (2 * DP));
#pragma unroll
    for (int i4 = 0; i4 < DP / 4; ++i4) {
      zl[i4] = make_float4(q[2 * i4].x, q[2 * i4].y, q[2 * i4 + 1].x, q[2 * i4 + 1].y);
      zl[DP / 4 + i4] = make_float4(p[2 * i4].x, p[2 * i4].y, p[2 * i4 + 1].x, p[2 * i4 + 1].y);
    }
  }
}

// true if the call is the production configuration served by kl_integrate_fast_kernel
static bool fast_path_ok(const IntegrateArgs& a, int drift_kind, int DP) {
  return a.d == DP && DP % 4 == 0 &&
         (drift_kind == PDEIP_DRIFT_GMM || drift_kind == PDEIP_DRIFT_LINEAR || drift_kind == PDEIP_DRIFT_MEANFIELD_TABLE) && !a.noise &&
         !a.tau0 && !a.tau && a.traj && a.z_last && a.emit_drift && a.emit_every == 1 && a.emit_offset == 0 &&
         a.schedule == PDEIP_SCHEDULE_REFERENCE && a.state_layout == PDEIP_LAYOUT_AOS &&
         (a.traj_layout == PDEIP_TRAJ_TIME_SOA || a.traj_layout == PDEIP_TRAJ_BLOCK128) &&
         getenv("PDEIP_NO_FAST_INTEGRATOR") == nullptr;
}

template <int DP>
static int launch_integrate_fast(const IntegrateArgs& a, int drift_kind, cudaStream_t st) {
  if constexpr (DP % 4 == 0) {
    const int block = 128;
    const int64_t grid = (a.n + block - 1) / block;
    if (drift_kind == PDEIP_DRIFT_GMM) {
      const int k_pad = (a.n_gaussian + kGmmTile - 1) / kGmmTile * kGmmTile;
      const size_t smem = sizeof(float) * (size_t)k_pad * DP;
      PDEIP_REQUIRE(smem <= 48 * 1024, PDEIP_ERR_UNSUPPORTED, "GMM centres exceed 48 KB of shared memory");
      if (a.traj_layout == PDEIP_TRAJ_BLOCK128)
        kl_integrate_fast_kernel<DP, PDEIP_DRIFT_GMM, true><<<(unsigned)grid, block, smem, st>>>(a, k_pad);
      else
        kl_integrate_fast_kernel<DP, PDEIP_DRIFT_GMM, false><<<(unsigned)grid, block, smem, st>>>(a, k_pad);
    } else if (drift_kind == PDEIP_DRIFT_MEANFIELD_TABLE) {
      if (a.traj_layout == PDEIP_TRAJ_BLOCK128)
        kl_integrate_fast_kernel<DP, PDEIP_DRIFT_MEANFIELD_TABLE, true><<<(unsigned)grid, block, sizeof(float) * DP * DP, st>>>(a, 0);
      else
        kl_integrate_fast_kernel<DP, PDEIP_DRIFT_MEANFIELD_TABLE, false><<<(unsigned)grid, block, sizeof(float) * DP * DP, st>>>(a, 0);
    } else {
      if (a.traj_layout == PDEIP_TRAJ_BLOCK128)
        kl_integrate_fast_kernel<DP, PDEIP_DRIFT_LINEAR, true><<<(unsigned)grid, block, sizeof(float) * DP * DP, st>>>(a, 0);
      else
        kl_integrate_fast_kernel<DP, PDEIP_DRIFT_LINEAR, false><<<(unsigned)grid, block, sizeof(float) * DP * DP, st>>>(a, 0);
    }
    PDEIP_LAUNCH_OK();
    return PDEIP_OK;
  } else {
    return PDEIP_ERR_UNSUPPORTED;
  }
}

template <int DP>
static int launch_integrate(const IntegrateArgs& a, int drift_kind, int path, cudaStream_t st) {
  if (fast_path_ok(a, drift_kind, DP)) {
    // PDEIP_PATH_TENSOR: the GMM distance contraction on tcgen05 where that kernel exists, else the fp32 kernel
    if (path == PDEIP_PATH_TENSOR && integrate_tensor_ok(a, drift_kind)) return launch_integrate_tensor(a, st);
    return launch_integrate_fast<DP>(a, drift_kind, st);
  }
  const int block = 128;
  const int64_t grid = (a.n + block - 1) / block;
  size_t smem = 0;
  switch (drift_kind) {
    case PDEIP_DRIFT_NONE:
      kl_integrate_kernel<DP, PDEIP_DRIFT_NONE><<<(unsigned)grid, block, 0, st>>>(a);
      break;
    case PDEIP_DRIFT_LINEAR:
      smem = sizeof(float) * DP * DP;
      kl_integrate_kernel<DP, PDEIP_DRIFT_LINEAR><<<(unsigned)grid, block, smem, st>>>(a);
      break;
    case PDEIP_DRIFT_MEANFIELD:
      smem = sizeof(float) * (DP * DP + DP);
      kl_integrate_kernel<DP, PDEIP_DRIFT_MEANFIELD><<<(unsigned)grid, block, smem, st>>>(a);
      break;
    case PDEIP_DRIFT_MEANFIELD_TABLE:
      PDEIP_REQUIRE(a.schedule == PDEIP_SCHEDULE_REFERENCE, PDEIP_ERR_UNSUPPORTED,
                    "PDEIP_DRIFT_MEANFIELD_TABLE needs the REFERENCE schedule (table row = step index)");
      smem = sizeof(float) * DP * DP;
      kl_integrate_kernel<DP, PDEIP_DRIFT_MEANFIELD_TABLE><<<(unsigned)grid, block, smem, st>>>(a);
      break;
    case PDEIP_DRIFT_GMM:
      smem = sizeof(float) * (size_t)a.n_gaussian * DP;
      PDEIP_REQUIRE(smem <= 48 * 1024, PDEIP_ERR_UNSUPPORTED, "GMM centres exceed 48 KB of shared memory");
      kl_integrate_kernel<DP, PDEIP_DRIFT_GMM><<<(unsigned)grid, block, smem, st>>>(a);
      break;
    default:
      PDEIP_REQUIRE(false, PDEIP_ERR_INVALID_ARG, "unknown drift kind %d", drift_kind);
  }
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}

// K1 under a hypothesis model's potential: the generic kernel with the affine (quadratic model) or MLP drift; under
// PDEIP_PATH_TENSOR the MLP drift of the tcgen05 kernel's envelope (integrator_mlp_tc.cu).
template <int DP>
static int launch_integrate_model(const IntegrateArgs& a, int model_kind, int path, cudaStream_t st) {
  if (model_kind == PDEIP_MODEL_MLP && path == PDEIP_PATH_TENSOR && integrate_mlp_tensor_ok(a))
    return launch_integrate_mlp_tensor(a, st);
  const unsigned grid = (unsigned)((a.n + 127) / 128);
  if (model_kind == PDEIP_MODEL_QUADRATIC) {
    kl_integrate_kernel<DP, kDriftAffine><<<grid, 128, sizeof(float) * (DP * DP + DP), st>>>(a);
  } else {
    // at most 9 768 floats (d = 32, 8 layers): below the 48 KB of shared memory a launch gets without opt-in
    const size_t smem = sizeof(float) * (size_t)MlpShape<32>{a.d, a.layers}.num_params();
    if (a.layers <= 2) kl_integrate_kernel<DP, kDriftMlp, 2><<<grid, 128, smem, st>>>(a);
    else if (a.layers <= 4) kl_integrate_kernel<DP, kDriftMlp, 4><<<grid, 128, smem, st>>>(a);
    else kl_integrate_kernel<DP, kDriftMlp, 8><<<grid, 128, smem, st>>>(a);
  }
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}

// K1-OD: the overdamped step on the generic kernel, every analytic drift and configuration (the entry point has
// rejected PDEIP_DRIFT_MEANFIELD_TABLE and unknown kinds); under PDEIP_PATH_TENSOR the GMM drift of K1-T-OD's envelope
// (integrator_tc.cu)
template <int DP>
static int launch_overdamped(const IntegrateArgs& a, int drift_kind, int path, cudaStream_t st) {
  if (path == PDEIP_PATH_TENSOR && overdamped_tensor_ok(a, drift_kind)) return launch_overdamped_tensor(a, st);
  const unsigned grid = (unsigned)((a.n + 127) / 128);
  switch (drift_kind) {
    case PDEIP_DRIFT_NONE:
      kl_integrate_kernel<DP, PDEIP_DRIFT_NONE, 0, true><<<grid, 128, 0, st>>>(a);
      break;
    case PDEIP_DRIFT_LINEAR:
      kl_integrate_kernel<DP, PDEIP_DRIFT_LINEAR, 0, true><<<grid, 128, sizeof(float) * DP * DP, st>>>(a);
      break;
    case PDEIP_DRIFT_MEANFIELD:
      kl_integrate_kernel<DP, PDEIP_DRIFT_MEANFIELD, 0, true><<<grid, 128, sizeof(float) * (DP * DP + DP), st>>>(a);
      break;
    default: {  // PDEIP_DRIFT_GMM
      const size_t smem = sizeof(float) * (size_t)a.n_gaussian * DP;
      PDEIP_REQUIRE(smem <= 48 * 1024, PDEIP_ERR_UNSUPPORTED, "GMM centres exceed 48 KB of shared memory");
      kl_integrate_kernel<DP, PDEIP_DRIFT_GMM, 0, true><<<grid, 128, smem, st>>>(a);
    }
  }
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}

// K1-OD under a hypothesis model's potential; under PDEIP_PATH_TENSOR the MLP drift of the tcgen05 kernel's envelope
template <int DP>
static int launch_overdamped_model(const IntegrateArgs& a, int model_kind, int path, cudaStream_t st) {
  if (model_kind == PDEIP_MODEL_MLP && path == PDEIP_PATH_TENSOR && overdamped_mlp_tensor_ok(a))
    return launch_overdamped_mlp_tensor(a, st);
  const unsigned grid = (unsigned)((a.n + 127) / 128);
  if (model_kind == PDEIP_MODEL_QUADRATIC) {
    kl_integrate_kernel<DP, kDriftAffine, 0, true><<<grid, 128, sizeof(float) * (DP * DP + DP), st>>>(a);
  } else {
    const size_t smem = sizeof(float) * (size_t)MlpShape<32>{a.d, a.layers}.num_params();
    if (a.layers <= 2) kl_integrate_kernel<DP, kDriftMlp, 2, true><<<grid, 128, smem, st>>>(a);
    else if (a.layers <= 4) kl_integrate_kernel<DP, kDriftMlp, 4, true><<<grid, 128, smem, st>>>(a);
    else kl_integrate_kernel<DP, kDriftMlp, 8, true><<<grid, 128, smem, st>>>(a);
  }
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}

// ------------------------------------------------------------------------------------------
// noise dumps (what the integrator draws in Philox mode) and the Gaussian initial ensemble
// ------------------------------------------------------------------------------------------
__global__ void philox_normals_kernel(float* out, int64_t n, int n_draws, int d, uint64_t seed,
                                      uint64_t particle_offset, uint32_t step_offset) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // (particle, draw)
  if (idx >= n * n_draws) return;
  const int64_t p = idx / n_draws;
  const int s = (int)(idx - p * n_draws);
  for (int j = 0; j < (d + 3) / 4; ++j) {
    float r4[4];
    philox_normal4(seed, particle_offset + (uint64_t)p, step_offset + (uint32_t)s, (uint32_t)j, r4);
    for (int k = 0; k < 4; ++k)
      if (4 * j + k < d) out[idx * d + 4 * j + k] = r4[k];
  }
}

__global__ void philox_uniforms_kernel(float* out, int64_t n, uint64_t seed, uint64_t particle_offset) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n) out[p] = philox_uniform01(seed, particle_offset + (uint64_t)p, kTagTau0);
}

__global__ void philox_raw_kernel(const uint32_t* ctr, const uint32_t* key, uint32_t* out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t c0 = ctr[4 * i], c1 = ctr[4 * i + 1], c2 = ctr[4 * i + 2], c3 = ctr[4 * i + 3];
  philox4x32_10(c0, c1, c2, c3, key[0], key[1]);
  out[4 * i] = c0; out[4 * i + 1] = c1; out[4 * i + 2] = c2; out[4 * i + 3] = c3;
}

// ------------------------------------------------------------------------------------------------------------
// Mean-field drift  grad U = A (x - xbar_t),  xbar_t = empirical mean over ALL particles of all ranks  (README.md:54-62:
// -grad Phi * rho_t for Phi = x'Ax/2).  On the common time grid (tau0 == 0: step 0 has h = 0, steps 1..S have h = dt) the
// ensemble mean obeys a closed recursion, because the interaction term A (xbar - xbar) vanishes in the mean:
//     pbar_{s+1} = (1 - gamma dt) pbar_s + sqrt(2 dt) xibar_s,   qbar_{s+1} = qbar_s + dt pbar_{s+1},
// xibar_s = mean over particles of the step-s normals.  The noise is counter-based (Philox keyed by the global particle
// id), so xibar_s for ALL steps comes from one pre-pass over the particles, ONE all-reduce of (S+1) d + 2 d doubles
// replaces S per-step exchanges of sum x, and the integrator itself runs without any synchronisation.  The table is
// exactly what per-step recomputation gives in exact arithmetic (rounding differs at 1e-7; tests compare with the
// oracle's per-step empirical mean).
// ------------------------------------------------------------------------------------------------------------
// sums [(n_draws) d + 2 d] doubles, accumulated with atomics (caller zeroes): [s][i] sum xi_{s,i};  tail: sum q0, sum p0
__global__ void __launch_bounds__(256) meanfield_noise_sums_kernel(const float* __restrict__ z0, int64_t n, int d,
                                                                   int n_draws, uint64_t seed, uint64_t particle_offset,
                                                                   uint32_t step_offset, double* __restrict__ sums) {
  __shared__ float red[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t first = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (int s = -1; s < n_draws; ++s) {  // s == -1: the initial state sums (2 passes of up to 32 components)
    for (int half = 0; half < (s < 0 ? 2 : 1); ++half) {
      float acc[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[i] = 0.f;
      for (int64_t p = first; p < n; p += stride) {
        if (s < 0) {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (i < d) acc[i] += z0[p * 2 * d + half * d + i];
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (4 * j < d) {
              float r4[4];
              philox_normal4(seed, particle_offset + (uint64_t)p, step_offset + (uint32_t)s, (uint32_t)j, r4);
#pragma unroll
              for (int k = 0; k < 4; ++k)
                if (4 * j + k < d) acc[4 * j + k] += r4[k];
            }
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        if (i < d) {
          const float w = warp_sum(acc[i]);
          if (lane == 0) red[warp][i] = w;
        }
      }
      __syncthreads();
      if (threadIdx.x < d) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += (double)red[w][threadIdx.x];
        double* dst = s < 0 ? sums + (int64_t)n_draws * d + half * d : sums + (int64_t)s * d;
        atomicAdd(dst + threadIdx.x, t);
      }
      __syncthreads();
    }
  }
}

// one block, d <= 32 threads active: xbar [n_draws][d] (mean position BEFORE step s) and shift [n_draws][d] = A xbar_s
__global__ void meanfield_xbar_table_kernel(const double* __restrict__ sums, double inv_n, int d, int n_draws, double dt,
                                            double gamma, const float* __restrict__ A, float* __restrict__ xbar,
                                            float* __restrict__ shift) {
  __shared__ double qs[32];
  const int i = threadIdx.x;
  double q = 0.0, p = 0.0;
  if (i < d) {
    q = sums[(int64_t)n_draws * d + i] * inv_n;
    p = sums[(int64_t)n_draws * d + d + i] * inv_n;
  }
  for (int s = 0; s < n_draws; ++s) {
    if (i < d) qs[i] = q;
    __syncthreads();
    if (i < d) {
      if (xbar) xbar[(int64_t)s * d + i] = (float)q;
      double a = 0.0;
      for (int k = 0; k < d; ++k) a += (double)A[i * d + k] * qs[k];
      shift[(int64_t)s * d + i] = (float)a;
      const double h = s == 0 ? 0.0 : dt;  // tau0 == 0: the first step of the reference schedule has h = 0
      p = (1.0 - gamma * h) * p + sqrt(2.0 * h) * (sums[(int64_t)s * d + i] * inv_n);
      q += h * p;
    }
    __syncthreads();
  }
}

// z = mu + cov_half xi   (core/distribution.py:64-65); one thread per sample, dim <= 64
__global__ void gaussian_sample_kernel(float* out, int64_t n, int dim, const float* __restrict__ mu,
                                       const float* __restrict__ cov_half, uint64_t seed,
                                       uint64_t particle_offset, int layout) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  float xi[64];
  for (int j = 0; j < (dim + 3) / 4; ++j) {
    float r4[4];
    philox_normal4(seed, particle_offset + (uint64_t)p, kTagInit, (uint32_t)j, r4);
    for (int k = 0; k < 4; ++k) xi[4 * j + k] = r4[k];
  }
  for (int i = 0; i < dim; ++i) {
    float s = mu ? mu[i] : 0.0f;
    if (cov_half) {
      for (int k = 0; k < dim; ++k) s = fmaf(cov_half[i * dim + k], xi[k], s);
    } else {
      s += xi[i];
    }
    out[elem_index(layout, p, i, n, dim)] = s;
  }
}

}  // namespace pdeip

using namespace pdeip;

// validates the arguments common to every K1 entry point and fills the argument block
static int integrate_args(IntegrateArgs& a, const float* z0, float* z_last, float* traj, float* tau,
                          int64_t n_particles, int d, int n_steps, float dt, float gamma, const float* noise,
                          const float* tau0, uint64_t seed, uint64_t particle_offset, uint32_t step_offset, int schedule,
                          int state_layout, int traj_layout, int emit_every, int emit_offset, int emit_drift, int path) {
  PDEIP_REQUIRE(path == PDEIP_PATH_FP32 || path == PDEIP_PATH_TENSOR, PDEIP_ERR_INVALID_ARG, "unknown path %d", path);
  PDEIP_REQUIRE(z0 != nullptr, PDEIP_ERR_INVALID_ARG, "z0 is NULL");
  PDEIP_REQUIRE(n_particles >= 0 && d >= 1 && d <= 32, PDEIP_ERR_UNSUPPORTED,
                "integrator supports 1 <= d <= 32 (got d=%d)", d);
  PDEIP_REQUIRE(n_steps >= 1, PDEIP_ERR_INVALID_ARG, "n_steps must be >= 1");
  PDEIP_REQUIRE(schedule == PDEIP_SCHEDULE_REFERENCE || schedule == PDEIP_SCHEDULE_UNIFORM,
                PDEIP_ERR_INVALID_ARG, "unknown schedule %d", schedule);
  PDEIP_REQUIRE(state_layout == PDEIP_LAYOUT_AOS || state_layout == PDEIP_LAYOUT_SOA, PDEIP_ERR_INVALID_ARG,
                "unknown state layout %d", state_layout);
  PDEIP_REQUIRE(traj_layout >= 0 && traj_layout <= 3, PDEIP_ERR_INVALID_ARG, "unknown trajectory layout %d",
                traj_layout);
  PDEIP_REQUIRE(traj_layout != PDEIP_TRAJ_BLOCK128 || traj == nullptr || n_particles % 128 == 0, PDEIP_ERR_INVALID_ARG,
                "PDEIP_TRAJ_BLOCK128 needs n_particles %% 128 == 0 (got %lld)", (long long)n_particles);
  PDEIP_REQUIRE(emit_every >= 1 && emit_offset >= 0 && emit_offset < emit_every, PDEIP_ERR_INVALID_ARG,
                "emit_every/emit_offset out of range");
  a.z0 = z0; a.z_last = z_last; a.traj = traj; a.tau = tau; a.n = n_particles; a.d = d;
  a.n_steps = n_steps; a.dt = dt; a.gamma = gamma; a.drift_params = nullptr;
  a.n_gaussian = 0; a.inv_sigma2 = 1.0f; a.layers = 0;
  a.noise = noise; a.tau0 = tau0; a.seed = seed; a.particle_offset = particle_offset;
  a.step_offset = step_offset; a.schedule = schedule; a.state_layout = state_layout;
  a.traj_layout = traj_layout; a.emit_every = emit_every; a.emit_offset = emit_offset;
  a.emit_drift = emit_drift ? 1 : 0;
  a.rk = philox_round_keys(seed);
  const int n_samples = n_steps;  // both schedules expose n_steps samples
  a.s_emit = (n_samples - emit_offset + emit_every - 1) / emit_every;
  return PDEIP_OK;
}

extern "C" int pdeip_kl_integrate_path(const float* z0, float* z_last, float* traj, float* tau,
                                       int64_t n_particles, int d, int n_steps, float dt, float gamma,
                                       int drift_kind, const float* drift_params, int n_gaussian, float sigma,
                                       const float* noise, const float* tau0, uint64_t seed,
                                       uint64_t particle_offset, uint32_t step_offset, int schedule,
                                       int state_layout, int traj_layout, int emit_every, int emit_offset,
                                       int emit_drift, int path, void* stream) {
  IntegrateArgs a;
  const int rc = integrate_args(a, z0, z_last, traj, tau, n_particles, d, n_steps, dt, gamma, noise, tau0, seed,
                                particle_offset, step_offset, schedule, state_layout, traj_layout, emit_every,
                                emit_offset, emit_drift, path);
  if (rc != PDEIP_OK) return rc;
  PDEIP_REQUIRE(drift_kind == PDEIP_DRIFT_NONE || drift_params != nullptr, PDEIP_ERR_INVALID_ARG,
                "drift_params is NULL");
  PDEIP_REQUIRE(drift_kind != PDEIP_DRIFT_GMM || (n_gaussian >= 1 && sigma > 0.0f), PDEIP_ERR_INVALID_ARG,
                "GMM drift needs n_gaussian >= 1 and sigma > 0");
  if (n_particles == 0) return PDEIP_OK;
  a.drift_params = drift_params;
  a.n_gaussian = n_gaussian; a.inv_sigma2 = drift_kind == PDEIP_DRIFT_GMM ? 1.0f / (sigma * sigma) : 1.0f;
  cudaStream_t st = (cudaStream_t)stream;
  if (d <= 2) return launch_integrate<2>(a, drift_kind, path, st);
  if (d <= 4) return launch_integrate<4>(a, drift_kind, path, st);
  if (d <= 8) return launch_integrate<8>(a, drift_kind, path, st);
  if (d <= 16) return launch_integrate<16>(a, drift_kind, path, st);
  return launch_integrate<32>(a, drift_kind, path, st);
}

extern "C" int pdeip_kl_integrate_model(const float* z0, float* z_last, float* traj, float* tau,
                                        int64_t n_particles, int d, int n_steps, float dt, float gamma,
                                        int model_kind, const float* params, int hidden, int layers, int n_gaussian,
                                        const float* noise, const float* tau0, uint64_t seed,
                                        uint64_t particle_offset, uint32_t step_offset, int schedule,
                                        int state_layout, int traj_layout, int emit_every, int emit_offset,
                                        int emit_drift, int path, void* stream) {
  PDEIP_REQUIRE(model_kind == PDEIP_MODEL_MLP || model_kind == PDEIP_MODEL_GMM || model_kind == PDEIP_MODEL_QUADRATIC,
                PDEIP_ERR_INVALID_ARG, "unknown model kind %d", model_kind);
  PDEIP_REQUIRE(params != nullptr, PDEIP_ERR_INVALID_ARG, "params is NULL");
  PDEIP_REQUIRE(d >= 1 && d <= 32, PDEIP_ERR_UNSUPPORTED, "integrator supports 1 <= d <= 32 (got d=%d)", d);
  if (model_kind == PDEIP_MODEL_GMM) {
    // the parametric GMM model (learned centres, sigma = 1) is exactly the GMM drift, on all of its kernels
    PDEIP_REQUIRE(n_gaussian >= 1, PDEIP_ERR_INVALID_ARG, "GMM model needs n_gaussian >= 1 (got %d)", n_gaussian);
    return pdeip_kl_integrate_path(z0, z_last, traj, tau, n_particles, d, n_steps, dt, gamma, PDEIP_DRIFT_GMM, params,
                                   n_gaussian, 1.0f, noise, tau0, seed, particle_offset, step_offset, schedule,
                                   state_layout, traj_layout, emit_every, emit_offset, emit_drift, path, stream);
  }
  if (model_kind == PDEIP_MODEL_MLP) {
    PDEIP_REQUIRE(hidden == 32, PDEIP_ERR_UNSUPPORTED,
                  "MLP drift is built for hidden_dim == 32 (pad smaller widths with zeros); got %d", hidden);
    PDEIP_REQUIRE(layers >= 1 && layers <= 8, PDEIP_ERR_UNSUPPORTED, "MLP drift supports 1 <= layers <= 8 (got %d)",
                  layers);
  }
  IntegrateArgs a;
  const int rc = integrate_args(a, z0, z_last, traj, tau, n_particles, d, n_steps, dt, gamma, noise, tau0, seed,
                                particle_offset, step_offset, schedule, state_layout, traj_layout, emit_every,
                                emit_offset, emit_drift, path);
  if (rc != PDEIP_OK) return rc;
  if (n_particles == 0) return PDEIP_OK;
  a.drift_params = params;
  a.layers = model_kind == PDEIP_MODEL_MLP ? layers : 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (d <= 2) return launch_integrate_model<2>(a, model_kind, path, st);
  if (d <= 4) return launch_integrate_model<4>(a, model_kind, path, st);
  if (d <= 8) return launch_integrate_model<8>(a, model_kind, path, st);
  if (d <= 16) return launch_integrate_model<16>(a, model_kind, path, st);
  return launch_integrate_model<32>(a, model_kind, path, st);
}

// the arguments of the overdamped entry points: those of K1 on the UNIFORM schedule with no friction, tau or tau0
static int overdamped_args(IntegrateArgs& a, const float* x0, float* x_last, float* traj, int64_t n_particles, int d,
                           int n_steps, float dt, const float* noise, uint64_t seed, uint64_t particle_offset,
                           uint32_t step_offset, int state_layout, int traj_layout, int emit_every, int emit_offset,
                           int emit_drift, int path) {
  PDEIP_REQUIRE(x0 != nullptr, PDEIP_ERR_INVALID_ARG, "x0 is NULL");
  return integrate_args(a, x0, x_last, traj, nullptr, n_particles, d, n_steps, dt, 0.0f, noise, nullptr, seed,
                        particle_offset, step_offset, PDEIP_SCHEDULE_UNIFORM, state_layout, traj_layout, emit_every,
                        emit_offset, emit_drift, path);
}

extern "C" int pdeip_overdamped_integrate(const float* x0, float* x_last, float* traj, int64_t n_particles, int d,
                                          int n_steps, float dt, int drift_kind, const float* drift_params,
                                          int n_gaussian, float sigma, const float* noise, uint64_t seed,
                                          uint64_t particle_offset, uint32_t step_offset, int state_layout,
                                          int traj_layout, int emit_every, int emit_offset, int emit_drift, int path,
                                          void* stream) {
  PDEIP_REQUIRE(drift_kind != PDEIP_DRIFT_MEANFIELD_TABLE, PDEIP_ERR_UNSUPPORTED,
                "PDEIP_DRIFT_MEANFIELD_TABLE encodes the underdamped mean recursion; the overdamped step does not take it");
  PDEIP_REQUIRE(drift_kind == PDEIP_DRIFT_NONE || drift_kind == PDEIP_DRIFT_LINEAR || drift_kind == PDEIP_DRIFT_GMM ||
                    drift_kind == PDEIP_DRIFT_MEANFIELD,
                PDEIP_ERR_INVALID_ARG, "unknown drift kind %d", drift_kind);
  IntegrateArgs a;
  const int rc = overdamped_args(a, x0, x_last, traj, n_particles, d, n_steps, dt, noise, seed, particle_offset,
                                 step_offset, state_layout, traj_layout, emit_every, emit_offset, emit_drift, path);
  if (rc != PDEIP_OK) return rc;
  PDEIP_REQUIRE(drift_kind == PDEIP_DRIFT_NONE || drift_params != nullptr, PDEIP_ERR_INVALID_ARG,
                "drift_params is NULL");
  PDEIP_REQUIRE(drift_kind != PDEIP_DRIFT_GMM || (n_gaussian >= 1 && sigma > 0.0f), PDEIP_ERR_INVALID_ARG,
                "GMM drift needs n_gaussian >= 1 and sigma > 0");
  if (n_particles == 0) return PDEIP_OK;
  a.drift_params = drift_params;
  a.n_gaussian = n_gaussian; a.inv_sigma2 = drift_kind == PDEIP_DRIFT_GMM ? 1.0f / (sigma * sigma) : 1.0f;
  cudaStream_t st = (cudaStream_t)stream;
  if (d <= 2) return launch_overdamped<2>(a, drift_kind, path, st);
  if (d <= 4) return launch_overdamped<4>(a, drift_kind, path, st);
  if (d <= 8) return launch_overdamped<8>(a, drift_kind, path, st);
  if (d <= 16) return launch_overdamped<16>(a, drift_kind, path, st);
  return launch_overdamped<32>(a, drift_kind, path, st);
}

extern "C" int pdeip_overdamped_integrate_model(const float* x0, float* x_last, float* traj, int64_t n_particles,
                                                int d, int n_steps, float dt, int model_kind, const float* params,
                                                int hidden, int layers, int n_gaussian, const float* noise,
                                                uint64_t seed, uint64_t particle_offset, uint32_t step_offset,
                                                int state_layout, int traj_layout, int emit_every, int emit_offset,
                                                int emit_drift, int path, void* stream) {
  PDEIP_REQUIRE(model_kind == PDEIP_MODEL_MLP || model_kind == PDEIP_MODEL_GMM || model_kind == PDEIP_MODEL_QUADRATIC,
                PDEIP_ERR_INVALID_ARG, "unknown model kind %d", model_kind);
  PDEIP_REQUIRE(params != nullptr, PDEIP_ERR_INVALID_ARG, "params is NULL");
  PDEIP_REQUIRE(d >= 1 && d <= 32, PDEIP_ERR_UNSUPPORTED, "integrator supports 1 <= d <= 32 (got d=%d)", d);
  if (model_kind == PDEIP_MODEL_GMM) {
    // the parametric GMM model (learned centres, sigma = 1) is exactly the GMM drift
    PDEIP_REQUIRE(n_gaussian >= 1, PDEIP_ERR_INVALID_ARG, "GMM model needs n_gaussian >= 1 (got %d)", n_gaussian);
    return pdeip_overdamped_integrate(x0, x_last, traj, n_particles, d, n_steps, dt, PDEIP_DRIFT_GMM, params,
                                      n_gaussian, 1.0f, noise, seed, particle_offset, step_offset, state_layout,
                                      traj_layout, emit_every, emit_offset, emit_drift, path, stream);
  }
  if (model_kind == PDEIP_MODEL_MLP) {
    PDEIP_REQUIRE(hidden == 32, PDEIP_ERR_UNSUPPORTED,
                  "MLP drift is built for hidden_dim == 32 (pad smaller widths with zeros); got %d", hidden);
    PDEIP_REQUIRE(layers >= 1 && layers <= 8, PDEIP_ERR_UNSUPPORTED, "MLP drift supports 1 <= layers <= 8 (got %d)",
                  layers);
  }
  IntegrateArgs a;
  const int rc = overdamped_args(a, x0, x_last, traj, n_particles, d, n_steps, dt, noise, seed, particle_offset,
                                 step_offset, state_layout, traj_layout, emit_every, emit_offset, emit_drift, path);
  if (rc != PDEIP_OK) return rc;
  if (n_particles == 0) return PDEIP_OK;
  a.drift_params = params;
  a.layers = model_kind == PDEIP_MODEL_MLP ? layers : 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (d <= 2) return launch_overdamped_model<2>(a, model_kind, path, st);
  if (d <= 4) return launch_overdamped_model<4>(a, model_kind, path, st);
  if (d <= 8) return launch_overdamped_model<8>(a, model_kind, path, st);
  if (d <= 16) return launch_overdamped_model<16>(a, model_kind, path, st);
  return launch_overdamped_model<32>(a, model_kind, path, st);
}

extern "C" int pdeip_kl_integrate(const float* z0, float* z_last, float* traj, float* tau,
                                  int64_t n_particles, int d, int n_steps, float dt, float gamma,
                                  int drift_kind, const float* drift_params, int n_gaussian, float sigma,
                                  const float* noise, const float* tau0, uint64_t seed,
                                  uint64_t particle_offset, uint32_t step_offset, int schedule,
                                  int state_layout, int traj_layout, int emit_every, int emit_offset,
                                  int emit_drift, void* stream) {
  return pdeip_kl_integrate_path(z0, z_last, traj, tau, n_particles, d, n_steps, dt, gamma, drift_kind, drift_params,
                                 n_gaussian, sigma, noise, tau0, seed, particle_offset, step_offset, schedule,
                                 state_layout, traj_layout, emit_every, emit_offset, emit_drift, PDEIP_PATH_FP32, stream);
}

extern "C" int pdeip_philox_normals(float* out, int64_t n_particles, int n_draws, int d, uint64_t seed,
                                    uint64_t particle_offset, uint32_t step_offset, void* stream) {
  PDEIP_REQUIRE(out && n_particles >= 0 && n_draws >= 1 && d >= 1, PDEIP_ERR_INVALID_ARG, "bad arguments");
  const int64_t total = n_particles * n_draws;
  if (total == 0) return PDEIP_OK;
  philox_normals_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      out, n_particles, n_draws, d, seed, particle_offset, step_offset);
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}

extern "C" int pdeip_philox_uniforms(float* out, int64_t n_particles, uint64_t seed, uint64_t particle_offset,
                                     void* stream) {
  PDEIP_REQUIRE(out && n_particles >= 0, PDEIP_ERR_INVALID_ARG, "bad arguments");
  if (n_particles == 0) return PDEIP_OK;
  philox_uniforms_kernel<<<(unsigned)((n_particles + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      out, n_particles, seed, particle_offset);
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}

extern "C" int pdeip_philox_raw(const uint32_t* ctr, const uint32_t* key, uint32_t* out, int64_t n,
                                void* stream) {
  PDEIP_REQUIRE(ctr && key && out && n >= 0, PDEIP_ERR_INVALID_ARG, "bad arguments");
  if (n == 0) return PDEIP_OK;
  philox_raw_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ctr, key, out, n);
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}

extern "C" int pdeip_gaussian_sample(float* out, int64_t n, int dim, const float* mu, const float* cov_half,
                                     uint64_t seed, uint64_t particle_offset, int layout, void* stream) {
  PDEIP_REQUIRE(out && n >= 0 && dim >= 1 && dim <= 64, PDEIP_ERR_UNSUPPORTED,
                "gaussian_sample supports 1 <= dim <= 64 (got %d)", dim);
  PDEIP_REQUIRE(layout == PDEIP_LAYOUT_AOS || layout == PDEIP_LAYOUT_SOA, PDEIP_ERR_INVALID_ARG, "bad layout");
  if (n == 0) return PDEIP_OK;
  gaussian_sample_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      out, n, dim, mu, cov_half, seed, particle_offset, layout);
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}

extern "C" int pdeip_meanfield_noise_sums(const float* z0, int64_t n_particles, int d, int n_steps, uint64_t seed,
                                          uint64_t particle_offset, uint32_t step_offset, double* sums, void* stream) {
  PDEIP_REQUIRE(z0 && sums, PDEIP_ERR_INVALID_ARG, "NULL argument");
  PDEIP_REQUIRE(n_particles >= 0 && d >= 1 && d <= 32 && n_steps >= 1, PDEIP_ERR_UNSUPPORTED,
                "meanfield_noise_sums supports 1 <= d <= 32, n_steps >= 1");
  if (n_particles == 0) return PDEIP_OK;
  int64_t blocks = (n_particles + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (blocks > cap) blocks = cap;
  meanfield_noise_sums_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(z0, n_particles, d, n_steps + 1, seed,
                                                                                 particle_offset, step_offset, sums);
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}

extern "C" int pdeip_meanfield_xbar_table(const double* sums, int64_t n_global, int d, int n_steps, float dt, float gamma,
                                          const float* A, float* xbar, float* drift_table, void* stream) {
  PDEIP_REQUIRE(sums && A && drift_table, PDEIP_ERR_INVALID_ARG, "NULL argument");
  PDEIP_REQUIRE(n_global >= 1 && d >= 1 && d <= 32 && n_steps >= 1, PDEIP_ERR_UNSUPPORTED,
                "meanfield_xbar_table supports 1 <= d <= 32, n_steps >= 1, n_global >= 1");
  meanfield_xbar_table_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(sums, 1.0 / (double)n_global, d, n_steps + 1, (double)dt,
                                                                  (double)gamma, A, xbar, drift_table);
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}
