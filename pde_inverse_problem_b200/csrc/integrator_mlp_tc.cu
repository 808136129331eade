// integrator_mlp_tc.cu — K1 under a fitted MLP's potential on the tensor cores (PDEIP_PATH_TENSOR of
// pdeip_kl_integrate_model, MLP 32 x 2, d = 8, 16 or 32).
//
// One CTA = 128 particles = one 128-row tcgen05 tile, thread = particle = TMEM lane; (q, p) stay in registers for all
// S + 1 steps.  grad V_theta(x) of V = |u|^2 (core/model.py:51-62) is the primal chain and its input-gradient chain:
//
//   F0  z0 = x W0            -> t0 = tanh(z0 + b0)        TMEM cols [0, 32)   (z0 stays there for B0's epilogue)
//   F1  z1 = t0 W1           -> t1 = tanh(z1 + b1)        TMEM cols [32, 64)  (z1 stays there for B2's epilogue)
//   F2  u  = t1 W2 (N = 48)  -> za = 2 (u + b2)           TMEM cols [64, 112)
//   B2  za W2^T              -> za1 = . (1 - t1^2)         TMEM cols [64, 96)
//   B1  za1 W1^T             -> za0 = . (1 - t0^2)
//   B0  za0 W0^T (N = d)     -> grad V_theta, state update
//
// Weights stay resident in shared memory as bf16 hi + lo tiles W_l^T [out][in]: the forward GEMMs read them K-major, the
// backward GEMMs read the same bytes through the MN-major (transposed) view.  Every GEMM carries the hi + lo split on
// both operands (a_hi w_hi + a_lo w_hi + a_hi w_lo, ~2^-17 relative per product); the biases, tanh and the state update
// are fp32.  The step's Philox normals are drawn while F0 is in flight.  Bounded mbarrier waits set status word 1 (the
// integrator word) on a timeout, as kl_integrate_tc_kernel does.  Same Philox stream, tau0, step schedule and outputs
// as the fp32 kernel of pdeip_kl_integrate_model.
//
// OD = true is the overdamped variant (PDEIP_PATH_TENSOR of pdeip_overdamped_integrate_model): the state per thread is
// x alone, S steps x' = x - dt grad V_theta(x) + sqrt(2 dt) xi with no tau0; x + sqrt(2 dt) xi is formed while F0 runs
// and B0's epilogue subtracts dt grad V_theta and emits [x, grad V_theta].  A trajectory run makes one extra drift
// evaluation (GEMM chain without an update) for the last sample's drift.  Same weight tiles, TMEM map and hand-offs.
#include "common.cuh"
#include "integrator_args.cuh"
#include "mlp_thread.cuh"
#include "philox.cuh"
#include "umma.cuh"

#include <stdlib.h>

namespace pdeip {

int* tensor_status_word();  // residual_tensor.cu

namespace imlp {
using namespace umma;

constexpr int kH = 32, kNO = 48;  // hidden width, output width padded to a multiple of 16

template <int DP>
struct Cfg {
  static constexpr int DK = DP < 16 ? 16 : DP;                // K of F0 / N of B0 (multiple of 16)
  static constexpr uint32_t A_BYTES = 128 * 2 * kNO * 2;      // activation tile [128][a_hi(KW) | a_lo(KW)], KW <= 48
  static constexpr uint32_t RG_W0 = (DK / 8) * 128, RG_W = (kH / 8) * 128;
  static constexpr uint32_t W0_BYTES = kH * DK * 2, W1_BYTES = kH * kH * 2, W2_BYTES = kNO * kH * 2;
  static constexpr uint32_t O_A = 0;
  static constexpr uint32_t O_W0H = O_A + A_BYTES, O_W0L = O_W0H + W0_BYTES;
  static constexpr uint32_t O_W1H = O_W0L + W0_BYTES, O_W1L = O_W1H + W1_BYTES;
  static constexpr uint32_t O_W2H = O_W1L + W1_BYTES, O_W2L = O_W2H + W2_BYTES;
  static constexpr uint32_t O_B = O_W2L + W2_BYTES;            // fp32 biases b0 (32) | b1 (32) | b2 (48, zero padded)
  static constexpr uint32_t O_MISC = O_B + (2 * kH + kNO) * 4;  // mbarrier (8 B), TMEM base (4 B), dead flag (4 B)
  static constexpr uint32_t TOTAL = O_MISC + 64;
  static constexpr uint32_t TMEM_COLS = 128;
};

__device__ __forceinline__ uint32_t pack_bf2(float a, float b) {
  const __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&t);
}
// v = hi + lo, both bf16
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  hi = pack_bf2(a, b);
  lo = pack_bf2(a - __uint_as_float(hi << 16), b - __uint_as_float(hi & 0xffff0000u));
}
__device__ __forceinline__ void tm_ld16(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tm_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// this thread's row of the activation tile: v[0, KW) as hi (columns [0, KW)) and lo (columns [KW, 2 KW))
template <int KW>
__device__ __forceinline__ void store_split_row(uint8_t* tileA, int tid, const float (&v)[KW]) {
  constexpr uint32_t RG = (2 * KW / 8) * 128;
  uint8_t* const row = tileA + (uint32_t)(tid & 7) * 16u + (uint32_t)(tid >> 3) * RG;
#pragma unroll
  for (int cg = 0; cg < KW / 8; ++cg) {
    uint4 hi, lo;
    split2(v[8 * cg], v[8 * cg + 1], hi.x, lo.x);
    split2(v[8 * cg + 2], v[8 * cg + 3], hi.y, lo.y);
    split2(v[8 * cg + 4], v[8 * cg + 5], hi.z, lo.z);
    split2(v[8 * cg + 6], v[8 * cg + 7], hi.w, lo.w);
    *reinterpret_cast<uint4*>(row + cg * 128) = hi;
    *reinterpret_cast<uint4*>(row + (KW / 8 + cg) * 128) = lo;
  }
}

// W^T tile [rows = out][cols = in] (hi and lo) of W [in][out] (row-major, n_in x n_out in global memory)
__device__ __forceinline__ void stage_weight(uint8_t* hi_t, uint8_t* lo_t, uint32_t rg, int rows, int cols,
                                             const float* __restrict__ W, int n_in, int n_out, int tid) {
  for (int idx = tid; idx < rows * cols; idx += 128) {
    const int r = idx / cols, c = idx - r * cols;  // r = out unit, c = in unit
    const float w = (r < n_out && c < n_in) ? W[c * n_out + r] : 0.f;
    const __nv_bfloat16 h = __float2bfloat16_rn(w);
    const __nv_bfloat16 l = __float2bfloat16_rn(w - __bfloat162float(h));
    const uint32_t off = chunk_off(r, c >> 3, rg) + (uint32_t)(c & 7) * 2u;
    *reinterpret_cast<__nv_bfloat16*>(hi_t + off) = h;
    *reinterpret_cast<__nv_bfloat16*>(lo_t + off) = l;
  }
}

// TRAJ: 0 = terminal state only, 1 = PDEIP_TRAJ_BLOCK128, 2 = PDEIP_TRAJ_TIME_SOA (both with grad V_theta)
template <int DP, int TRAJ, int MINB, bool OD = false>
__global__ void __launch_bounds__(128, MINB) kl_integrate_mlp_tc_kernel(const IntegrateArgs a, int* status) {
  using S = Cfg<DP>;
  constexpr int DK = S::DK;
  constexpr bool BLK = TRAJ == 1;
  extern __shared__ __align__(128) uint8_t sm[];
  const int tid = threadIdx.x, warp = tid >> 5;
  uint64_t* mbar_p = reinterpret_cast<uint64_t*>(sm + S::O_MISC);
  uint32_t* tmem_p = reinterpret_cast<uint32_t*>(sm + S::O_MISC + 8);
  volatile int* dead_p = reinterpret_cast<volatile int*>(sm + S::O_MISC + 12);
  const float* bias = reinterpret_cast<const float*>(sm + S::O_B);

  // ---- one-time set-up: TMEM, mbarrier, resident weight tiles ------------------------------------------------
  if (warp == 0) {
    tmem_alloc(smem_u32(tmem_p), S::TMEM_COLS);
    tmem_relinquish();
  }
  if (tid == 0) {
    mbar_init(smem_u32(mbar_p), 1);
    fence_mbar_init();
    *dead_p = 0;
  }
  const MlpShape<kH> sh{DP, 2};
  stage_weight(sm + S::O_W0H, sm + S::O_W0L, S::RG_W0, kH, DK, a.drift_params + sh.w_off(0), DP, kH, tid);
  stage_weight(sm + S::O_W1H, sm + S::O_W1L, S::RG_W, kH, kH, a.drift_params + sh.w_off(1), kH, kH, tid);
  stage_weight(sm + S::O_W2H, sm + S::O_W2L, S::RG_W, kNO, kH, a.drift_params + sh.w_off(2), kH, kOut, tid);
  {
    float* b = reinterpret_cast<float*>(sm + S::O_B);
    for (int i = tid; i < 2 * kH + kNO; i += 128) {
      float v = 0.f;
      if (i < kH) v = a.drift_params[sh.b_off(0) + i];
      else if (i < 2 * kH) v = a.drift_params[sh.b_off(1) + i - kH];
      else if (i - 2 * kH < kOut) v = a.drift_params[sh.b_off(2) + i - 2 * kH];
      b[i] = v;
    }
  }
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tbase = *tmem_p;
  const uint32_t t_row = tbase + ((uint32_t)(warp * 32) << 16);
  const uint32_t mbar = smem_u32(mbar_p);
  const uint32_t sA = smem_u32(sm + S::O_A);
  const uint32_t sW0H = smem_u32(sm + S::O_W0H), sW0L = smem_u32(sm + S::O_W0L), sW1H = smem_u32(sm + S::O_W1H),
                 sW1L = smem_u32(sm + S::O_W1L), sW2H = smem_u32(sm + S::O_W2H), sW2L = smem_u32(sm + S::O_W2L);
  constexpr uint32_t RG_X = (2 * DK / 8) * 128, RG_32 = (2 * kH / 8) * 128, RG_48 = (2 * kNO / 8) * 128;
  uint32_t phase = 0;

  // Rows past the end of a ragged last tile repeat the last particle (same id, same values to the same addresses).
  const int64_t n_raw = (int64_t)blockIdx.x * 128 + tid;
  const int64_t n = n_raw < a.n ? n_raw : a.n - 1;
  const uint64_t pid = a.particle_offset + (uint64_t)n;
  float q[DP], p[DP];
  if constexpr (OD) {
    const float4* z4 = reinterpret_cast<const float4*>(a.z0 + n * DP);
#pragma unroll
    for (int i4 = 0; i4 < DP / 4; ++i4) {
      const float4 tq = z4[i4];
      q[4 * i4] = tq.x; q[4 * i4 + 1] = tq.y; q[4 * i4 + 2] = tq.z; q[4 * i4 + 3] = tq.w;
    }
  } else {
    const float4* z4 = reinterpret_cast<const float4*>(a.z0 + n * (2 * DP));
#pragma unroll
    for (int i4 = 0; i4 < DP / 4; ++i4) {
      const float4 tq = z4[i4], tp = z4[DP / 4 + i4];
      q[4 * i4] = tq.x; q[4 * i4 + 1] = tq.y; q[4 * i4 + 2] = tq.z; q[4 * i4 + 3] = tq.w;
      p[4 * i4] = tp.x; p[4 * i4 + 1] = tp.y; p[4 * i4 + 2] = tp.z; p[4 * i4 + 3] = tp.w;
    }
  }
  const float t0 = OD ? 0.f : philox_uniform01(a.seed, pid, kTagTau0) * a.dt;  // sampling_utils.py:32
  const int Sn = a.n_steps;
  constexpr int CW = OD ? 2 * DP : 3 * DP;  // floats per emitted sample: [x, v, grad V] or (OD) [x, grad V]
  // BLK: element (sample s, tile t, component c, lane l) at ((s T + t) CW + c) 128 + l ; SOA: c S N + s N + n
  const int64_t plane = BLK ? 128 : (int64_t)Sn * a.n;
  const int64_t sstride = BLK ? (int64_t)gridDim.x * (CW * 128) : a.n;
  float* o = TRAJ == 0 ? nullptr : (BLK ? a.traj + ((int64_t)blockIdx.x * CW * 128 + tid) : a.traj + n);
  // OD: S steps, and with a trajectory one more drift evaluation (s == S) for the last sample
  const int s_end = OD ? Sn + (TRAJ != 0 ? 1 : 0) : Sn + 1;

  auto wait_commit = [&]() {
    if (!*dead_p) {
      if (!mbar_wait(mbar, phase, 1u << 22)) {
        *dead_p = 1;
        atomicExch(status, 2);
      }
    }
    phase ^= 1u;
    fence_after_sync();
  };
  auto handoff = [&]() {  // the activation tile is written: make it visible to the tensor cores
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
  };
  // tanh(z_l + b_l) of the 32 hidden units of layer l from this thread's TMEM row
  auto hidden = [&](int l, float (&t)[kH]) {
    tm_ld16(t_row + 32 * l, t);
    tm_ld16(t_row + 32 * l + 16, t + 16);
    tm_wait_ld();
#pragma unroll
    for (int j = 0; j < kH; ++j) t[j] = tanhf(t[j] + bias[kH * l + j]);
  };

#pragma unroll 1
  for (int s = 0; OD ? s < s_end : s <= Sn; ++s) {
    const float h = OD ? a.dt : ((s == 0) ? t0 : ((s == Sn) ? a.dt - t0 : a.dt));  // sampling_utils.py:33,45-46
    const float sq = sqrtf(h) * 1.41421356237309515f;
    const float dmp = 1.f - a.gamma * h;

    {  // F0
      float x[DK];
#pragma unroll
      for (int i = 0; i < DK; ++i) x[i] = i < DP ? q[i] : 0.f;
      store_split_row<DK>(sm + S::O_A, tid, x);
    }
    handoff();
    if (warp == 0 && elect_one()) {
      fence_after_sync();
      gemm_kk(tbase, sA, RG_X, 0, sW0H, S::RG_W0, 0, DK, kH, 0u);
      gemm_kk(tbase, sA, RG_X, DK, sW0H, S::RG_W0, 0, DK, kH, 1u);
      gemm_kk(tbase, sA, RG_X, 0, sW0L, S::RG_W0, 0, DK, kH, 1u);
      commit(mbar);
    }
    __syncwarp();
    // the drift-independent part of the kick while F0 runs: p <- p (1 - gamma h) + sqrt(2h) xi
    // (OD: x <- x + sqrt(2h) xi; x is in the activation tile already)
    if (!OD || s < Sn) {
#pragma unroll
      for (int j = 0; j < DP / 4; ++j) {
        float r4[4];
        philox_normal4_rk(a.rk, pid, a.step_offset + (uint32_t)s, (uint32_t)j, r4);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if constexpr (OD) q[4 * j + k] = fmaf(sq, r4[k], q[4 * j + k]);
          else p[4 * j + k] = fmaf(sq, r4[k], p[4 * j + k] * dmp);
        }
      }
    }
    wait_commit();

    {  // F0 epilogue -> F1
      float t[kH];
      hidden(0, t);
      store_split_row<kH>(sm + S::O_A, tid, t);
    }
    handoff();
    if (warp == 0 && elect_one()) {
      fence_after_sync();
      gemm_kk(tbase + 32, sA, RG_32, 0, sW1H, S::RG_W, 0, kH, kH, 0u);
      gemm_kk(tbase + 32, sA, RG_32, kH, sW1H, S::RG_W, 0, kH, kH, 1u);
      gemm_kk(tbase + 32, sA, RG_32, 0, sW1L, S::RG_W, 0, kH, kH, 1u);
      commit(mbar);
    }
    __syncwarp();
    wait_commit();

    {  // F1 epilogue -> F2
      float t[kH];
      hidden(1, t);
      store_split_row<kH>(sm + S::O_A, tid, t);
    }
    handoff();
    if (warp == 0 && elect_one()) {
      fence_after_sync();
      gemm_kk(tbase + 64, sA, RG_32, 0, sW2H, S::RG_W, 0, kH, kNO, 0u);
      gemm_kk(tbase + 64, sA, RG_32, kH, sW2H, S::RG_W, 0, kH, kNO, 1u);
      gemm_kk(tbase + 64, sA, RG_32, 0, sW2L, S::RG_W, 0, kH, kNO, 1u);
      commit(mbar);
    }
    __syncwarp();
    wait_commit();

    {  // F2 epilogue: za = 2 (u + b2) -> B2
      float u[kNO];
      tm_ld16(t_row + 64, u);
      tm_ld16(t_row + 80, u + 16);
      tm_ld16(t_row + 96, u + 32);
      tm_wait_ld();
#pragma unroll
      for (int j = 0; j < kNO; ++j) u[j] = 2.f * (u[j] + bias[2 * kH + j]);
      store_split_row<kNO>(sm + S::O_A, tid, u);
    }
    handoff();
    if (warp == 0 && elect_one()) {
      fence_after_sync();
      gemm_km(tbase + 64, sA, RG_48, 0, sW2H, S::RG_W, 0, 0, kNO, kH, 0u);
      gemm_km(tbase + 64, sA, RG_48, kNO, sW2H, S::RG_W, 0, 0, kNO, kH, 1u);
      gemm_km(tbase + 64, sA, RG_48, 0, sW2L, S::RG_W, 0, 0, kNO, kH, 1u);
      commit(mbar);
    }
    __syncwarp();
    wait_commit();

    // B2 epilogue -> B1, B1 epilogue -> B0: za_{l-1} = (za_l W_l^T) (1 - t_{l-1}^2)
#pragma unroll 1
    for (int l = 1; l >= 0; --l) {
      {
        float t[kH], aa[kH];
        hidden(l, t);
        tm_ld16(t_row + 64, aa);
        tm_ld16(t_row + 80, aa + 16);
        tm_wait_ld();
#pragma unroll
        for (int j = 0; j < kH; ++j) aa[j] *= 1.f - t[j] * t[j];
        store_split_row<kH>(sm + S::O_A, tid, aa);
      }
      handoff();
      if (warp == 0 && elect_one()) {
        fence_after_sync();
        if (l == 1) {
          gemm_km(tbase + 64, sA, RG_32, 0, sW1H, S::RG_W, 0, 0, kH, kH, 0u);
          gemm_km(tbase + 64, sA, RG_32, kH, sW1H, S::RG_W, 0, 0, kH, kH, 1u);
          gemm_km(tbase + 64, sA, RG_32, 0, sW1L, S::RG_W, 0, 0, kH, kH, 1u);
        } else {
          gemm_km(tbase + 64, sA, RG_32, 0, sW0H, S::RG_W0, 0, 0, kH, DK, 0u);
          gemm_km(tbase + 64, sA, RG_32, kH, sW0H, S::RG_W0, 0, 0, kH, DK, 1u);
          gemm_km(tbase + 64, sA, RG_32, 0, sW0L, S::RG_W0, 0, 0, kH, DK, 1u);
        }
        commit(mbar);
      }
      __syncwarp();
      wait_commit();
    }

    // B0 epilogue: grad V_theta (of the state emitted as sample s - 1; at s = 0 it is parked in sample 0's slot, which
    // step 1 overwrites), then p' = p - h grad V, q' = q + h p'
    float g[DK];
#pragma unroll
    for (int c = 0; c < DK / 16; ++c) tm_ld16(t_row + 64 + 16 * c, g + 16 * c);
    tm_wait_ld();
    if constexpr (TRAJ != 0) {
      float* og = (s == 0 ? o : o - sstride) + (OD ? DP : 2 * DP) * plane;
#pragma unroll
      for (int k = 0; k < DP; ++k) __stcs(og + k * plane, g[k]);
    }
    if constexpr (OD) {  // x' = (x + sqrt(2h) xi) - h grad V_theta(x)
      if (s < Sn) {
#pragma unroll
        for (int k = 0; k < DP; ++k) q[k] = fmaf(-h, g[k], q[k]);
        if constexpr (TRAJ != 0) {
#pragma unroll
          for (int k = 0; k < DP; ++k) __stcs(o + k * plane, q[k]);
        }
      }
      if constexpr (TRAJ != 0) o += sstride;
    } else {
#pragma unroll
      for (int k = 0; k < DP; ++k) {
        p[k] = fmaf(-h, g[k], p[k]);
        q[k] = fmaf(h, p[k], q[k]);
      }
      if constexpr (TRAJ != 0) {
        if (s < Sn) {
#pragma unroll
          for (int k = 0; k < DP; ++k) {
            __stcs(o + k * plane, q[k]);
            __stcs(o + (DP + k) * plane, p[k]);
          }
        }
        o += sstride;
      }
    }
  }
  if constexpr (OD) {
    float4* zl = reinterpret_cast<float4*>(a.z_last + n * DP);
#pragma unroll
    for (int i4 = 0; i4 < DP / 4; ++i4) zl[i4] = make_float4(q[4 * i4], q[4 * i4 + 1], q[4 * i4 + 2], q[4 * i4 + 3]);
  } else {
    float4* zl = reinterpret_cast<float4*>(a.z_last + n * (2 * DP));
#pragma unroll
    for (int i4 = 0; i4 < DP / 4; ++i4) {
      zl[i4] = make_float4(q[4 * i4], q[4 * i4 + 1], q[4 * i4 + 2], q[4 * i4 + 3]);
      zl[DP / 4 + i4] = make_float4(p[4 * i4], p[4 * i4 + 1], p[4 * i4 + 2], p[4 * i4 + 3]);
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tbase, S::TMEM_COLS);
}

template <int DP, bool OD>
static int launch(const IntegrateArgs& a, int* status, cudaStream_t st) {
  using S = Cfg<DP>;
  constexpr int MINB = DP >= 16 ? 3 : 4;  // 128 TMEM columns per CTA: at most 4 CTAs per SM (d = 16 spills at 4)
  void (*kern)(const IntegrateArgs, int*);
  if (a.traj == nullptr) kern = kl_integrate_mlp_tc_kernel<DP, 0, MINB, OD>;
  else if (a.traj_layout == PDEIP_TRAJ_BLOCK128) kern = kl_integrate_mlp_tc_kernel<DP, 1, MINB, OD>;
  else kern = kl_integrate_mlp_tc_kernel<DP, 2, MINB, OD>;
  PDEIP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL));
  kern<<<(unsigned)((a.n + 127) / 128), 128, S::TOTAL, st>>>(a, status);
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}

}  // namespace imlp

bool integrate_mlp_tensor_ok(const IntegrateArgs& a) {
  return a.layers == 2 && (a.d == 8 || a.d == 16 || a.d == 32) && !a.noise && !a.tau0 && !a.tau && a.z_last &&
         a.schedule == PDEIP_SCHEDULE_REFERENCE && a.state_layout == PDEIP_LAYOUT_AOS && a.emit_every == 1 &&
         a.emit_offset == 0 &&
         (a.traj == nullptr ||
          (a.emit_drift && (a.traj_layout == PDEIP_TRAJ_BLOCK128 || a.traj_layout == PDEIP_TRAJ_TIME_SOA))) &&
         getenv("PDEIP_NO_TC_INTEGRATOR") == nullptr;
}

int launch_integrate_mlp_tensor(const IntegrateArgs& a, cudaStream_t st) {
  int* status = tensor_status_word();
  PDEIP_REQUIRE(status != nullptr, PDEIP_ERR_CUDA, "cannot allocate the tensor-path status word");
  status += 1;  // word 1: integrator
  if (a.d == 8) return imlp::launch<8, false>(a, status, st);
  if (a.d == 16) return imlp::launch<16, false>(a, status, st);
  return imlp::launch<32, false>(a, status, st);
}

// the overdamped arguments come on the UNIFORM schedule without tau0 (pdeip_overdamped_integrate_model)
bool overdamped_mlp_tensor_ok(const IntegrateArgs& a) {
  return a.layers == 2 && (a.d == 8 || a.d == 16 || a.d == 32) && !a.noise && a.z_last &&
         a.state_layout == PDEIP_LAYOUT_AOS && a.emit_every == 1 && a.emit_offset == 0 &&
         (a.traj == nullptr ||
          (a.emit_drift && (a.traj_layout == PDEIP_TRAJ_BLOCK128 || a.traj_layout == PDEIP_TRAJ_TIME_SOA))) &&
         getenv("PDEIP_NO_TC_INTEGRATOR") == nullptr;
}

int launch_overdamped_mlp_tensor(const IntegrateArgs& a, cudaStream_t st) {
  int* status = tensor_status_word();
  PDEIP_REQUIRE(status != nullptr, PDEIP_ERR_CUDA, "cannot allocate the tensor-path status word");
  status += 1;  // word 1: integrator
  if (a.d == 8) return imlp::launch<8, true>(a, status, st);
  if (a.d == 16) return imlp::launch<16, true>(a, status, st);
  return imlp::launch<32, true>(a, status, st);
}

}  // namespace pdeip
