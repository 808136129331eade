// integrator_tc.cu — K1 with the GMM drift on the tensor cores (PDEIP_PATH_TENSOR of pdeip_kl_integrate_path).
//
// Replaces utils/sampling_utils.py:6-52 with potential_grad = GMMPotential.gradient (core/potential.py:32-61): the
// particle x centre distance contraction (4 K d FLOP per particle-step) is what bounds the CUDA-core kernel (22 % of
// the HBM roofline at C5: d = 32, K = 64; 56 % at C3: d = 8, K = 16).  One CTA = 128 particles = one 128-row tcgen05
// tile, thread = particle = TMEM lane; (q, p) stay in registers for all S + 1 steps.  Per step (d = 16, 32; the d = 8
// kernel further down packs the same operands into full K = 16 steps):
//
//   GEMM 1   L[128 x K]  = [1 | x_hi | x_lo | x_hi] . [b ; mu~_hi ; mu~_hi ; mu~_lo]^T       (tcgen05.mma, bf16 -> fp32)
//            mu~ = mu log2(e) / sigma^2,  b_k = -|mu~_k|^2 / (2 log2(e) / sigma^2)  (three bf16 terms through a ones column)
//            => L_k = log2 of the unnormalised softmax weight up to the row constant -c |x|^2 / 2, which cancels
//   softmax  m = max_k L_k ; e_k = ex2(L_k - m) (MUFU) ; se = sum e_k ; e = e_hi + e_lo (bf16 pair) -> shared memory
//   GEMM 2   A[128 x d]  = [e_hi | e_lo | e_hi] . [mu~_hi ; mu~_hi ; mu~_lo]   (the same centre tiles, MN-major view)
//   update   grad U = (x - A / (c se)) / sigma^2 ; p' = p (1 - gamma h) - h grad U + sqrt(2h) xi ; q' = q + h p'
//
// Operands are split hi + lo (two bf16 terms) so that the contraction carries ~2^-17 relative error instead of 2^-9:
// the result equals the fp32 closed form evaluated at inputs perturbed by < 1e-5 relative (tests: 2e-3 on whole
// trajectories against the fp32 kernel; tolerance class "bf16 GEMM paths" = 1e-2).  The Philox noise of a step does
// not depend on the drift, so it is generated while the step's GEMMs are in flight.  Same Philox stream, tau0, step
// schedule and outputs ([S][N/128][3d][128] or [3d][S][N] trajectory with grad U, final state) as
// kl_integrate_fast_kernel (integrator.cu).  Measured: 70.8 % (d = 32, K = 64) and 69 % (d = 8, K = 16) of the HBM copy
// bandwidth; bound by instruction issue and MUFU together (profiles/r01_summary_tc_integrator.md).
//
// OD = true is the overdamped variant (K1-T-OD, PDEIP_PATH_TENSOR of pdeip_overdamped_integrate with the GMM drift):
// the state per thread is x alone, S steps x' = (x + sqrt(2h) xi_s) - h grad U(x) with h = dt and no tau0.  The
// registers that hold p in the kinetic step hold x + sqrt(2h) xi_s, formed while the GEMMs run, because the epilogue
// still needs x.  An emitted sample is [x, grad U(x)] ([S][N/128][2d][128] or [2d][S][N]); a trajectory run makes one
// more drift-only iteration (s = S: GEMMs and epilogue, no noise, no update) for the last sample's drift, and TRAJ =
// false (OD only) writes the terminal state alone.  Same operand tiles, TMEM map, splits and status word.
#include "common.cuh"
#include "integrator_args.cuh"
#include "philox.cuh"
#include "umma.cuh"

#include <stdlib.h>

#ifndef PDEIP_ITC_MINB
#define PDEIP_ITC_MINB 3  // CTAs (= 128-particle tiles) per SM the register budget is sized for
#endif

namespace pdeip {

int* tensor_status_word();  // residual_tensor.cu: per-device status / debug buffer

namespace itc {
using namespace umma;

template <int DP, int KP>
struct Cfg {
  static_assert(DP == 16 || DP == 32, "d must be 16 or 32");
  static_assert(KP % 16 == 0 && KP >= 16 && KP <= 64, "padded centre count: multiple of 16, <= 64");
  static constexpr uint32_t RG_X = (2 * DP / 8) * 128;  // x tile [128][x_hi(DP) | x_lo(DP)]
  static constexpr uint32_t RG_W = (2 * KP / 8) * 128;  // e tile [128][e_hi(KP) | e_lo(KP)] (aliases the x tile)
  static constexpr uint32_t A_BYTES = 128 * 2 * (KP > DP ? KP : DP) * 2;
  static constexpr uint32_t RG_ONES = 2 * 128;          // [128][16]: columns 0..2 = 1
  static constexpr uint32_t RG_MU = (DP / 8) * 128;     // centre tiles [KP][DP]
  static constexpr uint32_t MU_BYTES = KP * DP * 2;
  static constexpr uint32_t RG_BIAS = 2 * 128;          // [KP][16]: columns 0..2 = b_hi, b_mid, b_lo
  static constexpr uint32_t O_A = 0;
  static constexpr uint32_t O_ONES = O_A + A_BYTES;
  static constexpr uint32_t O_MUH = O_ONES + 128 * 16 * 2;
  static constexpr uint32_t O_MUL = O_MUH + MU_BYTES;
  static constexpr uint32_t O_BIAS = O_MUL + MU_BYTES;
  static constexpr uint32_t O_MISC = O_BIAS + KP * 16 * 2;  // mbarrier (8 B), TMEM base (4 B), dead flag (4 B)
  static constexpr uint32_t TOTAL = O_MISC + 64;
  static constexpr uint32_t TMEM_COLS = (KP + DP) <= 32 ? 32 : ((KP + DP) <= 64 ? 64 : 128);
};

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_bf2(float a, float b) {
  const __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&t);
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

// v = hi + lo, both bf16 (round to nearest twice), for two pairs at once
__device__ __forceinline__ void split2(float2 ab, uint32_t& hi, uint32_t& lo) {
  hi = pack_bf2(ab.x, ab.y);
  const float2 hf = make_float2(__uint_as_float(hi << 16), __uint_as_float(hi & 0xffff0000u));
  const float2 r = __ffma2_rn(hf, make_float2(-1.f, -1.f), ab);
  lo = pack_bf2(r.x, r.y);
}

// BLK = true: trajectory in PDEIP_TRAJ_BLOCK128 ([S][N/128][3d][128]: every store of a step is base + immediate);
// false: PDEIP_TRAJ_TIME_SOA ([3d][S][N]).  OD: the overdamped step (see above); TRAJ = false: no trajectory (OD only).
template <int DP, int KP, bool BLK, int MINB, bool OD = false, bool TRAJ = true>
__global__ void __launch_bounds__(128, MINB) kl_integrate_tc_kernel(const IntegrateArgs a, int* status) {
  static_assert(TRAJ || OD, "a kinetic launch always writes its trajectory");
  using S = Cfg<DP, KP>;
  extern __shared__ __align__(128) uint8_t sm[];
  const int tid = threadIdx.x, warp = tid >> 5;
  uint64_t* mbar_p = reinterpret_cast<uint64_t*>(sm + S::O_MISC);
  uint32_t* tmem_p = reinterpret_cast<uint32_t*>(sm + S::O_MISC + 8);
  volatile int* dead_p = reinterpret_cast<volatile int*>(sm + S::O_MISC + 12);

  // ---- one-time set-up: TMEM, mbarrier, constant operand tiles ------------------------------------------------
  if (warp == 0) {
    tmem_alloc(smem_u32(tmem_p), S::TMEM_COLS);
    tmem_relinquish();
  }
  if (tid == 0) {
    mbar_init(smem_u32(mbar_p), 1);
    fence_mbar_init();
    *dead_p = 0;
  }
  const float cs = a.inv_sigma2 * 1.4426950408889634f;  // logits come out of GEMM 1 in log2 units
  for (int idx = tid; idx < KP * DP; idx += 128) {      // centre tiles: row = centre, column = coordinate
    const int r = idx / DP, c = idx - r * DP;
    const float w = (r < a.n_gaussian) ? cs * a.drift_params[r * DP + c] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(w);
    const __nv_bfloat16 lo = __float2bfloat16_rn(w - __bfloat162float(hi));
    const uint32_t off = chunk_off(r, c >> 3, S::RG_MU) + (uint32_t)(c & 7) * 2u;
    *reinterpret_cast<__nv_bfloat16*>(sm + S::O_MUH + off) = hi;
    *reinterpret_cast<__nv_bfloat16*>(sm + S::O_MUL + off) = lo;
  }
  {  // ones tile: this thread's row
    const uint4 one = make_uint4(0x3F803F80u, 0x00003F80u, 0u, 0u), zero = make_uint4(0u, 0u, 0u, 0u);
    *reinterpret_cast<uint4*>(sm + S::O_ONES + chunk_off(tid, 0, S::RG_ONES)) = one;
    *reinterpret_cast<uint4*>(sm + S::O_ONES + chunk_off(tid, 1, S::RG_ONES)) = zero;
  }
  __syncthreads();
  if (tid < KP) {  // bias row of centre tid: -|mu~|^2 / (2 cs) of the centre as the GEMMs see it (hi + lo)
    float b = -1.0e30f;  // padding centres: weight exactly 0
    if (tid < a.n_gaussian) {
      float s2 = 0.f;
      for (int c = 0; c < DP; ++c) {
        const uint32_t off = chunk_off(tid, c >> 3, S::RG_MU) + (uint32_t)(c & 7) * 2u;
        const float m = __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(sm + S::O_MUH + off)) +
                        __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(sm + S::O_MUL + off));
        s2 = fmaf(m, m, s2);
      }
      b = -0.5f * s2 / cs;
    }
    const __nv_bfloat16 b0 = __float2bfloat16_rn(b);
    const float r1 = b - __bfloat162float(b0);
    const __nv_bfloat16 b1 = __float2bfloat16_rn(r1);
    const __nv_bfloat16 b2 = __float2bfloat16_rn(r1 - __bfloat162float(b1));
    uint4 c0 = make_uint4(0u, 0u, 0u, 0u);
    c0.x = (uint32_t)__bfloat16_as_ushort(b0) | ((uint32_t)__bfloat16_as_ushort(b1) << 16);
    c0.y = (uint32_t)__bfloat16_as_ushort(b2);
    *reinterpret_cast<uint4*>(sm + S::O_BIAS + chunk_off(tid, 0, S::RG_BIAS)) = c0;
    *reinterpret_cast<uint4*>(sm + S::O_BIAS + chunk_off(tid, 1, S::RG_BIAS)) = make_uint4(0u, 0u, 0u, 0u);
  }
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tbase = *tmem_p;
  const uint32_t t_row = tbase + ((uint32_t)(warp * 32) << 16);
  const uint32_t t_logit = t_row, t_acc = t_row + KP;  // this thread's lane, first column of each accumulator
  const uint32_t mbar = smem_u32(mbar_p);
  const uint32_t sA = smem_u32(sm + S::O_A), sOnes = smem_u32(sm + S::O_ONES), sMuH = smem_u32(sm + S::O_MUH),
                 sMuL = smem_u32(sm + S::O_MUL), sBias = smem_u32(sm + S::O_BIAS);
  uint8_t* const rowA = sm + S::O_A + (uint32_t)(tid & 7) * 16u;  // + (tid >> 3) * row-group bytes + chunk * 128
  uint32_t phase = 0;

  // ---- state.  Rows past the end of a ragged last tile repeat the last particle (same id, same values written to
  // the same addresses), so that no load or store in the step loop needs a predicate. ----------------------------
  const int64_t n_raw = (int64_t)blockIdx.x * 128 + tid;
  const int64_t n = n_raw < a.n ? n_raw : a.n - 1;
  const uint64_t pid = a.particle_offset + (uint64_t)n;
  float2 q[DP / 2], p[DP / 2];  // OD: q = x, p = x + sqrt(2h) xi of the current step
  if constexpr (OD) {
    const float4* z4 = reinterpret_cast<const float4*>(a.z0 + n * DP);
#pragma unroll
    for (int i4 = 0; i4 < DP / 4; ++i4) {
      const float4 tq = z4[i4];
      q[2 * i4] = make_float2(tq.x, tq.y); q[2 * i4 + 1] = make_float2(tq.z, tq.w);
    }
  } else {
    const float4* z4 = reinterpret_cast<const float4*>(a.z0 + n * (2 * DP));
#pragma unroll
    for (int i4 = 0; i4 < DP / 4; ++i4) {
      const float4 tq = z4[i4], tp = z4[DP / 4 + i4];
      q[2 * i4] = make_float2(tq.x, tq.y); q[2 * i4 + 1] = make_float2(tq.z, tq.w);
      p[2 * i4] = make_float2(tp.x, tp.y); p[2 * i4 + 1] = make_float2(tp.z, tp.w);
    }
  }
  const float t0 = OD ? 0.f : philox_uniform01(a.seed, pid, kTagTau0) * a.dt;  // sampling_utils.py:32
  const int Sn = a.n_steps;
  constexpr int CW = OD ? 2 * DP : 3 * DP;  // floats per emitted sample: [x, v, grad U] or (OD) [x, grad U]
  // BLK: element (sample s, tile t, component c, lane l) at ((s T + t) CW + c) 128 + l ; else c S N + s N + n
  const int64_t plane = BLK ? 128 : (int64_t)Sn * a.n;               // floats between components of a sample
  const int64_t sstride = BLK ? (int64_t)gridDim.x * (CW * 128) : a.n;  // floats between samples
  float* o = !TRAJ ? nullptr : (BLK ? a.traj + ((int64_t)blockIdx.x * CW * 128 + tid) : a.traj + n);  // sample 0, component 0
  const float rcs = 1.0f / cs;
  // OD: S steps, and with a trajectory one more drift-only iteration (s = S) for the last sample's drift
  const int s_end = OD ? Sn + (TRAJ ? 1 : 0) : Sn + 1;

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
  // p <- p (1 - gamma h) + sqrt(2h) xi for coordinate blocks [j0, j1) (4 coordinates each): the drift-independent part
  // (OD: p <- x + sqrt(2h) xi; the drift-only iteration s = S draws nothing)
  auto kick = [&](int s, float dmp, float sq, int j0, int j1) {
    if (OD && s == Sn) return;
    const float2 dmp2 = make_float2(dmp, dmp), sq2 = make_float2(sq, sq);
#pragma unroll
    for (int j = j0; j < j1; ++j) {
      float r4[4];
      philox_normal4_rk(a.rk, pid, a.step_offset + (uint32_t)s, (uint32_t)j, r4);
      if constexpr (OD) {
        p[2 * j] = __ffma2_rn(sq2, make_float2(r4[0], r4[1]), q[2 * j]);
        p[2 * j + 1] = __ffma2_rn(sq2, make_float2(r4[2], r4[3]), q[2 * j + 1]);
      } else {
        p[2 * j] = __ffma2_rn(sq2, make_float2(r4[0], r4[1]), __fmul2_rn(p[2 * j], dmp2));
        p[2 * j + 1] = __ffma2_rn(sq2, make_float2(r4[2], r4[3]), __fmul2_rn(p[2 * j + 1], dmp2));
      }
    }
  };

#pragma unroll 1
  for (int s = 0; OD ? s < s_end : s <= Sn; ++s) {
    const float h = OD ? a.dt : ((s == 0) ? t0 : ((s == Sn) ? a.dt - t0 : a.dt));  // sampling_utils.py:33,45-46
    const float sq = sqrtf(h) * 1.41421356237309515f;
    const float dmp = 1.f - a.gamma * h;

    // (1) x -> [x_hi | x_lo] rows of the A tile
    {
      uint8_t* const row = rowA + (uint32_t)(tid >> 3) * S::RG_X;
#pragma unroll
      for (int cg = 0; cg < DP / 8; ++cg) {
        uint4 hi, lo;
        split2(q[4 * cg], hi.x, lo.x);
        split2(q[4 * cg + 1], hi.y, lo.y);
        split2(q[4 * cg + 2], hi.z, lo.z);
        split2(q[4 * cg + 3], hi.w, lo.w);
        *reinterpret_cast<uint4*>(row + cg * 128) = hi;
        *reinterpret_cast<uint4*>(row + (DP / 8 + cg) * 128) = lo;
      }
    }
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    if (warp == ((2 * s) & 3) && elect_one()) {  // the issuing duty rotates over the four warps
      fence_after_sync();
      mma_bf16(tbase, make_desc(sOnes, 128u, S::RG_ONES), make_desc(sBias, 128u, S::RG_BIAS), make_idesc(KP, 0, 0), 0u);
      gemm_kk(tbase, sA, S::RG_X, 0, sMuH, S::RG_MU, 0, DP, KP, 1u);   // x_hi . mu_hi
      gemm_kk(tbase, sA, S::RG_X, DP, sMuH, S::RG_MU, 0, DP, KP, 1u);  // x_lo . mu_hi
      gemm_kk(tbase, sA, S::RG_X, 0, sMuL, S::RG_MU, 0, DP, KP, 1u);   // x_hi . mu_lo
      commit(mbar);
    }
    __syncwarp();
    kick(s, dmp, sq, 0, DP / 8);  // first half of the noise while GEMM 1 runs
    wait_commit();

    // (2) softmax over the centres: two passes over the TMEM row (max, then exponentials)
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < KP / 16; ++c) {
      float l[16];
      tm_ld16(t_logit + 16 * c, l);
      tm_wait_ld();
#pragma unroll
      for (int i = 0; i < 16; ++i) m = fmaxf(m, l[i]);
    }
    float2 se2 = make_float2(0.f, 0.f);
    {
      const float2 nm2 = make_float2(-m, -m);
      uint8_t* const row = rowA + (uint32_t)(tid >> 3) * S::RG_W;
#pragma unroll
      for (int c = 0; c < KP / 16; ++c) {
        float l[16];
        tm_ld16(t_logit + 16 * c, l);
        tm_wait_ld();
        float2 e[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float2 t = __fadd2_rn(make_float2(l[2 * i], l[2 * i + 1]), nm2);
          e[i] = make_float2(ex2f(t.x), ex2f(t.y));
          se2 = __fadd2_rn(se2, e[i]);
        }
#pragma unroll
        for (int hcg = 0; hcg < 2; ++hcg) {
          uint4 hi, lo;
          split2(e[4 * hcg], hi.x, lo.x);
          split2(e[4 * hcg + 1], hi.y, lo.y);
          split2(e[4 * hcg + 2], hi.z, lo.z);
          split2(e[4 * hcg + 3], hi.w, lo.w);
          *reinterpret_cast<uint4*>(row + (2 * c + hcg) * 128) = hi;
          *reinterpret_cast<uint4*>(row + (KP / 8 + 2 * c + hcg) * 128) = lo;
        }
      }
    }
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    if (warp == ((2 * s + 1) & 3) && elect_one()) {
      fence_after_sync();
      gemm_km(tbase + KP, sA, S::RG_W, 0, sMuH, S::RG_MU, 0, 0, KP, DP, 0u);   // e_hi . mu_hi
      gemm_km(tbase + KP, sA, S::RG_W, KP, sMuH, S::RG_MU, 0, 0, KP, DP, 1u);  // e_lo . mu_hi
      gemm_km(tbase + KP, sA, S::RG_W, 0, sMuL, S::RG_MU, 0, 0, KP, DP, 1u);   // e_hi . mu_lo
      commit(mbar);
    }
    __syncwarp();
    kick(s, dmp, sq, DP / 8, DP / 4);  // second half of the noise while GEMM 2 runs
    wait_commit();

    // (3) grad U = (x - A / (cs se)) / sigma^2 ; finish the step.  grad U belongs to the state emitted as sample
    // s - 1; at s = 0 it is parked in sample 0's slot, which step 1 overwrites.
    const float rn = -rcs / (se2.x + se2.y);
    const float2 rn2 = make_float2(rn, rn), is2 = make_float2(a.inv_sigma2, a.inv_sigma2);
    const float2 nh2 = make_float2(-h, -h), h2 = make_float2(h, h);
    float* og = (s == 0 ? o : o - sstride) + (OD ? DP : 2 * DP) * plane;
#pragma unroll
    for (int c = 0; c < DP / 16; ++c) {
      float acc[16];
      tm_ld16(t_acc + 16 * c, acc);
      tm_wait_ld();
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int k = 8 * c + i;
        const float2 g = __fmul2_rn(__ffma2_rn(make_float2(acc[2 * i], acc[2 * i + 1]), rn2, q[k]), is2);
        if constexpr (TRAJ) {
          if constexpr (BLK) {
            __stcs(og + (2 * k) * 128, g.x);
            __stcs(og + (2 * k + 1) * 128, g.y);
          } else {
            __stcs(og, g.x);
            __stcs(og + plane, g.y);
            og += 2 * plane;
          }
        }
        if constexpr (OD) {  // x' = (x + sqrt(2h) xi) - h grad U(x)
          if (s < Sn) q[k] = __ffma2_rn(nh2, g, p[k]);
        } else {
          p[k] = __ffma2_rn(nh2, g, p[k]);
          q[k] = __ffma2_rn(h2, p[k], q[k]);
        }
      }
    }
    if (TRAJ && s < Sn) {  // the state as sample s: [x, v] (OD: x; its drift follows in the next iteration)
      if constexpr (BLK) {
#pragma unroll
        for (int i = 0; i < DP / 2; ++i) {
          __stcs(o + (2 * i) * 128, q[i].x);
          __stcs(o + (2 * i + 1) * 128, q[i].y);
          if constexpr (!OD) {
            __stcs(o + (DP + 2 * i) * 128, p[i].x);
            __stcs(o + (DP + 2 * i + 1) * 128, p[i].y);
          }
        }
      } else {
        float* w = o;
#pragma unroll
        for (int i = 0; i < DP / 2; ++i) {
          __stcs(w, q[i].x);
          __stcs(w + plane, q[i].y);
          w += 2 * plane;
        }
        if constexpr (!OD) {
#pragma unroll
          for (int i = 0; i < DP / 2; ++i) {
            __stcs(w, p[i].x);
            __stcs(w + plane, p[i].y);
            w += 2 * plane;
          }
        }
      }
    }
    if constexpr (TRAJ) o += sstride;
  }
  if constexpr (OD) {
    float4* zl = reinterpret_cast<float4*>(a.z_last + n * DP);
#pragma unroll
    for (int i4 = 0; i4 < DP / 4; ++i4) zl[i4] = make_float4(q[2 * i4].x, q[2 * i4].y, q[2 * i4 + 1].x, q[2 * i4 + 1].y);
  } else {
    float4* zl = reinterpret_cast<float4*>(a.z_last + n * (2 * DP));
#pragma unroll
    for (int i4 = 0; i4 < DP / 4; ++i4) {
      zl[i4] = make_float4(q[2 * i4].x, q[2 * i4].y, q[2 * i4 + 1].x, q[2 * i4 + 1].y);
      zl[DP / 4 + i4] = make_float4(p[2 * i4].x, p[2 * i4].y, p[2 * i4 + 1].x, p[2 * i4 + 1].y);
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tbase, S::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------------------
// d = 8 (C3: K = 16).  Same step, operands packed so that every MMA has a full K = 16:
//   A tile [128][32]  = [x_hi | x_lo | x_hi | 1 1 1 0 0 0 0 0]          B tile [K][32] = [mu~_hi | mu~_hi | mu~_lo | b0 b1 b2 0..]
//   GEMM 1  L[128 x K]  = A . B^T                                       (two MMAs)
//   GEMM 2  Acc[128 x 16] = e_hi . B[:, 0:16] + e_lo . B[:, 0:16] + e_hi . B[:, 16:32]   (MN-major views of the B tile;
//           columns 0..7 of Acc are sum_k e_k mu~_k, columns 8..15 are never read)
// ------------------------------------------------------------------------------------------------------------
template <int KP>
struct Cfg8 {
  static_assert(KP % 16 == 0 && KP >= 16 && KP <= 64, "padded centre count: multiple of 16, <= 64");
  static constexpr uint32_t RG_X = 4 * 128, RG_B = 4 * 128, RG_W = (2 * KP / 8) * 128;
  static constexpr uint32_t O_X = 0, O_W = O_X + 16 * RG_X, O_B = O_W + 16 * RG_W, O_MISC = O_B + (KP / 8) * RG_B;
  static constexpr uint32_t TOTAL = O_MISC + 64;
  static constexpr uint32_t TMEM_COLS = (KP + 16) <= 32 ? 32 : ((KP + 16) <= 64 ? 64 : 128);
};

#ifndef PDEIP_ITC8_MINB
#define PDEIP_ITC8_MINB 8
#endif
template <int KP, bool BLK, int MINB, bool OD = false, bool TRAJ = true>
__global__ void __launch_bounds__(128, MINB) kl_integrate_tc8_kernel(const IntegrateArgs a, int* status) {
  static_assert(TRAJ || OD, "a kinetic launch always writes its trajectory");
  using S = Cfg8<KP>;
  constexpr int DP = 8;
  extern __shared__ __align__(128) uint8_t sm[];
  const int tid = threadIdx.x, warp = tid >> 5;
  uint64_t* mbar_p = reinterpret_cast<uint64_t*>(sm + S::O_MISC);
  uint32_t* tmem_p = reinterpret_cast<uint32_t*>(sm + S::O_MISC + 8);
  volatile int* dead_p = reinterpret_cast<volatile int*>(sm + S::O_MISC + 12);

  if (warp == 0) {
    tmem_alloc(smem_u32(tmem_p), S::TMEM_COLS);
    tmem_relinquish();
  }
  if (tid == 0) {
    mbar_init(smem_u32(mbar_p), 1);
    fence_mbar_init();
    *dead_p = 0;
  }
  const float cs = a.inv_sigma2 * 1.4426950408889634f;
  if (tid < KP) {  // B tile row of centre tid
    float hi_f[8], lo_f[8], s2 = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float w = (tid < a.n_gaussian) ? cs * a.drift_params[tid * DP + c] : 0.f;
      hi_f[c] = __bfloat162float(__float2bfloat16_rn(w));
      lo_f[c] = __bfloat162float(__float2bfloat16_rn(w - hi_f[c]));
      const float m = hi_f[c] + lo_f[c];
      s2 = fmaf(m, m, s2);
    }
    const float b = (tid < a.n_gaussian) ? -0.5f * s2 / cs : -1.0e30f;  // padding centres: weight exactly 0
    const float b0 = __bfloat162float(__float2bfloat16_rn(b));
    const float b1 = __bfloat162float(__float2bfloat16_rn(b - b0));
    const float b2 = __bfloat162float(__float2bfloat16_rn(b - b0 - b1));
    const float bias[8] = {b0, b1, b2, 0.f, 0.f, 0.f, 0.f, 0.f};
    store_chunk(sm + S::O_B, chunk_off(tid, 0, S::RG_B), hi_f);
    store_chunk(sm + S::O_B, chunk_off(tid, 1, S::RG_B), hi_f);
    store_chunk(sm + S::O_B, chunk_off(tid, 2, S::RG_B), lo_f);
    store_chunk(sm + S::O_B, chunk_off(tid, 3, S::RG_B), bias);
  }
  *reinterpret_cast<uint4*>(sm + S::O_X + chunk_off(tid, 3, S::RG_X)) = make_uint4(0x3F803F80u, 0x00003F80u, 0u, 0u);
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tbase = *tmem_p;
  const uint32_t t_row = tbase + ((uint32_t)(warp * 32) << 16);
  const uint32_t t_logit = t_row, t_acc = t_row + KP;
  const uint32_t mbar = smem_u32(mbar_p);
  const uint32_t sX = smem_u32(sm + S::O_X), sW = smem_u32(sm + S::O_W), sB = smem_u32(sm + S::O_B);
  uint8_t* const rowX = sm + S::O_X + (uint32_t)(tid & 7) * 16u + (uint32_t)(tid >> 3) * S::RG_X;
  uint8_t* const rowW = sm + S::O_W + (uint32_t)(tid & 7) * 16u + (uint32_t)(tid >> 3) * S::RG_W;
  uint32_t phase = 0;

  const int64_t n_raw = (int64_t)blockIdx.x * 128 + tid;
  const int64_t n = n_raw < a.n ? n_raw : a.n - 1;  // ragged last tile: repeat the last particle (see above)
  const uint64_t pid = a.particle_offset + (uint64_t)n;
  float2 q[4], p[4];  // OD: q = x, p = x + sqrt(2h) xi of the current step
  if constexpr (OD) {
    const float4* z4 = reinterpret_cast<const float4*>(a.z0 + n * 8);
    const float4 q0 = z4[0], q1 = z4[1];
    q[0] = make_float2(q0.x, q0.y); q[1] = make_float2(q0.z, q0.w); q[2] = make_float2(q1.x, q1.y); q[3] = make_float2(q1.z, q1.w);
  } else {
    const float4* z4 = reinterpret_cast<const float4*>(a.z0 + n * 16);
    const float4 q0 = z4[0], q1 = z4[1], p0 = z4[2], p1 = z4[3];
    q[0] = make_float2(q0.x, q0.y); q[1] = make_float2(q0.z, q0.w); q[2] = make_float2(q1.x, q1.y); q[3] = make_float2(q1.z, q1.w);
    p[0] = make_float2(p0.x, p0.y); p[1] = make_float2(p0.z, p0.w); p[2] = make_float2(p1.x, p1.y); p[3] = make_float2(p1.z, p1.w);
  }
  const float t0 = OD ? 0.f : philox_uniform01(a.seed, pid, kTagTau0) * a.dt;  // sampling_utils.py:32
  const int Sn = a.n_steps;
  constexpr int CW = OD ? 2 * DP : 3 * DP;  // floats per emitted sample
  const int64_t plane = BLK ? 128 : (int64_t)Sn * a.n;
  const int64_t sstride = BLK ? (int64_t)gridDim.x * (CW * 128) : a.n;
  float* o = !TRAJ ? nullptr : (BLK ? a.traj + ((int64_t)blockIdx.x * CW * 128 + tid) : a.traj + n);
  const float rcs = 1.0f / cs;
  const int s_end = OD ? Sn + (TRAJ ? 1 : 0) : Sn + 1;  // OD: + the drift-only iteration of a trajectory run

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
  auto kick = [&](int s, float dmp, float sq, int j) {  // p <- p (1 - gamma h) + sqrt(2h) xi, coordinates 4j .. 4j+3
    if (OD && s == Sn) return;                          // (OD: p <- x + sqrt(2h) xi; none at s = S)
    const float2 dmp2 = make_float2(dmp, dmp), sq2 = make_float2(sq, sq);
    float r4[4];
    philox_normal4_rk(a.rk, pid, a.step_offset + (uint32_t)s, (uint32_t)j, r4);
    if constexpr (OD) {
      p[2 * j] = __ffma2_rn(sq2, make_float2(r4[0], r4[1]), q[2 * j]);
      p[2 * j + 1] = __ffma2_rn(sq2, make_float2(r4[2], r4[3]), q[2 * j + 1]);
    } else {
      p[2 * j] = __ffma2_rn(sq2, make_float2(r4[0], r4[1]), __fmul2_rn(p[2 * j], dmp2));
      p[2 * j + 1] = __ffma2_rn(sq2, make_float2(r4[2], r4[3]), __fmul2_rn(p[2 * j + 1], dmp2));
    }
  };

#pragma unroll 1
  for (int s = 0; OD ? s < s_end : s <= Sn; ++s) {
    const float h = OD ? a.dt : ((s == 0) ? t0 : ((s == Sn) ? a.dt - t0 : a.dt));  // sampling_utils.py:33,45-46
    const float sq = sqrtf(h) * 1.41421356237309515f;
    const float dmp = 1.f - a.gamma * h;
    {
      uint4 hi, lo;
      split2(q[0], hi.x, lo.x);
      split2(q[1], hi.y, lo.y);
      split2(q[2], hi.z, lo.z);
      split2(q[3], hi.w, lo.w);
      *reinterpret_cast<uint4*>(rowX) = hi;
      *reinterpret_cast<uint4*>(rowX + 128) = lo;
      *reinterpret_cast<uint4*>(rowX + 256) = hi;
    }
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    if (warp == ((2 * s) & 3) && elect_one()) {
      fence_after_sync();
      gemm_kk(tbase, sX, S::RG_X, 0, sB, S::RG_B, 0, 32, KP, 0u);
      commit(mbar);
    }
    __syncwarp();
    kick(s, dmp, sq, 0);
    wait_commit();

    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < KP / 16; ++c) {
      float l[16];
      tm_ld16(t_logit + 16 * c, l);
      tm_wait_ld();
#pragma unroll
      for (int i = 0; i < 16; ++i) m = fmaxf(m, l[i]);
    }
    float2 se2 = make_float2(0.f, 0.f);
    {
      const float2 nm2 = make_float2(-m, -m);
#pragma unroll
      for (int c = 0; c < KP / 16; ++c) {
        float l[16];
        tm_ld16(t_logit + 16 * c, l);
        tm_wait_ld();
        float2 e[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float2 t = __fadd2_rn(make_float2(l[2 * i], l[2 * i + 1]), nm2);
          e[i] = make_float2(ex2f(t.x), ex2f(t.y));
          se2 = __fadd2_rn(se2, e[i]);
        }
#pragma unroll
        for (int hcg = 0; hcg < 2; ++hcg) {
          uint4 hi, lo;
          split2(e[4 * hcg], hi.x, lo.x);
          split2(e[4 * hcg + 1], hi.y, lo.y);
          split2(e[4 * hcg + 2], hi.z, lo.z);
          split2(e[4 * hcg + 3], hi.w, lo.w);
          *reinterpret_cast<uint4*>(rowW + (2 * c + hcg) * 128) = hi;
          *reinterpret_cast<uint4*>(rowW + (KP / 8 + 2 * c + hcg) * 128) = lo;
        }
      }
    }
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    if (warp == ((2 * s + 1) & 3) && elect_one()) {
      fence_after_sync();
      gemm_km(tbase + KP, sW, S::RG_W, 0, sB, S::RG_B, 0, 0, KP, 16, 0u);    // e_hi . [mu_hi | mu_hi]
      gemm_km(tbase + KP, sW, S::RG_W, KP, sB, S::RG_B, 0, 0, KP, 16, 1u);   // e_lo . [mu_hi | mu_hi]
      gemm_km(tbase + KP, sW, S::RG_W, 0, sB, S::RG_B, 16, 0, KP, 16, 1u);   // e_hi . [mu_lo | bias]
      commit(mbar);
    }
    __syncwarp();
    kick(s, dmp, sq, 1);
    wait_commit();

    const float rn = -rcs / (se2.x + se2.y);
    const float2 rn2 = make_float2(rn, rn), is2 = make_float2(a.inv_sigma2, a.inv_sigma2);
    const float2 nh2 = make_float2(-h, -h), h2 = make_float2(h, h);
    float* og = (s == 0 ? o : o - sstride) + (OD ? DP : 2 * DP) * plane;
    float acc[8];
    tmem_ld8(t_acc, acc);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 g = __fmul2_rn(__ffma2_rn(make_float2(acc[2 * k], acc[2 * k + 1]), rn2, q[k]), is2);
      if constexpr (TRAJ) {
        __stcs(og + (2 * k) * plane, g.x);
        __stcs(og + (2 * k + 1) * plane, g.y);
      }
      if constexpr (OD) {  // x' = (x + sqrt(2h) xi) - h grad U(x)
        if (s < Sn) q[k] = __ffma2_rn(nh2, g, p[k]);
      } else {
        p[k] = __ffma2_rn(nh2, g, p[k]);
        q[k] = __ffma2_rn(h2, p[k], q[k]);
      }
    }
    if (TRAJ && s < Sn) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        __stcs(o + (2 * i) * plane, q[i].x);
        __stcs(o + (2 * i + 1) * plane, q[i].y);
        if constexpr (!OD) {
          __stcs(o + (DP + 2 * i) * plane, p[i].x);
          __stcs(o + (DP + 2 * i + 1) * plane, p[i].y);
        }
      }
    }
    if constexpr (TRAJ) o += sstride;
  }
  if constexpr (OD) {
    float4* zl = reinterpret_cast<float4*>(a.z_last + n * 8);
    zl[0] = make_float4(q[0].x, q[0].y, q[1].x, q[1].y);
    zl[1] = make_float4(q[2].x, q[2].y, q[3].x, q[3].y);
  } else {
    float4* zl = reinterpret_cast<float4*>(a.z_last + n * 16);
    zl[0] = make_float4(q[0].x, q[0].y, q[1].x, q[1].y);
    zl[1] = make_float4(q[2].x, q[2].y, q[3].x, q[3].y);
    zl[2] = make_float4(p[0].x, p[0].y, p[1].x, p[1].y);
    zl[3] = make_float4(p[2].x, p[2].y, p[3].x, p[3].y);
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tbase, S::TMEM_COLS);
}

// CTAs per SM the overdamped instances are sized for (fixed; the PDEIP_ITC*_MINB knobs tune the kinetic instances):
// the kinetic defaults where ptxas fits them without a stack frame.  At d = 8 a budget of 8 CTAs (64 registers) needs
// one, so the trajectory instances take 6.  The terminal-only ones need one at 6 (K >= 48) and at 5 (K = 64): they take
// 5, and 4 at K = 64, where a CTA's 128 TMEM columns allow no more than 4 CTAs per SM anyway.
constexpr int kOdMinb16 = 3, kOdMinb32 = 3, kOdMinb8Traj = 6;
template <int KP>
constexpr int kOdMinb8Terminal = KP == 64 ? 4 : 5;

template <int KP, bool OD>
static int launch8(const IntegrateArgs& a, int* status, cudaStream_t st) {
  using S = Cfg8<KP>;
  const int64_t grid = (a.n + 127) / 128;
  void (*kern)(const IntegrateArgs, int*);
  if constexpr (OD) {
    constexpr int MB = kOdMinb8Traj;
    if (a.traj == nullptr) kern = kl_integrate_tc8_kernel<KP, false, kOdMinb8Terminal<KP>, true, false>;
    else if (a.traj_layout == PDEIP_TRAJ_BLOCK128) kern = kl_integrate_tc8_kernel<KP, true, MB, true>;
    else kern = kl_integrate_tc8_kernel<KP, false, MB, true>;
  } else {
    const char* mb = getenv("PDEIP_ITC8_MINB");  // tuning knob: CTAs per SM the register budget is sized for
    const bool eight = mb ? (mb[0] == '8') : (PDEIP_ITC8_MINB == 8);
    if (a.traj_layout == PDEIP_TRAJ_BLOCK128)
      kern = eight ? kl_integrate_tc8_kernel<KP, true, 8> : kl_integrate_tc8_kernel<KP, true, 6>;
    else
      kern = eight ? kl_integrate_tc8_kernel<KP, false, 8> : kl_integrate_tc8_kernel<KP, false, 6>;
  }
  PDEIP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL));
  kern<<<(unsigned)grid, 128, S::TOTAL, st>>>(a, status);
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}

template <int DP, int KP, bool OD>
static int launch(const IntegrateArgs& a, int* status, cudaStream_t st) {
  using S = Cfg<DP, KP>;
  const int64_t grid = (a.n + 127) / 128;
  void (*kern)(const IntegrateArgs, int*);
  if constexpr (OD) {
    constexpr int MB = DP == 32 ? kOdMinb32 : kOdMinb16;
    if (a.traj == nullptr) kern = kl_integrate_tc_kernel<DP, KP, false, MB, true, false>;
    else if (a.traj_layout == PDEIP_TRAJ_BLOCK128) kern = kl_integrate_tc_kernel<DP, KP, true, MB, true>;
    else kern = kl_integrate_tc_kernel<DP, KP, false, MB, true>;
  } else {
    const char* mb = getenv("PDEIP_ITC_MINB");  // tuning knob: CTAs per SM the register budget is sized for
    const bool four = mb ? (mb[0] == '4') : (PDEIP_ITC_MINB == 4);
    if (a.traj_layout == PDEIP_TRAJ_BLOCK128)
      kern = four ? kl_integrate_tc_kernel<DP, KP, true, 4> : kl_integrate_tc_kernel<DP, KP, true, 3>;
    else
      kern = four ? kl_integrate_tc_kernel<DP, KP, false, 4> : kl_integrate_tc_kernel<DP, KP, false, 3>;
  }
  PDEIP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL));
  kern<<<(unsigned)grid, 128, S::TOTAL, st>>>(a, status);
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}

}  // namespace itc

// true if the call is served by the tensor-core kernel: the production configuration of kl_integrate_fast_kernel
// (checked by the caller) with the GMM drift, d = 8, 16 or 32 and at most 64 centres
bool integrate_tensor_ok(const IntegrateArgs& a, int drift_kind) {
  return drift_kind == PDEIP_DRIFT_GMM && (a.d == 8 || a.d == 16 || a.d == 32) && a.n_gaussian >= 1 && a.n_gaussian <= 64 &&
         getenv("PDEIP_NO_TC_INTEGRATOR") == nullptr;
}

namespace itc {
template <bool OD>
static int launch_d_k(const IntegrateArgs& a, cudaStream_t st) {
  int* status = tensor_status_word();
  PDEIP_REQUIRE(status != nullptr, PDEIP_ERR_CUDA, "cannot allocate the tensor-path status word");
  status += 1;  // word 1: integrator (word 0: residual kernel)
  const int kp = (a.n_gaussian + 15) / 16 * 16;
  if (a.d == 8) {
    if (kp == 16) return launch8<16, OD>(a, status, st);
    if (kp == 32) return launch8<32, OD>(a, status, st);
    if (kp == 48) return launch8<48, OD>(a, status, st);
    return launch8<64, OD>(a, status, st);
  }
  if (a.d == 32) {
    if (kp == 16) return launch<32, 16, OD>(a, status, st);
    if (kp == 32) return launch<32, 32, OD>(a, status, st);
    if (kp == 48) return launch<32, 48, OD>(a, status, st);
    return launch<32, 64, OD>(a, status, st);
  }
  if (kp == 16) return launch<16, 16, OD>(a, status, st);
  if (kp == 32) return launch<16, 32, OD>(a, status, st);
  if (kp == 48) return launch<16, 48, OD>(a, status, st);
  return launch<16, 64, OD>(a, status, st);
}
}  // namespace itc

int launch_integrate_tensor(const IntegrateArgs& a, cudaStream_t st) { return itc::launch_d_k<false>(a, st); }

// true if an overdamped GMM call is served by K1-T-OD: d = 8, 16 or 32, 1..64 centres, Philox noise, AoS state with a
// terminal-state output, every sample emitted, and either no trajectory or a BLOCK128 / TIME_SOA trajectory with the
// drift (the arguments come on the UNIFORM schedule without tau0, pdeip_overdamped_integrate)
bool overdamped_tensor_ok(const IntegrateArgs& a, int drift_kind) {
  return drift_kind == PDEIP_DRIFT_GMM && (a.d == 8 || a.d == 16 || a.d == 32) && a.n_gaussian >= 1 &&
         a.n_gaussian <= 64 && !a.noise && a.z_last && a.state_layout == PDEIP_LAYOUT_AOS && a.emit_every == 1 &&
         a.emit_offset == 0 &&
         (a.traj == nullptr ||
          (a.emit_drift && (a.traj_layout == PDEIP_TRAJ_BLOCK128 || a.traj_layout == PDEIP_TRAJ_TIME_SOA))) &&
         getenv("PDEIP_NO_TC_INTEGRATOR") == nullptr;
}

int launch_overdamped_tensor(const IntegrateArgs& a, cudaStream_t st) { return itc::launch_d_k<true>(a, st); }

}  // namespace pdeip
