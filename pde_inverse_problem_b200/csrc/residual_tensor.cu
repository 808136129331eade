// residual_tensor.cu — K3/K4 on the 5th-generation tensor cores (tcgen05 + TMEM), KFP 0T point set, version 2.
//
// Mathematics: SURVEY.md §9 (reference: methods/consistency_instances/kinetic_fokker_planck.py:11-69), restated
// phase by phase in tests/tensor_v2_model.py (float64 twin, checked against oracle/taylor.py to 1e-16).
// Per point (x, v):  l = |g|^2 - 2 D_v^2 V + 2 gamma D_v V,  g = grad_x V,  V = |MLP(x)|^2,  and dl/dtheta.
//
// Organisation.  One CTA per SM, persistent over 128-point tiles; NS tiles ("slots") are in flight per CTA so
// that one slot's epilogue hides the other's GEMM hand-off latency (NS = 2 for d <= 8, 1 otherwise).
//   * epilogue warps: thread = (point row == TMEM lane, one part of the units; Team): 16 warps in the one-slot kernels
//     (8 of the 32 hidden units, 8 + 2 of the 40 outputs), 8 in the two-slot kernel (16 / 24); 1 MMA warp: one elected
//     lane issues every tcgen05.mma of both slots.
//   * operands: bf16 in shared memory, no-swizzle core-matrix layout (umma.cuh); every tile is written once and
//     used K-major (layer GEMMs, points x units) and through the transposed view (batch-reduced dW GEMMs).
//     Weights and the input x are split hi + lo (two bf16 terms), activations are rounded to bf16 once.
//   * accumulators: fp32 in TMEM.  Values an epilogue needs again later are "parked" in TMEM as packed bf16 pairs
//     (s1 = 1 - t^2 of both hidden layers, the partial seed s0p, the pz terms).
//   * streams.  Forward Taylor streams along v: a (primal), a1, a2^ = -a2 / 2.  Input gradient chain za^ = 4 za,
//     aa^ = 4 aa.  Stop-gradient stream along g^ = g / 2 (order 1).  The adjoints of the a2 and g streams are
//     proportional to the input-gradient chain (zbar2 = -2 za, zbar_g = 2 za), so only TWO adjoint streams need
//     GEMMs: the primal (zbar0) and the order-1 stream (zbar1); the latter rides along with the input-gradient chain
//     (P3..P5).  With c = a2^ + ag^:  a2^T zbar2 + ag^T zbar_g = c^T za^.
//   * dW_l = t^T zbar0 + a1^T zbar1 + c^T za^ accumulates over ALL tiles of the CTA in persistent TMEM
//     columns: each term is an M = 128 GEMM over the 128 points whose A operand is the transposed view of the
//     activation tile started at the band of that stream ("band-shifted accumulate"): rows 0..31 of D are the
//     wanted 32 x N block, rows >= 32 are never read.  db_l = sum_p zbar0 is kept per row (registers, or TMEM: C_DB).
//   phases  P0 z0,z1_0 | P1 z1,z1_1,z2^_1 | P2 u,u1,u2^ | P3 aa2, ab1_2 (+dW2: a1) | P4 aa1, ab1_1 (+dW1: a1) |
//           P5 g (+dW0: v) | P6 zg^_0 | P7 zg^_1 | P8 ug^ | P9 ab_2, aa2 (+dW2: t, c) | P10 ab_1, aa1 (+dW1: t, c) |
//           P11 (dW0: x_hi, x_lo, g^).   E_k = epilogue between P_{k-1} and P_k.
//   parity  rtol 1e-2 (BASELINE.json, bf16 GEMM path); measured against the oracle in tests/test_gpu_tensor.py.
//
// FP 0T set (methods/consistency_instances/fokker_planck.py:33-63: |g|^2 - 2 sum_i D_{e_i}^2 V, the d forward-mode
// tangents of jacfwd(grad V)) on the same kernel: the d tangent streams e_1..e_d of a point are STACKED ALONG M, one
// tile row (x, v = e_i) per direction, with gamma = 0 and the |g|^2 coefficient c_g = 1/d per row, so that the rows of a
// point add up to  sum_i (|g|^2 / d - 2 D_{e_i}^2 V) = |g|^2 - 2 Laplacian V  (and the same for the parameter gradient;
// the g-stream is linear in its direction, so c_g enters once, as the direction c_g g / 2 written in E6).  a.fp_dirs = d: virtual tile T is
// (point tile T / d, direction T % d): the d tiles of one point tile are consecutive (its inputs stay in L1 / L2) and
// every row of a tile has the same direction.  Cost: d KFP evaluations per point (the primal, the input-gradient chain
// and the g-stream are recomputed per direction: ~2x the executed FLOPs of a shared-primal kernel).
#include "mlp_thread.cuh"
#include "residual_common.cuh"
#include "umma.cuh"

namespace pdeip {

int mlp_residual_accumulate_fp32(int set_kind, const ResidualArgs& a, int hidden, cudaStream_t st);

namespace tc {

using namespace umma;

constexpr int H = 32;
constexpr int OP = 48;  // output width 40 padded to a multiple of 16

// ---- TMEM column map: [0, 112) persistent dW accumulators, then NS slots of 200 columns -----------------------
constexpr uint32_t C_DW2 = 0, C_DW1 = 48, C_DW0 = 80, C_SLOT0 = 112, SLOT_COLS = 200;
// slot-relative
constexpr uint32_t C_S1P1 = 0, C_S1P2 = 16;  // parked s1 of hidden layers 1 / 2 (packed bf16 pairs, 16 columns)
constexpr uint32_t C_R = 32;                  // 144 transient columns
constexpr uint32_t C_Z0 = C_R + 0, C_Z10 = C_R + 32;                       // P0
constexpr uint32_t C_Z1 = C_R + 64, C_Z11 = C_R + 96, C_Z21 = C_R + 0;      // P1
constexpr uint32_t C_U = C_R + 0, C_U1 = C_R + 48, C_U2 = C_R + 96;         // P2
constexpr uint32_t C_S0P = 176;                                            // parked s0p (24 columns)
constexpr uint32_t C_AA2 = C_R + 0, C_AB12 = C_R + 32, C_PZ2 = C_R + 128;   // P3 / E4
constexpr uint32_t C_AA1 = C_R + 64, C_AB11 = C_R + 96, C_PZ1 = C_R + 0;    // P4 / E5
constexpr uint32_t C_G = C_R + 16;                                         // P5
constexpr uint32_t C_ZG0 = C_R + 64, C_ZG1 = C_R + 96, C_UG = C_R + 48;     // P6, P7, P8
constexpr uint32_t C_AB2 = C_R + 16, C_AA2R = C_R + 96;                     // P9
constexpr uint32_t C_AB1 = C_R + 48, C_AA1R = C_R + 96;                     // P10

// PDEIP_TC_TS (on; round-1 verdict item 1a).  One-slot kernels (d > 8) use 312 of the 512 TMEM columns: the next 48 hold
// the A OPERAND of the layer GEMMs (tcgen05.mma [d], [a_tmem], b_desc: lane = point row, column c = the bf16 pair
// (k = 2c, 2c + 1) of that row): the epilogue thread that packs an 8-unit chunk for the shared-memory tile (which the
// batch-reduced dW GEMMs still read through the transposed view) also stores the same four words to TMEM.
// Cost model measured with tools/umma_cost.py (profiles/r02_umma_cost.txt): a 128 x N x 16 MMA with both operands in
// shared memory costs (4 KB of A + 32 N bytes of B) / 128 B per clock + 4 = 44 / 47 cycles at N = 32 / 48 (shared-memory
// operand bandwidth, whatever the accumulator or the operand rotation); with A in TMEM it costs N / 2 + 2 = 18 / 27
// cycles (the math).  The first measurement of this switch saw no gain because the MMA warp itself was the bottleneck
// (24 registers after setmaxnreg: 75 spill instructions and R2UR chains in front of the MMAs of every phase); with the
// MMA warp on the uniform datapath the GEMM phases shorten by ~100 cycles each: d = 32 2.055e9 -> 2.24e9 evals/s.
constexpr uint32_t C_AOP = C_SLOT0 + SLOT_COLS;  // [312, 360): columns = 4 x (chunk index within the operand)
constexpr uint32_t C_AOPX = C_AOP + 48;           // [360, 408): the A operands of P0 ([x_hi | x_lo], v) when E0 runs a tile ahead (PIPE_X)
// [408, 512): one-slot kernels keep the per-row bias-gradient sums here, 26 per epilogue part (db0 8, db1 8, db2 10):
// db0 at [408 + 8 part, +8), db1 at [440 + 8 part, +8), db2 chunk units at [472 + 8 part, +8), db2 pair at [504 + 2 part, +2)
constexpr uint32_t C_DB = C_AOPX + 48;
static_assert(C_DB + 4 * 26 == 512, "TMEM column map");

// ---- shared memory ---------------------------------------------------------------------------------------------
// Z tile chunk map (24 chunks of 8 columns)
constexpr int ZC_ZA2 = 0, ZC_ZA1 = 6, ZC_ZA0 = 10, ZC_TA = 14, ZC_TB = 20;
// A tile chunk map (12 chunks): t | a1 (later the g-stream operand ag^) | a2^ (later c = a2^ + ag^)
constexpr int AC_T = 0, AC_A1 = 4, AC_C = 8;

// Thread shape.  Epilogue thread = (point row == TMEM lane, one "part" of the units): warp w reads TMEM lane quadrant
// q = w & 3 and owns part w >> 2.  One-slot kernels run 16 epilogue warps (4 parts: 8 of the 32 hidden units, and of
// the 40 output units 8 + 2, see OutCols), the two-slot kernel 8 (2 parts: 16 hidden units, 24 of the 48 output
// columns): with one slot nothing overlaps an epilogue phase, so its length is the tile's critical path, and it is
// bound by the latency of each thread's dependent chain, which more warps per scheduler shorten.
template <int NS>
struct Team {
  static constexpr int kEpiWarps = NS == 1 ? 16 : 8;
  static constexpr int kParts = kEpiWarps / 4;
  static constexpr int kEpiThreads = 32 * kEpiWarps;
  static constexpr int kThreads = kEpiThreads + 32;  // + one MMA-issuing warp (threads taking part in the named barriers)
  // Launched with a full extra warpgroup (the MMA warp and three idle warps) so that `setmaxnreg` can move registers:
  // the register file is 16 K per scheduler and each scheduler hosts kEpiWarps / 4 epilogue warps and one warp of the
  // extra group; the extra group shrinks and the epilogue groups grow (Regs<NS> below; no spills).
  static constexpr int kLaunchThreads = kEpiThreads + 128;
  // registers per thread the kernel is compiled and launched at (__launch_bounds__(kLaunchThreads, 1): the register
  // file over the threads, rounded down to the allocation granule of 8); tests/test_residual_tc_resources.py checks
  // that ptxas reports exactly this
  static constexpr int kLaunchRegs = 65536 / kLaunchThreads / 8 * 8;
};
template <int DP, int NS>
struct Cfg {
  static constexpr int XC = DP / 8;                  // chunks per input band
  static constexpr int NX = 4 * XC;                  // x_hi | x_lo | v | g^
  static constexpr int KX = 2 * DP;                  // K of the x GEMM ([x_hi | x_lo] against [W0; W0])
  static constexpr int KV = DP < 16 ? 16 : DP;       // K of the v / g^ GEMMs, N of the g GEMM
  static constexpr int XC_HI = 0, XC_LO = XC, XC_V = 2 * XC, XC_G = 3 * XC;
  static constexpr uint32_t RG_X = NX * 128, RG_A = 12 * 128, RG_Z = 24 * 128;
  static constexpr uint32_t SZ_X = 16 * RG_X, SZ_A = 16 * RG_A, SZ_Z = 16 * RG_Z;
  static constexpr uint32_t O_X = 0, O_A1 = O_X + SZ_X, O_A2 = O_A1 + SZ_A, O_Z = O_A2 + SZ_A, SLOT = O_Z + SZ_Z;
  // PDEIP_TC_PIPE_X (one-slot kernels; on): the x | v | g^ bands are double-buffered by tile parity, so that E0 of the
  // NEXT tile (the bf16 hi / lo split of its inputs) runs behind E10's hand-off while P10 executes, P0 of the next tile
  // is issued with P11 behind E11's hand-off, and the tile has 10 GEMM -> epilogue round trips instead of 11.
#ifndef PDEIP_TC_PIPE_X
#define PDEIP_TC_PIPE_X 1
#endif
#ifndef PDEIP_TC_STAGE
#define PDEIP_TC_STAGE 0  // (see STAGE_BYTES below)
#endif
  static constexpr bool PIPE_X = PDEIP_TC_PIPE_X && NS == 1 && !PDEIP_TC_STAGE;
  // second x | v | g^ buffer (odd tiles).  It sits between the slot and the weights, NOT at the end of the allocation: the
  // M = 64 band-shifted dW chains read 64 operand columns from the start of a band, i.e. up to (8 - XC) x 128 B past the
  // last row group of the tile (the cross-term rows that nobody reads) — harmless while something is mapped behind the
  // tile, an illegal-address fault when the tile is the last thing in shared memory (measured).
  static constexpr uint32_t O_X2 = NS * SLOT;
  // weights (rows = output units, columns = input units), hi and lo halves
  static constexpr uint32_t RG_T0X = KX / 8 * 128, SZ_T0X = 4 * RG_T0X;
  static constexpr uint32_t RG_T0V = KV / 8 * 128, SZ_T0V = 4 * RG_T0V;
  static constexpr uint32_t RG_T1 = 512, SZ_T1 = 4 * RG_T1, RG_T2 = 512, SZ_T2 = 6 * RG_T2;
  static constexpr uint32_t O_T0XH = NS * SLOT + (PIPE_X ? SZ_X : 0u), O_T0XL = O_T0XH + SZ_T0X, O_T0VH = O_T0XL + SZ_T0X,
                            O_T0VL = O_T0VH + SZ_T0V, O_T1H = O_T0VL + SZ_T0V, O_T1L = O_T1H + SZ_T1,
                            O_T2H = O_T1L + SZ_T1, O_T2L = O_T2H + SZ_T2,
                            // Gram tile G = c_g W0 W0^T / 8 ([32 hidden][32 hidden], hi + lo): one-slot kernels only
                            O_TGH = O_T2L + SZ_T2, O_TGL = O_TGH + (NS == 1 ? SZ_T1 : 0u),
                            O_BIAS = O_TGL + (NS == 1 ? SZ_T1 : 0u);
  static constexpr uint32_t TP_BYTES = NS == 2 ? 2048 : 4096;
  // PDEIP_TC_STAGE (off by default; round-1 verdict item 8, built and measured in round 2).  One-slot kernels have shared
  // memory to spare: the next tile of a BLOCK128 point set ([3 DP][128] floats, one contiguous block) can be staged by ONE
  // bulk copy of the TMA unit (cp.async.bulk global -> shared, mbarrier complete_tx; UBLKCP in SASS) issued five phases
  // ahead, instead of 48 LDG per thread behind a bulk L2 prefetch, and E0 / E6 read their row from it.  Correct (all GPU
  // tests pass with it), but 5-7 % SLOWER (d = 32: 1.94e9 -> 1.80-1.84e9 evals/s, d = 16: 2.15e9 -> 2.01-2.07e9): the
  // inputs are 1.3 % of the stall samples already (L2 hits landing behind the wait for P11), and the 49 KB write through
  // the async proxy competes with the operand fetches of the dW chains for shared-memory bandwidth.
#ifndef PDEIP_TC_STAGE
#define PDEIP_TC_STAGE 0
#endif
  static constexpr uint32_t STAGE_BYTES = (PDEIP_TC_STAGE && NS == 1) ? 128u * 3u * DP * 4u : 0u;
  // one-slot kernels: the five loss sums of every epilogue thread, [5][epilogue threads] floats (see kSumsSmem)
  static constexpr uint32_t SUMS_BYTES = NS == 1 ? 5u * 4u * Team<NS>::kEpiThreads : 0u;
  static constexpr uint32_t O_TRUE = O_BIAS + 512, O_MISC = O_TRUE + TP_BYTES, O_STAGE = O_MISC + 128,
                            O_SUMS = O_STAGE + STAGE_BYTES, TOTAL = O_SUMS + SUMS_BYTES;
  static_assert(TOTAL <= 227u * 1024u && O_STAGE % 128 == 0 && O_X2 % 1024 == 0, "shared-memory budget");
};

#ifndef PDEIP_TC_G_CHAIN_EARLY
#define PDEIP_TC_G_CHAIN_EARLY 1
#endif
#ifndef PDEIP_TC_NLO_FWD
// Measured (tools/nlo_study.sh, tools/tensor_errors.py): the lo halves matter for the primal stream (it feeds tanh) and
// for the input-gradient chain (|g|^2 enters the loss); on the tangent streams and the order-1 adjoint they change
// neither the loss nor the gradient error (1.4e-3 at d = 8 either way) and cost 3 % (8 of the 24 MMAs of P1 + P2).
#define PDEIP_TC_NLO_FWD 1  // streams of P1 / P2 (primal, order 1, order 2) that get the lo halves of W1 / W2
#endif
#ifndef PDEIP_TC_NLO_BWD
#define PDEIP_TC_NLO_BWD 1  // streams of P3 / P4 (input-gradient chain, order-1 adjoint) that get the lo halves
#endif
#ifndef PDEIP_TC_LO_FWD
#define PDEIP_TC_LO_FWD true  // lo halves of W1, W2 in the forward layer GEMMs P1, P2
#endif
// (epilogue, extra group) register budgets after setmaxnreg
#ifndef PDEIP_TC_REGS1_EPI
#define PDEIP_TC_REGS1_EPI 104
#define PDEIP_TC_REGS1_MMA 40
#endif
#ifndef PDEIP_TC_REGS2_EPI
#define PDEIP_TC_REGS2_EPI 208
#define PDEIP_TC_REGS2_MMA 88
#endif
template <int NS>
struct Regs {
  static constexpr int kEpi = NS == 2 ? PDEIP_TC_REGS2_EPI : PDEIP_TC_REGS1_EPI;
  static constexpr int kMma = NS == 2 ? PDEIP_TC_REGS2_MMA : PDEIP_TC_REGS1_MMA;
  // measured: a scheduler's epilogue warps can only grow into what its warp of the extra group releases, i.e. the
  // pool is (epilogue warps per scheduler + 1) x the launch count (two-slot kernel at 168: 2 x 216 + 80 = 512 never
  // returns; 2 x 208 + 88 = 504 works).  One-slot kernels at 96: 4 x 104 + 40 = 456 <= 480; 4 x 112 + 40 does not fit.
  static constexpr int kEpiPerSched = Team<NS>::kEpiWarps / 4, kLaunch = Team<NS>::kLaunchRegs;
  static_assert(kEpiPerSched * kEpi + kMma <= (kEpiPerSched + 1) * kLaunch && kEpi >= kLaunch && kMma <= kLaunch &&
                    kEpi % 8 == 0 && kMma % 8 == 0 && kMma >= 24 && kEpi <= 256,
                "setmaxnreg budgets: an impossible request never returns (the kernel hangs)");
};

template <int V>
struct IC {
  static constexpr int value = V;
};

// PDEIP_TC_TRACE builds: clock stamps SUMMED over kTraceTiles steady-state tile rounds of CTA 0 (differences of the sums
// are sums of the differences; the tool divides): trace[(ph * 2 + slot) * 8 + k],
// k = 0 epilogue wait start, 1 wait end, 2 arrive;  4 MMA warp operands ready, 5 fast GEMMs issued, 6 all issued
#ifdef PDEIP_TC_TRACE
constexpr int kTraceTiles = 64;
// (fire-and-forget reductions: a load-add-store would stall the stamped thread on the load)
#define TC_TRACE(k) do { if (trace_on) atomicAdd(reinterpret_cast<unsigned long long*>(trace) + (ph * 2 + s) * 8 + (k), (unsigned long long)clock64()); } while (0)
#define TC_FINE(k) do { if (trace_on && ph == 4) atomicAdd(reinterpret_cast<unsigned long long*>(trace) + 240 + s * 8 + (k), (unsigned long long)clock64()); } while (0)
#define TC_TRACE_DECL_MMA                                                     \
  long long* trace = reinterpret_cast<long long*>(status) + 512;              \
  const bool trace_on = blockIdx.x == 0 && base >= tile_begin + (int64_t)16 * tile_stride && base < tile_begin + (int64_t)(16 + kTraceTiles) * tile_stride
#else
#define TC_TRACE(k) do { } while (0)
#define TC_FINE(k) do { } while (0)
#define TC_TRACE_DECL_MMA do { } while (0)
#endif

#ifdef PDEIP_TC_PROBE
#define TC_PROBE(id, unit0, arr, n)                                                              \
  do {                                                                                           \
    if (probe_on) {                                                                              \
      for (int _i = 0; _i < (n); ++_i) probe[((id) * 128 + row) * 48 + (unit0) + _i] = (arr)[_i]; \
    }                                                                                            \
  } while (0)
#else
#define TC_PROBE(id, unit0, arr, n) do { } while (0)
#endif
// the output-layer units of this thread (OutCols oc)
#define TC_PROBE_OUT(id, arr)                                                                       \
  do {                                                                                              \
    TC_PROBE(id, oc.unit0(), arr, 8 * OutCols<NP>::NC);                                             \
    if constexpr (OutCols<NP>::PAIR) TC_PROBE(id, oc.pair_unit(), (arr) + 8 * OutCols<NP>::NC, 2); \
  } while (0)

// epilogue side: operands written -> visible to the tensor core; TMEM accesses ordered; signal the MMA warp
template <int NS, bool PROXY_FENCE = true>
__device__ __forceinline__ void epi_arrive(int slot) {
  if constexpr (PROXY_FENCE) fence_async_smem();
  fence_before_sync();
  asm volatile("bar.arrive %0, %1;" ::"r"(1 + slot), "n"(Team<NS>::kThreads) : "memory");
}
// MMA warp: wait until every epilogue thread has arrived
template <int NS>
__device__ __forceinline__ void mma_wait_operands(int slot) {
  asm volatile("bar.sync %0, %1;" ::"r"(1 + slot), "n"(Team<NS>::kThreads) : "memory");
  fence_after_sync();
}

// ---- descriptors as (lo, hi) 32-bit halves; advancing = one add on lo (addresses stay below 256 KB) ----------
struct Desc {
  uint32_t lo, hi;
};
__device__ __forceinline__ Desc mk_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  Desc d;
  d.lo = ((saddr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
  d.hi = ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14);  // descriptor version 1 (bit 46)
  return d;
}
// the same descriptor from base16 = (1024-aligned shared-window address) >> 4 and a compile-time byte offset: ONE add
// (shared addresses stay below 2^18, so the 14-bit address field cannot carry into the LBO field)
__device__ __forceinline__ Desc mk_desc16(uint32_t base16, uint32_t off_bytes, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  Desc d;
  d.lo = base16 + ((off_bytes >> 4) | (((lbo_bytes >> 4) & 0x3FFFu) << 16));
  d.hi = ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14);
  return d;
}
// value the compiler can neither hoist out of a loop nor keep live across it (the MMA warp runs on a small register
// budget after setmaxnreg: everything it needs is re-derived from two bases inside each phase)
__device__ __forceinline__ uint32_t opaque(uint32_t v) {
  uint32_t r;
  asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(v));
  return r;
}
__device__ __forceinline__ void mma(uint32_t d_tmem, Desc a, uint32_t a_adv, Desc b, uint32_t b_adv, uint32_t idesc,
                                    uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a.lo + (a_adv >> 4)), "r"(a.hi), "r"(b.lo + (b_adv >> 4)), "r"(b.hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, Desc b, uint32_t b_adv, uint32_t idesc,
                                       uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 db;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "r"(b.lo + (b_adv >> 4)), "r"(b.hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// the same GEMMs with the A operands in TMEM: a_col[g] = first TMEM column of stream g's operand (8 columns per k-step)
template <int K, int N, int NG, bool LO = true, int NLO = NG>
__device__ __forceinline__ void mm_fwd_ts(const uint32_t (&d)[NG], const uint32_t (&a_col)[NG], Desc w_hi, Desc w_lo) {
  constexpr uint32_t idesc = make_idesc(N, 0, 0);
#pragma unroll
  for (int k = 0; k < K; k += 16)
#pragma unroll
    for (int g = 0; g < NG; ++g) mma_ts(d[g], a_col[g] + (k >> 1), w_hi, k * 16, idesc, k > 0 ? 1u : 0u);
  if constexpr (LO) {
#pragma unroll
    for (int k = 0; k < K; k += 16)
#pragma unroll
      for (int g = 0; g < NLO; ++g) mma_ts(d[g], a_col[g] + (k >> 1), w_lo, k * 16, idesc, 1u);
  }
}
template <int K, int N, int NG, bool LO = true, int NLO = NG>
__device__ __forceinline__ void mm_bwd_ts(const uint32_t (&d)[NG], const uint32_t (&a_col)[NG], Desc w_hi_m, Desc w_lo_m,
                                          uint32_t w_rg) {
  constexpr uint32_t idesc = make_idesc(N, 0, 1);
#pragma unroll
  for (int k = 0; k < K; k += 16)
#pragma unroll
    for (int g = 0; g < NG; ++g) mma_ts(d[g], a_col[g] + (k >> 1), w_hi_m, (k >> 3) * w_rg, idesc, k > 0 ? 1u : 0u);
  if constexpr (LO) {
#pragma unroll
    for (int k = 0; k < K; k += 16)
#pragma unroll
      for (int g = 0; g < NLO; ++g) mma_ts(d[g], a_col[g] + (k >> 1), w_lo_m, (k >> 3) * w_rg, idesc, 1u);
  }
}

// NG independent forward GEMMs D_g[128 x N] = A_g(K-major, K columns) * W^T(K-major tile [N][K]), hi + lo halves of
// the weights, issued round-robin over g.  a_off[g] / d[g]: byte offset of the A band / TMEM column of GEMM g.
// NLO: the lo weight halves are applied to the first NLO of the NG streams only
template <int K, int N, int NG, bool LO = true, int NLO = NG>
__device__ __forceinline__ void mm_fwd(const uint32_t (&d)[NG], Desc a, const uint32_t (&a_off)[NG], Desc w_hi, Desc w_lo) {
  constexpr uint32_t idesc = make_idesc(N, 0, 0);
#pragma unroll
  for (int k = 0; k < K; k += 16)
#pragma unroll
    for (int g = 0; g < NG; ++g) mma(d[g], a, a_off[g] + k * 16, w_hi, k * 16, idesc, k > 0 ? 1u : 0u);
  if constexpr (LO) {
#pragma unroll
    for (int k = 0; k < K; k += 16)
#pragma unroll
      for (int g = 0; g < NLO; ++g) mma(d[g], a, a_off[g] + k * 16, w_lo, k * 16, idesc, 1u);
  }
}
// NG backward GEMMs D_g[128 x N] = A_g(K-major, K columns) * W (transposed view of the weight tile, rows = K)
template <int K, int N, int NG, bool LO = true, int NLO = NG>
__device__ __forceinline__ void mm_bwd(const uint32_t (&d)[NG], Desc a, const uint32_t (&a_off)[NG], Desc w_hi_m,
                                       Desc w_lo_m, uint32_t w_rg) {
  constexpr uint32_t idesc = make_idesc(N, 0, 1);
#pragma unroll
  for (int k = 0; k < K; k += 16)
#pragma unroll
    for (int g = 0; g < NG; ++g) mma(d[g], a, a_off[g] + k * 16, w_hi_m, (k >> 3) * w_rg, idesc, k > 0 ? 1u : 0u);
  if constexpr (LO) {
#pragma unroll
    for (int k = 0; k < K; k += 16)
#pragma unroll
      for (int g = 0; g < NLO; ++g) mma(d[g], a, a_off[g] + k * 16, w_lo_m, (k >> 3) * w_rg, idesc, 1u);
  }
}
// band-shifted batch-reduced outer product: D[m][n] += sum_points A[p][a_col0 + m] * B[p][b_col0 + n]
// (both operands transposed views; a_off / b_off = byte offsets of the first chunk of the band)
template <int N>
__device__ __forceinline__ void mm_outer(uint32_t d, Desc a_m, uint32_t a_off, uint32_t a_rg, Desc b_m, uint32_t b_off,
                                         uint32_t b_rg, uint32_t accumulate) {
  // M = 64 instruction shape: only rows 0..31 of a dW block are wanted, and the A fetch (the cost of these MMAs:
  // both operands come from shared memory) halves.  Row i of D lands in TMEM lane (i % 16) + 32 (i / 16)
  // (measured: tools/umma_m64_probe.py, tests/test_gpu_umma.py).
  constexpr uint32_t idesc = (make_idesc(N, 1, 1) & ~(0x1Fu << 24)) | ((uint32_t)(64 >> 4) << 24);
#pragma unroll
  for (int k = 0; k < 128; k += 16)
    mma(d, a_m, a_off + (k >> 3) * a_rg, b_m, b_off + (k >> 3) * b_rg, idesc, k > 0 ? 1u : accumulate);
}

// MUFU tanh (max relative error ~2^-11, below the bf16 rounding applied to every activation operand)
__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---- packed bf16 helpers -----------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&p);
}
__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
// 8 floats <- one 16-byte chunk of an operand tile
__device__ __forceinline__ void load_chunk(const uint8_t* tile, uint32_t off, float* v) {
  const uint4 q = *reinterpret_cast<const uint4*>(tile + off);
  v[0] = bf_lo(q.x); v[1] = bf_hi(q.x); v[2] = bf_lo(q.y); v[3] = bf_hi(q.y);
  v[4] = bf_lo(q.z); v[5] = bf_hi(q.z); v[6] = bf_lo(q.w); v[7] = bf_hi(q.w);
}
__device__ __forceinline__ void put_chunk(uint8_t* tile, uint32_t off, const float* v) {
  uint4 q;
  q.x = pack2(v[0], v[1]); q.y = pack2(v[2], v[3]); q.z = pack2(v[4], v[5]); q.w = pack2(v[6], v[7]);
  *reinterpret_cast<uint4*>(tile + off) = q;
}
// ---- TMA bulk copy (global -> shared, completion on an mbarrier) --------------------------------------------------
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
               "l"(src), "r"(bytes), "r"(mbar)
               : "memory");
}
__device__ __forceinline__ void tm_st4(uint32_t taddr, const uint32_t* r);
// the chunk to shared memory AND (TS) the same four packed words to the A-operand columns of this thread's TMEM lane
template <bool TS>
__device__ __forceinline__ void put_op(uint8_t* tile, uint32_t off, uint32_t taddr, const float* v) {
  uint4 q;
  q.x = pack2(v[0], v[1]); q.y = pack2(v[2], v[3]); q.z = pack2(v[4], v[5]); q.w = pack2(v[6], v[7]);
  *reinterpret_cast<uint4*>(tile + off) = q;
  if constexpr (TS) tm_st4(taddr, reinterpret_cast<const uint32_t*>(&q));
}
// TMEM: raw loads (no wait), 8 or 16 consecutive 32-bit columns of this thread's lane
__device__ __forceinline__ void tm_ld8(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tm_ld4(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tm_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tm_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tm_st8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tm_st4(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3])
               : "memory");
}
__device__ __forceinline__ void tm_ld2(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tm_ld1(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r[0]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tm_st2(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1,%2};" ::"r"(taddr), "r"(r[0]), "r"(r[1]) : "memory");
}
__device__ __forceinline__ void tm_st1(uint32_t taddr, uint32_t r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(r) : "memory");
}
// NU fp32 columns (NU = 8, 16 or 24) -> floats, no wait
template <int NU>
__device__ __forceinline__ void tm_ldf(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  if constexpr (NU == 8) {
    tm_ld8(taddr, r);
  } else {
    tm_ld16(taddr, r);
    if constexpr (NU == 24) tm_ld8(taddr + 16, r + 16);
  }
}
// NU parked values = NU / 2 columns of packed bf16 pairs
template <int NU>
__device__ __forceinline__ void tm_ldp(uint32_t taddr, uint32_t* r) {
  if constexpr (NU == 8) {
    tm_ld4(taddr, r);
  } else {
    tm_ld8(taddr, r);
    if constexpr (NU == 24) tm_ld4(taddr + 8, r + 8);
  }
}
// stores only (the caller waits with tm_wait_st)
template <int NU>
__device__ __forceinline__ void tm_park_st(uint32_t taddr, const float* v) {
  uint32_t r[NU / 2];
#pragma unroll
  for (int i = 0; i < NU / 2; ++i) r[i] = pack2(v[2 * i], v[2 * i + 1]);
  if constexpr (NU == 8) {
    tm_st4(taddr, r);
  } else {
    tm_st8(taddr, r);
    if constexpr (NU == 24) tm_st4(taddr + 8, r + 8);
  }
}
template <int NU>
__device__ __forceinline__ void tm_park(uint32_t taddr, const float* v) {
  tm_park_st<NU>(taddr, v);
  tm_wait_st();
}

// Output-layer units (48 columns, 40 real) of epilogue part `part` out of NP.  NP = 2: columns [24 part, +24).  NP = 4:
// chunk `part` (columns [8 part, +8)) plus the pair 32 + 2 part, 33 + 2 part of chunk 4, 10 units per thread; chunk 5
// (columns 40..47) is padding with zero weights and bias that no thread owns.  Every array over a thread's output units
// holds the NC chunk units first, then the PAIR units.  Packed bf16 values (parked in TMEM or stored as an operand)
// follow the same map: column pair k of the chunk units at word 4 NC part + k, the pair at word 16 + part.
template <int NP>
struct OutCols {
  static constexpr int NC = NP == 2 ? 3 : 1;  // full 8-unit chunks per thread
  static constexpr bool PAIR = NP == 4;
  static constexpr int NU = 8 * NC + (PAIR ? 2 : 0);
  const int part;
  __device__ __forceinline__ int unit0() const { return 8 * NC * part; }  // first chunk unit
  __device__ __forceinline__ int chunk0() const { return NC * part; }
  __device__ __forceinline__ int pair_unit() const { return 32 + 2 * part; }
  __device__ __forceinline__ int unit(int i) const { return i < 8 * NC ? unit0() + i : pair_unit() + i - 8 * NC; }
  // NU fp32 accumulator columns of this thread (no wait)
  __device__ __forceinline__ void ldf(uint32_t taddr, float* v) const {
    tm_ldf<8 * NC>(taddr + unit0(), v);
    if constexpr (PAIR) tm_ld2(taddr + pair_unit(), reinterpret_cast<uint32_t*>(v + 8 * NC));
  }
  // NU / 2 parked words (no wait)
  __device__ __forceinline__ void ldp(uint32_t taddr, uint32_t* r) const {
    tm_ldp<8 * NC>(taddr + 4 * NC * part, r);
    if constexpr (PAIR) tm_ld1(taddr + 16 + part, r + 4 * NC);
  }
  __device__ __forceinline__ void park(uint32_t taddr, const float* v) const {
    tm_park_st<8 * NC>(taddr + 4 * NC * part, v);
    if constexpr (PAIR) tm_st1(taddr + 16 + part, pack2(v[8 * NC], v[8 * NC + 1]));
    tm_wait_st();
  }
  // bias (or any 48-float vector in shared memory) of this thread's units
  __device__ __forceinline__ void ld_smem(const float* b, float* v) const {
#pragma unroll
    for (int i = 0; i < 2 * NC; ++i)
      *reinterpret_cast<float4*>(v + 4 * i) = *reinterpret_cast<const float4*>(b + unit0() + 4 * i);
    if constexpr (PAIR) *reinterpret_cast<float2*>(v + 8 * NC) = *reinterpret_cast<const float2*>(b + pair_unit());
  }
  // this thread's units of a 48-column band of an operand tile (first chunk c0; `row` = the thread's row offset) and,
  // with TS, of its A-operand copy in TMEM (first word w0 of the band in this thread's lane)
  template <bool TS>
  __device__ __forceinline__ void put(uint8_t* row, int c0, uint32_t w0, const float* v) const {
#pragma unroll
    for (int c = 0; c < NC; ++c) put_op<TS>(row, (c0 + NC * part + c) * 128, w0 + 4 * (NC * part + c), v + 8 * c);
    if constexpr (PAIR) {
      const uint32_t w = pack2(v[8 * NC], v[8 * NC + 1]);
      *reinterpret_cast<uint32_t*>(row + (c0 + 4) * 128 + 4 * part) = w;
      if constexpr (TS) tm_st1(w0 + 16 + part, w);
    }
  }
};

// inline true gradient (LINEAR: A x; GMM: core/potential.py:32-37), components [8 cg, 8 cg + 8) of point p (p < 0: none).
// Cold path (tests and the reference-shaped API; the pipeline stores grad U next to the point): kept out of line.
template <int DP>
__device__ __noinline__ void true_grad_chunk(const ResidualArgs& a, const float* __restrict__ tp, int64_t p, int dimw,
                                             int cg, float* gt) {
  const int d = a.d;
  float x[DP];
#pragma unroll
  for (int u = 0; u < DP; ++u)
    x[u] = (p >= 0 && u < d) ? __ldg(a.points + elem_index(a.layout, p, u, a.n_points, dimw)) : 0.f;
  if (a.tg.kind == PDEIP_DRIFT_LINEAR) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int u = cg * 8 + e;
      float acc = 0.f;
      if (u < d) {
#pragma unroll
        for (int k = 0; k < DP; ++k)
          if (k < d) acc = fmaf(tp[u * d + k], x[k], acc);
      }
      gt[e] = acc;
    }
  } else {
    float m = -INFINITY;
    for (int k = 0; k < a.tg.n_gaussian; ++k) {
      float s2 = 0.f;
#pragma unroll
      for (int u = 0; u < DP; ++u)
        if (u < d) {
          const float r = x[u] - tp[k * d + u];
          s2 = fmaf(r, r, s2);
        }
      m = fmaxf(m, -0.5f * a.tg.inv_sigma2 * s2);
    }
    float se = 0.f, wm[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) wm[e] = 0.f;
    for (int k = 0; k < a.tg.n_gaussian; ++k) {
      float s2 = 0.f;
#pragma unroll
      for (int u = 0; u < DP; ++u)
        if (u < d) {
          const float r = x[u] - tp[k * d + u];
          s2 = fmaf(r, r, s2);
        }
      const float ek = __expf(-0.5f * a.tg.inv_sigma2 * s2 - m);
      se += ek;
#pragma unroll
      for (int e = 0; e < 8; ++e)
        if (cg * 8 + e < d) wm[e] = fmaf(ek, tp[k * d + cg * 8 + e], wm[e]);
    }
    const float inv = 1.f / se;
#pragma unroll
    for (int e = 0; e < 8; ++e) gt[e] = (cg * 8 + e < d) ? (x[cg * 8 + e] - wm[e] * inv) * a.tg.inv_sigma2 : 0.f;
  }
}
__device__ __forceinline__ float unp(const uint32_t* r, int i) { return (i & 1) ? bf_hi(r[i >> 1]) : bf_lo(r[i >> 1]); }

// ---- packed fp32x2 epilogue arithmetic (FFMA2 / FMUL2 / FADD2: one issue slot per two values).  Every array of
// the epilogues is paired (2 i, 2 i + 1): adjacent TMEM columns, the two halves of a packed bf16 word. -------------
#ifndef PDEIP_TC_PACKED
#define PDEIP_TC_PACKED 1
#endif
__device__ __forceinline__ float2 pr(const float* v, int i) { return make_float2(v[2 * i], v[2 * i + 1]); }
__device__ __forceinline__ void st2(float* v, int i, float2 x) { v[2 * i] = x.x; v[2 * i + 1] = x.y; }
__device__ __forceinline__ float2 unp2(const uint32_t* r, int i) { return make_float2(bf_lo(r[i]), bf_hi(r[i])); }
__device__ __forceinline__ float2 bc2(float x) { return make_float2(x, x); }

// BND: the KFP boundary sets (kinetic_fokker_planck.py:34-39,48-50: l = coef grad V . v, coef = +-2/T) on the same phase
// schedule with the seeds of that loss (alpha = 0, beta = coef, no |g|^2 term: za^ = 0, so the input-gradient chain, the
// g-stream and the c chains carry zeros) and the lo weight halves on EVERY stream: mean D_v V over a boundary set is a
// heavily cancelling sum, and the systematic part of the bf16 weight rounding (the same for every point, it does not
// average out) showed at 1.1e-2 in that term with hi-only tangent streams (profiles/r01_summary_tensor_v2.md item 7).
// MODE: 0 KFP 0T set, 1 KFP boundary set (BND), 2 FP 0T set as direction tiles (FPM) — compile-time, so that the 0T kernel
// carries none of the other modes' code (the epilogue is instruction-fetch sensitive).
constexpr int kModeKfp0T = 0, kModeBnd = 1, kModeFp0T = 2;
template <int DP, int NS, int MODE>
__global__ void __launch_bounds__(Team<NS>::kLaunchThreads, 1) mlp_residual_tc_kernel(const ResidualArgs a, int* status) {
  constexpr bool BND = MODE == kModeBnd, FPM = MODE == kModeFp0T;
#ifndef PDEIP_TC_TS
#define PDEIP_TC_TS 1  // see C_AOP above
#endif
  constexpr bool kTS = PDEIP_TC_TS && NS == 1;  // layer-GEMM A operands from TMEM (the two-slot kernel has no columns left)
#ifndef PDEIP_TC_GRAM
#define PDEIP_TC_GRAM 1
#endif
  // One-slot kernels: zg^_0 = g^ W0 = za^0 (W0 W0^T) c_g / 8 comes out of P5 itself through the Gram tile (hi + lo; the
  // two-slot kernel has no shared memory for it), so that E6 and E7 run back to back and the P6 hand-off disappears:
  // 11 GEMM -> epilogue round trips per tile instead of 12, and zg^_0 no longer passes through the bf16 rounding of g^.
  constexpr bool kGram = PDEIP_TC_GRAM && NS == 1;
  // Two-stage hand-off (one-slot kernels with the A operands in TMEM): the layer GEMMs of a phase read TMEM and the
  // weights only, so they are released by a first arrive right behind tcgen05.wait::st; the generic -> async proxy fence,
  // which only the dW chains of the phase need (they read the activation bands from shared memory), follows on a second
  // named barrier while the layer GEMMs already execute.
#ifndef PDEIP_TC_TWO_STAGE
#define PDEIP_TC_TWO_STAGE 1
#endif
  constexpr bool kTwoStage = PDEIP_TC_TWO_STAGE && kTS;
  constexpr bool kPipeX = Cfg<DP, NS>::PIPE_X;  // E0 / P0 of the next tile ride behind E10 / with P11 (see Cfg)
  constexpr bool kPipeFlow = kPipeX;  // the schedule that goes with the second buffer
  using S = Cfg<DP, NS>;
  constexpr int kEpiThreads = Team<NS>::kEpiThreads, kThreads = Team<NS>::kThreads, kLaunchThreads = Team<NS>::kLaunchThreads;
  constexpr int NP = Team<NS>::kParts;  // epilogue parts (see Team)
  constexpr int UH = 32 / NP;           // hidden units per epilogue thread
  constexpr int HC = UH / 8;            // ... in 8-unit chunks
  extern __shared__ __align__(1024) uint8_t sm[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool is_mma_warp = warp == kEpiThreads / 32;
  const int q = warp & 3;         // TMEM lane quadrant of this warp
  const int part = warp >> 2;      // which UH of the 32 hidden units (and which output units, OutCols) this thread owns
  const int row = q * 32 + lane;  // point within the tile == TMEM lane == operand tile row
  const int d = a.d;
  const MlpShape<H> sh{d, 2};
  const int P = sh.num_params();
  float* bias_s = reinterpret_cast<float*>(sm + S::O_BIAS);   // b0[32] b1[32] b2[48]
  float* tp = reinterpret_cast<float*>(sm + S::O_TRUE);
  uint64_t* mbar_p = reinterpret_cast<uint64_t*>(sm + S::O_MISC);  // [slot]
  uint32_t* tmem_p = reinterpret_cast<uint32_t*>(sm + S::O_MISC + 64);

  // Every CTA owns a CONTIGUOUS range of tiles (a multiple of NS): its input stream walks one region of the point set
  // front to back (one new 2 MB page every ~170 tiles at d = 8 instead of every tile with a grid-strided assignment).
  // n_tiles is the END of this CTA's range.
  const uint32_t fpd = FPM ? (uint32_t)a.fp_dirs : 1u;                         // FP: d direction tiles per point tile
  const int64_t n_tiles_all = (a.n_points + 127) / 128 * fpd;                  // (virtual) tiles of this point set
  const int64_t per_cta = ((n_tiles_all + gridDim.x - 1) / gridDim.x + NS - 1) / NS * NS;
  const int64_t tile_begin = (int64_t)blockIdx.x * per_cta;
  if (tile_begin >= n_tiles_all) return;  // nothing to do for this CTA (uniform)
  const int64_t n_tiles = tile_begin + per_cta < n_tiles_all ? tile_begin + per_cta : n_tiles_all;

  // ---- one-time set-up: TMEM, mbarriers, zeroed operand tiles, split weights in core-matrix layout ------------
  if (warp == 0) {
    tmem_alloc(smem_u32(tmem_p), 512);
    tmem_relinquish();
  }
  if (tid == 0) {
    for (int s = 0; s < NS; ++s) mbar_init(smem_u32(mbar_p + s), 1);
    mbar_init(smem_u32(mbar_p + 4), 1);  // input staging (one-slot kernels)
    fence_mbar_init();
  }
  // every operand byte is finite from the start: zero-weight columns multiply whatever the neighbouring band holds
  for (uint32_t o = tid * 16; o < S::O_BIAS; o += kLaunchThreads * 16) *reinterpret_cast<uint4*>(sm + o) = make_uint4(0, 0, 0, 0);
  if constexpr (S::PIPE_X)
    for (uint32_t o = tid * 16; o < S::SZ_X; o += kLaunchThreads * 16) *reinterpret_cast<uint4*>(sm + S::O_X2 + o) = make_uint4(0, 0, 0, 0);
  __syncthreads();
  {
    const float* W0 = a.params + sh.w_off(0);
    const float* W1 = a.params + sh.w_off(1);
    const float* W2 = a.params + sh.w_off(2);
    auto put = [&](uint32_t o_hi, uint32_t o_lo, uint32_t rg, int r, int c, float w) {
      const __nv_bfloat16 hi = __float2bfloat16_rn(w);
      const __nv_bfloat16 lo = __float2bfloat16_rn(w - __bfloat162float(hi));
      const uint32_t off = chunk_off(r, c >> 3, rg) + (uint32_t)(c & 7) * 2u;
      *reinterpret_cast<__nv_bfloat16*>(sm + o_hi + off) = hi;
      *reinterpret_cast<__nv_bfloat16*>(sm + o_lo + off) = lo;
    };
    for (int idx = tid; idx < 32 * S::KX; idx += kLaunchThreads) {  // T0X[r = out][c] = W0[c mod DP][r]  ([W0; W0])
      const int r = idx / S::KX, c = idx % S::KX, ci = c % DP;
      put(S::O_T0XH, S::O_T0XL, S::RG_T0X, r, c, ci < d ? W0[ci * H + r] : 0.f);
    }
    for (int idx = tid; idx < 32 * S::KV; idx += kLaunchThreads) {  // T0V[r = out][c = in] = W0[c][r], columns >= d zero
      const int r = idx / S::KV, c = idx % S::KV;
      put(S::O_T0VH, S::O_T0VL, S::RG_T0V, r, c, c < d ? W0[c * H + r] : 0.f);
    }
    for (int idx = tid; idx < 32 * 32; idx += kLaunchThreads) {
      const int r = idx / 32, c = idx % 32;
      put(S::O_T1H, S::O_T1L, S::RG_T1, r, c, W1[c * H + r]);
    }
    for (int idx = tid; idx < OP * 32; idx += kLaunchThreads) {  // T2[r = out (48)][c = in] = W2[c][r], rows >= 40 zero
      const int r = idx / 32, c = idx % 32;
      put(S::O_T2H, S::O_T2L, S::RG_T2, r, c, r < kOut ? W2[c * kOut + r] : 0.f);
    }
    if constexpr (kGram) {  // TG[i][j] = (c_g / 8) sum_k W0[k][i] W0[k][j]  (k over the d inputs)
      const float sc = 0.125f / (float)fpd;
      for (int idx = tid; idx < 32 * 32; idx += kLaunchThreads) {
        const int r = idx / 32, c = idx % 32;
        float acc = 0.f;
        for (int k = 0; k < d; ++k) acc = fmaf(W0[k * H + r], W0[k * H + c], acc);
        put(S::O_TGH, S::O_TGL, S::RG_T1, r, c, sc * acc);
      }
    }
    for (int j = tid; j < 32; j += kLaunchThreads) {
      bias_s[j] = a.params[sh.b_off(0) + j];
      bias_s[32 + j] = a.params[sh.b_off(1) + j];
    }
    for (int j = tid; j < OP; j += kLaunchThreads) bias_s[64 + j] = j < kOut ? a.params[sh.b_off(2) + j] : 0.f;
    int ntg = 0;
    if (a.tg.kind == PDEIP_DRIFT_LINEAR) ntg = d * d;
    else if (a.tg.kind == PDEIP_DRIFT_GMM) ntg = a.tg.n_gaussian * d;
    for (int i = tid; i < ntg; i += kLaunchThreads) tp[i] = a.tg.params[i];
  }
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();

  const uint32_t TB = *tmem_p;
  const int64_t tile_stride = NS;

  // ==========================================================================================================
  // MMA warp: one lane issues every tcgen05.mma, phase by phase, slot by slot
  // ==========================================================================================================
  if (warp >= kEpiThreads / 32) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(Regs<NS>::kMma));
  }
  if (is_mma_warp) {
    // Descriptors are NOT kept in registers across the tile loop (18 weight views + 8 slot views would not fit the
    // budget left by setmaxnreg and were spilled: 75 LDL / STL in front of the MMAs of every phase, profiles/
    // r02_summary_residual.md): each phase re-derives the few it needs from the shared-memory base with one add each.
    const uint32_t sm16 = smem_u32(sm) >> 4;
    constexpr uint32_t CH = 128;  // bytes per chunk (8 operand columns)
    uint32_t dw_started = 0;      // becomes 1 after the first tile's P3..P5 background GEMMs
    // dW chains whose operands are final before the tail are issued where the tensor pipe idles (P6..P8: 1-2 MMAs per
    // phase) instead of in the tail P9..P11, which is bound by it: g^^T za0 behind P6's commit, and — two-slot kernel
    // only: with one slot a chain in front of the next layer GEMM is fully exposed (d = 32: -2.5 %) — c_1^T za1 behind
    // P7's and c_2^T za2 behind P8's.  d = 8: 2.98e9 -> 3.01e9 evals/s.
    constexpr bool kCChainsEarly = PDEIP_TC_G_CHAIN_EARLY && NS == 2;
    constexpr int kNloFwd = BND ? 2 : PDEIP_TC_NLO_FWD;  // BND: primal and order-1 streams get the lo halves
    constexpr int kNloBwd = BND ? 2 : PDEIP_TC_NLO_BWD;
    // NOTE: a compact switch over the phase (about 13 KB of code) measured FASTER than the fully written-out sequence
    // (26 KB): the epilogue warps are instruction-fetch sensitive and the larger MMA stream evicts their code.
    // The lo halves of the weights are skipped for the g-stream (P6..P8) and adjoint (P9, P10) GEMMs: their effect on
    // the result is below 1e-3 (tests/tensor_v2_model.py study), the forward and input-gradient GEMMs keep hi + lo.
    uint32_t xb = 0;  // PIPE_X: which x | v | g^ buffer holds the current tile
    uint32_t tsb = 0;  // two-stage hand-off: which of the two second-stage barriers is next
#pragma unroll 1
    for (int64_t base = tile_begin; base < n_tiles; base += tile_stride) {
#pragma unroll 1
      for (int ph = (kPipeFlow && base != tile_begin) ? 1 : 0; ph < 12; ++ph) {  // PIPE_X: P0 was issued with the previous P11
        if (kGram && ph == 6) continue;  // no P6: its GEMM rides in P5, its dW chain in P7
#pragma unroll 1
        for (int s = 0; s < NS; ++s) {
          const uint32_t w16 = opaque(sm16), b16 = opaque(sm16 + (uint32_t)s * (S::SLOT >> 4));
          // x | v | g^ bands of the current tile / of the next one (PIPE_X: two buffers; else both are the slot's own)
          const uint32_t x16 = kPipeX ? opaque(sm16 + (xb ? (S::O_X2 >> 4) : 0u)) : b16;
          const uint32_t x16n = kPipeX ? opaque(sm16 + (xb ? 0u : (S::O_X2 >> 4))) : b16;
          const uint32_t TBo = opaque(TB);
          const uint32_t TS = TBo + C_SLOT0 + (uint32_t)s * SLOT_COLS;
          const uint32_t mb = smem_u32(mbar_p + s);
          const uint32_t AOP = TBo + C_AOP;  // A-operand columns (kTS)
          // weights: K-major views (LBO = 128: next 8 columns, SBO = row-group bytes) and transposed views
          const Desc T0XHK = mk_desc16(w16, S::O_T0XH, 128, S::RG_T0X), T0XLK = mk_desc16(w16, S::O_T0XL, 128, S::RG_T0X);
          const Desc T0VHK = mk_desc16(w16, S::O_T0VH, 128, S::RG_T0V), T0VLK = mk_desc16(w16, S::O_T0VL, 128, S::RG_T0V);
          const Desc T1HK = mk_desc16(w16, S::O_T1H, 128, S::RG_T1), T1LK = mk_desc16(w16, S::O_T1L, 128, S::RG_T1);
          const Desc T2HK = mk_desc16(w16, S::O_T2H, 128, S::RG_T2), T2LK = mk_desc16(w16, S::O_T2L, 128, S::RG_T2);
          const Desc TGHK = mk_desc16(w16, S::O_TGH, 128, S::RG_T1), TGLK = mk_desc16(w16, S::O_TGL, 128, S::RG_T1);
          const Desc T0VHM = mk_desc16(w16, S::O_T0VH, S::RG_T0V, 128), T0VLM = mk_desc16(w16, S::O_T0VL, S::RG_T0V, 128);
          const Desc T1HM = mk_desc16(w16, S::O_T1H, S::RG_T1, 128), T1LM = mk_desc16(w16, S::O_T1L, S::RG_T1, 128);
          const Desc T2HM = mk_desc16(w16, S::O_T2H, S::RG_T2, 128), T2LM = mk_desc16(w16, S::O_T2L, S::RG_T2, 128);
          const Desc XK = mk_desc16(x16, S::O_X, 128, S::RG_X), A1K = mk_desc16(b16, S::O_A1, 128, S::RG_A),
                     A2K = mk_desc16(b16, S::O_A2, 128, S::RG_A), ZK = mk_desc16(b16, S::O_Z, 128, S::RG_Z);
          const Desc XM = mk_desc16(x16, S::O_X, S::RG_X, 128), ZM = mk_desc16(b16, S::O_Z, S::RG_Z, 128);
          const uint32_t AOPX = kPipeX ? TBo + C_AOPX : AOP;  // A operands of P0
          // P0: z0 = [x_hi | x_lo] [W0; W0],  z1_0 = v W0   (xk: K-major view of the tile's x | v bands)
          auto issue_p0 = [&](const Desc xk) {
            if constexpr (kTS) {
              mm_fwd_ts<S::KX, 32, 1>({TS + C_Z0}, {AOPX}, T0XHK, T0XLK);
              mm_fwd_ts<S::KV, 32, 1, (PDEIP_TC_NLO_FWD >= 2 || BND)>({TS + C_Z10}, {AOPX + S::KX / 2}, T0VHK, T0VLK);
            } else {
              mm_fwd<S::KX, 32, 1>({TS + C_Z0}, xk, {S::XC_HI * CH}, T0XHK, T0XLK);
              mm_fwd<S::KV, 32, 1, (PDEIP_TC_NLO_FWD >= 2 || BND)>({TS + C_Z10}, xk, {S::XC_V * CH}, T0VHK, T0VLK);  // tangent stream
            }
          };
          TC_TRACE_DECL_MMA;
          mma_wait_operands<NS>(s);
          if (elect_one()) {
            TC_TRACE(4);
            switch (ph) {
              case 0: {
                issue_p0(XK);
                commit(mb);
              } break;
              case 1: {  // z1, z1_1, z2^_1
                if constexpr (kTS) mm_fwd_ts<32, 32, 3, PDEIP_TC_LO_FWD, kNloFwd>({TS + C_Z1, TS + C_Z11, TS + C_Z21}, {AOP + 4 * AC_T, AOP + 4 * AC_A1, AOP + 4 * AC_C}, T1HK, T1LK);
                else mm_fwd<32, 32, 3, PDEIP_TC_LO_FWD, kNloFwd>({TS + C_Z1, TS + C_Z11, TS + C_Z21}, A1K, {AC_T * CH, AC_A1 * CH, AC_C * CH}, T1HK, T1LK);
                commit(mb);
              } break;
              case 2: {  // u, u1, u2^
                if constexpr (kTS) mm_fwd_ts<32, OP, 3, PDEIP_TC_LO_FWD, kNloFwd>({TS + C_U, TS + C_U1, TS + C_U2}, {AOP + 4 * AC_T, AOP + 4 * AC_A1, AOP + 4 * AC_C}, T2HK, T2LK);
                else mm_fwd<32, OP, 3, PDEIP_TC_LO_FWD, kNloFwd>({TS + C_U, TS + C_U1, TS + C_U2}, A2K, {AC_T * CH, AC_A1 * CH, AC_C * CH}, T2HK, T2LK);
                commit(mb);
              } break;
              case 3: {  // aa2 = za2 W2^T, ab1_2 = s1v W2^T;  dW2 += a1_2^T s1v
                if constexpr (kTS) mm_bwd_ts<OP, 32, 2, true, kNloBwd>({TS + C_AA2, TS + C_AB12}, {AOP, AOP + 24}, T2HM, T2LM, S::RG_T2);
                else mm_bwd<OP, 32, 2, true, kNloBwd>({TS + C_AA2, TS + C_AB12}, ZK, {ZC_ZA2 * CH, ZC_TA * CH}, T2HM, T2LM, S::RG_T2);
                commit(mb);
              } break;
              case 4: {  // aa1 = za1 W1^T, ab1_1 = zbar1' W1^T;  dW1 += a1_1^T zbar1'
                if constexpr (kTS) mm_bwd_ts<32, 32, 2, true, kNloBwd>({TS + C_AA1, TS + C_AB11}, {AOP, AOP + 16}, T1HM, T1LM, S::RG_T1);
                else mm_bwd<32, 32, 2, true, kNloBwd>({TS + C_AA1, TS + C_AB11}, ZK, {ZC_ZA1 * CH, ZC_TB * CH}, T1HM, T1LM, S::RG_T1);
                commit(mb);
              } break;
              case 5: {  // g = za0 W0^T;  dW0 += v^T zbar1''
                if constexpr (kTS) mm_bwd_ts<32, S::KV, 1>({TS + C_G}, {AOP}, T0VHM, T0VLM, S::RG_T0V);
                else mm_bwd<32, S::KV, 1>({TS + C_G}, ZK, {ZC_ZA0 * CH}, T0VHM, T0VLM, S::RG_T0V);
                if constexpr (kGram) {  // zg^_0 (the same A operand as the g GEMM)
                  if constexpr (kTS) mm_fwd_ts<32, 32, 1, true>({TS + C_ZG0}, {AOP}, TGHK, TGLK);
                  else mm_fwd<32, 32, 1, true>({TS + C_ZG0}, ZK, {ZC_ZA0 * CH}, TGHK, TGLK);
                }
                commit(mb);
              } break;
              case 6: {  // zg^_0 = g^ W0
                if constexpr (kTS) mm_fwd_ts<S::KV, 32, 1, false>({TS + C_ZG0}, {AOP}, T0VHK, T0VLK);
                else mm_fwd<S::KV, 32, 1, false>({TS + C_ZG0}, XK, {S::XC_G * CH}, T0VHK, T0VLK);
                commit(mb);
#if PDEIP_TC_G_CHAIN_EARLY
                // dW0 += g^^T za0: both operands are final since E6 / E5, and the tensor pipe idles through P6..P8 (1-2
                // MMAs per phase) while the tail P9..P11 is bound by it: issued here, behind this slot's commit
                mm_outer<32>(TBo + C_DW0, XM, S::XC_G * CH, S::RG_X, ZM, ZC_ZA0 * CH, S::RG_Z, 1u);
#endif
              } break;
              case 7: {  // zg^_1 = ag^_1 W1  (operand in the a1 band)
                if constexpr (kTS) mm_fwd_ts<32, 32, 1, false>({TS + C_ZG1}, {AOP}, T1HK, T1LK);
                else mm_fwd<32, 32, 1, false>({TS + C_ZG1}, A1K, {AC_A1 * CH}, T1HK, T1LK);
                commit(mb);
                if constexpr (kGram && !kTwoStage)  // dW0 += g^^T za0 (P6's chain; g^ was written in E6, ordered by E7's arrive)
                  mm_outer<32>(TBo + C_DW0, XM, S::XC_G * CH, S::RG_X, ZM, ZC_ZA0 * CH, S::RG_Z, 1u);
                if constexpr (kCChainsEarly) {  // dW1 += c_1^T za1: c_1 is final since E7 (just arrived), za1 since E4
                  const Desc A1M = mk_desc16(b16, S::O_A1, S::RG_A, 128);
                  mm_outer<32>(TBo + C_DW1, A1M, AC_C * CH, S::RG_A, ZM, ZC_ZA1 * CH, S::RG_Z, 1u);
                }
              } break;
              case 8: {  // ug^ = ag^_2 W2
                if constexpr (kTS) mm_fwd_ts<32, OP, 1, false>({TS + C_UG}, {AOP}, T2HK, T2LK);
                else mm_fwd<32, OP, 1, false>({TS + C_UG}, A2K, {AC_A1 * CH}, T2HK, T2LK);
                commit(mb);
                if constexpr (kCChainsEarly) {  // dW2 += c_2^T za2: c_2 is final since E8 (just arrived), za2 since E3
                  const Desc A2M = mk_desc16(b16, S::O_A2, S::RG_A, 128);
                  mm_outer<OP>(TBo + C_DW2, A2M, AC_C * CH, S::RG_A, ZM, ZC_ZA2 * CH, S::RG_Z, 1u);
                }
              } break;
              case 9: {  // ab_2 = s0 W2^T, aa2 again;  dW2 += t2^T s0 + c_2^T za2
                if constexpr (kTS) {  // s0 from TMEM; za2 (written in E3) only exists in shared memory by now
                  mm_bwd_ts<OP, 32, 1, BND, 1>({TS + C_AB2}, {AOP}, T2HM, T2LM, S::RG_T2);
                  mm_bwd<OP, 32, 1, false>({TS + C_AA2R}, ZK, {ZC_ZA2 * CH}, T2HM, T2LM, S::RG_T2);
                } else {
                  mm_bwd<OP, 32, 2, BND, 1>({TS + C_AB2, TS + C_AA2R}, ZK, {ZC_TA * CH, ZC_ZA2 * CH}, T2HM, T2LM, S::RG_T2);
                }
                commit(mb);
              } break;
              case 10: {  // ab_1 = zbar0' W1^T, aa1 again;  dW1 += t1^T zbar0' + c_1^T za1
                if constexpr (kTS) {
                  mm_bwd_ts<32, 32, 1, BND, 1>({TS + C_AB1}, {AOP}, T1HM, T1LM, S::RG_T1);
                  mm_bwd<32, 32, 1, false>({TS + C_AA1R}, ZK, {ZC_ZA1 * CH}, T1HM, T1LM, S::RG_T1);
                } else {
                  mm_bwd<32, 32, 2, BND, 1>({TS + C_AB1, TS + C_AA1R}, ZK, {ZC_TB * CH, ZC_ZA1 * CH}, T1HM, T1LM, S::RG_T1);
                }
                commit(mb);
              } break;
              default: {  // dW0 += x_hi^T zbar0'' (+ x_lo^T zbar0'' if PDEIP_TC_XLO_DW) + g^^T za0
                const bool p0_next = kPipeFlow && base + tile_stride < n_tiles;
                if (p0_next) {  // PIPE_X: the next tile's x | v bands were written behind E10: its P0 goes first, the dW0
                                // chain of this tile follows in the background (covered by the next commit)
                  issue_p0(mk_desc16(x16n, S::O_X, 128, S::RG_X));
                  commit(mb);
                }
                if constexpr (!kTwoStage) {  // (two-stage hand-off: the chain is issued behind the second barrier, below)
                  mm_outer<32>(TBo + C_DW0, XM, S::XC_HI * CH, S::RG_X, ZM, ZC_TA * CH, S::RG_Z, 1u);
#ifdef PDEIP_TC_XLO_DW  // measured: +2 % time, no visible effect on the gradient error (x_lo = x - bf16(x) averages out)
                  mm_outer<32>(TBo + C_DW0, XM, S::XC_LO * CH, S::RG_X, ZM, ZC_TA * CH, S::RG_Z, 1u);
#endif
#if !PDEIP_TC_G_CHAIN_EARLY
                  mm_outer<32>(TBo + C_DW0, XM, S::XC_G * CH, S::RG_X, ZM, ZC_ZA0 * CH, S::RG_Z, 1u);
#endif
                  if (!p0_next) commit(mb);  // the next tile's E0 overwrites the x | v bands (PIPE_X: last tile, for the drain)
                }
              } break;
            }
            TC_TRACE(6);
          }
          __syncwarp();
        }
        // background (batch-reduced dW) GEMMs of this phase, issued after the fast GEMMs of BOTH slots so that the
        // second slot's fast GEMMs do not queue behind the first slot's dW chains (the tensor pipe runs in issue order)
        if (ph == 3 || ph == 4 || ph == 5 || ph == 9 || ph == 10 || (kTwoStage && (ph == 7 || ph == 11))) {
#pragma unroll 1
          for (int s = 0; s < NS; ++s) {
            if constexpr (kTwoStage) {  // second stage of the hand-off: the activation bands are visible to the async proxy.
              // TWO named barriers (4, 5) used alternately: the epilogue's next second-stage arrive follows its wait for
              // this phase's commit, which is issued BEFORE this barrier — with a single barrier a slow MMA warp could
              // be overtaken (two generations of arrivals on one barrier: a deadlock seen once in ~1e4 launches).  With
              // two, the arrive after next needs the commit of the next phase, which this warp issues behind this sync.
              asm volatile("bar.sync %0, %1;" ::"r"(4 + (int)tsb), "n"(kThreads) : "memory");
              tsb ^= 1u;
              fence_after_sync();
            }
            const uint32_t b16 = opaque(sm16 + (uint32_t)s * (S::SLOT >> 4)), TBo = opaque(TB);
            const uint32_t x16 = kPipeX ? opaque(sm16 + (xb ? (S::O_X2 >> 4) : 0u)) : b16;
            const Desc XM = mk_desc16(x16, S::O_X, S::RG_X, 128), A1M = mk_desc16(b16, S::O_A1, S::RG_A, 128),
                       A2M = mk_desc16(b16, S::O_A2, S::RG_A, 128), ZM = mk_desc16(b16, S::O_Z, S::RG_Z, 128);
            const uint32_t acc_first = (dw_started | (uint32_t)s) ? 1u : 0u;
            if (elect_one()) {
              switch (ph) {
                case 3:  // dW2 += a1_2^T s1v
                  mm_outer<OP>(TBo + C_DW2, A2M, AC_A1 * CH, S::RG_A, ZM, ZC_TA * CH, S::RG_Z, acc_first);
                  break;
                case 4:  // dW1 += a1_1^T zbar1'
                  mm_outer<32>(TBo + C_DW1, A1M, AC_A1 * CH, S::RG_A, ZM, ZC_TB * CH, S::RG_Z, acc_first);
                  break;
                case 5:  // dW0 += v^T zbar1''
                  mm_outer<32>(TBo + C_DW0, XM, S::XC_V * CH, S::RG_X, ZM, ZC_TA * CH, S::RG_Z, acc_first);
                  break;
                case 9:  // dW2 += t2^T s0 + c_2^T za2
                  mm_outer<OP>(TBo + C_DW2, A2M, AC_T * CH, S::RG_A, ZM, ZC_TA * CH, S::RG_Z, 1u);
                  if constexpr (!kCChainsEarly)
                    mm_outer<OP>(TBo + C_DW2, A2M, AC_C * CH, S::RG_A, ZM, ZC_ZA2 * CH, S::RG_Z, 1u);
                  break;
                case 10:  // dW1 += t1^T zbar0' + c_1^T za1
                  mm_outer<32>(TBo + C_DW1, A1M, AC_T * CH, S::RG_A, ZM, ZC_TB * CH, S::RG_Z, 1u);
                  if constexpr (!kCChainsEarly)
                    mm_outer<32>(TBo + C_DW1, A1M, AC_C * CH, S::RG_A, ZM, ZC_ZA1 * CH, S::RG_Z, 1u);
                  break;
                case 7:  // (two-stage hand-off) dW0 += g^^T za0: P6's chain, g^ written in E6 and fenced in E7
                  if constexpr (kGram) mm_outer<32>(TBo + C_DW0, XM, S::XC_G * CH, S::RG_X, ZM, ZC_ZA0 * CH, S::RG_Z, 1u);
                  break;
                default: {  // (two-stage hand-off) P11: dW0 += x_hi^T zbar0''; the drain's commit on the last tile
                  mm_outer<32>(TBo + C_DW0, XM, S::XC_HI * CH, S::RG_X, ZM, ZC_TA * CH, S::RG_Z, 1u);
#ifdef PDEIP_TC_XLO_DW
                  mm_outer<32>(TBo + C_DW0, XM, S::XC_LO * CH, S::RG_X, ZM, ZC_TA * CH, S::RG_Z, 1u);
#endif
#if !PDEIP_TC_G_CHAIN_EARLY
                  mm_outer<32>(TBo + C_DW0, XM, S::XC_G * CH, S::RG_X, ZM, ZC_ZA0 * CH, S::RG_Z, 1u);
#endif
                  if (!(kPipeFlow && base + tile_stride < n_tiles)) commit(smem_u32(mbar_p + s));
                } break;
              }
            }
            __syncwarp();
          }
        }
      }
      dw_started = 1u;
      xb ^= 1u;
    }
  } else if (warp < kEpiThreads / 32) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(Regs<NS>::kEpi));
    // ========================================================================================================
    // epilogue warps
    // ========================================================================================================
    bool ok = true;
    uint32_t par = 0;  // bit s = parity of slot s's mbarrier
#ifdef PDEIP_TC_PROBE
    float* probe = reinterpret_cast<float*>(status) + 2048;
#endif
    const OutCols<NP> oc{part};
    constexpr int UO = OutCols<NP>::NU;  // output units per thread
    // bias-gradient sums over this thread's row: hidden units [UH part, +UH), output units of oc.  The two-slot kernel
    // keeps them in registers.  One-slot kernels keep them in TMEM (C_DB; 104 registers per thread do not hold them next
    // to the phase temporaries): E9, E10 and E11 load them with their other TMEM reads in front of the GEMM wait and store
    // them with the operand stores that their hand-off waits for anyway.
    constexpr bool kDbTmem = NS == 1;
    static_assert(!kDbTmem || (UH == 8 && UO == 10), "C_DB map: 8 + 8 + 10 columns per part");
    const uint32_t LDB = TB + ((uint32_t)(q * 32) << 16) + C_DB;
    const uint32_t cdb0 = LDB + 8 * part, cdb1 = LDB + 32 + 8 * part, cdb2 = LDB + 64 + 8 * part, cdb2p = LDB + 96 + 2 * part;
    auto db_ld = [&](uint32_t col, float* v) { tm_ld8(col, reinterpret_cast<uint32_t*>(v)); };
    auto db_st = [&](uint32_t col, const float* v) { tm_st8(col, reinterpret_cast<const uint32_t*>(v)); };
    auto db2_ld = [&](float* v) { db_ld(cdb2, v); tm_ld2(cdb2p, reinterpret_cast<uint32_t*>(v + 8)); };
    auto db2_st = [&](const float* v) { db_st(cdb2, v); tm_st2(cdb2p, reinterpret_cast<const uint32_t*>(v + 8)); };
    float db0[UH], db1[UH], db2[UO];
#pragma unroll
    for (int i = 0; i < UH; ++i) { db0[i] = 0.f; db1[i] = 0.f; }
#pragma unroll
    for (int i = 0; i < UO; ++i) db2[i] = 0.f;
    if constexpr (kDbTmem) {
      db_st(cdb0, db0);
      db_st(cdb1, db1);
      db2_st(db2);
      tm_wait_st();
    }
    // loss sums of this thread's row: registers in the two-slot kernel; one-slot kernels keep them in shared memory
    // (S::O_SUMS, [k][thread]), read and written once per tile by E3 (d1, d2) and E6 (g2, gt2, gd2), as the db sums
    constexpr bool kSumsSmem = NS == 1;
    float* const sums_s = reinterpret_cast<float*>(sm + S::O_SUMS) + tid;
    float sum_g2 = 0.f, sum_gt2 = 0.f, sum_gd2 = 0.f, sum_d1 = 0.f, sum_d2 = 0.f;
    if constexpr (kSumsSmem)
      for (int k = 0; k < 5; ++k) sums_s[k * kEpiThreads] = 0.f;
    const float gamma = a.coef, gamma4 = 4.f * a.coef;
    const float cgw = 1.f / (float)fpd;  // coefficient of the |g|^2 term per row (FP: 1/d per direction row; else 1)
    const int dimw = (FPM ? d : 2 * d) + (a.tg.kind == PDEIP_DRIFT_IN_POINTS ? d : 0);  // floats per point
    // byte offsets of this thread's row inside the operand tiles (chunk c adds c * 128)
    const uint32_t offX = (uint32_t)(row & 7) * 16u + (uint32_t)(row >> 3) * S::RG_X;
    const uint32_t offA = (uint32_t)(row & 7) * 16u + (uint32_t)(row >> 3) * S::RG_A;
    const uint32_t offZ = (uint32_t)(row & 7) * 16u + (uint32_t)(row >> 3) * S::RG_Z;
    const uint32_t LA0 = TB + ((uint32_t)(q * 32) << 16) + C_SLOT0;
    const uint32_t LOP = TB + ((uint32_t)(q * 32) << 16) + C_AOP;  // this thread's lane of the A-operand columns (kTS)
    const int uh = UH * part;  // first hidden unit owned
    // prefetched input chunks: item j = part + NP i;  j in [0, XC): x chunk j;  [XC, 2 XC): v;  [2 XC, 3 XC): stored gt
    constexpr int NI = (3 * S::XC + NP - 1) / NP;
    float xin0[NI][8], xin1[NI][8];
    // BLOCK128 point sets with d == DP (the pipeline's layout and the benchmark widths): the tile is one block of
    // [dimw][128] floats, so every component of this thread's row sits at a COMPILE-TIME offset from one base pointer:
    // 48 loads with immediate offsets at d = 32 instead of ~12 instructions of 64-bit index arithmetic per load (the
    // generic path below: 560 instructions and ~2.3 k cycles per tile in the phase trace).
    const bool fast_in = !FPM && a.layout == PDEIP_LAYOUT_BLOCK128 && d == DP;
    // items of the bands in `bands` (bit 0 x, bit 1 v, bit 2 stored gt)
    auto load_into = [&](float (&xin)[NI][8], int64_t t, const int bands = 7) {
      if (fast_in) {
        const int64_t pp = t * 128 + row;
        const bool inside = t < n_tiles && pp < a.n_points;
        // item j = part + NP i holds components [8 j, 8 j + 8) of the row (band j / XC, chunk j % XC, DP = 8 XC): the
        // runtime part goes into the base pointer, the rest is an immediate
        const float* const pb = a.points + (inside ? t * (int64_t)(128 * dimw) + row : (int64_t)0) + part * (8 * 128);
        const bool has_gt = a.tg.kind == PDEIP_DRIFT_IN_POINTS;
#pragma unroll
        for (int i = 0; i < NI; ++i) {
          if (part + NP * i >= 3 * S::XC) continue;       // (d = 8: the fourth item does not exist)
          if (!((bands >> ((part + NP * i) / S::XC)) & 1)) continue;
          if (part + NP * i >= 2 * S::XC && !has_gt) continue;  // stored true gradient: only if the rows carry it
#pragma unroll
          for (int e = 0; e < 8; ++e) xin[i][e] = __ldg(pb + (8 * NP * i + e) * 128);
        }
        return;
      }
      const int64_t cstride = comp_stride(a.layout, a.n_points);
      // FP: virtual tile -> (point tile, direction); tile counts stay below 2^31
      const uint32_t tq = FPM ? (uint32_t)t / fpd : 0u;
      const int dir = FPM ? (int)((uint32_t)t - tq * fpd) : -1;
      const int64_t pp = (FPM ? (int64_t)tq : t) * 128 + row;
      const int64_t pc = (t < n_tiles && pp < a.n_points) ? pp : 0;
      const float* const pbase = a.points + point_base(a.layout, pc, dimw);
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const int j = part + NP * i;
        if (j < 3 * S::XC && !((bands >> (j / S::XC)) & 1)) continue;
        const int band = (j / S::XC) < 3 ? (j / S::XC) : 0, cg = j % S::XC;
        const int bandc = (band < 2 || a.tg.kind == PDEIP_DRIFT_IN_POINTS) ? band : 0;
        // FP rows hold [x (d), grad V_true (d, IN_POINTS)]: the gt band sits right after x, the v band is e_dir
        const int bandm = FPM ? (bandc == 2 ? 1 : 0) : bandc;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int u = cg * 8 + e;
          const int uc = u < d ? u : 0;
          const float val = __ldg(pbase + (bandm * d + uc) * cstride);
          xin[i][e] = (FPM && band == 1) ? (u == dir ? 1.f : 0.f) : val;
        }
      }
    };
    // input staging by the TMA unit (one-slot kernels, BLOCK128 point sets: a tile is one contiguous block)
    constexpr bool kStage = PDEIP_TC_STAGE && NS == 1;
    const bool use_stage = kStage && a.layout == PDEIP_LAYOUT_BLOCK128 && (reinterpret_cast<uintptr_t>(a.points) & 15u) == 0;
    const float* const stage = reinterpret_cast<const float*>(sm + S::O_STAGE) + row;  // component c of this row: [c * 128]
    const uint32_t stage_mbar = smem_u32(mbar_p + 4);
    uint32_t spar = 0;
    auto stage_issue = [&](int64_t t) {  // called by ONE thread, after every warp has finished reading the buffer
      if (t >= n_tiles) return;
      const int64_t pt = FPM ? (int64_t)((uint32_t)t / fpd) : t;
      const uint32_t bytes = 512u * (uint32_t)dimw;
      mbar_expect_tx(stage_mbar, bytes);
      bulk_g2s(smem_u32(sm + S::O_STAGE), a.points + pt * 128 * dimw, bytes, stage_mbar);
    };
    if (use_stage && tid == 0) stage_issue(tile_begin);
    // two separate branches: each slot's loads target its own registers directly (no select on the loaded value)
    auto load_inputs = [&](int s, int64_t t, const int bands = 7) {
      if (NS == 2 && s == 1) load_into(xin1, t, bands);
      else load_into(xin0, t, bands);
    };
#ifndef PDEIP_TC_L2_PREFETCH
#define PDEIP_TC_L2_PREFETCH 1
#endif
    // Input staging.  A register prefetch issued one tile ahead (in E10) shares a scoreboard with the phase's own
    // LDS / TMEM loads, so the first wait after it sits out the full DRAM latency (~1.4 k cycles per slot and tile in the
    // phase trace).  Instead E10 only asks the TMA unit to pull the next tile into L2 (cp.async.bulk.prefetch.L2: no
    // destination register, nothing to wait for; prefetch.global.L2 = CCTL.PF2 measured ~700 cycles per phase) and E0
    // issues the loads itself, before its commit wait: they hit L2 and land behind that wait.
    auto prefetch_inputs = [&](int64_t t) {
      if (FPM || t >= n_tiles || (t + 1) * 128 > a.n_points) return;  // FP tiles / ragged last tile: not worth a special case
      if (a.layout == PDEIP_LAYOUT_SOA) {  // dimw component segments of 512 B
        if ((a.n_points & 3) == 0 && part == 0 && row < dimw)
          asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a.points + (int64_t)row * a.n_points + t * 128),
                       "r"(512u)
                       : "memory");
      } else if (part == 0 && row == 0) {  // AOS and BLOCK128: the tile is one contiguous block of 128 x dimw floats
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a.points + t * 128 * dimw),
                     "r"((uint32_t)(512 * dimw))
                     : "memory");
      }
    };
#if !PDEIP_TC_L2_PREFETCH
    load_inputs(0, tile_begin);
    if constexpr (NS == 2) load_inputs(1, tile_begin + 1);
#endif

    bool first = true;
    int64_t base = tile_begin;
    uint32_t xb = 0;  // PIPE_X: which x | v | g^ buffer holds the current tile
    uint32_t tsb = 0;  // two-stage hand-off: which of the two second-stage barriers is next
    const uint32_t LOPX = kPipeX ? TB + ((uint32_t)(q * 32) << 16) + C_AOPX : LOP;  // this thread's lane of P0's A-operand columns
    // E0: x (hi + lo) and v bands of a tile from its prefetched inputs (Xd: this thread's row of the destination buffer)
    auto emit_x = [&](const float (&xin)[NI][8], const bool valid_t, uint8_t* const Xd) {
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const int j = part + NP * i;
        const int band = j / S::XC, cg = j % S::XC;
        if (band == 0) {
          float hi[8], lo[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float xv = (valid_t && cg * 8 + e < d) ? xin[i][e] : 0.f;
            hi[e] = __bfloat162float(__float2bfloat16_rn(xv));
            lo[e] = xv - hi[e];
          }
          put_op<kTS>(Xd, (S::XC_HI + cg) * 128, LOPX + 4 * cg, hi);
          put_op<kTS>(Xd, (S::XC_LO + cg) * 128, LOPX + 4 * (S::XC + cg), lo);
        } else if (band == 1) {
          float vv[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) vv[e] = (valid_t && cg * 8 + e < d) ? xin[i][e] : 0.f;
          put_op<kTS>(Xd, (S::XC_V + cg) * 128, LOPX + S::KX / 2 + 4 * cg, vv);
        }
      }
    };

    // one epilogue phase of one slot: wait for the previous GEMM phase of that slot, compute, signal the MMA warp
    // The phase bodies are shared by the two slots (runtime slot offsets): E_k(slot 0) and E_k(slot 1) run back to
    // back on the same ~20 KB of instructions, so the second pass is served by the instruction cache.
    auto phase = [&](auto PHc, const int s) {
      constexpr int ph = decltype(PHc)::value;
      uint8_t* const X = sm + (kPipeX ? (xb ? S::O_X2 : 0u) : (uint32_t)s * S::SLOT) + S::O_X + offX;
      uint8_t* const A1 = sm + (uint32_t)s * S::SLOT + S::O_A1 + offA;
      uint8_t* const A2 = sm + (uint32_t)s * S::SLOT + S::O_A2 + offA;
      uint8_t* const Z = sm + (uint32_t)s * S::SLOT + S::O_Z + offZ;
      const uint32_t LA = LA0 + (uint32_t)s * SLOT_COLS;
      const int64_t tile = base + s;
      const int64_t p = (FPM ? (int64_t)((uint32_t)tile / fpd) : tile) * 128 + row;  // point of this thread's row
      const bool valid = tile < n_tiles && p < a.n_points;
      const float mk = valid ? 1.f : 0.f;
#ifdef PDEIP_TC_PROBE
      const bool probe_on = blockIdx.x == 0 && tile == 0;
#endif
#ifdef PDEIP_TC_TRACE
      long long* trace = reinterpret_cast<long long*>(status) + 512;
      const bool trace_on = blockIdx.x == 0 && tid == 0 && base >= tile_begin + (int64_t)16 * tile_stride &&
                            base < tile_begin + (int64_t)(16 + kTraceTiles) * tile_stride;
#endif
      // wait for the GEMMs of the previous phase of this slot (P11 of the previous tile before E0).  Phases that also
      // read operands which do not come from those GEMMs (own bf16 chunks in shared memory, parked TMEM values) issue
      // and unpack them BEFORE this wait, so that the hand-off latency is spent on useful work.
      auto wait_gemm = [&]() {
        TC_TRACE(0);
        if (!(ph == 0 && first)) {
          if (ok && !mbar_wait(smem_u32(mbar_p + s), (par >> s) & 1u)) {
            ok = false;
            atomicExch(status, 1);
          }
          par ^= 1u << s;
          TC_TRACE(3);
          fence_after_sync();
        }
        TC_TRACE(1);
      };
      constexpr bool kEarlyLoads = true;  // (at d = 32 this used to spill; the shorter life of the input registers fixed that)
#if PDEIP_TC_L2_PREFETCH
      if constexpr (ph == 0) {
        if (!use_stage) load_inputs(s, tile, kPipeFlow ? 3 : 7);  // (PIPE_X: first tile only; stored gt below)
      }
      // PIPE_X: this tile's stored true gradient (an L2 hit since the prefetch in E4 one tile ago) for E6, read in front
      // of E5's GEMM wait.  Read in E10 with x and v, its 8 registers would live across six phases and spill at d = 32.
      if constexpr (kPipeFlow && ph == 5) {
        if (a.tg.kind == PDEIP_DRIFT_IN_POINTS) load_inputs(s, tile, 4);
      }
#endif
      if constexpr (kStage && ph == 0) {
        if (use_stage) {  // this tile's block has landed in shared memory (bulk copy issued one tile ago, in E7): the
                          // row is read before the wait for P11, like the global loads of the other layouts
          if (ok && !mbar_wait(stage_mbar, spar)) {
            ok = false;
            atomicExch(status, 1);
          }
          spar ^= 1u;
          const int dir = FPM ? (int)((uint32_t)tile % fpd) : -1;
#pragma unroll
          for (int i = 0; i < NI; ++i) {
            const int j = part + NP * i;
            const int band = (j / S::XC) < 3 ? (j / S::XC) : 0, cg = j % S::XC;
            if (band < 2) {
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int u = cg * 8 + e;
                const float val = stage[(band * d + (u < d ? u : 0)) * 128];
                xin0[i][e] = (FPM && band == 1) ? (u == dir ? 1.f : 0.f) : val;
              }
            }
          }
        }
      }
      if constexpr (ph <= 3 || ph == 6 || !kEarlyLoads) wait_gemm();
      if constexpr (ph == 0) {  // E0: x (hi + lo) and v bands of this tile
        if (NS == 2 && s == 1) emit_x(xin1, valid, X);
        else emit_x(xin0, valid, X);
      } else if constexpr (ph == 1 || ph == 2) {
        // E1: t1, a1_1 = s1 z1, a2^_1 = t a1 z1      E2: t2, a1_2, a2^_2 = s1 z2^ + t a1 z1     (a2^ = -a2 / 2)
        constexpr bool l1 = ph == 1;
        uint8_t* const At = l1 ? A1 : A2;
        float z0[UH], z1[UH], z2[UH];
        tm_ldf<UH>(LA + (l1 ? C_Z0 : C_Z1) + uh, z0);
        tm_ldf<UH>(LA + (l1 ? C_Z10 : C_Z11) + uh, z1);
        if constexpr (!l1) tm_ldf<UH>(LA + C_Z21 + uh, z2);
        float bb[UH];
#pragma unroll
        for (int i = 0; i < UH / 4; ++i)
          *reinterpret_cast<float4*>(bb + 4 * i) = *reinterpret_cast<const float4*>(bias_s + (l1 ? 0 : 32) + uh + 4 * i);
        tm_wait_ld();
        float t[UH], s1[UH], q1[UH], q2[UH];
#if PDEIP_TC_PACKED
#pragma unroll
        for (int i = 0; i < UH / 2; ++i) {
          const float2 zb = __fadd2_rn(pr(z0, i), pr(bb, i));
          const float2 t2 = make_float2(tanh_fast(zb.x), tanh_fast(zb.y));
          const float2 s2 = __ffma2_rn(__fmul2_rn(t2, bc2(-1.f)), t2, bc2(1.f));
          const float2 z12 = pr(z1, i);
          const float2 q = __fmul2_rn(s2, z12);
          float2 r = __fmul2_rn(__fmul2_rn(t2, q), z12);
          if constexpr (!l1) r = __ffma2_rn(s2, pr(z2, i), r);
          st2(t, i, t2); st2(s1, i, s2); st2(q1, i, q); st2(q2, i, r);
        }
#else
#pragma unroll
        for (int i = 0; i < UH; ++i) {
          t[i] = tanh_fast(z0[i] + bb[i]);
          s1[i] = fmaf(-t[i], t[i], 1.f);
          q1[i] = s1[i] * z1[i];
          const float w = t[i] * q1[i];
          q2[i] = l1 ? w * z1[i] : fmaf(s1[i], z2[i], w * z1[i]);
        }
#endif
#pragma unroll
        for (int c = 0; c < HC; ++c) {
          put_op<kTS>(At, (AC_T + HC * part + c) * 128, LOP + 4 * (AC_T + HC * part + c), t + 8 * c);
          put_op<kTS>(At, (AC_A1 + HC * part + c) * 128, LOP + 4 * (AC_A1 + HC * part + c), q1 + 8 * c);
          put_op<kTS>(At, (AC_C + HC * part + c) * 128, LOP + 4 * (AC_C + HC * part + c), q2 + 8 * c);
        }
        tm_park<UH>(LA + (l1 ? C_S1P1 : C_S1P2) + UH / 2 * part, s1);
        TC_PROBE(l1 ? 0 : 3, uh, t, UH);
        TC_PROBE(l1 ? 1 : 4, uh, q1, UH);
        TC_PROBE(l1 ? 2 : 5, uh, q2, UH);
      } else if constexpr (ph == 3) {
        // E3: za^2 = 8 u, s1v = -8 u1 + 4 gamma u, s0p = 8 u2^ + 4 gamma u1, D_v V, D_v^2 V
        float u[UO], u1[UO], u2[UO];
        oc.ldf(LA + C_U, u);
        oc.ldf(LA + C_U1, u1);
        oc.ldf(LA + C_U2, u2);
        float bb[UO];
        oc.ld_smem(bias_s + 64, bb);
        tm_wait_ld();
        // seeds of l = alpha D_v^2 V + beta D_v V (+ |g|^2):  0T set alpha = -2, beta = 2 gamma;  BND alpha = 0, beta = coef
        const float k8 = BND ? 0.f : 8.f * mk, kg = (BND ? 2.f * a.coef : gamma4) * mk;
        float d1 = 0.f, d2a = 0.f, d2b = 0.f;
        float za[UO], sv[UO], sp[UO];
#if PDEIP_TC_PACKED
        {
          float2 e1 = bc2(0.f), e2a = bc2(0.f), e2b = bc2(0.f);
          const float2 k82 = bc2(k8), nk82 = bc2(-k8), kg2 = bc2(kg);
#pragma unroll
          for (int i = 0; i < UO / 2; ++i) {
            const float2 uu = __fadd2_rn(pr(u, i), pr(bb, i));
            const float2 v1 = pr(u1, i), v2 = pr(u2, i);
            e1 = __ffma2_rn(uu, v1, e1);
            e2a = __ffma2_rn(v1, v1, e2a);
            e2b = __ffma2_rn(uu, v2, e2b);
            st2(za, i, __fmul2_rn(k82, uu));
            st2(sv, i, __ffma2_rn(nk82, v1, __fmul2_rn(kg2, uu)));
            st2(sp, i, __ffma2_rn(k82, v2, __fmul2_rn(kg2, v1)));
          }
          d1 = e1.x + e1.y; d2a = e2a.x + e2a.y; d2b = e2b.x + e2b.y;
        }
#else
#pragma unroll
        for (int i = 0; i < UO; ++i) {
          const float uu = u[i] + bb[i];
          d1 = fmaf(uu, u1[i], d1);
          d2a = fmaf(u1[i], u1[i], d2a);
          d2b = fmaf(uu, u2[i], d2b);
          za[i] = k8 * uu;
          sv[i] = fmaf(-k8, u1[i], kg * uu);
          sp[i] = fmaf(k8, u2[i], kg * u1[i]);
        }
#endif
        oc.template put<kTS>(Z, ZC_ZA2, LOP, za);
        oc.template put<kTS>(Z, ZC_TA, LOP + 24, sv);
        oc.park(LA + C_S0P, sp);
        // this thread's share of D_v V = 2 u.u1 and D_v^2 V = 2 (u1.u1 + u.u2), u2 = -2 u2^
        if constexpr (kSumsSmem) {
          sum_d1 = sums_s[3 * kEpiThreads];
          sum_d2 = sums_s[4 * kEpiThreads];
        }
        sum_d1 = fmaf(2.f * mk, d1, sum_d1);
        sum_d2 = fmaf(mk, 2.f * d2a - 4.f * d2b, sum_d2);
        if constexpr (kSumsSmem) {
          sums_s[3 * kEpiThreads] = sum_d1;
          sums_s[4 * kEpiThreads] = sum_d2;
        }
        TC_PROBE_OUT(6, za);
        TC_PROBE_OUT(7, sv);
        TC_PROBE_OUT(8, sp);
      } else if constexpr (ph == 4 || ph == 5) {
        if constexpr (kPipeFlow && ph == 4) prefetch_inputs(tile + tile_stride);  // read in E10
        // E4 (hidden layer 2) / E5 (hidden layer 1):  aa^ = 4 aa from the GEMM of za^
        //   za^' = aa^ s1,  zbar1' = s1 ab1 + 2 t aa^ a1,  pz = a1 (aa^ a1 - 2 t ab1)
        constexpr bool l2 = ph == 4;
        const uint8_t* At = l2 ? A2 : A1;
        float aa[UH], ab1[UH], t[UH], a1[UH];
        uint32_t s1p[UH / 2];
        tm_ldp<UH>(LA + (l2 ? C_S1P2 : C_S1P1) + UH / 2 * part, s1p);
#pragma unroll
        for (int c = 0; c < HC; ++c) {
          load_chunk(At, (AC_T + HC * part + c) * 128, t + 8 * c);
          load_chunk(At, (AC_A1 + HC * part + c) * 128, a1 + 8 * c);
        }
        tm_wait_ld();
        if constexpr (kEarlyLoads) wait_gemm();
        tm_ldf<UH>(LA + (l2 ? C_AA2 : C_AA1) + uh, aa);
        tm_ldf<UH>(LA + (l2 ? C_AB12 : C_AB11) + uh, ab1);
        tm_wait_ld();
        TC_FINE(0);
        float za[UH], zb[UH], pz[UH];
#if PDEIP_TC_PACKED
#pragma unroll
        for (int i = 0; i < UH / 2; ++i) {
          const float2 s2 = unp2(s1p, i), aa2 = pr(aa, i), a12 = pr(a1, i), ab2 = pr(ab1, i);
          const float2 tt = __fmul2_rn(pr(t, i), bc2(2.f));
          const float2 qq = __fmul2_rn(aa2, a12);
          st2(za, i, __fmul2_rn(aa2, s2));
          st2(zb, i, __ffma2_rn(tt, qq, __fmul2_rn(s2, ab2)));
          st2(pz, i, __fmul2_rn(a12, __ffma2_rn(__fmul2_rn(tt, bc2(-1.f)), ab2, qq)));
        }
#else
#pragma unroll
        for (int i = 0; i < UH; ++i) {
          const float s1 = unp(s1p, i);
          za[i] = aa[i] * s1;
          const float qq = aa[i] * a1[i];
          zb[i] = fmaf(2.f * t[i], qq, s1 * ab1[i]);
          pz[i] = a1[i] * fmaf(-2.f * t[i], ab1[i], qq);
        }
#endif
#pragma unroll
        for (int c = 0; c < HC; ++c) {
          put_op<kTS>(Z, ((l2 ? ZC_ZA1 : ZC_ZA0) + HC * part + c) * 128, LOP + 4 * (HC * part + c), za + 8 * c);
          // zbar1' is an A operand of P4; zbar1'' (E5) only feeds the dW0 chain (shared memory)
          put_op<(kTS && l2)>(Z, ((l2 ? ZC_TB : ZC_TA) + HC * part + c) * 128, LOP + 16 + 4 * (HC * part + c), zb + 8 * c);
        }
        TC_FINE(1);
        tm_park<UH>(LA + (l2 ? C_PZ2 : C_PZ1) + UH / 2 * part, pz);
        TC_FINE(2);
        TC_PROBE(l2 ? 9 : 12, uh, za, UH);
        TC_PROBE(l2 ? 10 : 13, uh, zb, UH);
        TC_PROBE(l2 ? 11 : 14, uh, pz, UH);
      } else if constexpr (ph == 6) {
        // E6: g^ = g / 2 band (the GEMM gives 4 g);  |g|^2, |g_true|^2, |g_true - g|^2
        if constexpr (kSumsSmem) {
          sum_g2 = sums_s[0];
          sum_gt2 = sums_s[kEpiThreads];
          sum_gd2 = sums_s[2 * kEpiThreads];
        }
        // which items carry the sums: the stored gt band, else the x band (gt from the true potential, or zero)
        const bool gt_stored = a.tg.kind == PDEIP_DRIFT_IN_POINTS;
        const float mkc = mk * cgw;  // FP: each of the d direction rows of a point carries 1/d of the per-point sums
        auto add_sums = [&](const float* gv, const float* gt) {
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float df = gt[e] - gv[e];
            sum_g2 = fmaf(mkc * gv[e], gv[e], sum_g2);
            sum_gt2 = fmaf(mkc * gt[e], gt[e], sum_gt2);
            sum_gd2 = fmaf(mkc * df, df, sum_gd2);
          }
        };
        // g^ band first (the operand of the next GEMM), then the sums; the sums of the true-potential kinds come last, so
        // that no input register is live across their out-of-line true_grad_chunk call (a call clobbers the caller-saved
        // registers: at 104 registers the stored-gt items spilled around it)
        auto g_chunk = [&](int cg, float* gv) {
          tm_ld8(LA + C_G + 8 * cg, reinterpret_cast<uint32_t*>(gv));
          tm_wait_ld();
#pragma unroll
          for (int e = 0; e < 8; ++e) gv[e] *= 0.25f;
        };
#pragma unroll
        for (int i = 0; i < NI; ++i) {
          const int j = part + NP * i;
          const int band = j / S::XC, cg = j % S::XC;
          if (band == 0) {
            float gv[8], gh[8];
            g_chunk(cg, gv);
#pragma unroll
            for (int e = 0; e < 8; ++e) gh[e] = (0.5f * cgw) * gv[e];  // the g-stream is linear in its direction: c_g g / 2
            put_op<kTS>(X, (S::XC_G + cg) * 128, LOP + 4 * cg, gh);
            TC_PROBE(15, cg * 8, gv, 8);
          }
        }
        if (gt_stored) {
#pragma unroll
          for (int i = 0; i < NI; ++i) {
            const int j = part + NP * i;
            const int band = j / S::XC, cg = j % S::XC;
            if (j < 3 * S::XC && band == 2) {
              float gv[8], gt[8];
              g_chunk(cg, gv);
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int u = cg * 8 + e;
                float val;
                if (kStage && use_stage) val = stage[((FPM ? d : 2 * d) + (u < d ? u : 0)) * 128];  // still this tile's block
                else val = (NS == 2 && s == 1) ? xin1[i][e] : xin0[i][e];
                gt[e] = (valid && u < d) ? val : 0.f;
              }
              add_sums(gv, gt);
            }
          }
        } else {
#pragma unroll
          for (int i = 0; i < NI; ++i) {
            const int j = part + NP * i;
            const int band = j / S::XC, cg = j % S::XC;
            if (band == 0) {
              float gv[8], gt[8];
              g_chunk(cg, gv);
#pragma unroll
              for (int e = 0; e < 8; ++e) gt[e] = 0.f;
              if (a.tg.kind == PDEIP_DRIFT_LINEAR || a.tg.kind == PDEIP_DRIFT_GMM)
                true_grad_chunk<DP>(a, tp, valid ? p : (int64_t)-1, dimw, cg, gt);
              add_sums(gv, gt);
            }
          }
        }
        if constexpr (kSumsSmem) {
          sums_s[0] = sum_g2;
          sums_s[kEpiThreads] = sum_gt2;
          sums_s[2 * kEpiThreads] = sum_gd2;
        }
      } else if constexpr (ph == 7 || ph == 8) {
        // E7: ag^_1 = s1_1 zg^_0 -> a1 band of A1;  c_1 = a2^_1 + ag^_1       E8: the same for hidden layer 2
        constexpr bool l1 = ph == 7;
        uint8_t* const At = l1 ? A1 : A2;
        float zg[UH], a2[UH];
        uint32_t s1p[UH / 2];
        tm_ldp<UH>(LA + (l1 ? C_S1P1 : C_S1P2) + UH / 2 * part, s1p);
#pragma unroll
        for (int c = 0; c < HC; ++c) load_chunk(At, (AC_C + HC * part + c) * 128, a2 + 8 * c);
        tm_wait_ld();
        if constexpr (kEarlyLoads && !(kGram && l1)) wait_gemm();  // kGram: zg^_0 is a P5 result, already waited for in E6
        if constexpr (kStage && l1) {
          // P6 is committed, so every warp has arrived at the end of E6 (its last read of the staged block, ordered by
          // the proxy fence of that arrive): the next tile's block may overwrite it, five phases ahead of its E0
          if (use_stage && tid == 0) stage_issue(tile + tile_stride);
        }
        tm_ldf<UH>(LA + (l1 ? C_ZG0 : C_ZG1) + uh, zg);
        tm_wait_ld();
        float ag[UH], cc[UH];
#if PDEIP_TC_PACKED
#pragma unroll
        for (int i = 0; i < UH / 2; ++i) {
          const float2 g2 = __fmul2_rn(unp2(s1p, i), pr(zg, i));
          st2(ag, i, g2);
          st2(cc, i, __fadd2_rn(pr(a2, i), g2));
        }
#else
#pragma unroll
        for (int i = 0; i < UH; ++i) {
          ag[i] = unp(s1p, i) * zg[i];
          cc[i] = a2[i] + ag[i];
        }
#endif
#pragma unroll
        for (int c = 0; c < HC; ++c) {
          put_op<kTS>(At, (AC_A1 + HC * part + c) * 128, LOP + 4 * (HC * part + c), ag + 8 * c);
          put_chunk(At, (AC_C + HC * part + c) * 128, cc + 8 * c);
        }
        TC_PROBE(l1 ? 16 : 17, uh, cc, UH);
      } else if constexpr (ph == 9) {
        // E9: s0 = s0p + 8 ug^;  db2 += s0
        float ug[UO], s0[UO];
        uint32_t spp[UO / 2];
        oc.ldp(LA + C_S0P, spp);
        if constexpr (kDbTmem) db2_ld(db2);
        tm_wait_ld();
        if constexpr (kEarlyLoads) wait_gemm();
        oc.ldf(LA + C_UG, ug);
        tm_wait_ld();
#if PDEIP_TC_PACKED
#pragma unroll
        for (int i = 0; i < UO / 2; ++i) {
          const float2 v = __ffma2_rn(bc2(8.f), pr(ug, i), unp2(spp, i));
          st2(s0, i, v);
          st2(db2, i, __fadd2_rn(pr(db2, i), v));
        }
#else
#pragma unroll
        for (int i = 0; i < UO; ++i) {
          s0[i] = fmaf(8.f, ug[i], unp(spp, i));
          db2[i] += s0[i];
        }
#endif
        oc.template put<kTS>(Z, ZC_TA, LOP, s0);
        if constexpr (kDbTmem) db2_st(db2);
        TC_PROBE_OUT(18, s0);
      } else {
        // E10: zbar0' = s1_2 ab_2 + pz2 - 2 t2 aa^2 c_2;  db1       E11: zbar0'' likewise with hidden layer 1;  db0
        constexpr bool l2 = ph == 10;
        // next tile of this slot: issue the input loads first, so that the DRAM latency overlaps this phase's work (the
        // proxy fence of epi_arrive waits for every outstanding load of the thread: a load issued late in a phase is a
        // blocking load)
#if PDEIP_TC_L2_PREFETCH
        if constexpr (l2) {
          if constexpr (kPipeFlow) {  // the x and v items of the next tile (16 registers at d = 32, 8 at d = 16; L2
                                      // prefetch issued in E4) are read here and land behind this phase (measured with 8
                                      // epilogue warps: more than 16 registers here costs more in E10 than the hidden
                                      // latency gives back); its stored gt is read in its own E5
            if (tile + tile_stride < n_tiles) load_inputs(s, tile + tile_stride, 3);
          } else if (!use_stage) {
            prefetch_inputs(tile + tile_stride);
          }
        }
#else
        if constexpr (l2) load_inputs(s, tile + tile_stride);
#endif
        const uint8_t* At = l2 ? A2 : A1;
        float ab[UH], aa[UH], t[UH], cc[UH];
        uint32_t s1p[UH / 2], pzp[UH / 2];
        tm_ldp<UH>(LA + (l2 ? C_S1P2 : C_S1P1) + UH / 2 * part, s1p);
        tm_ldp<UH>(LA + (l2 ? C_PZ2 : C_PZ1) + UH / 2 * part, pzp);
#pragma unroll
        for (int c = 0; c < HC; ++c) {
          load_chunk(At, (AC_T + HC * part + c) * 128, t + 8 * c);
          load_chunk(At, (AC_C + HC * part + c) * 128, cc + 8 * c);
        }
        if constexpr (kDbTmem) db_ld(l2 ? cdb1 : cdb0, l2 ? db1 : db0);
        tm_wait_ld();
        if constexpr (kEarlyLoads) wait_gemm();
        tm_ldf<UH>(LA + (l2 ? C_AB2 : C_AB1) + uh, ab);
        tm_ldf<UH>(LA + (l2 ? C_AA2R : C_AA1R) + uh, aa);
        tm_wait_ld();
        float zb[UH];
#if PDEIP_TC_PACKED
#pragma unroll
        for (int i = 0; i < UH / 2; ++i) {
          const float2 m0 = __ffma2_rn(unp2(s1p, i), pr(ab, i), unp2(pzp, i));
          const float2 ta = __fmul2_rn(__fmul2_rn(pr(t, i), bc2(-2.f)), pr(aa, i));
          const float2 v = __ffma2_rn(ta, pr(cc, i), m0);
          st2(zb, i, v);
          if (l2) st2(db1, i, __fadd2_rn(pr(db1, i), v));
          else st2(db0, i, __fadd2_rn(pr(db0, i), v));
        }
#else
#pragma unroll
        for (int i = 0; i < UH; ++i) {
          const float m0 = fmaf(unp(s1p, i), ab[i], unp(pzp, i));
          zb[i] = fmaf(-2.f * t[i] * aa[i], cc[i], m0);
          if (l2) db1[i] += zb[i];
          else db0[i] += zb[i];
        }
#endif
#pragma unroll
        for (int c = 0; c < HC; ++c)  // zbar0' is an A operand of P10; zbar0'' (E11) only feeds the dW0 chain
          put_op<(kTS && l2)>(Z, ((l2 ? ZC_TB : ZC_TA) + HC * part + c) * 128, LOP + 4 * (HC * part + c), zb + 8 * c);
        if constexpr (kDbTmem) db_st(l2 ? cdb1 : cdb0, l2 ? db1 : db0);
        TC_PROBE(l2 ? 19 : 20, uh, zb, UH);
      }
      if constexpr (!(kGram && ph == 6)) {  // kGram: no hand-off after E6, E7 follows immediately (zg^_0 came out of P5)
        if constexpr (kTS) tm_wait_st();  // the A-operand columns are complete before the hand-off
        TC_TRACE(7);
        if constexpr (kTwoStage && (ph == 3 || ph == 4 || ph == 5 || ph == 7 || ph == 9 || ph == 10 || ph == 11)) {
          epi_arrive<NS, false>(s);  // layer GEMMs (A from TMEM, B = weights): go
          fence_async_smem();    // the bands this phase wrote -> async proxy, for the dW chains behind the second barrier
          asm volatile("bar.arrive %0, %1;" ::"r"(4 + (int)tsb), "n"(kThreads) : "memory");
          tsb ^= 1u;
        } else {
#ifdef PDEIP_TC_TRACE
        fence_async_smem();
        TC_FINE(3);
        fence_before_sync();
        TC_FINE(4);
        asm volatile("bar.arrive %0, %1;" ::"r"(1 + s), "n"(kThreads) : "memory");
#else
        // The generic -> async proxy fence orders this thread's shared-memory writes before the MMAs that READ them.  With
        // the layer-GEMM A operands in TMEM (kTS) the GEMMs of P0, P1, P2 and P8 read no activation bytes from shared
        // memory, and the bands written by E0, E1, E2, E8 are first read by dW chains issued behind LATER hand-offs
        // (P3 / P4 / P5 / P9 ...), whose fences (same thread, later in program order) cover these writes too.
        constexpr bool kNeedProxyFence = !(kTS && (ph == 0 || ph == 1 || ph == 2 || ph == 8));
        epi_arrive<NS, kNeedProxyFence>(s);
#endif
        }
        TC_TRACE(2);
      }
      if constexpr (kPipeFlow && ph == 10) {  // E0 of the NEXT tile, while P10 executes (its TMEM stores and shared-memory
                                          // writes are ordered before P0 by the wait::st / proxy fence of E11's hand-off)
        // (its x and v items were read at the start of E10)
        const int64_t tn = tile + tile_stride;
        const int64_t pn = (FPM ? (int64_t)((uint32_t)tn / fpd) : tn) * 128 + row;
        if (tn < n_tiles) emit_x(xin0, pn < a.n_points, sm + (xb ? 0u : S::O_X2) + S::O_X + offX);
      }
    };
#define PDEIP_TC_PHASE(PH)                       \
  _Pragma("unroll 1") for (int s_ = 0; s_ < NS; ++s_) phase(IC<PH>{}, s_);

#pragma unroll 1
    for (; base < n_tiles; base += tile_stride) {
      if (!kPipeFlow || first) { PDEIP_TC_PHASE(0) }
      PDEIP_TC_PHASE(1) PDEIP_TC_PHASE(2) PDEIP_TC_PHASE(3) PDEIP_TC_PHASE(4) PDEIP_TC_PHASE(5)
      PDEIP_TC_PHASE(6) PDEIP_TC_PHASE(7) PDEIP_TC_PHASE(8) PDEIP_TC_PHASE(9) PDEIP_TC_PHASE(10) PDEIP_TC_PHASE(11)
      first = false;
      xb ^= 1u;
    }
#undef PDEIP_TC_PHASE
    // ---- drain: wait for P11 of the last tile of every slot (covers every MMA issued before it) --------------
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      if (ok && !mbar_wait(smem_u32(mbar_p + s), (par >> s) & 1u)) {
        ok = false;
        atomicExch(status, 1);
      }
    }
    fence_after_sync();
    asm volatile("bar.sync 3, %0;" ::"n"(kEpiThreads) : "memory");

    // ---- write-out: this CTA's partial (one writer per index, fixed order -> bit-reproducible) ------------------
    float* wsp = a.ws + (int64_t)blockIdx.x * a.pstride;
    float* red = reinterpret_cast<float*>(sm);  // [4 quadrants][128] bias sums + [epilogue warps][8] loss sums
    static_assert((512 + 8 * Team<NS>::kEpiWarps) * 4 <= S::O_BIAS, "write-out scratch inside the operand tiles");
    const float wt = a.weight;
    if (ok && q < 2) {  // M = 64 dW blocks: input unit i = 16 q + lane sits in TMEM lane 32 q + lane, lane < 16
      const uint32_t LQ = TB + ((uint32_t)(q * 32) << 16);
      const int iu = 16 * q + lane;
      float w2[UO], w1[UH], w0[UH];
      oc.ldf(LQ + C_DW2, w2);
      tm_ldf<UH>(LQ + C_DW1 + uh, w1);
      tm_ldf<UH>(LQ + C_DW0 + uh, w0);
      tm_wait_ld();
      if (lane < 16) {
#pragma unroll
        for (int i = 0; i < UO; ++i)
          if (oc.unit(i) < kOut) wsp[sh.w_off(2) + iu * kOut + oc.unit(i)] += wt * w2[i];
#pragma unroll
        for (int i = 0; i < UH; ++i) wsp[sh.w_off(1) + iu * H + uh + i] += wt * w1[i];
        if (iu < d) {
#pragma unroll
          for (int i = 0; i < UH; ++i) wsp[sh.w_off(0) + iu * H + uh + i] += wt * w0[i];
        }
      }
    }
    // bias gradients: sum over the 32 rows of the warp, then over the 4 quadrants through shared memory
    // red layout: [q][0..31] db0, [32..63] db1, [64..111] db2
    if constexpr (kDbTmem) {
      db_ld(cdb0, db0);
      db_ld(cdb1, db1);
      db2_ld(db2);
      tm_wait_ld();
    }
#pragma unroll
    for (int i = 0; i < UH; ++i) {
      const float r0 = warp_sum(db0[i]), r1 = warp_sum(db1[i]);
      if (lane == 0) {
        red[q * 128 + uh + i] = r0;
        red[q * 128 + 32 + uh + i] = r1;
      }
    }
#pragma unroll
    for (int i = 0; i < UO; ++i) {
      const float r2 = warp_sum(db2[i]);
      if (lane == 0) red[q * 128 + 64 + oc.unit(i)] = r2;
    }
    {
      if constexpr (kSumsSmem) {
        sum_g2 = sums_s[0];
        sum_gt2 = sums_s[kEpiThreads];
        sum_gd2 = sums_s[2 * kEpiThreads];
        sum_d1 = sums_s[3 * kEpiThreads];
        sum_d2 = sums_s[4 * kEpiThreads];
      }
      const float sums5[5] = {sum_g2, sum_gt2, sum_gd2, sum_d1, sum_d2};
#pragma unroll
      for (int k = 0; k < 5; ++k) {
        const float sk = warp_sum(sums5[k]);
        if (lane == 0) red[512 + warp * 8 + k] = sk;
      }
    }
    asm volatile("bar.sync 3, %0;" ::"n"(kEpiThreads) : "memory");
    if (ok) {
      if (tid < 112) {
        const float v = (red[tid] + red[128 + tid]) + (red[256 + tid] + red[384 + tid]);
        if (tid < 32) wsp[sh.b_off(0) + tid] += wt * v;
        else if (tid < 64) wsp[sh.b_off(1) + tid - 32] += wt * v;
        else if (tid - 64 < kOut) wsp[sh.b_off(2) + tid - 64] += wt * v;
      }
      if (tid == 128) {
        float t5[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        for (int w = 0; w < Team<NS>::kEpiWarps; ++w)
          for (int k = 0; k < 5; ++k) t5[k] += red[512 + w * 8 + k];
        const float g2 = wt * t5[0], gt2 = wt * t5[1], gd2 = wt * t5[2], D1 = wt * t5[3], D2 = wt * t5[4];
        if constexpr (BND) {  // residual_mlp.cu, KFP_BOUNDARY: sum coef grad V . v
          wsp[P + PDEIP_SUM_BOUNDARY] += a.coef * D1;
          wsp[P + PDEIP_SUM_LOSS] += a.coef * D1;
        } else {
          wsp[P + PDEIP_SUM_G2] += g2;
          wsp[P + PDEIP_SUM_GTRUE2] += gt2;
          wsp[P + PDEIP_SUM_GT] += gd2;
          if (!FPM) wsp[P + PDEIP_SUM_D1] += D1;  // FP rows: D_{e_i} V is not a loss term (fokker_planck.py:50-51)
          wsp[P + PDEIP_SUM_D2] += D2;
          wsp[P + PDEIP_SUM_LOSS] += g2 + gt2 - 2.f * D2 + 2.f * gamma * D1;
        }
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(TB, 512);
}

}  // namespace tc

// one status / debug buffer per device (the "no allocation inside the entry points" rule has this one exception: a
// few hundred KB allocated once per device on the first tensor-path launch)
int* tensor_status_word() {
  static int* w[64] = {nullptr};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  if (!w[dev]) {
    const size_t bytes = 8192 + 24 * 128 * 48 * sizeof(float);
    if (cudaMalloc(&w[dev], bytes) != cudaSuccess) return nullptr;
    cudaMemset(w[dev], 0, bytes);
  }
  return w[dev];
}

#ifdef PDEIP_HAVE_TENSOR_PATH
template <int DP, int NS, int MODE>
static int launch_tc(const ResidualArgs& a, int* status, cudaStream_t st) {
  using S = tc::Cfg<DP, NS>;
  auto kern = tc::mlp_residual_tc_kernel<DP, NS, MODE>;
  PDEIP_REQUIRE(true_grad_floats(a.tg, a.d) * sizeof(float) <= S::TP_BYTES, PDEIP_ERR_UNSUPPORTED,
                "tensor path: true-gradient parameters exceed %u bytes", (unsigned)S::TP_BYTES);
  PDEIP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::TOTAL));
  kern<<<residual_grid(), tc::Team<NS>::kLaunchThreads, S::TOTAL, st>>>(a, status);
  PDEIP_LAUNCH_OK();
  return PDEIP_OK;
}

int mlp_residual_accumulate_tensor(int set_kind, const ResidualArgs& a, int hidden, cudaStream_t st) {
  // FP boundary (coef V) and KMV pairs stay on the fp32 kernel
  if (set_kind != PDEIP_SET_KFP_0T && set_kind != PDEIP_SET_FP_0T && set_kind != PDEIP_SET_KFP_BOUNDARY)
    return mlp_residual_accumulate_fp32(set_kind, a, hidden, st);
  PDEIP_REQUIRE(hidden == 32 && a.layers == 2, PDEIP_ERR_UNSUPPORTED,
                "tensor path is built for hidden_dim == 32, layers == 2 (got %d, %d)", hidden, a.layers);
  PDEIP_REQUIRE(a.d >= 1 && a.d <= 32, PDEIP_ERR_UNSUPPORTED, "tensor path supports 1 <= d <= 32 (got %d)", a.d);
  int* status = tensor_status_word();
  PDEIP_REQUIRE(status != nullptr, PDEIP_ERR_CUDA, "cannot allocate the tensor-path status word");
  ResidualArgs b = a;
  int mode = tc::kModeKfp0T;
  if (set_kind == PDEIP_SET_FP_0T) {  // d tangent streams stacked along M: one tile row (x, e_i) per direction, gamma = 0
    PDEIP_REQUIRE((a.n_points + 127) / 128 * (int64_t)a.d < ((int64_t)1 << 31), PDEIP_ERR_UNSUPPORTED,
                  "FP tensor path: n_points * d / 128 must stay below 2^31");
    b.fp_dirs = a.d;
    b.coef = 0.f;
    mode = tc::kModeFp0T;
  } else if (set_kind == PDEIP_SET_KFP_BOUNDARY) {
    b.tg.kind = PDEIP_DRIFT_NONE;  // boundary points are rows [x, v]
    mode = tc::kModeBnd;
  }
#define PDEIP_TC_DISPATCH(DP, NS)                                                     \
  (mode == tc::kModeKfp0T ? launch_tc<DP, NS, tc::kModeKfp0T>(b, status, st)          \
   : mode == tc::kModeBnd ? launch_tc<DP, NS, tc::kModeBnd>(b, status, st)            \
                          : launch_tc<DP, NS, tc::kModeFp0T>(b, status, st))
  if (a.d <= 8) return PDEIP_TC_DISPATCH(8, 2);
  if (a.d <= 16) return PDEIP_TC_DISPATCH(16, 1);
  return PDEIP_TC_DISPATCH(32, 1);
#undef PDEIP_TC_DISPATCH
}
#endif

// read-and-clear: bit 0 = a residual phase timed out, bit 1 = an integrator phase timed out since the last query / begin
int tensor_path_status(cudaStream_t st, int* out) {
  int* status = tensor_status_word();
  if (!status) return PDEIP_ERR_CUDA;
  int w[2] = {0, 0};
  if (cudaMemcpyAsync(w, status, 2 * sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess) return PDEIP_ERR_CUDA;
  if (cudaStreamSynchronize(st) != cudaSuccess) return PDEIP_ERR_CUDA;
  *out = (w[0] ? 1 : 0) | (w[1] ? 2 : 0);
  if (*out && cudaMemsetAsync(status, 0, 2 * sizeof(int), st) != cudaSuccess) return PDEIP_ERR_CUDA;
  return PDEIP_OK;
}

}  // namespace pdeip

// 0 = every tcgen05 phase completed; 1 = a bounded mbarrier wait timed out (results invalid).  Synchronises.
extern "C" int pdeip_tensor_path_status(void* stream, int* out_status) {
  PDEIP_REQUIRE(out_status != nullptr, PDEIP_ERR_INVALID_ARG, "out_status is NULL");
  return pdeip::tensor_path_status((cudaStream_t)stream, out_status);
}

// test hook: set status word `word` (0 residual, 1 integrator) as a timed-out kernel would
extern "C" int pdeip_debug_set_status(int word, int value, void* stream) {
  int* status = pdeip::tensor_status_word();
  if (!status || word < 0 || word > 1) return PDEIP_ERR_INVALID_ARG;
  if (cudaMemcpyAsync(status + word, &value, sizeof(int), cudaMemcpyHostToDevice, (cudaStream_t)stream) != cudaSuccess)
    return PDEIP_ERR_CUDA;
  if (cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess) return PDEIP_ERR_CUDA;
  return PDEIP_OK;
}

// debug (PDEIP_TC_TRACE builds): 24 x 8 clock stamps (see TC_TRACE)
extern "C" int pdeip_debug_tensor_trace(long long* out, int n) {
  int* status = pdeip::tensor_status_word();
  if (!status) return PDEIP_ERR_CUDA;
  if (n > 24 * 8 + 48 + 16) return PDEIP_ERR_INVALID_ARG;
  if (cudaDeviceSynchronize() != cudaSuccess) return PDEIP_ERR_CUDA;
  if (cudaMemcpy(out, reinterpret_cast<long long*>(status) + 512, sizeof(long long) * (size_t)n, cudaMemcpyDeviceToHost) !=
      cudaSuccess)
    return PDEIP_ERR_CUDA;
  if (cudaMemset(reinterpret_cast<long long*>(status) + 512, 0, sizeof(long long) * (size_t)n) != cudaSuccess)  // the stamps are sums
    return PDEIP_ERR_CUDA;
  return PDEIP_OK;
}

// debug (PDEIP_TC_PROBE builds): per-phase epilogue values of tile 0, [probe id][row 128][unit 48] floats
extern "C" int pdeip_debug_tensor_probe(float* out, int n_floats) {
  int* status = pdeip::tensor_status_word();
  if (!status) return PDEIP_ERR_CUDA;
  if (n_floats > 24 * 128 * 48) return PDEIP_ERR_INVALID_ARG;
  if (cudaDeviceSynchronize() != cudaSuccess) return PDEIP_ERR_CUDA;
  if (cudaMemcpy(out, reinterpret_cast<float*>(status) + 2048, sizeof(float) * (size_t)n_floats, cudaMemcpyDeviceToHost) !=
      cudaSuccess)
    return PDEIP_ERR_CUDA;
  return PDEIP_OK;
}
