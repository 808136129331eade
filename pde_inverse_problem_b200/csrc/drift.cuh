// drift.cuh — per-thread drift functors  grad U(q)  on register arrays.
//
//   GMM      : core/potential.py:32-37 — a_k = -|x-mu_k|^2/(2 sigma^2), U = -logsumexp(a),
//              grad U = (x - sum_k softmax(a)_k mu_k) / sigma^2   (closed form of jax.grad(gmm_V))
//   LINEAR   : grad U = A x  (kinetic OU tilde_F x, example_problems/kinetic_fokker_planck_example_OU.py:15-20;
//              QuadraticPotential.gradient with mu = 0, core/potential.py:20-24)
//   MEANFIELD: grad U = A (x - xbar)  (README.md:54-71)
//   AFFINE   : grad U = M x + b  (the quadratic hypothesis model V = y.(yK + b): M = K + K^T,
//              example_problems/kinetic_fokker_planck_example_OU.py:209-220)
//   MLP      : grad U = grad V_theta of the hypothesis MLP (core/model.py:51-62), mlp_thread.cuh
// Parameters live in shared memory, zero-padded to the compile-time width DP, so a runtime
// d <= DP needs no masking inside the arithmetic (padded components stay exactly zero).
#pragma once

#include "common.cuh"
#include "mlp_thread.cuh"

namespace pdeip {

// copy a row-major [rows][d] global matrix into smem as [rows][DP], zero padded
template <int DP>
__device__ __forceinline__ void load_padded(float* dst, const float* __restrict__ src, int rows, int d,
                                            int tid, int nthreads) {
  for (int idx = tid; idx < rows * DP; idx += nthreads) {
    const int r = idx / DP, c = idx - r * DP;
    dst[idx] = (c < d) ? src[r * d + c] : 0.0f;
  }
}

// online-softmax GMM gradient; mus_s: smem [K][DP]
template <int DP>
__device__ __forceinline__ void gmm_grad_thread(const float (&x)[DP], const float* __restrict__ mus_s, int K,
                                                float inv_sigma2, float (&g)[DP], float* value = nullptr) {
  float m = -INFINITY, se = 0.0f;
  float acc[DP];
#pragma unroll
  for (int i = 0; i < DP; ++i) acc[i] = 0.0f;
  for (int k = 0; k < K; ++k) {
    const float* mu = mus_s + k * DP;
    float mk[DP];
    if constexpr (DP % 4 == 0) {
#pragma unroll
      for (int i4 = 0; i4 < DP / 4; ++i4) {
        const float4 t = reinterpret_cast<const float4*>(mu)[i4];
        mk[4 * i4 + 0] = t.x; mk[4 * i4 + 1] = t.y; mk[4 * i4 + 2] = t.z; mk[4 * i4 + 3] = t.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < DP; ++i) mk[i] = mu[i];
    }
    float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
    for (int i = 0; i < DP; i += 2) {
      const float r0 = x[i] - mk[i];
      s0 = fmaf(r0, r0, s0);
      if (i + 1 < DP) {
        const float r1 = x[i + 1] - mk[i + 1];
        s1 = fmaf(r1, r1, s1);
      }
    }
    const float a = -0.5f * inv_sigma2 * (s0 + s1);
    if (a > m) {  // new running maximum: rescale what has been accumulated
      const float sc = expf(m - a);
      se *= sc;
#pragma unroll
      for (int i = 0; i < DP; ++i) acc[i] *= sc;
      m = a;
    }
    const float e = expf(a - m);
    se += e;
#pragma unroll
    for (int i = 0; i < DP; ++i) acc[i] = fmaf(e, mk[i], acc[i]);
  }
  const float inv = 1.0f / se;
#pragma unroll
  for (int i = 0; i < DP; ++i) g[i] = (x[i] - acc[i] * inv) * inv_sigma2;
  if (value) *value = -(m + logf(se));
}

// A_s: smem [DP][DP] row-major (padded); g = A (x - shift)
template <int DP>
__device__ __forceinline__ void linear_grad_thread(const float (&x)[DP], const float* __restrict__ A_s,
                                                   const float* __restrict__ shift_s, float (&g)[DP]) {
  float y[DP];
#pragma unroll
  for (int i = 0; i < DP; ++i) y[i] = shift_s ? x[i] - shift_s[i] : x[i];
#pragma unroll
  for (int i = 0; i < DP; ++i) {
    float s = 0.0f;
#pragma unroll
    for (int k = 0; k < DP; ++k) s = fmaf(A_s[i * DP + k], y[k], s);
    g[i] = s;
  }
}

// M_s: smem [DP][DP] row-major (padded), b_s: [DP];  g = M x + b
template <int DP>
__device__ __forceinline__ void affine_grad_thread(const float (&x)[DP], const float* __restrict__ M_s,
                                                   const float* __restrict__ b_s, float (&g)[DP]) {
#pragma unroll
  for (int i = 0; i < DP; ++i) {
    float s = 0.0f;
#pragma unroll
    for (int k = 0; k < DP; ++k) s = fmaf(M_s[i * DP + k], x[k], s);
    g[i] = s + b_s[i];
  }
}

// grad V_theta(x) of the hypothesis MLP, weights in smem (flat layout of pdeip.h, hidden width 32);
// g[i] = 0 for d <= i < DP.  The per-point activations live in the thread's local memory.
template <int DP, int LHMAX>
__device__ __forceinline__ void mlp_grad_thread(const float (&x)[DP], const MlpShape<32>& sh,
                                                const float* __restrict__ w_s, float (&g)[DP]) {
  PointState<32, LHMAX> st;
  MlpThread<32, LHMAX> net(sh, w_s, st);
#pragma unroll
  for (int i = 0; i < DP; ++i)
    if (i < sh.d) st.x[i] = x[i];
  net.primal_forward();
  float gl[kDMax];
  net.input_gradient(gl);
#pragma unroll
  for (int i = 0; i < DP; ++i) g[i] = i < sh.d ? gl[i] : 0.0f;
}

}  // namespace pdeip
