/*
 * pdeip.h — C ABI of the B200-native hot path of shenzebang/PDE-inverse-problem.
 *
 * One shared library (libpdeip.so, sm_100a).  Every entry point takes plain device pointers,
 * sizes, scalars and a CUDA stream (void* == cudaStream_t); the caller owns and allocates every
 * buffer (workspace sizes come from the *_workspace_bytes queries); calls enqueue work on the
 * stream and return without synchronising; they return 0 or a negative PDEIP_ERR_* code and never
 * throw.  The reference has no native code and no FFI: each entry point below replaces the JAX
 * function cited next to it (paths relative to the reference checkout), i.e. it is what an
 * XLA-FFI / ctypes binding for that function would bind (see INTEGRATION.md).
 *
 * Conventions
 *   - all floating-point data is float32 (the reference never enables x64);
 *   - kinetic states are rows [x(0..d-1), v(0..d-1)] of length 2d, as jnp.split(.., 2, axis=-1)
 *     in methods/consistency_instances/kinetic_fokker_planck.py:13-15;
 *   - `layout` arguments: PDEIP_LAYOUT_AOS  rows of `dim` floats, point-major        [n][dim]
 *                         PDEIP_LAYOUT_SOA  component planes                         [dim][n]
 *                         PDEIP_LAYOUT_BLOCK128  128-point blocks of component planes  [n/128][dim][128]
 *   - MLP parameters are one flat buffer [W0 (d x H, row-major [in][out]), b0 (H), W1 (H x H), b1,
 *     ..., W_last (H x 40), b_last (40)] — Flax's layers_i/{kernel,bias} order (core/model.py:42-43);
 *   - sums, not means: residual kernels return weighted SUMS over the points they were given
 *     (weight = 1/global count), so that shards add up under one all-reduce(sum).
 */
#ifndef PDEIP_H_
#define PDEIP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PDEIP_ABI_VERSION 1

#define PDEIP_OK               0
#define PDEIP_ERR_INVALID_ARG (-1)
#define PDEIP_ERR_UNSUPPORTED (-2)
#define PDEIP_ERR_WORKSPACE   (-3)
#define PDEIP_ERR_CUDA        (-4)

#define PDEIP_LAYOUT_AOS 0
#define PDEIP_LAYOUT_SOA 2
#define PDEIP_LAYOUT_BLOCK128 3 /* [n/128][dim][128]: blocks of 128 points, component planes inside a block (n % 128 == 0) */

/* trajectory layouts of pdeip_kl_integrate */
#define PDEIP_TRAJ_PARTICLE_MAJOR 0 /* [N][S_emit][2d]  (reference: utils/sampling_utils.py:52 under vmap) */
#define PDEIP_TRAJ_TIME_MAJOR     1 /* [S_emit][N][2d] */
#define PDEIP_TRAJ_TIME_SOA       2 /* [2d][S_emit][N]: an SOA point set of S_emit*N points, point = s*N + n */
#define PDEIP_TRAJ_BLOCK128       3 /* [S_emit][N/128][2d][128] (N % 128 == 0): a PDEIP_LAYOUT_BLOCK128 point set of
                                     S_emit*N points, point = s*N + n; all stores of a step are base + constant */

/* drift kinds */
#define PDEIP_DRIFT_NONE      0 /* VoidPotential, core/potential.py:27-29 */
#define PDEIP_DRIFT_LINEAR    1 /* grad U = A x          A row-major [d][d]  (kinetic OU, README.md:64-71) */
#define PDEIP_DRIFT_GMM       2 /* core/potential.py:32-61, params = mus [K][d] */
#define PDEIP_DRIFT_MEANFIELD 3 /* grad U = A (x - xbar), params = [A (d*d), xbar (d)] */
#define PDEIP_DRIFT_IN_POINTS 4 /* residual kernels only: grad V_true is stored after each point's own components */
#define PDEIP_DRIFT_MEANFIELD_TABLE 5 /* grad U = A (x - xbar_s) at step s (README.md:54-62 with Phi = x'Ax/2 and the EMPIRICAL
                                         mean of all particles): params = [A (d*d), A xbar_s for s = 0..n_steps ((n_steps+1)*d)]
                                         from pdeip_meanfield_xbar_table; REFERENCE schedule on the common time grid
                                         (tau0 == 0 unless injected: step 0 has h = 0, sample s is the state at time s dt) */

/* step schedules */
#define PDEIP_SCHEDULE_REFERENCE 0 /* step(tau0), (S-1) x step(dt), step(dt - tau0): sampling_utils.py:32-46 */
#define PDEIP_SCHEDULE_UNIFORM   1 /* S steps of dt, every state emitted (no tau0) */

/* model kinds for the residual kernels */
#define PDEIP_MODEL_MLP       0 /* core/model.py:32-62 */
#define PDEIP_MODEL_GMM       1 /* example_problems/kinetic_fokker_planck_example_GMM.py:214-234 */
#define PDEIP_MODEL_QUADRATIC 2 /* example_problems/kinetic_fokker_planck_example_OU.py:209-220 */

/* point-set kinds for pdeip_residual_accumulate */
#define PDEIP_SET_KFP_0T        0 /* |gV|^2 - 2 v'Hv + 2 gamma gV.v        kinetic_fokker_planck.py:40-45 */
#define PDEIP_SET_KFP_BOUNDARY  1 /* coef * gV.v  (coef = +-2/T)           kinetic_fokker_planck.py:34-39,48-50 */
#define PDEIP_SET_FP_0T         2 /* |gV|^2 - 2 Laplacian V               fokker_planck.py:50-51 */
#define PDEIP_SET_FP_BOUNDARY   3 /* coef * V                             fokker_planck.py:48-49,53 */
#define PDEIP_SET_KMV_PAIRS     4 /* pairwise residual                    kinetic_mckean_vlasov.py:74-97 */

/* arithmetic paths of the MLP residual */
#define PDEIP_PATH_FP32   0 /* CUDA-core fp32 (parity path, rtol 1e-5) */
#define PDEIP_PATH_TENSOR 1 /* tcgen05 tensor-core path (rtol 1e-2) */

/* slots of the `sums` output of pdeip_residual_finalize (all weighted sums) */
#define PDEIP_SUM_G2        0 /* sum |grad V|^2 over 0T                               */
#define PDEIP_SUM_D2        1 /* sum v'Hv (KFP/KMV) or Laplacian (FP) over 0T           */
#define PDEIP_SUM_D1        2 /* sum grad V . v over 0T (KFP) / sum c_j Phi (KMV)       */
#define PDEIP_SUM_GTRUE2    3 /* sum |grad V_true|^2 over 0T                            */
#define PDEIP_SUM_GT        4 /* sum |grad V_true - grad V|^2 over 0T ("loss ground truth") */
#define PDEIP_SUM_BOUNDARY  5 /* sum coef * (gV.v | V) over boundary sets              */
#define PDEIP_SUM_LOSS      6 /* assembled loss of the point sets accumulated so far   */
#define PDEIP_SUM_GRADNORM  7 /* ||grad||_2 of the accumulated gradient (common_utils.py:74-76) */
#define PDEIP_NUM_SUMS      8

int pdeip_abi_version(void);
/* human-readable message of the last failing call on this thread ("" if none) */
const char* pdeip_last_error(void);
/* number of SMs the library sizes its persistent grids for (148 when no device is visible) */
int pdeip_sm_count(void);

/* ---------------------------------------------------------------------------------------------
 * K1  kinetic-Langevin integrator.          replaces utils/sampling_utils.py:6-52
 *   p' = p - h gradU(q) + sqrt(2h) xi - gamma p h ;  q' = q + h p'
 * z0, z_last: [N][2d] (state_layout AOS) or [2d][N] (SOA).  traj: NULL for terminal-only, else
 * the emitted samples in `traj_layout`; sample s (0 <= s < S) is emitted iff s % emit_every ==
 * emit_offset, S_emit = number of such s.  tau (optional, [N][S] particle-major): tau0 + s*dt
 * (sampling_utils.py:48).  noise: NULL -> in-register Philox4x32-10 keyed by (seed, particle_offset
 * + n, step_offset + s); else injected normals [N][S+1][d] (REFERENCE schedule) / [N][S][d] (UNIFORM).
 * tau0: NULL -> Philox uniform [0,1)*dt; else injected [N] (REFERENCE schedule only).
 * emit_drift != 0: every emitted sample is [x, v, grad U(x)] (3d floats; the integrator evaluates grad U(x) anyway at
 * the following step), which the residual kernels accept as grad V_true via PDEIP_DRIFT_IN_POINTS.
 * ------------------------------------------------------------------------------------------- */
int pdeip_kl_integrate(const float* z0, float* z_last, float* traj, float* tau,
                       int64_t n_particles, int d, int n_steps, float dt, float gamma,
                       int drift_kind, const float* drift_params, int n_gaussian, float sigma,
                       const float* noise, const float* tau0,
                       uint64_t seed, uint64_t particle_offset, uint32_t step_offset,
                       int schedule, int state_layout, int traj_layout,
                       int emit_every, int emit_offset, int emit_drift, void* stream);

/* Same call with a kernel path.  PDEIP_PATH_FP32: CUDA-core fp32 arithmetic throughout (rtol 1e-5 class).
 * PDEIP_PATH_TENSOR: in the production configuration (Philox noise, REFERENCE schedule, AOS state, TIME_SOA
 * trajectory with emit_drift, emit_every 1) with the GMM drift, d = 8, 16 or 32 and n_gaussian <= 64, the particle x
 * centre contraction and the softmax-weighted centre sum run on tcgen05 with bf16 hi + lo split operands
 * ("bf16 GEMM path", rtol 1e-2 class; measured ~1e-4); every other configuration runs the fp32 kernels. */
int pdeip_kl_integrate_path(const float* z0, float* z_last, float* traj, float* tau,
                            int64_t n_particles, int d, int n_steps, float dt, float gamma,
                            int drift_kind, const float* drift_params, int n_gaussian, float sigma,
                            const float* noise, const float* tau0,
                            uint64_t seed, uint64_t particle_offset, uint32_t step_offset,
                            int schedule, int state_layout, int traj_layout,
                            int emit_every, int emit_offset, int emit_drift, int path, void* stream);

/* K1 with grad U = grad V_theta of a hypothesis model (model_kind / params / hidden / layers / n_gaussian exactly as
 * in pdeip_model_eval and the residual kernels).  Every other argument, output, layout, schedule, Philox stream and
 * emit_drift contract is that of pdeip_kl_integrate_path: the reference's underdamped_langevin_dynamics_scan driven by
 * jax.grad of a fitted net.apply (utils/sampling_utils.py:25-52 with potential_grad = grad V_theta).
 *   PDEIP_MODEL_MLP       hidden == 32 (narrower nets zero-padded), 1 <= layers <= 8, d <= 32; fp32 on the CUDA cores
 *                         (rtol 1e-5 class).  PDEIP_PATH_TENSOR with layers == 2, d = 8, 16 or 32, Philox noise, REFERENCE
 *                         schedule, AOS state, emit_every 1 and either traj == NULL (terminal state only, n arbitrary) or
 *                         a PDEIP_TRAJ_BLOCK128 / PDEIP_TRAJ_TIME_SOA trajectory with emit_drift: the six GEMMs of a step
 *                         (primal chain and input-gradient chain) run on tcgen05 with bf16 hi + lo split operands ("bf16
 *                         GEMM path", rtol 1e-2 class); every other call takes the fp32 kernel (PDEIP_NO_TC_INTEGRATOR=1
 *                         forces it);
 *   PDEIP_MODEL_GMM       learned centres, sigma = 1: exactly pdeip_kl_integrate_path(PDEIP_DRIFT_GMM, params,
 *                         n_gaussian, 1.0f, ...) on all of its kernels (bit-identical);
 *   PDEIP_MODEL_QUADRATIC V = y.(yK + b): grad V = (K + K^T) y + b, fp32 on both paths.
 * Rejected before any CUDA call: unknown model kind, NULL params (PDEIP_ERR_INVALID_ARG), d > 32, layers outside
 * [1, 8], hidden != 32 (PDEIP_ERR_UNSUPPORTED), GMM with n_gaussian < 1 (PDEIP_ERR_INVALID_ARG). */
int pdeip_kl_integrate_model(const float* z0, float* z_last, float* traj, float* tau,
                             int64_t n_particles, int d, int n_steps, float dt, float gamma,
                             int model_kind, const float* params, int hidden, int layers, int n_gaussian,
                             const float* noise, const float* tau0,
                             uint64_t seed, uint64_t particle_offset, uint32_t step_offset,
                             int schedule, int state_layout, int traj_layout,
                             int emit_every, int emit_offset, int emit_drift, int path, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K1-OD  overdamped Langevin integrator: dX = -grad U(X) dt + sqrt(2) dW (the Fokker-Planck instance,
 * example_problems/fokker_planck_example.py), Euler-Maruyama with S steps of size dt:
 *   x_{s+1} = x_s - dt grad U(x_s) + sqrt(2 dt) xi_s,   s = 0..S-1   (the sqrt(2) is fixed, as in K1)
 * Sample s is the state after step s; x_last is sample S-1.  No tau0, no reference schedule.
 * x0, x_last: [N][d] (state_layout AOS) or [d][N] (SOA).  noise: NULL -> Philox4x32-10 keyed by (seed, particle_offset
 * + n, step_offset + s), i.e. draw s of pdeip_philox_normals(n, S, d, seed, particle_offset, step_offset); else injected
 * normals [N][S][d].  traj: NULL for terminal-only, else sample s is emitted iff s % emit_every == emit_offset, in the
 * four K1 trajectory layouts with C = d components per sample, or C = 2d with emit_drift: [x, grad U(x)] (the drift
 * step s+1 evaluates anyway; the last sample takes one extra evaluation).  A PDEIP_TRAJ_BLOCK128 trajectory is directly
 * a PDEIP_LAYOUT_BLOCK128 FP point set, with PDEIP_DRIFT_IN_POINTS when the drift is emitted.
 * Drifts: PDEIP_DRIFT_NONE / _LINEAR / _GMM / _MEANFIELD, fp32 on the CUDA cores (rtol 1e-5 class).  PDEIP_PATH_TENSOR
 * with the GMM drift, d = 8, 16 or 32, 1 <= n_gaussian <= 64, Philox noise, AOS state with x_last, emit_every 1,
 * emit_offset 0 and either traj == NULL (terminal state only, n arbitrary) or a PDEIP_TRAJ_BLOCK128 /
 * PDEIP_TRAJ_TIME_SOA trajectory with emit_drift runs the centre contraction and the softmax-weighted centre sum on
 * tcgen05 (K1-T-OD, bf16 hi + lo split operands, "bf16 GEMM path", rtol 1e-2 class); every other call takes the fp32
 * kernel, bit-identical to PDEIP_PATH_FP32 (PDEIP_NO_TC_INTEGRATOR=1 forces it).  PDEIP_DRIFT_MEANFIELD_TABLE encodes the underdamped mean recursion and is rejected
 * (PDEIP_ERR_UNSUPPORTED).  Rejected before any CUDA call, with a pdeip_last_error message: unknown drift kind, path or
 * layout, NULL x0 or drift_params, n_steps < 1, bad emit_every / emit_offset (PDEIP_ERR_INVALID_ARG), BLOCK128 with
 * n % 128 != 0 (PDEIP_ERR_INVALID_ARG), d outside [1, 32] (PDEIP_ERR_UNSUPPORTED).
 * ------------------------------------------------------------------------------------------- */
int pdeip_overdamped_integrate(const float* x0, float* x_last, float* traj, int64_t n_particles, int d, int n_steps,
                               float dt, int drift_kind, const float* drift_params, int n_gaussian, float sigma,
                               const float* noise, uint64_t seed, uint64_t particle_offset, uint32_t step_offset,
                               int state_layout, int traj_layout, int emit_every, int emit_offset, int emit_drift,
                               int path, void* stream);

/* K1-OD with grad U = grad V_theta of a hypothesis model, with the envelope and rejections of pdeip_kl_integrate_model:
 *   PDEIP_MODEL_MLP       hidden == 32, 1 <= layers <= 8, d <= 32, fp32 on the CUDA cores.  PDEIP_PATH_TENSOR with
 *                         layers == 2, d = 8, 16 or 32, Philox noise, AOS state, emit_every 1 and either traj == NULL
 *                         (terminal state only, n arbitrary) or a PDEIP_TRAJ_BLOCK128 / PDEIP_TRAJ_TIME_SOA trajectory
 *                         with emit_drift runs the six GEMMs of a step on tcgen05 (K1-MT, bf16 hi + lo split operands);
 *                         every other call takes the fp32 kernel, bit-identical to PDEIP_PATH_FP32
 *                         (PDEIP_NO_TC_INTEGRATOR=1 forces it);
 *   PDEIP_MODEL_GMM       exactly pdeip_overdamped_integrate(PDEIP_DRIFT_GMM, params, n_gaussian, 1.0f, ...);
 *   PDEIP_MODEL_QUADRATIC grad V = (K + K^T) y + b, fp32 on both paths. */
int pdeip_overdamped_integrate_model(const float* x0, float* x_last, float* traj, int64_t n_particles, int d,
                                     int n_steps, float dt, int model_kind, const float* params, int hidden, int layers,
                                     int n_gaussian, const float* noise, uint64_t seed, uint64_t particle_offset,
                                     uint32_t step_offset, int state_layout, int traj_layout, int emit_every,
                                     int emit_offset, int emit_drift, int path, void* stream);

/* Mean-field drift (interacting system, README.md:54-62): the ensemble mean on the common time grid obeys
 *   pbar' = (1 - gamma dt) pbar + sqrt(2 dt) xibar_s,  qbar' = qbar + dt pbar'   (the interaction cancels in the mean),
 * xibar_s = mean over ALL particles of the step-s Philox normals.  noise_sums accumulates (atomically, caller zeroes)
 * sums [(n_steps+1)*d + 2d] doubles over this rank's particles: [s][i] = sum xi_{s,i}, then sum q0 (d), sum p0 (d);
 * after ONE all-reduce(sum) over ranks, xbar_table turns them into xbar [n_steps+1][d] (nullable; mean position before
 * step s) and drift_table [n_steps+1][d] = A xbar_s, the tail of the PDEIP_DRIFT_MEANFIELD_TABLE parameter block.
 * No per-step exchange of sum x is needed: S exchanges collapse into that one all-reduce. */
int pdeip_meanfield_noise_sums(const float* z0, int64_t n_particles, int d, int n_steps, uint64_t seed,
                               uint64_t particle_offset, uint32_t step_offset, double* sums, void* stream);
int pdeip_meanfield_xbar_table(const double* sums, int64_t n_global, int d, int n_steps, float dt, float gamma,
                               const float* A, float* xbar, float* drift_table, void* stream);

/* the normals / uniforms pdeip_kl_integrate draws in Philox mode (for parity tests):
 * normals [N][n_draws][d] for steps step_offset..step_offset+n_draws-1; uniforms [N] (tau0/dt). */
int pdeip_philox_normals(float* out, int64_t n_particles, int n_draws, int d, uint64_t seed,
                         uint64_t particle_offset, uint32_t step_offset, void* stream);
int pdeip_philox_uniforms(float* out, int64_t n_particles, uint64_t seed, uint64_t particle_offset,
                          void* stream);
/* raw Philox4x32-10 blocks (known-answer test): ctr [n][4], key [2] -> out [n][4] (all uint32) */
int pdeip_philox_raw(const uint32_t* ctr, const uint32_t* key, uint32_t* out, int64_t n, void* stream);

/* initial ensemble  z = mu + cov_half xi          replaces core/distribution.py:64-65
 * out [N][dim] AOS or [dim][N] SOA; cov_half row-major [dim][dim] (NULL -> identity); mu NULL -> 0 */
int pdeip_gaussian_sample(float* out, int64_t n, int dim, const float* mu, const float* cov_half,
                          uint64_t seed, uint64_t particle_offset, int layout, void* stream);

/* exact samplers feeding the residual in "online / exact" mode.
 * grouped: sample p of group g = p / per_group is mus[g] + cov_halves[g] xi    (mus [G][dim], cov_halves
 *   [G][dim][dim]; replaces Gaussian(mean_t, cov_t).sample per time stamp,
 *   example_problems/kinetic_fokker_planck_example_OU.py:140-190);  out [G*per_group][dim].
 * ou_exact: overdamped OU at a per-sample random time t ~ U(t_min, t_max), closed form in the eigenbasis of F
 *   (example_problems/fokker_planck_example.py:48-55,84-96): U [d][d], s [d], B0 = U^T P0 U, B = U^T L U,
 *   mt0 = U^T m0;  out [n][d], out_t [n] (nullable). */
int pdeip_gaussian_sample_grouped(float* out, int64_t n_groups, int per_group, int dim, const float* mus,
                                  const float* cov_halves, uint64_t seed, uint64_t particle_offset, void* stream);
int pdeip_ou_exact_sample(float* out, float* out_t, int64_t n, int d, const float* U, const float* s,
                          const float* B0, const float* B, const float* mt0, float t_min, float t_max,
                          uint64_t seed, uint64_t particle_offset, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K2  GMM potential value / gradient.       replaces core/potential.py:32-61
 *   a_k = -|x - mu_k|^2 / (2 sigma^2);  U = -logsumexp(a);  grad U = (x - sum_k softmax(a)_k mu_k)/sigma^2
 * x [n][d]; out_value [n] (nullable); out_grad [n][d] (nullable).
 * ------------------------------------------------------------------------------------------- */
int pdeip_gmm_value_grad(const float* x, const float* mus, int n_gaussian, float sigma,
                         float* out_value, float* out_grad, int64_t n, int d, void* stream);
/* linear drift  out = x A^T  (QuadraticPotential.gradient with mu = 0, core/potential.py:20-24) */
int pdeip_linear_grad(const float* x, const float* A, float* out, int64_t n, int d, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Model evaluation (forward_fn / jax.grad / hessian_vector_product of one model at many points).
 *   replaces core/model.py:51-62 under jax.vmap(jax.grad) and utils/common_utils.py:6-14
 * x [n][d]; v [n][d] nullable; out_value [n], out_grad [n][d], out_vHv [n] (v'Hv), out_lap [n]
 * (Laplacian, tr Hessian) — each nullable.  model_kind / params as in the residual kernels.
 * ------------------------------------------------------------------------------------------- */
int pdeip_model_eval(int model_kind, const float* params, int d, int hidden, int layers, int n_gaussian,
                     const float* x, const float* v, float* out_value, float* out_grad,
                     float* out_vHv, float* out_lap, int64_t n, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K3/K4/K5  self-consistency residual: loss terms + parameter gradient.
 *   replaces methods/consistency_instances/{kinetic_fokker_planck.py:11-69, fokker_planck.py:33-63,
 *   kinetic_mckean_vlasov.py:11-120} (value_and_grad_fn)
 * Protocol: begin (zero the accumulators) -> accumulate (once per point set / chunk, any number of
 * times) -> finalize (deterministic reduction to sums[PDEIP_NUM_SUMS] and grad[n_params]).
 * ------------------------------------------------------------------------------------------- */
int64_t pdeip_model_num_params(int model_kind, int d, int hidden, int layers, int n_gaussian);
size_t pdeip_residual_workspace_bytes(int model_kind, int d, int hidden, int layers, int n_gaussian);
int pdeip_residual_begin(void* workspace, size_t workspace_bytes, int model_kind, int d, int hidden,
                         int layers, int n_gaussian, void* stream);

/* One point set.  points: [n][dim] (AOS) or [dim][n] (SOA), dim = 2d (kinetic kinds) or d (FP kinds).
 * weight multiplies every per-point contribution (use 1 / global point count).
 * coef: KFP_0T -> gamma_friction;  *_BOUNDARY -> +-2/T;  FP_0T, KMV -> unused.
 * true_kind/true_params/true_n_gaussian/true_sigma: drift spec (PDEIP_DRIFT_LINEAR / _GMM / _NONE) of
 *   grad V_true, used by the *_0T kinds for sum|gV_true|^2 and "loss ground truth"; PDEIP_DRIFT_IN_POINTS: the points
 *   carry d extra components holding grad V_true (rows of dim + d floats / dim + d planes).
 * path: PDEIP_PATH_FP32 or PDEIP_PATH_TENSOR (MLP model 32 x 2; KFP_0T and FP_0T run on tcgen05 — FP_0T as d
 *   direction rows (x, e_i) per point stacked along the GEMM M dimension —, the boundary kinds stay fp32). */
int pdeip_residual_accumulate(void* workspace, size_t workspace_bytes, int set_kind, int model_kind,
                              const float* params, int d, int hidden, int layers, int n_gaussian,
                              const float* points, int64_t n_points, int layout, float weight, float coef,
                              int true_kind, const float* true_params, int true_n_gaussian, float true_sigma,
                              int path, void* stream);

/* KMV pairwise set (kinetic_mckean_vlasov.py:20-97):  pairs (i,j,t), Delta = x[j,t] - x[i,t].
 * xv [n][nt][2d]; G [n][nt][d] = mean_i grad Phi(Delta_ij) (from pdeip_kmv_mean_grad; nullable -> skip the
 * |G|^2 gradient term); c [n][nt] = d_ss log rho + (d_s log rho)^2 + gamma d_s log rho. weight = 1/(n*n*nt). */
size_t pdeip_kmv_workspace_bytes(int64_t n, int nt, int d);
/* out_G [n][nt][d]; out_Gtrue (nullable) = mean_i grad Phi_true(Delta_ij) with Phi_true = D' A D / 2 (true_A [d][d]) */
int pdeip_kmv_mean_grad(int model_kind, const float* params, int d, int hidden, int layers,
                        const float* xv, int64_t n, int nt, float* out_G, float* out_Gtrue,
                        const float* true_A, void* workspace, size_t workspace_bytes, void* stream);
/* accumulates the pair terms and, when G is given, mean|G|^2 + mean|G_true|^2 (loss) and mean|G_true - G|^2 */
int pdeip_residual_accumulate_kmv(void* workspace, size_t workspace_bytes, int model_kind, const float* params,
                                  int d, int hidden, int layers, const float* xv, int64_t n, int nt,
                                  const float* G, const float* G_true, const float* c, float weight, void* stream);

/* Reference set != batch (SURVEY.md §7.6): Delta = x[j,t] - ref[i,t], ref [m][nt][2d] (x part used), weight =
 * 1/(m*n*nt); ref == NULL -> the batch itself (m = n, the reference's choice, kinetic_mckean_vlasov.py:20-23).
 * A sub-sampled reference set is ref = xv, m < n (the first m trajectories). */
size_t pdeip_kmv_workspace_bytes_ref(int64_t n, int nt, int d, int64_t m);
int pdeip_kmv_mean_grad_ref(int model_kind, const float* params, int d, int hidden, int layers,
                            const float* xv, int64_t n, int nt, const float* ref, int64_t m, float* out_G,
                            float* out_Gtrue, const float* true_A, void* workspace, size_t workspace_bytes, void* stream);
int pdeip_residual_accumulate_kmv_ref(void* workspace, size_t workspace_bytes, int model_kind, const float* params,
                                      int d, int hidden, int layers, const float* xv, int64_t n, int nt,
                                      const float* ref, int64_t m, const float* G, const float* G_true, const float* c,
                                      float weight, void* stream);
/* Moment closure for PDEIP_MODEL_QUADRATIC (Phi = D'W D + b.D): the pair set against the full reference set equals the
 * pair set against its MEAN (ref = rbar [1][nt][2d], m = 1, weight 1/(n*nt)) plus
 *   loss += sum_jt 2 c_jt weight tr(W C_t),  dW += sum_jt 2 c_jt weight C_t,   C_t = cov of the reference x at t
 * (cov [nt][d][d], 1/m normalisation).  O(n) instead of O(n m) at any ensemble size. */
int pdeip_kmv_closure_correction(void* workspace, size_t workspace_bytes, const float* params, int d, int64_t n, int nt,
                                 const float* c, const float* cov, float weight, void* stream);
/* d_s log rho, d_ss log rho of the Gaussian x-marginal and c = d_ss + d_s^2 + gamma d_s on the device
 * (example_problems/kinetic_mckean_vlasov_example_quadratic.py:51-69,120-177).  coef [nt][3d + 2 + 2d^2] =
 * [mean1 | a1 | a2 | k1 | k2 | M1 | M2] per time stamp (host float64, once per time stamp):
 *   d_s = -a1.diff + k1 - diff'M1 diff/2,  d_ss = -a2.diff + k2 - diff'M2 diff/2,  diff = mean1 - x.
 * xv [n][nt][2d]; outputs (each nullable) are [nt][n] row-major, which the reference reshapes to [n][nt]
 * (kinetic_mckean_vlasov.py:57-72). */
int pdeip_kmv_density_terms(const float* xv, int64_t n, int nt, int d, const float* coef, float gamma,
                            float* out_c, float* out_ps, float* out_ps2, void* stream);

/* loss assembly: loss = G2 - 2 D2 + 2 gamma_or_1 * D1 + GTRUE2 + BOUNDARY  (coefficients already folded in
 * by accumulate, see csrc/residual_common.cuh); sums/grad are device buffers. */
int pdeip_residual_finalize(void* workspace, size_t workspace_bytes, int model_kind, int d, int hidden,
                            int layers, int n_gaussian, float* sums, float* grad, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K6  optimizer step.     replaces main.py:20-26 (add_decayed_weights + adam) and core/trainer.py:61-70,110
 *   g <- grad_scale*g + wd p;  m,v Adam moments; p <- p - lr * mhat/(sqrt(vhat)+eps), bias correction with
 *   `count` (= 1-based update index);  optional EMA: ema <- decay ema + (1-decay) p_new, p <- ema.
 *   norms[0] = ||grad_scale*g||_2 (before weight decay), norms[1] = ||p_new||_2 (trainer.py:110).
 * ------------------------------------------------------------------------------------------- */
int pdeip_adam_l2_step(float* params, const float* grad, float* m, float* v, float* ema,
                       int64_t n, float lr, float b1, float b2, float eps, float weight_decay,
                       int64_t count, float grad_scale, int use_ema, float ema_decay,
                       float* norms, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K7  ensemble moments   sum z, sum z z^T   (validation against OU.py:73-93)
 * z [n][dim] (AOS) or [dim][n] (SOA); out [dim + dim*dim] raw sums (deterministic).
 * ------------------------------------------------------------------------------------------- */
size_t pdeip_moments_workspace_bytes(int dim);
int pdeip_ensemble_moments(const float* z, int64_t n, int dim, int layout, float* out,
                           void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * offline 0T sub-sampler (device gather).   replaces methods/consistency.py:102-118
 * dataset [n_traj][n_time][dim]; sample_index [n_sel] (int64); time index t_k = k*interval + shift,
 * k < n_time_sel.  out [n_sel*n_time_sel][dim].
 * ------------------------------------------------------------------------------------------- */
int pdeip_gather_0T(const float* dataset, int64_t n_traj, int n_time, int dim, const int64_t* sample_index,
                    int64_t n_sel, int interval, int shift, int n_time_sel, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * self-test of the tcgen05 building blocks (one 128 x N x K bf16 GEMM through the helpers of csrc/umma.cuh);
 * mode 0: D = A B^T (K-major A [128][K], B [N][K]); 1: D = A B (B [K][N], transposed view); 2: D = A^T B
 * (A [K][128], B [K][N], both transposed views); 3: TMEM st/ld round trip.  status (device int) != 0 on timeout.
 * ------------------------------------------------------------------------------------------- */
/* Status of the PDEIP_PATH_TENSOR launches since the last query / pdeip_residual_begin: 0 = every tcgen05 phase
 * completed; bit 0 = a bounded mbarrier wait of the residual kernel timed out, bit 1 = of the integrator (results
 * invalid).  Read-and-clear; synchronises the stream.  The product path does not need to poll it:
 * pdeip_residual_begin clears both words and pdeip_residual_finalize writes NaN into sums and grad when either is
 * set, so the caller's NaN check on the loss (core/trainer.py:112) fires. */
int pdeip_tensor_path_status(void* stream, int* out_status);
int pdeip_debug_umma(int mode, const float* A, const float* B, float* D, int K, int N, int* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PDEIP_H_ */
