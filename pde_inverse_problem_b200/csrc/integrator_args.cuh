// integrator_args.cuh — argument block shared by the K1 kernels (integrator.cu, integrator_tc.cu).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "philox.cuh"

namespace pdeip {

struct IntegrateArgs {
  const float* z0;
  float* z_last;
  float* traj;
  float* tau;
  int64_t n;
  int d;
  int n_steps;
  float dt;
  float gamma;
  const float* drift_params;
  int n_gaussian;
  float inv_sigma2;
  int layers;  // hidden layers of the MLP hypothesis model (pdeip_kl_integrate_model)
  const float* noise;
  const float* tau0;
  uint64_t seed;
  uint64_t particle_offset;
  uint32_t step_offset;
  int schedule;
  int state_layout;
  int traj_layout;
  int emit_every;
  int emit_offset;
  int s_emit;  // number of emitted samples
  int emit_drift;  // 1: every emitted sample carries grad U(x) as components [2d, 3d)
  PhiloxRoundKeys rk;  // round keys of `seed`
};

// integrator_tc.cu: GMM drift on the tensor cores (PDEIP_PATH_TENSOR)
bool integrate_tensor_ok(const IntegrateArgs& a, int drift_kind);
int launch_integrate_tensor(const IntegrateArgs& a, cudaStream_t st);

// integrator_mlp_tc.cu: MLP (32 x 2) drift on the tensor cores (PDEIP_PATH_TENSOR of pdeip_kl_integrate_model)
bool integrate_mlp_tensor_ok(const IntegrateArgs& a);
int launch_integrate_mlp_tensor(const IntegrateArgs& a, cudaStream_t st);
// ... and its overdamped variant (PDEIP_PATH_TENSOR of pdeip_overdamped_integrate_model)
bool overdamped_mlp_tensor_ok(const IntegrateArgs& a);
int launch_overdamped_mlp_tensor(const IntegrateArgs& a, cudaStream_t st);

}  // namespace pdeip
