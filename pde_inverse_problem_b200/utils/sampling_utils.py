"""Mirror of utils/sampling_utils.py:25-52 on the K1 CUDA integrator, and its overdamped counterpart (K1-OD)."""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from .. import _lib as L
from .. import ops


def drift_spec(potential_grad):
    """Map the `potential_grad` callable the reference passes (Potential.gradient, GMM.py:120) to the drift of the
    C ABI: (drift kind, parameter tensor, n_gaussian, sigma) for an analytic Potential, (ModelSpec, flat parameters)
    for a core.potential.ModelPotential (a fitted hypothesis model)."""
    owner = getattr(potential_grad, "__self__", None)
    if owner is None or not hasattr(owner, "drift_spec"):
        raise NotImplementedError(
            "potential_grad must be the .gradient method of a pde_inverse_problem_b200.core.potential.Potential "
            "(GMMPotential, LinearPotential, QuadraticPotential, VoidPotential, or ModelPotential(net, params) for a "
            "fitted model's grad V_theta); arbitrary Python callables cannot run inside the fused CUDA integrator")
    return owner.drift_spec()


def underdamped_langevin_dynamics_scan(q0_p0: torch.Tensor, n_steps: int, dt: float, key, potential_grad,
                                       gamma_friction: float, *, noise: Optional[torch.Tensor] = None,
                                       tau0: Optional[torch.Tensor] = None, particle_offset: int = 0,
                                       traj_layout: int = L.TRAJ_PARTICLE_MAJOR, want_trajectory: bool = True,
                                       path: int = L.PATH_FP32,
                                       ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Returns (last_sample [N,2d], trajectory [N,n_steps,2d], tau_trajectory [N,n_steps]) exactly like the
    vmapped reference (sampling_utils.py:52).  `key` is an integer seed (the reference passes one jax key
    per particle; here the per-particle stream is Philox(seed, particle_offset + n)).  `noise`/`tau0` inject
    the random draws for parity runs.  `path`: the kernel path of pdeip_kl_integrate_path (see pdeip.h)."""
    spec = drift_spec(potential_grad)
    common = dict(noise=noise, tau0=tau0, seed=int(key), particle_offset=particle_offset,
                  schedule=L.SCHEDULE_REFERENCE, traj_layout=traj_layout, want_traj=want_trajectory, want_tau=True,
                  path=path)
    if isinstance(spec[0], ops.ModelSpec):
        model_spec, flat = spec
        return ops.kl_integrate_model(q0_p0, n_steps, float(dt), float(gamma_friction), model_spec, flat, **common)
    kind, params, n_gaussian, sigma = spec
    return ops.kl_integrate(q0_p0, n_steps, float(dt), float(gamma_friction), kind, params, n_gaussian=n_gaussian,
                            sigma=sigma, **common)


def overdamped_langevin_dynamics_scan(x0: torch.Tensor, n_steps: int, dt: float, key, potential_grad, *,
                                      noise: Optional[torch.Tensor] = None, particle_offset: int = 0,
                                      traj_layout: int = L.TRAJ_PARTICLE_MAJOR, want_trajectory: bool = True,
                                      path: int = L.PATH_FP32,
                                      ) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """Overdamped Langevin dX = -grad U(X) dt + sqrt(2) dW, the SDE of the Fokker-Planck instance, by n_steps
    Euler-Maruyama steps x' = x - dt grad U(x) + sqrt(2 dt) xi (pdeip_overdamped_integrate).  Returns (x_last [N,d],
    trajectory of the n_steps samples in `traj_layout` ([N,n_steps,d] by default), or None without want_trajectory); sample s is the state after
    step s.  `potential_grad` is what underdamped_langevin_dynamics_scan takes: the .gradient of an analytic Potential or
    of a ModelPotential(net, params).  `key` is an integer seed (Philox(seed, particle_offset + n)); `noise` [N,n_steps,d]
    injects the draws for parity runs."""
    spec = drift_spec(potential_grad)
    common = dict(noise=noise, seed=int(key), particle_offset=particle_offset, traj_layout=traj_layout,
                  want_traj=want_trajectory, path=path)
    if isinstance(spec[0], ops.ModelSpec):
        model_spec, flat = spec
        return ops.overdamped_integrate_model(x0, n_steps, float(dt), model_spec, flat, **common)
    kind, params, n_gaussian, sigma = spec
    return ops.overdamped_integrate(x0, n_steps, float(dt), kind, params, n_gaussian=n_gaussian, sigma=sigma,
                                    **common)
