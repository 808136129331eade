"""Distribution-level validation of a fitted potential on the kinetic and the Fokker-Planck instances: simulate the
particles under the fitted drift and under the true one, synchronously coupled.

The integrator's noise is counter-based (Philox keyed by seed, global particle id and step), so two runs from the same
initial ensemble with the same seed share every Brownian increment and every initial time shift.  The RMS distance
between the coupled terminal states is then an upper bound on the W2 distance between the true and the fitted terminal
laws.  The kinetic instances run the underdamped integrator, the Fokker-Planck instance (no `gamma_friction` in its
configuration) the overdamped one.  The reference has no such metric (its kinetic test_fn is commented out); this module
is not wired into test_fn.
"""
from __future__ import annotations

import functools
from typing import Dict, Optional

import torch

from .. import _lib as L
from .. import ops
from ..core.model import model_of
from ..core.potential import ModelPotential
from . import rng as jrandom
from .sampling_utils import overdamped_langevin_dynamics_scan, underdamped_langevin_dynamics_scan


def _instance_n_steps(pde_instance) -> int:
    """The step count the instance integrates its own terminal samples with: the offline GMM dataset uses
    n_steps_terminal, online sampling n_steps (kinetic_fokker_planck_example_GMM.py)."""
    cfg = pde_instance.cfg.pde_instance
    if getattr(cfg, "sample_mode", "online") == "offline":
        return int(cfg.n_steps_terminal)
    return int(cfg.n_steps)


def _mean_cov(z: torch.Tensor):
    s1, s2 = ops.ensemble_moments(z)
    n = z.shape[0]
    mean = s1 / n
    return mean, s2 / n - torch.outer(mean, mean)


def coupled_simulation_error(pde_instance, forward_fn, n_particles: int, rng, n_steps: Optional[int] = None,
                             path: int = L.PATH_FP32) -> Dict[str, torch.Tensor]:
    """Integrate one initial ensemble (drawn from pde_instance.distribution_initial) to the terminal time twice, with
    the same seed: under pde_instance.potential and under the fitted model `forward_fn` (= functools.partial(net.apply,
    params), as test_fn receives it).  dt = total_evolving_time / n_steps, n_steps defaults to the instance's own on the
    kinetic instances; the Fokker-Planck instance has no step count of its own, so there n_steps is required.

    Returns 0-d CUDA tensors (no host synchronisation; every reduction is one ensemble_moments call), over the full
    state ((x, v) on the kinetic instances, x on the Fokker-Planck one):
      "coupled rms distance terminal"      sqrt(mean |z_true - z_fit|^2)  (>= W2 of the two terminal laws)
      "relative mean error terminal"       |mean_fit - mean_true| / |mean_true|
      "relative covariance error terminal" |C_fit - C_true|_F / |C_true|_F
    """
    potential = getattr(pde_instance, "potential", None)
    if potential is None or not hasattr(pde_instance, "distribution_initial"):
        raise NotImplementedError("coupled_simulation_error needs an instance with a true `potential` "
                                  "(kinetic Fokker-Planck, GMM or OU, or Fokker-Planck)")
    if not isinstance(forward_fn, functools.partial) or not forward_fn.args:
        raise NotImplementedError("forward_fn must be functools.partial(net.apply, params), as test_fn receives it")
    net, params = model_of(forward_fn), forward_fn.args[0]
    overdamped = "gamma_friction" not in pde_instance.initial_configuration
    if n_steps is None:
        if overdamped:
            raise ValueError("n_steps is required on the Fokker-Planck instance: its configuration has no step count")
        n_steps = _instance_n_steps(pde_instance)
    n_steps = int(n_steps)
    dt = float(pde_instance.total_evolving_time) / n_steps
    rng_init, rng_sde = jrandom.split(rng)
    z0 = pde_instance.distribution_initial.sample(n_particles, rng_init)
    fitted = ModelPotential(net, params).gradient
    if overdamped:
        z_true, _ = overdamped_langevin_dynamics_scan(z0, n_steps, dt, rng_sde, potential.gradient,
                                                      want_trajectory=False, path=path)
        z_fit, _ = overdamped_langevin_dynamics_scan(z0, n_steps, dt, rng_sde, fitted, want_trajectory=False, path=path)
    else:
        gamma = float(pde_instance.initial_configuration["gamma_friction"])
        z_true, _, _ = underdamped_langevin_dynamics_scan(z0, n_steps, dt, rng_sde, potential.gradient, gamma,
                                                          want_trajectory=False, path=path)
        z_fit, _, _ = underdamped_langevin_dynamics_scan(z0, n_steps, dt, rng_sde, fitted, gamma,
                                                         want_trajectory=False, path=path)
    _, diff_second = ops.ensemble_moments(z_true - z_fit)
    rms = torch.sqrt(torch.trace(diff_second) / n_particles)
    m_true, c_true = _mean_cov(z_true)
    m_fit, c_fit = _mean_cov(z_fit)
    tiny = torch.finfo(torch.float32).tiny
    return {
        "coupled rms distance terminal": rms,
        "relative mean error terminal": torch.linalg.vector_norm(m_fit - m_true)
        / torch.linalg.vector_norm(m_true).clamp_min(tiny),
        "relative covariance error terminal": torch.linalg.matrix_norm(c_fit - c_true)
        / torch.linalg.matrix_norm(c_true).clamp_min(tiny),
    }
