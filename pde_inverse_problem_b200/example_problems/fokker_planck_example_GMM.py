"""The Fokker-Planck instance under a Gaussian-mixture potential: dX = -grad V(X) dt + sqrt(2) dW with V the GMM
potential of the kinetic GMM instance (kinetic_fokker_planck_example_GMM.py).  Its law has no closed form, so the
ground truth is sampled through the SDE with the overdamped integrator K1-OD, as the kinetic GMM instance samples its
own (GMM.py:104-142).  Selected by pde_instance.potential = "GMM" on the "fokker_planck" configuration."""
from __future__ import annotations

from math import prod

import torch

from .. import _lib as L
from .. import ops
from ..api import ProblemInstance
from ..core.distribution import Gaussian
from ..core.potential import GMMPotential
from ..utils import rng as jrandom
from ..utils.sampling_utils import overdamped_langevin_dynamics_scan


def initialize_configuration(domain_dim: int, rng, n_Gaussian: int = 3, device="cuda"):
    """mus ~ U[-4, 4]^d from a torch generator seeded by `rng` (as the kinetic GMM instance), sigma = 1, initial law
    N(0, 4 I) (the x-block of the kinetic instance's).  No gamma_friction: the dynamics are overdamped."""
    g = torch.Generator().manual_seed(int(rng) & 0x7FFFFFFFFFFFFFFF)
    mus = (torch.rand(n_Gaussian, domain_dim, generator=g, dtype=torch.float64) * 8.0 - 4.0).float()
    return {
        "n_Gaussian": n_Gaussian,
        "m_0": torch.zeros(domain_dim).to(device), "P_0": torch.diag(torch.full((domain_dim,), 4.0)).to(device),
        "GMM": {"mus": mus.to(device).contiguous()},
    }


class OverdampedTerminal:
    """The terminal law of the instance: .sample(n, rng) integrates n particles drawn from the initial law to the
    terminal time (terminal state only, the instance's n_steps)."""

    def __init__(self, pde_instance):
        self.pde_instance = pde_instance

    def sample(self, batch_size: int, key):
        pde = self.pde_instance
        rng_init, rng_sde = jrandom.split(key)
        x0 = pde.distribution_initial.sample(batch_size, rng_init)
        x_T, _ = overdamped_langevin_dynamics_scan(x0, pde.n_steps, pde.total_evolving_time / pde.n_steps, rng_sde,
                                                   pde.potential.gradient, want_trajectory=False)
        return x_T


class FokkerPlanckGMM(ProblemInstance):
    def __init__(self, cfg, rng, device="cuda"):
        super().__init__(cfg, rng, device)
        rng_initial_config, _ = jrandom.split(rng)
        self.initial_configuration = initialize_configuration(
            cfg.pde_instance.domain_dim, rng_initial_config, n_Gaussian=int(cfg.pde_instance.get("n_gaussian", 3)),
            device=self.device)
        self.n_steps = int(cfg.pde_instance.get("n_steps", 100))
        self.potential = GMMPotential(self.initial_configuration["GMM"]["mus"], 1.0)
        self.sample_scheme = "SDE"
        self.sample_mode = cfg.pde_instance.get("sample_mode", "online")
        if self.sample_mode != "online":
            raise NotImplementedError(f"the Fokker-Planck GMM instance samples online only (sample_mode "
                                      f"{self.sample_mode!r}: it has no offline dataset)")
        self.distribution_initial = Gaussian(self.initial_configuration["m_0"], self.initial_configuration["P_0"])
        self.distribution_terminal = OverdampedTerminal(self)

    def V_true_fn(self, x: torch.Tensor):
        if x.ndim in (1, 2):
            return self.potential.value(x)
        raise ValueError("x should be either 1D (unbatched) or 2D (batched) array.")

    def true_grad_spec(self):
        return ops.TrueGrad(L.DRIFT_GMM, self.potential.mus, sigma=self.potential.sigma)

    def sample_ground_truth(self, rng, batch_size: int):
        """(initial, terminal, 0T) as the kinetic GMM instance draws them (GMM.py:104-142) with the overdamped
        integrator: 0T = all n_steps samples of batch_size trajectories ([batch_size * n_steps, d]), initial = 30 x
        batch_size draws of the initial law, terminal = the terminal states of 30 x batch_size more trajectories."""
        rng, rng2, rng_init, rng_init2, rng_init3 = jrandom.split(rng, 5)
        multiple_init = 30
        multiple_terminal = 30
        dt = self.total_evolving_time / self.n_steps
        x0 = self.distribution_initial.sample(batch_size, rng_init)
        _, sample_0T = overdamped_langevin_dynamics_scan(x0, self.n_steps, dt, rng, self.potential.gradient)
        sample_0T = sample_0T.reshape((prod(sample_0T.shape[:2]), *sample_0T.shape[2:]))
        sample_initial = self.distribution_initial.sample(batch_size * multiple_init, rng_init2)
        x02 = self.distribution_initial.sample(batch_size * multiple_terminal, rng_init3)
        sample_final, _ = overdamped_langevin_dynamics_scan(x02, self.n_steps, dt, rng2, self.potential.gradient,
                                                            want_trajectory=False)
        return sample_initial, sample_final, sample_0T
