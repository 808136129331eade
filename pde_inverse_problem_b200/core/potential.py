"""Mirror of core/potential.py on the K2 CUDA kernels."""
from __future__ import annotations

import warnings

import torch

from .. import _lib as L
from .. import ops


class Potential(object):
    """core/potential.py:6-8."""

    def gradient(self, x: torch.Tensor):
        raise NotImplementedError

    def drift_spec(self):
        raise NotImplementedError


class QuadraticPotential(Potential):
    """core/potential.py:11-24: gradient = inv(cov) (x - mu)."""

    def __init__(self, mu: torch.Tensor, cov: torch.Tensor):
        assert mu.ndim == 1 and cov.ndim == 2 and cov.shape[0] == cov.shape[1] and cov.shape[0] == mu.shape[0]
        warnings.warn("cov is assumed to be positive definite!")
        self.dim = mu.shape[0]
        self.mu = mu
        self.cov = cov
        self.inv_cov = torch.linalg.inv(cov.double()).float().contiguous()  # host-side setup, once

    def gradient(self, x):
        if x.ndim == 1:
            return ops.linear_grad((x - self.mu)[None].contiguous(), self.inv_cov)[0]
        return ops.linear_grad((x - self.mu).contiguous(), self.inv_cov)

    def drift_spec(self):
        params = torch.cat([self.inv_cov.reshape(-1), self.mu.reshape(-1)]).contiguous()
        return L.DRIFT_MEANFIELD, params, 0, 1.0


class LinearPotential(Potential):
    """U = x^T A x / 2 with symmetric A: gradient A x (kinetic OU drift tilde_F x,
    example_problems/kinetic_fokker_planck_example_OU.py:15-20,130-131)."""

    def __init__(self, A: torch.Tensor):
        self.A = A.contiguous()
        self.dim = A.shape[0]

    def gradient(self, x):
        if x.ndim == 1:
            return ops.linear_grad(x[None].contiguous(), self.A)[0]
        return ops.linear_grad(x, self.A)

    def drift_spec(self):
        return L.DRIFT_LINEAR, self.A, 0, 1.0


class VoidPotential(Potential):
    """core/potential.py:27-29."""

    def gradient(self, x: torch.Tensor):
        return torch.zeros_like(x)

    def drift_spec(self):
        return L.DRIFT_NONE, None, 0, 1.0


class GMMPotential(Potential):
    """core/potential.py:48-61 (uniform weights, shared sigma)."""

    def __init__(self, mus: torch.Tensor, sigma):
        self.mus = mus.contiguous()
        self.sigma = float(sigma)

    def value(self, x):
        if x.ndim == 1:
            return ops.gmm_value_grad(x[None].contiguous(), self.mus, self.sigma, want_value=True,
                                      want_grad=False)[0][0]
        return ops.gmm_value_grad(x, self.mus, self.sigma, want_value=True, want_grad=False)[0]

    def gradient(self, x):
        if len(x.shape) == 1:
            return ops.gmm_value_grad(x[None].contiguous(), self.mus, self.sigma)[1][0]
        return ops.gmm_value_grad(x, self.mus, self.sigma)[1]

    def drift_spec(self):
        return L.DRIFT_GMM, self.mus, int(self.mus.shape[0]), self.sigma


class ModelPotential(Potential):
    """The potential V_theta of a fitted hypothesis model: `net` is a core.model model (V_hypothesis /
    V_parametric_GMM / V_parametric_quadratic), `params` its parameter tree.  What the reference gets from
    jax.grad(lambda x: net.apply(params, x)[0]): passing `ModelPotential(net, params).gradient` as `potential_grad`
    to utils.sampling_utils.underdamped_langevin_dynamics_scan integrates the particles under the fitted drift
    (pdeip_kl_integrate_model).

    The parameter tree is held by reference and its flat buffer is looked up at every call.  The trainer updates
    params["_flat"] in place, so one instance follows the fit; copy the tree to freeze a snapshot."""

    def __init__(self, net, params):
        self.net = net
        self.params = params
        self.dim = net.spec.d

    def value(self, x):
        if x.ndim == 1:
            return self.net.apply(self.params, x)[0]
        return self.net.apply(self.params, x)

    def gradient(self, x):
        if x.ndim == 1:
            return self.net.gradient(self.params, x[None].contiguous())[0]
        return self.net.gradient(self.params, x)

    def drift_spec(self):
        """(ModelSpec, flat parameter buffer) of pdeip_kl_integrate_model."""
        return self.net.spec, self.net.flat(self.params)
