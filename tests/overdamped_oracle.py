"""Float64 definition of the overdamped Langevin integrator K1-OD (test infrastructure, like oracle/integrator.py for
the kinetic one), with the noise injected so that the CUDA kernel and this restatement consume identical draws:

    x_{s+1} = x_s - dt grad U(x_s) + sqrt(dt) sqrt(2) xi_s,   s = 0..S-1,   noise [N, S, d] = xi

Sample s is the state after step s; the last sample is the terminal state.
"""
from __future__ import annotations

import math
from typing import Callable, Tuple

import torch


def overdamped_langevin_scan(x0: torch.Tensor, n_steps: int, dt: float, noise: torch.Tensor,
                             potential_grad: Callable) -> Tuple[torch.Tensor, torch.Tensor]:
    """Returns (last [N,d], traj [N,S,d]) particle-major; potential_grad maps [N,d] -> [N,d]."""
    n, d = x0.shape
    assert noise.shape == (n, n_steps, d), noise.shape
    x = x0.clone()
    sq = math.sqrt(dt) * math.sqrt(2.0)
    traj = []
    for s in range(n_steps):
        x = x - dt * potential_grad(x) + sq * noise[:, s]
        traj.append(x)
    return x, torch.stack(traj, 1)


def linear_moment_recursion(F: torch.Tensor, m0: torch.Tensor, P0: torch.Tensor, n_steps: int, dt: float):
    """Exact mean and covariance of the scheme under grad U = F x from x0 ~ (m0, P0):
    m' = (I - dt F) m,  P' = (I - dt F) P (I - dt F)^T + 2 dt I."""
    A = torch.eye(F.shape[0], dtype=F.dtype) - dt * F
    m, P = m0.clone(), P0.clone()
    for _ in range(n_steps):
        m = A @ m
        P = A @ P @ A.T + 2.0 * dt * torch.eye(F.shape[0], dtype=F.dtype)
    return m, P
