"""CPU: pdeip_kl_integrate_model argument validation (no device), the dispatch of underdamped_langevin_dynamics_scan on
ModelPotential, and the float64 oracle of the fitted-model drift (torch.func.grad of the MLP) against finite
differences of V."""
import math

import pytest
import torch

from oracle import integrator as o_int
from oracle import model as o_model


def _call(lib, *, z0=1, d=4, model_kind=0, params=1, hidden=32, layers=2, n_gaussian=0):
    # z0 / params are never dereferenced: every case below is rejected before any CUDA call
    return lib.pdeip_kl_integrate_model(z0, None, None, None, 10, d, 5, 0.1, 1.0, model_kind, params, hidden, layers,
                                        n_gaussian, None, None, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, None)


def test_integrate_model_rejects_bad_arguments_without_gpu():
    from pde_inverse_problem_b200 import _lib as L
    lib = L.load()
    cases = [
        (dict(model_kind=7), -1, b"model kind"),
        (dict(layers=0), -2, b"layers"),
        (dict(layers=9), -2, b"layers"),
        (dict(d=33), -2, b"32"),
        (dict(params=None), -1, b"params"),
        (dict(model_kind=L.MODEL_GMM, n_gaussian=0), -1, b"n_gaussian"),
        (dict(hidden=20), -2, b"hidden"),
        (dict(z0=None), -1, b"z0"),
    ]
    for kw, code, msg in cases:
        assert _call(lib, **kw) == code, kw
        assert msg in lib.pdeip_last_error(), (kw, lib.pdeip_last_error())
    # the quadratic model takes no hidden / layers
    assert _call(lib, model_kind=L.MODEL_QUADRATIC, hidden=0, layers=0, z0=None) == -1
    assert b"z0" in lib.pdeip_last_error()


def _mlp(d=4, hidden=32, layers=2):
    from pde_inverse_problem_b200.core.model import V_hypothesis
    net = V_hypothesis(output_dim=1, hidden_dims=[hidden] * layers, dim=d)
    return net, net.init(11, torch.zeros(d))


def test_model_potential_routes_to_the_model_entry_point(monkeypatch):
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    from pde_inverse_problem_b200.core.potential import GMMPotential, ModelPotential
    from pde_inverse_problem_b200.utils import sampling_utils as su
    net, params = _mlp()
    pot = ModelPotential(net, params)
    spec, flat = su.drift_spec(pot.gradient)
    assert spec is net.spec and spec.kind == L.MODEL_MLP and spec.hidden == 32 and spec.layers == 2
    assert flat is params["_flat"]  # held by reference: in-place updates of the fit are followed
    calls = []
    monkeypatch.setattr(ops, "kl_integrate_model", lambda *a, **k: calls.append(("model", a, k)) or (None, None, None))
    monkeypatch.setattr(ops, "kl_integrate", lambda *a, **k: calls.append(("drift", a, k)) or (None, None, None))
    z0 = torch.zeros(8, 8)
    su.underdamped_langevin_dynamics_scan(z0, 5, 0.1, 3, pot.gradient, 0.5)
    (name, args, kw), = calls
    assert name == "model" and args[4] is net.spec and args[5] is params["_flat"]
    assert kw["path"] == L.PATH_FP32 and kw["seed"] == 3 and kw["want_tau"]
    su.underdamped_langevin_dynamics_scan(z0, 5, 0.1, 3, pot.gradient, 0.5, path=L.PATH_TENSOR)
    assert calls[-1][0] == "model" and calls[-1][2]["path"] == L.PATH_TENSOR
    # the analytic potentials keep their route
    su.underdamped_langevin_dynamics_scan(z0, 5, 0.1, 3, GMMPotential(torch.zeros(3, 4), 1.0).gradient, 0.5)
    assert calls[-1][0] == "drift" and calls[-1][1][4] == L.DRIFT_GMM and calls[-1][2]["path"] == L.PATH_FP32


def test_arbitrary_callable_still_raises():
    from pde_inverse_problem_b200.utils import sampling_utils as su
    with pytest.raises(NotImplementedError, match="ModelPotential"):
        su.underdamped_langevin_dynamics_scan(torch.zeros(4, 8), 5, 0.1, 0, lambda x: 2 * x, 0.5)
    with pytest.raises(NotImplementedError, match="ModelPotential"):
        su.drift_spec(torch.sin)


def _oracle_grad(params):
    """grad_x V of the float64 oracle MLP, batched (points are independent, so grad of the sum = per-point grads)."""
    return lambda x: torch.func.grad(lambda y: o_model.mlp_apply(params, y).sum())(x)


@pytest.mark.parametrize("d,hidden,layers", [(2, 32, 1), (8, 20, 2), (5, 32, 8)])
def test_oracle_model_drift_matches_finite_differences(d, hidden, layers):
    params = o_model.init_mlp_params(d, hidden, layers, seed=d + layers)
    grad = _oracle_grad(params)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(64, d, generator=g, dtype=torch.float64)
    gx = grad(x)
    fd = fd_grad(params, x)
    assert ((gx - fd).abs().max() / gx.abs().max()).item() < 1e-7
    # the oracle integrator takes the callable as it stands (utils/sampling_utils.py:6-52 with jax.grad(net.apply))
    n, S, dt, gamma = 64, 3, 0.01, 0.5
    z0 = torch.randn(n, 2 * d, generator=g, dtype=torch.float64)
    noise = torch.randn(n, S + 1, d, generator=g, dtype=torch.float64)
    tau0 = torch.rand(n, generator=g, dtype=torch.float64) * dt
    last, traj, _ = o_int.underdamped_langevin_dynamics_scan(z0, S, dt, noise, tau0, grad, gamma)
    # first step by hand: p' = p - h gradV(q) + sqrt(2h) xi - gamma h p ; q' = q + h p'
    q, p, h = z0[:, :d], z0[:, d:], tau0[:, None]
    p1 = p - h * fd_grad(params, q) + torch.sqrt(h) * math.sqrt(2.0) * noise[:, 0] - gamma * p * h
    assert torch.allclose(traj[:, 0, d:], p1, rtol=0, atol=1e-9)
    assert torch.allclose(traj[:, 0, :d], q + h * p1, rtol=0, atol=1e-9)
    assert traj.shape == (n, S, 2 * d) and torch.isfinite(last).all()


def fd_grad(params, x, h=1e-5):
    """central finite differences of the oracle V"""
    d = x.shape[1]
    out = torch.empty_like(x)
    for i in range(d):
        e = torch.zeros(d, dtype=x.dtype)
        e[i] = h
        out[:, i] = (o_model.mlp_apply(params, x + e)[0] - o_model.mlp_apply(params, x - e)[0]) / (2 * h)
    return out
