"""CPU: the overdamped integrator K1-OD (pdeip_overdamped_integrate*): exported symbols, argument validation before any
CUDA call, the dispatch of overdamped_langevin_dynamics_scan and coupled_simulation_error, and known answers of the
float64 definition (tests/overdamped_oracle.py) under the linear drift."""
import math

import pytest
import torch

from overdamped_oracle import linear_moment_recursion, overdamped_langevin_scan


def test_overdamped_entry_points_declared_bound_and_registered():
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import torch_ops
    names = set(L.header_functions())
    assert {"pdeip_overdamped_integrate", "pdeip_overdamped_integrate_model"} <= names
    assert names == set(L.SIGNATURES)
    lib = L.load()  # binds every declared symbol, or raises
    assert lib.pdeip_overdamped_integrate and lib.pdeip_overdamped_integrate_model
    assert {"overdamped_integrate", "overdamped_integrate_model"} <= set(torch_ops.REGISTERED)


def _call(lib, *, x0=1, traj=None, n=10, d=4, n_steps=5, drift_kind=1, drift_params=1, n_gaussian=0, sigma=1.0,
          state_layout=0, traj_layout=0, emit_every=1, emit_offset=0, path=0):
    # x0 / drift_params are never dereferenced: every case below is rejected before any CUDA call
    return lib.pdeip_overdamped_integrate(x0, None, traj, n, d, n_steps, 0.01, drift_kind, drift_params, n_gaussian,
                                          sigma, None, 0, 0, 0, state_layout, traj_layout, emit_every, emit_offset, 0,
                                          path, None)


def _call_model(lib, *, x0=1, d=4, model_kind=0, params=1, hidden=32, layers=2, n_gaussian=0, state_layout=0):
    return lib.pdeip_overdamped_integrate_model(x0, None, None, 10, d, 5, 0.01, model_kind, params, hidden, layers,
                                                n_gaussian, None, 0, 0, 0, state_layout, 0, 1, 0, 0, 0, None)


def test_overdamped_rejects_bad_arguments_without_gpu():
    from pde_inverse_problem_b200 import _lib as L
    lib = L.load()
    cases = [
        (dict(x0=None), -1, b"x0"),
        (dict(drift_params=None), -1, b"drift_params"),
        (dict(d=0), -2, b"d=0"),
        (dict(d=33), -2, b"d=33"),
        (dict(state_layout=1), -1, b"state layout"),
        (dict(traj_layout=4), -1, b"trajectory layout"),
        (dict(traj=1, traj_layout=L.TRAJ_BLOCK128, n=200), -1, b"BLOCK128"),
        (dict(drift_kind=L.DRIFT_MEANFIELD_TABLE), -2, b"MEANFIELD_TABLE"),
        (dict(drift_kind=L.DRIFT_IN_POINTS), -1, b"drift kind"),
        (dict(drift_kind=L.DRIFT_GMM, n_gaussian=0), -1, b"n_gaussian"),
        (dict(n_steps=0), -1, b"n_steps"),
        (dict(emit_every=2, emit_offset=2), -1, b"emit_every"),
        (dict(path=5), -1, b"path"),
    ]
    for kw, code, msg in cases:
        assert _call(lib, **kw) == code, kw
        assert msg in lib.pdeip_last_error(), (kw, lib.pdeip_last_error())
    model_cases = [
        (dict(model_kind=7), -1, b"model kind"),
        (dict(params=None), -1, b"params"),
        (dict(layers=0), -2, b"layers"),
        (dict(layers=9), -2, b"layers"),
        (dict(hidden=20), -2, b"hidden"),
        (dict(d=33), -2, b"32"),
        (dict(model_kind=L.MODEL_GMM, n_gaussian=0), -1, b"n_gaussian"),
        (dict(x0=None), -1, b"x0"),
        (dict(model_kind=L.MODEL_QUADRATIC, hidden=0, layers=0, state_layout=1), -1, b"state layout"),
    ]
    for kw, code, msg in model_cases:
        assert _call_model(lib, **kw) == code, kw
        assert msg in lib.pdeip_last_error(), (kw, lib.pdeip_last_error())


def test_overdamped_scan_routes_every_potential(monkeypatch):
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    from pde_inverse_problem_b200.core.model import V_hypothesis
    from pde_inverse_problem_b200.core.potential import LinearPotential, ModelPotential
    from pde_inverse_problem_b200.utils import sampling_utils as su
    net = V_hypothesis(output_dim=1, hidden_dims=[32, 32], dim=4)
    params = net.init(11, torch.zeros(4))
    calls = []
    monkeypatch.setattr(ops, "overdamped_integrate_model", lambda *a, **k: calls.append(("model", a, k)) or (None, None))
    monkeypatch.setattr(ops, "overdamped_integrate", lambda *a, **k: calls.append(("drift", a, k)) or (None, None))
    x0 = torch.zeros(8, 4)
    su.overdamped_langevin_dynamics_scan(x0, 5, 0.1, 3, ModelPotential(net, params).gradient, path=L.PATH_TENSOR)
    (name, args, kw), = calls
    assert name == "model" and args[3] is net.spec and args[4] is params["_flat"]
    assert kw["path"] == L.PATH_TENSOR and kw["seed"] == 3 and kw["want_traj"]
    A = torch.eye(4)
    su.overdamped_langevin_dynamics_scan(x0, 5, 0.1, 3, LinearPotential(A).gradient, want_trajectory=False)
    name, args, kw = calls[-1]
    assert name == "drift" and args[3] == L.DRIFT_LINEAR and args[4] is A and kw["path"] == L.PATH_FP32
    assert not kw["want_traj"]
    with pytest.raises(NotImplementedError, match="ModelPotential"):
        su.overdamped_langevin_dynamics_scan(x0, 5, 0.1, 0, lambda x: 2 * x)


def test_coupled_simulation_error_needs_n_steps_on_the_fp_instance():
    import functools
    import types
    from pde_inverse_problem_b200.core.model import V_hypothesis
    from pde_inverse_problem_b200.core.potential import LinearPotential
    from pde_inverse_problem_b200.utils.simulation import coupled_simulation_error
    net = V_hypothesis(output_dim=1, hidden_dims=[32, 32], dim=4)
    params = net.init(1, torch.zeros(4))
    fp_like = types.SimpleNamespace(potential=LinearPotential(torch.eye(4)), distribution_initial=object(),
                                    initial_configuration={"F": torch.eye(4)}, total_evolving_time=2.0)
    with pytest.raises(ValueError, match="n_steps"):
        coupled_simulation_error(fp_like, functools.partial(net.apply, params), 128, rng=0)


def _F(d, seed=3):
    g = torch.Generator().manual_seed(seed)
    B = torch.randn(d, d + 1, generator=g, dtype=torch.float64)
    return B @ B.T / d


def test_oracle_is_linear_in_initial_state_and_noise():
    d, n, S, dt = 3, 16, 7, 0.05
    F = _F(d)
    grad = lambda x: x @ F.T  # noqa: E731
    g = torch.Generator().manual_seed(0)
    x0, y0 = torch.randn(2, n, d, generator=g, dtype=torch.float64)
    xi, eta = torch.randn(2, n, S, d, generator=g, dtype=torch.float64)
    a, b = 0.7, -1.3
    lin, tr_lin = overdamped_langevin_scan(a * x0 + b * y0, S, dt, a * xi + b * eta, grad)
    lx, tx = overdamped_langevin_scan(x0, S, dt, xi, grad)
    ly, ty = overdamped_langevin_scan(y0, S, dt, eta, grad)
    assert torch.allclose(lin, a * lx + b * ly, rtol=0, atol=1e-12)
    assert torch.allclose(tr_lin, a * tx + b * ty, rtol=0, atol=1e-12)
    assert torch.equal(tr_lin[:, -1], lin) and tr_lin.shape == (n, S, d)


def test_oracle_zero_noise_follows_the_mean_recursion():
    d, S, dt = 4, 50, 0.02
    F = _F(d)
    x0 = torch.randn(5, d, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    last, traj = overdamped_langevin_scan(x0, S, dt, torch.zeros(5, S, d, dtype=torch.float64), lambda x: x @ F.T)
    A = torch.eye(d, dtype=torch.float64) - dt * F
    m = x0.clone()
    for s in range(S):
        m = m @ A.T
        assert (traj[:, s] - m).abs().max().item() < 1e-12
    m_rec, P_rec = linear_moment_recursion(F, x0[0], torch.zeros(d, d, dtype=torch.float64), S, dt)
    assert (last[0] - m_rec).abs().max().item() < 1e-12


def test_oracle_one_step_covariance_is_two_dt():
    d, n, dt = 3, 400_000, 0.03
    F = _F(d)
    x0 = torch.ones(n, d, dtype=torch.float64) * 0.5  # point mass
    xi = torch.randn(n, 1, d, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    last, _ = overdamped_langevin_scan(x0, 1, dt, xi, lambda x: x @ F.T)
    cov = torch.cov(last.T)
    # sample covariance of n normals: entries within a few 2 dt sqrt(2 / n)
    assert (cov - 2 * dt * torch.eye(d, dtype=torch.float64)).abs().max().item() < 6 * 2 * dt * math.sqrt(2 / n)
    _, P = linear_moment_recursion(F, x0[0], torch.zeros(d, d, dtype=torch.float64), 1, dt)
    assert torch.allclose(P, 2 * dt * torch.eye(d, dtype=torch.float64), rtol=0, atol=1e-15)
