"""CPU: the Fokker-Planck GMM instance's dispatch and configuration, the overdamped pipeline.HotPath (its
configuration checks, chunk sizing and the ops one step issues, captured without a device), and a float64 known answer
of the overdamped scheme under a one-centre GMM potential."""
import math

import pytest
import torch

from overdamped_oracle import linear_moment_recursion, overdamped_langevin_scan


def _cfg(potential=None, d=4, **over):
    from pde_inverse_problem_b200.config import make_config
    kw = {"pde_instance.domain_dim": d, **over}
    if potential is not None:
        kw["pde_instance.potential"] = potential
    return make_config("fokker_planck", **kw)


def test_registry_dispatch():
    from pde_inverse_problem_b200 import registry
    from pde_inverse_problem_b200.example_problems.fokker_planck_example import FokkerPlanck
    from pde_inverse_problem_b200.example_problems.fokker_planck_example_GMM import FokkerPlanckGMM
    assert registry.get_pde_instance(_cfg("GMM")) is FokkerPlanckGMM
    assert registry.FokkerPlanckPotential == {"Quadratic": FokkerPlanck, "GMM": FokkerPlanckGMM}
    for potential in (None, "Quadratic", "OU", "anything"):
        assert registry.get_pde_instance(_cfg(potential)) is FokkerPlanck, potential
    cfg = _cfg()
    del cfg.pde_instance["potential"]
    assert registry.get_pde_instance(cfg) is FokkerPlanck


def test_fp_gmm_configuration():
    from pde_inverse_problem_b200.example_problems import fokker_planck_example_GMM as fpg
    from pde_inverse_problem_b200.example_problems import kinetic_fokker_planck_example_GMM as kg
    from pde_inverse_problem_b200.utils import rng as jrandom
    pde = fpg.FokkerPlanckGMM(_cfg("GMM", d=5, **{"pde_instance.n_gaussian": 4}), rng=7, device="cpu")
    c = pde.initial_configuration
    assert "gamma_friction" not in c  # coupled_simulation_error picks the overdamped dynamics from its absence
    assert c["n_Gaussian"] == 4 and tuple(c["GMM"]["mus"].shape) == (4, 5) and pde.n_steps == 100
    assert c["GMM"]["mus"].abs().max() <= 4.0
    # the centres the kinetic GMM instance draws from the same seed
    kin = kg.initialize_configuration(5, jrandom.split(7)[0], n_Gaussian=4, device="cpu")
    assert torch.equal(c["GMM"]["mus"], kin["GMM"]["mus"])
    assert torch.equal(pde.distribution_initial.cov, torch.eye(5) * 4.0) and not pde.distribution_initial.mu.any()
    assert pde.potential.sigma == 1.0 and pde.sample_scheme == "SDE" and pde.sample_mode == "online"
    assert fpg.FokkerPlanckGMM(_cfg("GMM", **{"pde_instance.n_steps": 7}), rng=1, device="cpu").n_steps == 7
    with pytest.raises(NotImplementedError, match="offline"):
        fpg.FokkerPlanckGMM(_cfg("GMM", **{"pde_instance.sample_mode": "offline"}), rng=1, device="cpu")
    from pde_inverse_problem_b200.config import _PDE
    assert set(_PDE["fokker_planck"]) == {"domain_dim", "domain_min", "domain_max", "boundary_condition",
                                          "diffusion_coefficient", "total_evolving_time", "name", "potential"}


def _hp_cfg(**kw):
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200.pipeline import HotPathConfig
    base = dict(d=8, n_steps=10, total_time=2.0, gamma=0.5, drift_kind=L.DRIFT_GMM, n_gaussian=16, chunk=256,
                dynamics="overdamped")
    base.update(kw)
    return HotPathConfig(**base)


def test_hot_path_config_rejections():
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200.pipeline import HotPath, HotPathConfig
    assert HotPathConfig(d=4, n_steps=1, total_time=1.0, gamma=1.0, drift_kind=L.DRIFT_LINEAR).dynamics == "kinetic"
    with pytest.raises(ValueError, match="dynamics"):
        HotPath(_hp_cfg(dynamics="underdamped"), None, {}, None, None, device="cpu")
    with pytest.raises(ValueError, match="MEANFIELD_TABLE"):
        HotPath(_hp_cfg(drift_kind=L.DRIFT_MEANFIELD_TABLE), None, {}, None, None, device="cpu")


def test_integrator_wave_and_auto_chunk_overdamped():
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200.pipeline import auto_chunk, integrator_wave
    T = L.PATH_TENSOR
    assert integrator_wave(8, L.DRIFT_GMM, 16, T, sm_count=148, overdamped=True) == 148 * 6 * 128
    assert integrator_wave(16, L.DRIFT_GMM, 32, T, sm_count=148, overdamped=True) == 148 * 3 * 128
    assert integrator_wave(32, L.DRIFT_GMM, 64, T, sm_count=148, overdamped=True) == 148 * 3 * 128
    assert integrator_wave(32, L.DRIFT_GMM, 65, T, sm_count=148, overdamped=True) == 148 * 2 * 128
    assert integrator_wave(8, L.DRIFT_GMM, 16, L.PATH_FP32, sm_count=148, overdamped=True) == 148 * 4 * 128
    # positional calls keep their kinetic meaning
    assert integrator_wave(8, L.DRIFT_GMM, 16, T, 148) == 148 * 8 * 128
    assert auto_chunk(8, 200, L.DRIFT_GMM, 16, T, 1, 6.0e9, 148) == 2 * 148 * 8 * 128
    for d, K, S in ((8, 16, 200), (32, 64, 200), (16, 32, 2000)):
        w = integrator_wave(d, L.DRIFT_GMM, K, T, sm_count=148, overdamped=True)
        c = auto_chunk(d, S, L.DRIFT_GMM, K, T, sm_count=148, overdamped=True)
        per = 2 * d * S * 4
        assert c % w == 0 and c >= w
        assert c * per <= 6.0e9 or c == w
        assert (c + w) * per > 6.0e9


class _Fake:
    """stand-ins for CUDA streams and events on the CPU"""

    def __init__(self, *a, **k):
        pass

    def record(self, *a):
        pass

    def wait_event(self, *a):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def test_hot_path_step_issues_the_fp_ops(monkeypatch):
    """Which ops one overdamped step runs, with which layouts, weights and coefs: a BLOCK128 chunk and a ragged
    TIME_SOA chunk of a host-resident ensemble, the FP 0T set with DRIFT_IN_POINTS at 1 / (n S), the FP boundary sets on
    all terminal and initial states at +-2/T, 1 / n; finalize and Adam."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops, parallel, pipeline
    from pde_inverse_problem_b200.core.model import V_hypothesis
    from pde_inverse_problem_b200.core.optimizer import AdamL2
    calls = []

    class Acc:
        def __init__(self, spec, device):
            self.sums, self.grad = torch.zeros(L.NUM_SUMS), torch.zeros(spec.num_params)

        def begin(self):
            calls.append(("begin",))

        def accumulate(self, set_kind, params, points, weight, coef=0.0, layout=L.LAYOUT_AOS, true_grad=None,
                       path=L.PATH_FP32):
            calls.append(("acc", set_kind, tuple(points.shape), weight, coef, layout,
                          true_grad.kind if true_grad else None, path))

        def finalize(self):
            calls.append(("finalize",))
            return self.sums, self.grad

    def integrate(x0, n_steps, dt, drift_kind, drift_params, *, n_gaussian, sigma, seed, particle_offset, traj_layout,
                  emit_every, emit_drift, path, traj_out, x_last_out):
        n, d = x0.shape
        calls.append(("od", n, n_steps, dt, drift_kind, n_gaussian, seed, particle_offset, traj_layout, emit_drift,
                      path, traj_out.data_ptr(), tuple(x_last_out.shape)))
        x_last_out.copy_(x0 + 1.0)
        return x_last_out, traj_out[: n * n_steps * 2 * d]

    monkeypatch.setattr(pipeline.ops, "ResidualAccumulator", Acc)
    monkeypatch.setattr(pipeline.ops, "overdamped_integrate", integrate)
    monkeypatch.setattr(pipeline.ops, "kl_integrate", lambda *a, **k: pytest.fail("kinetic integrator called"))
    monkeypatch.setattr(pipeline.ops, "adam_l2_step", lambda *a, **k: calls.append(("adam",)))
    for name in ("Stream", "Event", "stream"):
        monkeypatch.setattr(torch.cuda, name, _Fake)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a: _Fake())
    monkeypatch.setattr(parallel.Shard, "current", staticmethod(lambda: parallel.Shard(0, 1)))
    d, K, S, T = 8, 16, 10, 2.0
    model = V_hypothesis(1, [32, 32], d)
    params = model.init(11, torch.zeros(d))
    opt = AdamL2(lambda count: 1e-3, 1e-3)
    hp = pipeline.HotPath(_hp_cfg(n_steps=S, total_time=T, path=L.PATH_TENSOR), model, params, torch.zeros(K, d),
                          None, optimizer=opt, device="cpu")
    assert hp.particle_steps(1000) == 1000 * S
    x0 = torch.randn(356, d)  # host-resident: a BLOCK128 chunk of 256, then a ragged chunk of 100
    hp.step(x0, seed=3, n_global=1000, particle_offset=40)
    dt = T / S
    od = [c for c in calls if c[0] == "od"]
    assert [c[1:11] for c in od] == [
        (256, S, dt, L.DRIFT_GMM, K, 3, 40, L.TRAJ_BLOCK128, True, L.PATH_TENSOR),
        (100, S, dt, L.DRIFT_GMM, K, 3, 296, L.TRAJ_TIME_SOA, True, L.PATH_TENSOR)]
    assert od[0][11] == od[1][11] == hp.traj.data_ptr() and od[0][12] == (256, d) and od[1][12] == (100, d)
    w0, wb = 1.0 / (1000 * S), 1.0 / 1000
    IN = L.DRIFT_IN_POINTS
    assert [c for c in calls if c[0] != "od"] == [
        ("begin",),
        ("acc", L.SET_FP_0T, (S * 256 // 128, 2 * d, 128), w0, 0.0, L.LAYOUT_BLOCK128, IN, L.PATH_TENSOR),
        ("acc", L.SET_FP_0T, (2 * d, S * 100), w0, 0.0, L.LAYOUT_SOA, IN, L.PATH_TENSOR),
        ("acc", L.SET_FP_BOUNDARY, (356, d), wb, 2.0 / T, L.LAYOUT_AOS, None, L.PATH_TENSOR),
        ("acc", L.SET_FP_BOUNDARY, (356, d), wb, -2.0 / T, L.LAYOUT_AOS, None, L.PATH_TENSOR),
        ("finalize",), ("adam",)]
    assert torch.equal(hp.z0_full, x0) and torch.equal(hp.z_last_full, x0 + 1.0)


def _gmm_grad(mus):
    def grad(x):
        w = torch.softmax(-((x[:, None, :] - mus[None]) ** 2).sum(-1) / 2.0, -1)
        return x - w @ mus
    return grad


def test_single_centre_gmm_known_answer_float64():
    """K = 1: grad U = x - mu, so the scheme is OU around mu and linear_moment_recursion with F = I, shifted by mu,
    gives its exact moments.  The scan is affine in (x0, xi): its mean is the zero-noise run from m0, its covariance
    J_x P0 J_x^T + J_xi J_xi^T (Jacobians of one particle's scan), both to 1e-12."""
    d, S, dt = 3, 25, 0.05
    g = torch.Generator().manual_seed(1)
    mu = torch.randn(1, d, generator=g, dtype=torch.float64)
    m0 = torch.randn(d, generator=g, dtype=torch.float64)
    P0 = torch.eye(d, dtype=torch.float64) * 2.0 + 0.3
    grad = _gmm_grad(mu)
    x = torch.randn(5, d, generator=g, dtype=torch.float64)
    assert torch.allclose(grad(x), x - mu, atol=1e-14, rtol=0)
    m, P = linear_moment_recursion(torch.eye(d, dtype=torch.float64), m0 - mu[0], P0, S, dt)

    def last(x0, xi):
        return overdamped_langevin_scan(x0[None], S, dt, xi[None], grad)[0][0]

    zero = torch.zeros(S, d, dtype=torch.float64)
    assert torch.allclose(last(m0, zero), m + mu[0], atol=1e-12, rtol=0)
    Jx, Jxi = torch.func.jacfwd(last, argnums=(0, 1))(m0, zero)
    Jxi = Jxi.reshape(d, S * d)
    cov = Jx @ P0 @ Jx.T + Jxi @ Jxi.T
    assert torch.allclose(cov, P, atol=1e-12, rtol=0)
    assert math.isclose(torch.trace(P).item(), torch.trace(cov).item(), rel_tol=1e-12)
