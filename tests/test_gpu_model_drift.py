"""GPU: K1 under a hypothesis model's potential (pdeip_kl_integrate_model) against the float64 oracle, the emitted
drift, exactness of the parametric models against the analytic drifts, kernel-path fallback, rank invariance and the
coupled simulation metric."""
import functools
import math

import pytest
import torch

from conftest import relmax
from oracle import integrator as o_int
from oracle import model as o_model

pytestmark = pytest.mark.gpu


def _mlp(d, hidden, layers, seed, device):
    """(net, params on device, the same network as a float64 oracle tree with the reference's shapes)"""
    from pde_inverse_problem_b200.core.model import V_hypothesis
    net = V_hypothesis(output_dim=1, hidden_dims=[hidden] * layers, dim=d)
    params = net.init(seed, torch.zeros(d, device=device))
    tree = net.tree(params["_flat"])["params"]
    ref = {"params": {k: {"kernel": v["kernel"].double().cpu(), "bias": v["bias"].double().cpu()}
                      for k, v in tree.items()}}
    return net, params, ref


def _oracle_grad(ref):
    return lambda x: torch.func.grad(lambda y: o_model.mlp_apply(ref, y).sum())(x)


def _setup(n, d, S, seed):
    g = torch.Generator().manual_seed(seed)
    z0 = torch.randn(n, 2 * d, generator=g, dtype=torch.float64)
    noise = torch.randn(n, S + 1, d, generator=g, dtype=torch.float64)
    tau0 = torch.rand(n, generator=g, dtype=torch.float64)
    return z0, noise, tau0


@pytest.mark.parametrize("hidden", [32, 20])
@pytest.mark.parametrize("layers", [1, 2, 8])
@pytest.mark.parametrize("d", [2, 8, 32])
def test_fp32_mlp_drift_one_step_matches_float64_oracle(cuda, d, layers, hidden):
    """Parity protocol (i): injected noise and tau0, S = 1 (two update_steps), rtol 1e-5 against float64; the emitted
    drift (grad V_theta at sample 0, evaluated by the second step) too."""
    from pde_inverse_problem_b200 import ops
    N, S, dt, gamma = 1031, 1, 0.01, 0.5
    net, params, ref = _mlp(d, hidden, layers, seed=d + 10 * layers + hidden, device=cuda)
    z0, noise, tau0 = _setup(N, d, S, seed=d * layers)
    tau0 = tau0 * dt
    grad = _oracle_grad(ref)
    last, traj, tau = o_int.underdamped_langevin_dynamics_scan(z0, S, dt, noise, tau0, grad, gamma)
    zl, tr, ta = ops.kl_integrate_model(z0.float().to(cuda), S, dt, gamma, net.spec, params["_flat"],
                                        noise=noise.float().to(cuda), tau0=tau0.float().to(cuda), want_tau=True,
                                        emit_drift=True)
    assert relmax(zl, last) < 1e-5
    assert relmax(tr[..., : 2 * d], traj) < 1e-5
    assert relmax(tr[:, 0, 2 * d:], grad(traj[:, 0, :d])) < 1e-5
    assert relmax(ta, tau) < 1e-6


def test_fp32_mlp_drift_multi_step_within_fp32_twin_band(cuda):
    """Parity protocol (ii), as for the GMM drift: the GPU error against the float64 oracle per step index stays within
    2x the error of the CPU float32 twin of the same restatement (plus a floor)."""
    from pde_inverse_problem_b200 import ops
    d, N, S, T, gamma = 8, 2048, 200, 2.0, 0.5
    dt = T / S
    net, params, ref = _mlp(d, 32, 2, seed=5, device=cuda)
    z0, noise, tau0 = _setup(N, d, S, seed=11)
    z0[:, :d] *= 2.0
    z0[:, d:] *= math.sqrt(0.1)
    tau0 = tau0 * dt
    _, traj64, _ = o_int.underdamped_langevin_dynamics_scan(z0, S, dt, noise, tau0, _oracle_grad(ref), gamma)
    ref32 = {"params": {k: {kk: vv.float() for kk, vv in v.items()} for k, v in ref["params"].items()}}
    _, traj32, _ = o_int.underdamped_langevin_dynamics_scan(z0.float(), S, dt, noise.float(), tau0.float(),
                                                            _oracle_grad(ref32), gamma)
    _, tr, _ = ops.kl_integrate_model(z0.float().to(cuda), S, dt, gamma, net.spec, params["_flat"],
                                      noise=noise.float().to(cuda), tau0=tau0.float().to(cuda))
    err_gpu = (tr.cpu().double() - traj64).abs()
    err_twin = (traj32.double() - traj64).abs()
    scale = traj64.abs().max().item()
    for s in (0, 9, 99, 199):
        g_max, t_max = err_gpu[:, s].max().item() / scale, err_twin[:, s].max().item() / scale
        g_med, t_med = err_gpu[:, s].median().item(), err_twin[:, s].median().item()
        assert g_max <= 2.0 * t_max + 1e-6, (s, g_max, t_max)
        assert g_med <= 2.0 * t_med + 1e-7, (s, g_med, t_med)
    assert relmax(tr[:, 0], traj64[:, 0]) < 1e-5


def _to_particle_major(tr, layout, L):
    if layout == L.TRAJ_TIME_MAJOR:
        return tr.permute(1, 0, 2)
    if layout == L.TRAJ_TIME_SOA:
        return tr.permute(2, 1, 0)
    if layout == L.TRAJ_BLOCK128:
        S, nb, C, _ = tr.shape
        return tr.permute(1, 3, 0, 2).reshape(nb * 128, S, C)
    return tr


@pytest.mark.parametrize("layout", ["particle", "time", "soa", "block"])
def test_emitted_drift_is_model_gradient_in_every_layout(cuda, layout):
    """emit_drift: each emitted sample is [x, v, grad V_theta(x)]; every trajectory layout holds the same numbers,
    with SOA state and emit_every / emit_offset, on both schedules."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    lay = {"particle": L.TRAJ_PARTICLE_MAJOR, "time": L.TRAJ_TIME_MAJOR, "soa": L.TRAJ_TIME_SOA,
           "block": L.TRAJ_BLOCK128}[layout]
    d, N, S, dt, gamma = 8, 384, 12, 0.02, 0.5
    net, params, _ = _mlp(d, 20, 3, seed=3, device=cuda)
    flat = params["_flat"]
    z0, noise, tau0 = _setup(N, d, S, seed=21)
    z0, noise, tau0 = z0.float().to(cuda), noise.float().to(cuda), (tau0 * dt).float().to(cuda)
    zl, tr, _ = ops.kl_integrate_model(z0, S, dt, gamma, net.spec, flat, noise=noise, tau0=tau0, traj_layout=lay,
                                       emit_drift=True, emit_every=3, emit_offset=1)
    tr = _to_particle_major(tr, lay, L)
    assert tr.shape == (N, 4, 3 * d)
    g = net.gradient(params, tr[..., :d].reshape(-1, d).contiguous()).reshape(N, 4, d)
    assert relmax(tr[..., 2 * d:], g) < 1e-5
    zl_p, tr_p, _ = ops.kl_integrate_model(z0, S, dt, gamma, net.spec, flat, noise=noise, tau0=tau0)
    assert torch.equal(tr[..., : 2 * d], tr_p[:, 1::3]) and torch.equal(zl, zl_p)
    # SOA state
    zl_s, _, _ = ops.kl_integrate_model(z0.t().contiguous(), S, dt, gamma, net.spec, flat, noise=noise, tau0=tau0,
                                        state_layout=L.LAYOUT_SOA, want_traj=False)
    assert torch.equal(zl_s.t(), zl)
    # UNIFORM schedule: the last sample has no following step, its drift is evaluated separately
    zl_u, tr_u, _ = ops.kl_integrate_model(z0, S, dt, gamma, net.spec, flat, noise=noise[:, :S].contiguous(),
                                           schedule=L.SCHEDULE_UNIFORM, traj_layout=lay, emit_drift=True)
    tr_u = _to_particle_major(tr_u, lay, L)
    x_last = tr_u[:, -1, :d].contiguous()
    assert relmax(tr_u[:, -1, 2 * d:], net.gradient(params, x_last)) < 1e-5
    assert torch.equal(tr_u[:, -1, : 2 * d], zl_u)


def _kgmm(cuda, d=4, K=3, **kw):
    from pde_inverse_problem_b200 import registry
    from pde_inverse_problem_b200.config import make_config
    cfg = make_config("kinetic_fokker_planck", **{"pde_instance.potential": "GMM", "pde_instance.domain_dim": d,
                                                  "pde_instance.n_gaussian": K, "pde_instance.n_steps": 50, **kw})
    return registry.get_pde_instance(cfg)(cfg=cfg, rng=7, device=cuda)


def _kou(cuda, d=4):
    from pde_inverse_problem_b200 import registry
    from pde_inverse_problem_b200.config import make_config
    cfg = make_config("kinetic_fokker_planck", **{"pde_instance.domain_dim": d, "pde_instance.n_steps": 50})
    return registry.get_pde_instance(cfg)(cfg=cfg, rng=7, device=cuda)


@pytest.mark.parametrize("production", [False, True])
def test_parametric_gmm_model_is_bit_identical_to_gmm_drift(cuda, production):
    """The parametric GMM model holding the true centres runs exactly the GMM drift, on the generic kernel (injected
    noise) and on the production kernels of both paths (Philox, [3d][S][N] trajectory with grad U)."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    from pde_inverse_problem_b200.core.model import V_parametric_GMM
    d, K, N, S, dt, gamma = 8, 16, 1000, 20, 0.01, 0.5
    g = torch.Generator().manual_seed(4)
    mus = (torch.rand(K, d, generator=g) * 8 - 4).to(cuda)
    z0 = (torch.randn(N, 2 * d, generator=g) * 1.5).to(cuda)
    net = V_parametric_GMM(d, K)
    params = net.tree(mus.reshape(-1).clone())
    if production:
        kw = dict(seed=9, particle_offset=77, traj_layout=L.TRAJ_TIME_SOA, emit_drift=True)
    else:
        kw = dict(noise=torch.randn(N, S + 1, d, generator=g).to(cuda), tau0=torch.rand(N, generator=g).mul(dt).to(cuda))
    for path in (L.PATH_FP32, L.PATH_TENSOR):
        a = ops.kl_integrate(z0, S, dt, gamma, L.DRIFT_GMM, mus, n_gaussian=K, sigma=1.0, path=path, **kw)
        b = ops.kl_integrate_model(z0, S, dt, gamma, net.spec, params["_flat"], path=path, **kw)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), path
    assert ops.tensor_path_status() == 0


def test_quadratic_model_equals_linear_drift(cuda):
    """V = y.(yK + b) with K = F/2, b = 0 has grad V = F y: the linear (kinetic OU) drift."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    from pde_inverse_problem_b200.core.model import V_parametric_quadratic
    pde = _kou(cuda, d=6)
    F = pde.initial_configuration["tilde_F"]
    d, N, S, dt, gamma = 6, 2000, 50, 0.02, 1.0
    net = V_parametric_quadratic(d)
    flat = torch.cat([(F / 2).reshape(-1), torch.zeros(d, device=cuda)]).contiguous()
    z0 = torch.randn(N, 2 * d, generator=torch.Generator().manual_seed(1)).to(cuda)
    for kw in (dict(seed=3), dict(seed=3, traj_layout=L.TRAJ_TIME_SOA, emit_drift=True)):
        a = ops.kl_integrate(z0, S, dt, gamma, L.DRIFT_LINEAR, F, **kw)
        b = ops.kl_integrate_model(z0, S, dt, gamma, net.spec, flat, **kw)
        assert relmax(b[0], a[0]) < 1e-6 and relmax(b[1], a[1]) < 1e-6


def test_coupled_simulation_error_vanishes_for_the_true_parametric_models(cuda):
    from pde_inverse_problem_b200.core.model import V_parametric_GMM, V_parametric_quadratic
    from pde_inverse_problem_b200.utils.simulation import coupled_simulation_error
    kgmm = _kgmm(cuda)
    net = V_parametric_GMM(4, 3)
    params = net.tree(kgmm.potential.mus.reshape(-1).clone())
    out = coupled_simulation_error(kgmm, functools.partial(net.apply, params), 4096, rng=5)
    kou = _kou(cuda)
    qnet = V_parametric_quadratic(4)
    F = kou.initial_configuration["tilde_F"]
    qparams = qnet.tree(torch.cat([(F / 2).reshape(-1), torch.zeros(4, device=cuda)]).contiguous())
    out_ou = coupled_simulation_error(kou, functools.partial(qnet.apply, qparams), 4096, rng=5)
    for o in (out, out_ou):
        assert set(o) == {"coupled rms distance terminal", "relative mean error terminal",
                          "relative covariance error terminal"}
        for k, v in o.items():
            assert v.is_cuda and v.ndim == 0
            assert v.item() <= 1e-6, (k, v.item())


def test_coupled_simulation_error_of_a_random_mlp_is_positive(cuda):
    from pde_inverse_problem_b200.utils.simulation import coupled_simulation_error
    kgmm = _kgmm(cuda)
    net, params, _ = _mlp(4, 32, 2, seed=1, device=cuda)
    out = coupled_simulation_error(kgmm, functools.partial(net.apply, params), 4096, rng=5)
    for k, v in out.items():
        assert math.isfinite(v.item()) and v.item() > 0, (k, v.item())
    # the instance's own step count (online sampling: n_steps), or the caller's
    out2 = coupled_simulation_error(kgmm, functools.partial(net.apply, params), 4096, rng=5, n_steps=50)
    assert out2["coupled rms distance terminal"].item() == out["coupled rms distance terminal"].item()


@pytest.mark.parametrize("d,layers", [(4, 2), (8, 3)])
def test_tensor_path_takes_the_fp32_kernel_outside_its_envelope(cuda, d, layers):
    """layers != 2 or d not in {8, 16, 32}: PDEIP_PATH_TENSOR runs the fp32 kernel, bit for bit."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    net, params, _ = _mlp(d, 32, layers, seed=2, device=cuda)
    z0 = torch.randn(512, 2 * d, generator=torch.Generator().manual_seed(2)).to(cuda)
    kw = dict(seed=4, traj_layout=L.TRAJ_BLOCK128, emit_drift=True)
    a = ops.kl_integrate_model(z0, 30, 0.01, 0.5, net.spec, params["_flat"], path=L.PATH_FP32, **kw)
    b = ops.kl_integrate_model(z0, 30, 0.01, 0.5, net.spec, params["_flat"], path=L.PATH_TENSOR, **kw)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.parametrize("model", ["mlp", "gmm"])
def test_rank_invariance_with_particle_offset(cuda, model):
    """One launch over n particles equals two launches over the halves with particle_offset, bit for bit."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    from pde_inverse_problem_b200.core.model import V_parametric_GMM
    d, n, S = 8, 2048, 40
    if model == "mlp":
        net, params, _ = _mlp(d, 32, 2, seed=8, device=cuda)
    else:
        net = V_parametric_GMM(d, 16)
        params = net.init(3, torch.zeros(d, device=cuda))
    z0 = torch.randn(n, 2 * d, generator=torch.Generator().manual_seed(6)).to(cuda)
    for path in (L.PATH_FP32, L.PATH_TENSOR):
        run = functools.partial(ops.kl_integrate_model, n_steps=S, dt=0.01, gamma=0.5, spec=net.spec,
                                params=params["_flat"], seed=31, path=path, traj_layout=L.TRAJ_TIME_SOA,
                                emit_drift=True)
        full = run(z0, particle_offset=100)[0]
        lo = run(z0[: n // 2].contiguous(), particle_offset=100)[0]
        hi = run(z0[n // 2:].contiguous(), particle_offset=100 + n // 2)[0]
        assert torch.equal(full, torch.cat([lo, hi])), path


def _blocked_to_particle_major(tr):
    S, nb, C, _ = tr.shape
    return tr.permute(1, 3, 0, 2).reshape(nb * 128, S, C)


@pytest.mark.parametrize("hidden", [32, 20])
@pytest.mark.parametrize("d", [8, 16, 32])
def test_tensor_mlp_drift_one_step_matches_float64_oracle(cuda, d, hidden):
    """PDEIP_PATH_TENSOR (tcgen05 MLP drift, bf16 hi + lo operands) for one step against the float64 oracle fed with the
    same Philox draws; the emitted grad V_theta too.  Tolerance class "bf16 GEMM paths": 1e-2."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    n, S, dt, gamma, seed, off = 256, 1, 0.01, 0.5, 17, 300
    net, params, ref = _mlp(d, hidden, 2, seed=d + hidden, device=cuda)
    z0 = torch.randn(n, 2 * d, generator=torch.Generator().manual_seed(d), dtype=torch.float64).float().double()
    noise = ops.philox_normals(n, S + 1, d, seed=seed, particle_offset=off, device=cuda).double().cpu()
    tau0 = ops.philox_uniforms(n, seed=seed, particle_offset=off, device=cuda).float().mul(dt).double().cpu()
    grad = _oracle_grad(ref)
    last, traj, _ = o_int.underdamped_langevin_dynamics_scan(z0, S, dt, noise, tau0, grad, gamma)
    zl, tr, _ = ops.kl_integrate_model(z0.float().to(cuda), S, dt, gamma, net.spec, params["_flat"], seed=seed,
                                       particle_offset=off, traj_layout=L.TRAJ_BLOCK128, emit_drift=True,
                                       path=L.PATH_TENSOR)
    torch.cuda.synchronize()
    assert ops.tensor_path_status() == 0
    got = _blocked_to_particle_major(tr)
    e = (relmax(got[..., : 2 * d], traj), relmax(got[:, 0, 2 * d:], grad(traj[:, 0, :d])), relmax(zl, last))
    print(f"tensor one step d={d} hidden={hidden}: state {e[0]:.2e} grad V {e[1]:.2e} last {e[2]:.2e}")
    assert max(e) < 1e-2, e


@pytest.mark.parametrize("d", [8, 16, 32])
def test_tensor_mlp_drift_full_trajectories_match_fp32_kernel(cuda, d):
    """200 steps on the tcgen05 MLP drift against the fp32 kernel on the same Philox draws (rtol 1e-2, per-tensor
    max-norm): terminal-only (ragged n = 1000 and full tiles), BLOCK128 and TIME_SOA with grad V_theta.  Inside that
    envelope, the criterion of the GMM kernel's full-length test (tests/test_gpu_integrator.py): median |err| < 1e-4 and
    99.9 % of the entries within 1e-2 of the trajectory (and drift) scale, terminal ensemble mean and second moment
    within 1e-3."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    S, dt, gamma, seed = 200, 0.01, 0.5, 5
    net, params, _ = _mlp(d, 32, 2, seed=40 + d, device=cuda)
    flat = params["_flat"]
    z = torch.randn(1024, 2 * d, generator=torch.Generator().manual_seed(9)).to(cuda)
    z[:, d:] *= 0.3

    def run(n, path, **kw):
        out = ops.kl_integrate_model(z[:n].contiguous(), S, dt, gamma, net.spec, flat, seed=seed, path=path, **kw)
        torch.cuda.synchronize()
        return out

    for n in (1000, 1024):
        zt, _, _ = run(n, L.PATH_TENSOR, want_traj=False)
        assert ops.tensor_path_status() == 0
        zf, _, _ = run(n, L.PATH_FP32, want_traj=False)
        err = relmax(zt, zf)
        print(f"tensor vs fp32 d={d} terminal n={n}: last {err:.2e}")
        assert torch.isfinite(zt).all() and err < 1e-2
        _assert_statistics(zt, zf, f"terminal n={n}")
        _assert_moments(zt, zf)
    for layout in (L.TRAJ_BLOCK128, L.TRAJ_TIME_SOA):
        zt, tt, _ = run(1024, L.PATH_TENSOR, traj_layout=layout, emit_drift=True)
        assert ops.tensor_path_status() == 0
        zf, tf, _ = run(1024, L.PATH_FP32, traj_layout=layout, emit_drift=True)
        e_traj = relmax(tt.reshape(-1, 3 * d, 128)[:, : 2 * d] if layout == L.TRAJ_BLOCK128 else tt[: 2 * d],
                        tf.reshape(-1, 3 * d, 128)[:, : 2 * d] if layout == L.TRAJ_BLOCK128 else tf[: 2 * d])
        e_drift = relmax(tt.reshape(-1, 3 * d, 128)[:, 2 * d:] if layout == L.TRAJ_BLOCK128 else tt[2 * d:],
                         tf.reshape(-1, 3 * d, 128)[:, 2 * d:] if layout == L.TRAJ_BLOCK128 else tf[2 * d:])
        e_last = relmax(zt, zf)
        print(f"tensor vs fp32 d={d} layout={layout}: traj {e_traj:.2e} grad V {e_drift:.2e} last {e_last:.2e}")
        assert max(e_traj, e_drift, e_last) < 1e-2
        blocks = (lambda t: (t.reshape(-1, 3 * d, 128)[:, : 2 * d], t.reshape(-1, 3 * d, 128)[:, 2 * d:])) \
            if layout == L.TRAJ_BLOCK128 else (lambda t: (t[: 2 * d], t[2 * d:]))
        for name, a, b in zip(("traj", "grad V"), blocks(tt), blocks(tf)):
            _assert_statistics(a, b, f"layout={layout} {name}")
        _assert_moments(zt, zf)


def _assert_statistics(t, f, what):
    """median |err| < 1e-4 and 99.9 % of the entries within 1e-2, both relative to the scale max |f|"""
    e = (t.double().cpu() - f.double().cpu()).abs() / f.abs().max().item()
    med, frac = e.median().item(), (e < 1e-2).double().mean().item()
    print(f"  {what}: median {med:.1e}, fraction within 1e-2 {frac:.5f}")
    assert med < 1e-4 and frac > 0.999, (what, med, frac)


def _assert_moments(zt, zf):
    """terminal ensemble mean and second moment within 1e-3"""
    zt, zf = zt.double().cpu(), zf.double().cpu()
    assert (zt.mean(0) - zf.mean(0)).abs().max() < 1e-3 * max(1.0, zf.abs().max().item())
    m2, m2r = (zt ** 2).mean(0), (zf ** 2).mean(0)
    assert ((m2 - m2r).abs() / m2r.abs().max()).max() < 1e-3
