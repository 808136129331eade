"""GPU: the overdamped integrator K1-OD (pdeip_overdamped_integrate*) against its float64 definition
(tests/overdamped_oracle.py), the Philox stream, trajectory layouts and emitted drift, rank invariance, a known answer
on the Fokker-Planck instance, the tcgen05 MLP drift against float64 and against the fp32 kernel, the composition with
the FP residual through PDEIP_DRIFT_IN_POINTS, and the coupled simulation metric on the FP instance."""
import functools
import math

import numpy as np
import pytest
import torch

from conftest import relmax
from imlp_model import TOL_MT
from oracle import model as o_model
from oracle import potential as o_pot
from overdamped_oracle import linear_moment_recursion, overdamped_langevin_scan

pytestmark = pytest.mark.gpu


def _mlp(d, hidden, layers, seed, device, bias=True):
    """(net, params on device with non-zero biases, the same network as a float64 oracle tree)"""
    from pde_inverse_problem_b200.core.model import V_hypothesis
    net = V_hypothesis(output_dim=1, hidden_dims=[hidden] * layers, dim=d)
    params = net.init(seed, torch.zeros(d, device=device))
    tree = net.tree(params["_flat"])["params"]
    if bias:
        g = torch.Generator().manual_seed(seed)
        for k in tree:
            tree[k]["bias"].copy_(0.1 * torch.randn(tree[k]["bias"].shape, generator=g))
    ref = {"params": {k: {"kernel": v["kernel"].double().cpu(), "bias": v["bias"].double().cpu()}
                      for k, v in tree.items()}}
    return net, params, ref


def _mlp_grad(ref):
    return lambda x: torch.func.grad(lambda y: o_model.mlp_apply(ref, y).sum())(x)


def _F(d):
    from pde_inverse_problem_b200.example_problems.fokker_planck_example import initialize_configuration
    return torch.as_tensor(initialize_configuration(d)["F"], dtype=torch.float32)


def _drift(name, d, cuda):
    """(runner(x0, S, dt, **kw) -> (x_last, traj), float64 grad U of the same fp32 parameters, float32 twin grad)"""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    from pde_inverse_problem_b200.core.model import V_parametric_GMM, V_parametric_quadratic
    g = torch.Generator().manual_seed(7 + d)
    if name == "linear":
        F = _F(d)
        run = functools.partial(ops.overdamped_integrate, drift_kind=L.DRIFT_LINEAR, drift_params=F.to(cuda))
        return run, lambda x: x @ F.T.to(x.dtype)
    if name == "none":
        return functools.partial(ops.overdamped_integrate, drift_kind=L.DRIFT_NONE), torch.zeros_like
    if name.startswith("gmm"):  # gmm3, gmm16: the analytic drift; gmm_model: the parametric model, sigma = 1
        K = 3 if name == "gmm3" else 16
        mus = torch.rand(K, d, generator=g) * 6 - 3
        sigma = 1.0 if name == "gmm_model" else 1.3
        if name == "gmm_model":
            net = V_parametric_GMM(d, K)
            run = functools.partial(ops.overdamped_integrate_model, spec=net.spec, params=mus.reshape(-1).to(cuda))
        else:
            run = functools.partial(ops.overdamped_integrate, drift_kind=L.DRIFT_GMM, drift_params=mus.to(cuda),
                                    n_gaussian=K, sigma=sigma)
        return run, lambda x: o_pot.gmm_gradient_closed_form(x, mus.to(x.dtype), sigma)
    if name == "quadratic":
        net = V_parametric_quadratic(d)
        B = torch.randn(d, d, generator=g)
        R = torch.randn(d, d, generator=g)
        K = B @ B.T / (2 * d) + 0.1 * (R - R.T)  # asymmetric, K + K^T = B B^T / d positive semi-definite (stable)
        b = torch.randn(d, generator=g) * 0.3
        run = functools.partial(ops.overdamped_integrate_model, spec=net.spec,
                                params=torch.cat([K.reshape(-1), b]).to(cuda))
        return run, lambda x: x @ (K + K.T).to(x.dtype).T + b.to(x.dtype)
    _, layers, hidden = name.split("_")  # mlp_<layers>_<hidden>
    net, params, ref = _mlp(d, int(hidden), int(layers), seed=d + 10 * int(layers) + int(hidden), device=cuda)
    run = functools.partial(ops.overdamped_integrate_model, spec=net.spec, params=params["_flat"])
    ref32 = {"params": {k: {kk: vv.float() for kk, vv in v.items()} for k, v in ref["params"].items()}}
    grad64, grad32 = _mlp_grad(ref), _mlp_grad(ref32)
    return run, lambda x: grad64(x) if x.dtype == torch.float64 else grad32(x)


DRIFTS = ["linear", "gmm3", "gmm16", "none", "quadratic", "gmm_model", "mlp_1_32", "mlp_2_32", "mlp_3_32", "mlp_1_20",
          "mlp_2_20", "mlp_3_20"]


def _inputs(n, d, S, seed, scale=1.5):
    g = torch.Generator().manual_seed(seed)
    x0 = (torch.randn(n, d, generator=g, dtype=torch.float64) * scale).float().double()
    noise = torch.randn(n, S, d, generator=g, dtype=torch.float64).float().double()
    return x0, noise


@pytest.mark.parametrize("name", DRIFTS)
def test_fp32_one_step_matches_float64(cuda, name):
    """Injected noise, one step, rtol 1e-5; the emitted drift of the one sample (the extra evaluation) too."""
    d, n, dt = 6, 1031, 0.01
    run, grad = _drift(name, d, cuda)
    x0, noise = _inputs(n, d, 1, seed=1)
    last, traj = overdamped_langevin_scan(x0, 1, dt, noise, grad)
    xl, tr = run(x0.float().to(cuda), 1, dt, noise=noise.float().to(cuda), emit_drift=True)
    assert tr.shape == (n, 1, 2 * d)
    assert relmax(xl, last) < 1e-5 and relmax(tr[..., :d], traj) < 1e-5
    if name != "none":
        assert relmax(tr[:, 0, d:], grad(traj[:, 0])) < 1e-5
    else:
        assert not tr[..., d:].any()


@pytest.mark.parametrize("name", ["linear", "gmm3", "gmm16", "gmm_model", "quadratic", "mlp_2_32", "mlp_3_20"])
def test_fp32_200_steps_against_float64(cuda, name):
    """200 steps on injected noise.  Linear drifts: rtol 1e-5.  Nonlinear drifts: BASELINE section 5 criterion, the GPU
    error against float64 per step index within 2x the error of the CPU float32 twin of the same restatement, in the
    median and the 99.9th percentile at every reported step and in the maximum up to step 9.  Later, the maximum over
    the 12 288 entries is one particle's rounding amplified by a locally unstable drift, an extreme value of two
    independent rounding sequences rather than a property of the kernel (MLP 32 x 2, step 199: 8.1e-5 against the
    twin's 2.3e-5 on a B200 with equal medians); it is printed, not asserted."""
    d, n, S, dt = 6, 2048, 200, 0.01
    run, grad = _drift(name, d, cuda)
    x0, noise = _inputs(n, d, S, seed=2)
    _, traj64 = overdamped_langevin_scan(x0, S, dt, noise, grad)
    _, tr = run(x0.float().to(cuda), S, dt, noise=noise.float().to(cuda))
    err_gpu = (tr.cpu().double() - traj64).abs()
    scale = traj64.abs().max().item()
    if name in ("linear", "quadratic"):
        assert err_gpu.max().item() / scale < 1e-5
        return
    _, traj32 = overdamped_langevin_scan(x0.float(), S, dt, noise.float(), grad)
    err_twin = (traj32.double() - traj64).abs()
    for s in (0, 9, 99, 199):
        g_max, t_max = err_gpu[:, s].max().item() / scale, err_twin[:, s].max().item() / scale
        g_med, t_med = err_gpu[:, s].median().item(), err_twin[:, s].median().item()
        g_p, t_p = (torch.quantile(e[:, s].reshape(-1), 0.999).item() / scale for e in (err_gpu, err_twin))
        print(f"{name} step {s}: gpu max {g_max:.2e} twin {t_max:.2e}, p99.9 {g_p:.2e} / {t_p:.2e}, "
              f"median {g_med:.2e} / {t_med:.2e}")
        if s <= 9:
            assert g_max <= 2.0 * t_max + 1e-6, (s, g_max, t_max)
        assert g_p <= 2.0 * t_p + 1e-6, (s, g_p, t_p)
        assert g_med <= 2.0 * t_med + 1e-7, (s, g_med, t_med)


@pytest.mark.parametrize("name", ["linear", "mlp_2_32", "gmm16"])
def test_philox_mode_equals_injected_philox_normals(cuda, name):
    """Step s draws exactly draw s of philox_normals(n, S, d, seed, particle_offset, step_offset): bit for bit."""
    from pde_inverse_problem_b200 import ops
    d, n, S, dt, seed, off, so = 6, 777, 30, 0.01, 91, 12345, 7
    run, _ = _drift(name, d, cuda)
    x0 = _inputs(n, d, 1, seed=3)[0].float().to(cuda)
    a = run(x0, S, dt, seed=seed, particle_offset=off, step_offset=so, emit_drift=True)
    nz = ops.philox_normals(n, S, d, seed=seed, particle_offset=off, step_offset=so, device=cuda)
    b = run(x0, S, dt, noise=nz, emit_drift=True)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


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
@pytest.mark.parametrize("name", ["linear", "gmm16", "mlp_3_20"])
def test_layouts_emission_and_emitted_drift(cuda, name, layout):
    """Every trajectory layout and both state layouts hold the same numbers bit for bit; emit_every / emit_offset pick
    samples 1, 4, 7, 10 of 12; the emitted drift is linear_grad / gmm_value_grad / model_eval at the emitted positions."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    lay = {"particle": L.TRAJ_PARTICLE_MAJOR, "time": L.TRAJ_TIME_MAJOR, "soa": L.TRAJ_TIME_SOA,
           "block": L.TRAJ_BLOCK128}[layout]
    d, n, S, dt = 8, 384, 12, 0.02
    run, _ = _drift(name, d, cuda)
    x0, noise = _inputs(n, d, S, seed=4)
    x0, noise = x0.float().to(cuda), noise.float().to(cuda)
    xl, tr = run(x0, S, dt, noise=noise, traj_layout=lay, emit_drift=True, emit_every=3, emit_offset=1)
    tr = _to_particle_major(tr, lay, L)
    assert tr.shape == (n, 4, 2 * d)
    xl_p, tr_p = run(x0, S, dt, noise=noise)
    assert torch.equal(tr[..., :d], tr_p[:, 1::3]) and torch.equal(xl, xl_p) and torch.equal(tr_p[:, -1], xl)
    xs = tr[..., :d].reshape(-1, d).contiguous()
    kw = run.keywords
    if name == "linear":
        want = ops.linear_grad(xs, kw["drift_params"])
    elif name == "gmm16":
        want = ops.gmm_value_grad(xs, kw["drift_params"], kw["sigma"])[1]
    else:
        want = ops.model_eval(kw["spec"], kw["params"], xs, want=("grad",))["grad"]
    assert relmax(tr[..., d:].reshape(-1, d), want) < 1e-5
    # SOA state
    xl_s, _ = run(x0.t().contiguous(), S, dt, noise=noise, state_layout=L.LAYOUT_SOA, want_traj=False)
    assert torch.equal(xl_s.t(), xl)


@pytest.mark.parametrize("model", ["mlp", "gmm"])
def test_rank_invariance_with_particle_offset(cuda, model):
    """One launch over n particles equals two launches over the halves with particle_offset, bit for bit, on both paths
    (the MLP 32 x 2 at d = 8 runs tcgen05 on PDEIP_PATH_TENSOR)."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    d, n, S = 8, 2048, 40
    run, _ = _drift("mlp_2_32" if model == "mlp" else "gmm_model", d, cuda)
    x0 = _inputs(n, d, 1, seed=6)[0].float().to(cuda)
    for path in (L.PATH_FP32, L.PATH_TENSOR):
        for kw in (dict(want_traj=False), dict(traj_layout=L.TRAJ_TIME_SOA, emit_drift=True)):
            full = run(x0, S, 0.01, seed=31, particle_offset=100, path=path, **kw)
            lo = run(x0[: n // 2].contiguous(), S, 0.01, seed=31, particle_offset=100, path=path, **kw)
            hi = run(x0[n // 2:].contiguous(), S, 0.01, seed=31, particle_offset=100 + n // 2, path=path, **kw)
            assert torch.equal(full[0], torch.cat([lo[0], hi[0]])), (path, kw)
            if full[1] is not None:
                assert torch.equal(full[1], torch.cat([lo[1], hi[1]], -1)), (path, kw)
    assert ops.tensor_path_status() == 0


def _fp(cuda, d=4):
    from pde_inverse_problem_b200 import registry
    from pde_inverse_problem_b200.config import make_config
    cfg = make_config("fokker_planck", **{"pde_instance.domain_dim": d})
    return registry.get_pde_instance(cfg)(cfg=cfg, rng=7, device=cuda)


def test_fp_instance_moments_follow_the_discrete_recursion(cuda):
    """dt = 0.02, T = 2 on the FP instance's F (d = 4) from its initial law N(m_0, P_0): the ensemble mean and
    covariance match m' = (I - dt F) m, P' = (I - dt F) P (I - dt F)^T + 2 dt I within Monte-Carlo error.  The O(dt)
    gap of that recursion to the exact law OU_process(T) is reported, not asserted."""
    from pde_inverse_problem_b200.example_problems.fokker_planck_example import OU_process
    from pde_inverse_problem_b200.utils.sampling_utils import overdamped_langevin_dynamics_scan
    pde = _fp(cuda)
    n, S, dt = 1 << 19, 100, 0.02
    x0 = pde.distribution_initial.sample(n, 3)
    xl, _ = overdamped_langevin_dynamics_scan(x0, S, dt, 11, pde.potential.gradient, want_trajectory=False)
    x = xl.double().cpu()
    m_emp, C_emp = x.mean(0), torch.cov(x.T)
    cfgn = pde.np_configuration
    F = torch.as_tensor(pde.initial_configuration["F"].cpu().double())
    m, P = linear_moment_recursion(F, torch.as_tensor(cfgn["m_0"]), torch.as_tensor(cfgn["P_0"]), S, dt)
    mc = torch.sqrt(torch.diagonal(P) / n)
    rel_cov = (torch.linalg.matrix_norm(C_emp - P) / torch.linalg.matrix_norm(P)).item()
    m_ou, P_ou = OU_process(2.0, cfgn)
    gap = np.linalg.norm(P.numpy() - P_ou) / np.linalg.norm(P_ou)
    print(f"FP KAT: |mean - m| / MC sigma max {((m_emp - m).abs() / mc).max().item():.2f}, covariance rel Frobenius "
          f"{rel_cov:.2e}; O(dt) gap of the recursion to OU_process(T): mean {np.abs(m.numpy() - m_ou).max():.2e}, "
          f"covariance rel Frobenius {gap:.2e}")
    assert ((m_emp - m).abs() <= 5 * mc).all(), (m_emp, m, mc)
    assert rel_cov < 1e-2


@pytest.mark.parametrize("hidden", [32, 20])
@pytest.mark.parametrize("d", [8, 16, 32])
def test_tensor_mlp_drift_matches_float64(cuda, d, hidden):
    """PDEIP_PATH_TENSOR (tcgen05 MLP drift) for S = 4 steps fed the same Philox draws as the float64 definition: every
    emitted grad V_theta against float64 autodiff at the emitted position (TOL_MT), the samples against float64."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    n, S, dt, seed, off = 256, 4, 0.01, 17, 300
    net, params, ref = _mlp(d, hidden, 2, seed=d + hidden, device=cuda)
    x0 = _inputs(n, d, 1, seed=d)[0]
    noise = ops.philox_normals(n, S, d, seed=seed, particle_offset=off, device=cuda).double().cpu()
    grad = _mlp_grad(ref)
    last, traj = overdamped_langevin_scan(x0, S, dt, noise, grad)
    xl, tr = ops.overdamped_integrate_model(x0.float().to(cuda), S, dt, net.spec, params["_flat"], seed=seed,
                                            particle_offset=off, traj_layout=L.TRAJ_BLOCK128, emit_drift=True,
                                            path=L.PATH_TENSOR)
    torch.cuda.synchronize()
    assert ops.tensor_path_status() == 0
    got = _to_particle_major(tr, L.TRAJ_BLOCK128, L).cpu()
    x_emit = got[..., :d].double().reshape(-1, d)
    e_drift = relmax(got[..., d:].reshape(-1, d), grad(x_emit))
    e_state = max(relmax(got[..., :d], traj), relmax(xl, last))
    print(f"tensor overdamped d={d} hidden={hidden}: grad V {e_drift:.2e} (TOL_MT {TOL_MT:.0e}) state {e_state:.2e}")
    assert e_drift < TOL_MT and e_state < 1e-4


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


@pytest.mark.parametrize("hidden", [32, 20])
@pytest.mark.parametrize("d", [8, 16, 32])
def test_tensor_mlp_200_steps_match_fp32_kernel(cuda, d, hidden):
    """200 steps on the tcgen05 MLP drift against the fp32 kernel on the same Philox draws: max-norm 1e-2 and the
    full-length criterion of the kinetic K1-MT test, terminal-only (ragged n = 1000), BLOCK128 and TIME_SOA."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    S, dt, seed = 200, 0.01, 5
    net, params, _ = _mlp(d, hidden, 2, seed=40 + d + hidden, device=cuda)
    x = _inputs(1024, d, 1, seed=9)[0].float().to(cuda)

    def run(n, path, **kw):
        out = ops.overdamped_integrate_model(x[:n].contiguous(), S, dt, net.spec, params["_flat"], seed=seed,
                                             path=path, **kw)
        torch.cuda.synchronize()
        return out

    xt, _ = run(1000, L.PATH_TENSOR, want_traj=False)
    assert ops.tensor_path_status() == 0
    xf, _ = run(1000, L.PATH_FP32, want_traj=False)
    err = relmax(xt, xf)
    print(f"tensor vs fp32 overdamped d={d} hidden={hidden} terminal n=1000: {err:.2e}")
    assert torch.isfinite(xt).all() and err < 1e-2
    _assert_statistics(xt, xf, "terminal n=1000")
    _assert_moments(xt, xf)
    for layout in (L.TRAJ_BLOCK128, L.TRAJ_TIME_SOA):
        xt, tt = run(1024, L.PATH_TENSOR, traj_layout=layout, emit_drift=True)
        assert ops.tensor_path_status() == 0
        xf, tf = run(1024, L.PATH_FP32, traj_layout=layout, emit_drift=True)
        assert torch.equal(_to_particle_major(tt, layout, L)[:, -1, :d], xt)
        parts = (lambda t: (t[:, :, :d], t[:, :, d:])) if layout == L.TRAJ_BLOCK128 else (lambda t: (t[:d], t[d:]))
        errs = [relmax(a, b) for a, b in zip(parts(tt), parts(tf))] + [relmax(xt, xf)]
        print(f"tensor vs fp32 overdamped d={d} hidden={hidden} layout={layout}: traj {errs[0]:.2e} "
              f"grad V {errs[1]:.2e} last {errs[2]:.2e}")
        assert max(errs) < 1e-2
        for what, a, b in zip(("traj", "grad V"), parts(tt), parts(tf)):
            _assert_statistics(a, b, f"layout={layout} {what}")
        _assert_moments(xt, xf)


@pytest.mark.parametrize("case", ["layers3", "d12", "injected", "particle_major"])
def test_tensor_path_outside_envelope_is_fp32(cuda, case):
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    d = 12 if case == "d12" else 8
    net, params, _ = _mlp(d, 32, 3 if case == "layers3" else 2, seed=2, device=cuda)
    n, S = 512, 30
    x0, noise = _inputs(n, d, S, seed=2)
    kw = dict(seed=4, traj_layout=L.TRAJ_BLOCK128, emit_drift=True)
    if case == "injected":
        kw["noise"] = noise.float().to(cuda)
    if case == "particle_major":
        kw["traj_layout"] = L.TRAJ_PARTICLE_MAJOR
    a = ops.overdamped_integrate_model(x0.float().to(cuda), S, 0.01, net.spec, params["_flat"], path=L.PATH_FP32, **kw)
    b = ops.overdamped_integrate_model(x0.float().to(cuda), S, 0.01, net.spec, params["_flat"], path=L.PATH_TENSOR,
                                       **kw)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_block128_trajectory_feeds_the_fp_residual(cuda):
    """An overdamped BLOCK128 trajectory with emit_drift is a PDEIP_LAYOUT_BLOCK128 FP point set with
    PDEIP_DRIFT_IN_POINTS: SET_FP_0T on it equals the x-only points with TrueGrad(LINEAR, F) (fp32 path, 1e-5); the
    tensor residual takes it too."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    d, n, S, dt = 8, 1024, 16, 0.02
    F = _F(d).to(cuda)
    x0 = _inputs(n, d, 1, seed=12)[0].float().to(cuda)
    _, tr = ops.overdamped_integrate(x0, S, dt, L.DRIFT_LINEAR, F, seed=3, traj_layout=L.TRAJ_BLOCK128,
                                     emit_drift=True)
    pts_in = tr.reshape(S * n // 128, 2 * d, 128)
    pts_x = tr[:, :, :d].reshape(S * n // 128, d, 128).contiguous()
    spec = ops.ModelSpec(L.MODEL_MLP, d, 32, 2)
    flat = o_model.flatten_params(o_model.init_mlp_params(d, 32, 2, seed=5)).float().to(cuda)

    def residual(pts, tg, path):
        acc = ops.ResidualAccumulator(spec, device=cuda).begin()
        acc.accumulate(L.SET_FP_0T, flat, pts, 1.0 / (S * n), coef=1.0, layout=L.LAYOUT_BLOCK128, true_grad=tg,
                       path=path)
        s, g = acc.finalize()
        return s.cpu().double(), g.cpu().double()

    s_a, g_a = residual(pts_x, ops.TrueGrad(L.DRIFT_LINEAR, F), L.PATH_FP32)
    s_b, g_b = residual(pts_in, ops.TrueGrad(L.DRIFT_IN_POINTS), L.PATH_FP32)
    for k in (L.SUM_LOSS, L.SUM_GT, L.SUM_GTRUE2):
        assert relmax(s_b[k], s_a[k]) < 1e-5, k
    assert relmax(g_b, g_a) < 1e-5
    s_t, g_t = residual(pts_in, ops.TrueGrad(L.DRIFT_IN_POINTS), L.PATH_TENSOR)
    assert ops.tensor_path_status() == 0
    assert math.isfinite(s_t[L.SUM_LOSS].item()) and torch.isfinite(g_t).all()
    print(f"FP residual on the overdamped trajectory: tensor vs fp32 loss {relmax(s_t[L.SUM_LOSS], s_a[L.SUM_LOSS]):.2e}")


def test_coupled_simulation_error_on_the_fp_instance(cuda):
    """Exactly 0 for the quadratic model with W = F/2, b = 0 (its affine drift is the linear drift bit for bit), finite
    and positive for a random MLP, and a ValueError without n_steps (the FP configuration has no step count)."""
    from pde_inverse_problem_b200.core.model import V_parametric_quadratic
    from pde_inverse_problem_b200.utils.simulation import coupled_simulation_error
    pde = _fp(cuda)
    F = pde.initial_configuration["F"]
    qnet = V_parametric_quadratic(4)
    qparams = qnet.tree(torch.cat([(F / 2).reshape(-1), torch.zeros(4, device=cuda)]).contiguous())
    out = coupled_simulation_error(pde, functools.partial(qnet.apply, qparams), 4096, rng=5, n_steps=100)
    assert set(out) == {"coupled rms distance terminal", "relative mean error terminal",
                        "relative covariance error terminal"}
    for k, v in out.items():
        assert v.is_cuda and v.ndim == 0 and v.item() == 0.0, (k, v.item())
    net, params, _ = _mlp(4, 32, 2, seed=1, device=cuda)
    out = coupled_simulation_error(pde, functools.partial(net.apply, params), 4096, rng=5, n_steps=100)
    for k, v in out.items():
        assert math.isfinite(v.item()) and v.item() > 0, (k, v.item())
    with pytest.raises(ValueError, match="n_steps"):
        coupled_simulation_error(pde, functools.partial(net.apply, params), 4096, rng=5)
