"""The Fokker-Planck instance under a GMM potential on the GPU: the overdamped GMM drift on tcgen05 (K1-T-OD), the
FP-GMM problem instance, and the overdamped pipeline.HotPath.  Every test ends with ops.tensor_path_status() == 0."""
import functools
import math

import pytest
import torch

from conftest import relmax
from oracle import residuals as o_res
from overdamped_oracle import linear_moment_recursion, overdamped_langevin_scan

pytestmark = pytest.mark.gpu


def _mus(K, d, seed, scale=2.0):
    g = torch.Generator().manual_seed(seed)
    return ((torch.rand(K, d, generator=g, dtype=torch.float64) * 2.0 - 1.0) * scale).float()


def _gmm_grad64(mus, sigma=1.0):
    """float64 grad U of U = -log sum_k exp(-|x - mu_k|^2 / (2 sigma^2))"""
    m = mus.double()

    def grad(x):
        w = torch.softmax(-((x[:, None, :] - m[None]) ** 2).sum(-1) / (2 * sigma ** 2), -1)
        return (x - w @ m) / sigma ** 2
    return grad


def _run(x0, S, mus, path, dt=0.01, seed=5, **kw):
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    out = ops.overdamped_integrate(x0, S, dt, L.DRIFT_GMM, mus, n_gaussian=mus.shape[0], seed=seed, path=path, **kw)
    torch.cuda.synchronize()
    return out


def _pm(tr, layout, L):
    """trajectory -> particle-major [n, S, C]"""
    if layout == L.TRAJ_BLOCK128:
        S, nb, C, _ = tr.shape
        return tr.permute(1, 3, 0, 2).reshape(nb * 128, S, C)
    if layout == L.TRAJ_TIME_SOA:
        return tr.permute(2, 1, 0)
    if layout == L.TRAJ_TIME_MAJOR:
        return tr.permute(1, 0, 2)
    return tr


# ---------------------------------------------------------------------------------------------------------------------
# K1-T-OD on PDEIP_PATH_TENSOR
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [3, 16, 40, 64])
@pytest.mark.parametrize("d", [8, 16, 32])
def test_tensor_od_matches_float64(cuda, d, K):
    """S = 4 on the Philox draws of ops.philox_normals: the emitted drift against the float64 GMM gradient at the emitted
    positions, the emitted states and x_last against the float64 scan (rtol 1e-2 class, the max-norm is printed)."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    n, S, dt, seed = 1024, 4, 0.05, 11
    mus = _mus(K, d, seed=d + K)
    g = torch.Generator().manual_seed(3)
    x0 = (2.0 * torch.randn(n, d, generator=g)).to(cuda)
    noise = ops.philox_normals(n, S, d, seed).double().cpu()
    grad = _gmm_grad64(mus)
    last64, traj64 = overdamped_langevin_scan(x0.double().cpu(), S, dt, noise, grad)
    errs = {}
    for layout in (L.TRAJ_BLOCK128, L.TRAJ_TIME_SOA):
        xl, tr = _run(x0, S, mus.to(cuda), L.PATH_TENSOR, dt=dt, seed=seed, traj_layout=layout, emit_drift=True)
        pm = _pm(tr, layout, L).double().cpu()
        x_emit, g_emit = pm[:, :, :d], pm[:, :, d:]
        errs[f"drift{layout}"] = relmax(g_emit.reshape(-1, d), grad(x_emit.reshape(-1, d)))
        errs[f"states{layout}"] = relmax(x_emit, traj64)
        errs[f"last{layout}"] = relmax(xl, last64)
    xl, _ = _run(x0, S, mus.to(cuda), L.PATH_TENSOR, dt=dt, seed=seed, want_traj=False)
    errs["terminal"] = relmax(xl, last64)
    print(f"K1-T-OD vs float64 d={d} K={K}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert max(errs.values()) < 1e-2, errs
    assert ops.tensor_path_status() == 0


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


@pytest.mark.parametrize("dK", [(8, 16), (16, 32), (32, 64)])
def test_tensor_od_200_steps_match_fp32_kernel(cuda, dK):
    """200 steps on the same Philox draws, tensor against the fp32 kernel: max-norm 1e-2, median < 1e-4, 99.9 % within
    1e-2, moments within 1e-3; terminal-only at ragged n = 1000, BLOCK128 and TIME_SOA.  The last emitted sample is
    x_last bit for bit."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    d, K = dK
    S = 200
    mus = _mus(K, d, seed=100 + d).to(cuda)
    g = torch.Generator().manual_seed(9)
    x = (2.0 * torch.randn(1024, d, generator=g)).to(cuda)
    xt, _ = _run(x[:1000].contiguous(), S, mus, L.PATH_TENSOR, want_traj=False)
    assert ops.tensor_path_status() == 0
    xf, _ = _run(x[:1000].contiguous(), S, mus, L.PATH_FP32, want_traj=False)
    err = relmax(xt, xf)
    print(f"K1-T-OD vs fp32 d={d} K={K} terminal n=1000: {err:.2e}")
    assert torch.isfinite(xt).all() and err < 1e-2
    _assert_statistics(xt, xf, "terminal n=1000")
    _assert_moments(xt, xf)
    for layout in (L.TRAJ_BLOCK128, L.TRAJ_TIME_SOA):
        xt, tt = _run(x, S, mus, L.PATH_TENSOR, traj_layout=layout, emit_drift=True)
        assert ops.tensor_path_status() == 0
        xf, tf = _run(x, S, mus, L.PATH_FP32, traj_layout=layout, emit_drift=True)
        assert torch.equal(_pm(tt, layout, L)[:, -1, :d], xt)
        pt, pf = _pm(tt, layout, L), _pm(tf, layout, L)
        errs = [relmax(pt[..., :d], pf[..., :d]), relmax(pt[..., d:], pf[..., d:]), relmax(xt, xf)]
        print(f"K1-T-OD vs fp32 d={d} K={K} layout={layout}: traj {errs[0]:.2e} grad U {errs[1]:.2e} "
              f"last {errs[2]:.2e}")
        assert max(errs) < 1e-2
        _assert_statistics(pt[..., :d], pf[..., :d], f"layout={layout} traj")
        _assert_statistics(pt[..., d:], pf[..., d:], f"layout={layout} grad U")
        _assert_moments(xt, xf)
    assert ops.tensor_path_status() == 0


def test_tensor_od_single_centre_known_answer(cuda):
    """K = 1: grad U = x - mu, the scheme is OU around mu.  2^19 particles from N(m0, P0): the ensemble mean is within 5
    Monte-Carlo sigma of linear_moment_recursion(F = I) shifted by mu, the covariance within 1e-2 (relative Frobenius)."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    d, n, S, dt = 8, 1 << 19, 100, 0.01
    mu = _mus(1, d, seed=4)
    m0 = torch.full((d,), 0.5, dtype=torch.float64)
    P0 = torch.eye(d, dtype=torch.float64) * 2.0
    x0 = ops.gaussian_sample(n, d, m0.float().to(cuda), (P0.sqrt()).float().to(cuda), seed=3)
    xl, _ = _run(x0, S, mu.to(cuda), L.PATH_TENSOR, dt=dt, seed=8, want_traj=False)
    assert ops.tensor_path_status() == 0
    m, P = linear_moment_recursion(torch.eye(d, dtype=torch.float64), m0 - mu.double()[0], P0, S, dt)
    z = xl.double().cpu()
    mean, cov = z.mean(0), torch.cov(z.T)
    sig = torch.sqrt(torch.diagonal(P) / n)
    zscore = ((mean - (m + mu.double()[0])) / sig).abs().max().item()
    cov_err = (torch.linalg.matrix_norm(cov - P) / torch.linalg.matrix_norm(P)).item()
    print(f"K = 1 known answer: mean max |z| {zscore:.2f}, covariance {cov_err:.2e}")
    assert zscore < 5 and cov_err < 1e-2


@pytest.mark.parametrize("case", ["injected", "soa", "particle_major", "time_major", "emit_every2", "no_drift", "d12",
                                  "K65", "env"])
def test_tensor_od_outside_envelope_is_fp32(cuda, case, monkeypatch):
    """Outside K1-T-OD's envelope PDEIP_PATH_TENSOR runs the fp32 kernel: bit-identical to PDEIP_PATH_FP32."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    d = 12 if case == "d12" else 8
    K = 65 if case == "K65" else 16
    n, S = 512, 30
    mus = _mus(K, d, seed=2).to(cuda)
    g = torch.Generator().manual_seed(2)
    x0 = torch.randn(n, d, generator=g).to(cuda)
    kw = dict(traj_layout=L.TRAJ_BLOCK128, emit_drift=True)
    if case == "injected":
        kw["noise"] = torch.randn(n, S, d, generator=g).to(cuda)
    elif case == "soa":
        x0 = x0.T.contiguous()
        kw.update(state_layout=L.LAYOUT_SOA)
    elif case == "particle_major":
        kw["traj_layout"] = L.TRAJ_PARTICLE_MAJOR
    elif case == "time_major":
        kw["traj_layout"] = L.TRAJ_TIME_MAJOR
    elif case == "emit_every2":
        kw["emit_every"] = 2
    elif case == "no_drift":
        kw["emit_drift"] = False
    elif case == "env":
        monkeypatch.setenv("PDEIP_NO_TC_INTEGRATOR", "1")
    t = _run(x0, S, mus, L.PATH_TENSOR, **kw)
    f = _run(x0, S, mus, L.PATH_FP32, **kw)
    assert torch.equal(t[0], f[0]) and torch.equal(t[1], f[1]), case
    assert ops.tensor_path_status() == 0


@pytest.mark.parametrize("mode", ["terminal", "block128", "time_soa"])
def test_tensor_od_rank_invariance(cuda, mode):
    """Two launches over the halves with particle_offset equal one launch, bit for bit."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    d, n, S = 16, 2048, 40
    mus = _mus(16, d, seed=6).to(cuda)
    x0 = torch.randn(n, d, generator=torch.Generator().manual_seed(6)).to(cuda)
    kw = {"terminal": dict(want_traj=False), "block128": dict(traj_layout=L.TRAJ_BLOCK128, emit_drift=True),
          "time_soa": dict(traj_layout=L.TRAJ_TIME_SOA, emit_drift=True)}[mode]
    full = _run(x0, S, mus, L.PATH_TENSOR, seed=31, particle_offset=100, **kw)
    lo = _run(x0[: n // 2].contiguous(), S, mus, L.PATH_TENSOR, seed=31, particle_offset=100, **kw)
    hi = _run(x0[n // 2:].contiguous(), S, mus, L.PATH_TENSOR, seed=31, particle_offset=100 + n // 2, **kw)
    assert torch.equal(full[0], torch.cat([lo[0], hi[0]]))
    if mode == "block128":
        assert torch.equal(full[1], torch.cat([lo[1], hi[1]], 1))
    elif mode == "time_soa":
        assert torch.equal(full[1], torch.cat([lo[1], hi[1]], -1))
    assert ops.tensor_path_status() == 0


def test_model_gmm_forwards_to_the_tensor_kernel(cuda):
    """overdamped_integrate_model(MODEL_GMM) equals DRIFT_GMM with the same centres, bit for bit, on PATH_TENSOR."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    from pde_inverse_problem_b200.core.model import V_parametric_GMM
    d, K, n, S = 8, 16, 1024, 30
    net = V_parametric_GMM(dim=d, n_Gaussians=K)
    params = net.init(3, torch.zeros(d, device=cuda))
    mus = params["_flat"].view(K, d).clone()
    x0 = torch.randn(n, d, generator=torch.Generator().manual_seed(1)).to(cuda)
    for kw in (dict(want_traj=False), dict(traj_layout=L.TRAJ_BLOCK128, emit_drift=True)):
        a = ops.overdamped_integrate_model(x0, S, 0.01, net.spec, params["_flat"], seed=2, path=L.PATH_TENSOR, **kw)
        b = _run(x0, S, mus, L.PATH_TENSOR, seed=2, **kw)
        assert torch.equal(a[0], b[0]) and (a[1] is None or torch.equal(a[1], b[1]))
    assert ops.tensor_path_status() == 0


# ---------------------------------------------------------------------------------------------------------------------
# the FP-GMM problem instance
# ---------------------------------------------------------------------------------------------------------------------
def _instance(cuda, d=4, **over):
    from pde_inverse_problem_b200 import registry
    from pde_inverse_problem_b200.config import make_config
    cfg = make_config("fokker_planck", **{"pde_instance.domain_dim": d, "pde_instance.potential": "GMM",
                                          "estimation_mode": "non-parametric", "neural_network.layers": 2,
                                          "neural_network.hidden_dim": 32, "solver.train.batch_size_0T": 256, **over})
    return cfg, registry.get_pde_instance(cfg)(cfg=cfg, rng=7, device=cuda)


def _method(cfg, pde):
    from pde_inverse_problem_b200.methods.consistency import ConsistencyBased
    method = ConsistencyBased(pde_instance=pde, cfg=cfg, rng=1)
    net, params = method.create_model_fn()
    return method, net, params


def test_fp_gmm_sample_data(cuda):
    cfg, pde = _instance(cuda, **{"pde_instance.n_steps": 20})
    method, _, _ = _method(cfg, pde)
    data = method.sample_data(3)
    d, b = 4, 256
    assert tuple(data["0T"].shape) == (b * 20, d)
    assert tuple(data["initial"].shape) == (30 * b, d) and tuple(data["terminal"].shape) == (30 * b, d)
    assert all(torch.isfinite(v).all() for v in data.values())
    from pde_inverse_problem_b200 import ops
    assert ops.tensor_path_status() == 0


class _GmmProblem64:
    """what oracle.residuals.fp_value_and_grad_fn reads of the instance, in float64: T and V_true (the GMM potential,
    sigma = 1, up to its additive constant)"""

    def __init__(self, mus, T):
        self.mus, self.total_evolving_time = mus.double().cpu(), float(T)

    def V_true_fn(self, x):
        return -torch.logsumexp(-((x[None] - self.mus) ** 2).sum(-1) / 2.0, 0)


def test_fp_gmm_value_and_grad_matches_float64(cuda):
    """value_and_grad_fn on fp32 against oracle.residuals.fp_value_and_grad_fn in float64 on the same data (1e-5); the
    same sets accumulated on PATH_TENSOR (1e-2)."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    from pde_inverse_problem_b200.methods.consistency_instances import common
    from pde_inverse_problem_b200.methods.consistency_instances import fokker_planck as fp_mod
    from oracle import model as o_model
    cfg, pde = _instance(cuda, **{"pde_instance.n_steps": 10, "solver.train.batch_size_0T": 64})
    method, net, params = _method(cfg, pde)
    data = method.sample_data(5)
    out = fp_mod.value_and_grad_fn(net.apply, params, data, 0, pde)
    tree = net.tree(params["_flat"])["params"]
    p64 = {"params": {k: {"kernel": v["kernel"].double().cpu(), "bias": v["bias"].double().cpu()}
                      for k, v in tree.items()}}
    data64 = {k: v.double().cpu() for k, v in data.items()}
    ref = o_res.fp_value_and_grad_fn(o_model.mlp_apply, p64, data64, _GmmProblem64(pde.potential.mus,
                                                                                    pde.total_evolving_time))
    ref_grad = o_model.flatten_params(ref["grad"])
    e_loss = relmax(out["loss"], ref["loss"])
    e_grad = relmax(out["grad"]["_flat"], ref_grad)
    print(f"FP-GMM value_and_grad fp32 vs float64: loss {e_loss:.2e} grad {e_grad:.2e}")
    assert e_loss < 1e-5 and e_grad < 1e-5
    flat = net.flat(params)
    acc = common.accumulator_for(net, flat.device).begin()
    T = pde.total_evolving_time
    acc.accumulate(L.SET_FP_0T, flat, data["0T"], 1.0 / data["0T"].shape[0], true_grad=pde.true_grad_spec(),
                   path=L.PATH_TENSOR)
    acc.accumulate(L.SET_FP_BOUNDARY, flat, data["terminal"], 1.0 / data["terminal"].shape[0], coef=2.0 / T,
                   path=L.PATH_TENSOR)
    acc.accumulate(L.SET_FP_BOUNDARY, flat, data["initial"], 1.0 / data["initial"].shape[0], coef=-2.0 / T,
                   path=L.PATH_TENSOR)
    sums, grad = acc.finalize()
    e_loss = relmax(sums[L.SUM_LOSS], ref["loss"])
    e_grad = relmax(grad, ref_grad)
    print(f"FP-GMM value_and_grad tensor vs float64: loss {e_loss:.2e} grad {e_grad:.2e}")
    assert e_loss < 1e-2 and e_grad < 1e-2
    assert ops.tensor_path_status() == 0


def test_fp_gmm_test_fn_and_coupled_error(cuda):
    """test_fn keys are finite; coupled_simulation_error with V_parametric_GMM at the true centres is exactly 0 on both
    paths, and finite and positive for a random MLP."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    from pde_inverse_problem_b200.core.model import V_parametric_GMM
    from pde_inverse_problem_b200.utils.simulation import coupled_simulation_error
    cfg, pde = _instance(cuda, d=8, **{"pde_instance.n_steps": 30, "pde_instance.n_gaussian": 5})
    method, net, params = _method(cfg, pde)
    res = method.test_fn(net.apply, params, 4)
    assert res and all(torch.isfinite(v).all() for v in res.values()), res
    gmm = V_parametric_GMM(dim=8, n_Gaussians=5)
    gp = gmm.init(1, torch.zeros(8, device=cuda))
    gp["_flat"].copy_(pde.potential.mus.reshape(-1))
    for path in (L.PATH_FP32, L.PATH_TENSOR):
        r = coupled_simulation_error(pde, functools.partial(gmm.apply, gp), 4096, 9, n_steps=30, path=path)
        assert all(v.item() == 0.0 for v in r.values()), (path, r)
        r = coupled_simulation_error(pde, functools.partial(net.apply, params), 4096, 9, n_steps=30, path=path)
        assert all(math.isfinite(v.item()) and v.item() > 0 for v in r.values()), (path, r)
    assert ops.tensor_path_status() == 0


# ---------------------------------------------------------------------------------------------------------------------
# the overdamped HotPath
# ---------------------------------------------------------------------------------------------------------------------
def _hot_path(cuda, d, K, path, chunk=0):
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    from pde_inverse_problem_b200.core.model import V_hypothesis
    from pde_inverse_problem_b200.pipeline import HotPath, HotPathConfig
    mus = _mus(K, d, seed=20 + d).to(cuda)
    model = V_hypothesis(1, [32, 32], d)
    params = model.init(11, torch.zeros(d, device=cuda))
    cfg = HotPathConfig(d=d, n_steps=50, total_time=1.0, gamma=0.7, drift_kind=L.DRIFT_GMM, n_gaussian=K,
                        chunk=chunk, path=path, dynamics="overdamped")
    return HotPath(cfg, model, params, mus, ops.TrueGrad(L.DRIFT_IN_POINTS), device=cuda), mus, model, params


def test_hot_path_step_equals_composed_ops(cuda):
    """fp32: one step equals the integrator and residual ops composed by hand, bit for bit."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    d, K, n = 8, 16, 1024
    hp, mus, model, params = _hot_path(cuda, d, K, L.PATH_FP32)
    x0 = 2.0 * torch.randn(n, d, generator=torch.Generator().manual_seed(1)).to(cuda)
    out = hp.step(x0, seed=3, apply_optimizer=False)
    sums, grad = out["sums"].clone(), out["grad"].clone()
    S = hp.cfg.n_steps
    xl, tr = ops.overdamped_integrate(x0, S, 1.0 / S, L.DRIFT_GMM, mus, n_gaussian=K, seed=3,
                                      traj_layout=L.TRAJ_BLOCK128, emit_drift=True)
    acc = ops.ResidualAccumulator(model.spec, device=cuda).begin()
    flat = model.flat(params)
    acc.accumulate(L.SET_FP_0T, flat, tr.view(S * n // 128, 2 * d, 128), 1.0 / (n * S), layout=L.LAYOUT_BLOCK128,
                   true_grad=ops.TrueGrad(L.DRIFT_IN_POINTS))
    acc.accumulate(L.SET_FP_BOUNDARY, flat, xl, 1.0 / n, coef=2.0)
    acc.accumulate(L.SET_FP_BOUNDARY, flat, x0, 1.0 / n, coef=-2.0)
    s2, g2 = acc.finalize()
    assert torch.equal(sums, s2) and torch.equal(grad, g2)
    assert hp.particle_steps(n) == n * S
    assert ops.tensor_path_status() == 0


def test_hot_path_pinned_host_equals_device(cuda):
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    d, K, n = 8, 16, 1024 + 512
    hp, *_ = _hot_path(cuda, d, K, L.PATH_FP32, chunk=512)
    x0 = torch.randn(n, d, generator=torch.Generator().manual_seed(2)).to(cuda)
    a = {k: v.clone() for k, v in hp.step(x0, seed=4, apply_optimizer=False).items()}
    xh = torch.empty((n, d), dtype=torch.float32, pin_memory=True)
    xh.copy_(x0.cpu())
    b = hp.step(xh, seed=4, apply_optimizer=False)
    assert torch.equal(a["sums"], b["sums"]) and torch.equal(a["grad"], b["grad"])
    assert ops.tensor_path_status() == 0


def test_hot_path_ragged_chunks_match_single_chunk(cuda):
    """a BLOCK128 chunk plus a ragged TIME_SOA chunk against one chunk over all particles, 1e-6"""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    d, K, n = 8, 16, 1024 + 100
    hp1, *_ = _hot_path(cuda, d, K, L.PATH_FP32, chunk=1024)
    hp2, *_ = _hot_path(cuda, d, K, L.PATH_FP32, chunk=n)
    x0 = torch.randn(n, d, generator=torch.Generator().manual_seed(3)).to(cuda)
    a = {k: v.clone() for k, v in hp1.step(x0, seed=6, apply_optimizer=False).items()}
    b = hp2.step(x0, seed=6, apply_optimizer=False)
    e = (relmax(a["sums"][L.SUM_LOSS], b["sums"][L.SUM_LOSS]), relmax(a["grad"], b["grad"]))
    print(f"two chunks vs one: loss {e[0]:.2e} grad {e[1]:.2e}")
    assert max(e) < 1e-6
    assert ops.tensor_path_status() == 0


@pytest.mark.parametrize("dK", [(8, 16), (32, 64)])
def test_hot_path_tensor_step_matches_fp32(cuda, dK):
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    d, K = dK
    n = 4096
    x0 = 2.0 * torch.randn(n, d, generator=torch.Generator().manual_seed(4)).to(cuda)
    hpf, *_ = _hot_path(cuda, d, K, L.PATH_FP32)
    hpt, *_ = _hot_path(cuda, d, K, L.PATH_TENSOR)
    f = {k: v.clone() for k, v in hpf.step(x0, seed=7, apply_optimizer=False).items()}
    t = hpt.step(x0, seed=7, apply_optimizer=False)
    assert ops.tensor_path_status() == 0
    assert torch.isfinite(t["sums"]).all() and torch.isfinite(t["grad"]).all()
    e = (relmax(t["loss"], f["loss"]), relmax(t["grad"], f["grad"]))
    print(f"HotPath overdamped d={d} K={K} tensor vs fp32: loss {e[0]:.2e} grad {e[1]:.2e}")
    assert max(e) < 1e-2
