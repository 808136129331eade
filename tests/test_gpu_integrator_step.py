"""The tcgen05 integrators step by step: the drift class of the GMM drift at the kernel's own emitted positions, and a
bit-exact replay of every emitted step.

* Drift class of K1-T and K1-T-OD (csrc/integrator_tc.cu).  Every emitted grad U at its emitted position, against
  float64 (oracle/potential.py) and against the CPU twin of the kernel's arithmetic (tests/itc_model.py), for both
  dynamics and both trajectory layouts.  Comparing emitted pairs (x_s, g_s) takes the chaotic divergence of
  trajectories out of the measure.  Three ensembles, each with its own max-norm:
  - "normal": x ~ N(0, 4 I), centres ~ U[-4, 4]^d.  Against float64 at TOL_T max(1, sigma^-2): the logits scale as
    sigma^-2, and so does the split error of GEMM 1.  tests/test_itc_model.py shows that TOL_T rejects a formulation
    that loses any one of x_lo mu_hi, x_hi mu_lo, b1, e_lo mu_hi and e_hi mu_lo (at sigma = 1).
  - "bisector": x on the bisector of two centres.  The drift there is x less the mean of the two centres, small against
    x, and so is the max-norm it is measured in: against float64 at 4 times the "normal" bound, against the twin at
    TWIN_TOL_BISECTOR.
  - "far": x ~ N(0, (12 sigma)^2 I), tens of sigma from every centre, where the Gaussian weights underflow in fp32
    and only the max-subtracted softmax survives.  Against the twin only: the twin itself is within 5e-4 of float64
    there (tests/test_itc_model.py).
  "normal" and "far" are held to TWIN_TOL against the twin.
* Step replay of all four tcgen05 integrators: K1-T, K1-T-OD, K1-MT and K1-MT-OD (csrc/integrator_mlp_tc.cu).  The
  update is fixed by fused multiply-adds, so it is deterministic in fp32:
    kinetic     p <- fma(sq, xi_s, fl(p dmp)) ; p <- fma(-h, g, p) ; q <- fma(h, p, q)
    overdamped  x <- fma(-h, g, fma(sq, xi_s, x))
  with sq = fl(fl(sqrt(h)) fl32(sqrt 2)) and dmp = fl(1 - gamma h).  From the emitted [x, (v,) g] and the draws of
  ops.philox_normals, fma32 (tests/fp32_exact.py) replays every emitted step, and the replay must equal the kernel
  bit for bit (torch.equal).  dt = 2^-7 and gamma = 0.5 make gamma h exact, so dmp does not depend on whether the
  compiler fuses it.  Kinetic: samples 1 .. S-1 (h = dt); the first and last steps take h = tau0 and dt - tau0 and
  are not replayed.  Overdamped: every sample after the first, and the last sample is x_last.  The first sample
  needs grad U(x0), which is never emitted: it is held to the twin's drift at x0, within h TWIN_TOL of the scale.
  The replay also pins the noise: the kernels' Philox draws must equal ops.philox_normals bit for bit.

Measured on a B200 (1000 W power limit, profiles/r03_tc_precision.txt), the drift over the 60 cases: "normal" against
float64 1.5e-6 .. 1.1e-4 at sigma >= 1 and up to 2.3e-4 at sigma = 0.7 (bound 4.1e-4), against the twin <= 1.4e-5;
"bisector" against float64 up to 2.7 times the "normal" bound, against the twin <= 7.3e-5; "far" against the twin
<= 6.8e-6.  Replay: 0 differing elements in every case; the first step within 1/4 of its bound."""
import numpy as np
import pytest
import torch

from conftest import relmax
from fp32_exact import fma32
from imlp_model import mlp_drift_tensor_model
from itc_model import TOL_T, gmm_grad_tensor_model
from oracle import potential as o_pot

pytestmark = pytest.mark.gpu
# K1-T / K1-T-OD against the twin: ex2.approx, the tensor cores' fp32 accumulation order and the split pairs that
# follow from a last-bit difference.  About 3x the largest values measured on the B200 (1.4e-5, bisector 7.3e-5).
TWIN_TOL = 4e-5
TWIN_TOL_BISECTOR = 2.2e-4
TWIN_TOL_MT = 3e-5  # K1-MT against its twin (tests/test_gpu_mlp_drift_precision.py)
SQRT2 = np.float32(1.41421356237309515)


def _lib():
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    return L, ops


def _pm(tr, layout, L):
    """trajectory ([S][n/128][C][128] or [C][S][n]) -> particle-major [n, S, C]"""
    if layout == L.TRAJ_BLOCK128:
        S, nb, C, _ = tr.shape
        return tr.permute(1, 3, 0, 2).reshape(nb * 128, S, C)
    return tr.permute(2, 1, 0)


def _status_ok(ops):
    torch.cuda.synchronize()
    assert ops.tensor_path_status() == 0, "a tcgen05 phase timed out"


def _mus(K, d, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(K, d, generator=g) * 8 - 4


def _ensembles(n, d, mus, sigma, seed):
    """x0 [n, d] and the index sets of the three ensembles (normal | bisector | far)"""
    g = torch.Generator().manual_seed(seed)
    K = mus.shape[0]
    n1, n2 = n // 2, n // 4
    x = torch.randn(n, d, generator=g) * 2.0
    ia = torch.randint(0, K, (n2,), generator=g)
    ib = (ia + 1 + torch.randint(0, max(K - 1, 1), (n2,), generator=g)) % K
    dv = (mus[ia] - mus[ib]).double()
    w = torch.randn(n2, d, generator=g, dtype=torch.float64) * 0.5
    w -= (w * dv).sum(-1, keepdim=True) / (dv * dv).sum(-1, keepdim=True).clamp_min(1e-30) * dv
    x[n1:n1 + n2] = (0.5 * (mus[ia] + mus[ib]).double() + w).float()
    x[n1 + n2:] = torch.randn(n - n1 - n2, d, generator=g) * (12.0 * sigma)
    idx = torch.arange(n)
    return x, {"normal": idx[:n1], "bisector": idx[n1:n1 + n2], "far": idx[n1 + n2:]}


# (d, K, sigma, S): every K-padding case (K = 1, 3, 16, 17, 40, 64) at d = 8 and at d = 32, three at d = 16
_DRIFT_CASES = [
    (8, 1, 1.0, 20), (8, 3, 0.7, 2), (8, 16, 1.0, 20), (8, 17, 2.5, 20), (8, 40, 1.0, 1), (8, 64, 0.7, 20),
    (32, 1, 2.5, 2), (32, 3, 1.0, 20), (32, 16, 0.7, 20), (32, 17, 1.0, 1), (32, 40, 2.5, 20), (32, 64, 1.0, 20),
    (16, 3, 1.0, 20), (16, 40, 0.7, 2), (16, 64, 2.5, 20)]


@pytest.mark.parametrize("layout", ["block128", "time_soa"])
@pytest.mark.parametrize("dyn", ["kinetic", "overdamped"])
@pytest.mark.parametrize("d,K,sigma,S", _DRIFT_CASES)
def test_gmm_emitted_drift_class(cuda, d, K, sigma, S, dyn, layout):
    """Ragged n = 1000 (TIME_SOA) or 1024 (BLOCK128), dt = 1e-3, Philox noise: every emitted grad U against float64 and
    the twin at the emitted position.  S = 1 of the overdamped kernel emits one sample, whose drift comes from the
    drift-only last iteration."""
    L, ops = _lib()
    tl = L.TRAJ_BLOCK128 if layout == "block128" else L.TRAJ_TIME_SOA
    n = 1024 if layout == "block128" else 1000
    mus = _mus(K, d, seed=10 * d + K)
    x0, groups = _ensembles(n, d, mus, sigma, seed=d + K + S)
    if dyn == "kinetic":
        v0 = torch.randn(n, d, generator=torch.Generator().manual_seed(K)) * 0.3
        _, tr, _ = ops.kl_integrate(torch.cat([x0, v0], 1).to(cuda), S, 1e-3, 0.5, L.DRIFT_GMM, mus.to(cuda),
                                    n_gaussian=K, sigma=sigma, seed=17, particle_offset=333, traj_layout=tl,
                                    emit_drift=True, path=L.PATH_TENSOR)
    else:
        _, tr = ops.overdamped_integrate(x0.to(cuda), S, 1e-3, L.DRIFT_GMM, mus.to(cuda), n_gaussian=K, sigma=sigma,
                                         seed=17, particle_offset=333, traj_layout=tl, emit_drift=True,
                                         path=L.PATH_TENSOR)
    _status_ok(ops)
    pm = _pm(tr, tl, L)
    x, g = pm[..., :d], pm[..., -d:]
    assert torch.isfinite(g).all()
    tol64 = TOL_T * max(1.0, sigma ** -2)
    kp = (K + 15) // 16 * 16
    # the bound of each (ensemble, reference) pair; the far ensemble against the twin only
    bounds = {("normal", "float64"): tol64, ("normal", "twin"): TWIN_TOL, ("bisector", "float64"): 4 * tol64,
              ("bisector", "twin"): TWIN_TOL_BISECTOR, ("far", "twin"): TWIN_TOL}
    errs = {}
    for name, idx in groups.items():
        xs, gs = x[idx.to(cuda)].reshape(-1, d), g[idx.to(cuda)].reshape(-1, d)
        errs[name, "twin"] = relmax(gs, gmm_grad_tensor_model(xs.cpu(), mus, sigma, k_pad=kp))
        if (name, "float64") in bounds:
            errs[name, "float64"] = relmax(gs, o_pot.vg_gmm_V(xs.double(), mus.double().to(cuda), sigma))
    print(f"K1-T{'-OD' if dyn == 'overdamped' else ''} drift d={d} K={K} sigma={sigma} S={S} {layout}: " +
          ", ".join(f"{k[0]} vs {k[1]} {e:.2e}" for k, e in sorted(errs.items())))
    for k, e in errs.items():
        assert e < bounds[k], (k, e, bounds[k])


# ---------------------------------------------------------------------------------------------------------------------
# bit-exact step replay
# ---------------------------------------------------------------------------------------------------------------------
def _sq(h: float) -> np.float32:
    """sqrt(2h) as the kernels form it: sqrtf (correctly rounded) times sqrt 2 rounded to fp32, in fp32"""
    h32 = np.float32(h)
    return np.float32(np.sqrt(h32)) * SQRT2


def _c(v, like):
    return torch.tensor(float(v), dtype=torch.float32, device=like.device)


def _mismatch(a, b):
    return int((a != b).sum().item())


def _replay_od(x, g, xi, h):
    """x, g [n, S, d] emitted, xi [n, S, d] draws: x_{s+1} = fma(-h, g_s, fma(sq, xi_{s+1}, x_s)) for s = 0 .. S-2"""
    y = fma32(_c(_sq(h), x), xi[:, 1:], x[:, :-1])
    return fma32(_c(-np.float32(h), x), g[:, :-1], y)


def _replay_kinetic(q, p, g, xi, h, gamma):
    """samples 1 .. S-1 from samples 0 .. S-2 (h = dt) with draws 1 .. S-1"""
    h32 = np.float32(h)
    dmp = np.float32(1) - np.float32(gamma) * h32
    S = q.shape[1]
    p1 = fma32(_c(_sq(h), q), xi[:, 1:S], p[:, :-1] * _c(dmp, p))
    p2 = fma32(_c(-h32, q), g[:, :-1], p1)
    return fma32(_c(h32, q), p2, q[:, :-1]), p2


def _check_first_od(x0, x, xi, h, drift0, tol):
    """sample 0 = fma(-h, grad U(x0), fma(sq, xi_0, x0)): grad U(x0) is not emitted; with the twin's drift at x0 the
    replay is within h tol max|grad U| (+ one ulp of the sample)"""
    y = fma32(_c(_sq(h), x0), xi[:, 0], x0)
    pred = fma32(_c(-np.float32(h), x0), drift0.to(x0.device), y)
    err = (pred.double() - x[:, 0].double()).abs().max().item()
    ulp = (torch.nextafter(x[:, 0].abs(), torch.full_like(x[:, 0], float("inf"))) - x[:, 0].abs()).max().item()
    bound = float(h) * tol * drift0.abs().max().item() + ulp
    return err, bound


# (d, K, n, S, dt, layout): ragged n over several CTAs, both layouts, one case at n = 2^16, S = 50
_OD_REPLAY = [
    (8, 16, 1000, 20, 2 ** -7, "time_soa"), (16, 40, 777, 20, 2 ** -7, "time_soa"),
    (32, 64, 1000, 20, 2 ** -7, "time_soa"), (8, 3, 1024, 20, 2 ** -7, "block128"),
    (16, 1, 300, 20, 0.01, "time_soa"), (32, 17, 1024, 20, 0.01, "block128"),
    (32, 64, 1 << 16, 50, 2 ** -7, "block128")]


@pytest.mark.parametrize("d,K,n,S,dt,layout", _OD_REPLAY)
def test_od_gmm_step_replay(cuda, d, K, n, S, dt, layout):
    """K1-T-OD: every emitted step replayed bit for bit; the last sample is x_last; a terminal-only run ends on the same
    x_last and overdamped_integrate_model(MODEL_GMM) on the same outputs, bit for bit; the first step within the twin's
    drift class."""
    from pde_inverse_problem_b200.core.model import V_parametric_GMM
    L, ops = _lib()
    tl = L.TRAJ_BLOCK128 if layout == "block128" else L.TRAJ_TIME_SOA
    mus = _mus(K, d, seed=d + K).to(cuda)
    x0 = (torch.randn(n, d, generator=torch.Generator().manual_seed(n + d)) * 2.0).to(cuda)
    kw = dict(seed=91, particle_offset=501, step_offset=7)
    xl, tr = ops.overdamped_integrate(x0, S, dt, L.DRIFT_GMM, mus, n_gaussian=K, traj_layout=tl, emit_drift=True,
                                      path=L.PATH_TENSOR, **kw)
    _status_ok(ops)
    xl_t, _ = ops.overdamped_integrate(x0, S, dt, L.DRIFT_GMM, mus, n_gaussian=K, want_traj=False,
                                       path=L.PATH_TENSOR, **kw)
    _status_ok(ops)
    net = V_parametric_GMM(dim=d, n_Gaussians=K)
    xl_m, tr_m = ops.overdamped_integrate_model(x0, S, dt, net.spec, mus.reshape(-1).contiguous(), traj_layout=tl,
                                                emit_drift=True, path=L.PATH_TENSOR, **kw)
    _status_ok(ops)
    xi = ops.philox_normals(n, S, d, **kw)
    pm = _pm(tr, tl, L)
    x, g = pm[..., :d], pm[..., d:]
    rep = _replay_od(x, g, xi, dt)
    bad = _mismatch(rep, x[:, 1:])
    err0, bound0 = _check_first_od(x0, x, xi, dt, gmm_grad_tensor_model(x0.cpu(), mus.cpu(), 1.0,
                                                                          k_pad=(K + 15) // 16 * 16), TWIN_TOL)
    print(f"K1-T-OD replay d={d} K={K} n={n} S={S} dt={dt} {layout}: {bad} of {rep.numel()} elements differ; "
          f"first step {err0:.1e} (bound {bound0:.1e})")
    assert bad == 0
    assert torch.equal(x[:, -1], xl)
    assert torch.equal(xl_t, xl)
    assert torch.equal(xl_m, xl) and torch.equal(tr_m, tr)
    assert err0 <= bound0, (err0, bound0)


# (d, K, n, S, layout)
_KIN_REPLAY = [(8, 16, 1000, 20, "time_soa"), (16, 40, 1024, 20, "block128"), (32, 64, 1000, 20, "time_soa"),
               (8, 64, 384, 20, "block128"), (32, 7, 1 << 16, 50, "block128")]


@pytest.mark.parametrize("d,K,n,S,layout", _KIN_REPLAY)
def test_kinetic_gmm_step_replay(cuda, d, K, n, S, layout):
    """K1-T (REFERENCE schedule, iteration s draws xi_s of S + 1 draws): samples 1 .. S-1 replayed bit for bit."""
    L, ops = _lib()
    tl = L.TRAJ_BLOCK128 if layout == "block128" else L.TRAJ_TIME_SOA
    dt, gamma = 2 ** -7, 0.5
    mus = _mus(K, d, seed=d + K).to(cuda)
    gen = torch.Generator().manual_seed(n + d)
    z0 = torch.cat([torch.randn(n, d, generator=gen) * 2.0, torch.randn(n, d, generator=gen) * 0.3], 1).to(cuda)
    kw = dict(seed=92, particle_offset=502, step_offset=9)
    _, tr, _ = ops.kl_integrate(z0, S, dt, gamma, L.DRIFT_GMM, mus, n_gaussian=K, traj_layout=tl, emit_drift=True,
                                path=L.PATH_TENSOR, **kw)
    _status_ok(ops)
    xi = ops.philox_normals(n, S + 1, d, **kw)
    pm = _pm(tr, tl, L)
    q, p, g = pm[..., :d], pm[..., d:2 * d], pm[..., 2 * d:]
    rq, rp = _replay_kinetic(q, p, g, xi, dt, gamma)
    bad = (_mismatch(rq, q[:, 1:]), _mismatch(rp, p[:, 1:]))
    print(f"K1-T replay d={d} K={K} n={n} S={S} {layout}: {bad[0]} (x), {bad[1]} (v) of {rq.numel()} elements differ")
    assert bad == (0, 0)


def _mlp(d, cuda):
    from test_gpu_mlp_drift_precision import _mlp as mlp
    spec, flat, _ = mlp(d, 32, seed=70 + d, cuda=cuda)
    return spec, flat


@pytest.mark.parametrize("layout", ["block128", "time_soa"])
@pytest.mark.parametrize("d", [8, 16, 32])
def test_mlp_step_replay(cuda, d, layout):
    """K1-MT and K1-MT-OD (MLP 32 x 2, inside integrate_mlp_tensor_ok / overdamped_mlp_tensor_ok): every emitted step
    replayed bit for bit (kinetic: samples 1 .. S-1); overdamped: the last sample is x_last, the first step within
    the twin's drift class."""
    L, ops = _lib()
    tl = L.TRAJ_BLOCK128 if layout == "block128" else L.TRAJ_TIME_SOA
    n = 1024 if layout == "block128" else 1000
    S, dt, gamma = 20, 2 ** -7, 0.5
    spec, flat = _mlp(d, cuda)
    gen = torch.Generator().manual_seed(d)
    x0 = (torch.randn(n, d, generator=gen) * 1.5).to(cuda)
    v0 = (torch.randn(n, d, generator=gen) * 0.3).to(cuda)
    kw = dict(seed=93, particle_offset=503, step_offset=11)
    _, tr, _ = ops.kl_integrate_model(torch.cat([x0, v0], 1), S, dt, gamma, spec, flat, traj_layout=tl,
                                      emit_drift=True, path=L.PATH_TENSOR, **kw)
    _status_ok(ops)
    pm = _pm(tr, tl, L)
    q, p, g = pm[..., :d], pm[..., d:2 * d], pm[..., 2 * d:]
    rq, rp = _replay_kinetic(q, p, g, ops.philox_normals(n, S + 1, d, **kw), dt, gamma)
    bad_k = (_mismatch(rq, q[:, 1:]), _mismatch(rp, p[:, 1:]))

    xl, tr = ops.overdamped_integrate_model(x0, S, dt, spec, flat, traj_layout=tl, emit_drift=True,
                                            path=L.PATH_TENSOR, **kw)
    _status_ok(ops)
    xi = ops.philox_normals(n, S, d, **kw)
    pm = _pm(tr, tl, L)
    x, g = pm[..., :d], pm[..., d:]
    bad_o = _mismatch(_replay_od(x, g, xi, dt), x[:, 1:])
    err0, bound0 = _check_first_od(x0, x, xi, dt, mlp_drift_tensor_model(x0.cpu(), flat), TWIN_TOL_MT)
    print(f"K1-MT replay d={d} {layout}: kinetic {bad_k[0]} (x), {bad_k[1]} (v) differ; overdamped {bad_o} differ, "
          f"first step {err0:.1e} (bound {bound0:.1e})")
    assert bad_k == (0, 0) and bad_o == 0
    assert torch.equal(x[:, -1], xl)
    assert err0 <= bound0, (err0, bound0)
