"""Full-size checks through size-independent properties (BASELINE.json configs C2 / C3): analytic OU moments of the
production integrator kernel at 2^20 particles, and the chunked hot-path pipeline (tcgen05 residual against the fp32
residual on identical trajectories, shard invariance of the Philox streams)."""
import numpy as np
import pytest
import torch

from conftest import relmax
from oracle import moments as o_mom

pytestmark = pytest.mark.gpu


def _ops():
    from pde_inverse_problem_b200 import ops, _lib
    return ops, _lib


def test_c2_kinetic_ou_2e20_particles_match_analytic_moments(cuda):
    """C2: kinetic OU, d = 4, 2^20 particles, S = 100, T = 2 through the PRODUCTION kernel (reference schedule with
    per-particle tau0, Philox noise, [3d][S][N] trajectory with grad U).  The terminal ensemble matches the exact
    discrete-time moments of the scheme averaged over tau0 (KAT-2) to Monte-Carlo error and shows the scheme's own
    O(dt) gap to the continuous Lyapunov solution (KAT-1)."""
    ops, L = _ops()
    d, N, S, T = 4, 1 << 20, 100, 2.0
    dt = T / S
    cfg = o_mom.kinetic_ou_configuration(d)
    cfg["tilde_F"] = cfg["tilde_F"] / 4.0
    Z, I = np.zeros((d, d)), np.eye(d)
    cfg["F"] = np.block([[Z, I], [-cfg["tilde_F"], -cfg["gamma_friction"] * I]])
    A = torch.as_tensor(cfg["tilde_F"], dtype=torch.float32, device=cuda)
    z0 = ops.gaussian_sample(N, 2 * d, None, None, seed=5)
    chunk = 1 << 18
    traj = torch.empty(3 * d * S * chunk, device=cuda)
    zl = torch.empty_like(z0)
    for lo in range(0, N, chunk):
        ops.kl_integrate(z0[lo:lo + chunk], S, dt, cfg["gamma_friction"], L.DRIFT_LINEAR, A, seed=17, particle_offset=lo,
                         traj_layout=L.TRAJ_TIME_SOA, traj_out=traj, z_last_out=zl[lo:lo + chunk], emit_drift=True)
        # the emitted grad U of every sample is A x of that sample (last chunk checked below)
    tr = traj.view(3 * d, S, chunk)
    x_s = tr[:d, S // 2].T.double()
    g_s = tr[2 * d:, S // 2].T.double()
    assert relmax(g_s, x_s @ A.double().T) < 1e-5
    s1, s2 = ops.ensemble_moments(zl)
    mean = (s1 / N).cpu().double().numpy()
    cov = (s2 / N).cpu().double().numpy() - np.outer(mean, mean)
    # average the exact recursion over tau0 ~ U(0, dt) (mean zero => the covariance of the mixture is the average)
    taus = (np.arange(16) + 0.5) / 16 * dt
    P_d = np.mean([o_mom.discrete_mean_cov(S, dt, cfg, tau0=t)[1] for t in taus], axis=0)
    m_c, P_c = o_mom.lyapunov_mean_cov(T, cfg)
    rel_d = np.linalg.norm(cov - P_d) / np.linalg.norm(P_d)
    rel_c = np.linalg.norm(cov - P_c) / np.linalg.norm(P_c)
    gap = np.linalg.norm(P_d - P_c) / np.linalg.norm(P_c)
    assert rel_d < 6e-3, rel_d          # Monte-Carlo error at N = 2^20 (~0.3 %)
    assert np.abs(mean).max() < 6e-3
    assert abs(rel_c - gap) < 6e-3      # same statistical error / same O(dt) bias as the reference scheme


def _hot_path(cuda, path, chunk, n, offset=0, n_global=None, seed=3, d=8, K=16, S=40, host=False):
    import math
    from pde_inverse_problem_b200 import ops, _lib as L
    from pde_inverse_problem_b200.core.model import V_hypothesis
    from pde_inverse_problem_b200.pipeline import HotPath, HotPathConfig
    g = torch.Generator().manual_seed(1)
    mus = (torch.rand(K, d, generator=g) * 8 - 4).to(cuda)
    model = V_hypothesis(1, [32, 32], d)
    params = model.init(11, torch.zeros(d, device=cuda))
    cfg = HotPathConfig(d=d, n_steps=S, total_time=0.4, gamma=0.5, drift_kind=L.DRIFT_GMM, n_gaussian=K, chunk=chunk,
                        path=path)
    hp = HotPath(cfg, model, params, mus, ops.TrueGrad(L.DRIFT_GMM, mus, 1.0), optimizer=None, device=cuda)
    cov_half = torch.diag(torch.cat([torch.full((d,), 2.0), torch.full((d,), math.sqrt(0.1))])).to(cuda)
    z0 = ops.gaussian_sample(n, 2 * d, None, cov_half, seed=7, particle_offset=offset, device=cuda)
    if host:  # ensemble in pinned host memory: chunks are staged host -> device inside the step (double-buffered)
        zh = torch.empty((n, 2 * d), dtype=torch.float32, pin_memory=True)
        zh.copy_(z0)
        z0 = zh
    out = hp.step(z0, seed=seed, n_global=n_global or n, particle_offset=offset, apply_optimizer=False)
    torch.cuda.synchronize()
    return out["sums"].double().cpu(), out["grad"].double().cpu()


def test_pipeline_tensor_path_matches_fp32_path_and_is_chunk_invariant(cuda):
    """C3-shaped iteration (integrate -> 0T residual on the emitted trajectory -> boundary sets) on 2^15 particles x
    40 steps = 1.3 M residual points: tcgen05 path within 1e-2 of the fp32 path; the result does not depend on how the
    ensemble is chunked (Philox streams are keyed by the global particle id)."""
    from pde_inverse_problem_b200 import _lib as L
    n = 1 << 15
    s32, g32 = _hot_path(cuda, L.PATH_FP32, 1 << 13, n)
    stc, gtc = _hot_path(cuda, L.PATH_TENSOR, 1 << 13, n)
    assert relmax(stc[L.SUM_LOSS], s32[L.SUM_LOSS]) < 1e-2
    assert relmax(stc[L.SUM_GT], s32[L.SUM_GT]) < 1e-2
    assert relmax(gtc, g32) < 1e-2
    s32b, g32b = _hot_path(cuda, L.PATH_FP32, 1 << 12, n)
    assert relmax(s32b[L.SUM_LOSS], s32[L.SUM_LOSS]) < 1e-5
    assert relmax(g32b, g32) < 1e-5


def test_pipeline_shards_add_up(cuda):
    """Two half-ensembles with global particle offsets and 1/global weights add up to the single-rank result: the
    multi-GPU path needs one all-reduce(SUM) of [sums, grad] and nothing else."""
    from pde_inverse_problem_b200 import _lib as L
    n = 1 << 14
    s_all, g_all = _hot_path(cuda, L.PATH_TENSOR, 1 << 12, n)
    sa, ga = _hot_path(cuda, L.PATH_TENSOR, 1 << 12, n // 2, offset=0, n_global=n)
    sb, gb = _hot_path(cuda, L.PATH_TENSOR, 1 << 12, n // 2, offset=n // 2, n_global=n)
    assert relmax((sa + sb)[L.SUM_LOSS], s_all[L.SUM_LOSS]) < 1e-4
    assert relmax(ga + gb, g_all) < 1e-4


def test_pipeline_host_resident_ensemble_and_ragged_chunks(cuda):
    """The e2e configuration of bench.py (ensemble in pinned host memory, chunks copied on a side stream while the
    previous chunk is integrated) gives bit-identical sums and gradient to the device-resident run; a chunk size that
    is not a multiple of 128 (component-plane trajectory instead of 128-point blocks) agrees to rounding."""
    from pde_inverse_problem_b200 import _lib as L
    n = 1 << 14
    s_dev, g_dev = _hot_path(cuda, L.PATH_TENSOR, 1 << 12, n)
    s_host, g_host = _hot_path(cuda, L.PATH_TENSOR, 1 << 12, n, host=True)
    assert torch.equal(s_dev, s_host) and torch.equal(g_dev, g_host)
    s_rag, g_rag = _hot_path(cuda, L.PATH_TENSOR, 5000, n, host=True)
    assert relmax(s_rag[L.SUM_LOSS], s_dev[L.SUM_LOSS]) < 1e-4
    assert relmax(g_rag, g_dev) < 1e-4


def test_pipeline_c5_shape_tensor_integrator_matches_fp32(cuda):
    """C5-shaped iteration (d = 32, K = 64): integrator GMM contraction on tcgen05 + tcgen05 residual against the
    all-fp32 pipeline, tolerance class "bf16 GEMM paths" (1e-2)."""
    from pde_inverse_problem_b200 import _lib as L
    n = 1 << 12
    s32, g32 = _hot_path(cuda, L.PATH_FP32, 1 << 11, n, d=32, K=64, S=20)
    stc, gtc = _hot_path(cuda, L.PATH_TENSOR, 1 << 11, n, d=32, K=64, S=20)
    assert relmax(stc[L.SUM_LOSS], s32[L.SUM_LOSS]) < 1e-2
    assert relmax(stc[L.SUM_GT], s32[L.SUM_GT]) < 1e-2
    assert relmax(gtc, g32) < 1e-2


def test_bench_dumps_the_outputs_of_its_last_timed_step(cuda, tmp_path):
    """bench.py --dump-outputs DIR: the result of the last of exactly --steps timed steps, one float32 .npy per output
    (its loss is the loss of the JSON line), and the parameters that step left behind."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", "C3", "--particles", "8192",
                        "--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    j = json.loads(r.stdout)
    assert j["steps"] == 2
    names = {"loss", "loss_ground_truth", "sums", "grad", "grad_norm", "params_norm", "params"}
    assert {f[:-4] for f in os.listdir(tmp_path)} == names
    a = {k: np.load(tmp_path / (k + ".npy")) for k in names}
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert float(a["loss"]) == j["loss"]
    assert a["grad"].shape == a["params"].shape == (8 * 32 + 32 + 32 * 32 + 32 + 32 * 40 + 40,)
