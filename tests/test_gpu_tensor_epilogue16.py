"""One-slot tcgen05 residual kernels (d > 8, 16 epilogue warps: a thread owns 8 of the 32 hidden units and 8 + 2 of the
40 output units) against the fp32 path, at input widths whose last 8-component chunk is partly padding (d = 17, 20, 27)
or full (d = 32), over several tiles per CTA, in the three modes: KFP 0T set (stored true gradient in BLOCK128 rows,
the pipeline's layout), KFP boundary set and FP 0T set.  Tolerance as tests/test_gpu_tensor.py (rtol 1e-2, bf16 GEMM
operands)."""
import pytest
import torch

from conftest import relmax
from oracle import model as o_model

pytestmark = pytest.mark.gpu
TOL = 1e-2


def _ops():
    from pde_inverse_problem_b200 import ops, _lib
    return ops, _lib


def _flat(d, cuda, seed=5):
    p = o_model.init_mlp_params(d, 32, 2, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    for k in p["params"]:
        b = p["params"][k]["bias"]
        p["params"][k]["bias"] = 0.1 * torch.randn(b.shape, generator=g, dtype=torch.float64)
    return o_model.flatten_params(p).float().to(cuda)


def _run(ops, L, cuda, d, set_kind, flat, pts, n, path, **kw):
    acc = ops.ResidualAccumulator(ops.ModelSpec(L.MODEL_MLP, d, 32, 2), device=cuda).begin()
    acc.accumulate(set_kind, flat, pts, 1.0 / n, path=path, **kw)
    s, g = acc.finalize()
    assert ops.tensor_path_status() == 0, "a tcgen05 phase timed out"
    return s.cpu().double(), g.cpu().double()


@pytest.mark.parametrize("d", [17, 20, 27, 32])
def test_kfp_0t_block128_stored_gradient(cuda, d):
    ops, L = _ops()
    n = 128 * (148 * 3 + 5)  # 3-4 tiles per CTA
    g = torch.Generator().manual_seed(40 + d)
    rows = torch.randn(n, 3 * d, generator=g) * torch.cat([torch.full((d,), 1.5), torch.full((d,), 0.7), torch.ones(d)])
    pts = rows.reshape(n // 128, 128, 3 * d).transpose(1, 2).contiguous().to(cuda)  # [n / 128][3 d][128]
    flat = _flat(d, cuda)
    kw = dict(coef=0.5, true_grad=ops.TrueGrad(L.DRIFT_IN_POINTS), layout=L.LAYOUT_BLOCK128)
    s32, g32 = _run(ops, L, cuda, d, L.SET_KFP_0T, flat, pts, n, L.PATH_FP32, **kw)
    stc, gtc = _run(ops, L, cuda, d, L.SET_KFP_0T, flat, pts, n, L.PATH_TENSOR, **kw)
    for k in (L.SUM_LOSS, L.SUM_GT, L.SUM_G2, L.SUM_D2):
        assert relmax(stc[k], s32[k]) < TOL, (d, k)
    assert relmax(stc[L.SUM_GTRUE2], s32[L.SUM_GTRUE2]) < 1e-5  # stored gt: no GEMM in this term
    assert relmax(gtc, g32) < TOL
    _, gtc2 = _run(ops, L, cuda, d, L.SET_KFP_0T, flat, pts, n, L.PATH_TENSOR, **kw)
    assert torch.equal(gtc, gtc2)  # one writer per index, fixed order


@pytest.mark.parametrize("d", [17, 20, 27, 32])
def test_kfp_boundary_set(cuda, d):
    ops, L = _ops()
    n = 148 * 128 * 2 + 77  # ragged last tile
    g = torch.Generator().manual_seed(60 + d)
    pts = (torch.randn(n, 2 * d, generator=g) * 1.2).to(cuda)
    flat = _flat(d, cuda)
    s32, g32 = _run(ops, L, cuda, d, L.SET_KFP_BOUNDARY, flat, pts, n, L.PATH_FP32, coef=1.0)
    stc, gtc = _run(ops, L, cuda, d, L.SET_KFP_BOUNDARY, flat, pts, n, L.PATH_TENSOR, coef=1.0)
    # the boundary term is a cancelling mean (tests/test_gpu_tensor.py::test_boundary_sets_on_tensor_path): its error
    # is held against the mean |summand| scale, here that of the fp32 gradient
    assert abs(stc[L.SUM_BOUNDARY] - s32[L.SUM_BOUNDARY]) < TOL * g32.abs().max()
    assert relmax(gtc, g32) < TOL


@pytest.mark.parametrize("d", [17, 20, 27, 32])
def test_fp_0t_set(cuda, d):
    ops, L = _ops()
    n = 148 * 128 + 301  # d direction tiles per point tile: many tiles per CTA
    g = torch.Generator().manual_seed(80 + d)
    pts = (torch.randn(n, d, generator=g) * 1.5).to(cuda)
    mus = (torch.rand(8, d, generator=g) * 6 - 3).to(cuda)
    flat = _flat(d, cuda)
    kw = dict(true_grad=ops.TrueGrad(L.DRIFT_GMM, mus, 1.0))
    s32, g32 = _run(ops, L, cuda, d, L.SET_FP_0T, flat, pts, n, L.PATH_FP32, **kw)
    stc, gtc = _run(ops, L, cuda, d, L.SET_FP_0T, flat, pts, n, L.PATH_TENSOR, **kw)
    for k in (L.SUM_LOSS, L.SUM_GT, L.SUM_D2):
        assert relmax(stc[k], s32[k]) < TOL, (d, k)
    assert relmax(gtc, g32) < TOL
