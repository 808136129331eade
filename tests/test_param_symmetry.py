"""The parameter symmetries of tests/param_symmetry.py, checked in float64 through the closed-form residual twin
(oracle/taylor.py:point_set) before any kernel relies on them: each transform reproduces the loss, the per-term sums
and (through its gradient map) the parameter gradient to 1e-12, in the three point-set modes the residual kernels
implement (KFP 0T, KFP boundary, FP 0T), and the input permutation maps the true GMM and linear drifts as stated."""
import pytest
import torch

from oracle import model as o_model
from oracle import potential as o_pot
from oracle import taylor as o_tay
from param_symmetry import transforms, tree_of


def _flat(d, seed=5):
    p = o_model.init_mlp_params(d, 32, 2, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    for k in p["params"]:
        p["params"][k]["bias"] = 0.1 * torch.randn(p["params"][k]["bias"].shape, generator=g, dtype=torch.float64)
    return o_model.flatten_params(p)


def _residual(flat, d, pts, mode):
    """(loss, [per-term sums], flat gradient, g) of one point set, float64"""
    W, b = o_tay.unpack(tree_of(flat, d))
    x, v = pts[:, :d], pts[:, d:2 * d]
    n = x.shape[0]
    if mode == "kfp_0t":
        val, dW, db, terms, g = o_tay.point_set(W, b, x, [(v, -2.0, 2.0 * 0.5)], 0.0, 1.0, 1.0 / n)
    elif mode == "kfp_boundary":
        val, dW, db, terms, g = o_tay.point_set(W, b, x, [(v, 0.0, 1.0)], 0.0, 0.0, 1.0 / n)
    else:
        eye = torch.eye(d, dtype=x.dtype)
        val, dW, db, terms, g = o_tay.point_set(W, b, x, [(eye[i].expand(n, d), -2.0, 0.0) for i in range(d)],
                                                0.0, 1.0, 1.0 / n)
    sums = torch.stack([terms["V"], terms["g2"], sum(terms["D1"]), sum(terms["D2"])])
    grad = torch.cat([torch.cat([w_.reshape(-1), b_.reshape(-1)]) for w_, b_ in zip(dW, db)])
    return val, sums, grad, g


@pytest.mark.parametrize("mode", ["kfp_0t", "kfp_boundary", "fp_0t"])
@pytest.mark.parametrize("d", [5, 17])
def test_transforms_preserve_the_residual(d, mode):
    g = torch.Generator().manual_seed(d)
    flat = _flat(d)
    pts = torch.randn(300, 2 * d, generator=g, dtype=torch.float64) * 1.5
    val, sums, grad, gx = _residual(flat, d, pts, mode)
    for t in transforms(d, seed=3):
        val_t, sums_t, grad_t, gx_t = _residual(t.params(flat), d, t.points(pts, d), mode)
        scale = grad.abs().max()
        assert abs(val_t - val) <= 1e-12 * abs(val), t.name
        assert ((sums_t - sums).abs() <= 1e-12 * sums.abs().max()).all(), t.name
        assert (grad_t - t.grad(grad)).abs().max() <= 1e-12 * scale, t.name
        assert (gx_t - t.points(gx, d)).abs().max() <= 1e-12 * gx.abs().max(), t.name  # grad_x V moves with tau
        assert not torch.equal(t.params(flat), flat), t.name  # every transform moves something


@pytest.mark.parametrize("d", [5, 17])
def test_input_permutation_maps_the_true_drifts(d):
    """grad V_true of the transformed problem at the transformed points is the permuted true gradient: GMM centres
    mus[:, tau], linear drift F[tau][:, tau]."""
    g = torch.Generator().manual_seed(7)
    x = torch.randn(200, d, generator=g, dtype=torch.float64) * 2
    mus = torch.rand(9, d, generator=g, dtype=torch.float64) * 8 - 4
    F = torch.randn(d, d, generator=g, dtype=torch.float64)
    for t in transforms(d, seed=3):
        if t.tau is None:
            continue
        xt = t.points(x, d)
        ref = o_pot.vg_gmm_V(x, mus, 1.0)
        assert (o_pot.vg_gmm_V(xt, t.mus(mus), 1.0) - t.points(ref, d)).abs().max() < 1e-12, t.name
        assert (xt @ t.linear(F).T - t.points(x @ F.T, d)).abs().max() < 1e-12, t.name
