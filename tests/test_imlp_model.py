"""The split-operand formulation of the tensor-core MLP drift (tests/imlp_model.py, the CPU twin of
csrc/integrator_mlp_tc.cu) against float64 autodiff through oracle/model.py, and the power of its tolerance TOL_MT: a
kernel that lost any one split term of any one of its six GEMMs would fail it."""
import pytest
import torch

from conftest import relmax
from imlp_model import GEMMS, TOL_MT, mlp_drift_tensor_model, padded_flat
from oracle import model as o_model


def _case(d, hidden, seed=3, n=4096):
    """(x, padded flat float32 parameters, float64 grad V of the same fp32-rounded network at x)"""
    p = o_model.init_mlp_params(d, hidden, 2, seed=seed + d + hidden)
    g = torch.Generator().manual_seed(seed)
    for k in p["params"]:
        p["params"][k]["bias"] = 0.1 * torch.randn(p["params"][k]["bias"].shape, generator=g, dtype=torch.float64)
        p["params"][k] = {kk: vv.float().double() for kk, vv in p["params"][k].items()}
    x = (torch.randn(n, d, generator=g, dtype=torch.float64) * 1.5).float().double()
    ref = torch.func.grad(lambda y: o_model.mlp_apply(p, y).sum())(x)
    return x, padded_flat(p, d), ref


CASES = [(d, h) for d in (8, 16, 32) for h in (32, 20)]


@pytest.mark.parametrize("d,hidden", CASES)
def test_split_operand_mlp_drift_matches_float64(d, hidden):
    """hi + lo on both operands of all six GEMMs: measured 2e-5 .. 5e-5 against float64 (max-norm relative)."""
    x, flat, ref = _case(d, hidden)
    err = relmax(mlp_drift_tensor_model(x, flat), ref)
    print(f"K1-MT twin d={d} hidden={hidden}: {err:.2e}")
    assert err < TOL_MT / 2, err


@pytest.mark.parametrize("d,hidden", CASES)
def test_every_dropped_split_term_exceeds_the_tolerance(d, hidden):
    """Dropping a_lo w_hi or a_hi w_lo from any ONE GEMM, a_lo w_hi from all six, or both lo terms everywhere (hi only)
    costs at least 3 TOL_MT: the drift assertion of tests/test_gpu_mlp_drift_precision.py tells each such defect apart
    from the correct kernel (the 1e-2 class bound does not: most single drops stay below it)."""
    x, flat, ref = _case(d, hidden)
    variants = {f"{gm} -{t}": {gm: tuple(s for s in ("hh", "lh", "hl") if s != t)} for gm in GEMMS for t in ("lh", "hl")}
    variants["-lh everywhere"] = {gm: ("hh", "hl") for gm in GEMMS}
    variants["hi only"] = {gm: ("hh",) for gm in GEMMS}
    errs = {k: relmax(mlp_drift_tensor_model(x, flat, terms=v), ref) for k, v in variants.items()}
    worst = min(errs, key=errs.get)
    print(f"K1-MT twin d={d} hidden={hidden}: smallest defect {worst} {errs[worst]:.2e}")
    assert errs[worst] > 3 * TOL_MT, (worst, errs[worst])
