"""The split-operand formulation of the tensor-core GMM drift (tests/itc_model.py, the CPU twin of
csrc/integrator_tc.cu) against the float64 closed form of the reference (oracle/potential.py <- core/potential.py:32-61)."""
import pytest
import torch

from conftest import relmax
from itc_model import GEMM1, TERMS, TOL_T, gmm_grad_tensor_model
from oracle import potential as o_pot


@pytest.mark.parametrize("d,K,k_pad", [(8, 16, 16), (32, 64, 64), (16, 33, 48), (32, 7, 16), (8, 3, 16)])
def test_split_operand_gmm_gradient_matches_closed_form(d, K, k_pad):
    """C3 / C5 shaped ensembles (x0 ~ N(0, 4 I), centres ~ U[-4, 4]^d, GMM.py:17-42): two bf16 terms per operand keep
    the tensor-core formulation within 2e-4 (per-tensor max-norm) of the float64 gradient; a single bf16 term does not."""
    g = torch.Generator().manual_seed(d * 100 + K)
    x = torch.randn(4096, d, generator=g, dtype=torch.float64) * 2.0
    mus = torch.rand(K, d, generator=g, dtype=torch.float64) * 8 - 4
    ref = o_pot.vg_gmm_V(x, mus, 1.0)
    got = gmm_grad_tensor_model(x, mus, 1.0, k_pad=k_pad)
    assert torch.isfinite(got).all()
    assert relmax(got, ref) < 2e-4
    # what the split buys: plain bf16 operands (no lo terms) are orders of magnitude worse
    xb = x.to(torch.bfloat16).double()
    mb = mus.to(torch.bfloat16).double()
    assert relmax(o_pot.vg_gmm_V(xb, mb, 1.0), ref) > 10 * relmax(got, ref)


def test_split_operand_gmm_gradient_far_from_all_centres():
    """Particles tens of sigma away from every centre: the Gaussian weights underflow in fp32, the max-subtracted
    logits do not (the row constant -c |x|^2 / 2 is never formed)."""
    g = torch.Generator().manual_seed(5)
    mus = torch.rand(64, 32, generator=g, dtype=torch.float64) * 8 - 4
    x = torch.randn(512, 32, generator=g, dtype=torch.float64) * 12.0
    got = gmm_grad_tensor_model(x, mus, 1.0, k_pad=64)
    assert torch.isfinite(got).all()
    assert relmax(got, o_pot.vg_gmm_V(x, mus, 1.0)) < 5e-4


def test_sigma_scaling():
    g = torch.Generator().manual_seed(6)
    mus = torch.rand(16, 8, generator=g, dtype=torch.float64) * 8 - 4
    x = torch.randn(1000, 8, generator=g, dtype=torch.float64) * 2.0
    for sigma in (0.7, 1.0, 2.5):
        assert relmax(gmm_grad_tensor_model(x, mus, sigma, k_pad=16), o_pot.vg_gmm_V(x, mus, sigma)) < 3e-4


# (d, K) of C3 / C5 shaped ensembles; K = 17 leaves 15 padding centres in its second 16-centre chunk
_SHAPES = [(8, 16), (16, 32), (32, 64), (8, 3), (16, 40), (32, 7), (16, 17)]
# the split terms whose loss the drift tolerance must see; b2 (the third bias term, ~2^-17 of the bias) is below the
# resolution of the comparison with float64 (<= 1.7e-4) and is not claimed
_DETECTABLE = ("xl.muh", "xh.mul", "b1", "el.muh", "eh.mul")


def _ensemble(d, K, n=8192):
    g = torch.Generator().manual_seed(d * 100 + K)
    x = torch.randn(n, d, generator=g, dtype=torch.float64) * 2.0
    mus = torch.rand(K, d, generator=g, dtype=torch.float64) * 8 - 4
    return x, mus, o_pot.vg_gmm_V(x, mus, 1.0), (K + 15) // 16 * 16


@pytest.mark.parametrize("d,K", _SHAPES + [(8, 1), (32, 17)])
def test_twin_within_tol_t(d, K):
    """The full twin is within TOL_T of float64 (8192 points, x ~ N(0, 4 I), centres ~ U[-4, 4]^d)."""
    x, mus, ref, kp = _ensemble(d, K)
    err = relmax(gmm_grad_tensor_model(x, mus, 1.0, k_pad=kp), ref)
    print(f"GMM twin d={d} K={K}: vs float64 {err:.1e} (TOL_T {TOL_T:.0e})")
    assert err < TOL_T, err


@pytest.mark.parametrize("d,K", _SHAPES)
def test_tol_t_sees_every_dropped_split_term(d, K):
    """Each of x_lo mu_hi, x_hi mu_lo (GEMM 1), the second bias term b1, e_lo mu_hi and e_hi mu_lo (GEMM 2) left out costs
    more than 2 TOL_T against float64 on every shape, so the drift assertion of tests/test_gpu_integrator_step.py tells
    a kernel that lost one of them apart.  Printed: the error of every single-term variant (b2 included, not asserted)."""
    x, mus, ref, kp = _ensemble(d, K)
    errs = {t: relmax(gmm_grad_tensor_model(x, mus, 1.0, k_pad=kp, drop=(t,)), ref) for t in TERMS}
    print(f"GMM twin d={d} K={K} without: " + ", ".join(f"{t} {e:.1e}" for t, e in errs.items()))
    for t in _DETECTABLE:
        assert errs[t] > 2 * TOL_T, (t, errs[t])


def test_single_centre_sees_only_e_hi_mu_lo():
    """K = 1: the softmax weight is 2^0 = 1 whatever the logit, so GEMM 1, the bias terms b1, b2 and e_lo (= 0) do not
    reach the drift (bit-identical without them; b0 also carries the -1e30 of the 15 padding centres); e_hi mu_lo alone
    carries the lo part of the centre and is seen."""
    x, mus, ref, kp = _ensemble(8, 1, n=2048)
    full = gmm_grad_tensor_model(x, mus, 1.0, k_pad=kp)
    for t in GEMM1 + ("b1", "b2", "el.muh"):
        assert torch.equal(gmm_grad_tensor_model(x, mus, 1.0, k_pad=kp, drop=(t,)), full), t
    assert relmax(gmm_grad_tensor_model(x, mus, 1.0, k_pad=kp, drop=("eh.mul",)), ref) > 2 * TOL_T
