"""CPU twin of the tcgen05 GMM-drift arithmetic of csrc/integrator_tc.cu (K1-T and K1-T-OD, test infrastructure).

Restates, with torch bfloat16 casts and float32 accumulation, exactly what the kernel feeds the tensor cores:
centres scaled to log2 units and split hi + lo, the bias -|mu~|^2 / (2 c) as three bf16 terms through a ones column,
x split hi + lo, GEMM 1 = x_hi mu_hi^T + x_lo mu_hi^T + x_hi mu_lo^T + bias (the lo x lo term is dropped), softmax
weights e = 2^(L - max L) split hi + lo, GEMM 2 = e_hi mu_hi + e_lo mu_hi + e_hi mu_lo, and
grad U = (x - A / (c sum e)) / sigma^2   (core/potential.py:32-37 in closed form).

Each product term and each bias term can be dropped (`drop=("el.muh",)` loses e_lo mu_hi of GEMM 2), so that a test
can show which defects the drift tolerance TOL_T would catch (tests/test_itc_model.py).
"""
import torch

TOL_T = 2e-4  # K1-T / K1-T-OD emitted drift against float64, per-tensor max-norm (tests/test_itc_model.py shows its power)
GEMM1 = ("xh.muh", "xl.muh", "xh.mul")
BIAS = ("b0", "b1", "b2")
GEMM2 = ("eh.muh", "el.muh", "eh.mul")
TERMS = GEMM1 + BIAS + GEMM2


def _split(v: torch.Tensor, terms: int = 2):
    out, r = [], v.float()
    for _ in range(terms):
        h = r.to(torch.bfloat16).float()
        out.append(h)
        r = r - h
    return out


def gmm_grad_tensor_model(x: torch.Tensor, mus: torch.Tensor, sigma: float = 1.0, k_pad: int = 0,
                          drop=()) -> torch.Tensor:
    """x [N, d], mus [K, d] (any float dtype) -> grad U [N, d] float32, by the kernel's split-operand formulation.
    drop: names from TERMS left out of the GEMMs."""
    assert set(drop) <= set(TERMS), drop
    # 1 / sigma^2 and c = log2(e) / sigma^2 formed in fp32, as the launcher and the kernel form them
    inv_s2 = 1.0 / (torch.tensor(sigma, dtype=torch.float32) ** 2)
    cs = inv_s2 * torch.tensor(1.4426950408889634, dtype=torch.float32)
    mu_hi, mu_lo = _split(cs * mus.float())
    mu_rec = mu_hi + mu_lo
    b = -0.5 * (mu_rec * mu_rec).sum(-1) / cs
    if k_pad > mus.shape[0]:  # padding centres: zero rows, bias -1e30 (weight exactly 0)
        z = torch.zeros(k_pad - mus.shape[0], mus.shape[1])
        mu_hi, mu_lo = torch.cat([mu_hi, z]), torch.cat([mu_lo, z])
        b = torch.cat([b, torch.full((k_pad - mus.shape[0],), -1.0e30)])
    bias = dict(zip(BIAS, _split(b, 3)))
    x_hi, x_lo = _split(x)
    g1 = {"xh.muh": (x_hi, mu_hi), "xl.muh": (x_lo, mu_hi), "xh.mul": (x_hi, mu_lo)}
    logits = sum(a @ m.T for t, (a, m) in g1.items() if t not in drop)
    logits = logits + sum(v for t, v in bias.items() if t not in drop)
    m = logits.max(-1, keepdim=True).values
    e = torch.exp2(logits - m)
    se = e.sum(-1, keepdim=True)
    e_hi, e_lo = _split(e)
    g2 = {"eh.muh": (e_hi, mu_hi), "el.muh": (e_lo, mu_hi), "eh.mul": (e_hi, mu_lo)}
    acc = sum(a @ m for t, (a, m) in g2.items() if t not in drop)
    return (x.float() - acc / (cs * se)) * inv_s2
