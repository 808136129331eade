"""fma32 (tests/fp32_exact.py) against exact rational arithmetic: a * b + c formed as a Fraction and rounded to the
nearest fp32, ties to even."""
import math
from fractions import Fraction

import numpy as np
import torch

from fp32_exact import fma32


def _round_fp32(v: Fraction) -> float:
    """v rounded to the nearest fp32 (ties to even), returned as a Python float (exact)"""
    if v == 0:
        return 0.0
    sign, v = (-1.0 if v < 0 else 1.0), abs(v)
    e = v.numerator.bit_length() - v.denominator.bit_length()  # 2^e <= v < 2^(e + 2)
    if Fraction(2) ** e > v:
        e -= 1
    q = Fraction(2) ** (max(e, -126) - 23)  # the fp32 quantum of v's binade (subnormals: 2^-149)
    m = v / q
    k = math.floor(m)
    if m - k > Fraction(1, 2) or (m - k == Fraction(1, 2) and k % 2 == 1):
        k += 1
    r = k * q
    return sign * (math.inf if r > Fraction(float(np.finfo(np.float32).max)) else float(r))


def _check(a, b, c):
    a, b, c = (torch.tensor(v, dtype=torch.float32) for v in (a, b, c))
    got = fma32(a, b, c)
    want = [_round_fp32(Fraction(float(x)) * Fraction(float(y)) + Fraction(float(z)))
            for x, y, z in zip(a.tolist(), b.tolist(), c.tolist())]
    bad = [(i, a[i].item(), b[i].item(), c[i].item(), got[i].item(), w)
           for i, w in enumerate(want) if got[i].item() != w]
    assert not bad, bad[:5]
    return got


def test_fma32_random_matches_exact_rounding():
    """random significands over a spread of exponents, products and addends of both signs"""
    g = torch.Generator().manual_seed(0)
    n = 20000
    a = torch.randn(n, generator=g) * torch.exp2(torch.randint(-30, 30, (n,), generator=g).float())
    b = torch.randn(n, generator=g) * torch.exp2(torch.randint(-30, 30, (n,), generator=g).float())
    c = torch.randn(n, generator=g) * torch.exp2(torch.randint(-60, 60, (n,), generator=g).float())
    _check(a.tolist(), b.tolist(), c.tolist())
    # the update of the integrators: |c| ~ 1, a b ~ 2^-7 .. 2^-3
    _check((torch.rand(n, generator=g) * 0.1).tolist(), torch.randn(n, generator=g).tolist(),
           (torch.randn(n, generator=g) * 3).tolist())


def test_fma32_midpoints_and_exponent_gaps():
    """s = fl64(ab + c) exactly on an fp32 midpoint with a non-zero error e, where rounding s alone (ties to even)
    goes the wrong way; cancellation; addends far below and far above the product; subnormal results."""
    u = 2.0 ** -23
    cases = [
        # 1 + 2^-24 + 2^-70: the midpoint of 1 and 1 + 2^-23 plus a bit -> up (s alone would tie to 1)
        (-(1 + u) * 2.0 ** -12, (1 - u) * 2.0 ** -12, 1 + u),
        # 1 + 2^-23 + 2^-24 - 2^-70: the midpoint of 1 + 2^-23 and 1 + 2^-22 minus a bit -> down (s alone: up, even)
        ((1 + u) * 2.0 ** -12, (1 - u) * 2.0 ** -12, 1 + u),
        # the same two on the negative side
        ((1 + u) * 2.0 ** -12, (1 - u) * 2.0 ** -12, -(1 + u)),
        ((1 + u) * 2.0 ** -12, -(1 - u) * 2.0 ** -12, -(1 + u)),
        # exact midpoints (e = 0): ties to even
        (2.0 ** -12, 2.0 ** -12, 1.0), (2.0 ** -12, 2.0 ** -12, 1 + u), (-(2.0 ** -12), 2.0 ** -12, -(1 + u)),
        # cancellation to zero and to a tiny remainder
        (1 + u, 1 - u, -1.0), (3.0, 1.0 / 3.0, -1.0), (1 + u, 1 + u, -(1 + 2 * u)),
        # addend 2^-100 of the product and product 2^-100 of the addend
        (1.5, 1.25, 2.0 ** -100), (1.5, 1.25, -(2.0 ** -100)), (2.0 ** -60, 2.0 ** -41, 1.0),
        (2.0 ** -60, -(2.0 ** -41), 1.0), ((1 + u) * 2.0 ** -60, 2.0 ** -41, 1.0),
        # subnormal results
        (2.0 ** -75, 2.0 ** -75, 0.0), (1.5 * 2.0 ** -75, 1.5 * 2.0 ** -74, 2.0 ** -149), (2.0 ** -70, 2.0 ** -60, -1e-38),
    ]
    a, b, c = zip(*cases)
    got = _check(list(a), list(b), list(c))
    # the constructed cases do hit the midpoints: rounding fl64(ab + c) alone gets the first four wrong
    naive = (torch.tensor(a).double() * torch.tensor(b).double() + torch.tensor(c).double()).float()
    assert (naive[:4] != got[:4]).all()
