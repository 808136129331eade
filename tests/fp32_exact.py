"""Exactly rounded fp32 arithmetic on the host (test infrastructure): fma32 restates the fused multiply-add of the
CUDA kernels (fmaf, __ffma2_rn) on float32 tensors of any device, so that a test can replay a kernel's update bit
for bit.  Subnormal results are rounded exactly as well (the kernels are built without -ftz)."""
import torch


def fma32(a: torch.Tensor, b: torch.Tensor, c: torch.Tensor) -> torch.Tensor:
    """round-to-nearest-even fp32 of a * b + c, with a single rounding (float32 tensors, broadcast).

    a * b is exact in float64 (two 24-bit significands); TwoSum gives s = fl64(ab + c) and its exact error e; s rounded
    to fp32 is the answer, except where s lies exactly on an fp32 midpoint and e != 0: then the exact value lies on
    e's side of the midpoint and rounds that way."""
    a, b, c = (t.to(torch.float32) for t in (a, b, c))
    p = a.double() * b.double()
    cd = c.double()
    s = p + cd
    bb = s - p
    e = (p - (s - bb)) + (cd - bb)
    r = s.float()
    toward = torch.nextafter(r, torch.where(s > r.double(), torch.full_like(r, float("inf")),
                                            torch.full_like(r, float("-inf"))))
    mid = (s != r.double()) & ((r.double() + toward.double()) * 0.5 == s) & torch.isfinite(s)
    # on a midpoint: the exact value lies above s if e > 0; take the larger of the two neighbours, else the smaller
    hi, lo = torch.maximum(r, toward), torch.minimum(r, toward)
    fixed = torch.where(e > 0, hi, lo)
    return torch.where(mid & (e != 0), fixed, r)
