"""Exact symmetries of V = |MLP(x)|^2 (MLP 32 x 2, 40 outputs) on the flat Flax-order parameter buffer (test
infrastructure).

The buffer is layers_0 kernel [d][32], bias [32], layers_1 [32][32], bias, layers_2 [32][40], bias [40]
(oracle/model.py:flatten_params).  Each transform is a signed permutation M of the parameters under which the loss of
every residual is invariant: a permutation of the hidden units of either layer, a sign flip of hidden units (tanh is
odd), a permutation or sign flip of the 40 outputs (V sums their squares), or a permutation tau of the input
coordinates, which must be applied to the points (x, v, a stored true gradient) and to the true drift's parameters
(GMM centres mus[:, tau], linear F[tau][:, tau]) as well.  Since M is orthogonal, the gradient at M theta is M applied
to the gradient at theta: `grad` is the same map as `params`.

Transforms map bf16-rounded values onto bf16-rounded values, so a tensor-core kernel satisfies each relation up to
its fp32 summation order; a defect tied to one position (unit, part, lane, tile, CTA) moves with the transform.
"""
from dataclasses import dataclass
from typing import Callable, Optional

import torch

H, OUT = 32, 40


def _views(flat: torch.Tensor, d: int):
    """(W0 [d][32], b0, W1 [32][32], b1, W2 [32][40], b2) views of a flat buffer (torch, any device / dtype)"""
    shapes = [(d, H), (H,), (H, H), (H,), (H, OUT), (OUT,)]
    out, off = [], 0
    for s in shapes:
        n = s[0] * (s[1] if len(s) > 1 else 1)
        out.append(flat[off:off + n].view(s))
        off += n
    assert off == flat.numel(), (off, flat.numel())
    return out


@dataclass
class Transform:
    name: str
    params: Callable[[torch.Tensor], torch.Tensor]  # flat -> flat (a new tensor)
    tau: Optional[torch.Tensor] = None               # input permutation: column i of the new points = column tau[i]

    @property
    def grad(self):
        return self.params  # orthogonal: the gradient transforms as the parameters do

    def points(self, pts: torch.Tensor, d: int) -> torch.Tensor:
        """AoS rows [x | v | stored grad ...] (each block d wide) -> rows of the transformed problem"""
        if self.tau is None:
            return pts
        nb = pts.shape[1] // d
        idx = torch.cat([self.tau.to(pts.device) + k * d for k in range(nb)])
        return pts[:, idx].contiguous()

    def mus(self, mus: torch.Tensor) -> torch.Tensor:
        return mus if self.tau is None else mus[:, self.tau.to(mus.device)].contiguous()

    def linear(self, F: torch.Tensor) -> torch.Tensor:
        if self.tau is None:
            return F
        t = self.tau.to(F.device)
        return F[t][:, t].contiguous()


def _map(d, fn):
    def apply(flat):
        out = flat.clone()
        fn(_views(flat, d), _views(out, d))
        return out
    return apply


def hidden_perm(d: int, layer: int, perm: torch.Tensor, name: str) -> Transform:
    """units of hidden layer `layer` (0 or 1) reordered: W_l[:, perm], b_l[perm], W_{l+1}[perm, :]"""
    def fn(src, dst):
        p = perm.to(src[0].device)
        dst[2 * layer][:] = src[2 * layer][:, p]
        dst[2 * layer + 1][:] = src[2 * layer + 1][p]
        dst[2 * layer + 2][:] = src[2 * layer + 2][p, :]
    return Transform(name, _map(d, fn))


def hidden_sign(d: int, layer: int, signs: torch.Tensor, name: str) -> Transform:
    """units of hidden layer `layer` negated where signs == -1: W_l[:, j], b_l[j], W_{l+1}[j, :] (tanh is odd)"""
    def fn(src, dst):
        s = signs.to(src[0].device, src[0].dtype)
        dst[2 * layer][:] = src[2 * layer] * s[None, :]
        dst[2 * layer + 1][:] = src[2 * layer + 1] * s
        dst[2 * layer + 2][:] = src[2 * layer + 2] * s[:, None]
    return Transform(name, _map(d, fn))


def output_perm(d: int, perm: torch.Tensor, name: str) -> Transform:
    def fn(src, dst):
        p = perm.to(src[0].device)
        dst[4][:] = src[4][:, p]
        dst[5][:] = src[5][p]
    return Transform(name, _map(d, fn))


def output_sign(d: int, signs: torch.Tensor, name: str) -> Transform:
    def fn(src, dst):
        s = signs.to(src[0].device, src[0].dtype)
        dst[4][:] = src[4] * s[None, :]
        dst[5][:] = src[5] * s
    return Transform(name, _map(d, fn))


def input_perm(d: int, tau: torch.Tensor, name: str) -> Transform:
    def fn(src, dst):
        dst[0][:] = src[0][tau.to(src[0].device), :]
    return Transform(name, _map(d, fn), tau=tau)


def transforms(d: int, seed: int = 0):
    """The relations the tests check.  The reversals move every unit across every ownership boundary: j -> 31 - j sends
    each hidden unit to another part of both the 4-part (one-slot) and the 2-part (two-slot) residual kernels,
    j -> 39 - j swaps the output units 32..39 (the per-part "pair" units of the one-slot kernels) with chunk units,
    and i -> d - 1 - i moves the lone input component of a part-padded last chunk (d = 17) to chunk 0.  One seeded
    random permutation / sign pattern of each kind is added."""
    g = torch.Generator().manual_seed(seed)
    rev_h, rev_o, rev_i = torch.arange(H - 1, -1, -1), torch.arange(OUT - 1, -1, -1), torch.arange(d - 1, -1, -1)
    sign = lambda n: torch.where(torch.rand(n, generator=g) < 0.5, -1.0, 1.0)  # noqa: E731
    out = []
    for layer in (0, 1):
        out.append(hidden_perm(d, layer, rev_h, f"hidden{layer} reversed"))
        out.append(hidden_perm(d, layer, torch.randperm(H, generator=g), f"hidden{layer} random perm"))
        out.append(hidden_sign(d, layer, sign(H), f"hidden{layer} random signs"))
    out.append(output_perm(d, rev_o, "outputs reversed"))
    out.append(output_perm(d, torch.randperm(OUT, generator=g), "outputs random perm"))
    out.append(output_sign(d, sign(OUT), "outputs random signs"))
    out.append(input_perm(d, rev_i, "inputs reversed"))
    out.append(input_perm(d, torch.randperm(d, generator=g), "inputs random perm"))
    return out


def tree_of(flat: torch.Tensor, d: int):
    """flat buffer -> oracle parameter tree {"params": {"layers_i": {"kernel", "bias"}}}"""
    v = _views(flat, d)
    return {"params": {f"layers_{i}": {"kernel": v[2 * i], "bias": v[2 * i + 1]} for i in range(3)}}
