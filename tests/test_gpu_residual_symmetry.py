"""Symmetry relations of the MLP residual kernels (csrc/residual_tensor.cu and the fp32 path), each kernel compared with
itself: the loss and gradient of V = |MLP(x)|^2 are exactly equivariant under the signed permutations of
tests/param_symmetry.py (hidden units of either layer, outputs, input coordinates) and invariant under any permutation
of the points.  Every transform maps bf16-rounded values onto bf16-rounded values, so the tensor path satisfies each
relation up to fp32 summation order (and the rare bf16 rounding flip that order causes), far below its 1e-2 accuracy
class, while a defect tied to a position (a TMEM lane, an epilogue part, a hidden or output unit, a tile, a CTA, the
ragged tail) moves with the transform and shows at full size.

Point relations, on the same parameters: rows reversed inside every 128-point tile; tiles rotated by one (every tile
lands in another CTA and another turn of the persistent loop); a seeded global permutation (the ragged tail's points
move into the interior).  Coverage: both paths; KFP 0T in AoS with a GMM true gradient, KFP 0T in BLOCK128 with the
true gradient stored in the points, the KFP boundary set and the FP 0T set; d = 5, 8 (two-slot kernel), 12, 16 and
17, 32 (the one-slot kernels); n = (SM count) x 128 x 3 + r, so that every CTA runs several tiles.

Metric: each SUM_* entry relative to its own magnitude, the gradient per leaf (W0, b0, W1, b1, W2, b2), each leaf
normalised by its own max.  In the KFP sets v is drawn partly along grad V(x), so that D_v V is not a cancelling
mean.  Asserted at 1e-4 on the tensor path and 1e-5 on the fp32 path.  Measured on a B200 (1000 W), largest over all
cases and relations: tensor path sums 1.8e-5, gradient leaves 5.2e-5; fp32 path sums 8.3e-7, gradient leaves 8.9e-7
(profiles/r03_tc_precision.txt).  The hidden-unit sign flips go through tanh.approx, whose oddness is not documented;
the test prints whether that relation is bit-exact and does not require it (measured: bit-exact on both paths).

The same file holds the per-leaf tensor-versus-fp32 check of the one-slot kernels over several tiles per CTA (the
only case in which the TMEM-resident bias-gradient sums accumulate), at the rule of tests/test_gpu_tensor.py: weight
leaves 1e-2, bias leaves 1.5e-2."""
import pytest
import torch

from param_symmetry import transforms

pytestmark = pytest.mark.gpu
TOL = {"tensor": 1e-4, "fp32": 1e-5}
LEAVES = ("W0", "b0", "W1", "b1", "W2", "b2")
MODES = ["kfp0t_aos_gmm", "kfp0t_block_stored", "kfp_boundary", "fp0t"]


def _ops():
    from pde_inverse_problem_b200 import ops, _lib
    return ops, _lib


def _flat(d, seed):
    from oracle import model as o_model
    p = o_model.init_mlp_params(d, 32, 2, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    for k in p["params"]:  # non-zero biases: zero biases hide every bias-indexing defect
        p["params"][k]["bias"] = 0.1 * torch.randn(p["params"][k]["bias"].shape, generator=g, dtype=torch.float64)
    return o_model.flatten_params(p).float()


def _leaves(grad, d):
    sizes = (d * 32, 32, 32 * 32, 32, 32 * 40, 40)
    return torch.split(grad, sizes)


def _leaf_errs(a, b, d):
    return [((x - y).abs().max() / max(y.abs().max(), 1e-30)).item() for x, y in zip(_leaves(a, d), _leaves(b, d))]


def _sum_err(a, b):
    den = torch.where(b.abs() > 0, b.abs(), torch.ones_like(b))
    return ((a - b).abs() / den).max().item()


class Problem:
    """One residual accumulation: mode, d, rows (AoS [n, blocks * d] on the device), GMM centres."""

    def __init__(self, mode, d, flat, cuda):
        ops, L = _ops()
        self.ops, self.L, self.mode, self.d, self.cuda = ops, L, mode, d, cuda
        sm = torch.cuda.get_device_properties(0).multi_processor_count
        block = mode == "kfp0t_block_stored"
        self.n = sm * 128 * 3 + (128 * 5 if block else 77 + 8 * d)  # BLOCK128 needs whole tiles; else ragged
        g = torch.Generator().manual_seed(1000 + 10 * d + MODES.index(mode))
        nb = {"kfp0t_aos_gmm": 2, "kfp0t_block_stored": 3, "kfp_boundary": 2, "fp0t": 1}[mode]
        scale = torch.cat([torch.full((d,), 1.5), torch.full((d,), 0.7), torch.ones(d)])[: nb * d]
        self.rows = (torch.randn(self.n, nb * d, generator=g) * scale).to(cuda)
        self.mus = (torch.rand(8, d, generator=g) * 6 - 3).to(cuda)
        if nb > 1:
            # v partly along grad V(x): otherwise D_v V (the boundary set, and a term of the 0T loss) is a cancelling
            # mean of size |summand| / sqrt(n), and its own-magnitude relative error measures the cancellation
            gx = ops.model_eval(ops.ModelSpec(L.MODEL_MLP, d, 32, 2), flat, self.rows[:, :d].contiguous(),
                                want=("grad",))["grad"]
            self.rows[:, d:2 * d] = 0.6 * self.rows[:, d:2 * d] + 0.56 * gx / gx.pow(2).mean().sqrt()

    def run(self, flat, path, rows=None, mus=None):
        ops, L, d, n = self.ops, self.L, self.d, self.n
        rows = self.rows if rows is None else rows
        mus = self.mus if mus is None else mus
        acc = ops.ResidualAccumulator(ops.ModelSpec(L.MODEL_MLP, d, 32, 2), device=self.cuda).begin()
        if self.mode == "kfp0t_aos_gmm":
            acc.accumulate(L.SET_KFP_0T, flat, rows, 1.0 / n, coef=0.5, true_grad=ops.TrueGrad(L.DRIFT_GMM, mus, 1.0),
                           path=path)
        elif self.mode == "kfp0t_block_stored":
            blk = rows.reshape(n // 128, 128, 3 * d).transpose(1, 2).contiguous()
            acc.accumulate(L.SET_KFP_0T, flat, blk, 1.0 / n, coef=0.5, true_grad=ops.TrueGrad(L.DRIFT_IN_POINTS),
                           layout=L.LAYOUT_BLOCK128, path=path)
        elif self.mode == "kfp_boundary":
            acc.accumulate(L.SET_KFP_BOUNDARY, flat, rows, 1.0 / n, coef=1.0, path=path)
        else:
            acc.accumulate(L.SET_FP_0T, flat, rows, 1.0 / n, true_grad=ops.TrueGrad(L.DRIFT_GMM, mus, 1.0), path=path)
        s, gr = acc.finalize()
        s, gr = s.cpu().double(), gr.cpu().double()
        assert ops.tensor_path_status() == 0, "a tcgen05 phase timed out"
        return s, gr

    def point_perms(self):
        n = self.n
        idx = torch.arange(n)
        rev = idx.clone()
        for t0 in range(0, n, 128):  # reverse inside every tile (the ragged tail inside itself)
            rev[t0:min(t0 + 128, n)] = idx[t0:min(t0 + 128, n)].flip(0)
        g = torch.Generator().manual_seed(self.d)
        return {"rows reversed in tiles": rev, "tiles rotated by one": torch.roll(idx, -128),
                "random point perm": torch.randperm(n, generator=g)}


@pytest.mark.parametrize("d", [5, 8, 12, 16, 17, 32])
@pytest.mark.parametrize("mode", MODES)
def test_residual_symmetry_relations(cuda, mode, d):
    _, L = _ops()
    flat = _flat(d, seed=7 + d).to(cuda)
    prob = Problem(mode, d, flat, cuda)
    base, failed = {}, []
    for path_name, path in (("fp32", L.PATH_FP32), ("tensor", L.PATH_TENSOR)):
        s0, g0 = prob.run(flat, path)
        base[path_name] = (s0, g0)
        worst_s, worst_g, exact_sign = (0.0, ""), (0.0, ""), []
        cases = [(t.name, t.params(flat), t.points(prob.rows, d), t.mus(prob.mus), t.grad) for t in transforms(d, seed=d)]
        cases += [(name, flat, prob.rows[p.to(cuda)].contiguous(), prob.mus, lambda x: x)
                  for name, p in prob.point_perms().items()]
        for name, flat_t, rows_t, mus_t, gmap in cases:
            s, gr = prob.run(flat_t, path, rows_t, mus_t)
            expect = gmap(g0)
            es, eg = _sum_err(s, s0), max(_leaf_errs(gr, expect, d))
            worst_s, worst_g = max(worst_s, (es, name)), max(worst_g, (eg, name))
            if "signs" in name and name.startswith("hidden"):
                exact_sign.append(torch.equal(gr, expect) and torch.equal(s, s0))
            if es >= TOL[path_name]:
                failed.append((path_name, name, "sums", es, s.tolist(), s0.tolist()))
            if eg >= TOL[path_name]:
                failed.append((path_name, name, "grad leaves", dict(zip(LEAVES, _leaf_errs(gr, expect, d)))))
        print(f"symmetry {mode} d={d} {path_name}: sums {worst_s[0]:.1e} ({worst_s[1]}), grad leaves "
              f"{worst_g[0]:.1e} ({worst_g[1]}), hidden sign flips bit-exact: {all(exact_sign)}")
    assert not failed, failed
    if d > 8:  # one-slot kernels: per-leaf tensor vs fp32 over several tiles per CTA
        errs = dict(zip(LEAVES, _leaf_errs(base["tensor"][1], base["fp32"][1], d)))
        print(f"tensor vs fp32 {mode} d={d} per leaf: " + " ".join(f"{k} {v:.1e}" for k, v in errs.items()))
        for name, e in errs.items():
            assert e < (1.5e-2 if name.startswith("b") else 1e-2), (mode, d, name, e)
