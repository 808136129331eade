"""Precision class of the tcgen05 drifts of K1, below the 1e-2 "bf16 GEMM path" envelope.

* K1-MT (csrc/integrator_mlp_tc.cu): every GEMM splits both operands hi + lo, so grad V_theta is accurate to about
  2^-16, and the emitted drift is held at TOL_MT (tests/imlp_model.py) against float64 at the kernel's own emitted
  positions, which isolates the drift from trajectory divergence.  tests/test_imlp_model.py shows that TOL_MT rejects
  a kernel that lost any one split term of any one GEMM.  The kernel is also compared with its CPU twin.
* Symmetry relations of the emitted drift, each kernel against itself on the same Philox stream: K1-MT under a
  permutation of the hidden units and a sign flip of the outputs; the GMM drift K1-T under a permutation of the
  centres.

Measured on a B200 (1000 W, profiles/r03_tc_precision.txt): K1-MT drift against float64 2.0e-5 .. 6.4e-5 (TOL_MT 2e-4),
against its twin <= 1.1e-5; K1-MT relations: trajectories <= 6.4e-7, drift <= 1.8e-5, the output sign flip bit-exact;
K1-T centre permutations: trajectories <= 5.8e-8, drift <= 3.7e-6."""
import pytest
import torch

from conftest import relmax
from imlp_model import TOL_MT, mlp_drift_tensor_model
from oracle import model as o_model
from param_symmetry import hidden_perm, output_sign

pytestmark = pytest.mark.gpu
# K1-MT against its CPU twin.  Not fp32 order alone: a value that differs in its last fp32 bit splits into a different
# (hi, lo) pair, whose dropped lo x lo term and lo rounding (~2^-17 of each product) differ too.  Measured <= 1.1e-5.
TWIN_TOL = 3e-5


def _mlp(d, hidden, seed, cuda):
    """(spec, padded flat parameters with non-zero biases on the device, float64 oracle tree of the same fp32 values)"""
    from pde_inverse_problem_b200.core.model import V_hypothesis
    net = V_hypothesis(output_dim=1, hidden_dims=[hidden] * 2, dim=d)
    params = net.init(seed, torch.zeros(d, device=cuda))
    g = torch.Generator().manual_seed(seed)
    tree = params["params"]
    for k in tree:
        tree[k]["bias"].copy_(0.1 * torch.randn(tree[k]["bias"].shape, generator=g))
    ref = {"params": {k: {kk: vv.double().cpu() for kk, vv in v.items()} for k, v in tree.items()}}
    return net.spec, params["_flat"], ref


def _z0(n, d, seed):
    """positions N(0, 1.5^2) for half the particles, U[-4, 4] (saturated tanh) for the other half; v ~ N(0, 0.3^2)"""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, d, generator=g) * 1.5
    x[n // 2:] = torch.rand(n - n // 2, d, generator=g) * 8 - 4
    return torch.cat([x, torch.randn(n, d, generator=g) * 0.3], 1)


def _run_mt(cuda, spec, flat, z0, S, **kw):
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    zl, tr, _ = ops.kl_integrate_model(z0.to(cuda), S, 0.01, 0.5, spec, flat, seed=kw.pop("seed", 23),
                                       particle_offset=kw.pop("particle_offset", 501), traj_layout=L.TRAJ_TIME_SOA,
                                       emit_drift=True, path=L.PATH_TENSOR, **kw)
    torch.cuda.synchronize()
    assert ops.tensor_path_status() == 0, "a tcgen05 phase timed out"
    return zl.cpu(), tr.cpu()  # tr [3 d][S][n]


@pytest.mark.parametrize("hidden", [32, 20])
@pytest.mark.parametrize("d", [8, 16, 32])
def test_tensor_mlp_emitted_drift_within_split_operand_tolerance(cuda, d, hidden):
    """Ragged n = 1000, S = 20, Philox noise: every emitted grad V_theta against float64 autodiff at the emitted position
    (TOL_MT), and against the CPU twin of the kernel's arithmetic at the same positions (TWIN_TOL)."""
    n, S = 1000, 20
    spec, flat, ref = _mlp(d, hidden, seed=60 + d + hidden, cuda=cuda)
    _, tr = _run_mt(cuda, spec, flat, _z0(n, d, seed=d), S)
    x = tr[:d].permute(1, 2, 0).reshape(-1, d)
    got = tr[2 * d:].permute(1, 2, 0).reshape(-1, d)
    assert torch.isfinite(got).all()
    ref64 = torch.func.grad(lambda y: o_model.mlp_apply(ref, y).sum())(x.double())
    twin = mlp_drift_tensor_model(x, flat)
    e_ref, e_twin = relmax(got, ref64), relmax(got, twin)
    print(f"K1-MT drift d={d} hidden={hidden}: vs float64 {e_ref:.2e} (twin vs float64 {relmax(twin, ref64):.2e}), "
          f"vs twin {e_twin:.2e}")
    assert e_ref < TOL_MT, e_ref
    assert e_twin < TWIN_TOL, e_twin


@pytest.mark.parametrize("d", [8, 16, 32])
def test_tensor_mlp_drift_symmetries(cuda, d):
    """Hidden units of either layer reversed (j -> 31 - j) and randomly permuted, and a random sign flip of the 40
    outputs: the same trajectory and emitted drift on the same Philox stream, up to fp32 summation order and the
    split-representation difference it causes (TWIN_TOL above).  Measured: trajectories <= 6e-7, drift <= 1.8e-5."""
    n, S = 640, 20
    spec, flat, _ = _mlp(d, 32, seed=80 + d, cuda=cuda)
    z0 = _z0(n, d, seed=3 * d)
    zl0, tr0 = _run_mt(cuda, spec, flat, z0, S)
    g = torch.Generator().manual_seed(d)
    rel = [hidden_perm(d, 0, torch.arange(31, -1, -1), "hidden0 reversed"),
           hidden_perm(d, 1, torch.randperm(32, generator=g), "hidden1 random perm"),
           output_sign(d, torch.where(torch.rand(40, generator=g) < 0.5, -1.0, 1.0), "outputs random signs")]
    for t in rel:
        zl, tr = _run_mt(cuda, spec, t.params(flat), z0, S)
        e = (relmax(tr[:2 * d], tr0[:2 * d]), relmax(tr[2 * d:], tr0[2 * d:]), relmax(zl, zl0))
        print(f"K1-MT symmetry d={d} {t.name}: traj {e[0]:.1e} drift {e[1]:.1e} last {e[2]:.1e}, "
              f"bit-exact {torch.equal(tr, tr0)}")
        assert max(e[0], e[2]) < 1e-5 and e[1] < 5e-5, (t.name, e)


@pytest.mark.parametrize("d,K", [(8, 7), (16, 40), (32, 64), (32, 7)])
def test_tensor_gmm_drift_centre_permutation(cuda, d, K):
    """K1-T (kl_integrate, PDEIP_PATH_TENSOR): permuting the rows of mus (reversed, and a random permutation) leaves the
    trajectory and the emitted drift unchanged up to fp32 summation order.  K = 7 (padding centres), 40 and 64 (several
    16-centre chunks): the permutation moves centres across chunks and into the padded chunk."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    n, S = 1000, 12
    g = torch.Generator().manual_seed(d + K)
    z0 = (torch.randn(n, 2 * d, generator=g) * torch.cat([torch.full((d,), 2.0), torch.full((d,), 0.3)])).to(cuda)
    mus = (torch.rand(K, d, generator=g) * 8 - 4).to(cuda)

    def run(m):
        zl, tr, _ = ops.kl_integrate(z0, S, 0.01, 0.5, L.DRIFT_GMM, m.contiguous(), n_gaussian=K, seed=41,
                                     particle_offset=77, traj_layout=L.TRAJ_TIME_SOA, emit_drift=True,
                                     path=L.PATH_TENSOR)
        torch.cuda.synchronize()
        assert ops.tensor_path_status() == 0
        return zl.cpu(), tr.cpu()

    zl0, tr0 = run(mus)
    for name, perm in (("reversed", torch.arange(K - 1, -1, -1)), ("random", torch.randperm(K, generator=g))):
        zl, tr = run(mus[perm.to(cuda)])
        e = (relmax(tr[:2 * d], tr0[:2 * d]), relmax(tr[2 * d:], tr0[2 * d:]), relmax(zl, zl0))
        print(f"K1-T centre permutation d={d} K={K} {name}: traj {e[0]:.1e} drift {e[1]:.1e} last {e[2]:.1e}, "
              f"bit-exact {torch.equal(tr, tr0)}")
        assert max(e) < 1e-5, (name, e)
