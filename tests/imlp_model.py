"""CPU twin of the tcgen05 MLP-drift arithmetic of csrc/integrator_mlp_tc.cu (K1-MT, test infrastructure).

Restates what the kernel feeds the tensor cores for grad V_theta(x) of the MLP 32 x 2: both operands of each of the six
GEMMs split into bf16 hi + lo exactly as split2 / stage_weight do, the chosen products summed exactly (float64) and
rounded to fp32 (the tensor cores accumulate exact bf16 products in fp32), tanh, biases and the elementwise adjoint
factors in fp32.  The output layer is padded to 48 columns with zero weights and biases, as in the kernel.

    F0  z0 = x W0,   t0 = tanh(z0 + b0)        B2  za1 = (za W2^T) (1 - t1^2)
    F1  z1 = t0 W1,  t1 = tanh(z1 + b1)        B1  za0 = (za1 W1^T) (1 - t0^2)
    F2  u = t1 W2,   za = 2 (u + b2)           B0  grad V = za0 W0^T

Each GEMM's term set is selectable (`terms={"B1": ("hh", "hl")}` drops a_lo w_hi from B1 only), so a test can show
that the drift tolerance would catch a kernel that loses any one split term.
"""
import torch

TOL_MT = 2e-4  # K1-MT emitted drift against float64, per-tensor max-norm (tests/test_imlp_model.py shows its power)
GEMMS = ("F0", "F1", "F2", "B2", "B1", "B0")
ALL_TERMS = ("hh", "lh", "hl")
H, NO, OUT = 32, 48, 40


def split(v: torch.Tensor):
    hi = v.float().to(torch.bfloat16).float()
    return hi, (v.float() - hi).to(torch.bfloat16).float()


def mm(a: torch.Tensor, w: torch.Tensor, terms=ALL_TERMS) -> torch.Tensor:
    """a [N, K] @ w [K, M] from the selected bf16 products (a_hi w_hi, a_lo w_hi, a_hi w_lo), fp32 result"""
    (ah, al), (wh, wl) = split(a), split(w)
    ops = {"hh": (ah, wh), "lh": (al, wh), "hl": (ah, wl)}
    return sum(ops[t][0].double() @ ops[t][1].double() for t in terms).float()


def unflatten(flat: torch.Tensor, d: int):
    """padded flat MLP 32 x 2 buffer (kernel [d][32], bias, [32][32], bias, [32][40], bias) -> float32 W, b lists"""
    shapes = [((d, H), (H,)), ((H, H), (H,)), ((H, OUT), (OUT,))]
    W, b, off = [], [], 0
    for (ws, bs) in shapes:
        W.append(flat[off:off + ws[0] * ws[1]].float().reshape(ws))
        off += ws[0] * ws[1]
        b.append(flat[off:off + bs[0]].float())
        off += bs[0]
    assert off == flat.numel()
    return W, b


def padded_flat(params, d: int) -> torch.Tensor:
    """reference-shaped MLP tree (hidden <= 32, 2 layers) -> the zero-padded flat float32 buffer the kernels read"""
    out = []
    dims = [(d, H), (H, H), (H, OUT)]
    for i, (n_in, n_out) in enumerate(dims):
        leaf = params["params"][f"layers_{i}"]
        w = torch.zeros(n_in, n_out, dtype=torch.float64)
        w[: leaf["kernel"].shape[0], : leaf["kernel"].shape[1]] = leaf["kernel"]
        bb = torch.zeros(n_out, dtype=torch.float64)
        bb[: leaf["bias"].shape[0]] = leaf["bias"]
        out += [w.reshape(-1), bb]
    return torch.cat(out).float()


def mlp_drift_tensor_model(x: torch.Tensor, flat: torch.Tensor, terms=None) -> torch.Tensor:
    """x [N, d], flat padded parameters -> grad V_theta(x) [N, d] float32 by the K1-MT formulation.
    terms: {gemm name: tuple of "hh" / "lh" / "hl"}; GEMMs not named keep all three."""
    terms = terms or {}
    tm = lambda name: terms.get(name, ALL_TERMS)  # noqa: E731
    W, b = unflatten(flat.cpu(), x.shape[1])
    W2 = torch.cat([W[2], torch.zeros(H, NO - OUT)], 1)
    b2 = torch.cat([b[2], torch.zeros(NO - OUT)])
    t0 = torch.tanh(mm(x, W[0], tm("F0")) + b[0])
    t1 = torch.tanh(mm(t0, W[1], tm("F1")) + b[1])
    za = 2.0 * (mm(t1, W2, tm("F2")) + b2)
    za1 = mm(za, W2.T, tm("B2")) * (1.0 - t1 * t1)
    za0 = mm(za1, W[1].T, tm("B1")) * (1.0 - t0 * t0)
    return mm(za0, W[0].T, tm("B0"))
