"""Thin tensor-level wrappers over the C ABI (include/pdeip.h), dispatched as torch custom ops.

torch supplies device memory and the current CUDA stream; all arithmetic happens inside
libpdeip.so.  The hot-path entry points are registered as `torch.library.custom_op`s (torch_ops.py) and
called here as `torch.ops.pdeip.*`; the wrappers allocate the outputs (the C ABI never allocates) and
insist on CUDA float32 tensors — there is no CPU or eager fallback (the ops have no CPU kernel).
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Tuple

import torch

from . import _lib as L
from . import torch_ops as _T  # noqa: F401  (registers torch.ops.pdeip.*)
from ._lib import PdeipError  # noqa: F401  (re-export)
from .torch_ops import as_i64

_ops = torch.ops.pdeip

# count of libpdeip kernel launches issued through this module (bench.py reports it)
launch_counter = {"n": 0}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _f32(t: Optional[torch.Tensor], name: str, allow_none: bool = False) -> Optional[torch.Tensor]:
    if t is None:
        if allow_none:
            return None
        raise PdeipError(f"{name} is required")
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise PdeipError(f"{name} must be a CUDA tensor (got {type(t).__name__} on "
                         f"{getattr(t, 'device', 'n/a')}); the pdeip path has no CPU fallback")
    if t.dtype != torch.float32:
        raise PdeipError(f"{name} must be float32 (got {t.dtype})")
    return t if t.is_contiguous() else t.contiguous()


# ------------------------------------------------------------------------------------------------
# K1 integrator
# ------------------------------------------------------------------------------------------------
def _k1_buffers(z0, n_steps, noise, tau0, schedule, state_layout, traj_layout, want_traj, want_tau, emit_every,
                emit_offset, traj_out, z_last_out, emit_drift):
    """Checked inputs and the outputs of one K1 call: (z0, n, d, noise, tau0, z_last, traj|None, tau|None)."""
    z0 = _f32(z0, "z0")
    if state_layout == L.LAYOUT_AOS:
        n, two_d = z0.shape
    else:
        two_d, n = z0.shape
    d = two_d // 2
    noise = _f32(noise, "noise", allow_none=True)
    tau0 = _f32(tau0, "tau0", allow_none=True)
    n_draws = n_steps + 1 if schedule == L.SCHEDULE_REFERENCE else n_steps
    if noise is not None and tuple(noise.shape) != (n, n_draws, d):
        raise PdeipError(f"noise must have shape {(n, n_draws, d)}, got {tuple(noise.shape)}")
    if tau0 is not None and tuple(tau0.shape) != (n,):
        raise PdeipError(f"tau0 must have shape {(n,)}, got {tuple(tau0.shape)}")
    z_last = z_last_out if z_last_out is not None else torch.empty_like(z0)
    s_emit = (n_steps - emit_offset + emit_every - 1) // emit_every
    traj = None
    if want_traj:
        width = two_d + d if emit_drift else two_d
        shape = {L.TRAJ_PARTICLE_MAJOR: (n, s_emit, width), L.TRAJ_TIME_MAJOR: (s_emit, n, width),
                 L.TRAJ_TIME_SOA: (width, s_emit, n), L.TRAJ_BLOCK128: (s_emit, n // 128, width, 128)}[traj_layout]
        if traj_layout == L.TRAJ_BLOCK128 and n % 128:
            raise PdeipError(f"TRAJ_BLOCK128 needs n % 128 == 0, got n={n}")
        if traj_out is not None:
            if traj_out.numel() < n * s_emit * width:
                raise PdeipError("traj_out too small")
            traj = _f32(traj_out, "traj_out").view(-1)[: n * s_emit * width].view(shape)
        else:
            traj = torch.empty(shape, device=z0.device, dtype=torch.float32)
    tau = torch.empty((n, n_steps), device=z0.device, dtype=torch.float32) if want_tau else None
    return z0, n, d, noise, tau0, z_last, traj, tau


def kl_integrate(z0: torch.Tensor, n_steps: int, dt: float, gamma: float, drift_kind: int,
                 drift_params: Optional[torch.Tensor] = None, n_gaussian: int = 0, sigma: float = 1.0,
                 noise: Optional[torch.Tensor] = None, tau0: Optional[torch.Tensor] = None, seed: int = 0,
                 particle_offset: int = 0, step_offset: int = 0, schedule: int = L.SCHEDULE_REFERENCE,
                 state_layout: int = L.LAYOUT_AOS, traj_layout: int = L.TRAJ_PARTICLE_MAJOR,
                 want_traj: bool = True, want_tau: bool = False, emit_every: int = 1, emit_offset: int = 0,
                 traj_out: Optional[torch.Tensor] = None, z_last_out: Optional[torch.Tensor] = None,
                 emit_drift: bool = False, path: int = L.PATH_FP32,
                 ) -> Tuple[torch.Tensor, Optional[torch.Tensor], Optional[torch.Tensor]]:
    """pdeip_kl_integrate.  z0: [N,2d] (AOS) or [2d,N] (SOA).  Returns (z_last, traj|None, tau|None).
    emit_drift: every trajectory sample is [x, v, grad U(x)] (3d components).
    path: PATH_TENSOR runs the GMM drift contraction on tcgen05 where that kernel exists (see pdeip.h)."""
    z0, n, d, noise, tau0, z_last, traj, tau = _k1_buffers(
        z0, n_steps, noise, tau0, schedule, state_layout, traj_layout, want_traj, want_tau, emit_every, emit_offset,
        traj_out, z_last_out, emit_drift)
    drift_params = _f32(drift_params, "drift_params", allow_none=True)
    _ops.kl_integrate(z0, z_last, traj, tau, n, d, n_steps, float(dt), float(gamma), drift_kind, drift_params,
                      n_gaussian, float(sigma), noise, tau0, as_i64(seed), as_i64(particle_offset), step_offset, schedule,
                      state_layout, traj_layout, emit_every, emit_offset, 1 if emit_drift else 0, path)
    launch_counter["n"] += 1
    return z_last, traj, tau


def kl_integrate_model(z0: torch.Tensor, n_steps: int, dt: float, gamma: float, spec: "ModelSpec",
                       params: torch.Tensor, noise: Optional[torch.Tensor] = None, tau0: Optional[torch.Tensor] = None,
                       seed: int = 0, particle_offset: int = 0, step_offset: int = 0,
                       schedule: int = L.SCHEDULE_REFERENCE, state_layout: int = L.LAYOUT_AOS,
                       traj_layout: int = L.TRAJ_PARTICLE_MAJOR, want_traj: bool = True, want_tau: bool = False,
                       emit_every: int = 1, emit_offset: int = 0, traj_out: Optional[torch.Tensor] = None,
                       z_last_out: Optional[torch.Tensor] = None, emit_drift: bool = False, path: int = L.PATH_FP32,
                       ) -> Tuple[torch.Tensor, Optional[torch.Tensor], Optional[torch.Tensor]]:
    """pdeip_kl_integrate_model: kl_integrate with grad U = grad V_theta of the hypothesis model `spec` at the flat
    parameters `params` (the buffer model_eval takes).  Same outputs and keyword arguments as kl_integrate;
    emit_drift carries grad V_theta(x) of every emitted sample."""
    z0, n, d, noise, tau0, z_last, traj, tau = _k1_buffers(
        z0, n_steps, noise, tau0, schedule, state_layout, traj_layout, want_traj, want_tau, emit_every, emit_offset,
        traj_out, z_last_out, emit_drift)
    params = _f32(params, "params")
    if d != spec.d or params.numel() != spec.num_params:
        raise PdeipError(f"shape mismatch: the state has d={d}, params has {params.numel()} entries (expected "
                         f"d={spec.d}, {spec.num_params} params)")
    _ops.kl_integrate_model(z0, z_last, traj, tau, n, d, n_steps, float(dt), float(gamma), spec.kind, params,
                            spec.hidden, spec.layers, spec.n_gaussian, noise, tau0, as_i64(seed),
                            as_i64(particle_offset), step_offset, schedule, state_layout, traj_layout, emit_every,
                            emit_offset, 1 if emit_drift else 0, path)
    launch_counter["n"] += 1
    return z_last, traj, tau


def _od_buffers(x0, n_steps, noise, state_layout, traj_layout, want_traj, emit_every, emit_offset, emit_drift,
                traj_out=None, x_last_out=None):
    """Checked inputs and the outputs of one K1-OD call: (x0, n, d, noise, x_last, traj|None)."""
    x0 = _f32(x0, "x0")
    if state_layout == L.LAYOUT_AOS:
        n, d = x0.shape
    else:
        d, n = x0.shape
    noise = _f32(noise, "noise", allow_none=True)
    if noise is not None and tuple(noise.shape) != (n, n_steps, d):
        raise PdeipError(f"noise must have shape {(n, n_steps, d)}, got {tuple(noise.shape)}")
    s_emit = (n_steps - emit_offset + emit_every - 1) // emit_every
    traj = None
    if want_traj:
        width = 2 * d if emit_drift else d
        shape = {L.TRAJ_PARTICLE_MAJOR: (n, s_emit, width), L.TRAJ_TIME_MAJOR: (s_emit, n, width),
                 L.TRAJ_TIME_SOA: (width, s_emit, n), L.TRAJ_BLOCK128: (s_emit, n // 128, width, 128)}[traj_layout]
        if traj_layout == L.TRAJ_BLOCK128 and n % 128:
            raise PdeipError(f"TRAJ_BLOCK128 needs n % 128 == 0, got n={n}")
        if traj_out is not None:
            if traj_out.numel() < n * s_emit * width:
                raise PdeipError("traj_out too small")
            traj = _f32(traj_out, "traj_out").view(-1)[: n * s_emit * width].view(shape)
        else:
            traj = torch.empty(shape, device=x0.device, dtype=torch.float32)
    if x_last_out is not None:
        if tuple(x_last_out.shape) != tuple(x0.shape) or _f32(x_last_out, "x_last_out") is not x_last_out:
            raise PdeipError(f"x_last_out must be a contiguous {tuple(x0.shape)} tensor")
        return x0, n, d, noise, x_last_out, traj
    return x0, n, d, noise, torch.empty_like(x0), traj


def overdamped_integrate(x0: torch.Tensor, n_steps: int, dt: float, drift_kind: int,
                         drift_params: Optional[torch.Tensor] = None, n_gaussian: int = 0, sigma: float = 1.0,
                         noise: Optional[torch.Tensor] = None, seed: int = 0, particle_offset: int = 0,
                         step_offset: int = 0, state_layout: int = L.LAYOUT_AOS,
                         traj_layout: int = L.TRAJ_PARTICLE_MAJOR, want_traj: bool = True, emit_every: int = 1,
                         emit_offset: int = 0, emit_drift: bool = False, path: int = L.PATH_FP32, *,
                         traj_out: Optional[torch.Tensor] = None, x_last_out: Optional[torch.Tensor] = None,
                         ) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """pdeip_overdamped_integrate: n_steps overdamped Langevin steps x' = x - dt grad U(x) + sqrt(2 dt) xi.
    x0: [N,d] (AOS) or [d,N] (SOA).  noise: injected normals [N, n_steps, d], else Philox.  Returns (x_last,
    traj|None); with emit_drift every trajectory sample is [x, grad U(x)] (2d components).
    path: PATH_TENSOR runs the GMM drift on tcgen05 inside its envelope (see pdeip.h).  traj_out / x_last_out:
    buffers to write into (traj_out: at least the trajectory's size, viewed as its shape; x_last_out: x0's shape)."""
    x0, n, d, noise, x_last, traj = _od_buffers(x0, n_steps, noise, state_layout, traj_layout, want_traj, emit_every,
                                                emit_offset, emit_drift, traj_out, x_last_out)
    drift_params = _f32(drift_params, "drift_params", allow_none=True)
    _ops.overdamped_integrate(x0, x_last, traj, n, d, n_steps, float(dt), drift_kind, drift_params, n_gaussian,
                              float(sigma), noise, as_i64(seed), as_i64(particle_offset), step_offset, state_layout,
                              traj_layout, emit_every, emit_offset, 1 if emit_drift else 0, path)
    launch_counter["n"] += 1
    return x_last, traj


def overdamped_integrate_model(x0: torch.Tensor, n_steps: int, dt: float, spec: "ModelSpec", params: torch.Tensor,
                               noise: Optional[torch.Tensor] = None, seed: int = 0, particle_offset: int = 0,
                               step_offset: int = 0, state_layout: int = L.LAYOUT_AOS,
                               traj_layout: int = L.TRAJ_PARTICLE_MAJOR, want_traj: bool = True, emit_every: int = 1,
                               emit_offset: int = 0, emit_drift: bool = False, path: int = L.PATH_FP32,
                               ) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """pdeip_overdamped_integrate_model: overdamped_integrate with grad U = grad V_theta of the hypothesis model `spec`
    at the flat parameters `params`.  PATH_TENSOR runs the MLP 32 x 2 drift on tcgen05 inside its envelope (pdeip.h)."""
    x0, n, d, noise, x_last, traj = _od_buffers(x0, n_steps, noise, state_layout, traj_layout, want_traj, emit_every,
                                                emit_offset, emit_drift)
    params = _f32(params, "params")
    if d != spec.d or params.numel() != spec.num_params:
        raise PdeipError(f"shape mismatch: the state has d={d}, params has {params.numel()} entries (expected "
                         f"d={spec.d}, {spec.num_params} params)")
    _ops.overdamped_integrate_model(x0, x_last, traj, n, d, n_steps, float(dt), spec.kind, params, spec.hidden,
                                    spec.layers, spec.n_gaussian, noise, as_i64(seed), as_i64(particle_offset),
                                    step_offset, state_layout, traj_layout, emit_every, emit_offset,
                                    1 if emit_drift else 0, path)
    launch_counter["n"] += 1
    return x_last, traj


def philox_normals(n: int, n_draws: int, d: int, seed: int, particle_offset: int = 0, step_offset: int = 0,
                   device="cuda") -> torch.Tensor:
    out = torch.empty((n, n_draws, d), device=device, dtype=torch.float32)
    L.check(L.load().pdeip_philox_normals(_ptr(out), n, n_draws, d, seed & 0xFFFFFFFFFFFFFFFF, particle_offset,
                                          step_offset, _stream()), "pdeip_philox_normals")
    launch_counter["n"] += 1
    return out


def philox_uniforms(n: int, seed: int, particle_offset: int = 0, device="cuda") -> torch.Tensor:
    out = torch.empty((n,), device=device, dtype=torch.float32)
    L.check(L.load().pdeip_philox_uniforms(_ptr(out), n, seed & 0xFFFFFFFFFFFFFFFF, particle_offset, _stream()),
            "pdeip_philox_uniforms")
    launch_counter["n"] += 1
    return out


def philox_raw(ctr: torch.Tensor, key: torch.Tensor) -> torch.Tensor:
    """ctr [n,4] int32 (bit pattern of uint32), key [2] int32 -> [n,4] int32."""
    if not (ctr.is_cuda and key.is_cuda and ctr.dtype == torch.int32 and key.dtype == torch.int32):
        raise PdeipError("philox_raw expects CUDA int32 tensors")
    ctr = ctr.contiguous()
    out = torch.empty_like(ctr)
    L.check(L.load().pdeip_philox_raw(_ptr(ctr), _ptr(key.contiguous()), _ptr(out), ctr.shape[0], _stream()),
            "pdeip_philox_raw")
    launch_counter["n"] += 1
    return out


def gaussian_sample(n: int, dim: int, mu: Optional[torch.Tensor], cov_half: Optional[torch.Tensor], seed: int,
                    particle_offset: int = 0, layout: int = L.LAYOUT_AOS, device="cuda") -> torch.Tensor:
    mu = _f32(mu, "mu", allow_none=True)
    cov_half = _f32(cov_half, "cov_half", allow_none=True)
    shape = (n, dim) if layout == L.LAYOUT_AOS else (dim, n)
    out = torch.empty(shape, device=device, dtype=torch.float32)
    _ops.gaussian_sample(out, n, dim, mu, cov_half, as_i64(seed), as_i64(particle_offset), layout)
    launch_counter["n"] += 1
    return out


def gaussian_sample_grouped(n_groups: int, per_group: int, dim: int, mus: torch.Tensor, cov_halves: torch.Tensor,
                            seed: int, particle_offset: int = 0) -> torch.Tensor:
    """[n_groups, per_group, dim] samples, one (mean, cov_half) per group."""
    mus = _f32(mus, "mus")
    cov_halves = _f32(cov_halves, "cov_halves")
    if tuple(mus.shape) != (n_groups, dim) or tuple(cov_halves.shape) != (n_groups, dim, dim):
        raise PdeipError("mus must be [G,dim] and cov_halves [G,dim,dim]")
    out = torch.empty((n_groups, per_group, dim), device=mus.device, dtype=torch.float32)
    L.check(L.load().pdeip_gaussian_sample_grouped(_ptr(out), n_groups, per_group, dim, _ptr(mus), _ptr(cov_halves),
                                                   seed & 0xFFFFFFFFFFFFFFFF, particle_offset, _stream()),
            "pdeip_gaussian_sample_grouped")
    launch_counter["n"] += 1
    return out


def ou_exact_sample(n: int, U: torch.Tensor, s: torch.Tensor, B0: torch.Tensor, B: torch.Tensor, mt0: torch.Tensor,
                    t_min: float, t_max: float, seed: int, particle_offset: int = 0, want_t: bool = False):
    U, s, B0, B, mt0 = (_f32(t, nm) for t, nm in ((U, "U"), (s, "s"), (B0, "B0"), (B, "B"), (mt0, "mt0")))
    d = s.numel()
    out = torch.empty((n, d), device=U.device, dtype=torch.float32)
    out_t = torch.empty((n,), device=U.device, dtype=torch.float32) if want_t else None
    L.check(L.load().pdeip_ou_exact_sample(_ptr(out), _ptr(out_t), n, d, _ptr(U), _ptr(s), _ptr(B0), _ptr(B),
                                           _ptr(mt0), float(t_min), float(t_max), seed & 0xFFFFFFFFFFFFFFFF,
                                           particle_offset, _stream()), "pdeip_ou_exact_sample")
    launch_counter["n"] += 1
    return (out, out_t) if want_t else out


# ------------------------------------------------------------------------------------------------
# K2 potentials
# ------------------------------------------------------------------------------------------------
def gmm_value_grad(x: torch.Tensor, mus: torch.Tensor, sigma: float = 1.0, want_value: bool = False,
                   want_grad: bool = True) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    x = _f32(x, "x")
    mus = _f32(mus, "mus")
    n, d = x.shape
    if mus.shape[1] != d:
        raise PdeipError(f"mus must be [K,{d}], got {tuple(mus.shape)}")
    val = torch.empty((n,), device=x.device, dtype=torch.float32) if want_value else None
    grd = torch.empty_like(x) if want_grad else None
    _ops.gmm_value_grad(x, mus, mus.shape[0], float(sigma), val, grd, n, d)
    launch_counter["n"] += 1
    return val, grd


def linear_grad(x: torch.Tensor, A: torch.Tensor) -> torch.Tensor:
    x = _f32(x, "x")
    A = _f32(A, "A")
    n, d = x.shape
    out = torch.empty_like(x)
    _ops.linear_grad(x, A, out, n, d)
    launch_counter["n"] += 1
    return out


# ------------------------------------------------------------------------------------------------
# model evaluation and residual
# ------------------------------------------------------------------------------------------------
class ModelSpec:
    """(model_kind, d, hidden, layers, n_gaussian) + the flat parameter count."""

    def __init__(self, model_kind: int, d: int, hidden: int = 0, layers: int = 0, n_gaussian: int = 0):
        self.kind, self.d, self.hidden, self.layers, self.n_gaussian = model_kind, d, hidden, layers, n_gaussian
        self.num_params = int(L.load().pdeip_model_num_params(model_kind, d, hidden, layers, n_gaussian))
        if self.num_params <= 0:
            raise PdeipError(f"unknown model kind {model_kind}")

    def args(self):
        return (self.d, self.hidden, self.layers, self.n_gaussian)


def model_eval(spec: ModelSpec, params: torch.Tensor, x: torch.Tensor, v: Optional[torch.Tensor] = None,
               want: Sequence[str] = ("value", "grad")) -> Dict[str, torch.Tensor]:
    params = _f32(params, "params")
    x = _f32(x, "x")
    v = _f32(v, "v", allow_none=True)
    n, d = x.shape
    if d != spec.d or params.numel() != spec.num_params:
        raise PdeipError(f"shape mismatch: x is [{n},{d}], params has {params.numel()} (expected d={spec.d}, "
                         f"{spec.num_params} params)")
    out = {}
    if "value" in want:
        out["value"] = torch.empty((n,), device=x.device, dtype=torch.float32)
    if "grad" in want:
        out["grad"] = torch.empty((n, d), device=x.device, dtype=torch.float32)
    if "vHv" in want:
        out["vHv"] = torch.empty((n,), device=x.device, dtype=torch.float32)
    if "laplacian" in want:
        out["laplacian"] = torch.empty((n,), device=x.device, dtype=torch.float32)
    _ops.model_eval(spec.kind, params, spec.d, spec.hidden, spec.layers, spec.n_gaussian, x, v, out.get("value"),
                    out.get("grad"), out.get("vHv"), out.get("laplacian"), n)
    launch_counter["n"] += 1
    return out


class TrueGrad:
    """Specification of grad V_true for the 0T sets (LINEAR: A [d,d]; GMM: mus [K,d], sigma)."""

    def __init__(self, kind: int = L.DRIFT_NONE, params: Optional[torch.Tensor] = None, sigma: float = 1.0):
        self.kind = kind
        self.params = _f32(params, "true_params", allow_none=(kind in (L.DRIFT_NONE, L.DRIFT_IN_POINTS)))
        self.n_gaussian = int(self.params.shape[0]) if kind == L.DRIFT_GMM else 0
        self.sigma = float(sigma)


class ResidualAccumulator:
    """begin / accumulate / finalize protocol of the residual kernels (include/pdeip.h)."""

    def __init__(self, spec: ModelSpec, device="cuda"):
        self.spec = spec
        lib = L.load()
        self.ws_bytes = int(lib.pdeip_residual_workspace_bytes(spec.kind, *spec.args()))
        self.ws = torch.empty((self.ws_bytes // 4,), device=device, dtype=torch.float32)
        self.sums = torch.empty((L.NUM_SUMS,), device=device, dtype=torch.float32)
        self.grad = torch.empty((spec.num_params,), device=device, dtype=torch.float32)

    def begin(self):
        _ops.residual_begin(self.ws, self.spec.kind, *self.spec.args())
        return self

    def accumulate(self, set_kind: int, params: torch.Tensor, points: torch.Tensor, weight: float, coef: float = 0.0,
                   layout: int = L.LAYOUT_AOS, true_grad: Optional[TrueGrad] = None, path: int = L.PATH_FP32,
                   n_points: Optional[int] = None):
        params = _f32(params, "params")
        points = _f32(points, "points")
        if params.numel() != self.spec.num_params:
            raise PdeipError(f"params has {params.numel()} entries, expected {self.spec.num_params}")
        kinetic = set_kind in (L.SET_KFP_0T, L.SET_KFP_BOUNDARY)
        dim = 2 * self.spec.d if kinetic else self.spec.d
        if true_grad is not None and true_grad.kind == L.DRIFT_IN_POINTS:
            dim += self.spec.d  # grad V_true stored after the point's own components
        if n_points is None:
            if layout == L.LAYOUT_AOS:
                if points.ndim != 2 or points.shape[1] != dim:
                    raise PdeipError(f"points must be [n,{dim}], got {tuple(points.shape)}")
                n_points = points.shape[0]
            elif layout == L.LAYOUT_BLOCK128:
                if points.ndim != 3 or tuple(points.shape[1:]) != (dim, 128):
                    raise PdeipError(f"points must be [n/128,{dim},128], got {tuple(points.shape)}")
                n_points = points.shape[0] * 128
            else:
                if points.ndim != 2 or points.shape[0] != dim:
                    raise PdeipError(f"points must be [{dim},n], got {tuple(points.shape)}")
                n_points = points.shape[1]
        tg = true_grad or TrueGrad()
        _ops.residual_accumulate(self.ws, set_kind, self.spec.kind, params, *self.spec.args(), points, n_points, layout,
                                 float(weight), float(coef), tg.kind, tg.params, tg.n_gaussian, tg.sigma, path)
        launch_counter["n"] += 1
        return self

    def finalize(self) -> Tuple[torch.Tensor, torch.Tensor]:
        _ops.residual_finalize(self.ws, self.spec.kind, *self.spec.args(), self.sums, self.grad)
        launch_counter["n"] += 2
        return self.sums, self.grad


# ------------------------------------------------------------------------------------------------
# K6 / K7 / gather
# ------------------------------------------------------------------------------------------------
def adam_l2_step(params: torch.Tensor, grad: torch.Tensor, m: torch.Tensor, v: torch.Tensor, count: int, lr: float,
                 b1: float = 0.9, b2: float = 0.999, eps: float = 1e-4, weight_decay: float = 1e-3,
                 grad_scale: float = 1.0, ema: Optional[torch.Tensor] = None, use_ema: bool = False,
                 ema_decay: float = 0.999, norms: Optional[torch.Tensor] = None) -> torch.Tensor:
    """In-place optimizer step on the flat parameter buffer; returns norms [grad_norm, params_norm]."""
    for name, t in (("params", params), ("grad", grad), ("m", m), ("v", v)):
        if _f32(t, name) is not t:
            raise PdeipError(f"{name} must be contiguous (updated in place)")
    if norms is None:
        norms = torch.empty((2,), device=params.device, dtype=torch.float32)
    _ops.adam_l2_step(params, grad, m, v, ema, float(lr), float(b1), float(b2), float(eps), float(weight_decay),
                      int(count), float(grad_scale), 1 if use_ema else 0, float(ema_decay), norms)
    launch_counter["n"] += 1
    return norms


def ensemble_moments(z: torch.Tensor, layout: int = L.LAYOUT_AOS) -> Tuple[torch.Tensor, torch.Tensor]:
    """Raw sums (sum z [dim], sum z z^T [dim,dim])."""
    z = _f32(z, "z")
    n, dim = z.shape if layout == L.LAYOUT_AOS else (z.shape[1], z.shape[0])
    lib = L.load()
    ws_bytes = int(lib.pdeip_moments_workspace_bytes(dim))
    ws = torch.empty((ws_bytes // 4,), device=z.device, dtype=torch.float32)
    out = torch.empty((dim + dim * dim,), device=z.device, dtype=torch.float32)
    _ops.ensemble_moments(z, n, dim, layout, out, ws)
    launch_counter["n"] += 2
    return out[:dim], out[dim:].view(dim, dim)


def gather_0T(dataset: torch.Tensor, sample_index: torch.Tensor, interval: int, shift: int) -> torch.Tensor:
    """methods/consistency.py:102-118 as one device gather.  dataset [n_traj,n_time,dim]."""
    dataset = _f32(dataset, "dataset")
    if not (sample_index.is_cuda and sample_index.dtype == torch.int64):
        raise PdeipError("sample_index must be a CUDA int64 tensor")
    n_traj, n_time, dim = dataset.shape
    n_time_sel = n_time // interval
    n_sel = sample_index.numel()
    out = torch.empty((n_sel * n_time_sel, dim), device=dataset.device, dtype=torch.float32)
    _ops.gather_0T(dataset, n_traj, n_time, dim, sample_index.contiguous(), n_sel, interval, shift, n_time_sel, out)
    launch_counter["n"] += 1
    return out


# ------------------------------------------------------------------------------------------------
# KMV pairwise residual (kinetic_mckean_vlasov.py:11-120)
# ------------------------------------------------------------------------------------------------
def kmv_mean_grad(spec: ModelSpec, params: torch.Tensor, xv: torch.Tensor, true_A: Optional[torch.Tensor] = None,
                  ref: Optional[torch.Tensor] = None, m: Optional[int] = None):
    """G[j,t] = mean_i grad Phi(x[j,t] - ref[i,t]) and, if true_A is given, the same for Phi_true = D'AD/2.
    xv: [n, nt, 2d]; ref: [m, nt, 2d] (None: the batch itself, optionally only its first m trajectories)."""
    params = _f32(params, "params")
    xv = _f32(xv, "xv")
    true_A = _f32(true_A, "true_A", allow_none=True)
    ref = _f32(ref, "ref", allow_none=True)
    n, nt, two_d = xv.shape
    d = two_d // 2
    if ref is None and m is not None and m != n:
        ref = xv  # sub-sampled reference set: the first m trajectories of the batch
    m = int(n if ref is None else (ref.shape[0] if m is None else m))
    ws_bytes = int(L.load().pdeip_kmv_workspace_bytes_ref(n, nt, d, m))
    ws = torch.empty((ws_bytes // 4,), device=xv.device, dtype=torch.float32)
    G = torch.empty((n, nt, d), device=xv.device, dtype=torch.float32)
    Gt = torch.empty_like(G) if true_A is not None else None
    _ops.kmv_mean_grad(spec.kind, params, d, spec.hidden, spec.layers, xv, n, nt, ref, m, G, Gt, true_A, ws)
    launch_counter["n"] += 2
    return G, Gt


def kmv_density_terms(xv: torch.Tensor, coef: torch.Tensor, gamma: float, want_parts: bool = False):
    """c = d_ss log rho + (d_s log rho)^2 + gamma d_s log rho at every (time stamp, sample) on the device
    (kinetic_mckean_vlasov_example_quadratic.py:51-69,120-177).  xv [n, nt, 2d]; coef [nt, 3d + 2 + 2d^2]
    (utils/lyapunov.kmv_density_coefficients).  Returns c as [nt, n] (the reference reshapes it to [n, nt])."""
    xv = _f32(xv, "xv")
    coef = _f32(coef, "coef")
    n, nt, two_d = xv.shape
    d = two_d // 2
    if tuple(coef.shape) != (nt, 3 * d + 2 + 2 * d * d):
        raise PdeipError(f"coef must be [{nt},{3 * d + 2 + 2 * d * d}], got {tuple(coef.shape)}")
    c = torch.empty((nt, n), device=xv.device, dtype=torch.float32)
    ps = torch.empty_like(c) if want_parts else None
    ps2 = torch.empty_like(c) if want_parts else None
    _ops.kmv_density_terms(xv, n, nt, d, coef, float(gamma), c, ps, ps2)
    launch_counter["n"] += 1
    return (c, ps, ps2) if want_parts else c


def kmv_value_and_grad(model, params, flat: torch.Tensor, xv: torch.Tensor, c: torch.Tensor, true_A: torch.Tensor,
                       acc: "ResidualAccumulator", result_dict, m: Optional[int] = None, closure: bool = False):
    """Phase 1 (mean gradient per sample), then the pair set with the extra direction G_j and kappa = 2 c_j.
    m: reference-set size (the first m trajectories of the batch; None = the batch, as the reference).
    closure: quadratic model only — the pair set against the reference MEAN plus the covariance correction
    (exactly the full pair set, O(n) instead of O(n m))."""
    xv = _f32(xv, "xv")
    c = _f32(c, "c")
    n, nt, two_d = xv.shape
    d = two_d // 2
    spec = model.spec
    m = n if m is None else int(m)
    ref, m_eff, cov = None, m, None
    if closure:
        if spec.kind != L.MODEL_QUADRATIC:
            raise PdeipError("the moment closure is exact for the quadratic interaction model only")
        # per time stamp: mean and covariance of the reference x through the K7 moments kernel
        ref = torch.zeros((1, nt, two_d), device=xv.device, dtype=torch.float32)
        cov = torch.empty((nt, d, d), device=xv.device, dtype=torch.float32)
        for t in range(nt):
            s1, s2 = ensemble_moments(xv[:m, t, :d].contiguous())
            mean = s1 / m
            ref[0, t, :d] = mean
            cov[t] = s2 / m - torch.outer(mean, mean)
        m_eff = 1
    elif m != n:
        ref = xv
    G, Gt = kmv_mean_grad(spec, flat, xv, true_A, ref=ref, m=m_eff)
    acc.begin()
    w = 1.0 / (float(n) * m_eff * nt)
    _ops.residual_accumulate_kmv(acc.ws, spec.kind, flat, spec.d, spec.hidden, spec.layers, xv, n, nt, ref, m_eff, G, Gt, c, w)
    launch_counter["n"] += 2
    if closure:
        _ops.kmv_closure_correction(acc.ws, flat, d, n, nt, c, cov, w)
        launch_counter["n"] += 1
    sums, grad = acc.finalize()
    return result_dict(model, params, sums, grad)


# ------------------------------------------------------------------------------------------------
# mean-field drift: the ensemble-mean table of the interacting system (README.md:54-62)
# ------------------------------------------------------------------------------------------------
def meanfield_noise_sums(z0: torch.Tensor, n_steps: int, seed: int, particle_offset: int = 0, step_offset: int = 0,
                         out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Accumulates into `out` (float64 [(n_steps+1)*d + 2d], zero-initialised if None) the per-step sums of the Philox
    normals the integrator will draw for these particles, and sum q0, sum p0.  z0: [n, 2d] CUDA."""
    z0 = _f32(z0, "z0")
    n, two_d = z0.shape
    d = two_d // 2
    if out is None:
        out = torch.zeros(((n_steps + 1) * d + 2 * d,), device=z0.device, dtype=torch.float64)
    _ops.meanfield_noise_sums(z0, n, d, n_steps, as_i64(seed), as_i64(particle_offset), step_offset, out)
    launch_counter["n"] += 1
    return out


def meanfield_drift_params(sums: torch.Tensor, n_global: int, A: torch.Tensor, n_steps: int, dt: float, gamma: float):
    """(drift_params, xbar): drift_params = [A (d*d) | A xbar_s (n_steps+1, d)] for DRIFT_MEANFIELD_TABLE, xbar
    [n_steps+1, d] the ensemble mean before every step.  `sums` must already be reduced over ranks."""
    A = _f32(A, "A")
    d = A.shape[0]
    params = torch.empty((d * d + (n_steps + 1) * d,), device=A.device, dtype=torch.float32)
    params[: d * d] = A.reshape(-1)
    xbar = torch.empty((n_steps + 1, d), device=A.device, dtype=torch.float32)
    _ops.meanfield_xbar_table(sums, int(n_global), d, n_steps, float(dt), float(gamma), A, xbar, params[d * d:])
    launch_counter["n"] += 1
    return params, xbar


def tensor_path_status() -> int:
    """0 if every tcgen05 phase of the tensor-path launches so far completed (synchronises the stream)."""
    import ctypes as C
    out = C.c_int(-1)
    L.check(L.load().pdeip_tensor_path_status(_stream(), C.addressof(out)), "pdeip_tensor_path_status")
    return int(out.value)
