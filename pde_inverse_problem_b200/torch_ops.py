"""The C ABI (include/pdeip.h) registered as PyTorch custom ops: torch.ops.pdeip.*.

North-star boundary: "hand-written sm_100a CUDA kernels behind a thin C-ABI custom-call layer ... a torch custom op".
Every op below is a `torch.library.custom_op` whose CUDA implementation is ONE call into libpdeip.so on torch's
current stream: device pointers, sizes and scalars in, a status code out (raised as PdeipError).  The ops mutate
caller-allocated outputs (the C ABI never allocates), so their schemas carry `Tensor(a!)` annotations and return
nothing; `ops.py` allocates the outputs and is the only caller.  There is no CPU implementation: the ops are
registered for device type "cuda" only, so a CPU tensor fails in the dispatcher ("no kernel for backend CPU").

Replaces (reference file:line, as in pdeip.h): kl_integrate, kl_integrate_model — utils/sampling_utils.py:6-52;
overdamped_integrate, overdamped_integrate_model — the SDE of example_problems/fokker_planck_example.py;
gmm_value_grad — core/potential.py:32-61; model_eval — core/model.py:51-62 + utils/common_utils.py:6-14; residual_* —
methods/consistency_instances/{kinetic_fokker_planck.py:11-69, fokker_planck.py:33-63, kinetic_mckean_vlasov.py:11-120};
adam_l2_step — main.py:20-26 + core/trainer.py:61-70; ensemble_moments — example_problems/
kinetic_fokker_planck_example_OU.py:73-93 (ensemble side); gather_0T — methods/consistency.py:102-118;
gaussian_sample — core/distribution.py:64-65.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib as L

_U64 = 0xFFFFFFFFFFFFFFFF


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _u64(x: int) -> int:
    """schema ints are int64: seeds / offsets travel as the signed image of the uint64 the C ABI takes."""
    return int(x) & _U64


def as_i64(x: int) -> int:
    x = int(x) & _U64
    return x - (1 << 64) if x >= (1 << 63) else x


def _op(name, mutates):
    return torch.library.custom_op(f"pdeip::{name}", mutates_args=mutates, device_types="cuda")


@_op("kl_integrate", ("z_last", "traj", "tau"))
def kl_integrate(z0: torch.Tensor, z_last: torch.Tensor, traj: Optional[torch.Tensor], tau: Optional[torch.Tensor],
                 n_particles: int, d: int, n_steps: int, dt: float, gamma: float, drift_kind: int,
                 drift_params: Optional[torch.Tensor], n_gaussian: int, sigma: float, noise: Optional[torch.Tensor],
                 tau0: Optional[torch.Tensor], seed: int, particle_offset: int, step_offset: int, schedule: int,
                 state_layout: int, traj_layout: int, emit_every: int, emit_offset: int, emit_drift: int,
                 path: int) -> None:
    L.check(L.load().pdeip_kl_integrate_path(
        _p(z0), _p(z_last), _p(traj), _p(tau), n_particles, d, n_steps, dt, gamma, drift_kind, _p(drift_params),
        n_gaussian, sigma, _p(noise), _p(tau0), _u64(seed), _u64(particle_offset), step_offset, schedule, state_layout,
        traj_layout, emit_every, emit_offset, emit_drift, path, _stream()), "pdeip_kl_integrate_path")


@_op("kl_integrate_model", ("z_last", "traj", "tau"))
def kl_integrate_model(z0: torch.Tensor, z_last: torch.Tensor, traj: Optional[torch.Tensor],
                       tau: Optional[torch.Tensor], n_particles: int, d: int, n_steps: int, dt: float, gamma: float,
                       model_kind: int, params: torch.Tensor, hidden: int, layers: int, n_gaussian: int,
                       noise: Optional[torch.Tensor], tau0: Optional[torch.Tensor], seed: int, particle_offset: int,
                       step_offset: int, schedule: int, state_layout: int, traj_layout: int, emit_every: int,
                       emit_offset: int, emit_drift: int, path: int) -> None:
    L.check(L.load().pdeip_kl_integrate_model(
        _p(z0), _p(z_last), _p(traj), _p(tau), n_particles, d, n_steps, dt, gamma, model_kind, _p(params), hidden,
        layers, n_gaussian, _p(noise), _p(tau0), _u64(seed), _u64(particle_offset), step_offset, schedule,
        state_layout, traj_layout, emit_every, emit_offset, emit_drift, path, _stream()), "pdeip_kl_integrate_model")


@_op("overdamped_integrate", ("x_last", "traj"))
def overdamped_integrate(x0: torch.Tensor, x_last: torch.Tensor, traj: Optional[torch.Tensor], n_particles: int, d: int,
                         n_steps: int, dt: float, drift_kind: int, drift_params: Optional[torch.Tensor], n_gaussian: int,
                         sigma: float, noise: Optional[torch.Tensor], seed: int, particle_offset: int, step_offset: int,
                         state_layout: int, traj_layout: int, emit_every: int, emit_offset: int, emit_drift: int,
                         path: int) -> None:
    L.check(L.load().pdeip_overdamped_integrate(
        _p(x0), _p(x_last), _p(traj), n_particles, d, n_steps, dt, drift_kind, _p(drift_params), n_gaussian, sigma,
        _p(noise), _u64(seed), _u64(particle_offset), step_offset, state_layout, traj_layout, emit_every, emit_offset,
        emit_drift, path, _stream()), "pdeip_overdamped_integrate")


@_op("overdamped_integrate_model", ("x_last", "traj"))
def overdamped_integrate_model(x0: torch.Tensor, x_last: torch.Tensor, traj: Optional[torch.Tensor], n_particles: int,
                               d: int, n_steps: int, dt: float, model_kind: int, params: torch.Tensor, hidden: int,
                               layers: int, n_gaussian: int, noise: Optional[torch.Tensor], seed: int,
                               particle_offset: int, step_offset: int, state_layout: int, traj_layout: int,
                               emit_every: int, emit_offset: int, emit_drift: int, path: int) -> None:
    L.check(L.load().pdeip_overdamped_integrate_model(
        _p(x0), _p(x_last), _p(traj), n_particles, d, n_steps, dt, model_kind, _p(params), hidden, layers, n_gaussian,
        _p(noise), _u64(seed), _u64(particle_offset), step_offset, state_layout, traj_layout, emit_every, emit_offset,
        emit_drift, path, _stream()), "pdeip_overdamped_integrate_model")


@_op("meanfield_noise_sums", ("sums",))
def meanfield_noise_sums(z0: torch.Tensor, n_particles: int, d: int, n_steps: int, seed: int, particle_offset: int,
                         step_offset: int, sums: torch.Tensor) -> None:
    L.check(L.load().pdeip_meanfield_noise_sums(_p(z0), n_particles, d, n_steps, _u64(seed), _u64(particle_offset),
                                                step_offset, _p(sums), _stream()), "pdeip_meanfield_noise_sums")


@_op("meanfield_xbar_table", ("xbar", "drift_table"))
def meanfield_xbar_table(sums: torch.Tensor, n_global: int, d: int, n_steps: int, dt: float, gamma: float,
                         A: torch.Tensor, xbar: Optional[torch.Tensor], drift_table: torch.Tensor) -> None:
    L.check(L.load().pdeip_meanfield_xbar_table(_p(sums), n_global, d, n_steps, dt, gamma, _p(A), _p(xbar),
                                                _p(drift_table), _stream()), "pdeip_meanfield_xbar_table")


@_op("gmm_value_grad", ("out_value", "out_grad"))
def gmm_value_grad(x: torch.Tensor, mus: torch.Tensor, n_gaussian: int, sigma: float, out_value: Optional[torch.Tensor],
                   out_grad: Optional[torch.Tensor], n: int, d: int) -> None:
    L.check(L.load().pdeip_gmm_value_grad(_p(x), _p(mus), n_gaussian, sigma, _p(out_value), _p(out_grad), n, d,
                                          _stream()), "pdeip_gmm_value_grad")


@_op("linear_grad", ("out",))
def linear_grad(x: torch.Tensor, A: torch.Tensor, out: torch.Tensor, n: int, d: int) -> None:
    L.check(L.load().pdeip_linear_grad(_p(x), _p(A), _p(out), n, d, _stream()), "pdeip_linear_grad")


@_op("model_eval", ("out_value", "out_grad", "out_vHv", "out_lap"))
def model_eval(model_kind: int, params: torch.Tensor, d: int, hidden: int, layers: int, n_gaussian: int,
               x: torch.Tensor, v: Optional[torch.Tensor], out_value: Optional[torch.Tensor],
               out_grad: Optional[torch.Tensor], out_vHv: Optional[torch.Tensor], out_lap: Optional[torch.Tensor],
               n: int) -> None:
    L.check(L.load().pdeip_model_eval(model_kind, _p(params), d, hidden, layers, n_gaussian, _p(x), _p(v),
                                      _p(out_value), _p(out_grad), _p(out_vHv), _p(out_lap), n, _stream()),
            "pdeip_model_eval")


@_op("residual_begin", ("workspace",))
def residual_begin(workspace: torch.Tensor, model_kind: int, d: int, hidden: int, layers: int, n_gaussian: int) -> None:
    L.check(L.load().pdeip_residual_begin(_p(workspace), workspace.numel() * workspace.element_size(), model_kind, d,
                                          hidden, layers, n_gaussian, _stream()), "pdeip_residual_begin")


@_op("residual_accumulate", ("workspace",))
def residual_accumulate(workspace: torch.Tensor, set_kind: int, model_kind: int, params: torch.Tensor, d: int,
                        hidden: int, layers: int, n_gaussian: int, points: torch.Tensor, n_points: int, layout: int,
                        weight: float, coef: float, true_kind: int, true_params: Optional[torch.Tensor],
                        true_n_gaussian: int, true_sigma: float, path: int) -> None:
    L.check(L.load().pdeip_residual_accumulate(
        _p(workspace), workspace.numel() * workspace.element_size(), set_kind, model_kind, _p(params), d, hidden, layers,
        n_gaussian, _p(points), n_points, layout, weight, coef, true_kind, _p(true_params), true_n_gaussian, true_sigma,
        path, _stream()), "pdeip_residual_accumulate")


@_op("residual_finalize", ("sums", "grad"))
def residual_finalize(workspace: torch.Tensor, model_kind: int, d: int, hidden: int, layers: int, n_gaussian: int,
                      sums: torch.Tensor, grad: torch.Tensor) -> None:
    L.check(L.load().pdeip_residual_finalize(_p(workspace), workspace.numel() * workspace.element_size(), model_kind, d,
                                             hidden, layers, n_gaussian, _p(sums), _p(grad), _stream()),
            "pdeip_residual_finalize")


@_op("kmv_mean_grad", ("out_G", "out_Gtrue", "workspace"))
def kmv_mean_grad(model_kind: int, params: torch.Tensor, d: int, hidden: int, layers: int, xv: torch.Tensor, n: int,
                  nt: int, ref: Optional[torch.Tensor], m: int, out_G: torch.Tensor, out_Gtrue: Optional[torch.Tensor],
                  true_A: Optional[torch.Tensor], workspace: torch.Tensor) -> None:
    L.check(L.load().pdeip_kmv_mean_grad_ref(model_kind, _p(params), d, hidden, layers, _p(xv), n, nt, _p(ref), m,
                                             _p(out_G), _p(out_Gtrue), _p(true_A), _p(workspace),
                                             workspace.numel() * workspace.element_size(), _stream()),
            "pdeip_kmv_mean_grad_ref")


@_op("residual_accumulate_kmv", ("workspace",))
def residual_accumulate_kmv(workspace: torch.Tensor, model_kind: int, params: torch.Tensor, d: int, hidden: int,
                            layers: int, xv: torch.Tensor, n: int, nt: int, ref: Optional[torch.Tensor], m: int,
                            G: Optional[torch.Tensor], G_true: Optional[torch.Tensor], c: torch.Tensor,
                            weight: float) -> None:
    L.check(L.load().pdeip_residual_accumulate_kmv_ref(
        _p(workspace), workspace.numel() * workspace.element_size(), model_kind, _p(params), d, hidden, layers, _p(xv),
        n, nt, _p(ref), m, _p(G), _p(G_true), _p(c), weight, _stream()), "pdeip_residual_accumulate_kmv_ref")


@_op("kmv_closure_correction", ("workspace",))
def kmv_closure_correction(workspace: torch.Tensor, params: torch.Tensor, d: int, n: int, nt: int, c: torch.Tensor,
                           cov: torch.Tensor, weight: float) -> None:
    L.check(L.load().pdeip_kmv_closure_correction(_p(workspace), workspace.numel() * workspace.element_size(),
                                                  _p(params), d, n, nt, _p(c), _p(cov), weight, _stream()),
            "pdeip_kmv_closure_correction")


@_op("kmv_density_terms", ("out_c", "out_ps", "out_ps2"))
def kmv_density_terms(xv: torch.Tensor, n: int, nt: int, d: int, coef: torch.Tensor, gamma: float,
                      out_c: Optional[torch.Tensor], out_ps: Optional[torch.Tensor],
                      out_ps2: Optional[torch.Tensor]) -> None:
    L.check(L.load().pdeip_kmv_density_terms(_p(xv), n, nt, d, _p(coef), gamma, _p(out_c), _p(out_ps), _p(out_ps2),
                                             _stream()), "pdeip_kmv_density_terms")


@_op("adam_l2_step", ("params", "m", "v", "ema", "norms"))
def adam_l2_step(params: torch.Tensor, grad: torch.Tensor, m: torch.Tensor, v: torch.Tensor,
                 ema: Optional[torch.Tensor], lr: float, b1: float, b2: float, eps: float, weight_decay: float,
                 count: int, grad_scale: float, use_ema: int, ema_decay: float, norms: torch.Tensor) -> None:
    L.check(L.load().pdeip_adam_l2_step(_p(params), _p(grad), _p(m), _p(v), _p(ema), params.numel(), lr, b1, b2, eps,
                                        weight_decay, count, grad_scale, use_ema, ema_decay, _p(norms), _stream()),
            "pdeip_adam_l2_step")


@_op("ensemble_moments", ("out", "workspace"))
def ensemble_moments(z: torch.Tensor, n: int, dim: int, layout: int, out: torch.Tensor, workspace: torch.Tensor) -> None:
    L.check(L.load().pdeip_ensemble_moments(_p(z), n, dim, layout, _p(out), _p(workspace),
                                            workspace.numel() * workspace.element_size(), _stream()),
            "pdeip_ensemble_moments")


@_op("gather_0T", ("out",))
def gather_0T(dataset: torch.Tensor, n_traj: int, n_time: int, dim: int, sample_index: torch.Tensor, n_sel: int,
              interval: int, shift: int, n_time_sel: int, out: torch.Tensor) -> None:
    L.check(L.load().pdeip_gather_0T(_p(dataset), n_traj, n_time, dim, _p(sample_index), n_sel, interval, shift,
                                     n_time_sel, _p(out), _stream()), "pdeip_gather_0T")


@_op("gaussian_sample", ("out",))
def gaussian_sample(out: torch.Tensor, n: int, dim: int, mu: Optional[torch.Tensor], cov_half: Optional[torch.Tensor],
                    seed: int, particle_offset: int, layout: int) -> None:
    L.check(L.load().pdeip_gaussian_sample(_p(out), n, dim, _p(mu), _p(cov_half), _u64(seed), _u64(particle_offset),
                                           layout, _stream()), "pdeip_gaussian_sample")


REGISTERED = ("kl_integrate", "kl_integrate_model", "overdamped_integrate", "overdamped_integrate_model",
              "meanfield_noise_sums", "meanfield_xbar_table", "gmm_value_grad", "linear_grad",
              "model_eval", "residual_begin", "residual_accumulate", "residual_finalize", "kmv_mean_grad",
              "residual_accumulate_kmv", "kmv_closure_correction", "kmv_density_terms", "adam_l2_step",
              "ensemble_moments", "gather_0T", "gaussian_sample")
