"""The particle-ensemble hot path as one object: integrate -> residual -> (all-reduce) -> optimizer step.

This is the online "SDE" iteration of the reference at ensemble scale (methods/consistency.py:77-86 ->
example_problems/kinetic_fokker_planck_example_GMM.py:104-142 -> utils/sampling_utils.py:25-52 ->
methods/consistency_instances/kinetic_fokker_planck.py:11-69 -> core/trainer.py:61-70), restructured for
180 GB of HBM: particles are processed in chunks, each chunk's trajectory is emitted by K1 as one SOA point
set [2d][S*Nc] and consumed immediately by the residual kernel, so the full [N, S, 2d] trajectory (54 GB at
C3, 860 GB at C5) is never materialised.  Every emitted trajectory sample is a 0T point; the chunk's initial
and terminal states are the boundary sets (the variant at GMM.py:144-156).

HotPathConfig.dynamics = "overdamped" is the same iteration for the Fokker-Planck instance (dX = -grad U dt + sqrt(2) dW,
fokker_planck_example_GMM.py): K1-OD emits each chunk as [x, grad U(x)] samples, which are directly an FP point set
with DRIFT_IN_POINTS (SET_FP_0T), and the initial and terminal states are the FP boundary sets (SET_FP_BOUNDARY).

Estimator: the 0T set is the time marginals on the uniform step grid, and the boundary sets come from the same
ensemble as the 0T set.  The reference draws its 0T points at random times and its boundary samples independently;
both variants estimate the same expectations.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional

import torch

from . import _lib as L
from . import ops, parallel
from .core.optimizer import AdamL2, OptState


def integrator_wave(d: int, drift_kind: int, n_gaussian: int, path: int, sm_count: Optional[int] = None, *,
                    overdamped: bool = False) -> int:
    """Particles in one full wave of the production integrator grid (128 particles per CTA x CTAs per SM x SMs):
    the tcgen05 GMM kernels run 8 (d = 8) / 3 (d = 16, 32) CTAs per SM, their overdamped trajectory instances 6 (d = 8)
    / 3 (d = 16, 32), the fp32 kernel 4 (2 at d = 32) (csrc/integrator_tc.cu, csrc/integrator.cu launch bounds)."""
    sms = sm_count if sm_count is not None else L.load().pdeip_sm_count()
    tensor = path == L.PATH_TENSOR and drift_kind == L.DRIFT_GMM and d in (8, 16, 32) and 1 <= n_gaussian <= 64
    per_sm = ((6 if overdamped else 8) if d == 8 else 3) if tensor else (2 if d >= 32 else 4)
    return 128 * per_sm * sms


def auto_chunk(d: int, n_steps: int, drift_kind: int, n_gaussian: int, path: int, emit_every: int = 1,
               budget_bytes: float = 6.0e9, sm_count: Optional[int] = None, *, overdamped: bool = False) -> int:
    """Largest whole number of integrator waves whose [x, v, grad U] (overdamped: [x, grad U]) trajectory fits
    `budget_bytes` (at least one wave): no partially filled last wave, and a trajectory buffer far above the 126 MB L2."""
    wave = integrator_wave(d, drift_kind, n_gaussian, path, sm_count, overdamped=overdamped)
    s_emit = (n_steps + emit_every - 1) // emit_every
    per_particle = (2 if overdamped else 3) * d * s_emit * 4
    return wave * max(1, int(budget_bytes // (per_particle * wave)))


@dataclass
class HotPathConfig:
    d: int
    n_steps: int
    total_time: float
    gamma: float
    drift_kind: int
    n_gaussian: int = 0
    sigma: float = 1.0
    chunk: int = 0  # particles per integrate -> residual round trip; 0 = auto_chunk(...)
    emit_every: int = 1
    path: int = L.PATH_FP32
    dynamics: str = "kinetic"  # or "overdamped": K1-OD and the FP sets; the state is x [n, d] and gamma is ignored


class HotPath:
    def __init__(self, cfg: HotPathConfig, model, params: Dict, drift_params: Optional[torch.Tensor],
                 true_grad: ops.TrueGrad, optimizer: Optional[AdamL2] = None, device="cuda"):
        if cfg.dynamics not in ("kinetic", "overdamped"):
            raise ValueError(f"unknown dynamics {cfg.dynamics!r}: 'kinetic' or 'overdamped'")
        self.overdamped = cfg.dynamics == "overdamped"
        if self.overdamped and cfg.drift_kind == L.DRIFT_MEANFIELD_TABLE:
            raise ValueError("DRIFT_MEANFIELD_TABLE encodes the underdamped mean recursion; the overdamped dynamics "
                             "do not take it")
        if cfg.chunk <= 0:
            cfg.chunk = auto_chunk(cfg.d, cfg.n_steps, cfg.drift_kind, cfg.n_gaussian, cfg.path, cfg.emit_every,
                                   overdamped=self.overdamped)
        self.cfg, self.model, self.params = cfg, model, params
        self.drift_params, self.true_grad, self.optimizer = drift_params, true_grad, optimizer
        self.device = torch.device(device)
        self.acc = ops.ResidualAccumulator(model.spec, device=self.device)
        self.opt_state: Optional[OptState] = optimizer.init(params) if optimizer is not None else None
        self.norms = torch.empty(2, device=self.device, dtype=torch.float32)
        s_emit = (cfg.n_steps + cfg.emit_every - 1) // cfg.emit_every
        self.s_emit = s_emit
        # every sample carries [x, v, grad U(x)] (overdamped: [x, grad U(x)]): the integrator emits the drift it
        # evaluates anyway
        self.width = (2 if self.overdamped else 3) * cfg.d  # floats per emitted sample
        self.state = (1 if self.overdamped else 2) * cfg.d  # floats per state
        self.traj = torch.empty(self.width * s_emit * cfg.chunk, device=self.device, dtype=torch.float32)
        self.true_in_points = ops.TrueGrad(L.DRIFT_IN_POINTS)
        self.z_last = torch.empty((cfg.chunk, self.state), device=self.device, dtype=torch.float32)
        self.z_last_full: Optional[torch.Tensor] = None  # [n, 2d] ([n, d] overdamped) terminal states of all chunks (batched boundary sets)
        self.z0_full: Optional[torch.Tensor] = None      # [n, 2d] ([n, d]) device copy of the staged initial states (host-resident)
        # host-resident ensembles: two staging buffers and a copy stream, so that chunk k+1 crosses PCIe / NVLink-C2C
        # while chunk k is integrated
        self.z_stage = [torch.empty((cfg.chunk, self.state), device=self.device, dtype=torch.float32) for _ in range(2)]
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.stage_ready = [torch.cuda.Event() for _ in range(2)]  # H2D of the buffer finished
        self.stage_free = [torch.cuda.Event() for _ in range(2)]   # last kernel reading the buffer finished

    def particle_steps(self, n: int) -> int:
        if self.overdamped:
            return n * self.cfg.n_steps  # S Euler-Maruyama steps per trajectory
        return n * (self.cfg.n_steps + 1)  # the reference does S+1 update_steps per trajectory

    def residual_evals(self, n: int) -> int:
        return n * self.s_emit

    def meanfield_table(self, z0: torch.Tensor, seed: int, n_global: int, particle_offset: int) -> torch.Tensor:
        """Interacting system (drift A (x - xbar_t), xbar_t the empirical mean over ALL ranks' particles, README.md:54-62):
        one pre-pass over the local particles sums the Philox normals of every step (and z0), ONE all-reduce of
        (S+1) d + 2 d doubles replaces S per-step exchanges of sum x, and the closed recursion of the ensemble mean gives
        the per-step table the integrator reads (csrc/integrator.cu).  self.drift_params is A [d, d]."""
        c = self.cfg
        sums = torch.zeros(((c.n_steps + 1) * c.d + 2 * c.d,), device=self.device, dtype=torch.float64)
        n = z0.shape[0]
        for lo in range(0, n, c.chunk):
            hi = min(n, lo + c.chunk)
            zc = z0[lo:hi] if z0.is_cuda else self.z_stage[0][: hi - lo].copy_(z0[lo:hi], non_blocking=True)
            ops.meanfield_noise_sums(zc.contiguous(), c.n_steps, seed, particle_offset=particle_offset + lo, out=sums)
        if parallel.Shard.current().world > 1:  # float64 sums: not through the float32 packing of allreduce_sum_packed
            torch.distributed.all_reduce(sums, op=torch.distributed.ReduceOp.SUM)
        params, self.xbar = ops.meanfield_drift_params(sums, n_global, self.drift_params, c.n_steps,
                                                       c.total_time / c.n_steps, c.gamma)
        return params

    def step(self, z0: torch.Tensor, seed: int, n_global: Optional[int] = None, particle_offset: int = 0,
             apply_optimizer: bool = True, phase_events: Optional[list] = None) -> Dict[str, torch.Tensor]:
        """One iteration over the local ensemble z0 [n, 2d] (overdamped: x0 [n, d]) (CUDA, or pinned host memory: then
        each chunk is copied host->device inside the step).  n_global: ensemble size over all ranks (weights are 1/global
        counts so shards add up under one all-reduce).  phase_events: if a list, three CUDA events per chunk are
        appended to it (before the integrator, between integrator and 0T residual, after the 0T residual)."""
        c = self.cfg
        n = z0.shape[0]
        n_global = n if n_global is None else n_global
        dt = c.total_time / c.n_steps
        flat = self.model.flat(self.params)
        drift_params = self.drift_params
        if c.drift_kind == L.DRIFT_MEANFIELD_TABLE:
            drift_params = self.meanfield_table(z0, seed, n_global, particle_offset)
        w_0T = 1.0 / (n_global * self.s_emit)
        w_b = 1.0 / n_global
        self.acc.begin()
        main = torch.cuda.current_stream(self.device)
        staged = not z0.is_cuda
        # Boundary sets (initial / terminal states): the terminal states of all chunks are collected (and, for a
        # host-resident ensemble, the staged initial states too) and each set is ONE launch over n points per step: the
        # per-launch set-up of the residual kernel (weight staging, TMEM allocation) is paid twice per step instead of
        # twice per chunk (2.2 % -> 0.8 % of the C5 step), and both residencies accumulate in the same order
        # (bit-identical results).
        batched_boundary = n > c.chunk
        if batched_boundary and (self.z_last_full is None or self.z_last_full.shape[0] != n):
            self.z_last_full = torch.empty((n, self.state), device=self.device, dtype=torch.float32)
        if batched_boundary and staged and (self.z0_full is None or self.z0_full.shape[0] != n):
            self.z0_full = torch.empty((n, self.state), device=self.device, dtype=torch.float32)
        set_0T, set_b = (L.SET_FP_0T, L.SET_FP_BOUNDARY) if self.overdamped else (L.SET_KFP_0T, L.SET_KFP_BOUNDARY)

        def prefetch(k: int):  # H2D of chunk k into staging buffer k % 2 on the copy stream
            a, b = k * c.chunk, min(n, (k + 1) * c.chunk)
            with torch.cuda.stream(self.copy_stream):
                self.copy_stream.wait_event(self.stage_free[k % 2])
                self.z_stage[k % 2][: b - a].copy_(z0[a:b], non_blocking=True)
                self.stage_ready[k % 2].record(self.copy_stream)

        if staged:
            for ev in self.stage_free:
                ev.record(main)  # whatever used the buffers before this step is ordered before the first copies
            prefetch(0)
        for k, lo in enumerate(range(0, n, c.chunk)):
            hi = min(n, lo + c.chunk)
            nc = hi - lo
            if not staged:
                zc = z0[lo:hi]
            else:
                if hi < n:
                    prefetch(k + 1)
                main.wait_event(self.stage_ready[k % 2])
                zc = self.z_stage[k % 2][:nc]
            # 128-point blocks of component planes when the chunk allows it (every store of an integrator step and
            # every load of a residual tile is base + constant), else component planes over the whole chunk
            blocked = nc % 128 == 0
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)] if phase_events is not None else None
            if ev:
                ev[0].record()
            traj_layout = L.TRAJ_BLOCK128 if blocked else L.TRAJ_TIME_SOA
            z_last_out = self.z_last_full[lo:hi] if batched_boundary else self.z_last[:nc]
            if self.overdamped:
                z_last, traj = ops.overdamped_integrate(
                    zc, c.n_steps, dt, c.drift_kind, drift_params, n_gaussian=c.n_gaussian, sigma=c.sigma, seed=seed,
                    particle_offset=particle_offset + lo, traj_layout=traj_layout, emit_every=c.emit_every,
                    emit_drift=True, path=c.path, traj_out=self.traj, x_last_out=z_last_out)
            else:
                z_last, traj, _ = ops.kl_integrate(
                    zc, c.n_steps, dt, c.gamma, c.drift_kind, drift_params, n_gaussian=c.n_gaussian, sigma=c.sigma,
                    seed=seed, particle_offset=particle_offset + lo, traj_layout=traj_layout,
                    emit_every=c.emit_every, traj_out=self.traj, z_last_out=z_last_out, emit_drift=True, path=c.path)
            if ev:
                ev[1].record()
            coef_0T = 0.0 if self.overdamped else c.gamma
            if blocked:
                self.acc.accumulate(set_0T, flat, traj.view(self.s_emit * nc // 128, self.width, 128), w_0T,
                                    coef=coef_0T, layout=L.LAYOUT_BLOCK128, true_grad=self.true_in_points, path=c.path)
            else:
                self.acc.accumulate(set_0T, flat, traj.view(self.width, self.s_emit * nc), w_0T, coef=coef_0T,
                                    layout=L.LAYOUT_SOA, true_grad=self.true_in_points, path=c.path)
            if ev:
                ev[2].record()
                phase_events.append(ev)
            if not batched_boundary:
                self.acc.accumulate(set_b, flat, z_last, w_b, coef=2.0 / c.total_time, path=c.path)
                self.acc.accumulate(set_b, flat, zc, w_b, coef=-2.0 / c.total_time, path=c.path)
            if staged:
                if batched_boundary:
                    self.z0_full[lo:hi].copy_(zc, non_blocking=True)  # device-to-device, before the buffer is released
                self.stage_free[k % 2].record(main)
        if batched_boundary:
            self.acc.accumulate(set_b, flat, self.z_last_full, w_b, coef=2.0 / c.total_time, path=c.path)
            self.acc.accumulate(set_b, flat, self.z0_full if staged else z0, w_b, coef=-2.0 / c.total_time,
                                path=c.path)
        sums, grad = self.acc.finalize()
        shard = parallel.Shard.current()
        if shard.world > 1:
            sums_r, grad_r = parallel.allreduce_sum_packed([sums, grad])
            sums.copy_(sums_r)
            grad.copy_(grad_r)
            # the norm is not additive over ranks: recompute it from the reduced gradient (common_utils.py:74-76)
            sums[L.SUM_GRADNORM] = torch.linalg.vector_norm(grad)
        out = {"loss": sums[L.SUM_LOSS], "loss ground truth": sums[L.SUM_GT], "sums": sums, "grad": grad}
        if apply_optimizer and self.optimizer is not None:
            lr = self.optimizer.lr_schedule(self.opt_state.count)
            self.opt_state.count += 1
            ops.adam_l2_step(flat, grad, self.opt_state.m, self.opt_state.v, count=self.opt_state.count, lr=lr,
                             b1=self.optimizer.b1, b2=self.optimizer.b2, eps=self.optimizer.eps,
                             weight_decay=self.optimizer.weight_decay, norms=self.norms)
            out["grad_norm"] = self.norms[0]
            out["params_norm"] = self.norms[1]
        return out
