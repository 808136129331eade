#!/usr/bin/env python
"""bench.py — throughput of the particle-ensemble hot path on B200 (see DESIGN.md §Measurement).

One "step" = one pass of the hot path over one synthetic ensemble: K1 integrates every particle for S+1
kinetic-Langevin steps (in-register Philox noise, GMM / OU drift) emitting S trajectory samples, the residual
kernel evaluates loss terms + parameter gradient at every emitted sample (0T set) and at the initial /
terminal states (boundary sets), [all-reduce over ranks], and K6 applies Adam+L2.

  metric  particle-steps/s = (particles over all ranks) * (S+1) / step time    (BASELINE.json)
  also    residual evals/s = (particles over all ranks) * S_emit / step time
  value   inputs resident in HBM;   e2e: ensemble in pinned host memory, H2D per chunk and D2H of the loss
          inside the timed region.

Default workload: C5 (BASELINE.json configs[4], the north-star's scaling target): KGMM d=32, K=64, S=200 with
2^24 particles IN TOTAL, n = 2^24 / world per rank -> "scaling": "strong".  The C3 step (configs[2], 2^22 particles per
rank) is measured in the same run and reported as `extra.c3`.  C2 / C3 / C4 as --workload keep a fixed ensemble per
rank ("weak").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C2|C3|C4|C4mf|C5] [--path fp32|tensor]
                    [--dump-outputs DIR]
    python bench.py --impl reference ...     # CPU restatement of the reference (oracle port) on host cores

--dump-outputs DIR writes what the last timed step of the headline workload returned (loss, loss ground truth, the
residual sums, the parameter gradient, its norm, the parameter norm) and the parameters it left behind, one float32
DIR/<name>.npy each.  Inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# d, K (n_gaussian; 0 = linear OU drift), per-rank particles, S, T, gamma, chunk
WORKLOADS = {
    "C2": dict(name="KOU d=4 N=2^20 S=100 (kinetic OU, scripts/run_KOU.sh)", d=4, K=0, n=1 << 20, S=100, T=2.0,
               gamma=1.0, chunk=1 << 19),
    "C3": dict(name="KGMM d=8 K=16 N=2^22 S=200 (scripts/run_KGMM.sh)", d=8, K=16, n=1 << 22, S=200, T=2.0,
               gamma=0.5, chunk=303104),  # two whole waves of the tcgen05 integrator grid (148 SMs x 8 CTAs x 128 particles)
    "C4": dict(name="KMV-quadratic (-A x drift) d=16 N=2^22 S=100", d=16, K=0, n=1 << 22, S=100, T=2.0,
               gamma=1.0, chunk=1 << 18),
    "C4mf": dict(name="KMV interacting system d=16 N=2^22 S=100: drift A (x - xbar_t), xbar_t the empirical mean of ALL "
                      "ranks' particles (README.md:54-62); one noise pre-pass + ONE all-reduce per iteration",
                 d=16, K=0, n=1 << 22, S=100, T=2.0, gamma=1.0, chunk=1 << 18, meanfield=True),
    "C5": dict(name="KGMM d=32 K=64 N=2^24 total S=200, sharded over the ranks", d=32, K=64, n_total=1 << 24, S=200,
               T=2.0, gamma=0.5, chunk=56832),  # 148 SMs x 3 CTAs x 128 particles: one full wave of the tcgen05 integrator
}
HIDDEN, LAYERS, OUT = 32, 2, 40


def m1(d):
    return d * HIDDEN + HIDDEN * HIDDEN + OUT * HIDDEN


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            j = json.load(fh)
        return dict(hbm=j["hbm_gbs"], tf_burst=j["bf16_tflops"], tf_sust=j["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


def measured_traffic(kernel_key):
    """DRAM bytes per residual point of the dominant kernel from the committed ncu --set full capture
    (profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum / points of the captured launch)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(p) as fh:
            ent = json.load(fh).get(kernel_key)
    except (OSError, ValueError):
        ent = None
    if not ent:
        return None, "no ncu --set full capture of %s in profiles/traffic.json" % kernel_key
    return float(ent["dram_bytes_per_point"]), "profiles/traffic.json[%s] <- %s" % (kernel_key, ent["source"])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                     f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            busy = [s for s in sm if s > 0.5 * max(sm)] or sm
            out.update(sm_mhz=statistics.median(busy), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def build_problem(w, device, seed=1):
    """Synthetic problem of the named workload: centres / drift matrix, MLP, initial ensemble law."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    from pde_inverse_problem_b200.core.model import V_hypothesis
    from pde_inverse_problem_b200.core.optimizer import AdamL2, cosine_decay_schedule
    d, K = w["d"], w["K"]
    g = torch.Generator().manual_seed(seed)
    if K > 0:   # GMM.py:17-42: mu ~ U[-4,4]^d, x0 ~ N(0, 4I), v0 ~ N(0, 0.1 I), gamma = 0.5
        drift = (torch.rand(K, d, generator=g) * 8 - 4).to(device)
        drift_kind = L.DRIFT_GMM
        true = ops.TrueGrad(L.DRIFT_GMM, drift, 1.0)
        cov_half = torch.diag(torch.cat([torch.full((d,), 2.0), torch.full((d,), math.sqrt(0.1))])).to(device)
    else:       # OU.py:15-43: tilde_F = _F _F^T (scaled by 1/d so that dt*lambda_max stays stable at every d)
        _F = torch.randn(d, d + 1, generator=g, dtype=torch.float64)
        drift = ((_F @ _F.T) / d).float().to(device)
        drift_kind = L.DRIFT_MEANFIELD_TABLE if w.get("meanfield") else L.DRIFT_LINEAR
        true = ops.TrueGrad(L.DRIFT_LINEAR, drift)
        cov_half = None
    if w.get("model") == "parametric":  # what the reference's launch scripts train by default (config.yaml:40)
        from pde_inverse_problem_b200.core.model import V_parametric_GMM, V_parametric_quadratic
        model = V_parametric_GMM(d, K) if K > 0 else V_parametric_quadratic(d)
    else:
        model = V_hypothesis(1, [HIDDEN] * LAYERS, d)
    params = model.init(11, torch.zeros(d, device=device))
    opt = AdamL2(cosine_decay_schedule(1e-2, 20000, 0.001), 1e-3)
    return drift_kind, drift, true, cov_half, model, params, opt


def dump_outputs(out_dir, out, params):
    """The outputs of one hot-path step as out_dir/<name>.npy (float32): every tensor of the step's result dict and the
    flat parameter vector after its optimizer update.  Copied to the host at once: later steps reuse these buffers."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = dict(out, params=params)
    for key, t in arrays.items():
        np.save(os.path.join(out_dir, key.replace(" ", "_") + ".npy"), t.detach().float().cpu().numpy())


def measure(name, args, shard, device, local_rank, steps, warmup, with_clocks, dump_dir=None):
    """Warm-up + timed steps + e2e + per-kernel phases of one workload on this rank; returns the result dict (rank 0)
    after the max-over-ranks reduction of the times.  dump_dir: where rank 0 writes the outputs of the last timed step."""
    from pde_inverse_problem_b200 import _lib as L
    from pde_inverse_problem_b200 import ops
    from pde_inverse_problem_b200.pipeline import HotPath, HotPathConfig
    import torch.distributed as dist

    w = dict(WORKLOADS[name])
    w["model"] = args.model
    strong = "n_total" in w and not args.particles
    if args.particles:
        w["n"] = args.particles
    elif strong:
        assert w["n_total"] % shard.world == 0
        w["n"] = w["n_total"] // shard.world
    d, K, n, S = w["d"], w["K"], w["n"], w["S"]
    n_global = n * shard.world
    path = L.PATH_TENSOR if args.path == "tensor" else L.PATH_FP32
    drift_kind, drift, true, cov_half, model, params, opt = build_problem(w, device)
    cfg = HotPathConfig(d=d, n_steps=S, total_time=w["T"], gamma=w["gamma"], drift_kind=drift_kind,
                        n_gaussian=K, chunk=min(w["chunk"], n), path=path)
    hp = HotPath(cfg, model, params, drift, true, optimizer=opt, device=device)
    offset = shard.rank * n
    z0 = ops.gaussian_sample(n, 2 * d, None, cov_half, seed=7, particle_offset=offset, device=device)

    def barrier():
        if shard.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- phase timing helpers (events on torch's current stream, the stream the kernels launch on) --------
    def timed_phases(seed):
        """One more step of the same pipeline with CUDA events around the integrator and 0T-residual launches of
        every chunk (no optimizer update: the parameters of the timed steps are not touched)."""
        ev = []
        hp.step(z0, seed=seed, n_global=n_global, particle_offset=offset, apply_optimizer=False, phase_events=ev)
        torch.cuda.synchronize()
        t_int = sum(e[0].elapsed_time(e[1]) for e in ev) / 1e3
        t_res = sum(e[1].elapsed_time(e[2]) for e in ev) / 1e3
        return t_int, t_res, len(ev)

    # ---- warm-up ---------------------------------------------------------------------------------------
    for i in range(warmup):
        hp.step(z0, seed=100 + i, n_global=n_global, particle_offset=offset)
    barrier()

    # ---- timed region: EXACTLY K steps, inputs resident in HBM ---------------------------------------------
    sampler = ClockSampler(local_rank) if with_clocks else None
    if sampler:
        sampler.start()
    ops.launch_counter["n"] = 0
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        out = hp.step(z0, seed=1000 + i, n_global=n_global, particle_offset=offset)
    e1.record()
    barrier()
    launches = ops.launch_counter["n"]
    clocks = sampler.stop() if sampler else None
    t_dev = e0.elapsed_time(e1) / 1e3
    loss = float(out["loss"])
    assert math.isfinite(loss), "loss is not finite (a timed-out tcgen05 phase poisons it with NaN)"
    if dump_dir is not None and shard.rank == 0:
        dump_outputs(dump_dir, out, model.flat(params))

    # ---- e2e: ensemble in pinned host memory, H2D per chunk + D2H of the loss inside the timed region ----
    z0_host = torch.empty((n, 2 * d), dtype=torch.float32, pin_memory=True)
    z0_host.copy_(z0)
    result_host = torch.empty(2, dtype=torch.float32, pin_memory=True)
    hp.step(z0_host, seed=50, n_global=n_global, particle_offset=offset)  # warm the staging path
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(steps):
        o = hp.step(z0_host, seed=2000 + i, n_global=n_global, particle_offset=offset)
        result_host[0].copy_(o["loss"], non_blocking=True)
        result_host[1].copy_(o["grad_norm"], non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the caller reads the loss every iteration (trainer.py:112)
    f1.record()
    barrier()
    t_e2e = f0.elapsed_time(f1) / 1e3
    del z0_host

    # ---- per-kernel phases (separate pass, after the headline timing) ---------------------------------------
    t_int, t_res, n_chunks = timed_phases(seed=3000)

    # max over ranks
    times = torch.tensor([t_dev, t_e2e, t_int, t_res], device=device, dtype=torch.float64)
    if shard.world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    t_dev, t_e2e, t_int, t_res = [float(x) for x in times]
    del hp, z0
    torch.cuda.empty_cache()
    if shard.rank != 0:
        return None

    pk = peaks()
    psteps = n_global * (S + 1)
    s_emit = S
    evals = n_global * s_emit
    # dominant kernel = residual (tensor-pipe roofline, algorithmic 24*M1 FLOP per eval, SURVEY.md §8d)
    flop_eval = 24 * m1(d)
    res_rate = n * s_emit / t_res  # per GPU
    res_tflops = res_rate * flop_eval / 1e12
    dp, ns = (8, 2) if d <= 8 else ((16, 1) if d <= 16 else (32, 1))
    tensor_int = path == L.PATH_TENSOR and K > 0 and d in (8, 16, 32) and K <= 64
    parametric = args.model == "parametric"
    if parametric:  # closed-form model (K5): ~12 K d FLOP per eval, bound by the 3d*4 B it reads per point
        res_kernel = "gmm_param_residual_kernel (fp32, closed form)" if K > 0 else "quad_param_residual_kernel (fp32, closed form)"
        per_point, res_traffic_src = None, "not captured for the parametric kernels"
    elif path == L.PATH_TENSOR:
        res_kernel = "tc::mlp_residual_tc_kernel<%d,%d> (KFP 0T set, tcgen05)" % (dp, ns)
        per_point, res_traffic_src = measured_traffic("mlp_residual_tc<%d,%d>" % (dp, ns))
    else:
        res_kernel = "mlp_residual_kernel<32,2,KFP_0T,8> (fp32)"
        per_point, res_traffic_src = measured_traffic("mlp_residual_fp32")
    pts_launch = cfg.chunk * s_emit
    res_traffic = per_point * pts_launch if per_point is not None else None
    int_rate = n * (S + 1) / t_int
    int_written = n * s_emit * 3 * d * 4 / t_int / 1e9   # [x, v, grad U(x)] per emitted sample: the bytes really written
    int_alg = n * s_emit * 2 * d * 4 / t_int / 1e9       # SURVEY.md §8(d): 2d*4 B per emitted particle-step ([x, v])
    return {
        "metric": "particle-steps/s", "value": psteps * steps / t_dev, "unit": "particle-steps/s", "n_gpus": shard.world,
        "steps": steps, "warmup": warmup, "ms_per_step": t_dev / steps * 1e3, "higher_is_better": True,
        "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "f32" if path == L.PATH_FP32 else ("bf16 GEMM operands split hi+lo (MLP weights and x; GMM centres, x and softmax weights "
                                                  "in the integrator), f32 accumulate / epilogue / state"),
        "data": "synthetic",
        "config": {"workload": f"{name}: {w['name']}", "particles_per_rank": n, "particles_total": n_global,
                   "d": d, "n_gaussian": K, "n_steps": S,
                   "mlp": ("parametric model (closed-form residual)" if parametric else f"{d}->{HIDDEN}x{LAYERS}->{OUT}"),
                   "chunk": cfg.chunk, "residual_path": args.path,
                   "l2_policy": "inputs larger than L2: every chunk's trajectory (%.1f GB) streams through HBM"
                                % (3 * d * s_emit * cfg.chunk * 4 / 1e9)},
        "residual_evals_per_s": evals * steps / t_dev,
        "loss": loss,
        "e2e": {"value": psteps * steps / t_e2e, "unit": "particle-steps/s",
                "h2d_bytes_per_step": n * 2 * d * 4, "d2h_bytes_per_step": 8, "ms_per_step": t_e2e / steps * 1e3},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": ({"kernel": res_kernel, "bound": "hbm", "achieved": res_rate * 3 * d * 4 / 1e9, "peak": pk["hbm"],
                      "unit": "GB/s", "frac": res_rate * 3 * d * 4 / 1e9 / pk["hbm"], "traffic": None,
                      "traffic_source": res_traffic_src, "peak_source": pk["src"] + " copy bandwidth",
                      "evals_per_s_per_gpu": res_rate, "bytes_per_eval": 3 * d * 4} if parametric else
                     {"kernel": res_kernel, "bound": "tensor", "achieved": res_tflops,
                      "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": res_tflops / pk["tf_sust"],
                      "traffic": res_traffic, "traffic_source": res_traffic_src,
                      "peak_source": pk["src"] + " bf16 sustained",
                      "evals_per_s_per_gpu": res_rate, "flop_per_eval": flop_eval,
                      "frac_of_step": (n * s_emit * flop_eval / (t_dev / steps) / 1e12) / pk["tf_sust"]}),
        "kernels": {
            "kl_integrate": {"kernel": ("kl_integrate_tc_kernel (GMM contraction on tcgen05)" if tensor_int
                                        else "kl_integrate_fast_kernel (fp32)"), "bound": "hbm",
                             "achieved": int_written, "peak": pk["hbm"], "unit": "GB/s", "frac": int_written / pk["hbm"],
                             "bytes_per_emitted_step": 3 * d * 4,
                             "achieved_algorithmic": int_alg, "frac_algorithmic": int_alg / pk["hbm"],
                             "algorithmic_bytes_per_emitted_step": 2 * d * 4,
                             "particle_steps_per_s_per_gpu": int_rate, "ms_per_step": t_int * 1e3},
            "mlp_residual": {"ms_per_step": t_res * 1e3, "evals_per_s_per_gpu": res_rate},
        },
    }


def run_ours(args):
    from pde_inverse_problem_b200 import parallel
    import torch.distributed as dist

    shard = parallel.init_from_env("nccl")
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    line = measure(args.workload, args, shard, device, local_rank, args.steps, args.warmup, with_clocks=True,
                   dump_dir=args.dump_outputs)
    extra = None
    if args.workload == "C5" and not args.particles and not args.no_extra:
        # the C3 step (BASELINE.json configs[2], 2^22 particles per rank) in the same run
        c3 = measure("C3", args, shard, device, local_rank, args.steps, args.warmup, with_clocks=False)
        if c3 is not None:
            extra = {k: c3[k] for k in ("value", "unit", "ms_per_step", "scaling", "config", "residual_evals_per_s", "e2e",
                                        "roofline", "kernels", "steps", "warmup")}
    if shard.rank == 0:
        if extra is not None:
            line["extra"] = {"c3": extra}
        if not args.no_cpu_baseline and shard.world == 1:
            line["cpu_baseline"] = cpu_baseline(dict(WORKLOADS[args.workload]), seconds_hint=15.0)
        emit_result(line)
    if shard.world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (torch.func restatement of the reference), float32, all host threads
# ---------------------------------------------------------------------------------------------------------
def oracle_step(w, n_s, seed=0):
    """One hot-path step of the oracle on n_s particles: integrate S+1 steps, residual value+grad over the
    S*n_s trajectory points + boundary sets.  Returns seconds."""
    from oracle import integrator as o_int, model as o_model, potential as o_pot, residuals as o_res, problems as o_prob
    d, K, S = w["d"], w["K"], w["S"]
    g = torch.Generator().manual_seed(seed)
    dt = w["T"] / S
    if K > 0:
        pde = o_prob.KineticGMMProblem(d, K, T=w["T"], dtype=torch.float32)
        grad_fn = o_pot.GMMPotential(pde.mus, 1.0).gradient
    else:
        pde = o_prob.KineticOUProblem(d, T=w["T"], dtype=torch.float32)
        pde.initial_configuration["tilde_F"] = pde.initial_configuration["tilde_F"] / d
        grad_fn = o_pot.LinearDrift(pde.initial_configuration["tilde_F"], mean_field=bool(w.get("meanfield"))).gradient
    pde.initial_configuration["gamma_friction"] = w["gamma"]
    params = o_model.init_mlp_params(d, HIDDEN, LAYERS, dtype=torch.float32)
    z0 = torch.randn(n_s, 2 * d, generator=g)
    noise = torch.randn(n_s, S + 1, d, generator=g)
    tau0 = torch.rand(n_s, generator=g) * dt
    t0 = time.perf_counter()
    last, traj, _ = o_int.underdamped_langevin_dynamics_scan(z0, S, dt, noise, tau0, grad_fn, w["gamma"])
    data = {"initial": z0, "terminal": last, "0T": traj.reshape(-1, 2 * d)}
    out = o_res.kfp_value_and_grad_fn(o_model.mlp_apply, params, data, pde, chunk=8192)
    float(out["loss"])
    return time.perf_counter() - t0


def cpu_baseline(w, seconds_hint=15.0):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n_s = 64
    t = oracle_step(w, n_s)          # warm-up (torch.func tracing caches)
    t = oracle_step(w, n_s, seed=1)
    # scale the sample towards ~seconds_hint of CPU work, bounded
    n_big = int(min(4096, max(64, n_s * seconds_hint / max(t, 1e-3))))
    t_big = oracle_step(w, n_big, seed=2)
    psteps = n_big * (w["S"] + 1)
    return {"value": psteps / t_big, "unit": "particle-steps/s", "cores": cores, "kind": "port",
            "sample": f"{n_big} particles x (S+1={w['S'] + 1} steps + {w['S']} residual evals each), float32, "
                      f"torch.func autodiff restatement of the reference (JAX not installable), {t_big:.1f} s",
            "residual_evals_per_s": n_big * w["S"] / t_big}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = dict(WORKLOADS[args.workload])
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n_s = 256 if w["d"] <= 8 else 128
    for _ in range(max(1, args.warmup)):
        oracle_step(w, 64)
    times = [oracle_step(w, n_s, seed=10 + i) for i in range(args.steps)]
    t = sum(times)
    psteps = n_s * (w["S"] + 1) * args.steps
    value = psteps / t
    sample = (f"{n_s} particles per step x (S+1={w['S'] + 1} integrator steps + {w['S']} residual evals each), float32, "
              f"oracle port (torch.func restatement; the JAX reference is not installable here)")
    line = {"impl": "reference", "metric": "particle-steps/s", "value": value, "unit": "particle-steps/s",
            "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t / args.steps * 1e3, "higher_is_better": True,
            "scaling": "strong" if "n_total" in w else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {w['name']}", "sample_particles": n_s, "d": w["d"],
                       "n_gaussian": w["K"], "n_steps": w["S"], "mlp": f"{w['d']}->{HIDDEN}x{LAYERS}->{OUT}"},
            "residual_evals_per_s": n_s * w["S"] * args.steps / t,
            "cpu_baseline": {"value": value, "unit": "particle-steps/s", "cores": cores, "kind": "port",
                             "sample": sample},
            "e2e": {"value": value, "unit": "particle-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit_result(line)


_RESULT_OUT = None


def emit_result(line: dict) -> None:
    """The ONE JSON line of the run, on the process's original stdout."""
    out = _RESULT_OUT if _RESULT_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    # stdout carries exactly one JSON line.  Libraries write there too (NCCL prints its version banner from C with
    # NCCL_DEBUG=VERSION, whatever NCCL_DEBUG_FILE says at 8 ranks), so file descriptor 1 is pointed at stderr for the
    # whole run and the result goes to a private duplicate of the original stdout.
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C5", choices=sorted(WORKLOADS))
    ap.add_argument("--no-extra", action="store_true", help="skip the extra.c3 block of the default C5 run")
    ap.add_argument("--model", default="mlp", choices=["mlp", "parametric"],
                    help="hypothesis model: mlp = V_hypothesis d->32x2->40 (BASELINE metric), parametric = the closed-form "
                         "GMM / quadratic model the reference's launch scripts train by default (config.yaml:40)")
    ap.add_argument("--path", default=os.environ.get("PDEIP_BENCH_PATH", "tensor"), choices=["fp32", "tensor"],
                    help="residual kernel: tensor = tcgen05 bf16 GEMM path (rtol 1e-2, default), fp32 = CUDA-core parity path (rtol 1e-5)")
    ap.add_argument("--particles", type=int, default=0, help="override particles per rank")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: W >= 3
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
        run_ours(args)


if __name__ == "__main__":
    main()
