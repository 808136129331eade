"""Times the Fokker-Planck GMM hot path on PDEIP_PATH_FP32 and PDEIP_PATH_TENSOR, alternating the two paths in one
process:

  (a) the overdamped GMM integrator (pdeip_overdamped_integrate, PDEIP_DRIFT_GMM, sigma = 1) at (d, K) = (8, 16),
      (16, 32), (32, 64), n = 2^22, S = 200, in two modes:
        terminal  traj = NULL: only the terminal state;
        block128  every sample emitted as [x, grad U(x)] in PDEIP_TRAJ_BLOCK128 (the FP 0T point set), the particles
                  in chunks of --chunk with consecutive particle_offsets (the whole trajectory is 215 GB at d = 32).
      CUDA events around whole calls after one warm-up call per configuration; particle-steps/s and bytes written per
      second in the emitting mode (2d * 4 B per emitted particle-step).
  (b) one overdamped pipeline.HotPath step (MLP 32 x 2, no optimizer update) at (d, K) = (8, 16) and (32, 64), split
      with phase_events into the integrator, the FP 0T residual and the rest (boundary sets, finalize).

The device name and power limit are read in the same run.  Output: stdout and --out.

usage: python tools/fp_gmm_time.py [--out profiles/r03_fp_gmm_time.txt] [--n 4194304] [--steps 200] [--reps 2]
                                   [--chunk 262144] [--hp-n 1048576] [--hp-steps 100]
"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pde_inverse_problem_b200 import _lib as L, ops  # noqa: E402
from pde_inverse_problem_b200.core.model import V_hypothesis  # noqa: E402
from pde_inverse_problem_b200.pipeline import HotPath, HotPathConfig  # noqa: E402

PATHS = {"fp32": L.PATH_FP32, "tensor": L.PATH_TENSOR}


def power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def centres(d, K, dev):
    g = torch.Generator().manual_seed(1000 * d + K)
    return (torch.rand(K, d, generator=g) * 8.0 - 4.0).to(dev).contiguous()


def integrator(args, say, dev):
    n, S, chunk = args.n, args.steps, min(args.chunk, args.n)
    assert n % chunk == 0 and chunk % 128 == 0
    say(f"(a) overdamped GMM integrator, n = {n}, S = {S}, dt = 0.01, block128 chunk = {chunk}, {args.reps} timed "
        f"calls after 1 warm-up")
    for d, K in ((8, 16), (16, 32), (32, 64)):
        mus = centres(d, K, dev)
        x0 = 2.0 * torch.randn(n, d, device=dev)

        def run(mode, path):
            if mode == "terminal":
                ops.overdamped_integrate(x0, S, 0.01, L.DRIFT_GMM, mus, n_gaussian=K, seed=1, want_traj=False,
                                         path=path)
                return
            for c0 in range(0, n, chunk):
                ops.overdamped_integrate(x0[c0:c0 + chunk], S, 0.01, L.DRIFT_GMM, mus, n_gaussian=K, seed=1,
                                         particle_offset=c0, traj_layout=L.TRAJ_BLOCK128, emit_drift=True, path=path)

        for mode in ("terminal", "block128"):
            ms = {p: [] for p in PATHS.values()}
            for path in ms:
                run(mode, path)
            torch.cuda.synchronize()
            for _ in range(args.reps):
                for path in ms:  # alternate the two paths
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    run(mode, path)
                    e1.record()
                    torch.cuda.synchronize()
                    ms[path].append(e0.elapsed_time(e1))
            status = ops.tensor_path_status()
            for path, t in ms.items():
                best = min(t)
                line = (f"d={d:2d} K={K:2d} {mode:8s} {'tensor' if path else 'fp32':6s}: {best:9.2f} ms (calls: "
                        f"{', '.join(f'{x:.2f}' for x in t)})  {n * S / best * 1e3:.3e} particle-steps/s")
                if mode == "block128":
                    line += f"  {n * S * 2 * d * 4 / best / 1e6:7.1f} GB/s written"
                say(line + f"  status={status}")


def hot_path(args, say, dev):
    n, S = args.hp_n, args.hp_steps
    say(f"(b) one overdamped HotPath step (MLP 32 x 2, T = 2, no optimizer update), n = {n}, S = {S}, auto chunk; "
        f"best of {args.reps} after 1 warm-up")
    for d, K in ((8, 16), (32, 64)):
        mus = centres(d, K, dev)
        model = V_hypothesis(1, [32, 32], d)
        params = model.init(11, torch.zeros(d, device=dev))
        x0 = 2.0 * torch.randn(n, d, device=dev)
        hps = {}
        for name, path in PATHS.items():
            cfg = HotPathConfig(d=d, n_steps=S, total_time=2.0, gamma=0.0, drift_kind=L.DRIFT_GMM, n_gaussian=K,
                                path=path, dynamics="overdamped")
            hps[name] = HotPath(cfg, model, params, mus, ops.TrueGrad(L.DRIFT_IN_POINTS), device=dev)
            hps[name].step(x0, seed=5, apply_optimizer=False)
        torch.cuda.synchronize()
        res = {name: [] for name in PATHS}
        for _ in range(args.reps):
            for name, hp in hps.items():
                ev = []
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                hp.step(x0, seed=5, apply_optimizer=False, phase_events=ev)
                e1.record()
                torch.cuda.synchronize()
                total = e0.elapsed_time(e1)
                t_int = sum(e[0].elapsed_time(e[1]) for e in ev)
                t_res = sum(e[1].elapsed_time(e[2]) for e in ev)
                res[name].append((total, t_int, t_res, len(ev)))
        status = ops.tensor_path_status()
        for name, r in res.items():
            total, t_int, t_res, chunks = min(r)
            say(f"d={d:2d} K={K:2d} {name:6s}: step {total:9.2f} ms = integrator {t_int:9.2f} + 0T residual "
                f"{t_res:9.2f} + rest {total - t_int - t_res:7.2f} ms  ({chunks} chunks of {hps[name].cfg.chunk}, "
                f"{hps[name].particle_steps(n) / total * 1e3:.3e} particle-steps/s)  status={status}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_fp_gmm_time.txt"))
    ap.add_argument("--n", type=int, default=1 << 22)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--chunk", type=int, default=1 << 18)
    ap.add_argument("--hp-n", type=int, default=1 << 20)
    ap.add_argument("--hp-steps", type=int, default=100)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fp_gmm_time.py needs a CUDA device")
    dev = torch.device("cuda")
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say("# tools/fp_gmm_time.py: K1-OD under the GMM potential, fp32 kernel (kl_integrate_kernel<DP, GMM, 0, true>) "
        "against K1-T-OD (kl_integrate_tc*_kernel<..., OD = true>), and the overdamped HotPath step")
    say(f"device {torch.cuda.get_device_name(0)}, power limit {power_limit()}")
    integrator(args, say, dev)
    hot_path(args, say, dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
