"""Times the overdamped integrator under a fitted MLP's potential (pdeip_overdamped_integrate_model, MLP 32 x 2) on
PDEIP_PATH_FP32 and PDEIP_PATH_TENSOR, alternating the two paths in one process, for d in {8, 16, 32} and two modes:

  terminal  traj = NULL: only the terminal state (compute-bound);
  block128  every sample emitted as [x, grad V_theta(x)] in PDEIP_TRAJ_BLOCK128, the FP residual's point set.  The
            particles run in chunks of --chunk with consecutive particle_offsets (the whole trajectory of 2^22 particles
            is 215 GB at d = 32).

CUDA events around whole calls after one warm-up call per configuration.  Prints particle-steps/s, algorithmic FLOP/s at
4 M1 FLOP per drift evaluation (M1 = dH + H^2 + 40H: the primal chain and the input-gradient chain), written bytes per
second in the emitting mode (2d * 4 B per emitted particle-step), and the device name and power limit read in the same
run.

usage: python tools/overdamped_time.py [--n 4194304] [--steps 200] [--reps 2] [--chunk 262144] [--dims 8,16,32]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pde_inverse_problem_b200 import _lib as L, ops  # noqa: E402
from pde_inverse_problem_b200.core.model import V_hypothesis  # noqa: E402

H = 32


def power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 22)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--chunk", type=int, default=1 << 18)
    ap.add_argument("--dims", default="8,16,32")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("overdamped_time.py needs a CUDA device")
    dev = torch.device("cuda")
    n, S = args.n, args.steps
    chunk = min(args.chunk, n)
    assert n % chunk == 0 and chunk % 128 == 0
    print(f"device {torch.cuda.get_device_name(0)}, power limit {power_limit()}; overdamped, MLP {H} x 2, n = {n}, "
          f"S = {S}, block128 chunk = {chunk}, {args.reps} timed calls after 1 warm-up")
    for d in (int(x) for x in args.dims.split(",")):
        net = V_hypothesis(output_dim=1, hidden_dims=[H, H], dim=d)
        flat = net.init(11, torch.zeros(d, device=dev))["_flat"]
        x0 = torch.randn(n, d, device=dev)
        flop = 4 * (d * H + H * H + 40 * H)

        def run(mode, path):
            if mode == "terminal":
                ops.overdamped_integrate_model(x0, S, 0.01, net.spec, flat, seed=1, want_traj=False, path=path)
                return
            for c0 in range(0, n, chunk):
                ops.overdamped_integrate_model(x0[c0:c0 + chunk], S, 0.01, net.spec, flat, seed=1, particle_offset=c0,
                                               traj_layout=L.TRAJ_BLOCK128, emit_drift=True, path=path)

        for mode in ("terminal", "block128"):
            ms = {L.PATH_FP32: [], L.PATH_TENSOR: []}
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
            evals = S + (1 if mode == "block128" else 0)  # the last sample's drift takes one more evaluation
            for path, t in ms.items():
                best = min(t)
                ps = n * S / best * 1e3
                line = (f"d={d:2d} {mode:8s} {'tensor' if path else 'fp32':6s}: {best:9.2f} ms (calls: "
                        f"{', '.join(f'{x:.2f}' for x in t)})  {ps:.3e} particle-steps/s  "
                        f"{n * evals * flop / best / 1e9:7.2f} TFLOP/s")
                if mode == "block128":
                    line += f"  {n * S * 2 * d * 4 / best / 1e6:7.1f} GB/s written"
                print(line + f"  status={status}", flush=True)


if __name__ == "__main__":
    main()
