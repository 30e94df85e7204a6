"""Times the all-outputs device evaluation (residuals, Jacobian, gradient, cost; state resident in
HBM, cb200_engine_evaluate_device) of a BAL-shaped problem once per robust loss, with Huber as the
control, measured first and again last to show the drift of the machine over the run.

    python scripts/bench_losses.py --shape L --steps 20 --warmup 5

Per loss: the kernel time and the device time of a step (CUDA events on the engine's stream, mean
over --steps back-to-back evaluations after --warmup), and the ratio to the first Huber run.  The
GPU's name and power limit are read in the same run.  Writes one JSON file (--out) and prints it."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ceres_b200 import binding as B, problems as P  # noqa: E402

LOSSES = ["huber", "soft_l1", "arctan", "tolerant", "tukey", "cauchy", "huber"]


def gpu_info():
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_losses.py needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return {"torch_device_name": torch.cuda.get_device_name(0),
            "nvidia_smi_name_power_limit_max_sm_clock": q.stdout.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="L")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join("profiles", "r4_bench_losses_L.json"))
    args = ap.parse_args()
    info = gpu_info()
    spec = P.bal_shape(args.shape, args.scale)
    runs = []
    for name in LOSSES:
        kind, a, b = P.LOSS_BY_NAME[name]
        spec.rb_loss_kind[:], spec.rb_loss_a[:], spec.rb_loss_b[:] = kind, a, b
        t0 = time.perf_counter()
        cp = B.CudaProblem(spec, jacobian_format=0)
        setup_s = time.perf_counter() - t0
        ok, cost, *_ = cp.evaluate(cp.initial_state(), residuals=False, gradient=False,
                                   jacobian=False)  # uploads the state
        assert ok
        ok, _, _, _ = cp.evaluate_device_steps(args.warmup)
        assert ok
        ok, cost, kernel_ms, device_ms = cp.evaluate_device_steps(args.steps)
        assert ok
        runs.append({"loss": name, "kind": kind, "a": a, "b": b, "cost": cost,
                     "kernel_ms_mean": float(np.mean(kernel_ms)),
                     "kernel_ms_min": float(np.min(kernel_ms)),
                     "kernel_ms_max": float(np.max(kernel_ms)),
                     "device_ms_mean": float(np.mean(device_ms)), "setup_s": setup_s})
        cp.close()
        print(json.dumps(runs[-1]), file=sys.stderr)
    control = runs[0]["kernel_ms_mean"]
    for r in runs:
        r["kernel_ms_over_huber"] = r["kernel_ms_mean"] / control
    result = {
        "workload": f"synthetic BAL shape {args.shape} x {args.scale} ({spec.num_rb} residual "
                    "blocks), SnavelyReprojectionError<2,9,3>, BlockSparse, all outputs, state "
                    "in HBM",
        "steps": args.steps, "warmup": args.warmup, "gpu": info, "runs": runs,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
