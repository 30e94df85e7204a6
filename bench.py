#!/usr/bin/env python
"""Headline benchmark: residual blocks evaluated per second (residuals + Jacobian +
loss + gradient + cost) on a synthetic BAL problem of problem-13682-4456117 shape,
residual blocks sharded over --gpus B200s (BASELINE.json).

  python bench.py --gpus 1 --steps 20 --warmup 3
  python -m torch.distributed.run --nproc-per-node 8 ... bench.py --gpus 8 ...
  python bench.py --impl reference          # the reference algorithm on the host cores

A step is one Evaluator::Evaluate(state, &cost, residuals, gradient, jacobian) over
the whole problem.  `value` is measured with the state resident in HBM
(cb200_engine_evaluate_device); `e2e` goes through Evaluator::Evaluate with host
buffers, host<->device copies inside the timed region.  One JSON line on stdout.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT]

import numpy as np  # noqa: E402

# Workloads = BASELINE.json configs.  ALGORITHMIC bytes per residual block as derived in
# SURVEY.md section 8(d) / DESIGN.md "Roofline"; dense-Jet FLOP counts of the reference
# arithmetic from oracle/count_flops.cc.
#   BAL <2,9,3>, BlockSparse, all outputs: functor 16 + block ids 8 + cell positions 8 +
#     Jacobian 192 + residuals 16 + parameters and gradient amortised 2 x 3.7 = 248
#   L4 (SubsetManifold(9,{0}) cameras, CompressedRow): Jacobian 2 x 11 x 8 = 176 -> 236
#   P5 (pose graph <6,7,7>, EigenQuaternion x R^3): Jacobian 6 x 12 x 8 = 576 + residuals 48 +
#     functor 56 + ids/positions 16 + amortised state/gradient -> 700
WORKLOADS = {
    "S": dict(kind="bal", shape="S", fmt=0, bytes=248.0, flops=1763.0),
    "M": dict(kind="bal", shape="M", fmt=0, bytes=248.0, flops=1763.0),
    "L": dict(kind="bal", shape="L", fmt=0, bytes=248.0, flops=1763.0),
    "L4": dict(kind="bal", shape="L", fmt=1, bytes=236.0, flops=None, subset_manifold=True),
    "P5": dict(kind="pose", poses=2_500_000, edges=10_000_000, fmt=0, bytes=700.0, flops=None),
}
KERNEL_NAMES = {
    "bal": "EvaluateKernel<plain all-outputs, affine tables, SnavelyReprojectionError, HuberLossCUDA, 2, 9, 3>",
    "bal_subset": "EvaluateKernel<generic all-outputs, affine tables, SnavelyReprojectionError, HuberLossCUDA, 2, 9, 3>",
    "pose": "EvaluateKernel<generic all-outputs, RelativePoseError, TrivialLossCUDA, 6, 7, 7>",
}


METRIC = "residual blocks/s (residual+Jacobian+loss+gradient)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="L", choices=sorted(WORKLOADS),
                    help="S | M | L: BAL shapes, Huber, BlockSparse (configs 1-3); L4: L + "
                         "SubsetManifold(9,{0}) + CompressedRow (config 4); P5: pose graph (config 5)")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (debug)")
    ap.add_argument("--cpu-sample-blocks", type=int, default=None,
                    help="residual blocks of the CPU leg (default: 6 M inside the GPU arm, the "
                         "whole workload for --impl reference)")
    ap.add_argument("--no-multi-gpu-check", action="store_true")
    ap.add_argument("--pose-edge-order", default="temporal", choices=["temporal", "random"],
                    help="P5: edges sorted by their later pose (as g2o files list them) or the "
                         "loop closures in random order (worst case for locality)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to "
                         "DIR/<name>.npy (float64): cost, residuals, gradient, jacobian; arrays "
                         f"longer than {DUMP_SAMPLE} values as a fixed seeded sample whose "
                         "positions go to DIR/<name>_index.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


DUMP_SAMPLE = 1 << 20   # values kept per array: 3 arrays and their positions stay under 64 MB


def dump_outputs(path, cost, arrays):
    """Writes cost and each of `arrays` as float64 .npy files under path.  The sample positions
    depend only on an array's length, so two runs with the same arguments write the same ones."""
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "cost.npy"), np.array([cost], dtype=np.float64))
    for name, a in arrays.items():
        idx = np.arange(a.size) if a.size <= DUMP_SAMPLE else np.sort(
            np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))
        np.save(os.path.join(path, name + ".npy"), np.asarray(a[idx], dtype=np.float64))
        np.save(os.path.join(path, name + "_index.npy"), idx.astype(np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while running."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)),
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def make_spec(args):
    import ceres_b200  # noqa: F401
    from ceres_b200 import problems as P
    w = WORKLOADS[args.workload]
    if w["kind"] == "bal":
        return P.bal_shape(w["shape"], scale=args.scale,
                           subset_manifold=bool(w.get("subset_manifold")))
    return P.pose_graph_problem(max(10, int(w["poses"] * args.scale)),
                                max(20, int(w["edges"] * args.scale)), seed=5,
                                order=args.pose_edge_order)


def workload_config(args, spec):
    m, w = spec.meta, WORKLOADS[args.workload]
    if w["kind"] == "bal":
        what = (f"synthetic BAL {m['num_cameras']}x{m['num_points']} "
                f"({m['num_observations']} residual blocks), "
                "SnavelyReprojectionError<2,9,3> + HuberLossCUDA(1.0), " +
                ("SubsetManifold(9,{0}) on every camera, CompressedRowSparseMatrix Jacobian, "
                 if w.get("subset_manifold") else
                 "BlockSparseMatrix Jacobian (E=points, F=cameras), ") +
                "outputs: cost+residuals+gradient+Jacobian")
        jbytes = spec.num_rb * (176 if w.get("subset_manifold") else 192)
    else:
        what = (f"synthetic pose graph {spec.num_pb} poses / {spec.num_rb} edges, "
                "RelativePoseError<6,7,7>, ProductManifold<EigenQuaternion, Euclidean<3>>, pose 0 "
                f"constant, no loss, edges in {m.get('edge_order', 'temporal')} order, "
                "BlockSparseMatrix Jacobian, outputs: cost+residuals+gradient+Jacobian")
        jbytes = spec.num_rb * 576
    return {"workload": what, "shape": args.workload, "scale": args.scale, "seed": m["seed"],
            # identical in both arms: the reference arm evaluates the same problem on the host
            "parallelism": f"contiguous residual-block range per rank x{args.gpus}, parameters "
                           "replicated",
            "l2": "working set per step (Jacobian values alone %.2f GB) exceeds the 126 MB L2"
                  % (jbytes / 1e9)}


# ---------------------------------------------------------------- CPU reference arm
def cpu_sample(spec, max_blocks):
    """A bounded sample of the workload: the first max_blocks residual blocks (one
    residual-block type) with every parameter block they touch kept in place."""
    from ceres_b200 import problems as P
    n = spec.num_rb if not max_blocks else min(spec.num_rb, max_blocks)
    if n == spec.num_rb:
        return spec, n
    _, sizes, flen = P.COST_TYPES[int(spec.rb_type[0])]
    assert (spec.rb_type == spec.rb_type[0]).all()
    return P.ProblemSpec(
        pb_size=spec.pb_size, pb_values=spec.pb_values, rb_type=spec.rb_type[:n],
        rb_pb=spec.rb_pb[:len(sizes) * n], fdata=spec.fdata[:flen * n],
        pb_constant=spec.pb_constant,
        pb_manifold_kind=spec.pb_manifold_kind, pb_manifold_param=spec.pb_manifold_param,
        rb_loss_kind=spec.rb_loss_kind[:n], rb_loss_a=spec.rb_loss_a[:n],
        rb_loss_b=spec.rb_loss_b[:n], num_eliminate_blocks=spec.num_eliminate_blocks), n


def time_cpu(spec, max_blocks, steps, warmup, fmt=0):
    """Times the reference algorithm's CPU port (oracle/, ProgramEvaluator semantics,
    contiguous static partition over all host threads)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as O
    sample, n = cpu_sample(spec, max_blocks)
    cores = os.cpu_count() or 1
    op = O.OracleProblem(sample, jacobian_format=fmt, fast=True)  # -O3 -march=native, timing only
    x = op.initial_state()
    for _ in range(max(1, warmup)):
        op.evaluate(x, num_threads=cores)
    times = []
    for _ in range(max(1, steps)):
        t0 = time.perf_counter()
        ok, cost, r, g, j = op.evaluate(x, num_threads=cores)
        times.append(time.perf_counter() - t0)
        assert ok
    per_step = float(np.mean(times))
    outputs = (cost, {"residuals": r, "gradient": g, "jacobian": j[:op.num_jacobian_values]})
    return {"value": op.num_residual_blocks / per_step, "unit": "residual blocks/s",
            "cores": cores, "kind": "port",
            "build": "oracle/oracle_eval.cc, g++ -O3 -march=native, std::thread static partition",
            "sample": (f"all {spec.num_rb} residual blocks" if n == spec.num_rb else
                       f"first {op.num_residual_blocks} of {spec.num_rb} residual blocks "
                       f"(whole problem's parameter blocks)") +
                      f", full Evaluate, mean of {len(times)} calls after {max(1, warmup)} warm-up",
            "ms_per_step": per_step * 1e3, "best_ms": float(min(times)) * 1e3,
            "outputs": outputs}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    spec = make_spec(args)
    # A step is one Evaluate of the WHOLE workload unless --cpu-sample-blocks bounds it
    # (L: ~3 s per step on 16 threads).
    steps, warmup = args.steps, args.warmup
    cpu = time_cpu(spec, args.cpu_sample_blocks, steps, warmup, WORKLOADS[args.workload]["fmt"])
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *cpu["outputs"])
    line = {
        "impl": "reference", "metric": METRIC,
        "value": cpu["value"], "unit": "residual blocks/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": cpu["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(args, spec),
        "cpu_baseline": {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "build")},
        "e2e": {"value": cpu["value"], "unit": "residual blocks/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------- our arm
def measured_traffic(workload, scale, world):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, from
    the tracked ncu --set full summary of this workload (profiles/r2_traffic.json, written by
    scripts/ncu_traffic.py from the .ncu-rep); None when there is no capture for this case."""
    if scale != 1.0 or world != 1:
        return None, None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            rec = json.load(f)[workload]
        return float(rec["dram_bytes_per_launch"]), rec.get("source")
    except Exception:
        return None, None


def multi_gpu_check(B, P, dist, torch, rank, world, local_rank, fresh_id, scale=0.05):
    """Sharded against unsharded evaluation of the same problem (BAL L shape at 5 %) on every
    rank's GPU, before anything is timed: residual and Jacobian slices must agree to 1e-12,
    cost and gradient to 1e-10 (max over ranks)."""
    spec = P.bal_shape("L", scale=scale)
    full = B.CudaProblem(spec, jacobian_format=0, device=local_rank)
    x = full.initial_state()
    ok0, c0, r0, g0, j0 = full.evaluate(x)
    j0 = j0.copy()
    sh = B.CudaProblem(spec, jacobian_format=0, device=local_rank, rank=rank, world_size=world,
                       nccl_id=fresh_id())
    r = np.full(full.num_residuals, np.nan)
    sh.evaluate(x, out_residuals=r)
    ok, c, r, g, j = sh.evaluate(x, out_residuals=r)
    info = sh.shard_info()
    rs = slice(info["residual_begin"], info["residual_end"])
    errs = [abs(c - c0) / abs(c0),
            float(np.max(np.abs(g - g0)) / np.max(np.abs(g0))),
            float(np.max(np.abs(r[rs] - r0[rs])) / np.max(np.abs(r0))) if rs.stop > rs.start else 0.0,
            max([float(np.max(np.abs(j[gb:gb + ln] - j0[gb:gb + ln]))) for gb, ln, _ in
                 info["segments"]] + [0.0]) / float(np.max(np.abs(j0)))]
    full.close(); sh.close()
    t = torch.tensor(errs + [0.0 if (ok and ok0) else 1.0], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e = [float(v) for v in t.cpu()]
    return {"problem": f"BAL L shape x {scale}", "cost": e[0], "gradient": e[1], "residuals": e[2],
            "jacobian": e[3],
            "ok": bool(e[4] == 0.0 and max(e[0], e[1]) <= 1e-10 and max(e[2], e[3]) <= 1e-12)}


def run_ours(args):
    import torch
    import torch.distributed as dist
    import ceres_b200  # noqa: F401
    from ceres_b200 import binding as B
    from ceres_b200 import problems as P

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of one GPU: run it with --gpus 1")
    torch.cuda.set_device(local_rank)
    w = WORKLOADS[args.workload]

    def fresh_id():
        buf = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            buf.copy_(torch.frombuffer(bytearray(B.nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(buf, 0)
        return bytes(buf.cpu().numpy().tobytes())

    nccl_id, check = None, None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        if not args.no_multi_gpu_check:
            check = multi_gpu_check(B, P, dist, torch, rank, world, local_rank, fresh_id)
            if not check["ok"]:
                raise SystemExit(f"sharded evaluation does not match the unsharded one: {check}")
        nccl_id = fresh_id()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    spec = make_spec(args)
    t_setup = time.perf_counter()
    cp = B.CudaProblem(spec, jacobian_format=w["fmt"], device=local_rank, rank=rank,
                       world_size=world, nccl_id=nccl_id)
    setup_s = time.perf_counter() - t_setup
    nrb = cp.num_residual_blocks

    # The caller's buffers: pinned host memory, as INTEGRATION.md asks of the binding.
    state = B.PinnedArray(cp.num_parameters)
    residuals = B.PinnedArray(cp.num_residuals)
    gradient = B.PinnedArray(cp.num_effective_parameters)
    state.array[:] = cp.initial_state()

    def step_e2e():
        ok, cost, *_ = cp.evaluate(state.array, out_residuals=residuals.array,
                                   out_gradient=gradient.array)
        assert ok
        return cost

    def step_device():
        ok, cost = cp.evaluate_device()
        assert ok
        return cost

    for _ in range(max(3, args.warmup)):
        step_e2e()
    for _ in range(max(3, args.warmup)):
        step_device()
    launches_per_step = cp.timing()["launches"]

    sampler = ClockSampler(local_rank)
    sampler.start()
    # ---- timed region 1: state resident in HBM, outputs stay in HBM.
    # (the K steps run back to back inside the driver library: K complete
    # cb200_engine_evaluate_device calls, each with its own launches, cost read-back and
    # stream synchronisation, without interpreter time between them)
    barrier()
    t0 = time.perf_counter()
    ok, cost, kernel_ms, device_ms = cp.evaluate_device_steps(args.steps)
    assert ok
    barrier()
    wall_device = max_over_ranks(time.perf_counter() - t0)
    kernel_ms, device_ms = list(kernel_ms), list(device_ms)
    # ---- timed region 2: end to end through Evaluator::Evaluate with host buffers.
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cost = step_e2e()
    barrier()
    wall_e2e = max_over_ranks(time.perf_counter() - t0)
    e2e_engine_ms = cp.timing()["e2e_ms"]
    clocks = sampler.stop()
    if args.dump_outputs:
        # The last timed step: Evaluator::Evaluate into the caller's host buffers, at the state
        # the device-resident steps evaluated.
        dump_outputs(args.dump_outputs, cost, {
            "residuals": residuals.array, "gradient": gradient.array,
            "jacobian": cp.jacobian_values[:cp.num_jacobian_values]})
    # ---- the candidate-step evaluation of the minimizer (cost only), device time
    cost_only_ms = []
    for _ in range(max(3, args.warmup) + 5):
        cp.evaluate_device(residuals=False, gradient=False, jacobian=False)
        cost_only_ms.append(cp.timing()["kernel_ms"])
    cost_only = max_over_ranks(float(np.mean(cost_only_ms[-5:])))

    # Device time of a step = CUDA events on the engine's stream around kernels +
    # cost reduction + gradient exchange, max over ranks; the wall clock around the K calls
    # (launch + one host synchronisation each) is reported beside it.
    dev_ms = max_over_ranks(float(np.mean(device_ms)))
    ker_ms = max_over_ranks(float(np.mean(kernel_ms)))
    info = cp.shard_info()
    local_rb = info["rb_end"] - info["rb_begin"]
    local_j = sum(s[1] for s in info["segments"])
    h2d = 8 * cp.num_parameters
    d2h = 8 * ((info["residual_end"] - info["residual_begin"]) + cp.num_effective_parameters +
               local_j + 2)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peaks()
    achieved = w["bytes"] * local_rb / (ker_ms * 1e-3) / 1e9
    traffic, traffic_src = measured_traffic(args.workload, args.scale, world)
    kname = KERNEL_NAMES["pose" if w["kind"] == "pose" else
                         ("bal_subset" if w.get("subset_manifold") else "bal")]
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
            "kernel": kname, "algorithmic_bytes_per_block": w["bytes"],
            "blocks_per_launch": local_rb, "launch_ms": ker_ms, "peak_source": peak_src,
            "cost_only_kernel_ms": cost_only}
    if w["flops"]:
        roof["fp64"] = {"achieved_tflops": w["flops"] * local_rb / (ker_ms * 1e-3) / 1e12,
                        "algorithmic_flops_per_block": w["flops"],
                        "nominal_peak_tflops": 37.2,
                        # scripts/fp64_peak.cu on a B200 of this pool
                        "measured_peak_tflops": 33.78,
                        "peak_source": "profiles/r1_fp64_peak.json"}
    line = {
        "metric": METRIC,
        "value": nrb / (wall_device / args.steps), "unit": "residual blocks/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": wall_device / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, spec),
        "value_note": "state resident in HBM, outputs left in HBM (cb200_engine_evaluate_device); "
                      "e2e is Evaluator::Evaluate with host buffers",
        "device_ms_per_step": dev_ms, "kernel_ms_per_step": ker_ms,
        "e2e": {"value": nrb / (wall_e2e / args.steps), "unit": "residual blocks/s",
                "ms_per_step": wall_e2e / args.steps * 1e3, "engine_ms_last_step": e2e_engine_ms,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "note": "per rank; host buffers page-locked with cb200_host_pin"},
        "gpu_launches": launches_per_step * args.steps * 2,
        "clocks": clocks,
        "roofline": roof,
        "setup_s": setup_s, "cost": cost,
    }
    if check is not None:
        line["multi_gpu_check"] = check
    if world == 1 and not args.no_cpu_baseline:
        cpu = time_cpu(spec, args.cpu_sample_blocks or 6_000_000, 3, 1, w["fmt"])
        line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "build")}
    else:
        line["cpu_baseline"] = None
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    # Libraries (NCCL's version banner) print to fd 1; keep stdout for the one JSON line.
    _json_fd = os.dup(1)
    os.dup2(2, 1)
    _real_print = print

    def print(*args, **kw):  # noqa: A001
        if kw.get("flush") and args and isinstance(args[0], str) and args[0].startswith("{"):
            os.write(_json_fd, (args[0] + "\n").encode())
        else:
            _real_print(*args, **kw)

    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
