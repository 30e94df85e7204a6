"""Times the device-resident linear algebra on a BAL-shaped problem: one conjugate-gradient
iteration on the normal equations (one pass J'(J p), three vector kernels) with the Jacobian in HBM,
next to the evaluation that produced it.   python scripts/bench_solve.py --shape L
With --preconditioner scalar_jacobi,jacobi,... it also reports, per preconditioner, the pass that
accumulates blockdiag(J'J), the factorisation, the time per iteration and the iterations to reach
r_tolerance = 1e-6 on the same system.
Prints one JSON line; nothing here reads the oracle."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ceres_b200 import binding as B, problems as P  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="L")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--iterations", type=int, default=20)
    ap.add_argument("--preconditioner", default="",
                    help="comma-separated names of binding.PRECONDITIONERS to compare")
    args = ap.parse_args()
    names = [n for n in args.preconditioner.split(",") if n]
    for n in names:
        if n not in B.PRECONDITIONERS:
            ap.error(f"unknown preconditioner {n}")
    t0 = time.time()
    spec = P.bal_shape(args.shape, args.scale)
    nc, npts, nobs = spec.meta["num_cameras"], spec.meta["num_points"], spec.num_rb
    cp = B.CudaProblem(spec, jacobian_format=0)
    setup = time.time() - t0
    state = cp.initial_state()
    r = np.zeros(cp.num_residuals)
    g = np.zeros(cp.num_effective_parameters)
    cp.evaluate(state, jacobian=False, out_residuals=r, out_gradient=g)
    for _ in range(3):
        ok, cost = cp.evaluate_device()
    eval_ms = cp.timing()["device_ms"]
    d2 = cp.jacobian_squared_column_norm() / 1e4
    cp.cgnr_solve(d2, min_iterations=1, max_iterations=1)  # allocates the work vectors
    out = {}
    for iters in (2, 2 + args.iterations):
        _, s = cp.cgnr_solve(d2, min_iterations=iters, max_iterations=iters, r_tolerance=-1.0,
                             q_tolerance=-1.0)
        out[iters] = s
    per_iter = (out[2 + args.iterations]["ms"] - out[2]["ms"]) / args.iterations
    nnz = 24 * nobs
    # one iteration makes one pass over the values (J'(J p) fused)
    gbs = nnz * 8 / (per_iter * 1e-3) / 1e9
    result = {
        "workload": f"synthetic BAL {nc}x{npts} ({nobs} residual blocks), Jacobian in HBM",
        "evaluate_device_ms": eval_ms,
        "cg_iteration_ms": per_iter,
        "cg_fixed_cost_ms": out[2]["ms"] - 2 * per_iter,
        "jacobian_bytes": nnz * 8,
        "cg_iteration_jacobian_GBps": gbs,
        "setup_s": setup,
        "cost": cost,
    }
    if names:
        result["preconditioners"] = {n: _preconditioner(cp, d2, n, args.iterations) for n in names}
    print(json.dumps(result))


def _solve_ms(cp, d2, name, iterations, repeats=5):
    """Median device time of a solve with exactly `iterations` iterations."""
    times = []
    for _ in range(repeats):
        _, s = cp.cgnr_solve(d2, min_iterations=iterations, max_iterations=iterations,
                             r_tolerance=-1.0, q_tolerance=-1.0, preconditioner=name)
        times.append(s["ms"])
    return float(np.median(times))


def _preconditioner(cp, d2, name, iterations):
    """A solve with zero iterations is the set-up: J'b, the preconditioner, the model terms.
    Differences of such solves isolate the blockdiag(J'J) pass (recomputed after the values
    change, reused otherwise) and the factorisation with the first M^-1 r (over the scalar
    set-up).  Scaling the columns by one changes no value but invalidates blockdiag(J'J)."""
    ones = np.ones(cp.num_effective_parameters)
    cp.cgnr_solve(d2, min_iterations=1, max_iterations=1, preconditioner=name)  # allocates
    setup = _solve_ms(cp, d2, name, 0)
    out = {"setup_ms": setup,
           "factor_ms": setup - _solve_ms(cp, d2, "scalar_jacobi", 0)}
    if name == "jacobi":
        with_pass = []
        for _ in range(5):
            cp.jacobian_scale_columns(ones)
            _, s = cp.cgnr_solve(d2, min_iterations=0, max_iterations=0, r_tolerance=-1.0,
                                 q_tolerance=-1.0, preconditioner=name)
            with_pass.append(s["ms"])
        out["block_diagonal_pass_ms"] = float(np.median(with_pass)) - setup
    short, long = _solve_ms(cp, d2, name, 2), _solve_ms(cp, d2, name, 2 + iterations)
    out["cg_iteration_ms"] = (long - short) / iterations
    _, s = cp.cgnr_solve(d2, max_iterations=5000, r_tolerance=1e-6, q_tolerance=-1.0,
                         preconditioner=name)
    out.update({"iterations_to_1e-6": s["iterations"], "termination": s["termination"],
                "solve_to_1e-6_ms": s["ms"]})
    return out


if __name__ == "__main__":
    main()
