"""Solver::Options::preconditioner_type for the conjugate gradients on the device-resident
Jacobian: JACOBI (blockdiag(J'J + D^2)^-1, one dense block per parameter block), IDENTITY and
the default SCALAR_JACOBI.  The device iterates are checked against a numpy PCG on the oracle's
dense Jacobian of the same seeded problems, in both value layouts, with manifolds and constant
blocks."""
import numpy as np
import pytest

import oracle_py as O
from ceres_b200 import binding as B, lm, problems as P

gpu = pytest.mark.gpu


def _problems():
    bal = P.bal_problem(7, 90, 400, seed=11)
    sub = P.bal_problem(6, 60, 260, seed=12, subset_manifold=True, constant_cameras=1)
    pose = P.pose_graph_problem(40, 120, seed=13)
    return {"bal": bal, "bal_subset_constant": sub, "pose_graph": pose}


def _system(spec, fmt):
    """Dense J, residuals and the column ranges of the active parameter blocks."""
    op = O.OracleProblem(spec, jacobian_format=fmt)
    ok, cost, r, g, values = op.evaluate(op.initial_state())
    assert ok
    J = op.dense_jacobian(values)
    blocks = [(int(d), int(d) + int(t)) for _, _, d, t in op.pb_table() if d >= 0 and t > 0]
    return op, J, r, sorted(blocks)


def _block_inverse(A, blocks):
    M = np.zeros_like(A)
    for lo, hi in blocks:
        M[lo:hi, lo:hi] = np.linalg.inv(A[lo:hi, lo:hi])
    return M


def _pcg(A, b, M, k):
    """k iterations of preconditioned conjugate gradients from x = 0."""
    x = np.zeros_like(b)
    r = b.copy()
    z = M @ r
    p = z.copy()
    rho = r @ z
    for _ in range(k):
        q = A @ p
        alpha = rho / (p @ q)
        x += alpha * p
        r -= alpha * q
        z = M @ r
        rho_next = r @ z
        p = z + (rho_next / rho) * p
        rho = rho_next
    return x


def _rel(a, b):
    return float(np.max(np.abs(a - b))) / max(float(np.max(np.abs(b))), 1e-300)


@gpu
@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("name", ["bal", "bal_subset_constant", "pose_graph"])
def test_block_jacobi_iterates_match_numpy(name, fmt):
    spec = _problems()[name]
    op, J, r, blocks = _system(spec, fmt)
    assert sum(hi - lo for lo, hi in blocks) == J.shape[1]
    cp = B.CudaProblem(spec, jacobian_format=fmt)
    ok, *_ = cp.evaluate(op.initial_state())
    assert ok
    d2 = (J * J).sum(axis=0) / 1e4
    A = J.T @ J + np.diag(d2)
    M = _block_inverse(A, blocks)
    for k in (1, 2, 5):
        y, s = cp.cgnr_solve(d2, min_iterations=k, max_iterations=k, r_tolerance=-1.0,
                             q_tolerance=-1.0, preconditioner="jacobi")
        assert s["iterations"] == k and s["termination"] == 1, s
        assert _rel(y, _pcg(A, J.T @ r, M, k)) <= 1e-9, k


@gpu
def test_block_jacobi_is_exact_on_a_block_diagonal_system():
    """With every camera constant J'J is block diagonal (one 3 x 3 block per point): the
    preconditioner is the inverse and one iteration solves the system."""
    spec = P.bal_problem(6, 60, 260, seed=14, constant_cameras=6)
    op, J, r, blocks = _system(spec, 0)
    assert all(hi - lo == 3 for lo, hi in blocks)
    cp = B.CudaProblem(spec)
    cp.evaluate(op.initial_state())
    d2 = (J * J).sum(axis=0) / 1e4
    exact = np.linalg.solve(J.T @ J + np.diag(d2), J.T @ r)
    y, s = cp.cgnr_solve(d2, max_iterations=100, r_tolerance=1e-10, q_tolerance=-1.0,
                         preconditioner="jacobi")
    assert s["termination"] == 0 and s["iterations"] == 1, s
    assert _rel(y, exact) <= 1e-9
    _, s_scalar = cp.cgnr_solve(d2, max_iterations=100, r_tolerance=1e-10, q_tolerance=-1.0)
    assert s_scalar["termination"] == 0 and s_scalar["iterations"] > 1, s_scalar


@gpu
@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("preconditioner", ["identity", "jacobi"])
def test_converged_solution_matches_the_dense_solve(preconditioner, fmt):
    """On Jacobi-scaled columns, as ceres::Solve hands them to the solver: unpreconditioned
    conjugate gradients do not reach 1e-13 on the raw BAL columns (focal length ~1e3 next to
    distortion coefficients ~1e-7) within 5000 iterations."""
    spec = _problems()["bal"]
    op, J, r, _ = _system(spec, fmt)
    cp = B.CudaProblem(spec, jacobian_format=fmt)
    cp.evaluate(op.initial_state())
    scale = 1.0 / (1.0 + np.sqrt((J * J).sum(axis=0)))
    cp.jacobian_scale_columns(scale)
    J = J * scale
    d2 = (J * J).sum(axis=0) / 1e4
    exact = np.linalg.solve(J.T @ J + np.diag(d2), J.T @ r)
    y, s = cp.cgnr_solve(d2, max_iterations=5000, r_tolerance=1e-13, q_tolerance=-1.0,
                         preconditioner=preconditioner)
    assert s["termination"] == 0, s
    assert _rel(y, exact) <= 1e-7


@gpu
def test_block_jacobi_needs_fewer_iterations_than_the_scalar_diagonal():
    spec = _problems()["bal"]
    op, J, r, _ = _system(spec, 0)
    cp = B.CudaProblem(spec)
    cp.evaluate(op.initial_state())
    d2 = (J * J).sum(axis=0) / 1e4
    counts = {}
    for name in ("scalar_jacobi", "jacobi"):
        _, s = cp.cgnr_solve(d2, max_iterations=5000, r_tolerance=1e-10, q_tolerance=-1.0,
                             preconditioner=name)
        assert s["termination"] == 0, (name, s)
        counts[name] = s["iterations"]
    assert counts["jacobi"] < counts["scalar_jacobi"], counts


@gpu
def test_singular_block_falls_back_to_the_scalar_diagonal():
    """A camera seen once has a rank-2 9 x 9 block of J'J; without damping its Cholesky
    factorisation breaks down and the block takes the scalar rule instead of a NaN."""
    spec = P.bal_problem(12, 10, 20, seed=15)
    npts, nc = spec.meta["num_points"], spec.meta["num_cameras"]
    seen = np.bincount(spec.rb_pb[0::2] - npts, minlength=nc)
    assert (seen == 1).any()
    cp = B.CudaProblem(spec)
    cp.evaluate(cp.initial_state())
    y, s = cp.cgnr_solve(None, max_iterations=200, r_tolerance=1e-8, q_tolerance=-1.0,
                         preconditioner="jacobi")
    assert np.all(np.isfinite(y)), s
    assert s["termination"] in (0, 1), s


def _perturbed_bal(seed, subset_manifold=False):
    spec = P.bal_problem(12, 600, 2600, seed=seed, subset_manifold=subset_manifold)
    rng = np.random.default_rng(seed)
    spec.pb_values[:] += rng.normal(0, 0.02, spec.pb_values.size) * (np.abs(spec.pb_values) < 50)
    return spec


@gpu
def test_solve_with_block_jacobi_reaches_the_exact_solve_cost():
    spec = _perturbed_bal(31)
    out = B.solve(spec, B.CGNR, max_num_iterations=40, cuda_sparse=True, preconditioner="jacobi")
    assert out["usable"], out["message"]
    assert out["linear_solver_iterations"] > 0
    ref = lm.solve(O.OracleProblem(spec, jacobian_format=1), max_num_iterations=40)
    assert abs(out["initial_cost"] - ref["initial_cost"]) <= 1e-10 * ref["initial_cost"]
    assert out["final_cost"] <= 1.02 * ref["cost"]


@gpu
@pytest.mark.parametrize("kind", ["bal", "bal_subset", "pose_graph"])
def test_device_and_host_loops_take_the_same_block_jacobi_steps(kind, monkeypatch):
    if kind == "pose_graph":
        spec = P.pose_graph_problem(120, 420, seed=8)
    else:
        spec = _perturbed_bal(33, subset_manifold=kind == "bal_subset")
    monkeypatch.setenv("CB200_DRIVER_ETA", "1e-9")
    dev = B.solve(spec, B.CGNR, max_num_iterations=12, cuda_sparse=True, preconditioner="jacobi")
    monkeypatch.setenv("CB200_HOST_TRUST_REGION", "1")
    host = B.solve(spec, B.CGNR, max_num_iterations=12, cuda_sparse=True, preconditioner="jacobi")
    assert dev["usable"] and host["usable"], (dev["message"], host["message"])
    assert dev["iterations"] == host["iterations"]
    assert dev["successful_steps"] == host["successful_steps"]
    assert abs(dev["initial_cost"] - host["initial_cost"]) <= 1e-12 * host["initial_cost"]
    assert abs(dev["final_cost"] - host["final_cost"]) <= 1e-5 * host["final_cost"]
    assert np.max(np.abs(dev["x"] - host["x"])) <= 1e-3 * np.max(np.abs(host["x"]))
    assert dev["final_cost"] < 0.9 * dev["initial_cost"]


def test_options_accept_block_jacobi_only_for_the_device_cgnr():
    spec = P.bal_problem(2, 5, 10, seed=1)
    for name in ("identity", "jacobi"):
        ok, msg = B.options_is_valid(spec, 1, B.CGNR, cuda_sparse=True, preconditioner=name)
        assert ok, msg
        ok, msg = B.options_is_valid(spec, 1, B.ITERATIVE_SCHUR, cuda_sparse=True,
                                     preconditioner=name)
        assert not ok and "linear_solver_type" in msg and "sparse_linear_algebra" in msg, msg
        ok, msg = B.options_is_valid(spec, 1, B.CGNR, cuda_sparse=False, preconditioner=name)
        assert not ok and "CUDA_SPARSE" in msg, msg
    for lst in (B.CGNR, B.ITERATIVE_SCHUR, B.SPARSE_NORMAL_CHOLESKY):
        for cuda_sparse in (False, True):
            ok, msg = B.options_is_valid(spec, 1, lst, cuda_sparse=cuda_sparse)
            assert ok, msg
            ok, msg = B.options_is_valid(spec, 1, lst, cuda_sparse=cuda_sparse,
                                         preconditioner="scalar_jacobi")
            assert ok, msg
    with pytest.raises(ValueError):
        B.options_is_valid(spec, 1, B.CGNR, cuda_sparse=True, preconditioner="schur_jacobi")
