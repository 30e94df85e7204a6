"""ctypes binding of the test/bench driver (tests/driver/libceres_b200_driver.so),
which replays a ProblemSpec through the product's public C++ API and evaluates it
through the C ABI (include/ceres_b200.h).  No oracle, no CPU fallback: on a machine
without a CUDA device only the layout (structure) build works."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from . import problems as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(ROOT, "ceres-solver-cuda_b200", "lib", "libceres_b200.so")
DRIVER_PATH = os.path.join(ROOT, "tests", "driver", "libceres_b200_driver.so")
_DRV = None
_ABI = None

# Every symbol include/ceres_b200.h declares.
ABI_SYMBOLS = [
    "cb200_engine_create", "cb200_engine_destroy", "cb200_engine_last_error",
    "cb200_engine_set_parameter_blocks", "cb200_engine_add_residual_blocks",
    "cb200_engine_set_layout", "cb200_engine_set_shard", "cb200_engine_finalize",
    "cb200_nccl_unique_id", "cb200_engine_comm_init", "cb200_engine_evaluate",
    "cb200_engine_evaluate_device", "cb200_engine_device_ptr", "cb200_engine_shard_info",
    "cb200_engine_last_timing", "cb200_engine_exchange_plan", "cb200_engine_exchange_mode",
    "cb200_engine_state_upload", "cb200_engine_state_download", "cb200_engine_evaluate_state",
    "cb200_engine_jacobi_scale", "cb200_engine_trust_region_step",
    "cb200_engine_accept_candidate", "cb200_engine_gradient_max_norm",
    "cb200_engine_jacobian_multiply",
    "cb200_engine_jacobian_squared_column_norm", "cb200_engine_jacobian_scale_columns",
    "cb200_engine_cgnr_solve", "cb200_host_alloc", "cb200_host_pin", "cb200_host_free",
    "cb200_version",
]


def build(jobs=8):
    """Compiles libceres_b200.so and the driver for sm_100a (nvcc cross-compiles on CPU)."""
    subprocess.check_call(["make", "-C", ROOT, f"-j{jobs}", "all"], stdout=subprocess.DEVNULL)


def abi():
    global _ABI
    if _ABI is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run __graft_entry__.build() (no fallback)")
        _ABI = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        _ABI.cb200_version.restype = C.c_char_p
        _ABI.cb200_nccl_unique_id.argtypes = [C.c_void_p]
        _ABI.cb200_host_alloc.restype = C.c_void_p
        _ABI.cb200_host_alloc.argtypes = [C.c_uint64]
        _ABI.cb200_host_pin.argtypes = [C.c_void_p, C.c_uint64]
        _ABI.cb200_host_free.argtypes = [C.c_void_p]
    return _ABI


class PinnedArray:
    """float64 vector in cb200_host_alloc memory, page-locked (what a caller of the C
    ABI allocates for state / residuals / gradient to get full-rate copies)."""

    def __init__(self, n):
        L = abi()
        self.n = int(n)
        self.ptr = L.cb200_host_alloc(8 * max(self.n, 1))
        if not self.ptr:
            raise MemoryError("cb200_host_alloc failed")
        L.cb200_host_pin(self.ptr, 8 * max(self.n, 1))
        self.array = np.ctypeslib.as_array(C.cast(self.ptr, C.POINTER(C.c_double)),
                                           shape=(max(self.n, 1),))[:self.n]

    def free(self):
        if self.ptr:
            self.array = None
            abi().cb200_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def driver():
    global _DRV
    if _DRV is None:
        abi()
        if not os.path.exists(DRIVER_PATH):
            raise RuntimeError(f"{DRIVER_PATH} is missing: run __graft_entry__.build()")
        L = C.CDLL(DRIVER_PATH)
        L.drv_create.restype = C.c_void_p
        L.drv_create.argtypes = [C.c_int] + [C.c_void_p] * 5 + [C.c_int] + [C.c_void_p] * 6 + [C.c_int]
        L.drv_destroy.argtypes = [C.c_void_p]
        L.drv_error.restype = C.c_char_p
        L.drv_error.argtypes = [C.c_void_p]
        L.drv_build.argtypes = [C.c_void_p] + [C.c_int] * 8 + [C.c_void_p]
        L.drv_dims.argtypes = [C.c_void_p, C.c_void_p]
        L.drv_fixed_cost.restype = C.c_double
        L.drv_fixed_cost.argtypes = [C.c_void_p]
        L.drv_initial_state.argtypes = [C.c_void_p, C.c_void_p]
        L.drv_get_ints.restype = C.c_int64
        L.drv_get_ints.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.drv_pb_table.argtypes = [C.c_void_p, C.c_void_p]
        L.drv_jacobian_values.restype = C.POINTER(C.c_double)
        L.drv_jacobian_values.argtypes = [C.c_void_p]
        L.drv_evaluate.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_int]
        L.drv_evaluate_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.drv_timing.argtypes = [C.c_void_p, C.c_void_p]
        L.drv_evaluate_device_steps.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                                C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.drv_shard_info.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.drv_callback_info.argtypes = [C.c_void_p, C.c_void_p]
        L.drv_exchange_mode.argtypes = [C.c_void_p]
        L.drv_exchange_plan.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.drv_plus.argtypes = [C.c_void_p] * 4
        L.drv_plus_threads.argtypes = [C.c_void_p] * 4 + [C.c_int]
        L.drv_dense_jacobian.argtypes = [C.c_void_p, C.c_void_p]
        L.drv_solve_preconditioned.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.c_void_p, C.c_int, C.c_void_p]
        L.drv_problem_evaluate.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                           C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.drv_problem_evaluate_get.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.drv_evaluate_residual_block.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.drv_jacobian_multiply.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.drv_jacobian_squared_column_norm.argtypes = [C.c_void_p, C.c_void_p]
        L.drv_jacobian_scale_columns.argtypes = [C.c_void_p, C.c_void_p]
        L.drv_cgnr_solve_preconditioned.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                                    C.c_double, C.c_double, C.c_int, C.c_void_p,
                                                    C.c_void_p]
        L.drv_user_values.argtypes = [C.c_void_p, C.c_void_p]
        L.drv_options_is_valid_for.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.c_char_p, C.c_int]
        L.drv_argument_slot_ordering.argtypes = [C.c_void_p, C.c_void_p]
        L.drv_loss_evaluate.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double, C.c_void_p]
        L.drv_add_residual_blocks.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 6 + \
            [C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.drv_composed_loss_evaluate.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double,
                                                 C.c_void_p]
        _DRV = L
    return _DRV


def _create(spec, bulk):
    """drv_create for a ProblemSpec.  Specs with the loss kinds of driver_losses.h
    (problems.LOSS_SOFT_L1 and up) get their parameter blocks from drv_create and their residual
    blocks from drv_add_residual_blocks; the problem is the same one either way."""
    L = driver()
    if not (spec.rb_loss_kind >= P.LOSS_SOFT_L1).any():
        return L.drv_create(
            spec.num_pb, _p(spec.pb_size), _p(spec.pb_values), _p(spec.pb_constant),
            _p(spec.pb_manifold_kind), _p(spec.pb_manifold_param), spec.num_rb,
            _p(spec.rb_type), _p(spec.rb_pb), _p(spec.rb_loss_kind), _p(spec.rb_loss_a),
            _p(spec.rb_loss_b), _p(spec.fdata), int(bulk))
    h = L.drv_create(
        spec.num_pb, _p(spec.pb_size), _p(spec.pb_values), _p(spec.pb_constant),
        _p(spec.pb_manifold_kind), _p(spec.pb_manifold_param), 0, None, None, None, None, None,
        None, int(bulk))
    num_types = max(P.COST_TYPES) + 1
    blocks = np.zeros(num_types, dtype=np.int32)
    flen = np.zeros(num_types, dtype=np.int32)
    for t, (_, sizes, n) in P.COST_TYPES.items():
        blocks[t], flen[t] = len(sizes), n
    L.drv_add_residual_blocks(
        h, spec.num_rb, _p(spec.rb_type), _p(spec.rb_pb), _p(spec.rb_loss_kind),
        _p(spec.rb_loss_a), _p(spec.rb_loss_b), _p(spec.fdata), int(bulk) & 1, num_types,
        _p(blocks), _p(flen))
    return h


def nccl_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    rc = abi().cb200_nccl_unique_id(buf)
    if rc != 0:
        raise RuntimeError("cb200_nccl_unique_id failed (libnccl.so.2 not found?)")
    return buf.raw


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


_INT_ARRAYS = {
    "residual_layout": 0, "jacobian_per_residual_layout": 1, "jacobian_per_residual_offsets": 2,
    "program_rbs": 3, "program_pbs": 4, "col_block_size": 5, "col_block_pos": 6,
    "row_block_size": 7, "row_block_pos": 8, "row_cells_start": 9, "cell_block_id": 10,
    "cell_position": 11, "crs_rows": 12, "crs_cols": 13, "constant_pbs": 14,
    "jacobian_layout_storage": 15,
}


# ceres::LinearSolverType values (include/ceres/types.h of this repository)
SPARSE_NORMAL_CHOLESKY, DENSE_SCHUR, SPARSE_SCHUR, ITERATIVE_SCHUR, CGNR = 2, 3, 4, 5, 6

# Preconditioners by name: (ceres::PreconditionerType, CB200_PRECONDITIONER_*)
PRECONDITIONERS = {"identity": (0, 2), "jacobi": (1, 1), "scalar_jacobi": (2, 0)}


def _preconditioner(name, which):
    if name not in PRECONDITIONERS:
        raise ValueError(f"unknown preconditioner {name!r}; one of {sorted(PRECONDITIONERS)}")
    return PRECONDITIONERS[name][which]


def solve(spec, linear_solver_type=ITERATIVE_SCHUR, max_num_iterations=20, ordering=None,
          device=0, bulk=False, cuda_sparse=False, preconditioner="scalar_jacobi"):
    """ceres::Solve(options, ProblemCUDA*, summary) (reference: problem_cuda.h:490-502) on
    a ProblemSpec built through the per-block C++ API.  Returns a dict with the summary
    and the solution in the specification's parameter-block order.  preconditioner: a key of
    PRECONDITIONERS (Solver::Options::preconditioner_type)."""
    L = driver()
    h = _create(spec, int(bulk))
    err = L.drv_error(h)
    if err:
        raise RuntimeError(err.decode())
    out = np.zeros(9)
    o = None if ordering is None else np.ascontiguousarray(ordering, dtype=np.int32)
    ok = L.drv_solve_preconditioned(h, int(linear_solver_type), int(cuda_sparse),
                                    _preconditioner(preconditioner, 0), int(max_num_iterations),
                                    _p(o), int(device), _p(out))
    x = np.zeros(spec.pb_values.size)
    L.drv_user_values(h, _p(x))
    msg = L.drv_error(h).decode()
    L.drv_destroy(h)
    return dict(usable=bool(ok), initial_cost=out[0], final_cost=out[1], iterations=int(out[2]),
                successful_steps=int(out[3]), termination_type=int(out[4]),
                jacobian_evaluations=int(out[5]), residual_evaluations=int(out[6]),
                linear_solver_seconds=float(out[7]), linear_solver_iterations=int(out[8]),
                message=msg,
                x=x)


def argument_slot_ordering(spec):
    """internal::ArgumentSlotOrdering on the ProblemSpec (host code, no GPU): (found, group per
    parameter block)."""
    L = driver()
    h = _create(spec, 0)
    err = L.drv_error(h)
    if err:
        raise RuntimeError(err.decode())
    groups = np.zeros(spec.num_pb, dtype=np.int32)
    found = L.drv_argument_slot_ordering(h, _p(groups))
    L.drv_destroy(h)
    return bool(found), groups


def loss_evaluate(kind, a, b, s):
    """[rho(s), rho'(s), rho''(s)] of the product's loss class for a loss kind (problems.LOSS_*)
    with parameters a, b, evaluated on the host as Problem::EvaluateResidualBlock does."""
    rho = np.zeros(3)
    if not driver().drv_loss_evaluate(int(kind), float(a), float(b), float(s), _p(rho)):
        raise ValueError(f"loss kind {kind} has no loss object")
    return rho


def composed_loss_evaluate(which, a, b, s):
    """Host evaluation of ComposedLossCUDA<HuberLossCUDA, CauchyLossCUDA>(Huber(a), Cauchy(b))
    (which = 0) or ComposedLossCUDA<TolerantLossCUDA, TukeyLossCUDA>(Tolerant(a, b), Tukey(a))
    (which = 1)."""
    rho = np.zeros(3)
    if not driver().drv_composed_loss_evaluate(int(which), float(a), float(b), float(s), _p(rho)):
        raise ValueError(f"no composition {which}")
    return rho


def options_is_valid(spec, minimizer_type, linear_solver_type=None, cuda_sparse=False,
                     preconditioner=None):
    """Solver::Options::IsValid with use_cuda_for_evaluator (reference solver.cc:702-708);
    None keeps an option's default.  Returns (valid, message)."""
    L = driver()
    h = _create(spec, 0)
    msg = C.create_string_buffer(512)
    ok = L.drv_options_is_valid_for(
        h, int(minimizer_type), -1 if linear_solver_type is None else int(linear_solver_type),
        int(cuda_sparse), -1 if preconditioner is None else _preconditioner(preconditioner, 0),
        msg, 512)
    L.drv_destroy(h)
    return bool(ok), msg.value.decode()


class CudaProblem:
    """ProblemCUDA + Program + Evaluator for a ProblemSpec.

    with_device=False builds only the program and the Jacobian structure (host code,
    works without a GPU); evaluate() then raises."""

    def __init__(self, spec, jacobian_format=0, reduce=True, schur_reorder=False,
                 num_eliminate_blocks=None, with_device=True, device=0, rank=0, world_size=1,
                 nccl_id: bytes | None = None, bulk=None, evaluation_callback=False):
        L = driver()
        self.spec = spec
        if bulk is None:
            bulk = spec.num_rb > 5000
        bulk = int(bool(bulk)) | (2 if evaluation_callback else 0)
        self.h = _create(spec, int(bulk))
        err = L.drv_error(self.h)
        if err:
            raise RuntimeError(err.decode())
        ne = spec.num_eliminate_blocks if num_eliminate_blocks is None else num_eliminate_blocks
        self.jacobian_format = jacobian_format
        self.with_device = with_device
        idbuf = C.create_string_buffer(nccl_id, 128) if nccl_id else None
        ok = L.drv_build(self.h, int(reduce), int(schur_reorder), int(ne), int(jacobian_format),
                         int(with_device), int(device), int(rank), int(world_size), idbuf)
        if not ok:
            raise RuntimeError("drv_build failed: " + L.drv_error(self.h).decode())
        dims = np.zeros(10, dtype=np.int64)
        L.drv_dims(self.h, _p(dims))
        (self.num_parameters, self.num_effective_parameters, self.num_residuals,
         self.num_residual_blocks, self.num_parameter_blocks, self.num_jacobian_values,
         self.values_size, self.num_cells, self.offsets_size,
         self.num_constant_parameters) = (int(x) for x in dims)
        self.fixed_cost = float(L.drv_fixed_cost(self.h))
        ptr = L.drv_jacobian_values(self.h)
        # zero-copy view of the (pinned) values array of CreateJacobian()
        self.jacobian_values = np.ctypeslib.as_array(ptr, shape=(max(self.values_size, 1),))

    def close(self):
        if getattr(self, "h", None):
            self.jacobian_values = None
            driver().drv_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def ints(self, name):
        L = driver()
        n = L.drv_get_ints(self.h, _INT_ARRAYS[name], None)
        out = np.zeros(max(n, 0), dtype=np.int32)
        if n > 0:
            L.drv_get_ints(self.h, _INT_ARRAYS[name], _p(out))
        return out

    def pb_table(self):
        out = np.zeros((self.num_parameter_blocks, 4), dtype=np.int32)
        driver().drv_pb_table(self.h, _p(out))
        return out

    def initial_state(self):
        s = np.zeros(self.num_parameters)
        driver().drv_initial_state(self.h, _p(s))
        return s

    def callback_info(self):
        """What the problem's EvaluationCallback saw at its last notification."""
        out = np.zeros(4)
        driver().drv_callback_info(self.h, _p(out))
        return {"calls": int(out[0]), "evaluate_jacobians": bool(out[1]),
                "new_evaluation_point": bool(out[2]), "user_value_sum": float(out[3])}

    def evaluate(self, state=None, residuals=True, gradient=True, jacobian=True,
                 apply_loss_function=True, out_residuals=None, out_gradient=None,
                 new_evaluation_point=True):
        """Evaluator::Evaluate with host buffers.  Returns (ok, cost, r, g, jacobian_values)."""
        if not self.with_device:
            raise RuntimeError("built without a device: there is no CPU fallback")
        if state is None:
            state = self.initial_state()
        state = np.ascontiguousarray(state, dtype=np.float64)
        cost = np.zeros(1)
        r = g = None
        if residuals:
            r = out_residuals if out_residuals is not None else np.full(self.num_residuals, np.nan)
        if gradient:
            g = out_gradient if out_gradient is not None else \
                np.full(self.num_effective_parameters, np.nan)
        rc = driver().drv_evaluate(self.h, _p(state),
                                   int(apply_loss_function) | (0 if new_evaluation_point else 2),
                                   _p(cost), _p(r), _p(g), int(jacobian))
        if rc < 0:
            raise RuntimeError("no evaluator")
        j = self.jacobian_values[:self.values_size] if jacobian else None
        return bool(rc), float(cost[0]), r, g, j

    def evaluate_device(self, residuals=True, gradient=True, jacobian=True,
                        apply_loss_function=True):
        """Re-evaluates at the state already resident in HBM; outputs stay on the device."""
        cost = np.zeros(1)
        rc = driver().drv_evaluate_device(self.h, int(apply_loss_function), int(residuals),
                                          int(gradient), int(jacobian), _p(cost))
        if rc < 0:
            raise RuntimeError(f"evaluate_device failed ({rc})")
        return rc == 0, float(cost[0])

    def evaluate_device_steps(self, steps, residuals=True, gradient=True, jacobian=True,
                              apply_loss_function=True):
        """`steps` evaluations at the resident state, back to back inside the driver (no
        interpreter time between them).  Returns (ok, cost, kernel_ms[steps], device_ms[steps])."""
        cost, kernel_ms, device_ms = np.zeros(1), np.zeros(steps), np.zeros(steps)
        rc = driver().drv_evaluate_device_steps(
            self.h, int(steps), int(apply_loss_function), int(residuals), int(gradient),
            int(jacobian), _p(kernel_ms), _p(device_ms), _p(cost))
        if rc < 0:
            raise RuntimeError(f"evaluate_device_steps failed ({rc})")
        return rc == 0, float(cost[0]), kernel_ms, device_ms

    # ---- Problem::Evaluate / Problem::EvaluateResidualBlock (the user-level entry points)
    def problem_evaluate(self, parameter_blocks=None, residual_blocks=None,
                         apply_loss_function=True, device=0):
        """Problem::Evaluate(options, &cost, &residuals, &gradient, &jacobian) at the user
        state.  Returns (ok, cost, residuals, gradient, (rows, cols, values), (num_rows,
        num_cols))."""
        pb = None if parameter_blocks is None else np.ascontiguousarray(parameter_blocks, np.int32)
        rb = None if residual_blocks is None else np.ascontiguousarray(residual_blocks, np.int32)
        cost, dims = np.zeros(1), np.zeros(5, dtype=np.int64)
        ok = driver().drv_problem_evaluate(
            self.h, int(apply_loss_function), 0 if pb is None else pb.size, _p(pb),
            0 if rb is None else rb.size, _p(rb), int(device), _p(cost), _p(dims))
        r, g = np.zeros(dims[0]), np.zeros(dims[1])
        rows, cols = np.zeros(dims[2] + 1, np.int32), np.zeros(dims[4], np.int32)
        vals = np.zeros(dims[4])
        if ok:
            for which, arr in enumerate((r, g, rows, cols, vals)):
                if arr.size:
                    driver().drv_problem_evaluate_get(self.h, which, _p(arr))
        return bool(ok), float(cost[0]), r, g, (rows, cols, vals), (int(dims[2]), int(dims[3]))

    def evaluate_residual_block(self, rb, apply_loss_function=True, jacobians=True):
        """Problem::EvaluateResidualBlock on the host.  Returns (ok, cost, residuals, list of
        per-argument Jacobians (None for constant blocks), parameter block ids)."""
        from . import problems as P
        spec = self.spec
        kres, sizes, _ = P.COST_TYPES[int(spec.rb_type[rb])]
        cost, res = np.zeros(1), np.zeros(kres)
        jac = np.zeros(kres * sum(sizes))
        ids = np.zeros(len(sizes), np.int32)
        ok = driver().drv_evaluate_residual_block(self.h, int(rb), kres, int(apply_loss_function),
                                                  int(jacobians), _p(cost), _p(res), _p(jac), _p(ids))
        out, cursor = [], 0
        for j, pb in enumerate(ids):
            if not jacobians or spec.pb_constant[pb]:
                out.append(None)
                continue
            tangent = self.tangent_size(int(pb))
            out.append(jac[cursor:cursor + kres * tangent].reshape(kres, tangent).copy())
            cursor += kres * tangent
        return bool(ok), float(cost[0]), res, out, ids

    def tangent_size(self, pb):
        from . import problems as P
        spec = self.spec
        size, kind, param = int(spec.pb_size[pb]), int(spec.pb_manifold_kind[pb]), \
            int(spec.pb_manifold_param[pb])
        if kind in (P.MANIFOLD_SUBSET, P.MANIFOLD_OPAQUE_SUBSET):
            return size - bin(param).count("1")
        if kind in (P.MANIFOLD_QUATERNION, P.MANIFOLD_EIGEN_QUATERNION,
                    P.MANIFOLD_QUATERNION_X_EUCLIDEAN, P.MANIFOLD_EIGEN_QUATERNION_X_EUCLIDEAN):
            return size - 1
        return size

    # ---- linear algebra on the Jacobian the last evaluation left in HBM
    def _la_check(self, rc):
        if rc != 0:
            raise RuntimeError(f"device Jacobian operation failed ({rc}): "
                               f"{driver().drv_error(self.h).decode()}")

    def jacobian_multiply(self, x, transpose=False):
        """y = J x (or J' x) with the device-resident Jacobian of the last evaluation."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.zeros(self.num_effective_parameters if transpose else self.num_residuals)
        self._la_check(driver().drv_jacobian_multiply(self.h, int(transpose), _p(x), _p(y)))
        return y

    def jacobian_squared_column_norm(self):
        out = np.zeros(self.num_effective_parameters)
        self._la_check(driver().drv_jacobian_squared_column_norm(self.h, _p(out)))
        return out

    def jacobian_scale_columns(self, scale):
        scale = np.ascontiguousarray(scale, dtype=np.float64)
        self._la_check(driver().drv_jacobian_scale_columns(self.h, _p(scale)))

    def cgnr_solve(self, d_squared=None, min_iterations=0, max_iterations=500, r_tolerance=-1.0,
                   q_tolerance=0.1, preconditioner="scalar_jacobi"):
        """(J'J + diag(d_squared)) y = J'r on the device; returns (y, summary dict).
        preconditioner: a key of PRECONDITIONERS."""
        d2 = None if d_squared is None else np.ascontiguousarray(d_squared, dtype=np.float64)
        y = np.zeros(self.num_effective_parameters)
        out = np.zeros(8)
        self._la_check(driver().drv_cgnr_solve_preconditioned(
            self.h, _p(d2), int(min_iterations), int(max_iterations), float(r_tolerance),
            float(q_tolerance), _preconditioner(preconditioner, 1), _p(y), _p(out)))
        return y, dict(iterations=int(out[0]), termination=int(out[1]), gradient_norm=out[2],
                       residual_norm=out[3], jy_dot_b=out[4], jy_squared_norm=out[5], ms=out[6])

    def timing(self):
        """ms of the last evaluation: kernels, kernels+reductions+allreduce, whole call; launches."""
        out = np.zeros(4)
        driver().drv_timing(self.h, _p(out))
        return {"kernel_ms": out[0], "device_ms": out[1], "e2e_ms": out[2], "launches": int(out[3])}

    def shard_info(self):
        info = np.zeros(4, dtype=np.int32)
        seg = np.zeros(3 * 16, dtype=np.int64)
        n = driver().drv_shard_info(self.h, _p(info), _p(seg), 16)
        return {"rb_begin": int(info[0]), "rb_end": int(info[1]), "residual_begin": int(info[2]),
                "residual_end": int(info[3]),
                "segments": [tuple(int(x) for x in seg[3 * i:3 * i + 3]) for i in range(max(n, 0))]}

    def exchange_mode(self):
        """0: one rank; 1: NCCL all-reduce; 2: peer exchange fused into the evaluation kernel."""
        return int(driver().drv_exchange_mode(self.h))

    def exchange_plan(self):
        """This rank's gradient exchange plan (several ranks): None when the structure only
        allows the NCCL all-reduce, else {chunks: [n, 4] (first block, end block, gradient
        begin, gradient end), exclusive: (begin, length), shared_count}."""
        excl = np.zeros(2, dtype=np.int64)
        shared = np.zeros(1, dtype=np.int32)
        n = driver().drv_exchange_plan(self.h, None, 0, _p(excl), _p(shared))
        if n < 0:
            return None
        chunks = np.zeros((max(n, 1), 4), dtype=np.int32)
        driver().drv_exchange_plan(self.h, _p(chunks), n, _p(excl), _p(shared))
        return {"chunks": chunks[:n], "exclusive": (int(excl[0]), int(excl[1])),
                "shared_count": int(shared[0])}

    def plus(self, state, delta, num_threads=1):
        out = np.zeros(self.num_parameters)
        if num_threads > 1:
            driver().drv_plus_threads(self.h, _p(np.ascontiguousarray(state)),
                                      _p(np.ascontiguousarray(delta)), _p(out), int(num_threads))
            return out
        driver().drv_plus(self.h, _p(np.ascontiguousarray(state)), _p(np.ascontiguousarray(delta)),
                          _p(out))
        return out

    def dense_jacobian(self):
        J = np.zeros((self.num_residuals, self.num_effective_parameters))
        driver().drv_dense_jacobian(self.h, _p(J))
        return J
