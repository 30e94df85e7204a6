"""The SoftLOne, Arctan, Tolerant, Tukey and composed losses (include/ceres/loss_function_cuda.h,
after internal/ceres/loss_function.cc).

On the host: rho(0) = 0, rho' and rho'' against central differences (the checks of the
reference's loss_function_test.cc), the composition rule, and the product's host evaluation
(Problem::EvaluateResidualBlock, through HostLossThunk) against the restatement below to 1 ulp.

The oracle (oracle/oracle_eval.cc) restates the reference's losses only.  The new ones are
restated here in plain Python floats (IEEE double, no contraction, the platform's libm: what the
oracle's -ffp-contract=off C++ computes) and applied to the oracle's evaluation without a loss,
block by block, with the oracle's own Corrector (_OracleWithLoss).

On the GPU, against that with the parity tolerances of test_gpu_parity.py: every new loss
in both value layouts, the generic variant, the loss table, a pose graph, Tukey's zero rho' for
outliers, ceres::Solve on the device-resident loop, and the size-independent properties of
test_full_size_properties.py on BAL M."""
import math

import numpy as np
import pytest

import oracle_py as O
from ceres_b200 import binding as B, lm, problems as P

RTOL_VALUES = 1e-12
RTOL_SUMS = 1e-10
TINY = np.finfo(float).tiny  # numeric_limits<double>::min(), rho's floor

# (kind, a, b): a = 0.7 as in loss_function_test.cc; b = Tolerant's second parameter or the scale
KINDS = [
    (P.LOSS_SOFT_L1, 0.7, 0.0),
    (P.LOSS_ARCTAN, 0.7, 0.0),
    (P.LOSS_TOLERANT, 0.7, 0.4),
    (P.LOSS_TUKEY, 0.7, 0.0),
    (P.LOSS_SCALED_SOFT_L1, 0.7, 1.3),
    (P.LOSS_SCALED_TUKEY, 0.7, 1.3),
    (P.LOSS_COMPOSED, 0.7, 1.3),
]
KIND_IDS = ["soft_l1", "arctan", "tolerant", "tukey", "scaled_soft_l1", "scaled_tukey", "composed"]


def _branch_points(kind, a, b):
    """s on both sides of the kind's branch: Tolerant's switch to the linear tail at
    (s - a) / b = 36.7, Tukey's limit s = a^2."""
    if kind == P.LOSS_TOLERANT:
        return [a + 36.7 * b - 0.01, a + 36.7 * b + 0.01]
    if kind in (P.LOSS_TUKEY, P.LOSS_SCALED_TUKEY):
        return [a * a - 0.01, a * a + 0.01]
    return []


# ------------------------------------------------------------------ the losses, restated
def _soft_l1(a, s):
    b = a * a
    c = 1 / b
    total = 1.0 + s * c
    tmp = math.sqrt(total)
    d1 = max(TINY, 1.0 / tmp)
    return [2.0 * b * (tmp - 1.0), d1, -(c * d1) / (2.0 * total)]


def _arctan(a, s):
    b = 1 / (a * a)
    total = 1 + s * s * b
    inv = 1 / total
    return [a * math.atan2(s, a), max(TINY, inv), -2.0 * s * b * (inv * inv)]


def _tolerant(a, b, s):
    c = b * math.log(1.0 + math.exp(-a / b))
    x = (s - a) / b
    if x > 36.7:
        return [s - a - c, 1.0, 0.0]
    e_x = math.exp(x)
    try:
        cosh_x = math.cosh(x)
    except OverflowError:  # (C's cosh returns inf)
        cosh_x = math.inf
    return [b * math.log(1.0 + e_x) - c, max(TINY, e_x / (1.0 + e_x)), 0.5 / (b * (1.0 + cosh_x))]


def _tukey(a, s):
    a2 = a * a
    if s <= a2:
        value = 1.0 - s / a2
        value_sq = value * value
        return [a2 / 6.0 * (1.0 - value_sq * value), 0.5 * value_sq, -1.0 / a2 * value]
    return [a2 / 6.0, 0.0, 0.0]


def _cauchy(a, s):
    b = a * a
    c = 1 / b
    total = 1.0 + s * c
    inv = 1.0 / total
    return [b * math.log(total), max(TINY, inv), -c * (inv * inv)]


def _scaled(rho, b):
    return [rho[0] * b, rho[1] * b, rho[2] * b]


def _rho(kind, a, b, s):
    """[rho, rho', rho''] of the loss kind (problems.LOSS_*) with parameters a, b, as
    internal/ceres/loss_function.cc computes it."""
    s = float(s)
    if kind == P.LOSS_SOFT_L1:
        return np.array(_soft_l1(a, s))
    if kind == P.LOSS_ARCTAN:
        return np.array(_arctan(a, s))
    if kind == P.LOSS_TOLERANT:
        return np.array(_tolerant(a, b, s))
    if kind == P.LOSS_TUKEY:
        return np.array(_tukey(a, s))
    if kind == P.LOSS_SCALED_SOFT_L1:
        return np.array(_scaled(_soft_l1(a, s), b))
    if kind == P.LOSS_SCALED_TUKEY:
        return np.array(_scaled(_tukey(a, s), b))
    assert kind == P.LOSS_COMPOSED  # b SoftLOne(a) of Cauchy(a)
    g = _cauchy(a, s)
    f = _scaled(_soft_l1(a, g[0]), b)
    return np.array([f[0], f[1] * g[1], f[2] * g[1] * g[1] + f[1] * g[2]])


class _OracleWithLoss:
    """OracleProblem with the new losses: the oracle's evaluation without a loss, then per
    residual block rho(s) from _rho and the oracle's Corrector on the block's residuals and
    Jacobian rows (residual_block.cc:68-204), the gradient J'r of the corrected values.  The
    Jacobian is dense (`dense`); with the CompressedRow format evaluate() also returns its
    values, so that lm.solve can run on it."""

    def __init__(self, spec, jacobian_format=0):
        self.op = O.OracleProblem(spec, jacobian_format=jacobian_format)
        self.spec = spec
        self.jacobian_format = jacobian_format
        self.dense = None

    def __getattr__(self, name):
        return getattr(self.op, name)

    def evaluate(self, state=None, residuals=True, gradient=True, jacobian=True,
                 apply_loss_function=True):
        op, spec = self.op, self.spec
        if not apply_loss_function:
            return op.evaluate(state, residuals, gradient, jacobian, apply_loss_function=False)
        want_j = jacobian or gradient
        ok, _, r, _, jv = op.evaluate(state, residuals=True, gradient=False, jacobian=want_j,
                                      apply_loss_function=False)
        if not ok:
            return False, 0.0, None, None, None
        J = op.dense_jacobian(jv) if want_j else None
        rbs, first_row = op.ints("program_rbs"), op.ints("residual_layout")
        cost = 0.0
        for k, rb in enumerate(rbs):
            nres = P.COST_TYPES[int(spec.rb_type[rb])][0]
            rows = slice(first_row[k], first_row[k] + nres)
            s = 0.0
            for v in r[rows]:
                s += v * v
            rho = _rho(int(spec.rb_loss_kind[rb]), float(spec.rb_loss_a[rb]),
                       float(spec.rb_loss_b[rb]), s)
            cost += 0.5 * rho[0]
            if want_j:
                cols = np.flatnonzero(np.any(J[rows] != 0.0, axis=0))
                # (C order: oracle_py.corrector hands the array's memory to the oracle as rows)
                block = np.ascontiguousarray(J[rows][:, cols])
                r[rows], block = O.corrector(s, rho, r[rows], block)
                J[np.arange(rows.start, rows.stop)[:, None], cols[None, :]] = block
            else:
                r[rows], _ = O.corrector(s, rho, r[rows])
        self.dense = J
        g = J.T @ r if gradient else None
        values = None
        if jacobian and self.jacobian_format == 1:
            crs_rows, crs_cols = op.ints("crs_rows"), op.ints("crs_cols")
            n = op.num_jacobian_values
            values = J[np.repeat(np.arange(op.num_residuals), np.diff(crs_rows)), crs_cols[:n]]
        return True, cost, r if residuals else None, g, values


# ------------------------------------------------------------------------------ host
@pytest.mark.parametrize("kind,a,b", KINDS, ids=KIND_IDS)
def test_rho_is_zero_at_zero(kind, a, b):
    assert B.loss_evaluate(kind, a, b, 0.0)[0] == 0.0
    assert _rho(kind, a, b, 0.0)[0] == 0.0


@pytest.mark.parametrize("kind,a,b", KINDS, ids=KIND_IDS)
def test_derivatives_match_central_differences(kind, a, b):
    h = 1e-4
    for s in [0.357, 1.792] + _branch_points(kind, a, b):
        fwd, bwd = B.loss_evaluate(kind, a, b, s + h), B.loss_evaluate(kind, a, b, s - h)
        rho = B.loss_evaluate(kind, a, b, s)
        assert abs((fwd[0] - bwd[0]) / (2 * h) - rho[1]) <= 1e-6, (s, rho)
        assert abs((fwd[1] - bwd[1]) / (2 * h) - rho[2]) <= 1e-6, (s, rho)


def test_branches_take_the_reference_values():
    # Tolerant beyond the switch: rho = s - a - c, rho' = 1, rho'' = 0
    a, b = 0.7, 0.4
    c = b * np.log(1.0 + np.exp(-a / b))
    s = a + 40 * b
    rho = B.loss_evaluate(P.LOSS_TOLERANT, a, b, s)
    assert rho[1] == 1.0 and rho[2] == 0.0 and rho[0] == s - a - c
    assert B.loss_evaluate(P.LOSS_TOLERANT, a, b, 0.3)[2] > 0.0
    # Tukey beyond a^2: constant a^2 / 6, rho' = rho'' = 0
    rho = B.loss_evaluate(P.LOSS_TUKEY, 0.7, 0.0, 5.0)
    assert rho[0] == 0.7 * 0.7 / 6.0 and rho[1] == 0.0 and rho[2] == 0.0
    # Arctan and SoftLOne keep rho' at the smallest normal double
    assert B.loss_evaluate(P.LOSS_ARCTAN, 1.0, 0.0, 1e200)[1] == np.finfo(float).tiny
    assert B.loss_evaluate(P.LOSS_SOFT_L1, 1e-160, 0.0, 1e300)[1] == np.finfo(float).tiny


def _compose(f, g):
    return np.array([f[0], f[1] * g[1], f[2] * g[1] * g[1] + f[1] * g[2]])


@pytest.mark.parametrize("s", [0.0, 0.357, 0.6, 1.792, 40.0])
def test_composition_rule(s):
    a, b = 0.7, 1.3
    # Huber(a) of Cauchy(b): both rho'' <= 0, so the composition declares kNonPositiveCurvature
    g = B.loss_evaluate(P.LOSS_CAUCHY, b, 0.0, s)
    f = B.loss_evaluate(P.LOSS_HUBER, a, 0.0, g[0])
    np.testing.assert_array_equal(B.composed_loss_evaluate(0, a, b, s), _compose(f, g))
    # Tolerant(a, b) of Tukey(a)
    g = B.loss_evaluate(P.LOSS_TUKEY, a, 0.0, s)
    f = B.loss_evaluate(P.LOSS_TOLERANT, a, b, g[0])
    np.testing.assert_array_equal(B.composed_loss_evaluate(1, a, b, s), _compose(f, g))
    # the driver's composed kind: Scaled(SoftLOne(a), b) of Cauchy(a)
    g = B.loss_evaluate(P.LOSS_CAUCHY, a, 0.0, s)
    f = B.loss_evaluate(P.LOSS_SCALED_SOFT_L1, a, b, g[0])
    np.testing.assert_array_equal(B.loss_evaluate(P.LOSS_COMPOSED, a, b, s), _compose(f, g))


def _ulps(x, ref):
    x, ref = np.asarray(x, float), np.asarray(ref, float)
    return np.abs(x - ref) / np.spacing(np.maximum(np.abs(ref), np.finfo(float).tiny))


@pytest.mark.parametrize("kind,a,b", KINDS, ids=KIND_IDS)
def test_host_loss_matches_the_restatement(kind, a, b):
    for s in np.concatenate([[0.0], np.logspace(-8, 6, 57), _branch_points(kind, a, b)]):
        host, oracle = B.loss_evaluate(kind, a, b, s), _rho(kind, a, b, s)
        assert np.all(_ulps(host, oracle) <= 1.0), (s, host, oracle)


@pytest.mark.parametrize("kind,a,b", KINDS, ids=KIND_IDS)
def test_evaluate_residual_block_matches_the_restatement(kind, a, b):
    """Problem::EvaluateResidualBlock: the cost is 0.5 rho(s) of the restated loss to 1 ulp, and
    the corrected residuals are the oracle Corrector's."""
    spec = P.bal_problem(4, 20, 60, seed=6)
    spec.rb_loss_kind[:], spec.rb_loss_a[:], spec.rb_loss_b[:] = kind, a, b
    cp = B.CudaProblem(spec, with_device=False)
    for rb in range(spec.num_rb):
        ok, raw_cost, raw, _, _ = cp.evaluate_residual_block(rb, apply_loss_function=False,
                                                             jacobians=False)
        assert ok
        s = 2.0 * raw_cost
        ok, cost, res, _, _ = cp.evaluate_residual_block(rb, jacobians=False)
        assert ok
        rho = _rho(kind, a, b, s)
        assert _ulps(cost, 0.5 * rho[0]) <= 1.0, (rb, s, cost, rho)
        expected, _ = O.corrector(s, rho, raw)
        np.testing.assert_allclose(res, expected, rtol=4e-16, atol=0)


# ------------------------------------------------------------------------------- GPU
def _close(a, b, rtol, what):
    a, b = np.asarray(a, float), np.asarray(b, float)
    scale = max(float(np.max(np.abs(b))), 1e-300)
    err = float(np.max(np.abs(a - b))) / scale
    assert err <= rtol, f"{what}: max error / max magnitude = {err:.3e} > {rtol:.0e}"


def _check(spec, fmt=0, state=None, bulk=None):
    op = _OracleWithLoss(spec, jacobian_format=fmt)
    cp = B.CudaProblem(spec, jacobian_format=fmt, bulk=bulk)
    if state is None:
        state = op.initial_state()
    ok_o, c_o, r_o, g_o, _ = op.evaluate(state)
    cp.jacobian_values[:] = -1.0  # every value must be overwritten
    ok_c, c_c, r_c, g_c, _ = cp.evaluate(state)
    assert ok_o and ok_c
    _close(c_c, c_o, RTOL_SUMS, "cost")
    _close(r_c, r_o, RTOL_VALUES, "residuals")
    _close(cp.dense_jacobian(), op.dense, RTOL_VALUES, "jacobian")
    _close(g_c, g_o, RTOL_SUMS, "gradient")
    return op, cp


def _bal(kind, a, b, seed=4, **kw):
    spec = P.bal_problem(6, 80, 300, seed=seed, **kw)
    spec.rb_loss_kind[:], spec.rb_loss_a[:], spec.rb_loss_b[:] = kind, a, b
    return spec


def _raw_s(op):
    ok, _, r, _, _ = op.evaluate(residuals=True, gradient=False, jacobian=False,
                                 apply_loss_function=False)
    assert ok
    return (r.reshape(-1, 2) ** 2).sum(axis=1)


# a = 1 (b = 1 for Tolerant): the generator's 2 % outliers land past Tolerant's switch and
# Tukey's limit, the inliers before them
GPU_KINDS = [(P.LOSS_SOFT_L1, 1.0, 0.0), (P.LOSS_ARCTAN, 1.0, 0.0), (P.LOSS_TOLERANT, 1.0, 1.0),
             (P.LOSS_TUKEY, 1.0, 0.0), (P.LOSS_SCALED_SOFT_L1, 1.0, 0.7),
             (P.LOSS_SCALED_TUKEY, 1.0, 0.7), (P.LOSS_COMPOSED, 1.0, 0.7)]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("kind,a,b", GPU_KINDS, ids=KIND_IDS)
def test_parity_with_the_oracle(kind, a, b, fmt):
    spec = _bal(kind, a, b)
    op, _ = _check(spec, fmt)
    s = _raw_s(op)
    if kind == P.LOSS_TOLERANT:
        x = (s - a) / b
        assert (x > 36.7).any() and (x <= 36.7).any()
    if kind in (P.LOSS_TUKEY, P.LOSS_SCALED_TUKEY):
        assert (s > a * a).any() and (s <= a * a).any()
    # one AddResidualBlocks call with a shared loss object
    _check(spec, fmt, bulk=True)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", [0, 1])
def test_tolerant_with_rho_prime_at_its_floor(fmt):
    """a / b large: e^x underflows for every block, rho' sits at the smallest normal double and
    rho'' is positive, then denormal, then 0 - the Corrector's alpha branch with D far from 1,
    and its switch back to the plain scaling, on the device as on the host."""
    spec = _bal(P.LOSS_TOLERANT, 1000.0, 1.4)
    op, cp = _check(spec, fmt)
    x = (_raw_s(op) - 1000.0) / 1.4
    assert (x > -708.0).any() and (x < -710.5).any()
    # the blocks at the floor are scaled by ~1e-154 and vanish from the norm-wise comparison
    # above: compare the residuals block by block as well
    ok, _, r_o, _, _ = op.evaluate()
    ok_c, _, r_c, _, _ = cp.evaluate(op.initial_state())
    assert ok and ok_c
    r_o, r_c = r_o.reshape(-1, 2), r_c.reshape(-1, 2)
    scale = np.max(np.abs(r_o), axis=1)
    assert (scale > 0).all()
    assert np.all(np.max(np.abs(r_c - r_o), axis=1) <= 1e-9 * scale)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", [0, 1])
def test_tukey_points_seen_only_by_outliers(fmt):
    spec = _bal(P.LOSS_TUKEY, 1.0, 0.0)
    npts = spec.meta["num_points"]
    lonely = np.arange(5)  # every observation of these points becomes an outlier
    obs_point = spec.rb_pb[1::2]
    outliers = np.isin(obs_point, lonely)
    spec.fdata.reshape(-1, 2)[outliers] += 40.0
    op, cp = _check(spec, fmt)
    x = op.initial_state()
    ok, cost, r, g, _ = cp.evaluate(x)
    assert ok
    # residual rows of the outlier blocks, in program order
    program_rbs = cp.ints("program_rbs")
    row_of = cp.ints("residual_layout")
    rows = np.concatenate([row_of[k] + np.arange(2) for k in range(program_rbs.size)
                           if outliers[program_rbs[k]]])
    assert rows.size == 2 * int(outliers.sum())
    assert np.all(r[rows] == 0.0)
    J = cp.dense_jacobian()
    assert np.all(J[rows] == 0.0)
    table, program_pbs = cp.pb_table(), cp.ints("program_pbs")
    for k, pb in enumerate(program_pbs):
        if pb in lonely:
            assert np.all(g[table[k, 2]:table[k, 2] + 3] == 0.0)
    assert npts > lonely.size
    # the Jet-free variant: cost alone, and cost with the corrected residuals
    ok, cost_only, _, _, _ = cp.evaluate(x, residuals=False, gradient=False, jacobian=False)
    assert ok and abs(cost_only - cost) <= 1e-12 * cost
    ok, cost_r, r_only, _, _ = cp.evaluate(x, gradient=False, jacobian=False)
    assert ok and abs(cost_r - cost) <= 1e-12 * cost
    assert np.all(r_only[rows] == 0.0)
    _close(r_only, r, RTOL_VALUES, "residuals of the Jet-free variant")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", [0, 1])
def test_generic_variant(fmt):
    spec = P.bal_problem(12, 200, 800, seed=2, loss="soft_l1", subset_manifold=True,
                         constant_cameras=3)
    _check(spec, fmt)


@pytest.mark.gpu
def test_several_loss_objects_in_one_type():
    """The loss table + per-block index path."""
    spec = P.bal_problem(6, 80, 300, seed=5, loss="soft_l1")
    spec.rb_loss_a[::3] = 0.5
    spec.rb_loss_a[1::3] = 2.0
    _check(spec)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", [0, 1])
def test_pose_graph(fmt):
    spec = P.pose_graph_problem(300, 900, seed=5)
    spec.rb_loss_kind[:] = P.LOSS_SOFT_L1
    spec.rb_loss_a[:] = 0.05
    _check(spec, fmt)


@pytest.mark.gpu
@pytest.mark.parametrize("loss", ["soft_l1", "tukey"])
def test_device_resident_solve(loss, monkeypatch):
    """ceres::Solve with CGNR + CUDA_SPARSE: the device-resident loop takes the steps of the host
    loop around the same device Jacobian, and reaches the cost of the exact-step LM on the
    oracle."""
    spec = P.bal_problem(12, 600, 2600, seed=31, loss=loss)
    if loss == "tukey":
        # a = 4 px: the outliers past the limit, the inliers before it.  (With a = 1 px two thirds
        # of the blocks are past it and many points have no Jacobian at all; the two loops then
        # take the same number of steps but end 0.6 % apart.)
        spec.rb_loss_a[:] = 4.0
    rng = np.random.default_rng(31)
    spec.pb_values[:] += rng.normal(0, 0.02, spec.pb_values.size) * (np.abs(spec.pb_values) < 50)
    monkeypatch.setenv("CB200_DRIVER_ETA", "1e-9")
    dev = B.solve(spec, B.CGNR, max_num_iterations=12, cuda_sparse=True)
    monkeypatch.setenv("CB200_HOST_TRUST_REGION", "1")
    host = B.solve(spec, B.CGNR, max_num_iterations=12, cuda_sparse=True)
    monkeypatch.delenv("CB200_HOST_TRUST_REGION")
    assert dev["usable"] and host["usable"], (dev["message"], host["message"])
    assert dev["iterations"] == host["iterations"]
    # (the gradient is summed with atomics, so the steps differ in the last bits run to run:
    # measured up to 6e-10 apart on the final cost for SoftLOne on a B200)
    assert abs(dev["final_cost"] - host["final_cost"]) <= 1e-6 * host["final_cost"]
    ref = lm.solve(_OracleWithLoss(spec, jacobian_format=1), max_num_iterations=40)
    assert abs(dev["initial_cost"] - ref["initial_cost"]) <= 1e-10 * ref["initial_cost"]
    out = B.solve(spec, B.CGNR, max_num_iterations=40, cuda_sparse=True)
    assert out["usable"], out["message"]
    assert out["final_cost"] <= 1.02 * ref["cost"]


# ------------------------------------------------------------------ BAL M, properties
def _loss_on_host(loss, s):
    """(rho, rho') of SoftLOne(1) / Tukey(1) in numpy."""
    if loss == "soft_l1":
        t = np.sqrt(1.0 + s)
        return 2.0 * (t - 1.0), 1.0 / t
    v = 1.0 - s
    inlier = s <= 1.0
    return np.where(inlier, (1.0 - v ** 3) / 6.0, 1.0 / 6.0), np.where(inlier, 0.5 * v * v, 0.0)


@pytest.fixture(scope="module", params=["soft_l1", "tukey"])
def full(request):
    spec = P.bal_shape("M", loss=request.param)
    cp = B.CudaProblem(spec, jacobian_format=0)
    x = cp.initial_state()
    ok, cost, r, g, j = cp.evaluate(x)
    assert ok
    yield request.param, cp, x, cost, r.copy(), g.copy(), j
    cp.close()


@pytest.mark.gpu
def test_full_size_gradient_is_jt_r(full):
    loss, cp, x, cost, r, g, j = full
    jt_r = cp.jacobian_multiply(r, transpose=True)
    assert float(np.max(np.abs(jt_r - g))) <= 1e-10 * float(np.max(np.abs(g)))


@pytest.mark.gpu
def test_full_size_cost_and_corrected_residuals(full):
    loss, cp, x, cost, r, g, j = full
    ok, cost_raw, r_raw, _, _ = cp.evaluate(x, gradient=False, jacobian=False,
                                            apply_loss_function=False)
    assert ok
    s = (r_raw.reshape(-1, 2) ** 2).sum(axis=1)
    rho, rho1 = _loss_on_host(loss, s)
    assert abs(cost - 0.5 * rho.sum()) <= 1e-10 * cost
    err = np.max(np.abs(r.reshape(-1, 2) - r_raw.reshape(-1, 2) * np.sqrt(rho1)[:, None]))
    assert float(err) <= 1e-12 * float(np.max(np.abs(r)))
    if loss == "tukey":
        assert (rho1 == 0.0).any() and (rho1 > 0.0).any()


@pytest.mark.gpu
def test_full_size_evaluation_is_reproducible(full):
    loss, cp, x, cost, r, g, j = full
    j_first = j[:50_000_000].copy()
    ok, cost2, r2, g2, j2 = cp.evaluate(x)
    assert ok and cost2 == cost
    assert np.array_equal(r2, r)
    assert np.array_equal(j2[:50_000_000], j_first)
    assert float(np.max(np.abs(g2 - g))) <= 1e-12 * float(np.max(np.abs(g)))
    for _ in range(3):
        ok, cost3 = cp.evaluate_device()
        assert ok and cost3 == cost
