"""BASELINE.json's full-size configuration (synthetic BAL 13682 x 4456117, 28,987,644 residual
blocks) is too large for the oracle, so the CUDA path is checked there through properties that
do not depend on the size:

* linearity: the gradient the evaluation kernel accumulates with atomics equals J' r computed
  by an independent kernel (cb200_engine_jacobian_multiply) from the Jacobian and residuals it
  wrote;
* a prefix of the problem (the first residual blocks, all parameter blocks) evaluated by the
  oracle reproduces the corresponding residuals and Jacobian cells of the full evaluation;
* the cost equals the sum over residual blocks recomputed on the host from the uncorrected
  residuals (apply_loss_function = false) through the loss function;
* two evaluations give bit-identical residuals, Jacobian and cost (the gradient is summed with
  atomics and agrees to rounding).
(Sharded evaluation against unsharded is covered at small size in test_gpu_parity.py and on
several GPUs by scripts/check_multigpu.py.)
"""
import numpy as np
import pytest

import oracle_py as O
from ceres_b200 import binding as B, problems as P

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def full():
    spec = P.bal_shape("L")
    cp = B.CudaProblem(spec, jacobian_format=0)
    x = cp.initial_state()
    ok, cost, r, g, j = cp.evaluate(x)
    assert ok
    yield spec, cp, x, cost, r.copy(), g.copy(), j
    cp.close()


def test_gradient_is_jt_r(full):
    spec, cp, x, cost, r, g, j = full
    jt_r = cp.jacobian_multiply(r, transpose=True)
    scale = float(np.max(np.abs(g)))
    assert float(np.max(np.abs(jt_r - g))) <= 1e-10 * scale


def test_cost_is_the_sum_of_the_losses(full):
    spec, cp, x, cost, r, g, j = full
    ok, cost_raw, r_raw, _, _ = cp.evaluate(x, gradient=False, jacobian=False,
                                            apply_loss_function=False)
    assert ok
    s = (r_raw.reshape(-1, 2) ** 2).sum(axis=1)
    assert abs(cost_raw - 0.5 * s.sum()) <= 1e-10 * cost_raw
    a = float(spec.rb_loss_a[0])            # HuberLossCUDA(a): loss_function_cuda.h:78-96
    rho = np.where(s > a * a, 2.0 * a * np.sqrt(s) - a * a, s)
    assert abs(cost - 0.5 * rho.sum()) <= 1e-10 * cost
    # the corrected residuals are the raw ones scaled by sqrt(rho') (corrector.cc:112-124)
    sqrt_rho1 = np.where(s > a * a, np.sqrt(a / np.sqrt(np.maximum(s, 1e-300))), 1.0)
    assert float(np.max(np.abs(r.reshape(-1, 2) - r_raw.reshape(-1, 2) * sqrt_rho1[:, None]))) <= \
        1e-12 * float(np.max(np.abs(r)))


def test_prefix_matches_the_oracle(full):
    spec, cp, x, cost, r, g, j = full
    n = 200_000
    prefix = P.ProblemSpec(
        pb_size=spec.pb_size, pb_values=spec.pb_values, rb_type=spec.rb_type[:n],
        rb_pb=spec.rb_pb[:2 * n], fdata=spec.fdata[:2 * n], rb_loss_kind=spec.rb_loss_kind[:n],
        rb_loss_a=spec.rb_loss_a[:n], rb_loss_b=spec.rb_loss_b[:n],
        num_eliminate_blocks=spec.num_eliminate_blocks)
    # reduce=False keeps the untouched parameter blocks, so offsets match the full problem
    op = O.OracleProblem(prefix, jacobian_format=0, reduce=False)
    ok, c_o, r_o, g_o, j_o = op.evaluate(op.initial_state())
    assert ok
    assert float(np.max(np.abs(r[:2 * n] - r_o))) <= 1e-12 * float(np.max(np.abs(r_o)))
    # block-sparse values: E cells (points, 2x3) of the first n blocks come first in both
    assert float(np.max(np.abs(j[:6 * n] - j_o[:6 * n]))) <= 1e-12 * float(np.max(np.abs(j_o)))
    f_full, f_pre = 6 * spec.num_rb, 6 * n
    assert float(np.max(np.abs(j[f_full:f_full + 18 * n] - j_o[f_pre:f_pre + 18 * n]))) <= \
        1e-12 * float(np.max(np.abs(j_o)))


def test_evaluation_is_reproducible_except_for_the_atomic_gradient(full):
    spec, cp, x, cost, r, g, j = full
    j_first = j[:50_000_000].copy()
    ok, cost2, r2, g2, j2 = cp.evaluate(x)
    assert ok and cost2 == cost
    assert np.array_equal(r2, r)
    assert np.array_equal(j2[:50_000_000], j_first)
    assert float(np.max(np.abs(g2 - g))) <= 1e-12 * float(np.max(np.abs(g)))
    # warps draw their chunks of this problem in a different order every time
    for _ in range(10):
        ok, cost3 = cp.evaluate_device()
        assert ok and cost3 == cost
