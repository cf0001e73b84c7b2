"""Host-side bookkeeping of the device ADMM loop: the control block a solve starts from and the status it ends with
(no GPU needed)."""
import numpy as np
import pytest

from gglasso_b200._engine import boyd_status, control_block
from gglasso_b200._lib import CTRL_STRIDE, HIST_STRIDE, C_DONE, C_ITER, C_LAM1, C_LAM2, C_RHO, C_XSCALE


def _ctrl(done, iters):
    c = np.zeros(CTRL_STRIDE)
    c[C_DONE], c[C_ITER] = done, iters
    return c


def _hist(rows, cap=8):
    """residual history of ``cap`` iterations: ``rows`` = (r, s, eps_pri, eps_dual) of the executed ones, the rest
    holds values no status may read"""
    h = np.full((cap, HIST_STRIDE), -1.0)
    h[:len(rows), :4] = rows
    h[:len(rows), 4] = 1.0
    return h


# (done flag, last (r, s, eps_pri, eps_dual)) -> status; the done flag wins over the last residuals
OUTCOMES = [
    (1, (2.0, 3.0, 1.0, 1.0), "optimal"),
    (0, (1.0, 3.0, 1.0, 1.0), "primal optimal"),
    (0, (2.0, 0.5, 1.0, 1.0), "dual optimal"),
    (0, (2.0, 3.0, 1.0, 1.0), "max iterations reached"),
]


@pytest.mark.parametrize("done,last,expected", OUTCOMES)
def test_boyd_status_outcomes(done, last, expected):
    rows = [(5.0, 4.0, 0.1, 0.1), (3.0, 6.0, 0.1, 0.1), last]
    status, residual = boyd_status(_ctrl(done, len(rows)), _hist(rows))
    assert status == expected
    np.testing.assert_array_equal(residual, [5.0, 6.0, max(last[0], last[1])])


def test_boyd_status_mixed_batch():
    """one control row and history per problem, as run_admm reads them: each problem's own iteration count decides
    which history row is its last and how long its residual series is"""
    cap = 8
    ctrl = np.zeros((len(OUTCOMES), CTRL_STRIDE))
    hist = np.zeros((len(OUTCOMES), cap, HIST_STRIDE))
    for q, (done, last, _) in enumerate(OUTCOMES):
        n = q + 2
        rows = [(10.0 + i, 20.0 + i, 0.1, 0.1) for i in range(n - 1)] + [last]
        ctrl[q] = _ctrl(done, n)
        hist[q] = _hist(rows, cap)
    for q, (_, last, expected) in enumerate(OUTCOMES):
        status, residual = boyd_status(ctrl[q], hist[q])
        n = q + 2
        assert status == expected
        assert len(residual) == n
        np.testing.assert_array_equal(residual[:-1], 20.0 + np.arange(n - 1))
        assert residual[-1] == max(last[0], last[1])


def test_control_block_without_lambdas():
    c = control_block(3, 0.7)
    assert c.shape == (3, CTRL_STRIDE) and c.dtype == np.float64
    expected = np.zeros((3, CTRL_STRIDE))
    expected[:, C_RHO] = 0.7
    expected[:, C_XSCALE] = 1.0                 # no pending rescale of the scaled dual
    np.testing.assert_array_equal(c, expected)


def test_control_block_scalar_lambdas():
    c = control_block(2, 1.0, (0.05, 0.01))
    np.testing.assert_array_equal(c[:, C_LAM1], [0.05, 0.05])
    np.testing.assert_array_equal(c[:, C_LAM2], [0.01, 0.01])
    np.testing.assert_array_equal(c[:, C_RHO], 1.0)
    np.testing.assert_array_equal(c[:, C_XSCALE], 1.0)


def test_control_block_per_problem_lambdas():
    l1 = np.array([0.3, 0.01, 0.15])
    c = control_block(3, 2.0, (l1, 0.02))
    np.testing.assert_array_equal(c[:, C_LAM1], l1)
    np.testing.assert_array_equal(c[:, C_LAM2], 0.02)
    c = control_block(3, 2.0, (0.1, [0.1, 0.2, 0.3]))
    np.testing.assert_array_equal(c[:, C_LAM1], 0.1)
    np.testing.assert_array_equal(c[:, C_LAM2], [0.1, 0.2, 0.3])


def test_control_block_rejects_lambda_count_mismatch():
    with pytest.raises(ValueError):
        control_block(3, 1.0, (np.array([0.1, 0.2]), 0.01))
    with pytest.raises(ValueError):
        control_block(2, 1.0, (0.1, np.array([0.1, 0.2, 0.3])))
