"""The oracle's exact-sum mode (orc_set_sum_mode(1), oracleapi.sum_mode), which the GPU parity checks compare against: the group's
Wiener weight sum and useSD's mean / square sums are added in double and rounded to float once. Mode 0, the reference's serial
float sums, stays the default; the reference pins run in it."""
import numpy as np
import pytest

import golden_inputs as gi
from gpucheck import estimate

K, N = 16, 32
BOUND = N * 9 * K * K * 2.0 ** -24      # a serial float sum of the N * A * k^2 non-negative terms of a group, relative


@pytest.fixture(scope="module")
def inputs(oracle):
    _, _, sym = gi.pad_inputs(40, 48, 25.0)
    z = np.zeros_like(sym)
    mask, proc = np.ones(9, np.uint32), np.zeros(9, np.uint32)
    on, od = oracle.run_pass(1, sym, None, z, z, mask, proc, 4, 3, 25.0, 2.7, 18, 6, 16, 8, 4, oracle.ID, oracle.SADCT, oracle.HAAR)
    return sym, estimate(on, od, sym), z, mask, proc


def run(oracle, inputs, step, mode, useSD=0):
    sym, basic, z, mask, proc = inputs
    oracle.lib().orc_set_use_sd(useSD)
    try:
        with oracle.sum_mode(mode):
            return oracle.run_pass(step, sym, basic if step == 2 else None, z, z, mask, proc, 4, 3, 25.0, 2.7 if step == 1 else 0.0,
                                   18, 6, K, N, 4, oracle.DCT, oracle.SADCT, oracle.HAAR)
    finally:
        oracle.lib().orc_set_use_sd(0)


def rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def test_step1_bit_identical(oracle, inputs):
    """Step 1's weight is a count of coefficients, exact in float: the mode changes nothing."""
    n0, d0 = run(oracle, inputs, 1, 0)
    n1, d1 = run(oracle, inputs, 1, 1)
    assert np.array_equal(n0, n1) and np.array_equal(d0, d1)


@pytest.mark.parametrize("step,useSD", [(2, 0), (1, 1), (2, 1)])
def test_sums_move_within_the_float_bound(oracle, inputs, step, useSD):
    """The modes differ (the float sums do round), and by no more than the rounding bound of a serial float sum of the group."""
    n0, d0 = run(oracle, inputs, step, 0, useSD)
    n1, d1 = run(oracle, inputs, step, 1, useSD)
    for a, b in ((n0, n1), (d0, d1)):
        assert 0.0 < rel(a, b) <= BOUND, (rel(a, b), BOUND)


def test_mode_restored_after_an_exception(oracle, inputs):
    n0, d0 = run(oracle, inputs, 2, 0)
    with pytest.raises(RuntimeError):
        with oracle.sum_mode(1):
            raise RuntimeError("inside the block")
    n, d = oracle.run_pass(2, inputs[0], inputs[1], inputs[2], inputs[2], inputs[3], inputs[4], 4, 3, 25.0, 0.0, 18, 6, K, N, 4,
                           oracle.DCT, oracle.SADCT, oracle.HAAR)
    assert np.array_equal(n, n0) and np.array_equal(d, d0)
