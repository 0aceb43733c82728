"""CPU test of the rule that holds a render to the oracle channel by channel (tests/util.py assert_oracle_exact), on small
hand-made arrays: it lets through exactly the 1-LSB differences of two linear colours, 1e-9 apart, on either side of a
quantisation step, and nothing else."""
import numpy as np
import pytest

from tests.util import assert_oracle_exact, to_int_c


def oracle(linear):
    linear = np.asarray(linear, dtype=np.float64).reshape(1, -1, 3)
    return {"rgb_f64": linear, "rgb_u8": to_int_c(linear)}


# two pixels: a mid-level colour, and one whose red channel sits just below the step 99 -> 100 (255 * c = 100 - 1e-10)
BELOW = (100 - 1e-10) / 255
REF = [[0.5, 0.25, 0.125], [BELOW, 0.0, 1.0]]


def device(linear, pixels=None):
    linear = np.asarray(linear, dtype=np.float64).reshape(1, -1, 3)
    return (to_int_c(linear) if pixels is None else pixels), linear


def test_equal_colours_pass():
    assert assert_oracle_exact(*device(REF), oracle(REF)) == 0


def test_non_finite_colours_are_equal_to_themselves():
    ref = [[np.nan, np.inf, -np.inf], [0.5, 2.0, -1.0]]
    assert assert_oracle_exact(*device(ref), oracle(ref)) == 0


def test_a_straddled_step_may_differ_by_one():
    dev = [[0.5, 0.25, 0.125], [(100 + 1e-10) / 255, 0.0, 1.0]]   # 8e-13 relative above the oracle: the other side
    px, lin = device(dev)
    assert int(px[0, 1, 0]) - int(oracle(REF)["rgb_u8"][0, 1, 0]) == 1
    assert assert_oracle_exact(px, lin, oracle(REF)) == 1


def test_one_lsb_away_from_a_step_fails():
    ref = oracle(REF)
    ref["rgb_u8"] = ref["rgb_u8"].copy()
    ref["rgb_u8"][0, 0, 1] -= 1    # oracle bytes one below the device's, though the colours are equal and far from a step
    with pytest.raises(AssertionError, match="off the oracle's"):
        assert_oracle_exact(*device(REF), ref)


def test_a_difference_of_two_fails_even_at_a_step():
    dev = [[0.5, 0.25, 0.125], [(100 + 1e-10) / 255, 0.0, 1.0]]
    ref = oracle(REF)
    ref["rgb_u8"] = ref["rgb_u8"].copy()
    ref["rgb_u8"][0, 1, 0] -= 1    # 98: two below the device's 100
    with pytest.raises(AssertionError, match="straddle"):
        assert_oracle_exact(*device(dev), ref)
    px, lin = device(REF)
    px = px.copy()
    px[0, 0, 0] += 2
    with pytest.raises(AssertionError):
        assert_oracle_exact(px, lin, oracle(REF))


def test_bytes_that_are_not_the_devices_own_quantisation_fail():
    px, lin = device(REF)
    px = px.copy()
    px[0, 1, 0] += 1    # 100: the oracle's neighbour value at a step, but not toIntC of this linear colour
    with pytest.raises(AssertionError, match="not toIntC"):
        assert_oracle_exact(px, lin, oracle(REF))


def test_a_linear_colour_1e_6_off_fails():
    dev = np.array(REF)
    dev[0, 2] *= 1 + 1e-6   # same byte (31), but far beyond the summation order's roundings
    px, lin = device(dev)
    assert np.array_equal(px, oracle(REF)["rgb_u8"])
    with pytest.raises(AssertionError, match="linear channels"):
        assert_oracle_exact(px, lin, oracle(REF))
