"""CPU tests of the MT19937 jump-ahead (demethify_b200/mt_jump.py) that the row-sharded bicross-validation draws its rows of the
fold masks with: jumped states continue numpy's legacy stream bit for bit, and every rank's rows of a mask are the rows of the full
draw."""
import numpy as np
import pytest

from demethify_b200 import mt_jump
from demethify_b200.sharded import row_range

SEEDS = [0, 1, 2**32 - 1, [5]]


def test_stored_polynomial_is_berlekamp_massey_result():
    p = mt_jump.characteristic_polynomial()
    assert p.bit_length() - 1 == 19937
    assert p == sum(1 << k for k in mt_jump.PHI_TERMS)
    assert mt_jump._phi_source() == "PHI_TERMS = (" + ", ".join(map(str, mt_jump.PHI_TERMS)) + ")"


def test_jump_poly_is_x_to_the_j_mod_phi():
    # x^(a + b) = x^a x^b: two jumps compose into one
    for a, b in ((20000, 7), (19937, 19937), (123457, 10 ** 6)):
        pa, pb = mt_jump.jump_poly(a), mt_jump.jump_poly(b)
        prod = 0
        for k in range(pb.bit_length()):
            if (pb >> k) & 1:
                prod ^= pa << k
        assert mt_jump._mod_phi(prod) == mt_jump.jump_poly(a + b)
    with pytest.raises(ValueError):
        mt_jump.jump_poly(-1)


@pytest.mark.parametrize("seed", SEEDS, ids=str)
@pytest.mark.parametrize("k", [0, 1, 311, 312, 313, 10_000])
def test_jumped_state_continues_the_stream(seed, k):
    """From the state after k doubles, a jump by J words gives the next 1 000 doubles of one long random_sample, bit for bit."""
    rs = np.random.RandomState(seed)
    rs.random_sample(k)
    start = rs.get_state()
    for J in (0, 2, 622, 624, 626, 1248, 2 * 10 ** 7):
        other = np.random.RandomState()
        other.set_state(mt_jump.jump_state(start, J))
        got = other.random_sample(1000)
        rs.set_state(start)
        rs.random_sample(J // 2)
        want = rs.random_sample(1000)
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), (seed, k, J)


def test_odd_jump_and_words():
    """A jump by an odd number of words lands between the two words of a double: compare 32-bit words."""
    rs = np.random.RandomState(3)
    start = rs.get_state()
    want = rs.randint(0, 2 ** 32, size=5000, dtype=np.uint64)       # one word per value for the full 32-bit range
    for J in (1, 623, 625, 3001):
        other = np.random.RandomState()
        other.set_state(mt_jump.jump_state(start, J))
        assert np.array_equal(other.randint(0, 2 ** 32, size=100, dtype=np.uint64), want[J:J + 100])


@pytest.mark.parametrize("seed", SEEDS, ids=str)
def test_mask_rows_are_the_ranks_rows_of_the_full_mask(seed):
    for M, N in ((7, 5), (1, 3), (401, 9)):
        rs = np.random.RandomState(seed)
        rs.random_sample(17)                                      # a state off the regeneration boundary
        start = rs.get_state()
        full = rs.rand(M, N) < 0.3
        after = rs.random_sample(10)
        for world in (1, 2, 3, 8):
            for rank in range(world):
                lo, hi = row_range(M, rank, world)                # M = 1 leaves ranks without rows
                rows, end = mt_jump.mask_rows(start, M, N, lo, hi, 0.3)
                assert rows.shape == (hi - lo, N) and np.array_equal(rows, full[lo:hi])
                other = np.random.RandomState()
                other.set_state(end)
                assert np.array_equal(other.random_sample(10), after)
