"""CPU self-tests of oracle/exact.py: the bit budget that makes the moment references exact, the KKT certificates of the exact
NNLS, the exact NNLS against brute-force enumeration of passive sets, and the fp64 mirror of wls_nnls_kernel."""
import os
from fractions import Fraction

import numpy as np
import pytest

from oracle import exact as ex

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_bit_budget_is_exact_and_tight():
    rs = np.random.RandomState(0)
    bits, w_max = 10, 255
    # y = x: d z_p z_q <= 255 * 2^20 -> 28 bits per term, 2^20 rows fit in 48 bits
    assert ex.moment_bit_budget(1 << 20, bits, w_max, False) <= 53
    # y = d x: 255^3 2^20 -> 44 bits per term: at most 2^9 rows
    assert ex.moment_bit_budget(1 << 9, bits, w_max, True) <= 53
    assert ex.moment_bit_budget(1 << 10, bits, w_max, True) > 53
    # the int64 reference equals a Fraction sum, and fp64 sums of its terms in any order are exact within the budget
    M, N, K = 37, 3, 4
    X, R = ex.dyadic(rs, (M, N), bits), ex.dyadic(rs, (M, K), bits)
    D = rs.randint(0, w_max + 1, size=(M, N)).astype(np.float64)
    for y_is_dx in (False, True):
        mom = ex.wls_moments_exact(X, D, R, y_is_dx, bits)
        j = 2
        z = [np.ones(M), D[:, j] * X[:, j] if y_is_dx else X[:, j]] + [R[:, k] for k in range(K)]
        for p, q in ((0, 0), (1, 1), (1, 3), (5, 2)):
            terms = D[:, j] * z[p] * z[q]
            want = sum(Fraction(float(t)) for t in terms) * (1 << 2 * bits)
            assert want == int(mom[p, q, j])
            shuffled = terms[rs.permutation(M)]
            assert float(np.sum(shuffled)) * (1 << 2 * bits) == int(mom[p, q, j])


def test_moment_reference_rejects_non_dyadic_input():
    X = np.full((3, 1), 0.1)
    with pytest.raises(AssertionError, match="dyadic"):
        ex.wls_moments_exact(X, np.ones((3, 1)), np.zeros((3, 1)), False, 10)


def _random_problem(rs, K, zeros):
    """Exact moments of a small WLS problem whose true proportions have `zeros` exact zeros."""
    M, bits = 64, 10
    R = ex.dyadic(rs, (M, K), bits)
    a = np.zeros(K)
    a[rs.permutation(K)[: K - zeros]] = rs.dirichlet(np.ones(K - zeros))
    X = np.round(np.clip(R @ a + rs.normal(0, 0.05, M), 0, 1)[:, None] * 1024) / 1024
    D = rs.randint(1, 40, size=(M, 1)).astype(np.float64)
    return ex.centred_normal_equations(ex.wls_moments_exact(X, D, R, False, bits), 0)


@pytest.mark.parametrize("K", [1, 2, 3, 5, 8])
def test_nnls_exact_matches_brute_force(K):
    rs = np.random.RandomState(K)
    for trial in range(4):
        G, b = _random_problem(rs, K, zeros=min(trial, K - 1))
        got = ex.nnls_exact(G, b)
        x_bf, P_bf = ex.nnls_brute_force(G, b)
        assert got["x"] == x_bf and got["passive"] == P_bf
        assert got["kkt"][0] and got["kkt"][3] == 0


def test_kkt_certificate_rejects_non_optimal_points():
    G = [[Fraction(2), Fraction(1)], [Fraction(1), Fraction(2)]]
    b = [Fraction(1), Fraction(-1)]
    x = ex.nnls_exact(G, b)["x"]
    assert x == [Fraction(1, 2), Fraction(0)]
    assert not ex.kkt_certificate(G, b, [Fraction(1, 3), Fraction(0)])[0]          # stationarity fails
    assert not ex.kkt_certificate(G, b, [Fraction(1, 2), Fraction(1, 10)])[0]      # a positive entry with w != 0
    assert not ex.kkt_certificate(G, b, [Fraction(0), Fraction(0)])[0]             # w_0 > 0 on the active set


def test_nnls_exact_records_inner_loop_removal():
    """A problem on which Lawson-Hanson must drop a variable it added: the case the GPU test uses."""
    G = [[Fraction(1), Fraction(9, 10)], [Fraction(9, 10), Fraction(1)]]
    b = [Fraction(1), Fraction(1, 2)]
    # the unconstrained solution has x_1 < 0; x_0 enters first, x_1 never does
    assert ex.nnls_exact(G, b)["passive"] == [0]
    G3, b3 = REMOVAL_CASE
    r = ex.nnls_exact([[Fraction(v) for v in row] for row in G3], [Fraction(v) for v in b3])
    assert r["removals"] >= 1 and r["passive"] == [1, 2] and r["x"] == [0, Fraction(4, 39), Fraction(2, 3)]
    # the device algorithm takes the same path: the fp64 mirror steps through its inner loop once
    mom = np.zeros((5, 5, 1))
    mom[0, 0, 0] = 1.0
    mom[2:, 2:, 0] = G3
    mom[1, 2:, 0] = mom[2:, 1, 0] = b3
    _, status, raw, it, _ = ex.wls_nnls_mirror(mom, 0, 3, 1)
    assert status == 0 and it == 1 and raw[0] == 0.0


REMOVAL_CASE = ([[57, 32, 45], [32, 26, 26], [45, 26, 38]], [31, 20, 28])    # G = A^T A, b = A^T y for small integer A, y


def test_nnls_mirror_flags_the_iteration_limit():
    """wls_nnls_kernel stops its inner loop after 3 K steps.  On these (numerically singular) normal equations the mirror reaches
    the limit with a negative coefficient and no collinearity flag: the kernel now reports status 4 (DMF_E_STATE) instead of
    returning a negative proportion."""
    mom = np.load(os.path.join(GOLDEN, "wls_nnls_iteration_cap.npy"))
    K = mom.shape[0] - 2
    with np.errstate(all="ignore"):
        x, status, raw, it, capped = ex.wls_nnls_mirror(mom, 0, K, 1)
    assert capped and status == 4 and it == 3 * K and raw.min() < 0


def test_nnls_mirror_matches_exact_on_well_conditioned_problems():
    rs = np.random.RandomState(7)
    for K in (2, 4, 6):
        M, bits = 200, 10
        R = ex.dyadic(rs, (M, K), bits)
        a = rs.dirichlet(np.ones(K))
        a[0] = 0.0
        X = np.round(np.clip(R @ (a / a.sum()), 0, 1)[:, None] * 1024) / 1024
        D = rs.randint(1, 40, size=(M, 1)).astype(np.float64)
        mom = ex.wls_moments_exact(X, D, R, False, bits)
        r = ex.nnls_exact(*ex.centred_normal_equations(mom, 0))
        x, status, raw, _, _ = ex.wls_nnls_mirror(mom.astype(np.float64), 0, K, M)
        assert status == 0 and [p for p in range(K) if raw[p] > 0] == r["passive"]
        xs = np.array([float(v) for v in r["x"]])
        assert np.abs(raw - xs).max() <= 100 * K * float(r["cond"]) * ex.EPS * np.abs(xs).max()


def test_nndsvd_rule_tie_and_zero_sigma():
    U = np.array([[0.5, 0.5], [0.5, -0.5], [0.5, 0.5], [0.5, -0.5]])
    Vh = np.array([[0.6, 0.8], [0.5, -0.5]])
    W, H, pos = ex.nndsvd_rule_mp(U, np.array([4.0, 0.0]), Vh, 2)
    assert pos == [True, True]                                # |u+||v+| == |u-||v-| exactly: the positive pattern
    assert all(W[m][1] == 0 for m in range(4)) and all(H[1][j] == 0 for j in range(2))
    assert float(W[0][0]) == 1.0 and float(H[0][1]) == 1.6
