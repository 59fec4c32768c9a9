"""GPU tests of the reference's solver steps called one at a time (run with -m gpu on the B200 box): update_u, update_alpha and
frank_wolfe_nmf of demethify_b200.deconvolution against the oracle's restatement of deconvolution.py:81-102 / :280-302, outer loops
composed from them against the golden vectors and the oracle's solvers, resident-problem inputs, fp32 mode and the error paths."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SHAPES = [(1, 1, 1, 1), (350, 10, 5, 1), (5000, 64, 6, 2), (3000, 300, 6, 2), (1200, 24, 20, 9)]
N_ITER2 = [0, 1, 20]
TOL = 1e-10


def _a_after(n):
    a = 1.0
    for _ in range(n):
        a = (1 + np.sqrt(1 + 4 * a * a)) / 2           # deconvolution.py:84
    return a


A1S = [1.0, _a_after(37), 2.5]
# l_prev / l: 1.3 leaves beta = (a - 1) / a_next on the first step, 0.2 lets 0.9999 sqrt(l_prev / l) bind for a > 1
RATIOS = [1.3, 0.2]


@pytest.fixture(scope="module")
def dec():
    import torch
    assert torch.cuda.is_available()
    import __graft_entry__ as g
    g.build()
    from demethify_b200 import deconvolution
    return deconvolution


@pytest.fixture(scope="module")
def orc():
    from oracle import bssmf_numpy
    return bssmf_numpy


def synth(seed, M, N, K, n_u, depth=50):
    """X, D (int64), R_trunc, a current (u, alpha) and a previous (u_, alpha_) iterate."""
    rs = np.random.RandomState(seed)
    a = rs.uniform(0.2, 1.0, size=K + n_u)
    Rf = rs.beta(a, a, size=(M, K + n_u))
    A = rs.dirichlet(np.ones(K + n_u), N).T
    D = rs.poisson(depth, size=(M, N)) + 1
    X = rs.binomial(D, np.clip(Rf @ A, 0, 1)) / D
    u = rs.uniform(size=(M, n_u))
    u_prev = np.clip(u + 0.05 * rs.standard_normal((M, n_u)), 0, 1)
    A_prev = rs.dirichlet(np.ones(K + n_u), N).T
    return X, D.astype(np.int64), np.ascontiguousarray(Rf[:, :K]), u, A, u_prev, A_prev


def snapshot(*arrays):
    return [np.array(a, copy=True) for a in arrays]


def unchanged(before, *arrays):
    return all(np.array_equal(b, a, equal_nan=True) for b, a in zip(before, arrays))


def on_simplex(A):
    return A.min() >= 0 and np.abs(A.sum(0) - 1).max() <= 1e-12


# ------------------------------------------------------------------------------- single steps vs the oracle
@pytest.mark.parametrize("ratio", RATIOS)
@pytest.mark.parametrize("a1", A1S)
@pytest.mark.parametrize("n_iter2", N_ITER2)
@pytest.mark.parametrize("M,N,K,n_u", SHAPES)
def test_update_u_vs_oracle(dec, orc, M, N, K, n_u, n_iter2, a1, ratio):
    X, D, Rk, u, A, u_prev, _ = synth(M + 3 * N + K, M, N, K, n_u)
    l_w = np.linalg.norm(A[-n_u:]) ** 2 * D.max() ** 2
    l_w_ = ratio * l_w
    before = snapshot(u, A, u_prev, X, D, Rk)
    uo, uo_, a1o, lo_ = orc.u_inner_loop(u.copy(), A, n_iter2, a1, l_w_, l_w, u_prev.copy(), X, Rk, n_u, D.astype(float))
    ug, ug_, a1g, lg_ = dec.update_u(u, A, n_iter2, a1, l_w_, l_w, u_prev, X, Rk, n_u, D)
    assert unchanged(before, u, A, u_prev, X, D, Rk)
    assert a1g == a1o and lg_ == lo_
    if n_iter2 == 0:
        assert np.array_equal(ug, u) and np.array_equal(ug_, u_prev) and a1g == a1 and lg_ == l_w_
    assert ug.shape == (M, n_u) and ug_.shape == (M, n_u)
    assert np.abs(ug - uo).max() <= TOL and np.abs(ug_ - uo_).max() <= TOL


@pytest.mark.parametrize("ratio", RATIOS)
@pytest.mark.parametrize("a2", A1S)
@pytest.mark.parametrize("n_iter2", N_ITER2)
@pytest.mark.parametrize("M,N,K,n_u", SHAPES + [(700, 12, 4, 3), (500, 9, 0, 1)])    # Kt = 7 and Kt = 1: odd, the last reference-free
def test_update_alpha_vs_oracle(dec, orc, M, N, K, n_u, n_iter2, a2, ratio):
    X, D, Rk, u, A, _, A_prev = synth(M + 5 * N + K, M, N, K, n_u)
    R = np.hstack((Rk, u))
    l_h = np.linalg.norm(R) ** 2 * D.max() ** 2
    l_h_ = ratio * l_h
    before = snapshot(A, A_prev, R, X, D)
    ao, ao_, a2o, lo_ = orc.alpha_inner_loop(n_iter2, A.copy(), a2, l_h_, l_h, A_prev.copy(), R, D.astype(float), X)
    ag, ag_, a2g, lg_ = dec.update_alpha(n_iter2, A, a2, l_h_, l_h, A_prev, R, D, X)
    assert unchanged(before, A, A_prev, R, X, D)
    assert a2g == a2o and lg_ == lo_
    if n_iter2 == 0:
        assert np.array_equal(ag, A) and np.array_equal(ag_, A_prev) and a2g == a2 and lg_ == l_h_
    else:
        assert on_simplex(ag)
    assert np.abs(ag - ao).max() <= TOL and np.abs(ag_ - ao_).max() <= TOL


@pytest.mark.parametrize("n_iter2", [1, 50])
@pytest.mark.parametrize("purity_kind", ["zero", "one", "random"])
@pytest.mark.parametrize("n_u", [1, 2])
@pytest.mark.parametrize("K", [1, 6])
def test_frank_wolfe_nmf_vs_oracle(dec, orc, K, n_u, purity_kind, n_iter2):
    M, N = 2000, 24
    X, D, Rk, u, A, _, _ = synth(K * 10 + n_u, M, N, K, n_u)
    purity = {"zero": np.zeros(N), "one": np.ones(N), "random": np.random.RandomState(K).uniform(size=N)}[purity_kind]
    H1, H2 = A[:K] * purity / A[:K].sum(0), A[K:] * (1 - purity) / A[K:].sum(0)
    before = snapshot(Rk, u, X, H1, H2, purity, D)
    h1o, h2o = orc.frank_wolfe_alpha(Rk, u, X, H1, H2, purity, n_iter2, D.astype(float))
    h1, h2 = dec.frank_wolfe_nmf(Rk, u, X, H1, H2, purity, n_iter2, D)
    assert unchanged(before, Rk, u, X, H1, H2, purity, D)
    assert h1.shape == (K, N) and h2.shape == (n_u, N)
    assert np.abs(h1 - h1o).max() <= TOL and np.abs(h2 - h2o).max() <= TOL


# ------------------------------------------------------------------------------- outer loops composed from the steps
def test_partial_reference_loop_from_steps(dec, shipped, live):
    """mdwbssmf_deconv (deconvolution.py:190-223) written from update_u, update_alpha and cost_f_w: the momentum state the steps
    return carries across calls, so the loop stops at the reference's outer iteration with the reference's alpha."""
    X, D, Rk, n_u = shipped["X"], shipped["D"], shipped["Rk"], 1
    u, R, A = dec.init_BSSMF_md("uniform_", X, D, Rk, n_u, seed=1)
    a1 = a2 = 1.0
    u_, A_ = u.copy(), A.copy()
    dmax2 = D.max() ** 2
    l_w = np.linalg.norm(A[-n_u:]) ** 2 * dmax2
    l_w_ = l_w
    l_h = np.linalg.norm(R) ** 2 * dmax2
    l_h_ = l_h
    cf = dec.cost_f_w(X, R, A, D)
    n_outer = 0
    for _ in range(10000):
        cf0 = cf
        u, u_, a1, l_w_ = dec.update_u(u, A, 20, a1, l_w_, l_w, u_, X, Rk, n_u, D)
        R = np.hstack((Rk, u.reshape(-1, n_u)))
        l_h = np.linalg.norm(R) ** 2 * dmax2
        A, A_, a2, l_h_ = dec.update_alpha(20, A, a2, l_h_, l_h, A_, R, D, X)
        l_w = np.linalg.norm(A[-n_u:]) ** 2 * dmax2
        cf = dec.cost_f_w(X, R, A, D)
        n_outer += 1
        if abs(cf - cf0) < 1e-2:
            break
    assert n_outer == len(live["pr1_costs"]) - 1
    assert np.abs(A - live["pr1_a"]).max() <= 1e-6 and np.abs(A - shipped["partial_alpha"]).max() <= 1e-6


def test_purity_loop_from_steps(dec, orc, shipped):
    """mdwbssmf_deconv_p (deconvolution.py:305-337) written from update_u and frank_wolfe_nmf, three outer iterations."""
    X, D, Rk, n_u = shipped["X"], shipped["D"], shipped["Rk"], 1
    pur = 1 - shipped["purity_pct"] / 100.0
    u0, R0, a0 = dec.init_BSSMF_md_p("uniform_", X, D, Rk, n_u, pur, seed=1)
    uo, ao = orc.solve_purity(u0.copy(), R0, a0.copy(), X, D.astype(float), Rk, n_u, pur, n_iter1=3, n_iter2=50, tol=0.0)
    u, u_, a1 = u0, u0.copy(), 1.0
    A1, A2 = a0[:-n_u], a0[-n_u:]
    dmax2 = D.max() ** 2
    l_w = np.linalg.norm(A2) ** 2 * dmax2
    l_w_ = l_w
    for _ in range(3):
        u, u_, a1, l_w_ = dec.update_u(u, np.vstack((A1, A2)), 50, a1, l_w_, l_w, u_, X, Rk, n_u, D)
        A1, A2 = dec.frank_wolfe_nmf(Rk, u, X, A1, A2, pur, 50, D)
        l_w = np.linalg.norm(A2) ** 2 * dmax2
    assert np.abs(u - uo).max() <= TOL and np.abs(np.vstack((A1, A2)) - ao).max() <= TOL


# ------------------------------------------------------------------------------- resident problem, fp32
def test_resident_problem_is_bit_identical(dec):
    from demethify_b200.engine import DeviceProblem
    M, N, K, n_u = 5000, 64, 6, 2
    X, D, Rk, u, A, u_prev, A_prev = synth(17, M, N, K, n_u)
    prob = DeviceProblem(X, D, Rk)
    l_w = np.linalg.norm(A[-n_u:]) ** 2 * D.max() ** 2
    ref = dec.update_u(u, A, 20, 2.5, 0.2 * l_w, l_w, u_prev, X, Rk, n_u, D)
    res = dec.update_u(u, A, 20, 2.5, 0.2 * l_w, l_w, u_prev, prob, None, n_u, None)
    assert all(np.array_equal(r, s) for r, s in zip(ref, res))
    R = np.hstack((Rk, u))
    l_h = np.linalg.norm(R) ** 2 * D.max() ** 2
    ref = dec.update_alpha(20, A, 2.5, 0.2 * l_h, l_h, A_prev, R, D, X)
    res = dec.update_alpha(20, A, 2.5, 0.2 * l_h, l_h, A_prev, R, None, prob)
    assert all(np.array_equal(r, s) for r, s in zip(ref, res))
    pur = np.random.RandomState(2).uniform(size=N)
    H1, H2 = A[:K] * pur, A[K:] * (1 - pur) / A[K:].sum(0)
    ref = dec.frank_wolfe_nmf(Rk, u, X, H1, H2, pur, 30, D)
    res = dec.frank_wolfe_nmf(None, u, prob, H1, H2, pur, 30, None)
    assert all(np.array_equal(r, s) for r, s in zip(ref, res))
    assert prob.K == K          # update_alpha's per-call R leaves the resident problem's R_trunc alone


def test_fp32_steps(dec, orc):
    import demethify_b200
    M, N, K, n_u = 6000, 32, 6, 2
    X, D, Rk, u, A, u_prev, A_prev = synth(11, M, N, K, n_u)
    Df = D.astype(float)
    l_w = np.linalg.norm(A[-n_u:]) ** 2 * D.max() ** 2
    R = np.hstack((Rk, u))
    l_h = np.linalg.norm(R) ** 2 * D.max() ** 2
    uo, uo_, a1o, _ = orc.u_inner_loop(u.copy(), A, 20, 1.0, l_w, l_w, u_prev.copy(), X, Rk, n_u, Df)
    ao, ao_, a2o, _ = orc.alpha_inner_loop(20, A.copy(), 1.0, l_h, l_h, A_prev.copy(), R, Df, X)
    demethify_b200.set_precision("fp32")
    try:
        ug, ug_, a1g, _ = dec.update_u(u, A, 20, 1.0, l_w, l_w, u_prev, X, Rk, n_u, D)
        ag, ag_, a2g, _ = dec.update_alpha(20, A, 1.0, l_h, l_h, A_prev, R, D, X)
    finally:
        demethify_b200.set_precision("fp64")
    assert a1g == a1o and a2g == a2o          # the momentum scalars stay fp64
    assert np.abs(ug - uo).max() <= 1e-3 and np.abs(ug_ - uo_).max() <= 1e-3
    assert np.abs(ag - ao).max() <= 1e-4 and np.abs(ag_ - ao_).max() <= 1e-4


# ------------------------------------------------------------------------------- errors
def test_non_finite_input_raises(dec):
    from demethify_b200 import _lib
    X, D, Rk, u, A, _, A_prev = synth(7, 300, 5, 3, 1)
    X = X.copy(); X[10, 2] = np.nan
    R = np.hstack((Rk, u))
    l_h = np.linalg.norm(R) ** 2 * D.max() ** 2
    before = snapshot(X, A, A_prev, R)
    with pytest.raises(_lib.DmfError, match="non-finite"):
        dec.update_alpha(5, A, 1.0, l_h, l_h, A_prev, R, D, X)
    assert unchanged(before, X, A, A_prev, R)


def test_unsupported_width_keeps_the_library_message(dec):
    from demethify_b200 import _lib
    X, D, Rk, u, A, u_prev, A_prev = synth(3, 200, 6, 25, 7)        # even(25) + even(7) = 34
    with pytest.raises(_lib.DmfError, match=r"K \+ n_u \(even padded\) > 32"):
        dec.update_u(u, A, 2, 1.0, 1.0, 1.0, u_prev, X, Rk, 7, D)
    X, D, Rk, u, A, u_prev, A_prev = synth(3, 200, 6, 26, 7)        # R with Kt = 33 columns is split 32 + 1: even(32) + even(1) = 34
    with pytest.raises(_lib.DmfError, match=r"K \+ n_u \(even padded\) > 32"):
        dec.update_alpha(2, A, 1.0, 1.0, 1.0, A_prev, np.hstack((Rk, u)), D, X)


def test_mismatched_shapes_raise_value_error(dec):
    M, N, K, n_u = 300, 8, 4, 2
    X, D, Rk, u, A, u_prev, A_prev = synth(5, M, N, K, n_u)
    R = np.hstack((Rk, u))
    pur = np.full(N, 0.5)
    bad = [
        lambda: dec.update_u(u[:-1], A, 2, 1.0, 1.0, 1.0, u_prev, X, Rk, n_u, D),
        lambda: dec.update_u(u, A, 2, 1.0, 1.0, 1.0, u_prev[:, :1], X, Rk, n_u, D),
        lambda: dec.update_u(u, A[:, :-1], 2, 1.0, 1.0, 1.0, u_prev, X, Rk, n_u, D),
        lambda: dec.update_u(u, A, 2, 1.0, 1.0, 1.0, u_prev, X, Rk[:-1], n_u, D),
        lambda: dec.update_alpha(2, A, 1.0, 1.0, 1.0, A_prev[:-1], R, D, X),
        lambda: dec.update_alpha(2, A[:-1], 1.0, 1.0, 1.0, A_prev[:-1], R, D, X),
        lambda: dec.update_alpha(2, A, 1.0, 1.0, 1.0, A_prev, R[:-1], D, X),
        lambda: dec.update_alpha(2, A, 1.0, 1.0, 1.0, A_prev, R, D[:, :-1], X),
        lambda: dec.frank_wolfe_nmf(Rk, u, X, A[:K], A[K:-1], pur, 2, D),
        lambda: dec.frank_wolfe_nmf(Rk, u[:-1], X, A[:K], A[K:], pur, 2, D),
        lambda: dec.frank_wolfe_nmf(Rk, u, X, A[:K - 1], A[K:], pur, 2, D),
    ]
    for call in bad:
        with pytest.raises(ValueError):
            call()


def test_set_step_state_checks_and_writes_only_its_scalars():
    import __graft_entry__ as g
    g.build()
    from demethify_b200 import _lib
    from demethify_b200.engine import DeviceProblem, FitBatch
    X, D, Rk, u, A, _, _ = synth(1, 500, 10, 4, 2)
    b = FitBatch(DeviceProblem(X, D, Rk), 2, [u, u[::-1].copy()], [A, A], engine="stream")
    b.pass_init()
    s0 = b.states()
    for which, a, l, l_old in [(2, 1.0, 1.0, 1.0), (-1, 1.0, 1.0, 1.0), (0, 1.0, 0.0, 1.0), (1, 1.0, -2.0, 1.0),
                               (0, np.nan, 1.0, 1.0), (1, 1.0, np.inf, 1.0), (0, 1.0, 1.0, np.nan)]:
        with pytest.raises(_lib.DmfError):
            b.set_step_state(which, [1.0, a], [1.0, l], [1.0, l_old])        # fit 1 is bad: nothing is written
    s1 = b.states()
    assert [(s.a1, s.a2, s.l_w, s.l_h) for s in s1] == [(s.a1, s.a2, s.l_w, s.l_h) for s in s0]
    b.set_step_state(0, [2.0, 3.0], [5.0, 7.0], [6.0, 8.0])
    b.set_step_state(1, [4.0, 9.0], [11.0, 13.0], [12.0, 14.0])
    s2 = b.states()
    assert [(s.a1, s.l_w, s.a2, s.l_h) for s in s2] == [(2.0, 5.0, 4.0, 11.0), (3.0, 7.0, 9.0, 13.0)]
    assert [(s.cost, s.cost_prev, s.dmax, s.n_outer, s.done, s.u_slot, s.a_slot) for s in s2] == \
           [(s.cost, s.cost_prev, s.dmax, s.n_outer, s.done, s.u_slot, s.a_slot) for s in s0]
    b.close()
