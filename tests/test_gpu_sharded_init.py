"""GPU tests of the initial iterate on row-sharded data: the library's split WLS (dmf_wls_moments + dmf_wls_solve) and the residual
reductions of the SVD inits (dmf_resid_gram, dmf_resid_project, dmf_nndsvd_apply) driven by sharded.ShardedInit.  With one process
the all-reduce is the identity, so every result must equal the single-process path; several processes are covered on CPU
(tests/test_sharded_init_cpu.py, gloo) and on 2 GPUs by tools/sharded_check.py (torchrun)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
TOL = 1e-6


@pytest.fixture(scope="module")
def sh():
    import torch
    assert torch.cuda.is_available()
    import __graft_entry__ as g
    g.build()
    from demethify_b200 import sharded
    return sharded


@pytest.mark.parametrize("N", [1, 10, 64, 256, 512])
@pytest.mark.parametrize("K", [0, 5])
def test_resid_gram_matches_numpy(sh, N, K):
    rs = np.random.RandomState(N + K)
    M = 1001                                                  # not a multiple of any row tile
    X = rs.uniform(0, 1, size=(M, N))
    R = rs.uniform(0, 1, size=(M, K)) if K else None
    H1 = rs.dirichlet(np.ones(K), N).T * 0.7 if K else None
    be = sh.GpuInitBackend(X, np.ones((M, N)), R, precision="fp64")
    G1, neg = be.resid_gram(H1)
    G2, _ = be.resid_gram(H1)
    r = X if K == 0 else np.maximum(X - R @ H1, 1e-8)
    want = r.T @ r
    got = G1.cpu().numpy()
    assert int(neg.item()) == 0
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()
    assert np.array_equal(got, got.T) and np.array_equal(got, G2.cpu().numpy())          # symmetric, bit-reproducible


def test_resid_gram_flags_negative_input(sh):
    X = np.random.RandomState(0).uniform(0, 1, size=(300, 7))
    X[299, 6] = -1e-3
    _, neg = sh.GpuInitBackend(X, np.ones_like(X), None, precision="fp64").resid_gram(None)
    assert int(neg.item()) == 1
    with pytest.raises(ValueError, match="negative elements"):
        sh.unsupervised_init_sharded("SVD", X, np.ones_like(X), 2, seed=1)


@pytest.mark.parametrize("M,N,K,K2,y_is_dx", [(4000, 301, 13, 0, False), (2999, 10, 5, 2, False), (350, 10, 5, 0, True)])
def test_wls_moments_then_solve_equals_wls_fit_bitwise(sh, M, N, K, K2, y_is_dx):
    from demethify_b200.init_func import wls_all_samples
    rs = np.random.RandomState(M)
    R = rs.beta(0.5, 0.5, size=(M, K))
    E = rs.uniform(size=(M, K2)) if K2 else None
    D = rs.poisson(30, size=(M, N)) + 1
    X = rs.binomial(D, np.clip(R @ rs.dirichlet(np.ones(K), N).T, 0, 1)) / D
    want = wls_all_samples(X, D, R, extra=E, y_is_dx=y_is_dx)
    got = sh.wls_all_samples_sharded(X, D, R, extra=E, y_is_dx=y_is_dx)
    assert np.array_equal(got, want)


def test_wls_moments_symmetric_and_reproducible(sh, shipped):
    """Each moment has one writer: the matrix is exactly symmetric and repeated calls agree bit for bit (the reference-based fit
    on the shipped fixture, y = d o x, and a K + K2 = 15 shape whose 8 x 8 blocks include off-diagonal ones)."""
    from demethify_b200.init_func import wls_all_samples
    X, D, Rk = shipped["X"], shipped["D"], shipped["Rk"]
    rs = np.random.RandomState(1)
    E = rs.uniform(size=(X.shape[0], 10))
    for extra, y_is_dx in ((None, True), (E, False)):
        be = sh.GpuInitBackend(X, D, Rk)
        kz = Rk.shape[1] + (0 if extra is None else extra.shape[1]) + 2
        moms = [be.wls_moments(extra, y_is_dx).cpu().numpy().reshape(kz, kz, -1) for _ in range(5)]
        for m in moms:
            assert np.array_equal(m, np.transpose(m, (1, 0, 2))) and np.array_equal(m, moms[0])
        fits = [wls_all_samples(X, D, Rk, extra=extra, y_is_dx=y_is_dx) for _ in range(5)]
        assert all(np.array_equal(f, fits[0]) for f in fits)


def test_sharded_svd_init_and_fit_match_golden(sh, shipped, live):
    from demethify_b200 import deconvolution as dec
    X, D, Rk = shipped["X"], shipped["D"], shipped["Rk"]
    u0, a0 = sh.init_BSSMF_md_sharded("SVD", X, D, Rk, 2, seed=1)
    us, _, as_ = dec.init_BSSMF_md("SVD", X, D, Rk, 2, seed=1)
    assert np.abs(u0 - live["svd_u0"]).max() <= 1e-8 and np.abs(a0 - live["svd_a0"]).max() <= 1e-8
    assert np.abs(u0 - us).max() <= 1e-8 and np.abs(a0 - as_).max() <= 1e-8
    u, a, n_outer, _ = sh.mdwbssmf_deconv_sharded(u0, a0, X, D, Rk, 2, n_iter1=10000, n_iter2=20, tol=1e-2)
    assert n_outer == len(live["svd_costs"]) - 1
    assert np.abs(a - live["svd_a"]).max() <= TOL and np.abs(u - live["svd_u"]).max() <= TOL


def test_sharded_uniform_init_and_fit_match_golden(sh, shipped, live):
    from demethify_b200 import deconvolution as dec
    X, D, Rk = shipped["X"], shipped["D"], shipped["Rk"]
    u0, a0 = sh.init_BSSMF_md_sharded("uniform", X, D, Rk, 2, seed=2)
    us, _, as_ = dec.init_BSSMF_md("uniform", X, D, Rk, 2, seed=2)
    assert np.array_equal(u0, us) and np.abs(a0 - as_).max() <= 1e-12
    assert np.abs(a0 - live["uniform_a0"]).max() <= 1e-8
    u, a, n_outer, _ = sh.mdwbssmf_deconv_sharded(u0, a0, X, D, Rk, 2, n_iter1=10000, n_iter2=20, tol=1e-2)
    assert n_outer == len(live["uniform_costs"]) - 1
    assert np.abs(a - live["uniform_a"]).max() <= TOL and np.abs(u - live["uniform_u"]).max() <= TOL


def test_sharded_purity_svd_init_matches_single_process(sh):
    from demethify_b200 import deconvolution as dec
    rs = np.random.RandomState(4)
    M, N, K = 3001, 12, 5
    R = rs.beta(0.5, 0.5, size=(M, K + 2))
    D = rs.poisson(40, size=(M, N)) + 1
    X = rs.binomial(D, np.clip(R @ rs.dirichlet(np.ones(K + 2), N).T, 0, 1)) / D
    pur = rs.uniform(0.3, 0.9, size=N)
    u0, a0 = sh.init_BSSMF_md_p_sharded("SVD", X, D, R[:, :K], 2, pur, seed=3)
    us, _, as_ = dec.init_BSSMF_md_p("SVD", X, D, R[:, :K], 2, pur, seed=3)
    assert np.abs(u0 - us).max() <= 1e-8 and np.abs(a0 - as_).max() <= 1e-8


@pytest.mark.parametrize("n_u", [2, 4])
def test_sharded_reference_free_svd_init_matches_single_process(sh, shipped, n_u):
    from demethify_b200.deconvolution import projection_simplex_sort_2d
    from demethify_b200.init_func import nndsvd_initialize
    X, D = shipped["X"], shipped["D"]
    u0, a0 = sh.unsupervised_init_sharded("SVD", X, D, n_u, seed=1)
    W, H = nndsvd_initialize(X, rank=n_u)                     # unsupervised_deconv's SVD init (deconvolution.py:128-131)
    assert np.abs(u0 - W.clip(0, 1)).max() <= 1e-8 and np.abs(a0 - projection_simplex_sort_2d(H)).max() <= 1e-8


def test_sharded_reference_based_fit_matches_single_process(sh, shipped):
    from demethify_b200.init_func import wls_all_samples
    X, D, Rk = shipped["X"], shipped["D"], shipped["Rk"]
    got = sh.wls_all_samples_sharded(X, D, Rk, y_is_dx=True)
    assert np.array_equal(got, wls_all_samples(X, D, Rk, y_is_dx=True))
    assert np.abs(got - shipped["ref_based_alpha"]).max() <= 1e-9
