"""CPU tests of the reference's rules for the initial iterate (deconvolution.py:40-78, :107-150, :228-267): the `n_u > N` fallbacks,
the `uniform_` / `beta` draws, the option errors, the purity fallback message and the zero guard, through every public entry point
that can draw on a CPU - the single-process inits, the row-sharded ones with the numpy backend, and the bootstrap's private-stream
draws - against the numpy oracle, bit for bit."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import bssmf_numpy as orc
from test_sharded_init_cpu import NumpyInitBackend, synth

M, N, K = 37, 5, 3
PURITY = np.random.RandomState(4).uniform(0.3, 0.9, size=N)
MESSAGE = "The number of unknowns is greater than the number of samples, we'll go with a uniform initialisation. \n"
GRID = [(opt, n_u) for opt in ("uniform_", "beta") for n_u in (2, N + 2)]


def _data():
    return synth(11, M, N, K, 2)


def _oracle_free(opt, n_u, seed):
    """The draws of oracle.solve_unsupervised, in its order (the oracle has no standalone reference-free draw)."""
    rs = orc.legacy_stream(seed)
    if opt != "uniform_" and n_u > N:
        opt = "uniform_"
    u = rs.uniform(size=(M, n_u)) if opt == "uniform_" else rs.beta(np.ones((M, n_u)) * 0.5, np.ones((M, n_u)) * 0.5)
    return u, rs.dirichlet(np.ones(n_u), N).T


def _bootstrap_option(opt, n_u):
    return "uniform_" if n_u > N else opt          # bootstrap_fits resolves the fallback before it draws


@pytest.mark.parametrize("opt,n_u", GRID)
def test_partial_draws_equal_the_oracle(opt, n_u):
    from demethify_b200 import bootstrap, deconvolution as dc, sharded as sh
    X, D, Rk = _data()
    U, R, A = orc.draw_init(opt, X, D, Rk, n_u, seed=3)
    u, r, a = dc.init_BSSMF_md(opt, X, D, Rk, n_u, seed=3)
    assert np.array_equal(u, U) and np.array_equal(r, R) and np.array_equal(a, A)
    u, a = sh.init_BSSMF_md_sharded(opt, None, None, None, n_u, seed=3, backend=NumpyInitBackend(X, D, Rk))
    assert np.array_equal(u, U) and np.array_equal(a, A)
    u, a = bootstrap._shape_only_init(3, _bootstrap_option(opt, n_u), M, K, N, n_u, with_zero_guard=True)
    assert np.array_equal(u, U) and np.array_equal(a, A)


@pytest.mark.parametrize("opt,n_u", GRID)
def test_purity_draws_equal_the_oracle(opt, n_u):
    from demethify_b200 import bootstrap, deconvolution as dc, sharded as sh
    X, D, Rk = _data()
    U, R, A = orc.draw_init_purity(opt, X, D, Rk, n_u, PURITY, seed=5)
    u, r, a = dc.init_BSSMF_md_p(opt, X, D, Rk, n_u, PURITY, seed=5)
    assert np.array_equal(u, U) and np.array_equal(r, R) and np.array_equal(a, A)
    u, a = sh.init_BSSMF_md_p_sharded(opt, None, None, None, n_u, PURITY, seed=5, backend=NumpyInitBackend(X, D, Rk))
    assert np.array_equal(u, U) and np.array_equal(a, A)
    u, a = bootstrap._shape_only_init(5, _bootstrap_option(opt, n_u), M, K, N, n_u, with_zero_guard=False)
    assert np.array_equal(u, U) and np.array_equal(a, A)


@pytest.mark.parametrize("opt,n_u", GRID)
def test_reference_free_draws_equal_the_oracle(opt, n_u):
    from demethify_b200 import sharded as sh
    X, D, _ = _data()
    U, A = _oracle_free(opt, n_u, seed=7)
    u, a = sh.unsupervised_init_sharded(opt, None, None, n_u, seed=7, backend=NumpyInitBackend(X, D, None))
    assert np.array_equal(u, U) and np.array_equal(a, A)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


WINDOW_CASES = [(variant, opt, n_u) for variant in ("partial", "purity", "free") for opt, n_u in GRID]


def _draw_sharded(variant, opt, n_u, X, D, Rk):
    from demethify_b200 import sharded as sh
    if variant == "free":
        return sh.unsupervised_init_sharded(opt, None, None, n_u, seed=9, backend=NumpyInitBackend(X, D, None))
    if variant == "purity":
        return sh.init_BSSMF_md_p_sharded(opt, None, None, None, n_u, PURITY, seed=9, backend=NumpyInitBackend(X, D, Rk))
    return sh.init_BSSMF_md_sharded(opt, None, None, None, n_u, seed=9, backend=NumpyInitBackend(X, D, Rk))


def _window_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from demethify_b200 import sharded as sh
        X, D, Rk = _data()
        lo, hi = sh.row_range(M, rank, world)
        res = {}
        for i, case in enumerate(WINDOW_CASES):
            res[f"u{i}"], res[f"a{i}"] = _draw_sharded(*case, X[lo:hi], D[lo:hi], Rk[lo:hi])
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), lo=lo, hi=hi, **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_row_window_keeps_those_rows_of_the_full_draw(tmp_path):
    """Rank r of 3 gets exactly rows [lo, hi) of the world-size-1 draw, and the same alpha."""
    world = 3
    mp.spawn(_window_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    X, D, Rk = _data()
    for rank in range(world):
        q = np.load(tmp_path / f"rank{rank}.npz")
        lo, hi = int(q["lo"]), int(q["hi"])
        assert 0 < hi - lo < M
        for i, case in enumerate(WINDOW_CASES):
            u, a = _draw_sharded(*case, X, D, Rk)
            assert np.array_equal(q[f"u{i}"], u[lo:hi]) and np.array_equal(q[f"a{i}"], a), case


def test_option_errors():
    from demethify_b200 import deconvolution as dc, sharded as sh
    X, D, Rk = _data()

    def partial(opt, n_u=2):
        return dc.init_BSSMF_md(opt, X, D, Rk, n_u, seed=1)

    def purity(opt, n_u=2):
        return dc.init_BSSMF_md_p(opt, X, D, Rk, n_u, PURITY, seed=1)

    def partial_sharded(opt, n_u=2):
        return sh.init_BSSMF_md_sharded(opt, None, None, None, n_u, seed=1, backend=NumpyInitBackend(X, D, Rk))

    def purity_sharded(opt, n_u=2):
        return sh.init_BSSMF_md_p_sharded(opt, None, None, None, n_u, PURITY, seed=1, backend=NumpyInitBackend(X, D, Rk))

    def free(opt, n_u=2):
        return dc.unsupervised_deconv(X, n_u, D, opt, seed=1)

    def free_sharded(opt, n_u=2):
        return sh.unsupervised_init_sharded(opt, None, None, n_u, seed=1, backend=NumpyInitBackend(X, D, None))

    for f in (partial, purity, partial_sharded, purity_sharded, free, free_sharded):
        with pytest.raises(NotImplementedError):
            f("ICA")
    for f in (partial, purity, partial_sharded, purity_sharded):
        with pytest.raises(ValueError, match="unknown init option 'typo'"):
            f("typo")
    for f in (free, free_sharded):
        with pytest.raises(NameError, match="R_trunc"):
            f("uniform")
        with pytest.raises(NotImplementedError, match="'typo' is not available"):
            f("typo")
    # n_u > N: every option becomes uniform_ before the dispatch, so ICA draws instead of raising
    U, _, A = orc.draw_init("uniform_", X, D, Rk, N + 1, seed=1)
    for f in (partial, partial_sharded):
        got = f("ICA", N + 1)
        assert np.array_equal(got[0], U) and np.array_equal(got[-1], A)
    U, _, A = orc.draw_init_purity("uniform_", X, D, Rk, N + 1, PURITY, seed=1)
    for f in (purity, purity_sharded):
        got = f("ICA", N + 1)
        assert np.array_equal(got[0], U) and np.array_equal(got[-1], A)
    U, A = _oracle_free("uniform_", N + 1, seed=1)
    u, a = free_sharded("ICA", N + 1)
    assert np.array_equal(u, U) and np.array_equal(a, A)


def test_purity_fallback_prints_once(capsys):
    from demethify_b200 import bootstrap, deconvolution as dc, sharded as sh
    X, D, Rk = _data()
    dc.init_BSSMF_md_p("beta", X, D, Rk, N + 1, PURITY, seed=2)
    assert capsys.readouterr().out == MESSAGE
    sh.init_BSSMF_md_p_sharded("SVD", None, None, None, N + 1, PURITY, seed=2, backend=NumpyInitBackend(X, D, Rk))
    assert capsys.readouterr().out == MESSAGE
    dc.init_BSSMF_md_p("uniform", X, D, Rk, N + 1, PURITY, seed=2)      # `uniform` itself does not announce the fallback
    dc.init_BSSMF_md("beta", X, D, Rk, N + 1, seed=2)
    sh.init_BSSMF_md_sharded("SVD", None, None, None, N + 1, seed=2, backend=NumpyInitBackend(X, D, Rk))
    bootstrap._shape_only_init(2, "uniform_", M, K, N, N + 1, with_zero_guard=False)
    assert capsys.readouterr().out == ""


def test_bootstrap_purity_fallback_is_silent(capsys):
    """bootstrap_fits resolves the n_u > N fallback of a purity fit without the message; without a GPU the call then stops in
    the device layer."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from demethify_b200 import _lib
    from demethify_b200.bootstrap import bootstrap_fits
    X, D, Rk = _data()
    with pytest.raises(_lib.DmfError):
        bootstrap_fits(2, N + 1, X, D, Rk, "SVD", 5, 5, 1e-3, PURITY, 1)
    assert capsys.readouterr().out == ""


class _ZeroFirstUnknown(NumpyInitBackend):
    """The numpy backend with an exact zero in the first unknown row of the WLS result (sample 0)."""

    def wls_solve(self, mom, M, K2):
        a = super().wls_solve(mom, M, K2)
        a[self.K, 0] = 0.0
        self.fit = a.copy()
        return a


def test_zero_guard_partial_only():
    """deconvolution.py:74-76: a zero in the first unknown row of alpha sets that row to 1e-10 and scales the known rows by
    1 - 1e-10; init_BSSMF_md applies it, init_BSSMF_md_p does not."""
    from demethify_b200 import sharded as sh
    X, D, Rk = _data()
    n_u = 2
    U = orc.legacy_stream(8).uniform(size=(M, n_u))
    be = _ZeroFirstUnknown(X, D, Rk)
    u, a = sh.init_BSSMF_md_sharded("uniform", None, None, None, n_u, seed=8, backend=be)
    want = be.fit.copy()
    want[K] = 1e-10
    want[:K] = (1 - 1e-10) * want[:K]
    assert np.array_equal(u, U) and np.array_equal(a, want)
    be = _ZeroFirstUnknown(X, D, Rk)
    u, a = sh.init_BSSMF_md_p_sharded("uniform", None, None, None, n_u, PURITY, seed=8, backend=be)
    assert np.array_equal(u, U) and np.array_equal(a, be.fit)
