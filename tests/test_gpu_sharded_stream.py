"""GPU tests of the row-sharded stream engine: shapes the Gram form cannot run (more unknown types, Kt = 32, wide cohorts with many
types) through GpuShardBackend in one process, where the all-reduce is the identity.  Each fit must equal the reference-shaped
oracle and the unsharded single-GPU stream fit; the multi-process behaviour of the same orchestration is covered on CPU
(tests/test_sharded_stream_cpu.py, gloo) and under torchrun by tools/sharded_stream_check.py."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sharded():
    import torch
    assert torch.cuda.is_available()
    import __graft_entry__ as g
    g.build()
    from demethify_b200 import sharded
    return sharded


def synth(seed, M, N, K, n_true, depth=50):
    rs = np.random.RandomState(seed)
    a = rs.uniform(0.2, 1.0, size=K + n_true)
    Rf = rs.beta(a, a, size=(M, K + n_true))
    unk = rs.uniform(0, 0.9, size=N)
    Ak = rs.dirichlet(np.ones(max(K, 1)), N).T[:K] * (1 - unk)
    Au = rs.dirichlet(np.ones(n_true), N).T * unk
    D = rs.poisson(depth, size=(M, N)) + 1
    cnt = rs.binomial(D, np.clip(Rf @ np.vstack([Ak, Au]), 0, 1))
    return cnt / D, D.astype(np.int64), np.ascontiguousarray(Rf[:, :K])


def problem(mode, M, N, K, n_u, seeds):
    """(X, D, R_trunc or None, purity or None, [(u0, R0, alpha0)] one per seed) drawn like the reference."""
    from oracle import bssmf_numpy as orc
    X, D, Rk = synth(M + N + K + n_u, M, N, K, max(min(n_u, 4), 1))
    pur = np.random.RandomState(N).uniform(0.2, 0.9, size=N) if mode == "purity" else None
    inits = []
    for s in seeds:
        if mode == "free":
            rs = orc.legacy_stream(s)
            u0 = rs.uniform(size=(M, n_u))
            inits.append((u0, None, rs.dirichlet(np.ones(n_u), N).T))
        elif mode == "purity":
            inits.append(orc.draw_init_purity("uniform_", X, D, Rk, n_u, pur, seed=s))
        else:
            inits.append(orc.draw_init("uniform_", X, D, Rk, n_u, seed=s))
    return X, D, (None if mode == "free" else Rk), pur, inits


def oracle_fit(mode, X, D, Rk, n_u, pur, init, seed, it1, it2, tol):
    from oracle import bssmf_numpy as orc
    u0, R0, a0 = init
    tr = {}
    if mode == "partial":
        uo, ao = orc.solve_partial_reference(u0.copy(), R0, a0.copy(), X, D.astype(float), Rk, n_u, it1, it2, tol, trace=tr)
    elif mode == "purity":
        uo, ao = orc.solve_purity(u0.copy(), R0, a0.copy(), X, D.astype(float), Rk, n_u, pur, it1, it2, tol, trace=tr)
    else:
        uo, ao = orc.solve_unsupervised(X, n_u, D.astype(float), "uniform_", it1, it2, tol, seed=seed, trace=tr)
    return uo, ao, tr["n_outer"], tr["costs"][-1]


def unsharded_stream_fit(X, D, Rk, n_u, mode, pur, inits, it1, it2, tol, precision):
    from demethify_b200 import _lib
    from demethify_b200.engine import DeviceProblem, FitBatch
    m = {"partial": _lib.DMF_MODE_PARTIAL, "purity": _lib.DMF_MODE_PURITY, "free": _lib.DMF_MODE_UNSUPERVISED}[mode]
    b = FitBatch(DeviceProblem(X, D, Rk, precision=precision), n_u, [i[0] for i in inits], [i[2] for i in inits], mode=m, purity=pur)
    try:
        assert b.engine == "stream"
        b.fit(it1, it2, tol)
        return b.results()
    finally:
        b.close()


# name, mode, (M, N, K, n_u), precision, (n_iter1, n_iter2, tol), initial iterate seeds (one fit per seed)
CASES = [("K6_nu9", "partial", (3000, 40, 6, 9), "fp64", (5, 10, 1e-9), [7]),
         ("K8_nu5", "partial", (3000, 40, 8, 5), "fp64", (5, 10, 1e-9), [7]),
         ("K22_nu10_Kt32", "partial", (2000, 24, 22, 10), "fp64", (4, 6, 1e-9), [7]),
         ("K6_nu4_N400", "partial", (2000, 400, 6, 4), "fp64", (3, 5, 1e-9), [7]),
         ("purity_K7_nu5", "purity", (2500, 32, 7, 5), "fp64", (4, 25, 1e-9), [7]),
         ("free_nu10", "free", (2500, 32, 0, 10), "fp64", (4, 8, 1e-9), [7]),
         ("fp32_K6_nu9", "partial", (3000, 40, 6, 9), "fp32", (4, 8, 1e-9), [7]),
         ("no_inner_K6_nu9", "partial", (1500, 24, 6, 9), "fp64", (3, 0, 1e-9), [7]),
         ("batch3_K6_nu9", "partial", (3000, 40, 6, 9), "fp64", (60, 5, 1250.0), [7, 8, 9])]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_sharded_stream_single_rank(sharded, case):
    name, mode, (M, N, K, n_u), precision, (it1, it2, tol), seeds = case
    from demethify_b200 import _lib
    X, D, Rk, pur, inits = problem(mode, M, N, K, n_u, seeds)
    m = {"partial": _lib.DMF_MODE_PARTIAL, "purity": _lib.DMF_MODE_PURITY, "free": _lib.DMF_MODE_UNSUPERVISED}[mode]
    be = sharded.GpuShardBackend(X, D, Rk, n_u, [i[0] for i in inits], [i[2] for i in inits], mode=m, purity=pur, precision=precision)
    assert be.stream and be.batch.engine == "stream"
    got = sharded.fit_row_sharded(be, it1, it2, tol)
    want = unsharded_stream_fit(X, D, Rk, n_u, mode, pur, inits, it1, it2, tol, precision)
    tol_ua = 1e-6 if precision == "fp64" else 1e-4
    for (u, a, n_outer, cost), (u1, a1, n1, c1), init, s in zip(got, want, inits, seeds):
        uo, ao, no, co = oracle_fit(mode, X, D, Rk, n_u, pur, init, s, it1, it2, tol)
        assert n_outer == no and abs(cost - co) <= (1e-9 if precision == "fp64" else 1e-5) * co, (name, s, n_outer, no, cost, co)
        assert np.abs(a - ao).max() <= tol_ua and np.abs(u - uo).max() <= tol_ua, (name, s)
        # the same passes as the unsharded stream fit: only where the state is advanced differs
        assert n_outer == n1 and abs(cost - c1) <= 1e-12 * c1, (name, s)
        assert np.abs(a - a1).max() <= 1e-12 and np.abs(u - u1).max() <= 1e-12, (name, s)
    if name.startswith("batch"):                              # the fits stop at their own termination tests
        assert len({r[2] for r in got}) > 1 and max(r[2] for r in got) < it1
    # set-up: max and sum of the scalars; every issued outer iteration: ||u||^2, n_iter2 gradients, the cost
    from test_sharded_stream_cpu import issued_outer
    assert sharded.last_info["collectives"] == 2 + (it2 + 2) * issued_outer(max(r[2] for r in got), it1)


def test_resident_problem_keeps_its_reference(sharded):
    """A resident DeviceProblem that carries R_trunc (what the row-sharded AIC / BIC members pass) runs the partial fit."""
    from demethify_b200.engine import DeviceProblem
    X, D, Rk, pur, inits = problem("partial", 3000, 40, 6, 9, [7])
    u0, R0, a0 = inits[0]
    u, a, n_outer, cost = sharded.mdwbssmf_deconv_sharded(u0, a0, DeviceProblem(X, D, Rk), None, None, 9, n_iter1=4, n_iter2=6, tol=1e-9)
    uo, ao, no, co = oracle_fit("partial", X, D, Rk, 9, None, inits[0], 7, 4, 6, 1e-9)
    assert n_outer == no and abs(cost - co) <= 1e-9 * co
    assert np.abs(a - ao).max() <= 1e-6 and np.abs(u - uo).max() <= 1e-6


def test_sharded_stream_graph_replay(sharded):
    """DMF_SHARDED_GRAPH=1 path: an outer iteration of the stream branch captured once and replayed gives the eager result."""
    from demethify_b200 import _lib
    X, D, Rk, pur, inits = problem("partial", 3000, 40, 6, 9, [7])
    runs = []
    for use_graph in (False, True):
        be = sharded.GpuShardBackend(X, D, Rk, 9, inits[0][0], inits[0][2], mode=_lib.DMF_MODE_PARTIAL)
        try:
            assert be.stream and be.supports_graphs
            runs.append(sharded.RowShardedFit(be).fit(8, 6, 1e-9, use_graph=use_graph)[0])
        finally:
            be.close()
    (u0, a0, n0, c0), (u1, a1, n1, c1) = runs
    assert n0 == n1 == 8 and c0 == c1 and np.array_equal(a0, a1) and np.array_equal(u0, u1)


def test_gram_shapes_keep_their_engine(sharded):
    """Shapes the Gram form runs keep it (or the fused engine) when sharded, and the stream passes and commits, which would read its
    [G | bx | scal] blocks as a gradient, refuse such a batch."""
    from demethify_b200 import _lib
    X, D, Rk, pur, inits = problem("partial", 2000, 16, 6, 8, [7])
    be = sharded.GpuShardBackend(X, D, Rk, 8, inits[0][0], inits[0][2], mode=_lib.DMF_MODE_PARTIAL)
    try:
        assert not be.stream and be.batch.engine == "gram"
        for step in (be.pass_u, be.u_commit, lambda: be.pass_alpha(0), lambda: be.alpha_commit(0), lambda: be.cost(False, 0.0)):
            with pytest.raises(_lib.DmfError, match="row-sharded"):
                step()
    finally:
        be.close()
