"""CPU tests of the row-sharded stream engine's orchestration (sharded.RowShardedFit, stream branch) with the numpy restatement
of its per-rank steps (oracle/stream_numpy.py): on one process against the reference-shaped oracle, and at world sizes 2 and 3
over gloo against the unsharded run - the same n_outer on every rank, alpha bit-identical across ranks, the right rows of u and
n_iter2 + 2 collectives per issued outer iteration."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import bssmf_numpy as orc
from oracle.stream_numpy import NumpyStreamShardBackend
from demethify_b200.sharded import RowShardedFit, row_range


def synth(seed, M, N, K, n_true, depth=50):
    rs = np.random.RandomState(seed)
    a = rs.uniform(0.2, 1.0, size=K + n_true)
    Rf = rs.beta(a, a, size=(M, K + n_true))
    unk = rs.uniform(0, 0.9, size=N)
    Ak = rs.dirichlet(np.ones(max(K, 1)), N).T[:K] * (1 - unk)
    Au = rs.dirichlet(np.ones(n_true), N).T * unk
    D = rs.poisson(depth, size=(M, N)) + 1
    cnt = rs.binomial(D, np.clip(Rf @ np.vstack([Ak, Au]), 0, 1))
    return cnt / D, D.astype(np.float64), np.ascontiguousarray(Rf[:, :K])


class StreamBatch:
    """Several stream-form fits behind the interface of a multi-fit GpuShardBackend: one row of the statistics blocks per fit."""

    stream = True

    def __init__(self, fits):
        self.fits = fits
        self.local = torch.zeros((len(fits), fits[0].local.shape[1]), dtype=torch.float64)
        self.glob = torch.zeros_like(self.local)
        for i, f in enumerate(fits):
            f.local, f.glob = self.local[i:i + 1], self.glob[i:i + 1]
        self.scal_off, self.has_known = fits[0].scal_off, fits[0].has_known

    def stats_local(self):
        return self.local

    def stats_global(self):
        return self.glob

    def __getattr__(self, step):
        if step not in ("cost", "finalize_cost", "pass_u", "u_commit", "pass_alpha", "alpha_commit"):
            raise AttributeError(step)
        return lambda *args: [getattr(f, step)(*args) for f in self.fits] and None

    def all_done(self):
        return all(f.all_done() for f in self.fits)

    def results(self):
        return [r for f in self.fits for r in f.results()]


def issued_outer(n_outer, n_iter1):
    """Outer iterations RowShardedFit.fit issues before it sees every fit done: chunks of 2, 4, 8, 16, 16, ... between polls."""
    issued, chunk = 0, 2
    while issued < n_iter1:
        issued += min(chunk, n_iter1 - issued)
        if issued >= n_outer:
            break
        chunk = min(chunk * 2, 16)
    return issued


# name, (M, N, K, n_u), mode, (n_iter1, n_iter2, tol), initial iterate seeds (one fit per seed)
CASES = [("partial", (500, 7, 3, 2), "partial", (40, 10, 1e-1), [4]),
         ("purity", (400, 6, 3, 2), "purity", (4, 25, 1e-9), [5]),
         ("unsupervised", (450, 6, 0, 3), "unsupervised", (4, 10, 1e-9), [6]),
         ("no_inner", (300, 5, 2, 1), "partial", (5, 0, 1e-9), [7]),
         ("batch", (420, 6, 3, 2), "partial", (60, 5, 1.0), [8, 9, 10])]


def case_data(i):
    name, (M, N, K, n_u), mode, (it1, it2, tol), seeds = CASES[i]
    X, D, Rk = synth(20 + i, M, N, K, max(n_u, 1))
    pur = np.random.RandomState(i).uniform(0.2, 0.9, size=N) if mode == "purity" else None
    inits = []
    for s in seeds:
        if mode == "unsupervised":
            rs = orc.legacy_stream(s)
            u0 = rs.uniform(size=(M, n_u))
            inits.append((u0, None, rs.dirichlet(np.ones(n_u), N).T))
        elif mode == "purity":
            inits.append(orc.draw_init_purity("uniform_", X, D, Rk, n_u, pur, seed=s))
        else:
            inits.append(orc.draw_init("uniform_", X, D, Rk, n_u, seed=s))
    return X, D, None if mode == "unsupervised" else Rk, n_u, mode, pur, (it1, it2, tol), inits


def backend(X, D, Rk, n_u, mode, pur, inits, lo=0, hi=None):
    hi = X.shape[0] if hi is None else hi
    fits = [NumpyStreamShardBackend(X[lo:hi], D[lo:hi], None if Rk is None else Rk[lo:hi], n_u, u0[lo:hi], a0, mode=mode, purity=pur)
            for u0, _, a0 in inits]
    return fits[0] if len(fits) == 1 else StreamBatch(fits)


@pytest.mark.parametrize("i", range(len(CASES)), ids=[c[0] for c in CASES])
def test_stream_form_equals_reference_shape(i):
    X, D, Rk, n_u, mode, pur, (it1, it2, tol), inits = case_data(i)
    got = RowShardedFit(backend(X, D, Rk, n_u, mode, pur, inits)).fit(it1, it2, tol)
    for (u, a, n_outer, cost), (u0, R0, a0), s in zip(got, inits, CASES[i][4]):
        tr = {}
        if mode == "partial":
            uo, ao = orc.solve_partial_reference(u0.copy(), R0, a0.copy(), X, D, Rk, n_u, it1, it2, tol, trace=tr)
        elif mode == "purity":
            uo, ao = orc.solve_purity(u0.copy(), R0, a0.copy(), X, D, Rk, n_u, pur, it1, it2, tol, trace=tr)
        else:
            uo, ao = orc.solve_unsupervised(X, n_u, D, "uniform_", it1, it2, tol, seed=s, trace=tr)
        assert n_outer == tr["n_outer"] and abs(cost - tr["costs"][-1]) <= 1e-10 * cost, (CASES[i][0], s)
        assert np.abs(a - ao).max() <= 1e-10 and np.abs(u - uo).max() <= 1e-10, (CASES[i][0], s)
    if CASES[i][0] == "batch":                                  # the fits of the batch stop at their own tests
        assert len({r[2] for r in got}) > 1


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res = {}
        for i in range(len(CASES)):
            X, D, Rk, n_u, mode, pur, (it1, it2, tol), inits = case_data(i)
            lo, hi = row_range(X.shape[0], rank, world)
            fit = RowShardedFit(backend(X, D, Rk, n_u, mode, pur, inits, lo, hi))
            for f, (u, a, n_outer, cost) in enumerate(fit.fit(it1, it2, tol)):
                res.update({f"{i}_{f}_u": u, f"{i}_{f}_a": a, f"{i}_{f}_n": n_outer, f"{i}_{f}_c": cost})
            res[f"{i}_coll"] = fit.collectives
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(900)
@pytest.mark.parametrize("world", [2, 3])
def test_row_sharded_stream_fit_gloo(tmp_path, world):
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    r = [dict(np.load(tmp_path / f"rank{k}.npz")) for k in range(world)]
    for i, (name, _shape, _mode, (it1, it2, tol), seeds) in enumerate(CASES):
        X, D, Rk, n_u, mode, pur, _its, inits = case_data(i)
        want = RowShardedFit(backend(X, D, Rk, n_u, mode, pur, inits)).fit(it1, it2, tol)
        for f, (u1, a1, n1, c1) in enumerate(want):
            key = f"{i}_{f}_"
            assert all(int(q[key + "n"]) == n1 for q in r), (name, f)                        # the same termination decision everywhere
            assert all(np.array_equal(q[key + "a"], r[0][key + "a"]) for q in r), (name, f)  # alpha replicated bit for bit
            assert np.abs(r[0][key + "a"] - a1).max() <= 1e-10 and abs(float(r[0][key + "c"]) - c1) <= 1e-10 * c1, (name, f)
            assert np.abs(np.vstack([q[key + "u"] for q in r]) - u1).max() <= 1e-10, (name, f)
        # set-up: max and sum of the scalars; every issued outer iteration: ||u||^2, n_iter2 gradients, the cost
        want_coll = 2 + (it2 + 2) * issued_outer(max(w[2] for w in want), it1)
        assert all(int(q[f"{i}_coll"]) == want_coll for q in r), (name, [int(q[f"{i}_coll"]) for q in r], want_coll)
