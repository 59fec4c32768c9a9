"""CPU tests of the row-sharded CCC and BCV members (ic.consensus_runs_sharded, ic.bicross_validation_sharded) at world sizes 2 and
3 over gloo: the product's orchestration (initial iterates, fold planner, one multi-fit RowShardedFit per member, all-reduced test
errors) with numpy restatements of the library's per-rank steps, against the single-process numpy oracle's ic_sweep."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import bssmf_numpy as orc
from oracle.gram_numpy import NumpyShardBackend
from test_sharded_init_cpu import NumpyInitBackend, synth

IT1, IT2, TOL = 40, 10, 1e-7
N_RUNS = 3
# (criterion, init option, seed, shape (M, N, K), n_u values); BCV seed 0 on 6 x 2 skips fold 1 (an all-test mask)
CASES = [("CCC", "uniform_", 3, (240, 7, 3), [1, 2]), ("CCC", "beta", 4, (240, 7, 3), [1, 2]), ("CCC", "uniform", 5, (240, 7, 3), [1, 2]),
         ("CCC", "SVD", 6, (240, 7, 3), [1, 2]),
         ("BCV", "uniform_", 3, (240, 7, 3), [1, 2]), ("BCV", "beta", 4, (240, 7, 3), [1, 2]), ("BCV", "uniform", 5, (240, 7, 3), [1, 2]),
         ("BCV", "SVD", 6, (240, 7, 3), [1, 2]), ("BCV", "uniform_", [5], (240, 7, 3), [1]), ("BCV", "SVD", [7], (240, 7, 3), [2]),
         ("BCV", "uniform_", 0, (6, 2, 1), [1])]


class NumpyBatchBackend:
    """Several NumpyShardBackend fits behind the interface of a multi-fit GpuShardBackend: the (n_fits, doubles per fit) statistics
    blocks hold one row per fit, every step advances the fits that are still running, and the fits are done when all are."""

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

    def _each(self, step, *args):
        for f in self.fits:
            getattr(f, step)(*args)

    def rowgram(self, initial, tol):
        self._each("rowgram", initial, tol)

    def finalize_cost(self, initial, tol):
        self._each("finalize_cost", initial, tol)

    def u_inner(self, n_iter2):
        self._each("u_inner", n_iter2)

    def panels(self, known_block):
        self._each("panels", known_block)

    def alpha_inner(self, n_iter2):
        self._each("alpha_inner", n_iter2)

    def all_done(self):
        return all(f.all_done() for f in self.fits)

    def results(self):
        return [r for f in self.fits for r in f.results()]

    def close(self):
        pass


def numpy_fit_backend(log):
    def make(problems, n_u, U0s, A0s):
        log.append(len(U0s))
        problems = problems * len(U0s) if len(problems) == 1 else problems
        return NumpyBatchBackend([NumpyShardBackend(X, D, R, n_u, u, a) for (X, D, R), u, a in zip(problems, U0s, A0s)])
    return make


def numpy_cost(X, R, alpha, W):
    return float(np.sum(W * (X - R @ alpha) ** 2))


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
        from demethify_b200.ic import bicross_validation_sharded, consensus_runs_sharded
        from demethify_b200.sharded import row_range
        res = {}
        for c, (ic, opt, seed, (M, N, K), n_us) in enumerate(CASES):
            X, D, Rk = synth(11 + c, M, N, K, 2)
            lo, hi = row_range(M, rank, world)
            loc = (X[lo:hi], D[lo:hi], Rk[lo:hi])
            for n_u in n_us:
                log = []
                tag = f"c{c}_n{n_u}"
                if ic == "CCC":
                    runs, u, a = consensus_runs_sharded(*loc, M, lo, hi, n_u, opt, [seed + r for r in range(N_RUNS)], IT1, IT2, TOL,
                                                        init_backend=NumpyInitBackend, fit_backend=numpy_fit_backend(log))
                    res[tag + "_runs"] = np.stack(runs)
                else:
                    total, u, a, errors = bicross_validation_sharded(*loc, M, lo, hi, n_u, opt, seed, N_RUNS, IT1, IT2, TOL,
                                                                     init_backend=NumpyInitBackend, fit_backend=numpy_fit_backend(log),
                                                                     cost=numpy_cost)
                    res[tag + "_total"] = total
                    res[tag + "_errors"] = np.array([np.nan if e is None else e for e in errors])
                    res[tag + "_after"] = np.random.random_sample(4)      # where the global stream was left
                res[tag + "_u"], res[tag + "_a"], res[tag + "_nfits"] = u, a, np.array(log)
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


def _oracle_bcv_errors(X, D, Rk, n_u, opt, seed):
    """Per-fold test errors of the oracle's bicross_validation_press (NaN for a skipped fold): its totals over the first f folds."""
    totals = [0.0] + [orc.bicross_validation_press(X, n_u, D, IT1, IT2, TOL, f, seed, Rk, opt)[0] for f in range(1, N_RUNS + 1)]
    return np.array([t1 - t0 if t1 != t0 else np.nan for t0, t1 in zip(totals, totals[1:])])


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("world", [2, 3])
def test_row_sharded_ccc_and_bcv_match_oracle_gloo(tmp_path, world):
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    r = [dict(np.load(tmp_path / f"rank{k}.npz")) for k in range(world)]
    for c, (ic, opt, seed, (M, N, K), n_us) in enumerate(CASES):
        X, D, Rk = synth(11 + c, M, N, K, 2)
        want_u, want_a, want_best, want_values = orc.ic_sweep(X, Rk, D, opt, ic, seed, IT1, IT2, TOL, n_restarts=N_RUNS, n_u_values=n_us)
        values = []
        for n_u in n_us:
            tag, case = f"c{c}_n{n_u}", (ic, opt, seed, n_u)
            for q in r[1:]:                                     # alpha and the criteria are the same on every rank
                assert np.array_equal(q[tag + "_a"], r[0][tag + "_a"]), case
            u = np.vstack([q[tag + "_u"] for q in r])
            if ic == "CCC":
                runs = r[0][tag + "_runs"]
                assert all(np.array_equal(q[tag + "_runs"], runs) for q in r) and list(r[0][tag + "_nfits"]) == [N_RUNS], case
                for k in range(N_RUNS):
                    uo, _, ao = orc.fit_for_ic(X, D, Rk, n_u, opt, seed + k, IT1, IT2, TOL)
                    assert np.abs(runs[k] - ao).max() <= 1e-10, case
                assert np.abs(u - uo).max() <= 1e-10 and np.abs(r[0][tag + "_a"] - ao).max() <= 1e-10, case      # the last restart's
                values.append(-orc.consensus_ccc(list(runs)))
            else:
                errors = r[0][tag + "_errors"]
                assert all(np.array_equal(q[tag + "_errors"], errors, equal_nan=True) for q in r), case
                want_errors = _oracle_bcv_errors(X, D, Rk, n_u, opt, seed)
                assert np.array_equal(np.isnan(errors), np.isnan(want_errors)), case
                ok = ~np.isnan(errors)
                assert np.abs(errors[ok] - want_errors[ok]).max() <= 1e-10 * np.abs(want_errors[ok]).max(), case
                nfits = r[0][tag + "_nfits"]
                # at most two distinct folds per member: the SVD init draws nothing, so every fold repeats the first
                assert list(nfits) == [1 if opt == "SVD" else 2], case
                total, best_u, best_a = orc.bicross_validation_press(X, n_u, D, IT1, IT2, TOL, N_RUNS, seed, Rk, opt)
                assert abs(float(r[0][tag + "_total"]) - total) <= 1e-10 * total, case
                assert np.abs(u - best_u).max() <= 1e-10 and np.abs(r[0][tag + "_a"] - best_a).max() <= 1e-10, case
                want_after = np.random.random_sample(4)          # the oracle left the global stream where the reference leaves it
                assert all(np.array_equal(q[tag + "_after"], want_after) for q in r), case
                values.append(float(r[0][tag + "_total"]))
        assert np.allclose(values, want_values, rtol=0, atol=1e-10), (ic, opt, seed)
        assert n_us[int(np.argmin(values))] == want_best, (ic, opt, seed)
    skip_case = [c for c, case in enumerate(CASES) if case[3] == (6, 2, 1)][0]
    assert np.isnan(r[0][f"c{skip_case}_n1_errors"][0])              # the shape and seed that hit the skip branch do hit it
