"""CPU tests of the initial iterate on row-sharded data (no GPU needed): `ShardedInit` - the product's orchestration of the row
reductions (WLS moments, residual Gram matrix, NNDSVD column norms) - with a numpy restatement of the library's per-rank steps, at
world sizes 2 and 3 over gloo, against the single-process numpy oracle of the `uniform`, `SVD` (partial, purity, reference-free)
inits and the reference-based fit (n_u = 0)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import bssmf_numpy as orc


class NumpyInitBackend:
    """numpy restatement of demethify_b200.sharded.GpuInitBackend on this rank's rows: dmf_wls_moments / dmf_wls_solve
    (csrc/dmf_wls.cuh), dmf_resid_gram / dmf_resid_project / dmf_nndsvd_apply (csrc/dmf_resid.cuh)."""

    def __init__(self, X, D, Rk):
        self.X, self.D = np.asarray(X, dtype=np.float64), np.asarray(D, dtype=np.float64)
        self.Rk = None if Rk is None else np.asarray(Rk, dtype=np.float64)
        self.M, self.N = self.X.shape
        self.K = 0 if Rk is None else self.Rk.shape[1]
        self.device = torch.device("cpu")

    def wls_moments(self, extra, y_is_dx):
        y = self.D * self.X if y_is_dx else self.X
        regs = [r for r in (self.Rk, None if extra is None else np.asarray(extra, dtype=np.float64)) if r is not None]
        R = np.hstack(regs) if regs else np.zeros((self.M, 0))
        Z = np.empty((self.M, self.N, R.shape[1] + 2))
        Z[:, :, 0], Z[:, :, 1], Z[:, :, 2:] = 1.0, y, R[:, None, :]
        kz = Z.shape[2]
        return torch.from_numpy(np.einsum("mj,mjp,mjq->pqj", self.D, Z, Z).reshape(kz * kz, self.N).copy())

    def wls_solve(self, mom, M, K2):
        K = self.K + K2
        Z = mom.numpy().reshape(K + 2, K + 2, self.N)
        out = np.zeros((K, self.N))
        for j in range(self.N):
            z = Z[:, :, j]
            rbar = z[0, 2:] / z[0, 0]
            b = z[1, 2:] - rbar * z[0, 1]
            G = z[2:, 2:] - rbar[:, None] * z[0, 2:][None, :]
            x = _nnls_normal(G, b, M)
            out[:, j] = x / max(x.sum(), 1e-10)
        return out

    def _r(self, H1):
        return self.X if H1 is None else np.maximum(self.X - self.Rk @ np.asarray(H1), 1e-8)

    def resid_gram(self, H1):
        r = self._r(H1)
        neg = int(H1 is None and bool((self.X < 0).any()))
        return torch.from_numpy(r.T @ r), torch.tensor([neg], dtype=torch.int32)

    def resid_project(self, H1, Vh, inv_sigma):
        U = self._r(H1) @ Vh.numpy().T * inv_sigma.numpy()
        sums = np.concatenate([np.sum(np.maximum(U, 0) ** 2, axis=0), np.sum(np.maximum(-U, 0) ** 2, axis=0)])
        return U, torch.from_numpy(sums)

    def nndsvd_apply(self, U, Vh, sigma, sums):
        Vh, S, s = Vh.numpy(), sigma.numpy(), sums.numpy()
        rank = Vh.shape[0]
        W, H = np.zeros((self.M, rank)), np.zeros((rank, self.N))
        W[:, 0], H[0] = np.sqrt(S[0]) * np.abs(U[:, 0]), np.sqrt(S[0]) * np.abs(Vh[0])
        for i in range(1, rank):
            n_up, n_un = np.sqrt(s[i]), np.sqrt(s[rank + i])
            n_vp, n_vn = np.linalg.norm(np.maximum(Vh[i], 0)), np.linalg.norm(np.maximum(-Vh[i], 0))
            tp, tn = n_up * n_vp, n_un * n_vn
            if tp >= tn:
                W[:, i], H[i] = np.sqrt(S[i] * tp) / n_up * np.maximum(U[:, i], 0), np.sqrt(S[i] * tp) / n_vp * np.maximum(Vh[i], 0)
            else:
                W[:, i], H[i] = np.sqrt(S[i] * tn) / n_un * np.maximum(-U[:, i], 0), np.sqrt(S[i] * tn) / n_vn * np.maximum(-Vh[i], 0)
        W[W < 1e-11] = 0
        H[H < 1e-11] = 0
        return W, H


def _nnls_normal(G, b, M):
    """Lawson-Hanson on the normal equations (G, b), with the tolerances of wls_nnls_kernel (M = the global row count)."""
    K = len(b)
    tolx = 10.0 * max(M, K) * np.spacing(1.0)
    tol = tolx * np.abs(b).sum()
    x, passive, it = np.zeros(K), np.zeros(K, dtype=bool), 0

    def solve():
        s = np.zeros(K)
        if passive.any():
            s[passive] = np.linalg.solve(G[np.ix_(passive, passive)], b[passive])
        return s
    w = b - G @ x
    while True:
        cand = np.where(~passive & (w > tol), w, -np.inf)
        if not np.isfinite(cand).any():
            break
        passive[int(np.argmax(cand))] = True
        s = solve()
        while it < 3 * K and s[passive].min() <= 0:
            it += 1
            bad = passive & (s <= 0)
            step = (x[bad] / (x[bad] - s[bad])).min()
            x = x * (1 - step) + step * s
            passive[x <= tolx] = False
            x[~passive] = 0.0
            s = solve()
        x = s
        w = b - G @ x
    return x


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


M, N, K = 811, 9, 4
PURITY = np.random.RandomState(2).uniform(0.3, 0.9, size=N)
# (case, init option, n_u, seed)
CASES = [("partial", "uniform", 2, 3), ("partial", "SVD", 2, 1), ("partial", "SVD", 3, 5), ("purity", "SVD", 2, 4),
         ("purity", "uniform", 1, 6), ("free", "SVD", 3, 2), ("refbased", None, 0, None)]


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
        from demethify_b200 import sharded as sh
        X, D, Rk = synth(7, M, N, K, 3)
        lo, hi = sh.row_range(M, rank, world)
        res = {}
        for i, (case, opt, n_u, seed) in enumerate(CASES):
            if case == "free":
                u, a = sh.unsupervised_init_sharded(opt, None, None, n_u, seed=seed, backend=NumpyInitBackend(X[lo:hi], D[lo:hi], None))
            elif case == "refbased":
                u, a = np.zeros((hi - lo, 0)), sh.wls_all_samples_sharded(None, None, None, y_is_dx=True,
                                                                        backend=NumpyInitBackend(X[lo:hi], D[lo:hi], Rk[lo:hi]))
            elif case == "purity":
                u, a = sh.init_BSSMF_md_p_sharded(opt, None, None, None, n_u, PURITY, seed=seed,
                                                  backend=NumpyInitBackend(X[lo:hi], D[lo:hi], Rk[lo:hi]))
            else:
                u, a = sh.init_BSSMF_md_sharded(opt, None, None, None, n_u, seed=seed, backend=NumpyInitBackend(X[lo:hi], D[lo:hi], Rk[lo:hi]))
            res[f"u{i}"], res[f"a{i}"] = u, a
        # a negative entry of X: every rank raises (the flag is all-reduced), as nndsvd_initialize does
        Xn = X.copy()
        Xn[M - 1, 0] = -0.5
        try:
            sh.unsupervised_init_sharded("SVD", None, None, 2, seed=1, backend=NumpyInitBackend(Xn[lo:hi], D[lo:hi], None))
            res["neg"] = "none"
        except ValueError as e:
            res["neg"] = str(e)
        try:
            sh.ShardedInit(NumpyInitBackend(X[lo:hi], D[lo:hi], None)).nndsvd(N + 1)      # rank > min(M, N)
            res["rank"] = "none"
        except IndexError:
            res["rank"] = "IndexError"
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), lo=lo, hi=hi, **res)
    finally:
        dist.destroy_process_group()


def _single_process(case, opt, n_u, seed):
    X, D, Rk = synth(7, M, N, K, 3)
    if case == "free":
        W, H = orc.nndsvd_factors(X, n_u)
        return W.clip(0, 1), orc.simplex_project_columns(H)
    if case == "refbased":
        return np.zeros((M, 0)), orc.reference_based_fit(X, D, Rk)
    if case == "purity":
        u, _, a = orc.draw_init_purity(opt, X, D, Rk, n_u, PURITY, seed=seed)
        return u, a
    u, _, a = orc.draw_init(opt, X, D, Rk, n_u, seed=seed)
    return u, a


@pytest.mark.timeout(600)
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_init_matches_single_process_gloo(tmp_path, world):
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    r = [np.load(tmp_path / f"rank{k}.npz") for k in range(world)]
    assert int(r[0]["lo"]) == 0 and int(r[-1]["hi"]) == M
    for i, case in enumerate(CASES):
        u1, a1 = _single_process(*case)
        assert all(np.array_equal(r[0][f"a{i}"], q[f"a{i}"]) for q in r), case          # alpha is the same on every rank
        u = np.vstack([q[f"u{i}"] for q in r])
        assert np.abs(r[0][f"a{i}"] - a1).max() <= 1e-10, case
        assert u.shape == u1.shape and (u.size == 0 or np.abs(u - u1).max() <= 1e-10), case
    for q in r:
        assert str(q["neg"]) == "The input matrix contains negative elements." and str(q["rank"]) == "IndexError"


def test_numpy_backend_single_rank_wls_equals_oracle():
    """World 1 (no process group): the moment-form WLS of the numpy backend is the oracle's per-sample fit."""
    from demethify_b200 import sharded as sh
    X, D, Rk = synth(9, 500, 6, 5, 2)
    got = sh.wls_all_samples_sharded(None, None, None, backend=NumpyInitBackend(X, D, Rk))
    want = np.stack([orc.wls_simplex_fit(X[:, j], D[:, j], Rk) for j in range(6)], axis=1)
    assert np.abs(got - want).max() <= 1e-10
