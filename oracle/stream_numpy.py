"""numpy (fp64) restatement of the stream engine's row-sharded steps (demethify_b200/csrc/dmf_kernels.cuh with kFlagPartial, the
commit kernels of dmf_gram.cuh) as a shard backend.

TEST INFRASTRUCTURE — see oracle/__init__.py.  Same interface as the stream branch of demethify_b200.sharded.GpuShardBackend:
every pass publishes this shard's sums in the `local` block [alpha gradient (Kt*N) | scal (8)], and the state advances on the
all-reduced `global` block, so `RowShardedFit` can be exercised on CPU with the gloo backend for shapes without the Gram form.

Reference lines restated: set-up deconvolution.py:192-204, update_u :82-89 (unsupervised variant :157-164), update_alpha
:94-101 with projection :21-37, frank_wolfe_nmf :285-299, cost/termination :218-221.
"""
import numpy as np
import torch

from .bssmf_numpy import simplex_project_columns
from .gram_numpy import NumpyShardBackend


class NumpyStreamShardBackend(NumpyShardBackend):
    """One fit on this shard's rows.  The set-up and the termination test on the reduced scalars (finalize_cost), all_done and
    results are the Gram-form backend's; the passes below are one reference step each."""

    stream = True

    def __init__(self, X, D, Rk, n_u, U0, A0, mode="partial", purity=None):
        super().__init__(X, D, Rk, n_u, U0, A0, mode=mode, purity=purity)
        self.scal_off = self.Kt * self.N
        self.local = torch.zeros((1, self.scal_off + 8), dtype=torch.float64)
        self.glob = torch.zeros_like(self.local)

    def _R(self):
        return np.hstack([self.Rk, self.u])

    # ---- cost pass: cost of this shard's rows (and at set-up ||R_trunc||^2, ||u||^2, max d_x)
    def cost(self, initial, tol):
        if self.st["done"]:
            return
        sc = self.local[0, self.scal_off:].numpy()
        sc[0] = float(np.sum(self.D * (self.X - self._R() @ self.A) ** 2))
        if initial:
            sc[1], sc[2] = float(np.sum(self.Rk ** 2)), float(np.sum(self.u ** 2))
            sc[3] = float(self.D.max()) if self.D.size else 0.0
            sc[4] = sc[2]

    # ---- one update_u iteration, row-local; publishes ||u||^2 of this shard
    def pass_u(self):
        st = self.st
        if st["done"]:
            return
        self._mom(st["t_u"] + 1)
        l_w = st["l_w"]
        beta = min(self.mom_m[st["t_u"]], 0.9999 * np.sqrt(st["l_w_old"] / l_w))
        u, up = self.u, self.u_prev
        ut = u + beta * (u - up)
        ug = u if self.mode == "unsupervised" else ut
        Ak, Au = self.A[:self.K], self.A[self.K:]
        g = (self.D * ((self.X - self.Rk @ Ak) - ug @ Au)) @ Au.T
        self.u_prev, self.u = u, np.clip(ut + g / l_w, 0, 1)
        st["t_u"] += 1
        st["l_w_old"] = l_w
        self.local[0, self.scal_off + 4] = float(np.sum(self.u ** 2))

    def u_commit(self):
        st = self.st
        if st["done"]:
            return
        st["ssq_u"] = float(self.glob[0, self.scal_off + 4])
        st["l_h"] = np.sqrt(st["ssq_rk"] + st["ssq_u"]) ** 2 * st["dmax2"]

    def _beta_a(self):
        st = self.st
        return min(self.mom_m[st["t_a"]], 0.9999 * np.sqrt(st["l_h_old"] / st["l_h"]))

    # ---- gradient R^T (d o (x - R alpha_eval)) of this shard: alpha_temp (projected gradient) or alpha (Frank-Wolfe)
    def pass_alpha(self, k):
        st = self.st
        if st["done"]:
            return
        self._mom(st["t_a"] + 1)
        A = self.A if self.mode == "purity" else self.A + self._beta_a() * (self.A - self.A_prev)
        R = self._R()
        G = R.T @ (self.D * (self.X - R @ A))
        self.local[0, :self.scal_off] = torch.from_numpy(G.reshape(-1))

    # ---- the step on the all-reduced gradient, identical on every rank
    def alpha_commit(self, k):
        st = self.st
        if st["done"]:
            return
        G = self.glob[0, :self.scal_off].numpy().reshape(self.Kt, self.N)
        if self.mode != "purity":
            At = self.A + self._beta_a() * (self.A - self.A_prev)
            self.A_prev, self.A = self.A, simplex_project_columns(At + G / st["l_h"])
            st["t_a"] += 1
            st["l_h_old"] = st["l_h"]
        else:
            K, cols, grad = self.K, np.arange(self.N), -G
            S = np.zeros_like(self.A)
            S[np.argmin(grad[:K], axis=0), cols] = self.purity
            S[K + np.argmin(grad[K:], axis=0), cols] = 1 - self.purity
            gamma = 2 / (k + 2)
            self.A = (1 - gamma) * self.A + gamma * S
        st["l_w"] = np.linalg.norm(self.A[self.K:]) ** 2 * st["dmax2"]
