"""CpG-row sharding of ONE fit over the GPUs of a box (SURVEY.md 8 e1 (ii); BASELINE config 5).

One process per GPU (torch.distributed, NCCL over NVLink).  Rank r holds a contiguous row range of X, d_x, R_trunc
and u plus a replica of alpha and of the fit state.  Per outer iteration (deconvolution.py:206-221 / :320-335):

  U step      row-local, no communication          (dmf_gram_u_inner on the rows' statistics)
  alpha step  ONE sum all-reduce of the per-sample statistics [G_j | bx_j | ||u||^2]  (Kt (Kt + 1) N + 8 doubles per fit),
              then every rank runs the identical n_iter2 inner iterations on the reduced copy (dmf_gram_alpha_inner)
  cost        ONE sum all-reduce of 8 doubles per fit, then the identical termination test on every rank

plus one max all-reduce (max d_x) at set-up.  Shapes without the Gram form (more unknown types, or wider cohorts with many
types) run the stream engine's passes instead: n_iter2 U passes then ONE scalar all-reduce (||u||^2, l_h), n_iter2 x (alpha or
Frank-Wolfe pass, ONE all-reduce of the Kt x N gradient, the identical step on every rank), and the cost as above: n_iter2 + 2
collectives per outer iteration.  The initial iterate is computed on the same row shards (`ShardedInit`): the
`uniform` init and the reference-based fit all-reduce the WLS moment matrix, the SVD inits the N x N Gram matrix of the residual
and the NNDSVD column norms.  Every rank therefore holds the same alpha and makes the same termination
decision; u stays distributed.  `RowShardedFit` is the orchestration; the arithmetic sits behind a small backend
interface whose product implementation (`GpuShardBackend`) drives libdemethify_sm100 through `FitBatch`.
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from .deconvolution import _initial_iterate, _quiet, set_seed
from .engine import DeviceProblem, FitBatch, _handle, _stream_ptr, to_device
from .init_func import aligned_workspace, wls_desc

__all__ = ["row_range", "GpuShardBackend", "RowShardedFit", "mdwbssmf_deconv_sharded", "fit_row_sharded", "last_info", "GpuInitBackend",
           "ShardedInit", "wls_all_samples_sharded", "init_BSSMF_md_sharded", "init_BSSMF_md_p_sharded", "unsupervised_init_sharded"]

_peer_cache = {}    # (group, world, device) -> (symmetric buffer, rendezvous handle, bytes): see enable_peer_exchange
last_info = {}      # of the most recent row-sharded fit (fit_row_sharded): {"peer_exchange": bool, "peer_error": str | None, "collectives": int}


def row_range(M, rank, world):
    """Rows [lo, hi) of rank `rank`: row m belongs to rank floor(m * world / M) (SURVEY 8 e1)."""
    lo = (M * rank + world - 1) // world
    hi = (M * (rank + 1) + world - 1) // world
    return lo, hi


class GpuShardBackend:
    """This rank's rows on its GPU: a FitBatch in sharded mode on the fused, Gram-form or stream engine (by shape).  One fit, or several when U0_local and A0 are lists of
    initial iterates (CCC restarts, BCV folds); X_local is then one problem all fits share, or a list of resident DeviceProblems,
    one per fit.  Every fit has its own statistics block, all-reduced copy and peer slot, so one all-reduce per step covers all."""

    def __init__(self, X_local, D_local, Rk_local, n_u, U0_local, A0, mode=_lib.DMF_MODE_PARTIAL, purity=None, precision=None, engine=None):
        if isinstance(X_local, (list, tuple)):
            self.prob = list(X_local)
        else:
            self.prob = X_local if isinstance(X_local, DeviceProblem) else DeviceProblem(X_local, D_local, Rk_local, precision=precision)
        U0s, A0s = (list(U0_local), list(A0)) if isinstance(U0_local, (list, tuple)) else ([U0_local], [A0])
        self.batch = FitBatch(self.prob, n_u, U0s, A0s, mode=mode, purity=purity, engine=engine)
        lib, b = _lib.lib(), self.batch
        _lib.check(lib.dmf_batch_set_sharded(b.b, 1, _stream_ptr()))
        # fused engine where the shape allows it: ONE pass and ONE all-reduce per outer iteration (RowShardedFit.outer)
        self.fused = b.engine == "fused"
        self.stream = b.engine == "stream"         # shapes without the Gram form: one pass per reference step
        loc, glo, per, so = C.c_void_p(), C.c_void_p(), C.c_int64(), C.c_int64()
        _lib.check(lib.dmf_batch_stats_buffers(b.b, C.byref(loc), C.byref(glo), C.byref(per), C.byref(so)))
        base = b.ws.data_ptr()
        nbytes = per.value * 8 * b.n_fits

        def view(ptr):
            off = ptr - base
            return b.ws[off:off + nbytes].view(torch.float64).view(b.n_fits, per.value)
        self.local, self.glob = view(loc.value), view(glo.value)
        self.scal_off = so.value
        self.has_known = b.K > 0
        self.device = b.device
        self.supports_graphs = True
        self.peer = None

    def enable_peer_exchange(self, group=None):
        """All-reduce over NVLink peer memory inside one kernel of the library (dmf_gram_exchange) instead of NCCL: allocates a
        symmetric buffer that every rank of `group` maps (torch symmetric memory) and hands the peer pointers to the library.
        Returns False (and leaves the NCCL path in place) when symmetric memory is not available."""
        if not (dist.is_initialized() and dist.get_world_size(group) > 1):
            return False
        try:
            import torch.distributed._symmetric_memory as symm_mem
            lib, b = _lib.lib(), self.batch
            world, rank = dist.get_world_size(group), dist.get_rank(group)
            nbytes = C.c_size_t()
            _lib.check(lib.dmf_batch_peer_bytes(b.b, world, C.byref(nbytes)))
            # the symmetric buffer and its rendezvous (an exchange of IPC handles through the store: tens of ms) are kept for the
            # process and reused by later fits of the same or a smaller statistics block; every use starts from zeroed flags
            key = (id(group) if group is not None else 0, world, self.device.index)
            cached = _peer_cache.get(key)
            if cached is not None and cached[2] >= nbytes.value:
                buf, hdl = cached[0], cached[1]
            else:
                buf = symm_mem.empty((nbytes.value + 7) // 8, dtype=torch.float64, device=self.device)
                hdl = symm_mem.rendezvous(buf, group if group is not None else dist.group.WORLD)
                _peer_cache[key] = (buf, hdl, nbytes.value)
            buf.zero_()
            ptrs = (C.c_void_p * world)(*[int(p) for p in hdl.buffer_ptrs])
            torch.cuda.synchronize()
            dist.barrier(group)                      # every rank's buffer (flags) is zero before anybody pushes
            _lib.check(lib.dmf_batch_set_peers(b.b, rank, world, ptrs, nbytes.value, _stream_ptr()))
            self.peer = (buf, hdl)
        except Exception as e:                       # no symmetric memory on this system: keep NCCL
            self.peer_error = repr(e)
            self.peer = None
        # the ranks must take the same path: one rank on NCCL while the others wait in the exchange kernel would hang the job
        ok = torch.tensor([1 if self.peer is not None else 0], dtype=torch.int32, device=self.device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
        if int(ok.item()) == 0:
            self.peer = None
        return self.peer is not None

    def exchange(self, which):
        _lib.check(_lib.lib().dmf_gram_exchange(self.batch.b, int(which), _stream_ptr()))

    def reserve(self, n_inner_total):
        """Make the following steps allocation- and sync-free (CUDA-graph capture)."""
        _lib.check(_lib.lib().dmf_batch_reserve_momentum(self.batch.b, int(n_inner_total), _stream_ptr()))

    # ---- statistics blocks: (n_fits, doubles_per_fit) tensors, [G | bx | scal(8)] (Gram form, fused) or [alpha gradient | scal(8)] (stream)
    def stats_local(self):
        return self.local

    def stats_global(self):
        return self.glob

    # ---- this rank's arithmetic
    def rowgram(self, initial, tol):
        self.batch.gram_rowgram(initial, tol)

    def u_inner(self, n_iter2):
        self.batch.gram_u_inner(n_iter2)

    def panels(self, known_block):
        self.batch.gram_panels(known_block)

    def alpha_inner(self, n_iter2):
        self.batch.gram_alpha_inner(n_iter2)

    def fused_pass(self, n_iter2, tol):
        self.batch.fused_pass(n_iter2, tol)

    def fused_alpha_commit(self, n_iter2, tol):
        _lib.check(_lib.lib().dmf_fused_alpha_commit(self.batch.b, int(n_iter2), float(tol), _stream_ptr()))

    # ---- stream engine: [alpha gradient | scal(8)] blocks
    def cost(self, initial, tol):
        if initial:
            self.batch.pass_init()
        else:
            self.batch.pass_cost(tol)

    def pass_u(self):
        self.batch.pass_u()

    def u_commit(self):
        _lib.check(_lib.lib().dmf_pass_u_commit(self.batch.b, _stream_ptr()))

    def pass_alpha(self, k):
        if self.batch.mode == _lib.DMF_MODE_PURITY:
            self.batch.pass_fw(k)
        else:
            self.batch.pass_alpha()

    def alpha_commit(self, k):
        _lib.check(_lib.lib().dmf_pass_alpha_commit(self.batch.b, int(k), _stream_ptr()))

    def finalize_cost(self, initial, tol):
        _lib.check(_lib.lib().dmf_gram_finalize_cost(self.batch.b, int(bool(initial)), float(tol), _stream_ptr()))

    def all_done(self):
        sts = self.batch.states()
        bad = [i for i, s in enumerate(sts) if s.done == 3]
        if bad:
            raise _lib.DmfError(f"non-finite values reached the simplex projection (fit {bad[0]})")
        return all(s.done != 0 for s in sts)

    def results(self):
        """[(u_local, alpha, n_outer, cost)] — u holds only this rank's rows."""
        return self.batch.results()

    def close(self):
        self.batch.close()


class RowShardedFit:
    """Outer loop of the row-sharded fits of `backend` (one or several: each stops at its own termination test, the loop when every
    fit has); `backend` does this rank's arithmetic, `group` is the torch.distributed group."""

    def __init__(self, backend, group=None):
        self.be, self.group = backend, group
        self.so = backend.scal_off
        self.collectives = 0

    def _allreduce(self, t, op=dist.ReduceOp.SUM):
        if dist.is_initialized() and dist.get_world_size(self.group) > 1:
            dist.all_reduce(t, op=op, group=self.group)
        self.collectives += 1

    def _reduce_scal(self, with_max):
        if getattr(self.be, "peer", None) is not None:          # one kernel: push to the peers, wait, rank-ordered sum (max for max d_x)
            self.be.exchange(2 if with_max else 1)
            self.collectives += 1
            return
        loc, glo, so = self.be.stats_local(), self.be.stats_global(), self.so
        sc = loc[:, so:so + 8].contiguous()
        if with_max:
            mx = sc[:, 3].clone()
            self._allreduce(mx, dist.ReduceOp.MAX)
        self._allreduce(sc)
        if with_max:
            sc[:, 3] = mx
        glo[:, so:so + 8] = sc

    def init(self):
        """deconvolution.py:192-204: cost, ||R||^2, max d_x over ALL rows; then this rank's known x known statistics."""
        be = self.be
        stream = getattr(be, "stream", False)
        if stream:
            be.cost(True, 0.0)
        else:
            be.rowgram(True, 0.0)
        self._reduce_scal(with_max=True)
        be.finalize_cost(True, 0.0)
        if be.has_known and not stream:
            be.panels(True)

    def _reduce_blocks(self):
        be = self.be
        if getattr(be, "peer", None) is not None:
            be.exchange(0)                            # G_j, bx_j, scalars over all rows, over NVLink peer memory
            self.collectives += 1
        else:
            glo = be.stats_global()
            glo.copy_(be.stats_local())
            self._allreduce(glo)                      # the same through NCCL

    def use_fused(self, n_iter2):
        return getattr(self.be, "fused", False) and 1 <= n_iter2 <= 64

    def outer(self, n_iter2, tol):
        be = self.be
        if self.use_fused(n_iter2):
            # fused engine: cost of the incoming iterate + U step + panel in ONE pass over this rank's rows, ONE all-reduce of
            # [G_j | bx_j | cost, ||u||^2], then the test / commit / alpha iterations identically on every rank
            be.fused_pass(n_iter2, tol)
            self._reduce_blocks()
            be.fused_alpha_commit(n_iter2, tol)
            self.pending = True
            return
        if getattr(be, "stream", False):
            # stream engine: every pass publishes this rank's sums, the state advances on the all-reduced ones
            for _ in range(n_iter2):
                be.pass_u()                           # row-local; publishes ||u||^2 of this rank's rows
            self._reduce_scal(with_max=False)
            be.u_commit()                             # l_h from ||u||^2 over all rows
            for k in range(n_iter2):
                be.pass_alpha(k)                      # this rank's Kt x N gradient (Frank-Wolfe iteration k for purity fits)
                self._reduce_blocks()
                be.alpha_commit(k)                    # the identical step on every rank
            be.cost(False, tol)
            self._reduce_scal(with_max=False)
            be.finalize_cost(False, tol)
            return
        if n_iter2 > 0:
            be.u_inner(n_iter2)                       # row-local
            be.panels(False)
            if getattr(be, "peer", None) is not None:
                be.exchange(0)                        # G_j, bx_j, ||u||^2 over all rows, over NVLink peer memory
                self.collectives += 1
            else:
                glo = be.stats_global()
                glo.copy_(be.stats_local())
                self._allreduce(glo)                  # the same through NCCL
            be.alpha_inner(n_iter2)                   # identical on every rank
        be.rowgram(False, tol)
        self._reduce_scal(with_max=False)
        be.finalize_cost(False, tol)                  # identical termination decision on every rank

    def finish(self, tol):
        """Fused engine: the cost of the last iterate is still pending after the last outer() - one cost-only pass."""
        if getattr(self, "pending", False):
            self.pending = False
            if not self.be.all_done():
                self.be.rowgram(False, tol)
                self._reduce_scal(with_max=False)
                self.be.finalize_cost(False, tol)

    def capture_outer(self, n_iter2, tol):
        """One outer iteration (kernels, D2D copies and both NCCL all-reduces) as a CUDA graph: a replay costs one launch
        instead of ~12 host calls, which is what bounds strong scaling once a rank's share of the rows takes < 0.2 ms."""
        self.outer(n_iter2, tol)                      # eager once: NCCL and the allocator are warm before the capture
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self.outer(n_iter2, tol)
        return graph

    def fit(self, n_iter1, n_iter2, tol, use_graph=None):
        self.init()
        issued, chunk = 0, 2
        graph = None
        if use_graph is None:      # opt-in: DMF_SHARDED_GRAPH=1 (see DESIGN.md 6 for what was measured)
            import os
            use_graph = getattr(self.be, "supports_graphs", False) and n_iter1 > 4 and os.environ.get("DMF_SHARDED_GRAPH", "0") == "1"
        if use_graph:
            self.be.reserve((n_iter1 + 2) * max(n_iter2, 1))
            graph = self.capture_outer(n_iter2, tol)
            issued = 1
            if self.be.all_done():
                return self.be.results()
        while issued < n_iter1:
            todo = min(chunk, n_iter1 - issued)
            for _ in range(todo):
                if graph is not None:
                    graph.replay()
                else:
                    self.outer(n_iter2, tol)
            issued += todo
            if self.be.all_done():                    # the state is replicated: every rank leaves the loop together
                self.pending = False
                break
            chunk = min(chunk * 2, 16)
        self.finish(tol)
        return self.be.results()


def mdwbssmf_deconv_sharded(u_local, alpha, X_local, d_local, R_local, n_u, n_iter1=100000, n_iter2=50, tol=1e-3, purity=None,
                            group=None):
    """mdwbssmf_deconv / mdwbssmf_deconv_p (deconvolution.py:190-223, :305-337) on a row-sharded problem: every rank passes
    ITS rows of u, X, d_x, R_trunc (see `row_range`), or a resident DeviceProblem of them as X_local, and the full alpha; returns
    (u_local, alpha, n_outer, cost)."""
    has_ref = R_local is not None or (isinstance(X_local, DeviceProblem) and X_local.K > 0)
    mode = _lib.DMF_MODE_PURITY if purity is not None else (_lib.DMF_MODE_PARTIAL if has_ref else _lib.DMF_MODE_UNSUPERVISED)
    be = GpuShardBackend(X_local, d_local, R_local, n_u, np.asarray(u_local).reshape(-1, n_u), np.asarray(alpha), mode=mode, purity=purity)
    (u, a, n_outer, cost), = fit_row_sharded(be, n_iter1, n_iter2, tol, group)
    return u, a, n_outer, cost


def fit_row_sharded(be, n_iter1, n_iter2, tol, group=None):
    """Run every fit of the shard backend `be` to its own termination over `group`, then close the backend ->
    [(u_local, alpha, n_outer, cost)] per fit.  A GPU backend all-reduces in-kernel over NVLink peer memory unless DMF_PEER_XCHG=0
    (NCCL is the fall-back when symmetric memory is unavailable)."""
    import os
    if isinstance(be, GpuShardBackend) and os.environ.get("DMF_PEER_XCHG", "1") != "0":
        be.enable_peer_exchange(group)
    fit = RowShardedFit(be, group)
    try:
        return fit.fit(n_iter1, n_iter2, tol)
    finally:
        last_info.update(peer_exchange=getattr(be, "peer", None) is not None, peer_error=getattr(be, "peer_error", None),
                         collectives=fit.collectives)
        if isinstance(be, GpuShardBackend):
            torch.cuda.synchronize()
        be.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# The initial iterate on row-sharded data

class GpuInitBackend:
    """This rank's rows on its GPU for the initial iterate: the WLS moments (dmf_wls_moments / dmf_wls_solve) and the residual
    reductions of the SVD inits (dmf_resid_gram / dmf_resid_project / dmf_nndsvd_apply)."""

    def __init__(self, X_local, D_local, R_local, precision=None):
        self.prob = X_local if isinstance(X_local, DeviceProblem) else DeviceProblem(X_local, D_local, R_local, precision=precision)
        self.device = self.prob.device
        self.M, self.N, self.K = self.prob.M, self.prob.N, self.prob.K
        self.h = _handle(self.device.index if self.device.index is not None else torch.cuda.current_device())

    def _wls_ws(self, desc):
        nbytes = C.c_size_t()
        _lib.check(_lib.lib().dmf_wls_workspace_bytes(self.h, C.byref(desc), C.byref(nbytes)))
        return nbytes.value

    def wls_moments(self, extra, y_is_dx):
        """[(Kz Kz), N] moment matrix of this rank's rows (device tensor)."""
        desc, out, keep = wls_desc(self.prob, extra, y_is_dx)
        kz = self.K + (0 if extra is None else np.shape(extra)[1]) + 2
        mom = torch.empty((kz * kz, self.N), dtype=torch.float64, device=self.device)
        nbytes = self._wls_ws(desc) if self.M > 0 else 0
        ws, ws_ptr = aligned_workspace(nbytes, self.device)
        _lib.check(_lib.lib().dmf_wls_moments(self.h, C.byref(desc), C.c_void_p(mom.data_ptr()), ws_ptr, nbytes, _stream_ptr()))
        return mom

    def wls_solve(self, mom, M, K2):
        """Per-sample NNLS on the all-reduced moments; M is the global row count -> (K + K2) x N ndarray."""
        out = torch.zeros((self.K + K2, self.N), dtype=torch.float64, device=self.device)
        desc = _lib.WlsDesc(M=int(M), N=self.N, K=self.K, K2=int(K2), out=out.data_ptr())
        ws, ws_ptr = aligned_workspace(256, self.device)
        _lib.check(_lib.lib().dmf_wls_solve(self.h, C.byref(desc), C.c_void_p(mom.data_ptr()), ws_ptr, 256, _stream_ptr()))
        return out.cpu().numpy()

    def _resid(self, H1):
        """dmf_resid_desc_t over fp64 rows: r = max(x - R H1, 1e-8), or r = x when H1 is None (the reference-free init)."""
        p = self.prob
        X = p.X if p.dtype == torch.float64 else p.X.to(torch.float64)
        keep = [X]
        d = _lib.ResidDesc(M=p.M, N=p.N, K=0, ldx=X.shape[1], ldr=0, X=X.data_ptr())
        if H1 is not None:
            R = p.Rk if p.dtype == torch.float64 else p.Rk.to(torch.float64)
            H = to_device(np.ascontiguousarray(H1, dtype=np.float64), torch.float64, self.device)
            keep += [R, H]
            d.K, d.ldr, d.R, d.H1 = p.K, R.shape[1], R.data_ptr(), H.data_ptr()
        nbytes = C.c_size_t()
        _lib.check(_lib.lib().dmf_resid_workspace_bytes(self.h, C.byref(d), C.byref(nbytes)))
        ws, ws_ptr = aligned_workspace(nbytes.value, self.device)
        keep.append(ws)
        return d, ws_ptr, nbytes.value, keep

    def resid_gram(self, H1):
        """(sum over this rank's rows of r_m r_m^T (N x N), 1 where X has a negative entry (reference-free) else 0), device tensors."""
        d, ws_ptr, nbytes, keep = self._resid(H1)
        G = torch.empty((self.N, self.N), dtype=torch.float64, device=self.device)
        neg = torch.zeros(1, dtype=torch.int32, device=self.device)
        _lib.check(_lib.lib().dmf_resid_gram(self.h, C.byref(d), C.c_void_p(G.data_ptr()), C.c_void_p(neg.data_ptr()), ws_ptr, nbytes,
                                             _stream_ptr()))
        return G, neg

    def resid_project(self, H1, Vh, inv_sigma):
        """(U = r Vh^T diag(inv_sigma) of this rank's rows, [|u+|^2 per component, |u-|^2 per component] of those rows)."""
        d, ws_ptr, nbytes, keep = self._resid(H1)
        rank = Vh.shape[0]
        Vh, inv_sigma = Vh.contiguous(), inv_sigma.contiguous()
        U = torch.empty((self.M, rank), dtype=torch.float64, device=self.device)
        sums = torch.empty(2 * rank, dtype=torch.float64, device=self.device)
        _lib.check(_lib.lib().dmf_resid_project(self.h, C.byref(d), C.c_void_p(Vh.data_ptr()), C.c_void_p(inv_sigma.data_ptr()), rank,
                                                C.c_void_p(U.data_ptr()), C.c_void_p(sums.data_ptr()), ws_ptr, nbytes, _stream_ptr()))
        return U, sums

    def nndsvd_apply(self, U, Vh, sigma, sums):
        """NNDSVD factors (W rows of this rank, H) from U and the all-reduced sums -> ndarrays."""
        rank = Vh.shape[0]
        Vh, sigma, sums = Vh.contiguous(), sigma.contiguous(), sums.contiguous()
        W = torch.empty((self.M, rank), dtype=torch.float64, device=self.device)
        H = torch.empty((rank, self.N), dtype=torch.float64, device=self.device)
        _lib.check(_lib.lib().dmf_nndsvd_apply(C.c_void_p(U.data_ptr()), self.M, C.c_void_p(Vh.data_ptr()), C.c_void_p(sigma.data_ptr()),
                                               C.c_void_p(sums.data_ptr()), self.N, rank, C.c_void_p(W.data_ptr()),
                                               C.c_void_p(H.data_ptr()), _stream_ptr()))
        return W.cpu().numpy(), H.cpu().numpy()


class ShardedInit:
    """The row reductions of the initial iterate on row-sharded data; `backend` does this rank's arithmetic (GpuInitBackend, or a
    numpy restatement in the tests), every rank of `group` calls the same steps in the same order."""

    def __init__(self, backend, group=None):
        self.be, self.group = backend, group
        rows = torch.tensor([backend.M], dtype=torch.int64, device=backend.device)
        if self._multi():
            parts = [torch.zeros_like(rows) for _ in range(dist.get_world_size(group))]
            dist.all_gather(parts, rows, group=group)
            counts = [int(t.item()) for t in parts]
        else:
            counts = [backend.M]
        rank = dist.get_rank(group) if self._multi() else 0
        self.M = sum(counts)                          # global row count
        self.lo = sum(counts[:rank])                  # this rank's rows are lo .. lo + backend.M of the full matrix
        self.hi = self.lo + backend.M

    def _multi(self):
        return dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1

    def _allreduce(self, t, op=None):
        if self._multi():
            dist.all_reduce(t, op=op or dist.ReduceOp.SUM, group=self.group)
        return t

    def _broadcast(self, t):
        if self._multi():
            dist.broadcast(t, src=dist.get_global_rank(self.group, 0) if self.group is not None else 0, group=self.group)
        return t

    def wls(self, extra=None, y_is_dx=False):
        """wls_intercept of every sample over all rows (init_func.py:8-14): `extra` holds this rank's rows of the second regressor
        block.  -> (K + K2) x N ndarray, the same on every rank."""
        mom = self._allreduce(self.be.wls_moments(extra, y_is_dx))
        return self.be.wls_solve(mom, self.M, 0 if extra is None else np.shape(extra)[1])

    def nndsvd(self, rank, H1=None):
        """nndsvd_initialize (init_func.py:40-82, flag 0) of the residual max(X - R_trunc H1, 1e-8), or of X when H1 is None, over
        all rows -> (this rank's rows of W, H).  The right singular vectors and the singular values come from the eigen-
        decomposition of the all-reduced N x N Gram matrix (descending, sigma = sqrt(max(lambda, 0))), the left ones from
        projecting this rank's residual rows on them."""
        G, neg = self.be.resid_gram(H1)
        self._allreduce(G)
        if H1 is None and int(self._allreduce(neg, dist.ReduceOp.MAX).item()):
            raise ValueError("The input matrix contains negative elements.")
        if rank > min(self.M, self.be.N):
            raise IndexError(f"index {min(self.M, self.be.N)} is out of bounds for axis 1 with size {min(self.M, self.be.N)}")
        lam, V = torch.linalg.eigh(G)
        order = torch.arange(G.shape[0] - 1, G.shape[0] - 1 - rank, -1, device=G.device)
        Vh = V[:, order].T.contiguous()
        sigma = torch.sqrt(torch.clamp(lam[order], min=0.0)).contiguous()
        self._broadcast(Vh)                           # one decomposition for all ranks
        self._broadcast(sigma)
        inv = torch.where(sigma > 0, 1.0 / sigma, torch.zeros_like(sigma))
        U, sums = self.be.resid_project(H1, Vh, inv)
        self._allreduce(sums)
        return self.be.nndsvd_apply(U, Vh, sigma, sums)


def _init_of(backend, X_local, d_local, R_local, group):
    return ShardedInit(backend if backend is not None else GpuInitBackend(X_local, d_local, R_local), group)


def wls_all_samples_sharded(X_local, d_local, R_local, extra=None, y_is_dx=False, group=None, backend=None):
    """init_func.wls_all_samples over row-sharded data: every rank passes ITS rows (and its rows of `extra`) -> (K [+ K2], N)
    ndarray, the same on every rank.  With y_is_dx it is the reference-based fit (n_u = 0, demethify.py:209-213)."""
    return _init_of(backend, X_local, d_local, R_local, group).wls(extra, y_is_dx)


def init_BSSMF_md_sharded(init_option, X_local, d_local, R_local, n_u, seed=None, group=None, backend=None):
    """deconvolution.init_BSSMF_md over row-sharded data: every rank passes ITS rows of X, d_x and R_trunc (or a resident
    DeviceProblem of them) -> (u_local, alpha); alpha is the same on every rank and u_local holds this rank's rows of the
    single-process u."""
    set_seed(seed)
    si = _init_of(backend, X_local, d_local, R_local, group)
    return _initial_iterate("partial", init_option, si.M, si.be.N, si.be.K, n_u, rows=(si.lo, si.hi), wls=si.wls, nndsvd=si.nndsvd)


def init_BSSMF_md_p_sharded(init_option, X_local, d_local, R_local, n_u, purity, seed=None, group=None, backend=None):
    """deconvolution.init_BSSMF_md_p over row-sharded data -> (u_local, alpha); rank 0 prints the fallback message."""
    set_seed(seed)
    si = _init_of(backend, X_local, d_local, R_local, group)
    say = print if not si._multi() or dist.get_rank(group) == 0 else _quiet
    return _initial_iterate("purity", init_option, si.M, si.be.N, si.be.K, n_u, rows=(si.lo, si.hi), wls=si.wls, nndsvd=si.nndsvd,
                            purity=purity, say=say)


def unsupervised_init_sharded(init_option, X_local, d_local, n_u, seed=None, group=None, backend=None):
    """The initial iterate of deconvolution.unsupervised_deconv (deconvolution.py:107-150) over row-sharded data ->
    (u_local, alpha)."""
    set_seed(seed)
    si = _init_of(backend, X_local, d_local, None, group)
    return _initial_iterate("free", init_option, si.M, si.be.N, 0, n_u, rows=(si.lo, si.hi), wls=si.wls, nndsvd=si.nndsvd)
