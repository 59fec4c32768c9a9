"""Device-side plumbing between the reference-shaped Python API and the C ABI.

torch is used for device memory, streams and host<->device copies only; every arithmetic step on the
deconvolution path is a kernel of libdemethify_sm100.so reached through `_lib` (ctypes).

  DeviceProblem : X, d_x, R_trunc resident in HBM (d_x narrowed to uint16 when it is integer coverage)
  FitBatch      : a set of independent fits of one shape (restarts, bootstrap resamples, BCV folds)
"""
import ctypes as C

import numpy as np
import torch

from . import _lib, get_engine, get_precision

_handles = {}

# FitBatch gives the fused engine its four U slots wherever the shape qualifies; tests switch this off to exercise the
# Gram-form engine on the same shapes
FUSED_SLOTS = True


def _handle(device_index):
    if device_index not in _handles:
        h = C.c_void_p()
        _lib.check(_lib.lib().dmf_create(device_index, C.byref(h)))
        _handles[device_index] = h
    return _handles[device_index]


def _require_cuda():
    if not torch.cuda.is_available():
        raise _lib.DmfError("demethify_b200 needs a CUDA device (B200); there is no CPU fallback")


def current_device():
    _require_cuda()
    return torch.device("cuda", torch.cuda.current_device())


def _stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _tdtype(precision):
    return torch.float64 if precision == "fp64" else torch.float32


def device_free_bytes(device):
    free, _total = torch.cuda.mem_get_info(device)
    return int(free)


def _even(n):
    return n + (n & 1)


def _pad_cols(t, width):
    """Zero-pad a 2-D device tensor on the right to `width` columns (ABI: even pitches, zero padding)."""
    if t.shape[1] == width:
        return t.contiguous()
    out = torch.zeros((t.shape[0], width), dtype=t.dtype, device=t.device)
    out[:, :t.shape[1]].copy_(t)
    return out


def to_device(arr, dtype=None, device=None):
    """Host ndarray / tensor -> contiguous device tensor (async when the source is pinned)."""
    device = device or current_device()
    if isinstance(arr, torch.Tensor):
        t = arr
    else:
        a = np.asarray(arr)
        if not a.flags.c_contiguous:
            a = np.ascontiguousarray(a)        # pandas .values arrive F-ordered (SURVEY 8 a1)
        if not a.flags.writeable:
            a = a.copy()
        t = torch.from_numpy(a)
    t = t.to(device, non_blocking=True)
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


class DeviceProblem:
    """X (M x N), d_x (M x N) and R_trunc (M x K, optional) in HBM in the layout the kernels stream."""

    def __init__(self, X, D, Rk=None, precision=None, narrow_weights=True, device=None):
        _require_cuda()
        self.precision = precision or get_precision()
        self.device = device or current_device()
        self.dtype = _tdtype(self.precision)
        X = to_device(X, self.dtype, self.device)
        self.M, self.N = X.shape
        # Row pitches (include/demethify_b200.h): a row tile reaches shared memory as ONE bulk copy and keeps its pitch there, so
        # the pitch decides the shared-memory bank pattern of the kernels that walk several rows per warp instruction (the fused
        # engine's MMA fragments).  pitch = 16 bytes beyond a multiple of 128 bytes (X and u16 weights) is conflict free.
        es = 8 if self.dtype == torch.float64 else 4
        self.wide = self.N * es >= 512              # short rows: bank conflicts do not matter, padding would (tile geometry, bytes)
        self.ldx = ((self.N * es + 127) // 128 * 128 + 16) // es if self.wide else (self.N + 7) // 8 * 8
        self.X = _pad_cols(X, self.ldx)
        self._set_reference(Rk)
        self.set_weights(D, narrow_weights)

    def _set_reference(self, Rk):
        self.K = 0
        self.Rk = None
        if Rk is not None:
            Rk = to_device(Rk, self.dtype, self.device)
            if Rk.ndim != 2 or Rk.shape[0] != self.M:
                raise ValueError("R_trunc must be M x K")
            self.K = Rk.shape[1]
            self.Rk = _pad_cols(Rk, _even(self.K))

    @property
    def shape(self):
        """(M, N) like the meth_frequency array it holds (lets the reference-shaped entry points take a resident problem)."""
        return (self.M, self.N)

    def set_weights(self, D, narrow=True):
        """Upload d_x.  Integer coverage in [0, 65535] is stored as uint16 (2 B/entry instead of 8)."""
        raw = to_device(D, None, self.device)
        if tuple(raw.shape) != (self.M, self.N):
            raise ValueError("d_x must have the shape of meth_frequency")
        self.wtype = _lib.DMF_W_FLOAT
        self.D = None
        es = 8 if self.dtype == torch.float64 else 4
        self.ldd = self.ldx                                        # float weights: the pitch of X
        if raw.dtype == torch.uint16:                              # already narrow (the CLI reader stages coverage as uint16): no check needed
            ldd16 = ((self.N * 2 + 127) // 128 * 128 + 16) // 2 if self.wide else (self.N + 7) // 8 * 8
            self.D, self.wtype, self.ldd = _pad_cols(raw, ldd16), _lib.DMF_W_U16, ldd16
            return
        if narrow:
            kind = {torch.float64: 0, torch.float32: 1, torch.int64: 2}.get(raw.dtype)
            if kind is None:
                raw = raw.to(torch.float64)
                kind = 0
            # u16 weights: 16 bytes beyond a multiple of 128 (wide rows), else 16-byte aligned rows
            ldd16 = ((self.N * 2 + 127) // 128 * 128 + 16) // 2 if self.wide else (self.N + 7) // 8 * 8
            raw16 = _pad_cols(raw, ldd16)
            packed = torch.empty((self.M, ldd16), dtype=torch.uint16, device=self.device)
            bad = torch.zeros(1, dtype=torch.int32, device=self.device)
            _lib.check(_lib.lib().dmf_pack_weights_u16(C.c_void_p(raw16.data_ptr()), kind, raw16.numel(), C.c_void_p(packed.data_ptr()),
                                                       C.c_void_p(bad.data_ptr()), _stream_ptr()))
            if int(bad.item()) == 0:
                self.D, self.wtype, self.ldd = packed, _lib.DMF_W_U16, ldd16
            del raw16
        if self.D is None:
            self.D = _pad_cols(raw.to(self.dtype), self.ldx)

    def masked(self, mask):
        """Problem with weights d_x * mask (BCV training folds, ic.py:75): zero weight == entry left out, so X is shared."""
        m = to_device(np.ascontiguousarray(mask), None, self.device)
        if self.D.dtype == torch.uint16:        # 0/1 multiply through the int16 view (bit-exact for every u16 value)
            m = _pad_cols(m.to(torch.int16), self.ldd)
            return self.with_weights((self.D.view(torch.int16) * m).view(torch.uint16), self.wtype)
        m = _pad_cols(m.to(self.D.dtype), self.ldd)
        return self.with_weights(self.D * m, self.wtype)

    def gathered(self, idx):
        """New problem holding rows idx of X, d_x, R_trunc (row gather kernel of the library; bootstrap.py:28)."""
        rows = idx.to(self.device, torch.int32) if isinstance(idx, torch.Tensor) else to_device(np.asarray(idx, dtype=np.int32), torch.int32, self.device)
        other = object.__new__(DeviceProblem)
        other.__dict__.update(self.__dict__)
        n = rows.numel()
        lib = _lib.lib()

        def take(t):
            out = torch.empty((n, t.shape[1]), dtype=t.dtype, device=t.device)
            _lib.check(lib.dmf_gather_rows(C.c_void_p(t.data_ptr()), C.c_void_p(rows.data_ptr()), n, t.shape[1], t.element_size(),
                                           C.c_void_p(out.data_ptr()), _stream_ptr()))
            return out
        other.X, other.D = take(self.X), take(self.D)
        other.Rk = take(self.Rk) if self.Rk is not None else None
        other.M = n
        return other

    def gathered_many(self, idx):
        """One problem per row of idx (B x n int32 device tensor): the B resampled copies of X, d_x, R_trunc live in three stacked
        tensors (one allocation per matrix and wave instead of three per resample - the allocations dominated the set-up of a wave)."""
        rows = idx.to(self.device, torch.int32).contiguous()
        B, n = rows.shape
        lib = _lib.lib()

        def take(t):
            out = torch.empty((B, n, t.shape[1]), dtype=t.dtype, device=t.device)
            for k in range(B):
                _lib.check(lib.dmf_gather_rows(C.c_void_p(t.data_ptr()), C.c_void_p(rows[k].data_ptr()), n, t.shape[1], t.element_size(),
                                               C.c_void_p(out[k].data_ptr()), _stream_ptr()))
            return out
        Xs, Ds = take(self.X), take(self.D)
        Rs = take(self.Rk) if self.Rk is not None else None
        probs = []
        for k in range(B):
            other = object.__new__(DeviceProblem)
            other.__dict__.update(self.__dict__)
            other.X, other.D, other.Rk, other.M = Xs[k], Ds[k], (Rs[k] if Rs is not None else None), n
            probs.append(other)
        return probs

    def row_slice(self, lo, hi):
        """Rows [lo, hi) as a problem of its own sharing the device buffers (CpG-row shards, sharded.py)."""
        other = object.__new__(DeviceProblem)
        other.__dict__.update(self.__dict__)
        other.X, other.D = self.X[lo:hi], self.D[lo:hi]
        other.Rk = self.Rk[lo:hi] if self.Rk is not None else None
        other.M = hi - lo
        return other

    def with_weights(self, D_tensor, wtype):
        """Shallow copy sharing X / R_trunc with different weights (BCV folds, ic.py:75)."""
        other = object.__new__(DeviceProblem)
        other.__dict__.update(self.__dict__)
        other.D, other.wtype = D_tensor, wtype
        return other

    def with_reference(self, Rk):
        """Shallow copy sharing X / d_x with another R_trunc (M x K, or None): update_alpha gets a new R every outer iteration."""
        other = object.__new__(DeviceProblem)
        other.__dict__.update(self.__dict__)
        other._set_reference(Rk)
        return other


class FitBatch:
    """n_fits independent fits of one (M, N, K, n_u) shape, advanced together by single launches."""

    def __init__(self, problems, n_u, U0, A0, mode=_lib.DMF_MODE_PARTIAL, purity=None, rows=None, trace_cap=0,
                 max_ctas_per_fit=0, engine=None, mult=None, offs=None):
        probs = problems if isinstance(problems, (list, tuple)) else [problems]
        self.n_fits = len(U0)
        if len(probs) == 1:
            probs = list(probs) * self.n_fits
        if len(probs) != self.n_fits or len(A0) != self.n_fits:
            raise ValueError("one problem / U0 / A0 per fit expected")
        p0 = probs[0]
        self.p0, self.probs = p0, probs
        self.M, self.N, self.K, self.n_u = p0.M, p0.N, p0.K, int(n_u)
        self.Kt = self.K + self.n_u
        self.mode = mode
        dev, dt = p0.device, p0.dtype
        self.device = dev
        if rows is not None and mult is None:
            self.M = int(rows[0].shape[0])
        # ping-pong buffers: both slots start at the initial iterate (u_ = u.copy(), deconvolution.py:194-195)
        self.ldu = _even(self.n_u)
        self.u_slot = (self.M * self.ldu + 31) // 32 * 32          # slot stride keeps bulk copies 16-byte aligned
        # the fused engine writes the new (u, u_) pair next to the current one: 4 slots where it can apply
        self.u_slots = 4 if (FUSED_SLOTS and dt == torch.float64 and self.n_u <= 2 and rows is None and mult is None) else 2
        self.U = torch.zeros((self.n_fits, self.u_slots, self.u_slot), dtype=dt, device=dev)
        self.A = torch.empty((self.n_fits, 2, self.Kt, self.N), dtype=dt, device=dev)
        if isinstance(U0, torch.Tensor) and U0.ndim == 3:
            # stacked initial iterates (n_fits, M, n_u) / (n_fits, Kt, N): a handful of copies for the whole batch
            u = to_device(U0, dt, dev).reshape(self.n_fits, self.M, self.n_u)
            a = to_device(np.ascontiguousarray(A0) if not isinstance(A0, torch.Tensor) else A0, dt, dev).reshape(self.n_fits, self.Kt, self.N)
            for slot in (0, 1):
                self.U[:, slot, :self.M * self.ldu].view(self.n_fits, self.M, self.ldu)[:, :, :self.n_u] = u
                self.A[:, slot] = a
        else:
            for i in range(self.n_fits):
                u = to_device(U0[i], dt, dev).reshape(self.M, self.n_u)
                a = to_device(A0[i], dt, dev).reshape(self.Kt, self.N)
                self.u_view(i, 0).copy_(u); self.u_view(i, 1).copy_(u)
                self.A[i, 0].copy_(a); self.A[i, 1].copy_(a)
        self.purity = None
        if mode == _lib.DMF_MODE_PURITY:
            self.purity = to_device(np.asarray(purity, dtype=np.float64).reshape(-1), torch.float64, dev)
            if self.purity.numel() != self.N:
                raise ValueError("purity needs one value per sample")
        self.rows = None
        if rows is not None:
            if isinstance(rows, torch.Tensor) and rows.ndim == 2:           # stacked (n_fits, M) int32 device tensor
                self.rows = to_device(rows, torch.int32, dev)
            else:
                self.rows = [to_device(r if isinstance(r, torch.Tensor) else np.asarray(r, dtype=np.int32), torch.int32, dev) for r in rows]
        # bootstrap resamples in multiplicity form: per fit int32 device tensors mult (M) and offs (M + 1)
        self.mult, self.offs = mult, offs
        if (mult is None) != (offs is None) or (mult is not None and rows is None):
            raise ValueError("the multiplicity form needs mult, offs and rows (sorted source row of every position)")
        self.trace_cap = int(trace_cap)
        self.trace = torch.zeros((self.n_fits, max(self.trace_cap, 1)), dtype=torch.float64, device=dev) if trace_cap else None

        lib = _lib.lib()
        self.h = _handle(dev.index if dev.index is not None else torch.cuda.current_device())
        self.shape = _lib.Shape(M=self.M, N=self.N, K=self.K, n_u=self.n_u,
                                dtype=_lib.DMF_F64 if dt == torch.float64 else _lib.DMF_F32, wtype=p0.wtype, mode=mode,
                                n_fits=self.n_fits, max_ctas_per_fit=max_ctas_per_fit, ldx=p0.ldx, ldd=p0.ldd, ldr=_even(self.K),
                                ldu=self.ldu, u_slot=self.u_slot, u_slots=self.u_slots)
        nbytes = C.c_size_t()
        _lib.check(lib.dmf_batch_workspace_bytes(self.h, C.byref(self.shape), C.byref(nbytes)))
        self.ws = torch.empty(nbytes.value + 256, dtype=torch.uint8, device=dev)
        descs = (_lib.FitDesc * self.n_fits)()
        for i, p in enumerate(probs):
            if (p.N, p.K, p.wtype, p.dtype, p.ldd) != (p0.N, p0.K, p0.wtype, p0.dtype, p0.ldd):
                raise ValueError("all problems of a batch must share shape and storage types")
            d = descs[i]
            d.X, d.D = p.X.data_ptr(), p.D.data_ptr()
            d.Rk = p.Rk.data_ptr() if p.Rk is not None else None
            d.rows = self.rows[i].data_ptr() if self.rows is not None else None
            if self.mult is not None:      # rows of a stacked tensor are views: no .contiguous() copies, the pointers must stay valid
                d.mult, d.offs = self.mult[i].data_ptr(), self.offs[i].data_ptr()
            d.U, d.A = self.U[i].data_ptr(), self.A[i].data_ptr()
            d.purity = self.purity.data_ptr() if self.purity is not None else None
            d.cost_trace = self.trace[i].data_ptr() if self.trace is not None else None
            d.trace_cap = self.trace_cap
        ws_ptr = (self.ws.data_ptr() + 255) // 256 * 256
        self.b = C.c_void_p()
        _lib.check(lib.dmf_batch_create(self.h, C.byref(self.shape), descs, C.c_void_p(ws_ptr), nbytes.value, _stream_ptr(), C.byref(self.b)))
        engine = engine or get_engine()
        if engine != "auto":
            _lib.check(lib.dmf_batch_set_engine(self.b, {"gram": _lib.DMF_ENGINE_GRAM, "stream": _lib.DMF_ENGINE_STREAM,
                                                         "fused": _lib.DMF_ENGINE_FUSED}[engine]))

    @property
    def engine(self):
        e = C.c_int32()
        _lib.check(_lib.lib().dmf_batch_get_engine(self.b, C.byref(e)))
        return {_lib.DMF_ENGINE_GRAM: "gram", _lib.DMF_ENGINE_FUSED: "fused"}.get(e.value, "stream")

    def u_view(self, i, slot):
        return self.U[i, slot, :self.M * self.ldu].view(self.M, self.ldu)[:, :self.n_u]

    # -- single reference-shaped steps (one launch each)
    def pass_init(self):
        _lib.check(_lib.lib().dmf_pass_init(self.b, _stream_ptr()))

    def pass_u(self):
        _lib.check(_lib.lib().dmf_pass_u(self.b, _stream_ptr()))

    def pass_alpha(self):
        _lib.check(_lib.lib().dmf_pass_alpha(self.b, _stream_ptr()))

    def pass_fw(self, k):
        _lib.check(_lib.lib().dmf_pass_fw(self.b, int(k), _stream_ptr()))

    def pass_cost(self, tol):
        _lib.check(_lib.lib().dmf_pass_cost(self.b, float(tol), _stream_ptr()))

    def set_step_state(self, which, a, l, l_old):
        """Momentum state (one value per fit each) the next pass_u (which = 0: a1, l_w, l_w_old) or pass_alpha (which = 1: a2, l_h,
        l_h_old) steps start from."""
        if any(len(v) != self.n_fits for v in (a, l, l_old)):
            raise ValueError("one step-state value per fit expected")
        vals = [(C.c_double * self.n_fits)(*(float(x) for x in v)) for v in (a, l, l_old)]
        _lib.check(_lib.lib().dmf_batch_set_step_state(self.b, int(which), *vals, _stream_ptr()))

    # -- Gram-form engine steps
    def gram_init(self):
        _lib.check(_lib.lib().dmf_gram_init(self.b, _stream_ptr()))

    def gram_rowgram(self, initial=False, tol=0.0):
        _lib.check(_lib.lib().dmf_gram_rowgram(self.b, int(bool(initial)), float(tol), _stream_ptr()))

    def gram_u_inner(self, n_iter2):
        _lib.check(_lib.lib().dmf_gram_u_inner(self.b, int(n_iter2), _stream_ptr()))

    def gram_panels(self, known_block=False):
        _lib.check(_lib.lib().dmf_gram_panels(self.b, int(bool(known_block)), _stream_ptr()))

    def gram_alpha_inner(self, n_iter2):
        _lib.check(_lib.lib().dmf_gram_alpha_inner(self.b, int(n_iter2), _stream_ptr()))

    def gram_outer(self, n_iter2, tol):
        _lib.check(_lib.lib().dmf_gram_outer(self.b, int(n_iter2), float(tol), _stream_ptr()))

    # -- fused engine steps
    def fused_pass(self, n_iter2, tol):
        _lib.check(_lib.lib().dmf_fused_pass(self.b, int(n_iter2), float(tol), _stream_ptr()))

    def fused_outer(self, n_iter2, tol):
        _lib.check(_lib.lib().dmf_fused_outer(self.b, int(n_iter2), float(tol), _stream_ptr()))

    def fused_finish(self, tol):
        _lib.check(_lib.lib().dmf_fused_finish(self.b, float(tol), _stream_ptr()))

    def enqueue_outer(self, n_outer, n_iter2, tol):
        _lib.check(_lib.lib().dmf_enqueue_outer(self.b, int(n_outer), int(n_iter2), float(tol), _stream_ptr()))

    def fit(self, n_iter1, n_iter2, tol):
        """Run every fit to termination (|cf - cf_0| < tol) or n_iter1 outer iterations."""
        _lib.check(_lib.lib().dmf_fit_batched(self.b, int(n_iter1), int(n_iter2), float(tol), _stream_ptr()))
        return self.states()

    def states(self):
        out = (_lib.FitState * self.n_fits)()
        _lib.check(_lib.lib().dmf_batch_read_state(self.b, out, self.n_fits, _stream_ptr()))
        return list(out)

    def geometry(self):
        a, b, c = C.c_int32(), C.c_int32(), C.c_int32()
        _lib.check(_lib.lib().dmf_batch_geometry(self.b, C.byref(a), C.byref(b), C.byref(c)))
        return {"ctas_per_fit": a.value, "tile_rows": b.value, "smem_bytes": c.value}

    def launch_count(self):
        n = C.c_int64()
        _lib.check(_lib.lib().dmf_batch_launch_count(self.b, C.byref(n)))
        return n.value

    def current(self, i, states=None):
        """Device tensors (U, alpha) holding fit i's current iterate."""
        st = (states or self.states())[i]
        return self.u_view(i, st.u_slot), self.A[i, st.a_slot]

    def stacked_current(self, states=None):
        """(U (n_fits, M, n_u), alpha (n_fits, Kt, N)) device tensors holding every fit's current iterate."""
        states = states or self.states()
        ar = torch.arange(self.n_fits, device=self.device)
        us = torch.tensor([s.u_slot for s in states], device=self.device)
        as_ = torch.tensor([s.a_slot for s in states], device=self.device)
        U = self.U[ar, us][:, :self.M * self.ldu].view(self.n_fits, self.M, self.ldu)[:, :, :self.n_u]
        return U, self.A[ar, as_]

    def results(self, states=None):
        """[(u ndarray Mxn_u, alpha ndarray KtxN, n_outer, cost)] as float64 host arrays."""
        states = states or self.states()
        out = []
        for i, st in enumerate(states):
            u, a = self.current(i, states)
            out.append((u.to(torch.float64).contiguous().cpu().numpy(), a.to(torch.float64).cpu().numpy(), st.n_outer, st.cost))
        return out

    def close(self):
        if getattr(self, "b", None) is not None and self.b.value:
            _lib.lib().dmf_batch_destroy(self.b)
            self.b = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
