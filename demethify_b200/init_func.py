"""Mirror of the reference's demethify/init_func.py for the B200 path.

  wls_intercept        init_func.py:8-14   — weighted NNLS with intercept; one streaming moment pass + per-sample
                                            Lawson-Hanson on the GPU (dmf_wls_fit).  `wls_all_samples` is the batched
                                            form every internal caller uses (all sample columns in one launch set).
  nndsvd_initialize    init_func.py:40-82  — NNDSVD; the thin SVD runs in cuSOLVER through torch.linalg.svd (a library
                                            call made once per fit, SURVEY 2.1 row 3), the sign split / norms / scaling in
                                            a kernel of the library (dmf_nndsvd_split).
  constrained_nndsvd   init_func.py:17-37
ICA (init_func.py:99-176) forms an M x M covariance and is out of scope (SURVEY 2.1 row 4).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .engine import DeviceProblem, _handle, _stream_ptr, _even, _pad_cols, to_device


def wls_all_samples(X, d_x, R_full, extra=None, y_is_dx=False, precision=None):
    """wls_intercept for every column of X at once -> (K [+ K2], N) float64 ndarray.
    y = X, or d_x * X when y_is_dx (demethify.py:212).  `extra` is an optional second block of regressor columns
    (the unknown profiles u of deconvolution.py:51)."""
    prob = X if isinstance(X, DeviceProblem) else DeviceProblem(X, d_x, R_full, precision=precision)
    desc, out, _keep = wls_desc(prob, extra, y_is_dx)
    lib = _lib.lib()
    h = _handle(prob.device.index if prob.device.index is not None else torch.cuda.current_device())
    nbytes = C.c_size_t()
    _lib.check(lib.dmf_wls_workspace_bytes(h, C.byref(desc), C.byref(nbytes)))
    _ws, ws_ptr = aligned_workspace(nbytes.value, prob.device)
    _lib.check(lib.dmf_wls_fit(h, C.byref(desc), ws_ptr, nbytes.value, _stream_ptr()))
    return out.cpu().numpy()


def wls_desc(prob, extra=None, y_is_dx=False):
    """dmf_wls_desc_t of a resident problem with the optional second regressor block `extra` -> (desc, device output (K + K2) x N,
    the tensors the descriptor points to that must outlive the call)."""
    dev, dt = prob.device, prob.dtype
    K2, R2 = 0, None
    if extra is not None:
        e = to_device(extra, dt, dev)
        K2 = e.shape[1]
        R2 = _pad_cols(e, _even(K2))
    out = torch.zeros((prob.K + K2, prob.N), dtype=torch.float64, device=dev)
    desc = _lib.WlsDesc(M=prob.M, N=prob.N, K=prob.K, K2=K2, dtype=_lib.DMF_F64 if dt == torch.float64 else _lib.DMF_F32,
                        wtype=prob.wtype, y_is_dx=int(bool(y_is_dx)), ldx=prob.ldx, ldd=prob.ldd, ldr=_even(prob.K),
                        ldr2=_even(K2), X=prob.X.data_ptr(), D=prob.D.data_ptr(),
                        R1=prob.Rk.data_ptr() if prob.Rk is not None else None, R2=R2.data_ptr() if R2 is not None else None,
                        out=out.data_ptr())
    return desc, out, R2


def aligned_workspace(nbytes, device):
    """A device workspace of `nbytes` at a 256-byte aligned address -> (tensor that owns it, address)."""
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=device)
    return ws, C.c_void_p((ws.data_ptr() + 255) // 256 * 256)


def wls_intercept(x, d_x, R_full):
    """init_func.py:8-14.  x: (M,1) or (M,), d_x likewise, R_full: (M,K).  Returns (K,1) for 2-D x, (K,) for 1-D."""
    x = np.asarray(x)
    col = wls_all_samples(x.reshape(-1, 1), np.asarray(d_x).reshape(-1, 1), R_full)
    return col if x.ndim == 2 else col[:, 0]


def _nndsvd_device(Vt, rank):
    """NNDSVD factors of a non-negative device matrix: thin SVD in cuSOLVER (a library call made once per fit, SURVEY 2.1
    row 3), then sign split / norms / scaling in one kernel of the library (dmf_nndsvd_split) -> device (W, H)."""
    Ut, St, Vh = torch.linalg.svd(Vt, full_matrices=False)
    Ut, Vh = Ut.contiguous(), Vh.contiguous()
    M, N = Vt.shape
    W = torch.empty((M, rank), dtype=torch.float64, device=Vt.device)
    H = torch.empty((rank, N), dtype=torch.float64, device=Vt.device)
    _lib.check(_lib.lib().dmf_nndsvd_split(C.c_void_p(Ut.data_ptr()), Ut.shape[1], C.c_void_p(St.data_ptr()), C.c_void_p(Vh.data_ptr()),
                                           Vh.shape[1], M, N, int(rank), C.c_void_p(W.data_ptr()), C.c_void_p(H.data_ptr()), _stream_ptr()))
    return W, H


def nndsvd_initialize(V, rank, flag=0):
    """init_func.py:40-82: NNDSVD initialisation of a non-negative matrix; `flag` picks what replaces the zeros of the factors
    (0: nothing, 1: the mean of V, 2: mean(V) * uniform(0, 1) / 100 drawn from numpy's global stream, W first)."""
    Vt = to_device(np.asarray(V, dtype=np.float64), torch.float64)
    if bool((Vt < 0).any()):
        raise ValueError("The input matrix contains negative elements.")
    if rank > min(Vt.shape):
        raise IndexError(f"index {min(Vt.shape)} is out of bounds for axis 1 with size {min(Vt.shape)}")
    Wd, Hd = _nndsvd_device(Vt, rank)
    W, H = Wd.cpu().numpy(), Hd.cpu().numpy()
    if flag in (1, 2):
        avg = float(Vt.mean())
        for F in (W, H):
            zeros = F == 0
            F[zeros] = avg if flag == 1 else avg * np.random.uniform(0, 1, size=int(zeros.sum())) / 100
    return W, H


def constrained_nndsvd(Y, W1, counts, rank, flag=0):
    """init_func.py:17-37: reference-based fit of every sample, NNDSVD of the floored residual."""
    Y = np.asarray(Y, dtype=np.float64)
    W1 = np.asarray(W1, dtype=np.float64)
    H1 = wls_all_samples(Y, counts, W1)
    Y_residual = np.maximum(Y - W1 @ H1, 1e-8)
    W2, H2 = nndsvd_initialize(Y_residual, rank=rank, flag=flag)
    return np.hstack([W1, np.clip(W2, 0, 1)]), np.vstack([H1, H2])
