"""ctypes binding of libdemethify_sm100.so — the only way the Python layer reaches the GPU kernels.

Mirrors include/demethify_b200.h one to one.  Fails loudly if the library has not been built
(`python -c "import __graft_entry__ as g; g.build()"`): there is deliberately no fallback path.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DMF_LIB") or os.path.join(HERE, "libdemethify_sm100.so")      # DMF_LIB: an alternative build of the same sources (kernel experiments)

DMF_F64, DMF_F32 = 0, 1
DMF_W_FLOAT, DMF_W_U16 = 0, 1
DMF_MODE_PARTIAL, DMF_MODE_PURITY, DMF_MODE_UNSUPERVISED = 0, 1, 2
DMF_ENGINE_STREAM, DMF_ENGINE_GRAM, DMF_ENGINE_FUSED = 0, 1, 2
ABI_VERSION = 4


class Shape(C.Structure):
    _fields_ = [("M", C.c_int64), ("N", C.c_int32), ("K", C.c_int32), ("n_u", C.c_int32), ("dtype", C.c_int32),
                ("wtype", C.c_int32), ("mode", C.c_int32), ("n_fits", C.c_int32), ("max_ctas_per_fit", C.c_int32),
                ("ldx", C.c_int64), ("ldd", C.c_int64), ("ldr", C.c_int64), ("ldu", C.c_int64), ("u_slot", C.c_int64),
                ("u_slots", C.c_int32), ("reserved", C.c_int32)]


class FitDesc(C.Structure):
    _fields_ = [("X", C.c_void_p), ("D", C.c_void_p), ("Rk", C.c_void_p), ("rows", C.c_void_p), ("U", C.c_void_p),
                ("A", C.c_void_p), ("purity", C.c_void_p), ("cost_trace", C.c_void_p), ("trace_cap", C.c_int32),
                ("reserved", C.c_int32), ("mult", C.c_void_p), ("offs", C.c_void_p)]


class FitState(C.Structure):
    _fields_ = [("cost", C.c_double), ("cost_prev", C.c_double), ("l_w", C.c_double), ("l_h", C.c_double),
                ("a1", C.c_double), ("a2", C.c_double), ("dmax", C.c_double), ("n_outer", C.c_int32),
                ("done", C.c_int32), ("u_slot", C.c_int32), ("a_slot", C.c_int32)]


class WlsDesc(C.Structure):
    _fields_ = [("M", C.c_int64), ("N", C.c_int32), ("K", C.c_int32), ("K2", C.c_int32), ("dtype", C.c_int32),
                ("wtype", C.c_int32), ("y_is_dx", C.c_int32), ("reserved", C.c_int32), ("ldx", C.c_int64), ("ldd", C.c_int64),
                ("ldr", C.c_int64), ("ldr2", C.c_int64), ("X", C.c_void_p), ("D", C.c_void_p), ("R1", C.c_void_p),
                ("R2", C.c_void_p), ("out", C.c_void_p)]


class ResidDesc(C.Structure):
    _fields_ = [("M", C.c_int64), ("N", C.c_int32), ("K", C.c_int32), ("ldx", C.c_int64), ("ldr", C.c_int64), ("X", C.c_void_p),
                ("R", C.c_void_p), ("H1", C.c_void_p)]


EXPORTS = {
    "dmf_abi_version": (C.c_int, []),
    "dmf_last_error": (C.c_char_p, []),
    "dmf_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "dmf_destroy": (C.c_int, [C.c_void_p]),
    "dmf_sm_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "dmf_batch_workspace_bytes": (C.c_int, [C.c_void_p, C.POINTER(Shape), C.POINTER(C.c_size_t)]),
    "dmf_batch_create": (C.c_int, [C.c_void_p, C.POINTER(Shape), C.POINTER(FitDesc), C.c_void_p, C.c_size_t, C.c_void_p,
                                   C.POINTER(C.c_void_p)]),
    "dmf_batch_destroy": (C.c_int, [C.c_void_p]),
    "dmf_batch_geometry": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "dmf_pass_init": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dmf_pass_u": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dmf_pass_alpha": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dmf_pass_fw": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "dmf_pass_cost": (C.c_int, [C.c_void_p, C.c_double, C.c_void_p]),
    "dmf_batch_set_step_state": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                           C.c_void_p]),
    "dmf_batch_set_engine": (C.c_int, [C.c_void_p, C.c_int32]),
    "dmf_batch_get_engine": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "dmf_gram_rowgram": (C.c_int, [C.c_void_p, C.c_int32, C.c_double, C.c_void_p]),
    "dmf_gram_u_inner": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "dmf_gram_panels": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "dmf_gram_alpha_inner": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "dmf_batch_set_sharded": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "dmf_batch_stats_buffers": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dmf_gram_finalize_cost": (C.c_int, [C.c_void_p, C.c_int32, C.c_double, C.c_void_p]),
    "dmf_batch_peer_bytes": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_size_t)]),
    "dmf_batch_set_peers": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_void_p), C.c_size_t, C.c_void_p]),
    "dmf_gram_exchange": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "dmf_batch_reserve_momentum": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "dmf_gram_init": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dmf_gram_outer": (C.c_int, [C.c_void_p, C.c_int32, C.c_double, C.c_void_p]),
    "dmf_fused_pass": (C.c_int, [C.c_void_p, C.c_int32, C.c_double, C.c_void_p]),
    "dmf_fused_outer": (C.c_int, [C.c_void_p, C.c_int32, C.c_double, C.c_void_p]),
    "dmf_fused_finish": (C.c_int, [C.c_void_p, C.c_double, C.c_void_p]),
    "dmf_fused_alpha_commit": (C.c_int, [C.c_void_p, C.c_int32, C.c_double, C.c_void_p]),
    "dmf_enqueue_outer": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_double, C.c_void_p]),
    "dmf_fit_batched": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_double, C.c_void_p]),
    "dmf_batch_read_state": (C.c_int, [C.c_void_p, C.POINTER(FitState), C.c_int32, C.c_void_p]),
    "dmf_batch_launch_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "dmf_wls_workspace_bytes": (C.c_int, [C.c_void_p, C.POINTER(WlsDesc), C.POINTER(C.c_size_t)]),
    "dmf_wls_fit": (C.c_int, [C.c_void_p, C.POINTER(WlsDesc), C.c_void_p, C.c_size_t, C.c_void_p]),
    "dmf_wls_moments": (C.c_int, [C.c_void_p, C.POINTER(WlsDesc), C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dmf_wls_solve": (C.c_int, [C.c_void_p, C.POINTER(WlsDesc), C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dmf_resid_workspace_bytes": (C.c_int, [C.c_void_p, C.POINTER(ResidDesc), C.POINTER(C.c_size_t)]),
    "dmf_resid_gram": (C.c_int, [C.c_void_p, C.POINTER(ResidDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dmf_resid_project": (C.c_int, [C.c_void_p, C.POINTER(ResidDesc), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_size_t, C.c_void_p]),
    "dmf_nndsvd_apply": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                   C.c_void_p]),
    "dmf_pack_weights_u16": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dmf_nndsvd_split": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_void_p,
                                   C.c_void_p, C.c_void_p]),
    "dmf_rng_legacy_streams": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                         C.c_void_p]),
    "dmf_percentile_max_keep": (C.c_int, []),
    "dmf_percentile_bounds": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dmf_consensus": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dmf_gather_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
}

_lib = None


class DmfError(RuntimeError):
    pass


def lib():
    """The loaded library (dlopen only — no CUDA call is made here)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DmfError(f"{LIB_PATH} is missing: build it with __graft_entry__.build() "
                           "(demethify_b200 has no CPU fallback)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            fn = getattr(handle, name)        # AttributeError if the symbol is not exported
            fn.restype, fn.argtypes = res, args
        if handle.dmf_abi_version() != ABI_VERSION:
            raise DmfError("libdemethify_sm100.so ABI version mismatch")
        _lib = handle
    return _lib


def check(rc):
    if rc != 0:
        raise DmfError(f"libdemethify_sm100 error {rc}: {lib().dmf_last_error().decode()}")
