"""ctypes binding of libstag_b200.so -- the C ABI declared in include/stag_b200.h.

There is no CPU fallback: if the library cannot be loaded every operator raises
``StagLibraryError``.  PyTorch is used by the callers only for device memory and
streams; nothing here takes a torch type.
"""
import ctypes
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_C", "libstag_b200.so")

STAG_OK, STAG_EINVAL, STAG_ECUDA, STAG_EWORKSPACE, STAG_EUNSUPPORTED = 0, -1, -2, -3, -4
NOISE_NONE, NOISE_EXTERNAL, NOISE_NORMAL, NOISE_UNIFORM, NOISE_BERNOULLI = 0, 1, 2, 3, 4
NOISE_NORMAL_HADAMARD = 5
PARAM_SCALAR, PARAM_CHANNEL, PARAM_EDGE, PARAM_EDGE_CHANNEL = 0, 1, 2, 3

c_i32p = ctypes.POINTER(ctypes.c_int32)
c_i64p = ctypes.POINTER(ctypes.c_int64)
c_f32p = ctypes.POINTER(ctypes.c_float)


class StagLibraryError(RuntimeError):
    pass


class StagError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("stag_b200 error %d: %s" % (code, msg))
        self.code = code


class StagGraph(ctypes.Structure):
    _fields_ = [
        ("num_rows", ctypes.c_int64), ("num_cols", ctypes.c_int64), ("num_edges", ctypes.c_int64),
        ("indptr", ctypes.c_void_p), ("indices", ctypes.c_void_p), ("eid", ctypes.c_void_p),
        ("num_hubs", ctypes.c_int32), ("num_hub_segs", ctypes.c_int32),
        ("hub_rows", ctypes.c_void_p), ("hub_seg_ptr", ctypes.c_void_p), ("row_order", ctypes.c_void_p),
        ("items", ctypes.c_void_p), ("num_items", ctypes.c_int64), ("erow", ctypes.c_void_p), ("eidf", ctypes.c_void_p),
    ]


class StagNoise(ctypes.Structure):
    _fields_ = [
        ("kind", ctypes.c_int32), ("K", ctypes.c_int32), ("param_shape", ctypes.c_int32),
        ("relu", ctypes.c_int32), ("in_norm", ctypes.c_int32), ("sample_base", ctypes.c_int32),
        ("p0", ctypes.c_void_p), ("p1", ctypes.c_void_p), ("external", ctypes.c_void_p),
        ("seed", ctypes.c_uint64), ("offset", ctypes.c_uint64),
        ("counter", ctypes.c_void_p),   # optional device uint32 added to the call counter (CUDA-graph replays)
    ]


PRIOR_MAX_COMPONENTS = 8
PRIOR_NORMAL_MIXTURE = 1


class StagPrior(ctypes.Structure):
    _fields_ = [
        ("kind", ctypes.c_int32), ("M", ctypes.c_int32),
        ("weight", ctypes.c_float * PRIOR_MAX_COMPONENTS), ("loc", ctypes.c_float * PRIOR_MAX_COMPONENTS),
        ("scale", ctypes.c_float * PRIOR_MAX_COMPONENTS),
    ]


# name -> (restype, argtypes); mirrors include/stag_b200.h one to one
_V, _I, _I32, _I64, _SZ = ctypes.c_void_p, ctypes.c_int, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t
_GP, _NP = ctypes.POINTER(StagGraph), ctypes.POINTER(StagNoise)
SIGNATURES = {
    "stag_last_error": (ctypes.c_char_p, []),
    "stag_abi_version": (_I, []),
    "stag_launch_count": (ctypes.c_longlong, []),
    "stag_hub_threshold": (_I, []),
    "stag_hub_segment": (_I, []),
    "stag_csx_workspace_bytes": (_SZ, [_I64, _I64]),
    "stag_csx_items_capacity": (_I64, [_I64, _I64]),
    "stag_csx_build": (_I, [_V, _V, _I64, _I64, _I, _V, _V, _V, _V, _V, _V, _V, _V, _V, c_i32p, _V, _SZ, _V]),
    "stag_spmm_workspace_bytes": (_SZ, [_GP, _I32, _I32]),
    "stag_spmm_fwd": (_I, [_GP, _V, _I64, _I64, _I32, _I32, _NP, _V, _V, _V, _I64, _I64, _V, _V, _SZ, _V]),
    "stag_spmm_bwd": (_I, [_GP, _V, _I64, _I64, _V, _I64, _I64, _I32, _I32, _NP, _V, _V, _V, _I64, _I64,
                           _V, _V, _V, _V, _SZ, _V]),
    "stag_spmm_max_fwd": (_I, [_GP, _V, _I64, _I64, _I32, _I32, _NP, _V, _V, _I64, _I64, _V, _SZ, _V]),
    "stag_spmm_max_bwd": (_I, [_GP, _V, _I64, _I64, _V, _V, _I64, _I64, _I32, _I32, _NP, _V, _I64, _I64,
                               _V, _V, _V, _V, _SZ, _V]),
    "stag_noise_emit": (_I, [_NP, _I64, _I32, _V, _V, _V]),
    "stag_noise_kl_workspace_bytes": (_SZ, [_I32]),
    "stag_noise_kl": (_I, [_NP, _I64, _I32, ctypes.POINTER(StagPrior), _V, _V, _V, _V, _SZ, _V]),
    "stag_segment_reduce": (_I, [_V, _I64, _V, _I32, _I32, _I, _V, _I64, _V]),
    "stag_edge_softmax": (_I, [_GP, _V, _I32, _V, _V]),
    "stag_edge_softmax_bwd": (_I, [_GP, _V, _V, _I32, _V, _V]),
    "stag_attention_softmax": (_I, [_GP, _V, _V, _V, ctypes.c_float, _I32, _V, _V]),
    "stag_attention_softmax_bwd": (_I, [_GP, _V, _V, _V, ctypes.c_float, _I32, _V, _V, _V, _V, _V, _V]),
    "stag_attention_workspace_bytes": (_SZ, [_GP, _I32, _I32]),
    "stag_attention_softmax_s": (_I, [_GP, _V, _I64, _V, _I64, _I32, _I32, _NP, ctypes.c_float, _V, _V, _SZ, _V]),
    "stag_attention_softmax_s_bwd": (_I, [_GP, _V, _I64, _V, _I64, _I32, _I32, _NP, ctypes.c_float, _V, _V, _V, _V,
                                          _V, _V, _V, _V, _SZ, _V]),
    "stag_nll_workspace_bytes": (_SZ, [_I64, _I32]),
    "stag_nll": (_I, [_V, _I64, _I64, _I64, _I32, _I32, _I, _V, _I64, _V, _V, _V, _V, _V, _SZ, _V]),
    "stag_mc_accumulate": (_I, [_V, _I64, _I64, _I64, _I32, _I32, _I, _V, _V, _V]),
    "stag_mc_finalize": (_I, [_V, _V, _I64, _I32, _I64, _I, _V, _I64, _V, _V, _V, _V, _V, _V]),
    "stag_calibration_table_len": (_I64, [_I32, _I32]),
    "stag_calibration": (_I, [_V, _I64, _I64, _I32, _I, _V, _I64, _V, _I32, _V, _V]),
    "stag_gemm_workspace_bytes": (_SZ, [_I64, _I32, _I32]),
    "stag_gemm_tcgen05": (_I, [_V, _I64, _V, _I64, _I64, _I32, _I32, _V, _V, _I, _V, _I64, _V, _SZ, _V]),
    "stag_aggregate_host": (_I, [_I, _V, _V, _I64, _I64, _V, _V, _I32, _I32, _NP, _I, _V, _V]),
}

_lock = threading.Lock()
_lib = None


def load(path=None):
    """Load the shared library (once) and type every entry point."""
    global _lib
    with _lock:
        if _lib is not None and path is None:
            return _lib
        p = path or os.environ.get("STAG_B200_LIB") or LIB_PATH
        if not os.path.exists(p):
            raise StagLibraryError(
                "stag_b200: CUDA library %s is missing. Build it with `python -m stag_b200.build` "
                "(needs nvcc, sm_100a). There is no CPU fallback." % p)
        try:
            lib = ctypes.CDLL(p)
        except OSError as e:  # pragma: no cover - depends on the box
            raise StagLibraryError("stag_b200: cannot load %s: %s" % (p, e))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError -> a header symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if lib.stag_abi_version() != 2:
            raise StagLibraryError("stag_b200: ABI version mismatch")
        _lib = lib
        return lib


def check(rc):
    if rc != STAG_OK:
        msg = load().stag_last_error()
        raise StagError(rc, msg.decode() if msg else "")


def loaded_path():
    return LIB_PATH if _lib is not None else None
