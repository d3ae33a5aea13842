"""ctypes binding of libcss_b200.so (the C ABI declared in include/css_b200.h).

There is NO fallback: if the library is missing and cannot be built, or an entry point returns non-zero, a
RuntimeError is raised.  Nothing here imports `oracle`.
"""
import ctypes
import os
from ctypes import c_float, c_int, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcss_b200.so")

DTYPE_F32, DTYPE_BF16 = 0, 1
SIM_COS, SIM_SOFTMAX = 0, 1
FUSE_NONE, FUSE_MIX = 0, 1
LABEL_F32, LABEL_I64 = 0, 1
CUT_CUTOUT, CUT_CUTMIX, CUT_CLASSMIX = 0, 1, 2
UPDATE_LOCAL, UPDATE_GLOBAL = 0, 1
META_WORDS = 256
META_V, META_N_VALID, META_N_HARD, META_CLS_OF_SLOT, META_SLOT_OF_CLS = 0, 32, 64, 96, 128
META_ROWS_STALE = 164
CMAX = 32
D = 256

P = c_void_p
# name -> (restype, argtypes); must list every symbol include/css_b200.h declares (tests/test_abi.py checks it)
SIGNATURES = {
    "css_version": (c_int, []),
    "css_last_error": (ctypes.c_char_p, []),
    "css_sm_count": (c_int, []),
    "css_launch_count": (ctypes.c_ulonglong, []),
    "css_set_pdl": (c_int, [c_int]),
    "css_sim_map": (c_int, [P, c_int, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_float, P, P]),
    "css_upsample_label_fuse": (c_int, [P, P, c_float, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, P, P, P, P, P]),
    "css_select_tiles": (c_int, [c_int]),
    "css_select": (c_int, [P, P, P, c_float, c_int, c_int, c_int, c_int, P, P, P, P, P, P, P]),
    "css_rep_pass": (c_int, [P, c_int, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_float, P, P, P, P]),
    "css_set_rep_pass_path": (c_int, [c_int]),
    "css_set_scorer_path": (c_int, [c_int]),
    "css_rep_pass_nhwc": (c_int, [P, c_int, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_float, P, P, P]),
    "css_grad_scatter_nhwc": (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int, P, P]),
    "css_rows_refresh_nhwc": (c_int, [P, P, P, P, P, c_int, c_int, c_int, c_int, P]),
    "css_rows_refresh": (c_int, [P, c_int, P, P, P, c_int, c_int, c_int, c_int, P]),
    "css_class_blocks": (c_int, [c_int]),
    "css_class_stats": (c_int, [P, c_int, P, P, c_int, c_int, c_int, P, P, P, P]),
    "css_proto_ema": (c_int, [P, P, P, c_float, c_float, c_float, c_int, c_int, c_int, P, P, P]),
    "css_sample": (c_int, [P, P, c_uint64, c_uint64, c_int, c_int, c_int, P, P, P]),
    "css_score_ce": (c_int, [P, c_int, P, P, P, P, P, P, P, P, c_uint64, c_uint64, P, c_int, c_int, c_int, c_int, c_int, c_float,
                             P, P, P, P, P]),
    "css_grad_scatter": (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int, P, P]),
    "css_atl_blocks": (c_int, [c_int, c_int]),
    "css_atl_forward": (c_int, [P, P, P, c_float, c_int, c_int, c_int, c_int, P, P, P, P, P, P]),
    "css_atl_backward": (c_int, [P, P, P, P, P, c_int, c_int, c_int, c_int, P, P]),
    "css_ohem_workspace_bytes": (ctypes.c_size_t, [c_int, c_int, c_int]),
    "css_ohem_forward": (c_int, [P, P, P, ctypes.c_longlong, c_float, c_int, c_int, c_int, c_int, c_int, P, ctypes.c_size_t, P, P, P,
                                 P]),
    "css_ohem_backward": (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, P, ctypes.c_size_t, P, P]),
    "css_comm_bytes":(ctypes.c_size_t, [c_int]),
    "css_comm_alloc": (c_int, [c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "css_comm_free": (c_int, [P]),
    "css_comm_set_timeout_ms": (c_int, [ctypes.c_ulonglong]),
    "css_comm_timeouts": (c_int, [P]),
    "css_comm_stats": (c_int, [P, ctypes.POINTER(ctypes.c_ulonglong)]),
    "css_comm_export": (c_int, [P, ctypes.c_char_p]),
    "css_comm_open": (c_int, [ctypes.c_char_p, ctypes.POINTER(ctypes.c_void_p)]),
    "css_comm_close": (c_int, [P]),
    "css_stats_allreduce": (c_int, [P, P, P, c_int, c_int, c_int, c_int, P]),
    "css_aug_index": (c_int, [P, c_int, c_int, c_int, c_int, P, P, P]),
    "css_aug_maps": (c_int, [P, P, c_int, P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, P, P, P, P, P]),
    "css_aug_image_workspace_bytes": (ctypes.c_size_t, [c_int, c_int, c_int]),
    "css_aug_image": (c_int, [P, c_int, c_int, c_int, P, P, P, c_int, c_int, P, ctypes.c_size_t, P, P]),
    "css_cut_mix": (c_int, [P, P, P, P, P, P, P, P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, P, P, P, P, P, P]),
    "css_threshold_glue": (c_int, [P, P, P, c_float, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, P, P]),
}

_lib = None


def load():
    """Loads (building first if the .so is absent and nvcc is available) and returns the ctypes library."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        try:
            from . import build as _build
            _build.build()
        except Exception as e:  # no nvcc on this host
            raise RuntimeError(
                f"css_b200: {LIB_PATH} is missing and could not be built ({e}). "
                "Run `python -m css_b200.build` (needs nvcc). There is no CPU fallback.") from e
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().css_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"css_b200.{what} failed (rc={rc}): {msg}")


def ptr(t):
    """Device pointer of a (contiguous) CUDA tensor, None -> NULL."""
    return None if t is None else c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)
