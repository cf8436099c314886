"""ctypes binding of include/migan_b200.h.  Fails loudly when the library is missing:
there is no Python/CPU fallback for the compute path."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int64, c_size_t, c_void_p

from . import build as _build

OK, ERR_INVALID, ERR_CUDA, ERR_STATE, ERR_WORKSPACE = 0, 1, 2, 3, 4
PATH_SIMT, PATH_TC, PATH_TC_FAST = 0, 1, 2
PATHS = {"simt": PATH_SIMT, "tc": PATH_TC, "tc_fast": PATH_TC_FAST}

# Every symbol include/migan_b200.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("migan_last_error", c_char_p, []),
    ("migan_version", c_char_p, []),
    ("migan_create", c_int, [c_int, c_int, POINTER(c_void_p)]),
    ("migan_destroy", c_int, [c_void_p]),
    ("migan_num_weights", c_int, [c_void_p]),
    ("migan_weight_info", c_int, [c_void_p, c_int, POINTER(c_char_p), POINTER(c_int), POINTER(c_int64)]),
    ("migan_set_weight", c_int, [c_void_p, c_char_p, c_void_p, c_int64]),
    ("migan_finalize_weights", c_int, [c_void_p]),
    ("migan_workspace_bytes", c_size_t, [c_void_p, c_int]),
    ("migan_forward", c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_int, c_void_p]),
    ("migan_graph_staging_bytes", c_size_t, [c_void_p, c_int]),
    ("migan_forward_graph", c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_int, c_void_p]),
    ("migan_host_staging_bytes", c_size_t, [c_void_p, c_int]),
    ("migan_forward_host", c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_int, c_void_p]),
    ("migan_forward_host_async", c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_int, c_void_p]),
    ("migan_host_wait", c_int, [c_void_p]),
    ("migan_u8_staging_bytes", c_size_t, [c_void_p, c_int]),
    ("migan_forward_u8", c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_int, c_void_p]),
    ("migan_forward_u8_async", c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_int, c_void_p]),
    ("b200_preprocess_u8", c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    ("b200_postprocess_u8", c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    ("b200_feather_composite", c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    ("b200_pipeline_scratch_bytes", c_size_t, [c_int, c_int, c_int]),
    ("b200_resize_nearest_u8", c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    ("b200_hole_flags", c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    ("migan_crop_box", c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    ("b200_pipeline_preprocess", c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    ("b200_pipeline_postprocess", c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    ("b200_pipeline_batch_scratch_bytes", c_size_t, [c_void_p, c_int, c_int]),
    ("b200_pipeline_batch_boxes", c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    ("b200_pipeline_batch_preprocess", c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    ("b200_pipeline_batch_postprocess", c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    ("b200_reparam_filter", c_int, [c_void_p, c_int, c_int, c_int64, c_void_p, c_void_p]),
    ("b200_stream_memops_available", c_int, []),
    ("b200_stream_wait_value32", c_int, [c_void_p, c_void_p, ctypes.c_uint32]),
    ("b200_stream_write_value32", c_int, [c_void_p, c_void_p, ctypes.c_uint32]),
    ("b200_memcpy_async", c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    ("b200_enable_peer_access", c_int, [c_int]),
    ("migan_last_launch_count", c_int, [c_void_p]),
    ("migan_set_profiling", c_int, [c_void_p, c_int]),
    ("migan_profile_num_steps", c_int, [c_void_p]),
    ("migan_profile_step", c_int, [c_void_p, c_int, POINTER(c_char_p), POINTER(c_float), POINTER(ctypes.c_double), POINTER(ctypes.c_double)]),
    ("migan_set_tap", c_int, [c_void_p, c_char_p, c_void_p]),
    ("migan_tap_info", c_int, [c_void_p, c_int, c_int, POINTER(c_char_p), POINTER(c_int)]),
    ("migan_debug_tc_timeout", c_int, [c_int]),
    ("b200_upfirdn2d", c_int, [c_void_p, c_void_p, c_void_p] + [c_int] * 14 + [c_int, c_float, c_void_p]),
    ("b200_conv1x1_nhwc", c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p]),
    ("b200_bias_act", c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_float, c_float, c_float, c_void_p]),
]

# Every symbol include/comodgan_b200.h declares
COMOD_SYMBOLS = [
    ("comodgan_last_error", c_char_p, []),
    ("comodgan_create", c_int, [c_int, c_int, POINTER(c_void_p)]),
    ("comodgan_destroy", c_int, [c_void_p]),
    ("comodgan_num_weights", c_int, [c_void_p]),
    ("comodgan_weight_info", c_int, [c_void_p, c_int, POINTER(c_char_p), POINTER(c_int), POINTER(c_int64)]),
    ("comodgan_set_weight", c_int, [c_void_p, c_char_p, c_void_p, c_int64]),
    ("comodgan_finalize_weights", c_int, [c_void_p]),
    ("comodgan_workspace_bytes", c_size_t, [c_void_p, c_int]),
    ("comodgan_num_noise_planes", c_int, [c_void_p]),
    ("comodgan_noise_plane_res", c_int, [c_void_p, c_int]),
    ("comodgan_forward", c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_float, c_int, c_int, c_void_p,
                                 c_void_p, c_size_t, c_void_p]),
    ("comodgan_last_launch_count", c_int, [c_void_p]),
    ("comodgan_set_tap", c_int, [c_void_p, c_char_p, c_void_p]),
    ("b200_conv2d_resample", c_int, [c_void_p, c_void_p, c_void_p, c_void_p] + [c_int] * 18 +
     [c_void_p, c_size_t, POINTER(c_size_t), POINTER(c_int), POINTER(c_int), c_void_p]),
]

PIPE_BATCH_MAX = 64   # MIGAN_PIPE_BATCH_MAX


class PipeReq(ctypes.Structure):
    """migan_pipe_req: one request of a batched crop-pipeline call (device pointers, sizes)."""
    _fields_ = [("image_chw", c_void_p), ("mask_hw", c_void_p), ("H", c_int), ("W", c_int), ("mask_h", c_int), ("mask_w", c_int)]


PREPOST_SYMBOLS =[s for s in SYMBOLS if s[0] in ("b200_preprocess_u8", "b200_postprocess_u8", "b200_feather_composite")]

_lib = None


def bind(lib, symbols):
    """Set restype / argtypes for `symbols` on an already dlopen-ed library (AttributeError if an export is missing)."""
    for name, restype, argtypes in symbols:
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    return lib



class MiganError(RuntimeError):
    """A C-ABI call returned a non-zero code."""

    def __init__(self, code: int, message: str):
        super().__init__("migan_b200 error %d: %s" % (code, message))
        self.code = code


def library_path() -> str:
    return os.environ.get("MIGAN_B200_LIB", _build.LIBPATH)


def load(build_if_missing: bool = False):
    """dlopen the shared library and bind every declared symbol."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        if build_if_missing:
            _build.build()
        else:
            raise ImportError(
                "migan_b200: %s not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU / pure-PyTorch fallback." % path)
    lib = ctypes.CDLL(path)
    bind(lib, SYMBOLS)
    bind(lib, COMOD_SYMBOLS)
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().migan_last_error()
        raise MiganError(rc, msg.decode() if msg else "unknown error")


def check_comod(rc: int, lib=None) -> None:
    if rc != 0:
        msg = (lib or load()).comodgan_last_error()
        raise MiganError(rc, msg.decode() if msg else "unknown error")
