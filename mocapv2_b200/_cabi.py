"""ctypes binding of libmocap_b200.so -- the C-ABI declared in include/mocap_b200.h.

This is the whole FFI surface: plain pointers and sizes, no torch types.  The library is built in-tree by
``mocapv2_b200.build`` (nvcc, sm_100a).  There is no CPU implementation behind these symbols: if the shared
library is missing or no CUDA device is present the package raises instead of degrading.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIB = os.path.join(HERE, "libmocap_b200.so")

ABI_VERSION = 6
MAX_CAND = 8
MAX_CAMS = 16
CAM_STRIDE = 40
N_STAGES = 5

OK = 0
FLAG_RUN_OVERFLOW, FLAG_BLOB_OVERFLOW, FLAG_CONTOUR_OVERFLOW, FLAG_TILE_OVERFLOW, FLAG_DEPTH_OVERFLOW, FLAG_TRACE_OVERFLOW = 1, 2, 4, 8, 16, 32
FLAG_GENERAL_PATH = 64          # informational
FLAG_LENS_INDEX = 128           # the frame's lens index lies outside the lens set: count 0
FLAG_ERRORS = 1 | 2 | 4 | 8 | 32 | 128
CFLAG_GROUP_CAP, CFLAG_CAND_CAP, CFLAG_TIE = 1, 2, 4

_p = C.c_void_p
_i = C.c_int
_i64 = C.c_int64
_sz = C.c_size_t
_d = C.c_double


class LensSet(C.Structure):
    """MocapLensSet: n_lenses undistortion tables lens_stride bytes apart, frame_lens_dev [n] int32 (or NULL: lens 0)."""
    _fields_ = [("tables_dev", C.c_void_p), ("n_lenses", C.c_int), ("lens_stride", C.c_size_t), ("frame_lens_dev", C.c_void_p)]


_ls = C.POINTER(LensSet)

# name -> (restype, argtypes); mirrors include/mocap_b200.h declaration by declaration
SIGNATURES = {
    "mocap_status_string": (C.c_char_p, [_i]),
    "mocap_abi_version": (_i, []),
    "mocap_kernel_launch_count": (C.c_uint64, []),
    "mocap_undistort_table_bytes": (_sz, [_i, _i]),
    "mocap_undistort_table_build": (_i, [_p, _p, _i, _i, _p, _sz, _p]),
    "mocap_detect_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i]),
    "mocap_detect_batch": (_i, [_p, _i, _i, _i, _i64, _ls, _i, _d, _d, _i, _i, _i,
                                _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _p]),
    "mocap_detect_batch_subpixel": (_i, [_p, _i, _i, _i, _i64, _ls, _i, _d, _d, _i, _i, _i,
                                         _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _p]),
    "mocap_stage_timer_create": (_p, []),
    "mocap_stage_timer_destroy": (None, [_p]),
    "mocap_stage_timer_read": (_i, [_p, _p]),
    "mocap_stage_name": (C.c_char_p, [_i]),
    "mocap_detect_pipe_create": (_p, [_i]),
    "mocap_detect_pipe_destroy": (None, [_p]),
    "mocap_detect_pipelined_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _i]),
    "mocap_detect_batch_pipelined": (_i, [_p, _p, _i, _i, _i, _i64, _ls, _i, _d, _d, _i, _i, _i,
                                          _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _i, _i]),
    "mocap_detect_batch_pipelined_subpixel": (_i, [_p, _p, _i, _i, _i, _i64, _ls, _i, _d, _d, _i, _i, _i,
                                                   _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _i, _i]),
    "mocap_detect_pipe_timeline": (_i, [_p, _p, _i]),
    "mocap_detect_pipe_info": (_i, [_p, _p]),
    "mocap_scan_cells_batch": (_i, [_p, _i, _i, _i, _i64, _p, _i, _i, _p, _p, _sz, _p]),
    "mocap_filter_batch": (_i, [_p, _i, _i, _i, _i64, _p, _i, _p, _p, _sz, _p]),
    "mocap_blobs_batch": (_i, [_p, _i, _i, _i, _d, _d, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "mocap_draw_contours_batch": (_i, [_p, _p, _p, _i, _i, _i, _i, _p, _i, _p]),
    "mocap_blur5_batch": (_i, [_p, _i, _i, _i, _p, _p]),
    "mocap_median5_threshold_batch": (_i, [_p, _i, _i, _i, _i, _p, _p]),
    "mocap_bayer_gr2gray_batch": (_i, [_p, _i, _i, _i, _p, _p]),
    "mocap_bayer_gr2gray_scan_batch": (_i, [_p, _i, _i, _i, _p, _i, _p, _p, _sz, _p]),
    "mocap_undistort_batch": (_i, [_p, _i, _i, _i, _p, _p, _p]),
    "mocap_triangulate_batch": (_i, [_p, _p, _p, _i, _i64, _i, _p, _p, _p]),
    "mocap_ba_residuals_batch": (_i, [_p, _p, _i, _i, _i64, _p, _p]),
    "mocap_reproject_batch": (_i, [_p, _p, _p, _p, _i, _i64, _i, _p, _p]),
    "mocap_correspond_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "mocap_correspond_batch": (_i, [_p, _p, _i, _i, _i, _p, _p, _d, _i, _i, _i,
                                    _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "mocap_correspond_batch_blocked": (_i, [_p, _p, _i, _i, _i, _i, _p, _p, _d, _i, _i, _i,
                                            _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "mocap_correspond_batch_subpixel": (_i, [_p, _p, _i, _i, _i, _i, _p, _p, _d, _i, _i, _i,
                                             _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
}


class MocapError(RuntimeError):
    pass


def load(path: str | None = None) -> C.CDLL:
    """dlopen the C-ABI library and attach the prototypes.  Raises if it is not there (no fallback)."""
    path = path or os.environ.get("MOCAP_B200_LIB", DEFAULT_LIB)
    if not os.path.exists(path):
        raise MocapError(f"{path} not found: build it with `python -m mocapv2_b200.build` (nvcc, sm_100a); "
                         "there is no CPU implementation of this path")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.mocap_abi_version() != ABI_VERSION:
        raise MocapError(f"ABI mismatch: library {lib.mocap_abi_version()} != binding {ABI_VERSION}")
    return lib


def check(lib, status: int, what: str):
    if status != OK:
        raise MocapError(f"{what}: {lib.mocap_status_string(status).decode()} ({status})")
