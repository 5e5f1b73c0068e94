"""ctypes binding of libgvcnn_sm100.so (include/gvcnn_b200.h).

This is the binding a maintainer of the reference would add next to
nets/model.py (see INTEGRATION.md).  There is no fallback of any kind: if the
library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libgvcnn_sm100.so")

F32, BF16, F16 = 0, 1, 2
LAYOUT_BVD, LAYOUT_VBD, LAYOUT_PTRS = 0, 1, 2
LAYOUT_CHANNELS_FIRST = 0x10  # ORed into the layout of channel-major [C, HW] maps (GVCNN_LAYOUT_CHANNELS_FIRST)
POOL_MAX, POOL_MEAN = 0, 1
SCORE_REDUCE_SHAPE, SCORE_REDUCE_BATCH = 0, 1
ABI_VERSION = 2
EXCHANGE_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p)


def pool_variant(pool, variant=0):
    """GVCNN_POOL_VARIANT: A/B-test selection of the pooling kernel, carried in bits 8..11 of `pool`."""
    return pool | (variant << 8)
STATUS_WORDS = 4
STATUS_BIN_RANGE, STATUS_NAN, STATUS_NEAR_EDGE, STATUS_BAD_SCHEME = 0, 1, 2, 3
FLAG_NEAR_EDGE, FLAG_BIN_RANGE, FLAG_NAN, FLAG_ORDER_EDGE = 1, 2, 4, 8
MAX_VIEWS, MAX_GROUPS = 128, 4096
E_UNSUPPORTED = -10
E_COMM_TIMEOUT = -11
COMM_MAX_WORLD, COMM_MAX_FLOATS, COMM_HANDLE_BYTES = 8, 16384, 64

_vp, _i, _i64, _f, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_size_t

# name -> (restype, argtypes): exactly the declarations of include/gvcnn_b200.h
SIGNATURES = {
    "gvcnn_version": (_i, []),
    "gvcnn_strerror": (ctypes.c_char_p, [_i]),
    "gvcnn_check_device": (_i, []),
    "gvcnn_view_score_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "gvcnn_batch_sum_x": (_i, [_vp, _vp, _i, _i, _vp]),
    "gvcnn_score_bin": (_i, [_vp, _f, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _i, _i, _vp, _i, _vp]),
    "gvcnn_batch_mean_bin": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i64, _vp, _vp, _vp]),
    "gvcnn_score_bin_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i64, _vp, _vp, _vp]),
    "gvcnn_score_bin_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "gvcnn_gap_score_bin_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "gvcnn_bins_from_scores": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _i, _i, _vp]),
    "gvcnn_bins_to_scheme": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "gvcnn_scheme_to_bins": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "gvcnn_group_weight": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "gvcnn_pool_fuse_fwd": (_i, [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp,
                                 _i, _i, _i64, _i, _i, _f, _i, _i, _vp]),
    "gvcnn_pool_fuse_bwd": (_i, [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp,
                                 _i, _i, _i64, _i, _i, _i, _i, _vp]),
    "gvcnn_view_pooling_bwd": (_i, [_vp, _vp, _i64, _vp, _vp, _vp, _i, _i, _i64, _i, _i, _i, _i, _vp]),
    "gvcnn_grouping_fusion_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                       _i, _i, _i, _i64, _i, _i, _f, _i, _i, _i, _i, _i, _vp]),
    "gvcnn_grouping_fusion_batch_fwd": (_i, [_vp] * 13 + [_i, _i, _i, _i64, _i, _i, _i, _f, _i, _i, _i, _i, _i, _i64,
                                                       _vp, _vp, _vp]),
    "gvcnn_pool_fuse_gap_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "gvcnn_pool_fuse_gap_fwd": (_i, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _sz, _i, _i, _i, _i, _i, _i, _f, _i, _i, _vp]),
    "gvcnn_pool_fuse_gap_bwd": (_i, [_vp, _vp, _i64, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "gvcnn_pool_fuse_gap_weighted_fwd": (_i, [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _sz, _i, _i, _i, _i, _i, _i,
                                              _f, _i, _i, _vp]),
    "gvcnn_pool_fuse_gap_weighted_bwd": (_i, [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i,
                                              _vp]),
    "gvcnn_group_weight_from_scores": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "gvcnn_pool_fuse_bwd_weights": (_i, [_vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _i, _i, _i64, _i, _i, _i, _i, _vp]),
    "gvcnn_score_weight_bwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "gvcnn_view_score_bwd_workspace_bytes": (_sz, [_i, _i]),
    "gvcnn_view_score_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _i, _i, _i, _i, _i, _vp]),
    "gvcnn_pool_fuse_gap_bwd_weights_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "gvcnn_pool_fuse_gap_bwd_weights": (_i, [_vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _sz, _i, _i, _i, _i, _i, _i,
                                             _i, _i, _vp]),
    "gvcnn_gap_score_bwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "gvcnn_comm_create": (_i, [ctypes.POINTER(_vp), _i, _i, _vp]),
    "gvcnn_comm_connect": (_i, [_vp, _vp]),
    "gvcnn_comm_allreduce_f32": (_i, [_vp, _vp, _i, _vp]),
    "gvcnn_comm_allreduce_scaled_f32": (_i, [_vp, _vp, _i, _f, _vp]),
    "gvcnn_comm_error": (_i, [_vp]),
    "gvcnn_comm_destroy": (_i, [_vp]),
    "gvcnn_host_pipeline_create": (_i, [ctypes.POINTER(_vp), _i]),
    "gvcnn_host_pipeline_destroy": (_i, [_vp]),
    "gvcnn_host_workspace_bytes": (_sz, [_i, _i, _i, _i, _i64, _i, _i, _i]),
    "gvcnn_grouping_fusion_host": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                        _i, _i, _i, _i64, _i, _i, _f, _i, _i, _i64, _vp, _vp, _i, _vp, _sz]),
}

_lib = None


class GvcnnError(RuntimeError):
    def __init__(self, code, where):
        self.code = code
        msg = lib().gvcnn_strerror(code).decode() if _lib is not None else str(code)
        super().__init__("%s failed: %s (code %d)" % (where, msg, code))


def lib():
    """Loads libgvcnn_sm100.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(
                "libgvcnn_sm100.so is missing (%s). Build it with `python gvcnn-tf_b200/build.py` "
                "or `__graft_entry__.build()`; this package has no CPU or PyTorch fallback." % SO_PATH)
        L = ctypes.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)           # AttributeError if a declared symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code, where):
    if code != 0:
        raise GvcnnError(code, where)
