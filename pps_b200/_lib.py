"""ctypes binding of libpps_b200.so (the C ABI declared in include/pps_b200.h).

There is no CPU fallback: if the library cannot be loaded (or built), every entry point
raises.  Non-zero return codes become RuntimeError, mirroring how CAFFE_ENFORCE failures
surface in the reference (detectron/tests/test_zero_even_op.py:50-53).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

from . import build as _build

# ---- constants (keep in sync with include/pps_b200.h) ----
ABI_VERSION = 10
PPS_OK = 0
PPS_ERR_INVALID_ARG = -1
PPS_ERR_SHAPE = -2
PPS_ERR_ALIGN = -3
PPS_ERR_CUDA = -4
PPS_ERR_UNSUPPORTED = -5
PPS_ERR_WORKSPACE = -6
PPS_ERR_NO_VALID_QUERY = -7
PPS_ERR_TOPK_OVERFLOW = -8
PPS_ERR_PASS_RESIZE = -9
PASS_NO_EPILOGUE_TOPK = 1
PASS_SIZING = 2
PASS_NO_FUSED_COUNT = 4


def index_tkcap(n: int) -> int:
    """PPS_INDEX_TKCAP(n): pps_index_search test hook, candidate entries per query and chunk (pps_index_range_search: keys
    per query in the first pass's slices)."""
    return (n & 0xffff) << 8


def index_prefix(n: int) -> int:
    """PPS_INDEX_PREFIX(n): pps_index_search test hook, n * 256 rows in the materialised prefix."""
    return (n & 0x7f) << 24


def index_piece(n: int) -> int:
    """PPS_INDEX_PIECE(n): pps_index_remove test hook, at most n rows per move piece."""
    return (n & 0xffff) << 8

POOL_AVG_MAX = 0
POOL_MAX_AVE = 1
POOL_MAX_PARTS = 10

DTYPE_F32 = 0
DTYPE_F16 = 1
SPLIT_F16_SCALED = 0x100

PREC_BF16X1 = 1
PREC_BF16X3 = 3
PREC_BF16X6 = 6
PREC_F16X1 = 16
PREC_F16X3 = 19
PREC_FP32 = 32

DIST_SQUARED = 1
DIST_DOT = 2
DIST_KERNEL_1CTA = 0x100
DIST_CLUSTER4 = 0x400
DIST_SEPARATE_SMALL = 0x800
DIST_SQRT_RN = 0x1000

TOPK_MAX = 128
N_PHASES = 7
PHASE_NAMES = ["pairs_enqueue", "split", "dist_gemm", "pairs_wait_gather", "rank_count", "finalize", "d2h"]

PRECISIONS = {"bf16x1": PREC_BF16X1, "bf16x3": PREC_BF16X3, "bf16x6": PREC_BF16X6, "f16x3": PREC_F16X3,
              "fp16": PREC_F16X1, "fp32": PREC_FP32}
PLANES_FOR = {PREC_BF16X1: 1, PREC_BF16X3: 2, PREC_BF16X6: 3, PREC_F16X1: 1, PREC_F16X3: 2}


def split_planes_arg(prec: int) -> int:
    """`planes` argument of pps_split_rows for a precision code (PPS_PREC_F16X3 wants scaled fp16 planes)."""
    return (2 | SPLIT_F16_SCALED) if prec == PREC_F16X3 else PLANES_FOR[prec]

_vp, _ll, _i = C.c_void_p, C.c_longlong, C.c_int

# name -> (restype, argtypes); the order is the order of include/pps_b200.h
SIGNATURES = {
    "pps_abi_version": (_i, []),
    "pps_strerror": (C.c_char_p, [_i]),
    "pps_last_cuda_error": (C.c_char_p, []),
    "pps_pool_fwd": (_i, [_vp, _i, _i, _i, _i, _i, C.POINTER(_i), _i, C.POINTER(_i), _i, _vp, _ll, _ll, _vp]),
    "pps_pool_planes_fwd": (_i, [_vp, _i, _i, _i, _i, _i, C.POINTER(_i), _i, C.POINTER(_i), _i, _vp, _i, _vp]),
    "pps_pool_bwd": (_i, [_vp, _vp, _i, _i, _i, _i, _i, C.POINTER(_i), _i, C.POINTER(_i), _i, _ll, _ll, _vp, _vp]),
    "pps_kpad": (_i, [_i]),
    "pps_split_bytes": (_ll, [_ll, _i, _i]),
    "pps_split_rows": (_i, [_vp, _i, _ll, _i, _ll, _i, _vp, _vp, _vp]),
    "pps_split_rows_slab": (_i, [_vp, _i, _ll, _ll, _ll, _i, _ll, _i, _vp, _vp, _vp]),
    "pps_split_rows_gather": (_i, [_vp, _i, _vp, _ll, _ll, _i, _ll, _i, _vp, _vp, _vp]),
    "pps_dist_tc": (_i, [_vp, _vp, _ll, _i, _ll, _vp, _vp, _ll, _i, _ll, _i, _i, _i, _vp, _ll, _vp]),
    "pps_dist_fp32": (_i, [_vp, _ll, _vp, _ll, _vp, _ll, _vp, _ll, _i, _i, _vp, _ll, _vp]),
    "pps_row_sqnorm": (_i, [_vp, _i, _ll, _i, _ll, _vp, _vp]),
    "pps_pairs_count": (_ll, [_vp, _ll, _vp, _ll]),
    "pps_pairs_fill": (_i, [_vp, _vp, _ll, _vp, _vp, _ll, _vp, _vp, _vp, _vp]),
    "pps_pairs_workspace_bytes": (_ll, [_ll, _ll]),
    "pps_pairs_count_device": (_i, [_vp, _ll, _vp, _ll, _vp, _vp, _vp, _vp]),
    "pps_pairs_fill_device": (_i, [_vp, _vp, _ll, _vp, _vp, _ll, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _vp]),
    "pps_pairs_local_count": (_i, [_vp, _ll, _vp, _ll, _vp, C.POINTER(_vp), _vp]),
    "pps_pairs_offsets": (_i, [_vp, _i, _i, _ll, _ll, _vp, _vp, _vp, _vp]),
    "pps_pairs_fill_local": (_i, [_vp, _vp, _ll, _vp, _vp, _ll, _ll, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _vp]),
    "pps_pairs_unpack_pos": (_i, [_vp, _ll, _vp, _vp]),
    "pps_pairs_prefilter_workspace_bytes": (_ll, [_ll, _ll]),
    "pps_pairs_prefilter": (_i, [_vp, _ll, _vp, _vp, _ll, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pps_pairs_remap": (_i, [_vp, _ll, _vp, _ll, _vp]),
    "pps_pairs_compact_workspace_bytes": (_ll, [_ll]),
    "pps_pairs_compact_rows": (_i, [_vp, _ll, _vp, _vp, _vp, _ll, _ll, _ll, _vp, _vp, _vp, _vp, _vp]),
    "pps_rank_gather": (_i, [_vp, _ll, _ll, _ll, _ll, _vp, _vp, _ll, _vp, _vp]),
    "pps_rank_count": (_i, [_vp, _ll, _ll, _ll, _ll, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "pps_rank_finalize": (_i, [_ll, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pps_rank_tab_elems": (_ll, [_ll, _i]),
    "pps_rank_tab_prep": (_i, [_ll, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pps_dist_rank_tc": (_i, [_vp, _vp, _ll, _i, _ll, _vp, _vp, _ll, _i, _ll, _i, _i, _i, _ll, _i,
                              _vp, _vp, _vp, _vp, _vp, _vp]),
    "pps_dist_rank_topk_tc": (_i, [_vp, _vp, _ll, _i, _ll, _vp, _vp, _ll, _i, _ll, _i, _i, _i, _ll, _i,
                                   _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "pps_rank_tab_finish": (_i, [_ll, _i, _vp, _vp, _vp, _vp]),
    "pps_rank_count_eq": (_i, [_vp, _ll, _ll, _ll, _vp, _vp, _i, _vp, _vp]),
    "pps_rank_finalize_trapezoid": (_i, [_ll, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pps_topk_init": (_i, [_vp, _ll, _i, _vp]),
    "pps_topk_update": (_i, [_vp, _ll, _ll, _ll, _ll, _vp, _vp, _vp, _vp, _i, _vp]),
    "pps_rank_sweep": (_i, [_vp, _ll, _ll, _ll, _ll, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _i, _vp]),
    "pps_topk_bound": (_i, [_vp, _ll, _i, _vp, _vp, _vp]),
    "pps_dist_topk_tc": (_i, [_vp, _vp, _ll, _i, _ll, _vp, _vp, _ll, _i, _ll, _i, _i, _i, _vp, _ll,
                              _ll, _vp, _vp, _vp, _i, _vp]),
    "pps_topk_merge": (_i, [_vp, _ll, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    "pps_topk_unpack": (_i, [_vp, _ll, _i, _vp, _vp, _vp]),
    "pps_ctx_create": (_i, [_i, C.POINTER(_vp)]),
    "pps_ctx_destroy": (_i, [_vp]),
    "pps_evaluate_host_ctx": (_i, [_vp, _vp, _ll, _vp, _ll, _i, _vp, _vp, _vp, _vp, _i, _i, _i,
                                   _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pps_evaluate_device_ctx": (_i, [_vp, _vp, _ll, _vp, _ll, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp,
                                     _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pps_rank_begin": (_i, [_vp, _vp, _ll, _vp, _ll, _i, _vp, _vp, _vp, _vp, _ll, _i, _i, _i, _vp, _vp, C.POINTER(_vp)]),
    "pps_rank_thresholds": (_i, [_vp, _vp, _i, _vp, C.POINTER(_ll), C.POINTER(_vp), C.POINTER(_ll)]),
    "pps_rank_count_local": (_i, [_vp, _vp, C.POINTER(_vp), C.POINTER(_ll)]),
    "pps_rank_end": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pps_pass_begin": (_i, [_vp, _vp, _ll, _vp, _ll, _i, _i, _vp, _vp, _vp, _vp, _ll, _ll, _i, _i, _i, _i, _ll, _i, _vp,
                            C.POINTER(_vp), C.POINTER(_ll)]),
    "pps_pass_set_host_input": (_i, [_vp, _vp, _vp]),
    "pps_pass_stat": (_ll, [_vp, _i]),
    "pps_pass_count": (_i, [_vp, _vp, _vp, C.POINTER(_vp), C.POINTER(_ll)]),
    "pps_pass_end": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pps_ctx_set_timing": (_i, [_vp, _i]),
    "pps_ctx_phase_ms": (_i, [_vp, _vp]),
    "pps_evaluate_host": (_i, [_vp, _ll, _vp, _ll, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i,
                               _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pps_search_topk_tc": (_i, [_vp, _vp, _ll, _i, _ll, _vp, _vp, _ll, _i, _ll, _i, _i, _i, _ll, _vp, _vp, _vp, _i, _vp]),
    "pps_index_create": (_i, [_i, _i, _i, _i, C.POINTER(_vp)]),
    "pps_index_destroy": (_i, [_vp]),
    "pps_index_add": (_i, [_vp, _vp, _ll, _ll, _vp]),
    "pps_index_size": (_ll, [_vp]),
    "pps_index_search": (_i, [_vp, _vp, _ll, _ll, _i, _ll, _i, _vp, _vp]),
    "pps_search_topk_excl_tc": (_i, [_vp, _vp, _ll, _i, _ll, _vp, _vp, _ll, _i, _ll, _i, _i, _i, _ll, _vp, _vp, _vp, _i, _vp,
                                     _vp, _vp]),
    "pps_topk_update_excl": (_i, [_vp, _ll, _ll, _ll, _ll, _vp, _vp, _vp, _i, _vp, _vp]),
    "pps_index_add_tagged": (_i, [_vp, _vp, _ll, _ll, _vp, _vp]),
    "pps_index_search_excluding": (_i, [_vp, _vp, _ll, _ll, _vp, _i, _ll, _i, _vp, _vp]),
    "pps_index_remove": (_i, [_vp, _vp, _ll, _i, _vp, C.POINTER(_ll)]),
    "pps_search_range_tc": (_i, [_vp, _vp, _ll, _i, _ll, _vp, _vp, _ll, _i, _ll, _i, _i, _i, _ll, _vp, _vp, _vp, _vp, _vp,
                                 _vp, _vp, _vp]),
    "pps_index_range_search": (_i, [_vp, _vp, _ll, _ll, _vp, _vp, _ll, _i, _vp, _vp, C.POINTER(_ll)]),
    "pps_index_range_keys": (_i, [_vp, _vp, _vp]),
    "pps_sort_key_segments": (_i, [_vp, _vp, _ll, _vp, _vp]),
    "pps_index_add_grouped": (_i, [_vp, _vp, _ll, _ll, _vp, _vp, _vp]),
    "pps_index_search_groups": (_i, [_vp, _vp, _ll, _ll, _vp, _i, _ll, _i, _vp, _vp, _vp]),
    "pps_index_group_stats": (_i, [_vp, C.POINTER(_ll), C.POINTER(_ll), C.POINTER(_i)]),
    "pps_topk_group_update": (_i, [_vp, _ll, _ll, _ll, _ll, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "pps_topk_group_merge": (_i, [_vp, _vp, _ll, _i, _vp, _i, _vp, _vp, _vp, _ll, _vp, _vp]),
    "pps_topk_group_merge_lists": (_i, [_vp, _vp, _i, _ll, _i, _vp, _vp, _vp]),
    "pps_pairwise_distance_fwd": (_i, [_vp, _i, _i, _vp, _vp]),
    "pps_pairwise_distance_bwd": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "pps_batch_hard_fwd": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "pps_batch_hard_fused_fwd": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "pps_batch_hard_bwd": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "pps_embed_tc": (_i, [_vp, _i, _ll, _vp, _i, _i, _i, _i, _vp, _vp, _i, _vp, _ll, _vp]),
    "pps_l2_normalize_rows": (_i, [_vp, _ll, _i, _ll, _vp, _ll, _vp]),
    "pps_group_mean_rows": (_i, [_vp, _ll, _i, _vp, _vp, _ll, _vp, _ll, _vp]),
    "pps_rerank_vcap": (_i, []),
    "pps_rerank_normalize": (_i, [_vp, _ll, _ll, _vp, _vp, _ll, _vp]),
    "pps_rerank_krecip": (_i, [_vp, _i, _ll, _i, _vp, _ll, _vp, _vp, _vp, _vp]),
    "pps_rerank_expand": (_i, [_vp, _i, _ll, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "pps_rerank_invert": (_i, [_vp, _vp, _vp, _i, _ll, _ll, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pps_rerank_jaccard": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _ll, _ll, _vp, _ll, C.c_float, _vp, _ll, _vp]),
    "pps_kernel_launch_count": (C.c_ulonglong, []),
}

_lock = threading.Lock()
_lib = None


def lib_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True):
    """Return the loaded CDLL; build it first if it is missing and nvcc is available."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = _build.LIB_PATH
        if not os.path.exists(path):
            if not build_if_missing:
                raise RuntimeError("libpps_b200.so is not built (%s); run __graft_entry__.build()" % path)
            _build.build()
        lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)   # AttributeError here == ABI mismatch: fail loudly
            fn.restype = res
            fn.argtypes = args
        if lib.pps_abi_version() != ABI_VERSION:
            raise RuntimeError("libpps_b200.so ABI version mismatch")
        _lib = lib
    return _lib


def error_text(rc: int) -> str:
    lib = load()
    msg = lib.pps_strerror(rc).decode()
    if rc == PPS_ERR_CUDA:
        msg += ": " + lib.pps_last_cuda_error().decode()
    return msg


def check(rc: int, what: str = "") -> None:
    if rc != PPS_OK:
        raise RuntimeError("%s%s" % (what + ": " if what else "", error_text(rc)))


def launch_count() -> int:
    return int(load().pps_kernel_launch_count())


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("pps_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """device / host pointer of a torch tensor or numpy array (None -> NULL)"""
    if t is None:
        return C.c_void_p(0)
    if hasattr(t, "data_ptr"):
        return C.c_void_p(t.data_ptr())
    return C.c_void_p(t.ctypes.data)
