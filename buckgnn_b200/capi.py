"""ctypes binding of libbuckgnn_b200.so (include/buckgnn_b200.h).

Pointers cross as plain integers (`tensor.data_ptr()`), sizes as int64, the CUDA
stream as its integer handle.  A non-zero status raises `BuckGNNError` carrying
bg_last_error().  If the library has not been built, loading raises -- there is no
CPU or eager-PyTorch fallback for the hot path.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

from .build import LIB_PATH as _DEFAULT_LIB_PATH

# BG_LIB_PATH selects an instrumented build of the same ABI (tools/gemm_bench.py); default = the product library
LIB_PATH = os.environ.get("BG_LIB_PATH", _DEFAULT_LIB_PATH)

BG_BF16, BG_F32, BG_F16 = 0, 1, 2
BG_AGGR_MEAN, BG_AGGR_SUM, BG_AGGR_MAX = 0, 1, 2
BG_BIG_ROW_THRESHOLD = 64
BG_MAX_GEMM_SEGMENTS = 8
ABI_VERSION = 11

AGGR_CODES = {"mean": BG_AGGR_MEAN, "sum": BG_AGGR_SUM, "add": BG_AGGR_SUM, "max": BG_AGGR_MAX}

# every symbol include/buckgnn_b200.h declares (tests check the library exports all of them)
EXPORTED_SYMBOLS = (
    "bg_abi_version", "bg_last_error", "bg_device_check", "bg_watchdog_info_host", "bg_set_sm_partition",
    "bg_csr_max_big_rows", "bg_csr_workspace_bytes", "bg_csr_build",
    "bg_batch_info", "bg_graph_ptr_build", "bg_publish_words", "bg_encoder_front",
    "bg_aggregate_workspace_bytes", "bg_hubfold_workspace_bytes", "bg_sage_aggregate", "bg_gemm512",
    "bg_sage_fused512", "bg_sage_aggregate_hubs", "bg_gemm128", "bg_gemm128_gathered", "bg_pool_head128", "bg_pool_head_blocks128",
    "bg_wgrad512", "bg_pool_workspace_bytes", "bg_pool_head", "bg_pool_block_flags", "bg_pool_head_blocks", "bg_cast_f32", "bg_split_tf32",
    "bg_expand_rowptr", "bg_add",
    "bg_train_workspace_bytes", "bg_bn_batch_stats", "bg_bn_act_forward", "bg_sage_backward_rows",
    "bg_transpose_chunks", "bg_mask_narrow", "bg_reduce_partials", "bg_colsum_workspace_bytes", "bg_colsum", "bg_pool_backward",
    "bg_sgemm_workspace_bytes", "bg_sgemm", "bg_eigen_loss", "bg_dropout_mask", "bg_collate_ptr", "bg_collate", "bg_expand_wire",
    "bg_dropout_residual", "bg_grad_mask", "bg_segment_expand",
    "bg_sag_workspace_bytes", "bg_sag_select", "bg_sag_connect", "bg_gather_rows", "bg_index_invert", "bg_index_gather",
    "bg_sag_pool_backward", "bg_max_aggregate_backward", "bg_max_bwd_workspace_bytes",
    "bg_bn_batch_stats128", "bg_bn_act_forward128", "bg_sage_backward_rows128", "bg_pool_backward128",
    "bg_max_aggregate_backward128", "bg_wgrad128",
    "bg_dropout_residual128", "bg_grad_mask128", "bg_segment_expand128", "bg_wgrad128_ld", "bg_node_head128",
)


class BuckGNNError(RuntimeError):
    def __init__(self, status: int, where: str, message: str):
        super().__init__(f"{where} failed with status {status}: {message}")
        self.status = status


class GemmSegment(C.Structure):
    _fields_ = [("a", C.c_void_p), ("lda", C.c_int64), ("b", C.c_void_p), ("ldb", C.c_int64),
                ("k", C.c_int32), ("b_groups", C.c_int32)]


class Epilogue(C.Structure):
    _fields_ = [("bias_host", C.c_void_p), ("bn_scale_host", C.c_void_p), ("bn_shift_host", C.c_void_p),
                ("residual", C.c_void_p), ("ldr", C.c_int64), ("normalize", C.c_int32), ("relu", C.c_int32),
                ("gather", C.c_void_p * 2),
                ("gather_idx", C.c_void_p * 2), ("gather_ld", C.c_int64), ("inv_norm_out", C.c_void_p),
                ("pool_block_sums", C.c_void_p), ("pool_block_keep", C.c_void_p)]


class FusedAggregate(C.Structure):
    _fields_ = [("x", C.c_void_p), ("ldx", C.c_int64), ("rowptr", C.c_void_p), ("col", C.c_void_p),
                ("aggr", C.c_int32), ("n_big", C.c_int32), ("hub_agg", C.c_void_p), ("big_rows", C.c_void_p)]


_lib = None
_lock = threading.Lock()
_P, _I64, _I32, _SZP = C.c_void_p, C.c_int64, C.c_int32, C.POINTER(C.c_size_t)

_SIGNATURES = {
    "bg_abi_version": (C.c_int, []),
    "bg_last_error": (C.c_char_p, []),
    "bg_device_check": (C.c_int, []),
    "bg_watchdog_info_host": (C.c_int, [C.POINTER(C.c_uint32)]),
    "bg_set_sm_partition": (C.c_int, [C.c_int, C.c_int]),
    "bg_csr_max_big_rows": (_I64, [_I64]),
    "bg_csr_workspace_bytes": (C.c_int, [_I64, _I64, _SZP]),
    "bg_csr_build": (C.c_int, [_P, _I64, _I64, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, C.c_size_t, _P]),
    "bg_batch_info": (C.c_int, [_P, _I64, _P, _P]),
    "bg_publish_words": (C.c_int, [_P, _P, _I32, _P]),
    "bg_graph_ptr_build": (C.c_int, [_P, _I64, _I64, _P, _P]),
    "bg_encoder_front": (C.c_int, [_P, _I64, _I32, _P, _P, _P, _P, _P, _P, C.c_int, _P, _P]),
    "bg_expand_rowptr": (C.c_int, [_P, _I64, _I64, _P, _P, _P, C.c_int, C.c_int, _P]),
    "bg_add": (C.c_int, [_P, _P, _P, _P, C.c_int, _I64, _P]),
    "bg_aggregate_workspace_bytes": (C.c_int, [_I32, _SZP]),
    "bg_hubfold_workspace_bytes": (C.c_int, [_I64, C.c_int, _I32, _I32, _SZP]),
    "bg_sage_aggregate": (C.c_int, [_P, _P, C.c_int, _I64, _I32, _P, _P, _P, _I32, C.c_int, _P, _P, _I32, _P,
                                    C.c_size_t, _P]),
    "bg_gemm512": (C.c_int, [C.POINTER(GemmSegment), _I32, _I64, C.c_int, C.c_int, C.POINTER(Epilogue), _P,
                             C.c_int, _I64, C.c_int, _P]),
    "bg_sage_fused512": (C.c_int, [C.POINTER(GemmSegment), _I32, _I64, C.c_int, C.c_int, C.POINTER(Epilogue),
                                   C.POINTER(FusedAggregate), _P, C.c_int, _I64, _P]),
    "bg_sage_aggregate_hubs": (C.c_int, [_P, C.c_int, _P, _P, _P, _I32, C.c_int, _P, _P, C.c_size_t, _P]),
    "bg_gemm128": (C.c_int, [C.POINTER(GemmSegment), _I32, _I64, C.c_int, C.c_int, C.POINTER(Epilogue), _P,
                             C.c_int, _I64, C.c_int, _P]),
    "bg_gemm128_gathered": (C.c_int, [C.POINTER(GemmSegment), _I32, _I64, C.c_int, C.c_int, C.POINTER(Epilogue), _P,
                                      C.c_int, _I64, C.c_int, _P]),
    "bg_pool_head128": (C.c_int, [_P, C.c_int, _I64, _P, _I64, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _I32, _P, _P,
                                  _P, C.c_size_t, _P, _P]),
    "bg_pool_head_blocks128": (C.c_int, [_P, C.c_int, _I64, _P, _I64, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _I32, _P,
                                         _P, _P, _P, _P, C.c_size_t, _P, _P]),
    "bg_wgrad512": (C.c_int, [_P, _I64, _P, _I32, _I64, C.c_int, _I64, _I32, _I64, _P, _P]),
    "bg_pool_workspace_bytes": (C.c_int, [_I64, _SZP]),
    "bg_pool_head": (C.c_int, [_P, C.c_int, _I64, _P, _I64, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _I32, _P, _P,
                               _P, C.c_size_t, _P, _P]),
    "bg_pool_block_flags": (C.c_int, [_P, _I64, _I64, _P, _P]),
    "bg_pool_head_blocks": (C.c_int, [_P, C.c_int, _I64, _P, _I64, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _I32, _P, _P,
                                      _P, _P, _P, C.c_size_t, _P, _P]),
    "bg_cast_f32": (C.c_int, [_P, _P, C.c_int, _I64, _P]),
    "bg_split_tf32": (C.c_int, [_P, _P, _P, _I64, _P]),
    "bg_train_workspace_bytes": (C.c_int, [_I64, _SZP]),
    "bg_bn_batch_stats": (C.c_int, [_P, C.c_int, _I64, _P, _P, C.c_float, C.c_float, _P, _P, _P, _P, _P, _P, _P,
                                    _P, C.c_size_t, _P]),
    "bg_bn_act_forward": (C.c_int, [_P, _P, _P, C.c_int, _I64, _P, _P, C.c_float, C.c_uint64, _P]),
    "bg_sage_backward_rows": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, _I64, _P, _P, _P, _P, C.c_float, C.c_uint64,
                                        _P, _P, C.c_int, _P, _P, _P, _P, C.c_size_t, _P]),
    "bg_transpose_chunks": (C.c_int, [_P, C.c_int, _I64, _I32, _I64, _I32, _I64, _I32, _P, _P]),
    "bg_mask_narrow": (C.c_int, [_P, C.c_int, _I64, _P, C.c_int, _I64, _I64, _I32, _P, _P]),
    "bg_reduce_partials": (C.c_int, [_P, _I32, _I64, _P, C.c_int, _P]),
    "bg_colsum_workspace_bytes": (C.c_int, [_I64, _I32, _SZP]),
    "bg_colsum": (C.c_int, [_P, C.c_int, _I64, _I32, _I64, _P, C.c_int, _P, C.c_size_t, _P]),
    "bg_pool_backward": (C.c_int, [_P, _I64, _P, _I64, C.c_int, _I64, _P, C.c_int, _P]),
    "bg_sgemm_workspace_bytes": (C.c_int, [_I64, _I64, _I64, _SZP]),
    "bg_sgemm": (C.c_int, [_P, C.c_int, _I64, _I64, _P, C.c_int, _I64, _I64, _I64, _I64, _I64, _P, C.c_int, _P,
                           C.c_int, _I64, _P, C.c_int, _I64, C.c_int, _P, C.c_size_t, _P]),
    "bg_dropout_mask": (C.c_int, [C.c_uint64, C.c_float, _I64, _P, _P]),
    "bg_dropout_residual": (C.c_int, [_P, _P, _P, C.c_int, _I64, C.c_float, C.c_uint64, _P]),
    "bg_grad_mask": (C.c_int, [_P, _P, _P, _P, C.c_int, _I64, C.c_float, C.c_uint64, _P]),
    "bg_segment_expand": (C.c_int, [_P, _P, _I64, C.c_int, _P, C.c_int, _P]),
    "bg_collate_ptr": (C.c_int, [_P, _I64, _P, _P, _P, _P, _P]),
    "bg_expand_wire": (C.c_int, [_P, _I64, _P, _P, _P, _I64, _I64, _P, _P, _P]),
    "bg_collate": (C.c_int, [_P, _I32, _P, _I64, _P, _I32, _P, _P, _I64, _P, _P, _P, _P, _I64, _I64, _P, _P, _P, _P, _P, _P]),
    "bg_eigen_loss": (C.c_int, [_P, _P, _I64, C.c_float, C.c_float, C.c_float, _P, _P, _P, _P]),
    "bg_sag_workspace_bytes": (C.c_int, [_I64, _I64, _I64, _SZP]),
    "bg_sag_select": (C.c_int, [_P, C.c_int, _I64, _P, _P, _P, _I32, _P, _P, C.c_float, C.c_float, _P, _I64, C.c_float,
                                _P, _I64, _P, _P, _P, _P, _P, _P, _P, _P, C.c_size_t, _P]),
    "bg_sag_connect": (C.c_int, [_P, _I64, _I64, _P, _I64, _P, _P, _P, C.c_size_t, _P]),
    "bg_gather_rows": (C.c_int, [_P, C.c_int, _I64, _P, _P, _I64, _P, _I64, _P]),
    "bg_index_invert": (C.c_int, [_P, _I64, _P, _P]),
    "bg_index_gather": (C.c_int, [_P, _P, _I64, _P, _P]),
    "bg_max_bwd_workspace_bytes": (C.c_int, [_I32, _I32, _SZP]),
    "bg_max_aggregate_backward": (C.c_int, [_P, _P, _P, C.c_int, _I64, _P, _P, _P, _I32, _P, _P, _P, _I32, _P, _P, _P, C.c_size_t, _P]),
    "bg_sag_pool_backward": (C.c_int, [_P, _P, C.c_int, _I64, _I64, _P, _P, _P, C.c_float, _P, _P, _P, _I32, _P, _P, _P, _P, _P, _P]),
    "bg_bn_batch_stats128": (C.c_int, [_P, C.c_int, _I64, _P, _P, C.c_float, C.c_float, _P, _P, _P, _P, _P, _P, _P,
                                       _P, C.c_size_t, _P]),
    "bg_bn_act_forward128": (C.c_int, [_P, _P, _P, C.c_int, _I64, _P, _P, C.c_float, C.c_uint64, _P]),
    "bg_sage_backward_rows128": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, _I64, _P, _P, _P, _P, C.c_float, C.c_uint64,
                                           _P, _P, C.c_int, _P, _P, _P, _P, C.c_size_t, _P]),
    "bg_pool_backward128": (C.c_int, [_P, _I64, _P, _I64, C.c_int, _I64, _P, C.c_int, _P]),
    "bg_max_aggregate_backward128": (C.c_int, [_P, _P, _P, C.c_int, _I64, _P, _P, _P, _I32, _P, _P, _P, _I32, _P, _P, _P,
                                               C.c_size_t, _P]),
    "bg_wgrad128": (C.c_int, [_P, _P, _P, C.c_int, _I64, _I32, _I64, _P, _P, _P, C.c_int, _P]),
    "bg_dropout_residual128": (C.c_int, [_P, _P, _P, C.c_int, _I64, C.c_float, C.c_uint64, _P]),
    "bg_grad_mask128": (C.c_int, [_P, _P, _P, _P, C.c_int, _I64, C.c_float, C.c_uint64, _P]),
    "bg_segment_expand128": (C.c_int, [_P, _P, _I64, C.c_int, _P, C.c_int, _P]),
    "bg_wgrad128_ld": (C.c_int, [_P, _P, _P, C.c_int, _I64, _I32, _I64, _P, _P, _I64, _P, _I64, C.c_int, _P]),
    "bg_node_head128": (C.c_int, [_P, C.c_int, _I64, _P, _P, _P, _P, _I32, _P, _P]),
}


def library_path() -> str:
    return LIB_PATH


def load():
    """dlopen the in-tree library (once).  Raises if it is missing or has the wrong ABI."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise BuckGNNError(-100, "load", f"{LIB_PATH} not built: run `python -m buckgnn_b200.build` "
                               "(the BuckGNN hot path has no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        if lib.bg_abi_version() != ABI_VERSION:
            raise BuckGNNError(-101, "load", f"ABI version mismatch: library {lib.bg_abi_version()}, binding {ABI_VERSION}")
        _lib = lib
        return lib


def last_error() -> str:
    return load().bg_last_error().decode("utf-8", "replace")


def _check(status: int, where: str) -> None:
    if status != 0:
        raise BuckGNNError(status, where, last_error())


def device_check() -> None:
    _check(load().bg_device_check(), "bg_device_check")


def watchdog_info():
    buf = (C.c_uint32 * 4)()
    _check(load().bg_watchdog_info_host(buf), "bg_watchdog_info_host")
    return list(buf)


def csr_max_big_rows(n_edges: int) -> int:
    return int(load().bg_csr_max_big_rows(n_edges))


def _query(fn_name: str, *args) -> int:
    out = C.c_size_t(0)
    _check(getattr(load(), fn_name)(*args, C.byref(out)), fn_name)
    return int(out.value)


def csr_workspace_bytes(n_nodes: int, n_edges: int) -> int:
    return _query("bg_csr_workspace_bytes", n_nodes, n_edges)


def aggregate_workspace_bytes(n_big: int) -> int:
    return _query("bg_aggregate_workspace_bytes", n_big)


def pool_workspace_bytes(n_graphs: int) -> int:
    return _query("bg_pool_workspace_bytes", n_graphs)


def csr_build(edge_index, n_edges, n_nodes, key_row, rowptr, col, perm, big_rows, info, ws, ws_bytes, stream,
              hub_lo=None, hub_of_row=None):
    """`info` holds 8 int32 words (see include/buckgnn_b200.h)."""
    _check(load().bg_csr_build(edge_index, n_edges, n_nodes, key_row, rowptr, col, perm, big_rows, info,
                               hub_lo, hub_of_row, ws, ws_bytes, stream), "bg_csr_build")


def batch_info(batch, n_nodes, info, stream):
    _check(load().bg_batch_info(batch, n_nodes, info, stream), "bg_batch_info")


def publish_words(src, dst_host_mapped, n, stream):
    _check(load().bg_publish_words(src, dst_host_mapped, n, stream), "bg_publish_words")


def graph_ptr_build(batch, n_nodes, n_graphs, graph_ptr, stream):
    _check(load().bg_graph_ptr_build(batch, n_nodes, n_graphs, graph_ptr, stream), "bg_graph_ptr_build")


def encoder_front(x, n_nodes, n_features, w1, b1, w2, b2, out, out_dtype, stream, row_gather=None, nonfinite=None):
    _check(load().bg_encoder_front(x, n_nodes, n_features, w1, b1, w2, b2, row_gather, out, out_dtype, nonfinite, stream),
           "bg_encoder_front")


def expand_rowptr(rowptr, n_rows, n_entries, row_of, iota, nonempty, nonempty_dtype, stream, as_count=False):
    _check(load().bg_expand_rowptr(rowptr, n_rows, n_entries, row_of, iota, nonempty, nonempty_dtype,
                                   int(bool(as_count)), stream), "bg_expand_rowptr")


def add(a, b, c, out, dtype, n, stream):
    _check(load().bg_add(a, b, c, out, dtype, n, stream), "bg_add")


def hubfold_workspace_bytes(n_nodes: int, dtype: int, n_big: int, hub_max_degree: int) -> int:
    return _query("bg_hubfold_workspace_bytes", n_nodes, dtype, n_big, hub_max_degree)


def sage_aggregate(x, out, dtype, n_nodes, rowptr, col, big_rows, n_big, aggr, ws, ws_bytes, stream, width=512,
                   hub_lo=None, hub_of_row=None, hub_max_degree=0):
    _check(load().bg_sage_aggregate(x, out, dtype, n_nodes, width, rowptr, col, big_rows, n_big, aggr,
                                    hub_lo, hub_of_row, hub_max_degree, ws, ws_bytes, stream), "bg_sage_aggregate")


def _gemm(entry, segments, m, a_dtype, b_dtype, out, out_dtype, ldo, stream, *, bias=None, bn_scale=None,
          bn_shift=None, residual=None, ldr=0, normalize=False, relu=False, cta_group=2,
          gather=(), gather_ld, inv_norm_out=None, b_groups=0, pool_block_sums=None, pool_block_keep=None):
    n = len(segments)
    arr = (GemmSegment * n)(*[GemmSegment(a, lda, b, ldb, k, b_groups) for (a, lda, b, ldb, k) in segments])
    gm = (C.c_void_p * 2)(*([g[0] for g in gather] + [None] * (2 - len(gather))))
    gi = (C.c_void_p * 2)(*([g[1] for g in gather] + [None] * (2 - len(gather))))
    epi = Epilogue(bias, bn_scale, bn_shift, residual, ldr, int(bool(normalize)), int(bool(relu)),
                   gm, gi, gather_ld, inv_norm_out, pool_block_sums, pool_block_keep)
    _check(getattr(load(), entry)(arr, n, m, a_dtype, b_dtype, C.byref(epi), out, out_dtype, ldo, cta_group, stream),
           entry)


def gemm512(segments, m, a_dtype, b_dtype, out, out_dtype, ldo, stream, *, gather_ld=512, **epi):
    """segments: list of (a_ptr, lda, b_ptr, ldb, k); bias / bn_scale / bn_shift are HOST pointers;
    gather: up to two (matrix_ptr, index_ptr) pairs of gathered pre-activation addends;
    pool_block_sums / pool_block_keep: the pool-fused epilogue of the last layer (see the header)."""
    _gemm("bg_gemm512", segments, m, a_dtype, b_dtype, out, out_dtype, ldo, stream, gather_ld=gather_ld, **epi)


def gemm128(segments, m, a_dtype, b_dtype, out, out_dtype, ldo, stream, *, gather_ld=128, **epi):
    """bg_gemm128: gemm512 with 128-wide output rows (B [128, k], epilogue vectors [128]).  `gather` and `b_groups`
    are accepted only so that the library can reject them (BG_ERR_UNSUPPORTED)."""
    _gemm("bg_gemm128", segments, m, a_dtype, b_dtype, out, out_dtype, ldo, stream, gather_ld=gather_ld, **epi)


def gemm128_gathered(segments, m, a_dtype, b_dtype, out, out_dtype, ldo, stream, *, gather_ld=128, **epi):
    """bg_gemm128_gathered: gemm128 plus up to two (matrix_ptr, index_ptr) pairs of gathered pre-activation addends,
    [*, 128] rows of the output dtype with leading dimension gather_ld.  The library rejects them together with
    normalize, residual or pool fusion."""
    _gemm("bg_gemm128_gathered", segments, m, a_dtype, b_dtype, out, out_dtype, ldo, stream, gather_ld=gather_ld,
          **epi)


def sage_fused512(segments, m, a_dtype, b_dtype, out, out_dtype, ldo, stream, *, x, ldx, rowptr, col, aggr, hub_agg=None,
                  big_rows=None, n_big=0, bias=None, bn_scale=None, bn_shift=None, residual=None, ldr=0, relu=False,
                  pool_block_sums=None, pool_block_keep=None):
    """The fused SAGE layer: bg_gemm512 whose first segment's A operand (the neighbourhood aggregate of `x`) is gathered
    inside the kernel.  segments[0] = (None, 0, lin_l_ptr, ldb, 512), segments[1:] as in gemm512."""
    n = len(segments)
    arr = (GemmSegment * n)(*[GemmSegment(a, lda, b, ldb, k, 0) for (a, lda, b, ldb, k) in segments])
    none2 = (C.c_void_p * 2)(None, None)
    epi = Epilogue(bias, bn_scale, bn_shift, residual, ldr, 1, int(bool(relu)), none2, (C.c_void_p * 2)(None, None), 512,
                   None, pool_block_sums, pool_block_keep)
    fa = FusedAggregate(x, ldx, rowptr, col, aggr, n_big, hub_agg, big_rows)
    _check(load().bg_sage_fused512(arr, n, m, a_dtype, b_dtype, C.byref(epi), C.byref(fa), out, out_dtype, ldo, stream),
           "bg_sage_fused512")


def sage_aggregate_hubs(x, dtype, rowptr, col, big_rows, n_big, aggr, hub_out, ws, ws_bytes, stream):
    _check(load().bg_sage_aggregate_hubs(x, dtype, rowptr, col, big_rows, n_big, aggr, hub_out, ws, ws_bytes, stream),
           "bg_sage_aggregate_hubs")


POOL_MODES = {"mean": 0, "mlp": 0, "mean_no_super": 1, "mlp_no_super": 1, "supernode_only": 2,
              "supernode_with_pooling": 3}


def pool_head(x, dtype, n_nodes, graph_ptr, n_graphs, pool_mode, pre_w, pre_b, w1, b1, w2, b2, w3, b3, out_dim,
              pred, pooled_out, ws, ws_bytes, stream, nonfinite=None):
    _check(load().bg_pool_head(x, dtype, n_nodes, graph_ptr, n_graphs, pool_mode, pre_w, pre_b, w1, b1, w2, b2,
                               w3, b3, out_dim, pred, pooled_out, ws, ws_bytes, nonfinite, stream), "bg_pool_head")


def pool_head128(x, dtype, n_nodes, graph_ptr, n_graphs, pool_mode, pre_w, pre_b, w1, b1, w2, b2, w3, b3, out_dim,
                 pred, pooled_out, ws, ws_bytes, stream, nonfinite=None):
    _check(load().bg_pool_head128(x, dtype, n_nodes, graph_ptr, n_graphs, pool_mode, pre_w, pre_b, w1, b1, w2, b2,
                                  w3, b3, out_dim, pred, pooled_out, ws, ws_bytes, nonfinite, stream), "bg_pool_head128")


def node_head128(x, dtype, n_rows, w1, b1, w2, b2, out_dim, out, stream):
    """bg_node_head128: out [n_rows, out_dim] f32 = W2 relu(W1 x + b1) + b2 for x [n_rows, 128] of `dtype`, w1 [64, 128]
    in the operand format of dtype, b1 / w2 / b2 f32."""
    _check(load().bg_node_head128(x, dtype, n_rows, w1, b1, w2, b2, out_dim, out, stream), "bg_node_head128")


def pool_block_flags(graph_ptr, n_graphs, n_nodes, keep, stream):
    _check(load().bg_pool_block_flags(graph_ptr, n_graphs, n_nodes, keep, stream), "bg_pool_block_flags")


def pool_head_blocks(x, dtype, n_nodes, graph_ptr, n_graphs, pool_mode, pre_w, pre_b, w1, b1, w2, b2, w3, b3, out_dim,
                     pred, pooled_out, block_sums, keep, ws, ws_bytes, stream, nonfinite=None):
    _check(load().bg_pool_head_blocks(x, dtype, n_nodes, graph_ptr, n_graphs, pool_mode, pre_w, pre_b, w1, b1, w2, b2,
                                      w3, b3, out_dim, pred, pooled_out, block_sums, keep, ws, ws_bytes, nonfinite,
                                      stream), "bg_pool_head_blocks")


def pool_head_blocks128(x, dtype, n_nodes, graph_ptr, n_graphs, pool_mode, pre_w, pre_b, w1, b1, w2, b2, w3, b3, out_dim,
                        pred, pooled_out, block_sums, keep, ws, ws_bytes, stream, nonfinite=None):
    _check(load().bg_pool_head_blocks128(x, dtype, n_nodes, graph_ptr, n_graphs, pool_mode, pre_w, pre_b, w1, b1, w2,
                                         b2, w3, b3, out_dim, pred, pooled_out, block_sums, keep, ws, ws_bytes,
                                         nonfinite, stream), "bg_pool_head_blocks128")


def cast_f32(src, dst, dst_dtype, n, stream):
    _check(load().bg_cast_f32(src, dst, dst_dtype, n, stream), "bg_cast_f32")


def split_tf32(src, hi, lo, n, stream):
    _check(load().bg_split_tf32(src, hi, lo, n, stream), "bg_split_tf32")


# ----------------------------------------------------------------------------- training step
def train_workspace_bytes(n_rows: int) -> int:
    return _query("bg_train_workspace_bytes", n_rows)


def _w(name: str, width: int) -> str:
    """Entry point of a training-step kernel for the row width: `name` (512) or `name`128."""
    if width not in (512, 128):
        raise ValueError(f"{name}: width must be 512 or 128, got {width}")
    return name if width == 512 else name + "128"


def bn_batch_stats(u, dtype, n_rows, gamma, beta, eps, momentum, running_mean, running_var, num_batches_tracked,
                   a_out, shift_out, mean_out, invstd_out, ws, ws_bytes, stream, width=512):
    fn = _w("bg_bn_batch_stats", width)
    _check(getattr(load(), fn)(u, dtype, n_rows, gamma, beta, eps, momentum, running_mean, running_var,
                               num_batches_tracked, a_out, shift_out, mean_out, invstd_out, ws, ws_bytes, stream), fn)


def bn_act_forward(u, x_prev, y, dtype, n_rows, a, shift, dropout_p, seed, stream, width=512):
    fn = _w("bg_bn_act_forward", width)
    _check(getattr(load(), fn)(u, x_prev, y, dtype, n_rows, a, shift, dropout_p, seed, stream), fn)


def sage_backward_rows(u, dy, dy2, inv_norm, rowptr, dtype, n_rows, a, shift, mean, invstd, dropout_p, seed,
                       dgamma, dbeta, accumulate, dz, dz_scaled, g_out, ws, ws_bytes, stream, width=512):
    fn = _w("bg_sage_backward_rows", width)
    _check(getattr(load(), fn)(u, dy, dy2, inv_norm, rowptr, dtype, n_rows, a, shift, mean, invstd, dropout_p, seed,
                               dgamma, dbeta, int(bool(accumulate)), dz, dz_scaled, g_out, ws, ws_bytes, stream), fn)


def transpose_chunks(src, dtype, n_rows, n_cols, ld, n_chunks, chunk_k, out, stream, out_rows_per_chunk=0):
    _check(load().bg_transpose_chunks(src, dtype, n_rows, n_cols, ld, n_chunks, chunk_k, out_rows_per_chunk, out, stream),
           "bg_transpose_chunks")


def mask_narrow(src, src_dtype, ld_in, mask, mask_dtype, ld_mask, m, n_cols, out, stream):
    _check(load().bg_mask_narrow(src, src_dtype, ld_in, mask, mask_dtype, ld_mask, m, n_cols, out, stream), "bg_mask_narrow")


def reduce_partials(partial, n_chunks, n, out, accumulate, stream):
    _check(load().bg_reduce_partials(partial, n_chunks, n, out, int(bool(accumulate)), stream), "bg_reduce_partials")


def colsum_workspace_bytes(rows: int, cols: int) -> int:
    return _query("bg_colsum_workspace_bytes", rows, cols)


def colsum(src, dtype, rows, cols, ld, out, accumulate, ws, ws_bytes, stream):
    _check(load().bg_colsum(src, dtype, rows, cols, ld, out, int(bool(accumulate)), ws, ws_bytes, stream), "bg_colsum")


def pool_backward(dpooled, ldp, graph_ptr, n_graphs, pool_mode, n_nodes, dx, dtype, stream, width=512):
    fn = _w("bg_pool_backward", width)
    _check(getattr(load(), fn)(dpooled, ldp, graph_ptr, n_graphs, pool_mode, n_nodes, dx, dtype, stream), fn)


def sgemm_workspace_bytes(m: int, n: int, k: int) -> int:
    return _query("bg_sgemm_workspace_bytes", m, n, k)


def sgemm(a, a_dtype, sam, sak, b, b_dtype, sbk, sbn, m, n, k, bias, relu, mask, mask_dtype, mask_ld, out,
          out_dtype, ldo, accumulate, ws, ws_bytes, stream):
    _check(load().bg_sgemm(a, a_dtype, sam, sak, b, b_dtype, sbk, sbn, m, n, k, bias, int(bool(relu)), mask,
                           mask_dtype, mask_ld, out, out_dtype, ldo, int(bool(accumulate)), ws, ws_bytes, stream),
           "bg_sgemm")


def dropout_mask(seed, dropout_p, n_rows, keep, stream):
    _check(load().bg_dropout_mask(seed, dropout_p, n_rows, keep, stream), "bg_dropout_mask")


def eigen_loss(pred, y, n_graphs, scale, center, eps, out2, dpred, accum3, stream):
    _check(load().bg_eigen_loss(pred, y, n_graphs, scale, center, eps, out2, dpred, accum3, stream), "bg_eigen_loss")


def collate_ptr(sel, n_graphs, node_ptr, edge_ptr, out_node_ptr, out_edge_ptr, stream):
    _check(load().bg_collate_ptr(sel, n_graphs, node_ptr, edge_ptr, out_node_ptr, out_edge_ptr, stream), "bg_collate_ptr")


def collate(x_all, n_features, ei_all, e_all, ea_all, n_edge_features, y_all, sel, n_graphs, node_ptr, edge_ptr,
            out_node_ptr, out_edge_ptr, n_out, e_out, x, edge_index, edge_attr, batch, y, stream):
    _check(load().bg_collate(x_all, n_features, ei_all, e_all, ea_all, n_edge_features, y_all, sel, n_graphs, node_ptr,
                             edge_ptr, out_node_ptr, out_edge_ptr, n_out, e_out, x, edge_index, edge_attr, batch, y,
                             stream), "bg_collate")


def expand_wire(wire_edges, e_wire, node_ptr, wire_ptr, full_ptr, n_graphs, e_full, edge_index, batch, stream):
    _check(load().bg_expand_wire(wire_edges, e_wire, node_ptr, wire_ptr, full_ptr, n_graphs, e_full, edge_index, batch,
                                 stream), "bg_expand_wire")


def wgrad512(dz, ld_dz, act, act_cols, ld_act, dtype, n_rows, n_chunks, chunk_k, partial, stream):
    _check(load().bg_wgrad512(dz, ld_dz, act, act_cols, ld_act, dtype, n_rows, n_chunks, chunk_k, partial, stream),
           "bg_wgrad512")


def wgrad128(dz, agg, x, dtype, n_rows, n_chunks, chunk_k, partial, dwl, dwr, accumulate, stream):
    """bg_wgrad128: dwl (+)= dz^T agg, dwr (+)= dz^T x for [n_rows, 128] rows; partial [n_chunks * 256, 128] f32."""
    _check(load().bg_wgrad128(dz, agg, x, dtype, n_rows, n_chunks, chunk_k, partial, dwl, dwr, int(bool(accumulate)),
                              stream), "bg_wgrad128")


def wgrad128_ld(dz, a0, a1, dtype, n_rows, n_chunks, chunk_k, partial, dw0, ld0, dw1, ld1, accumulate, stream):
    """bg_wgrad128_ld: dw0[o*ld0 + i] (+)= (dz^T a0)[o, i] and, when a1 is given, dw1[o*ld1 + i] (+)= (dz^T a1)[o, i]
    for [n_rows, 128] rows; partial [n_chunks * 256, 128] f32."""
    _check(load().bg_wgrad128_ld(dz, a0, a1, dtype, n_rows, n_chunks, chunk_k, partial, dw0, ld0, dw1, ld1,
                                 int(bool(accumulate)), stream), "bg_wgrad128_ld")


def dropout_residual(x, x_prev, y, dtype, n_rows, dropout_p, seed, stream, width=512):
    fn = _w("bg_dropout_residual", width)
    _check(getattr(load(), fn)(x, x_prev, y, dtype, n_rows, dropout_p, seed, stream), fn)


def grad_mask(dy, dy2, act, out, dtype, n_rows, dropout_p, seed, stream, width=512):
    fn = _w("bg_grad_mask", width)
    _check(getattr(load(), fn)(dy, dy2, act, out, dtype, n_rows, dropout_p, seed, stream), fn)


def segment_expand(src, rowptr, n_rows, mean, out, dtype, stream, width=512):
    fn = _w("bg_segment_expand", width)
    _check(getattr(load(), fn)(src, rowptr, n_rows, int(bool(mean)), out, dtype, stream), fn)


# ----------------------------------------------------------------------------- SAGPooling
def sag_workspace_bytes(n_nodes: int, n_edges: int, n_graphs: int) -> int:
    return _query("bg_sag_workspace_bytes", n_nodes, n_edges, n_graphs)


def sag_select(x, dtype, n_nodes, rowptr, col, big_rows, n_big, w_l, w_r, bias, sign, graph_ptr, n_graphs, ratio,
               edge_index, n_edges, score, new_id, perm, batch_out, score_out, new_graph_ptr, info, ws, ws_bytes, stream):
    _check(load().bg_sag_select(x, dtype, n_nodes, rowptr, col, big_rows, n_big, w_l, w_r, bias, sign, graph_ptr,
                                n_graphs, ratio, edge_index, n_edges, score, new_id, perm, batch_out, score_out,
                                new_graph_ptr, info, ws, ws_bytes, stream), "bg_sag_select")


def sag_connect(edge_index, n_edges, n_nodes, new_id, n_edges_out, edge_index_out, kept_edge, ws, ws_bytes, stream):
    _check(load().bg_sag_connect(edge_index, n_edges, n_nodes, new_id, n_edges_out, edge_index_out, kept_edge, ws,
                                 ws_bytes, stream), "bg_sag_connect")


def gather_rows(x, dtype, ldx, row_index, row_scale, n_rows_out, out, ldo, stream):
    _check(load().bg_gather_rows(x, dtype, ldx, row_index, row_scale, n_rows_out, out, ldo, stream), "bg_gather_rows")


def index_invert(perm, n, out, stream):
    _check(load().bg_index_invert(perm, n, out, stream), "bg_index_invert")


def index_gather(table, idx, n, out, stream):
    _check(load().bg_index_gather(table, idx, n, out, stream), "bg_index_gather")


def sag_pool_backward(dx_pooled, x, dtype, n_nodes, n_nodes_out, perm, new_id, score, sign, rowptr_src, col_src,
                      big_rows_src, n_big_src, w_l, w_r, dx, t, dpre, stream):
    _check(load().bg_sag_pool_backward(dx_pooled, x, dtype, n_nodes, n_nodes_out, perm, new_id, score, sign, rowptr_src,
                                       col_src, big_rows_src, n_big_src, w_l, w_r, dx, t, dpre, stream),
           "bg_sag_pool_backward")


def max_bwd_workspace_bytes(n_big_tgt: int, n_big_src: int) -> int:
    return _query("bg_max_bwd_workspace_bytes", n_big_tgt, n_big_src)


def max_aggregate_backward(x, agg, dagg, dtype, n_nodes, rowptr_tgt, col_tgt, big_tgt, n_big_tgt, rowptr_src, col_src,
                           big_src, n_big_src, w_scratch, dx, ws, ws_bytes, stream, width=512):
    fn = _w("bg_max_aggregate_backward", width)
    _check(getattr(load(), fn)(x, agg, dagg, dtype, n_nodes, rowptr_tgt, col_tgt, big_tgt, n_big_tgt, rowptr_src, col_src,
                               big_src, n_big_src, w_scratch, dx, ws, ws_bytes, stream), fn)
