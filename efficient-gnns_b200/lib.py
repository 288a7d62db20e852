"""ctypes binding of ``libb200gnn.so`` — the C ABI declared in ``include/b200gnn.h``.

The library is the product: if it is missing or a symbol is absent this module
raises; nothing in this package falls back to PyTorch or CPU arithmetic.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import torch

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libb200gnn.so"

OK = 0
REDUCE_SUM = 0
REDUCE_MEAN = 1

_i32p = C.c_void_p
_f32p = C.c_void_p
_ptr = C.c_void_p
_i64 = C.c_int64
_i32 = C.c_int32
_int = C.c_int
_f32 = C.c_float
_u64 = C.c_uint64

# name -> (restype, argtypes).  tests/test_abi.py checks this table against the header.
SIGNATURES = {
    "b200gnn_abi_version": (_int, []),
    "b200gnn_error_string": (C.c_char_p, [_int]),
    "b200gnn_last_cuda_error": (C.c_char_p, []),
    "b200gnn_launch_count": (_i64, []),
    "b200gnn_reset_launch_count": (None, []),
    "b200gnn_csr_chunk_count": (_i64, [_i64, _i64, _i32, _i32]),
    "b200gnn_csr_chunk_plan": (_int, [_i32p, _i64, _i64, _i32, _i32, _i32p, _ptr]),
    "b200gnn_csr_hub_count": (_int, [_i32p, _i64, _i32, _i32, _i32p, _ptr]),
    "b200gnn_csr_hub_fill": (_int, [_i32p, _i64, _i32, _i32, _i32p, _i32p, _i64, _ptr]),
    "b200gnn_spmm_stat_slots": (_i64, [_i64, _i64]),
    "b200gnn_spmm_set_variant": (None, [_int]),
    "b200gnn_spmm_csr_f32": (_int, [_i32p, _i32p, _f32p, _f32p, _i64, _f32p, _i64, _i64, _i64, _i64, _int,
                                    _f32p, _f32p, _i32p, _i64, _i32, _i32, _i32p, _i32p, _i64, _i64, _f32p, _ptr]),
    "b200gnn_spmm_csr_scatter_f32": (_int, [_i32p, _i32p, _f32p, _f32p, _i64, _ptr, _ptr, _i32, _i64, _i64, _i64, _i64, _i64, _int,
                                            _f32p, _i32p, _i64, _i32, _i32, _i32p, _i32p, _i64, _i64, _f32p, _ptr]),
    "b200gnn_rows_slots": (_i64, [_i64]),
    "b200gnn_col_stats_f32": (_int, [_f32p, _i64, _i64, _f32p, _i64, _ptr]),
    "b200gnn_col_sum_f32": (_int, [_f32p, _i64, _i64, _f32p, _f32p, _i64, _ptr]),
    "b200gnn_bn_finalize_f32": (_int, [_f32p, _i64, _i64, _i64, _f32p, _f32p, _f32, _f32, _f32p, _f32p,
                                       _f32p, _f32p, _f32p, _f32p, _ptr]),
    "b200gnn_affine_relu_dropout_f32": (_int, [_f32p, _f32p, _i64, _i64, _f32p, _f32p, _int, _f32, _u64, _u64,
                                               _i32p, _u64, _u64, _ptr]),
    "b200gnn_affine_relu_dropout_mapped_f32": (_int, [_f32p, _f32p, _i64, _i64, _f32p, _f32p, _int, _f32, _u64, _u64,
                                                      _i32p, _u64, _i32p, _u64, _i64, _i64, _ptr]),
    "b200gnn_affine_relu_dropout_scatter_f32": (_int, [_f32p, _f32p, _i64, _i64, _f32p, _f32p, _int, _f32, _u64, _u64,
                                                       _i32p, _u64, _i32p, _u64, _i64, _i64, _ptr, _ptr, _i32, _i64, _ptr]),
    "b200gnn_dropout_mask_u8": (_int, [_ptr, _i64, _i64, _f32, _u64, _u64, _ptr]),
    "b200gnn_relu_dropout_bwd_f32": (_int, [_f32p, _f32p, _i64, _i64, _f32, _f32p, _ptr]),
    "b200gnn_relu_dropout_bwd_add_f32": (_int, [_f32p, _f32p, _i64, _i64, _f32p, _i64, _i64, _f32, _f32p, _ptr]),
    "b200gnn_bn_act_bwd_f32": (_int, [_f32p, _f32p, _f32p, _f32p, _f32p, _f32p, _i64, _i64, _f32, _f32p, _f32p,
                                      _f32p, _f32p, _f32p, _i64, _f32p, _ptr]),
    "b200gnn_bn_act_bwd_reduce_f32": (_int, [_f32p, _f32p, _f32p, _f32p, _f32p, _i64, _i64, _f32, _f32p, _i64, _ptr]),
    "b200gnn_bn_act_bwd_apply_f32": (_int, [_f32p, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, _i64, _i64, _i64, _i64, _f32,
                                            _f32p, _f32p, _f32p, _f32p, _f32p, _i64, _f32p, _ptr]),
    "b200gnn_partial_reduce_f32": (_int, [_f32p, _i64, _i64, _f32p, _ptr]),
    "b200gnn_adam_step_f32": (_int, [_f32p, _f32p, _f32p, _f32p, _i64, _f32, _f32, _f32, _f32, _i32p, _ptr]),
    "b200gnn_kd_partials": (_i64, [_i64]),
    "b200gnn_kd_loss_fwd_bwd_f32": (_int, [_f32p, _i64, _ptr, _i64, _ptr, _f32p, _i64, _i64, _f32, _f32, _i64, _f32p,
                                           _i64, _f32p, _f32p, _ptr]),
    "b200gnn_split_tf32_f32": (_int, [_f32p, _i64, _i64, _int, _f32p, _f32p, _ptr]),
    "b200gnn_gemm_tf32x3_f32": (_int, [_f32p, _i64, _f32p, _f32p, _i64, _f32p, _i64, _i64, _i64, _i64, _f32p, _ptr]),
    "b200gnn_random_walk_i64": (_int, [_i32p, _i32p, _i64, _ptr, _i64, _i32, _u64, _u64, _ptr, _ptr]),
    "b200gnn_saint_subgraph_count_i64": (_int, [_i32p, _i32p, _ptr, _i64, _i32p, _ptr, _ptr]),
    "b200gnn_saint_subgraph_fill_i64": (_int, [_i32p, _i32p, _ptr, _ptr, _i64, _i32p, _ptr, _ptr, _ptr, _ptr, _ptr]),
    "b200gnn_gemm_stat_slots": (_i64, [_i64, _i64]),
    "b200gnn_gemm_set_bnbwd_variant": (None, [_int]),
    "b200gnn_gemm_tf32x3_stats_f32": (_int, [_f32p, _i64, _f32p, _f32p, _i64, _f32p, _i64, _i64, _i64, _i64, _f32p, _int, _f32p, _i64,
                                             _ptr]),
    "b200gnn_gemm_tf32x3_bnbwd_f32": (_int, [_f32p, _i64, _f32p, _f32p, _i64, _f32p, _i64, _i64, _i64, _i64, _int,
                                             _f32p, _f32p, _f32p, _f32p, _f32, _f32p, _i64, _ptr]),
    "b200gnn_gemm_tf32x3_acc_f32": (_int, [_f32p, _i64, _f32p, _f32p, _i64, _f32p, _i64, _i64, _i64, _i64, _ptr]),
    "b200gnn_gemm_tf32x3_grouped_f32": (_int, [_f32p, _i64, _f32p, _i64, _i64, _ptr, _i32, _int, _ptr]),
    "b200gnn_gemm_tf32x3_scatter_f32": (_int, [_f32p, _i64, _f32p, _f32p, _i64, _ptr, _i32, _i64, _i64, _i64, _i64, _f32p, _ptr]),
    "b200gnn_gemm_tf32x3_bcast_f32": (_int, [_f32p, _i64, _f32p, _f32p, _i64, _ptr, _i32, _i64, _i64, _i64, _i64, _i64, _f32p, _ptr]),
    "b200gnn_wgrad_workspace_floats": (_i64, [_i64, _i64]),
    "b200gnn_wgrad_set_mode": (None, [_int]),
    "b200gnn_gemm_wgrad_tf32x3_f32": (_int, [_f32p, _i64, _f32p, _i64, _f32p, _i64, _i64, _i64, _f32p, _ptr]),
    "b200gnn_row_normalize_fwd_f32": (_int, [_f32p, _i64, _i64, _f32, _f32, _f32p, _f32p, _ptr]),
    "b200gnn_row_normalize_bwd_f32": (_int, [_f32p, _f32p, _f32p, _i64, _i64, _f32, _f32, _f32p, _int, _ptr]),
    "b200gnn_reduce_slots": (_i64, [_i64]),
    "b200gnn_mse_fwd_bwd_f32": (_int, [_f32p, _f32p, _i64, _f32, _f32p, _f32p, _f32p, _ptr]),
    "b200gnn_bce_logits_fwd_bwd_f32": (_int, [_f32p, _f32p, _int, _i64, _f32, _f32p, _f32p, _f32p, _ptr]),
    "b200gnn_row_sqnorm_f32": (_int, [_f32p, _i64, _i64, _f32p, _ptr]),
    "b200gnn_row_sqnorm_bwd_f32": (_int, [_f32p, _f32p, _i64, _i64, _f32p, _ptr]),
    "b200gnn_nce_rows_f32": (_int, [_f32p, _i64, _f32p, _f32p, _ptr]),
    "b200gnn_nce_rows_chunk_f32": (_int, [_f32p, _i64, _i64, _i64, _i64, _f32p, _ptr]),
    "b200gnn_nce_finish_f32": (_int, [_f32p, _i64, _f32p, _ptr]),
    "b200gnn_transpose_f32": (_int, [_f32p, _i64, _i64, _f32p, _ptr]),
    "b200gnn_gsp_pair_f32": (_int, [_f32p, _f32p, _f32p, _f32p, _i64, _int, _f32p, _f32p, _f32p, _ptr]),
    "b200gnn_row_axpy_f32": (_int, [_f32p, _f32p, _i64, _i64, _f32, _f32p, _ptr]),
    "b200gnn_edge_sim_f32": (_int, [_f32p, _i64, _i32p, _i32p, _i64, _int, _f32p, _ptr]),
    "b200gnn_lsp_partials": (_i64, [_i64]),
    "b200gnn_lsp_segment_f32": (_int, [_f32p, _f32p, _i32p, _i64, _i64, _int, _f32p, _f32p, _f32p, _ptr]),
    "b200gnn_edge_sim_bwd_f32": (_int, [_f32p, _i64, _i32p, _i32p, _i64, _int, _f32p, _f32p, _f32p, _ptr]),
    "b200gnn_lsp_bwd_values_f32": (_int, [_f32p, _i64, _i32p, _i32p, _i64, _int, _f32p, _f32p, _i32p, _i32p, _i32p, _i32p, _i64,
                                          _f32p, _f32p, _ptr]),
    "b200gnn_gat_edge_softmax_f32": (_int, [_i32p, _i32p, _f32p, _f32p, _i64, _i64, _f32, _f32, _f32p, _ptr, _ptr]),
    "b200gnn_gat_aggregate_f32": (_int, [_i32p, _i32p, _i32p, _f32p, _f32p, _i64, _f32p, _i64, _i64, _i64, _i64, _i32p, _i64,
                                         _i32, _i32, _i32p, _i32p, _i64, _i64, _f32p, _ptr]),
    "b200gnn_gat_bwd_rows_f32": (_int, [_i32p, _i32p, _f32p, _f32p, _i64, _f32p, _i64, _f32p, _f32p, _i64, _i64, _i64, _f32,
                                        _f32p, _f32p, _i32p, _i64, _i32, _i32, _i32p, _i32p, _i64, _i64, _f32p, _f32p, _ptr]),
    "b200gnn_segment_sum_heads_f32": (_int, [_i32p, _i32p, _f32p, _i64, _i64, _f32p, _ptr]),
    "b200gnn_graph_sort_workspace_bytes": (_i64, [_i64]),
    "b200gnn_graph_argsort_i64": (_int, [_ptr, _ptr, _i64, _i64, _i64, _i32p, _ptr, _ptr]),
    "b200gnn_graph_coalesce_i64": (_int, [_ptr, _ptr, _i64, _i64, _i64, _ptr, _ptr, _i32p, _ptr, _ptr, _ptr, _ptr]),
    "b200gnn_typed_gather_f32": (_int, [_ptr, _ptr, _i32, _ptr, _ptr, _i64, _i64, _f32p, _i64, _i32p, _ptr]),
    "b200gnn_typed_scatter_f32": (_int, [_f32p, _i64, _ptr, _ptr, _ptr, _i64, _i64, _ptr, _ptr, _i32, _ptr]),
    "b200gnn_arena_alloc": (_int, [_i64, C.POINTER(C.c_void_p)]),
    "b200gnn_arena_free": (_int, [_ptr]),
    "b200gnn_ipc_get_handle": (_int, [_ptr, _ptr]),
    "b200gnn_ipc_open_handle": (_int, [_ptr, C.POINTER(C.c_void_p)]),
    "b200gnn_ipc_close_handle": (_int, [_ptr]),
    "b200gnn_peer_copy2d_f32": (_int, [_ptr, _i32, _i64, _ptr]),
    "b200gnn_peer_barrier": (_int, [_ptr, _i32, _i32, _ptr, _ptr, _ptr]),
    "b200gnn_peer_exchange_f32": (_int, [_ptr, _i32, _i64, _ptr, _i32, _i32, _ptr, _ptr, _ptr, _ptr]),
}


class Copy2D(C.Structure):
    """struct b200gnn_copy2d (include/b200gnn.h)."""
    _fields_ = [("dst", C.c_void_p), ("src", C.c_void_p), ("ld_dst", C.c_int64), ("ld_src", C.c_int64), ("rows", C.c_int64)]


class GemmGroup(C.Structure):
    """struct b200gnn_gemm_group (include/b200gnn.h)."""
    _fields_ = [("B_hi", C.c_void_p), ("B_lo", C.c_void_p), ("ldb", C.c_int64), ("bias", C.c_void_p), ("row0", C.c_int64),
                ("rows", C.c_int64), ("K", C.c_int64)]


_lib = None


class B200GnnError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (once). Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise B200GnnError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU or PyTorch fallback for the b200gnn operators.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError => ABI mismatch, fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.b200gnn_abi_version() != 1:
        raise B200GnnError("libb200gnn.so ABI version mismatch; rebuild")
    _lib = lib
    report = os.environ.get("B200GNN_LAUNCH_REPORT")
    if report:          # evidence for out-of-process runs (the unmodified reference scripts on the shims): kernels launched
        import atexit
        atexit.register(lambda: Path(report).write_text(str(int(lib.b200gnn_launch_count()))))
    return lib


def check(rc: int, what: str) -> None:
    if rc != OK:
        lib = load()
        msg = lib.b200gnn_error_string(rc).decode()
        if rc == -3:
            msg += ": " + lib.b200gnn_last_cuda_error().decode()
        raise B200GnnError(f"{what} failed: {msg}")


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def dptr(t: torch.Tensor | None, dtype: torch.dtype, name: str) -> int | None:
    """Device pointer of a contiguous CUDA tensor of the given dtype (None passes through)."""
    if t is None:
        return None
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a tensor")
    if not t.is_cuda:
        raise B200GnnError(f"{name}: b200gnn operators need CUDA tensors (got {t.device}); there is no CPU fallback")
    if t.dtype != dtype:
        raise B200GnnError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise B200GnnError(f"{name}: tensor must be contiguous")
    return t.data_ptr()


def launch_count() -> int:
    return int(load().b200gnn_launch_count())


def reset_launch_count() -> None:
    load().b200gnn_reset_launch_count()
