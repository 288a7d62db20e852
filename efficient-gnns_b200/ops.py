"""Operators: thin, checked launches of the C ABI plus their autograd wiring.

Every function here ends in a ``libb200gnn.so`` call on the current CUDA stream;
PyTorch only provides the device buffers and the autograd tape.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import lib
from .sparse import CsrGraph, SparseTensor

_REDUCE = {"sum": lib.REDUCE_SUM, "add": lib.REDUCE_SUM, "mean": lib.REDUCE_MEAN}


def set_spmm_variant(variant: int) -> None:
    """0 = automatic kernel choice, 1 = force the register-staged SpMM kernel (A/B measurements)."""
    lib.load().b200gnn_spmm_set_variant(int(variant))


def stat_slots(g: CsrGraph) -> int:
    return int(lib.load().b200gnn_spmm_stat_slots(g.n_chunks, g.n_hub))


def spmm_csr(g: CsrGraph, x: torch.Tensor, reduce: str = "sum", bias: Optional[torch.Tensor] = None,
             out: Optional[torch.Tensor] = None, stat_partial: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Y = reduce_e val[e]·X[col[e]] (+bias), optional fused column statistics. No autograd."""
    if reduce not in _REDUCE:
        raise ValueError(f"reduce={reduce!r}: the engine implements sum/add/mean (what the reference path uses)")
    if x.dim() != 2:
        raise lib.B200GnnError("spmm: dense operand must be [n_src, K]")
    if x.shape[0] < g.n_cols:   # extra trailing rows are harmless (upstream accepts them: mag_pyg/gnn.py:151-162 infers
        raise lib.B200GnnError(  # the sparse sizes as max+1 and multiplies by the full per-type feature matrix)
            f"spmm: dense operand has {x.shape[0]} rows, matrix has {g.n_cols} columns")
    K = x.shape[1]
    if out is None:
        out = torch.empty(g.n_rows, K, dtype=torch.float32, device=x.device)
    if g.n_rows == 0 or K == 0:
        return out
    L = lib.load()
    ws = g.hub_workspace(K)
    rc = L.b200gnn_spmm_csr_f32(
        lib.dptr(g.rowptr, torch.int32, "rowptr"), lib.dptr(g.col, torch.int32, "col"),
        lib.dptr(g.val, torch.float32, "val"), lib.dptr(x, torch.float32, "x"), x.stride(0),
        lib.dptr(out, torch.float32, "out"), out.stride(0), g.n_rows, g.n_cols, K, _REDUCE[reduce],
        lib.dptr(bias, torch.float32, "bias"), lib.dptr(stat_partial, torch.float32, "stat_partial"),
        g.chunk_rowptr.data_ptr(), g.n_chunks, g.hub_threshold, g.seg_len,
        g.hub_rows.data_ptr() if g.n_hub else None, g.hub_segptr.data_ptr() if g.n_hub else None,
        g.n_hub, g.n_seg, None if ws is None else ws.data_ptr(), lib.stream_ptr())
    lib.check(rc, "spmm_csr_f32")
    return out


def _host_ptr_array(ptrs):
    import ctypes as C
    return (C.c_void_p * len(ptrs))(*[C.c_void_p(int(p)) for p in ptrs])


def _host_i32_array(vals):
    import ctypes as C
    return (C.c_int32 * len(vals))(*[int(v) for v in vals])


def spmm_csr_scatter(g: CsrGraph, x: torch.Tensor, dst_ptrs, row_off, ld_dst: int, col_dst: int, reduce: str = "sum",
                     bias: Optional[torch.Tensor] = None) -> None:
    """Y = A·X (+bias) with output row i stored to the R-layout buffer of the rank that owns it (raw device addresses
    dst_ptrs[q], rows row_off[q]..row_off[q+1], pitch ld_dst floats, column offset col_dst): the aggregation's epilogue performs
    the multi-GPU engine's C->R exchange."""
    K = x.shape[1]
    L = lib.load()
    ws = g.hub_workspace(K)
    rc = L.b200gnn_spmm_csr_scatter_f32(
        lib.dptr(g.rowptr, torch.int32, "rowptr"), lib.dptr(g.col, torch.int32, "col"), lib.dptr(g.val, torch.float32, "val"),
        lib.dptr(x, torch.float32, "x"), x.stride(0), _host_ptr_array(dst_ptrs), _host_i32_array(row_off), len(dst_ptrs),
        int(ld_dst), int(col_dst), g.n_rows, g.n_cols, K, _REDUCE[reduce], lib.dptr(bias, torch.float32, "bias"),
        g.chunk_rowptr.data_ptr(), g.n_chunks, g.hub_threshold, g.seg_len,
        g.hub_rows.data_ptr() if g.n_hub else None, g.hub_segptr.data_ptr() if g.n_hub else None,
        g.n_hub, g.n_seg, None if ws is None else ws.data_ptr(), lib.stream_ptr())
    lib.check(rc, "spmm_csr_scatter_f32")


class _SpMM(torch.autograd.Function):
    """matmul(adj, x, reduce): backward is the same kernel on the cached CSC view
    (upstream torch_sparse spmm backward, SURVEY Appendix A.4)."""

    @staticmethod
    def forward(ctx, x, adj: SparseTensor, reduce: str):
        st = adj.storage
        g = st.engine_csr() if st.value() is not None else st.engine_csr_unweighted()
        ctx.adj, ctx.reduce = adj, reduce
        return spmm_csr(g, x.contiguous(), reduce)

    @staticmethod
    def backward(ctx, grad_out):
        st = ctx.adj.storage
        if ctx.reduce == "mean":
            gt = st.engine_csc("mean" if st.value() is None else "mean_value")
        else:
            gt = st.engine_csc("value")
        return spmm_csr(gt, grad_out.contiguous(), "sum"), None, None


def matmul(adj: SparseTensor, x: torch.Tensor, reduce: str = "sum") -> torch.Tensor:
    """torch_sparse.matmul(adj, dense, reduce) for reduce in {sum, add, mean}."""
    if reduce not in _REDUCE:
        raise ValueError(f"reduce={reduce!r} not implemented (reference path uses add/mean)")
    v = adj.storage.value()
    if v is not None and v.requires_grad:
        raise NotImplementedError("gradients w.r.t. sparse values are never taken on the reference path")
    if x.dim() == 1:
        return matmul(adj, x.unsqueeze(-1), reduce).squeeze(-1)
    return _SpMM.apply(x, adj, reduce)


# ----------------------------------------------------------------------------- dense row passes (raw launches)
def _f32(t, name):
    return lib.dptr(t, torch.float32, name)


def _f32_rows(t, name):
    """Device pointer of a row-strided fp32 matrix view (unit column stride; the row pitch is passed separately)."""
    if t is None:
        return None
    if t.dim() != 2 or (t.stride(1) != 1 and t.shape[1] > 1):
        raise lib.B200GnnError(f"{name}: expected a 2-D view with unit column stride")
    if not t.is_cuda or t.dtype != torch.float32:
        raise lib.B200GnnError(f"{name}: expected a CUDA float32 tensor (got {t.device}, {t.dtype}); there is no CPU fallback")
    return t.data_ptr()


def rows_slots(n_rows: int) -> int:
    return int(lib.load().b200gnn_rows_slots(n_rows))


def col_stats(y: torch.Tensor, partial: Optional[torch.Tensor] = None) -> torch.Tensor:
    """partial[slots][2][K]: per-slot column sums / sums of squares of y [n,K]."""
    n, K = y.shape
    slots = rows_slots(n)
    if partial is None:
        partial = torch.empty(slots, 2, K, dtype=torch.float32, device=y.device)
    lib.check(lib.load().b200gnn_col_stats_f32(_f32(y, "y"), n, K, _f32(partial, "partial"), slots, lib.stream_ptr()),
              "col_stats_f32")
    return partial


def col_sum(y: torch.Tensor, out: Optional[torch.Tensor] = None, partial: Optional[torch.Tensor] = None) -> torch.Tensor:
    n, K = y.shape
    slots = rows_slots(n)
    if out is None:
        out = torch.empty(K, dtype=torch.float32, device=y.device)
    if partial is None:
        partial = torch.empty(slots, 2, K, dtype=torch.float32, device=y.device)
    lib.check(lib.load().b200gnn_col_sum_f32(_f32(y, "y"), n, K, _f32(out, "out"), _f32(partial, "partial"), slots,
                                             lib.stream_ptr()), "col_sum_f32")
    return out


def bn_finalize(partial: torch.Tensor, n_rows: int, gamma, beta, eps: float = 1e-5, momentum: float = 0.1,
                running_mean=None, running_var=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Returns a [4,K] tensor: rows = mean, invstd, scale, shift."""
    slots, _, K = partial.shape
    if out is None:
        out = torch.empty(4, K, dtype=torch.float32, device=partial.device)
    lib.check(lib.load().b200gnn_bn_finalize_f32(
        _f32(partial, "partial"), slots, K, n_rows, _f32(gamma, "gamma"), _f32(beta, "beta"), eps, momentum,
        _f32(running_mean, "running_mean"), _f32(running_var, "running_var"),
        out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(), out[3].data_ptr(), lib.stream_ptr()), "bn_finalize_f32")
    return out


def affine_relu_dropout(y: torch.Tensor, scale=None, shift=None, relu: bool = True, p: float = 0.0, seed: int = 0,
                        offset: int = 0, out: Optional[torch.Tensor] = None, step_dev: Optional[torch.Tensor] = None,
                        step_mul: int = 0, row_offset: int = 0) -> torch.Tensor:
    n, K = y.shape
    if out is None:
        out = torch.empty_like(y)
    lib.check(lib.load().b200gnn_affine_relu_dropout_f32(
        _f32(y, "y"), _f32(out, "out"), n, K, _f32(scale, "scale"), _f32(shift, "shift"), int(relu), p, seed, offset,
        lib.dptr(step_dev, torch.int32, "step_dev"), step_mul, row_offset, lib.stream_ptr()), "affine_relu_dropout_f32")
    return out


def affine_relu_dropout_mapped(y: torch.Tensor, scale=None, shift=None, relu: bool = True, p: float = 0.0, seed: int = 0,
                               offset: int = 0, out: Optional[torch.Tensor] = None, step_dev: Optional[torch.Tensor] = None,
                               step_mul: int = 0, rowmap: Optional[torch.Tensor] = None, row_offset: int = 0,
                               k_global: Optional[int] = None, col_offset: int = 0) -> torch.Tensor:
    """affine_relu_dropout on a row/column BLOCK of an [N, k_global] activation matrix: local row r is node
    rowmap[r] (int32) or r + row_offset, local columns start at col_offset.  Masks match the full-matrix call."""
    n, K = y.shape
    if out is None:
        out = torch.empty_like(y)
    lib.check(lib.load().b200gnn_affine_relu_dropout_mapped_f32(
        _f32(y, "y"), _f32(out, "out"), n, K, _f32(scale, "scale"), _f32(shift, "shift"), int(relu), p, seed, offset,
        lib.dptr(step_dev, torch.int32, "step_dev"), step_mul, lib.dptr(rowmap, torch.int32, "rowmap"), row_offset,
        K if k_global is None else k_global, col_offset, lib.stream_ptr()), "affine_relu_dropout_mapped_f32")
    return out


def affine_relu_dropout_scatter(y: torch.Tensor, scale, shift, relu: bool, p: float, seed: int, offset: int, out: torch.Tensor,
                                step_dev, step_mul: int, rowmap, k_global: int, col_offset: int, dst_ptrs, row_off,
                                ld_dst: int) -> torch.Tensor:
    """affine_relu_dropout_mapped that ALSO stores every output row into the R-layout buffer of the rank owning the node
    (the multi-GPU engine's C->R exchange fused into the activation pass)."""
    n, K = y.shape
    lib.check(lib.load().b200gnn_affine_relu_dropout_scatter_f32(
        _f32(y, "y"), _f32(out, "out"), n, K, _f32(scale, "scale"), _f32(shift, "shift"), int(relu), p, seed, offset,
        lib.dptr(step_dev, torch.int32, "step_dev"), step_mul, lib.dptr(rowmap, torch.int32, "rowmap"), 0, k_global, col_offset,
        _host_ptr_array(dst_ptrs), _host_i32_array(row_off), len(dst_ptrs), int(ld_dst), lib.stream_ptr()),
        "affine_relu_dropout_scatter_f32")
    return out


def relu_dropout_bwd(d_out: torch.Tensor, x_out: torch.Tensor, p: float, out: Optional[torch.Tensor] = None,
                     extra: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Backward of x_out = dropout_p(relu(y)): d_y = d_out * [x_out > 0] / (1-p); ``out`` may be ``d_out``.  With ``extra``
    (a row-strided [n, K_extra] view, K_extra <= K, e.g. the gradient of a loss on the unpadded hidden activation) the
    upstream gradient is d_out + extra (zero past K_extra), added before the scaling."""
    n, K = x_out.shape
    out = torch.empty_like(x_out) if out is None else out
    if extra is None:
        lib.check(lib.load().b200gnn_relu_dropout_bwd_f32(_f32(d_out, "d_out"), _f32(x_out, "x_out"), n, K, float(p),
                                                          _f32(out, "out"), lib.stream_ptr()), "relu_dropout_bwd_f32")
        return out
    if extra.dim() != 2 or extra.shape[0] != n:
        raise lib.B200GnnError(f"relu_dropout_bwd: extra must be [{n}, K_extra], got {tuple(extra.shape)}")
    lib.check(lib.load().b200gnn_relu_dropout_bwd_add_f32(_f32(d_out, "d_out"), _f32_rows(extra, "extra"), extra.stride(0),
                                                          extra.shape[1], _f32(x_out, "x_out"), n, K, float(p),
                                                          _f32(out, "out"), lib.stream_ptr()), "relu_dropout_bwd_add_f32")
    return out


def dropout_mask(n_rows: int, K: int, p: float, seed: int, offset: int, device="cuda") -> torch.Tensor:
    """The keep-mask (uint8 [n,K]) that affine_relu_dropout uses for (seed, offset)."""
    mask = torch.empty(n_rows, K, dtype=torch.uint8, device=device)
    lib.check(lib.load().b200gnn_dropout_mask_u8(mask.data_ptr(), n_rows, K, p, seed, offset, lib.stream_ptr()),
              "dropout_mask_u8")
    return mask


def bn_act_bwd(d_out, x_out, y, mean, invstd, gamma, p: float, d_y=None, d_gamma=None, d_beta=None, d_bias=None,
               partial=None, coef=None, want_dbias: bool = True):
    """Backward of x_out = dropout_p(relu(BN_train(y))). Returns (d_y, d_gamma, d_beta, d_bias)."""
    n, K = y.shape
    dev = y.device
    slots = rows_slots(n)
    d_y = torch.empty_like(y) if d_y is None else d_y
    d_gamma = torch.empty(K, device=dev) if d_gamma is None else d_gamma
    d_beta = torch.empty(K, device=dev) if d_beta is None else d_beta
    if want_dbias and d_bias is None:
        d_bias = torch.empty(K, device=dev)
    partial = torch.empty(slots, 2, K, device=dev) if partial is None else partial
    coef = torch.empty(3, K, device=dev) if coef is None else coef
    lib.check(lib.load().b200gnn_bn_act_bwd_f32(
        _f32(d_out, "d_out"), _f32(x_out, "x_out"), _f32(y, "y"), _f32(mean, "mean"), _f32(invstd, "invstd"),
        _f32(gamma, "gamma"), n, K, p, _f32(d_y, "d_y"), _f32(d_gamma, "d_gamma"), _f32(d_beta, "d_beta"),
        _f32(d_bias, "d_bias") if want_dbias else None, _f32(partial, "partial"), slots, _f32(coef, "coef"),
        lib.stream_ptr()), "bn_act_bwd_f32")
    return d_y, d_gamma, d_beta, d_bias


def adam_step(params, grads, exp_avg, exp_avg_sq, step: torch.Tensor, lr: float, betas=(0.9, 0.999), eps: float = 1e-8):
    lib.check(lib.load().b200gnn_adam_step_f32(
        _f32(params, "params"), _f32(grads, "grads"), _f32(exp_avg, "exp_avg"), _f32(exp_avg_sq, "exp_avg_sq"),
        params.numel(), lr, betas[0], betas[1], eps, lib.dptr(step, torch.int32, "step"), lib.stream_ptr()),
        "adam_step_f32")


def kd_loss_fwd_bwd(logits, labels, train_idx, teacher_logits=None, alpha: float = 0.9, T: float = 4.0,
                    d_logits=None, loss_out=None, partial=None, n_norm: int = 0):
    """Fused CE / logit-KD over rows train_idx of FULL [N,C] matrices (row-strided views accepted, e.g. the first C columns
    of a padded buffer); returns (loss_out[3], d_logits [N,C])."""
    N, C = logits.shape
    n_train = train_idx.numel() if train_idx is not None else N
    L = lib.load()
    if d_logits is None:
        d_logits = torch.zeros_like(logits)
    if loss_out is None:
        loss_out = torch.empty(3, dtype=torch.float32, device=logits.device)
    if partial is None:
        partial = torch.empty(2 * int(L.b200gnn_kd_partials(max(n_train, 1))), dtype=torch.float32, device=logits.device)
    lib.check(L.b200gnn_kd_loss_fwd_bwd_f32(
        _f32_rows(logits, "logits"), logits.stride(0), lib.dptr(train_idx, torch.int64, "train_idx"), n_train,
        lib.dptr(labels, torch.int64, "labels"), _f32_rows(teacher_logits, "teacher_logits"),
        teacher_logits.stride(0) if teacher_logits is not None else 0, C, alpha, T, n_norm, _f32_rows(d_logits, "d_logits"),
        d_logits.stride(0), _f32(loss_out, "loss_out"), _f32(partial, "partial"), lib.stream_ptr()), "kd_loss_fwd_bwd_f32")
    return loss_out, d_logits


# ----------------------------------------------------------------------------- tcgen05 3xTF32 GEMM
def split_tf32(w: torch.Tensor, transpose: bool = False, hi: Optional[torch.Tensor] = None,
               lo: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """(hi, lo) tf32 split of a small [rows, cols] matrix; transposed ([cols, rows]) output if requested."""
    rows, cols = w.shape
    shape = (cols, rows) if transpose else (rows, cols)
    hi = torch.empty(shape, dtype=torch.float32, device=w.device) if hi is None else hi
    lo = torch.empty(shape, dtype=torch.float32, device=w.device) if lo is None else lo
    lib.check(lib.load().b200gnn_split_tf32_f32(_f32(w, "w"), rows, cols, int(transpose), _f32(hi, "hi"), _f32(lo, "lo"),
                                                lib.stream_ptr()), "split_tf32_f32")
    return hi, lo


def gemm_tf32x3(a: torch.Tensor, b_hi: torch.Tensor, b_lo: torch.Tensor, bias: Optional[torch.Tensor] = None,
                out: Optional[torch.Tensor] = None, accumulate: bool = False) -> torch.Tensor:
    """out[M,N] (+)= a[M,K] @ b[N,K]^T (+bias) with fp32 fidelity on the tensor cores (b pre-split by split_tf32); a and out
    may be row-strided views."""
    M, K = a.shape
    N = b_hi.shape[0]
    assert b_hi.shape == b_lo.shape and b_hi.shape[1] == K
    if out is None:
        assert not accumulate
        out = torch.empty(M, N, dtype=torch.float32, device=a.device)
    L = lib.load()
    if accumulate:
        assert bias is None
        lib.check(L.b200gnn_gemm_tf32x3_acc_f32(_f32_rows(a, "a"), a.stride(0), _f32(b_hi, "b_hi"), _f32(b_lo, "b_lo"),
                                                b_hi.stride(0), _f32_rows(out, "out"), out.stride(0), M, N, K, lib.stream_ptr()),
                  "gemm_tf32x3_acc_f32")
        return out
    lib.check(L.b200gnn_gemm_tf32x3_f32(_f32_rows(a, "a"), a.stride(0), _f32(b_hi, "b_hi"), _f32(b_lo, "b_lo"),
                                        b_hi.stride(0), _f32_rows(out, "out"), out.stride(0), M, N, K,
                                        _f32(bias, "bias"), lib.stream_ptr()), "gemm_tf32x3_f32")
    return out


def gemm_tf32x3_grouped(a: torch.Tensor, out: torch.Tensor, groups, accumulate: bool = False) -> torch.Tensor:
    """One launch of out[r0:r0+m, :N] (+)= a[r0:r0+m, :K_g] @ b_g[N, K_g]^T (+bias_g) over the groups
    ``(row0, rows, b_hi, b_lo, bias)`` (b pre-split by split_tf32, K_g = b_hi.shape[1], bias may be None; b_hi None means
    K_g = 0).  ``a`` and ``out`` may be row-strided views (unit column stride)."""
    N = out.shape[1]
    arr = (lib.GemmGroup * max(len(groups), 1))()
    for i, (row0, rows, b_hi, b_lo, bias) in enumerate(groups):
        if b_hi is not None:
            assert b_hi.shape == b_lo.shape and b_hi.shape[0] == N and b_hi.stride(0) == b_lo.stride(0)
            arr[i].B_hi, arr[i].B_lo, arr[i].ldb, arr[i].K = _f32_rows(b_hi, "b_hi"), _f32_rows(b_lo, "b_lo"), b_hi.stride(0), b_hi.shape[1]
        arr[i].bias = _f32(bias, "bias")
        arr[i].row0, arr[i].rows = int(row0), int(rows)
    lib.check(lib.load().b200gnn_gemm_tf32x3_grouped_f32(_f32_rows(a, "a"), a.stride(0), _f32_rows(out, "out"), out.stride(0), N,
                                                         arr, len(groups), int(accumulate), lib.stream_ptr()),
              "gemm_tf32x3_grouped_f32")
    return out


def gemm_stat_slots(m: int, n: int) -> int:
    """Slots of the [slots, 2, n] partial buffer the statistics-fused GEMMs fill."""
    return int(lib.load().b200gnn_gemm_stat_slots(m, n))


def gemm_stats_supported(n: int) -> bool:
    return n % 32 == 0 and 48 < n <= 256


def gemm_tf32x3_stats(a: torch.Tensor, b_hi: torch.Tensor, b_lo: torch.Tensor, bias: Optional[torch.Tensor], out: torch.Tensor,
                      partial: torch.Tensor, accumulate: bool = False) -> torch.Tensor:
    """out = a @ b^T + bias (or out += a @ b^T) with the BatchNorm batch statistics of the final ``out`` reduced in the epilogue:
    partial[slots, 2, N] = per-slot (column sum, column sum of squares) — feed to ``bn_finalize`` (no sweep over out)."""
    M, K = a.shape
    N = b_hi.shape[0]
    lib.check(lib.load().b200gnn_gemm_tf32x3_stats_f32(_f32(a, "a"), a.stride(0), _f32(b_hi, "b_hi"), _f32(b_lo, "b_lo"),
                                                       b_hi.stride(0), _f32(out, "out"), out.stride(0), M, N, K, _f32(bias, "bias"),
                                                       int(accumulate), _f32(partial, "partial"), partial.shape[0], lib.stream_ptr()),
              "gemm_tf32x3_stats_f32")
    return out


def gemm_tf32x3_bnbwd(a: torch.Tensor, b_hi: torch.Tensor, b_lo: torch.Tensor, out: torch.Tensor, x_out: torch.Tensor,
                      y: torch.Tensor, mean: torch.Tensor, invstd: torch.Tensor, p: float, partial: torch.Tensor,
                      accumulate: bool = False) -> torch.Tensor:
    """Input-gradient GEMM with pass 1 of the BatchNorm/ReLU/dropout backward in its epilogue: d_out = a @ b^T (+ out),
    and what is STORED to ``out`` is dz = d_out * [x_out > 0] / (1-p); partial[slots, 2, N] = per-slot (sum dz, sum dz*xhat).
    Follow with ``bn_act_bwd_apply(out, None, y, ..., sums=partial, ...)``."""
    M, K = a.shape
    N = b_hi.shape[0]
    assert out.shape == x_out.shape == y.shape and out.stride(0) == x_out.stride(0) == y.stride(0)
    lib.check(lib.load().b200gnn_gemm_tf32x3_bnbwd_f32(_f32(a, "a"), a.stride(0), _f32(b_hi, "b_hi"), _f32(b_lo, "b_lo"),
                                                       b_hi.stride(0), _f32(out, "out"), out.stride(0), M, N, K, int(accumulate),
                                                       _f32(x_out, "x_out"), _f32(y, "y"), _f32(mean, "mean"),
                                                       _f32(invstd, "invstd"), float(p), _f32(partial, "partial"),
                                                       partial.shape[0], lib.stream_ptr()), "gemm_tf32x3_bnbwd_f32")
    return out


def gemm_tf32x3_scatter(a: torch.Tensor, b_hi: torch.Tensor, b_lo: torch.Tensor, dst_ptrs, row_off: int,
                        bias: Optional[torch.Tensor] = None) -> None:
    """a[M,K] @ b[N,K]^T with column block q of the result stored to the [*, N/world] matrix at raw device address
    dst_ptrs[q] (rows row_off + m): the GEMM epilogue performs the multi-GPU engine's R->C exchange (peer-mapped targets)."""
    import ctypes as C
    M, K = a.shape
    N = b_hi.shape[0]
    world = len(dst_ptrs)
    arr = (C.c_void_p * world)(*[C.c_void_p(int(p)) for p in dst_ptrs])
    lib.check(lib.load().b200gnn_gemm_tf32x3_scatter_f32(_f32(a, "a"), a.stride(0), _f32(b_hi, "b_hi"), _f32(b_lo, "b_lo"),
                                                         b_hi.stride(0), arr, world, int(row_off), M, N, K, _f32(bias, "bias"),
                                                         lib.stream_ptr()), "gemm_tf32x3_scatter_f32")


def gemm_tf32x3_bcast(a: torch.Tensor, b_hi: torch.Tensor, b_lo: torch.Tensor, dst_ptrs, row_off: int, ldc: int,
                      bias: Optional[torch.Tensor] = None) -> None:
    """a[M,K] @ b[N,K]^T stored to EVERY buffer at raw address dst_ptrs[q] (rows row_off + m, pitch ldc): the multi-GPU
    engine's row all-gather of a narrow result fused into the GEMM epilogue."""
    M, K = a.shape
    N = b_hi.shape[0]
    lib.check(lib.load().b200gnn_gemm_tf32x3_bcast_f32(_f32(a, "a"), a.stride(0), _f32(b_hi, "b_hi"), _f32(b_lo, "b_lo"),
                                                       b_hi.stride(0), _host_ptr_array(dst_ptrs), len(dst_ptrs), int(row_off), int(ldc),
                                                       M, N, K, _f32(bias, "bias"), lib.stream_ptr()), "gemm_tf32x3_bcast_f32")


def wgrad_supported(k_in: int, n_out: int) -> bool:
    return k_in in (128, 256) and n_out % 4 == 0 and 0 < n_out <= 256


def gemm_wgrad_tf32x3(x: torch.Tensor, g: torch.Tensor, out: Optional[torch.Tensor] = None,
                      workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[Kin,Nout] = x[Nn,Kin]^T @ g[Nn,Nout] on the tensor cores with fp32 fidelity (split-K over nodes); x and g may be
    row-strided views."""
    nn_, k_in = x.shape
    n_out = g.shape[1]
    assert g.shape[0] == nn_
    L = lib.load()
    if out is None:
        out = torch.empty(k_in, n_out, dtype=torch.float32, device=x.device)
    if workspace is None:
        workspace = torch.empty(int(L.b200gnn_wgrad_workspace_floats(k_in, n_out)), dtype=torch.float32, device=x.device)
    lib.check(L.b200gnn_gemm_wgrad_tf32x3_f32(_f32_rows(x, "x"), x.stride(0), _f32_rows(g, "g"), g.stride(0), _f32(out, "out"), nn_,
                                              k_in, n_out, _f32(workspace, "workspace"), lib.stream_ptr()),
              "gemm_wgrad_tf32x3_f32")
    return out


def partial_reduce(partial: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """[slots, 2, K] (or [slots, K2]) partial sums -> [2, K] / [K2] totals (before a cross-rank all-reduce)."""
    slots = partial.shape[0]
    k2 = partial.numel() // slots
    if out is None:
        out = torch.empty(partial.shape[1:], dtype=torch.float32, device=partial.device)
    lib.check(lib.load().b200gnn_partial_reduce_f32(_f32(partial, "partial"), slots, k2, _f32(out, "out"), lib.stream_ptr()),
              "partial_reduce_f32")
    return out


def bn_act_bwd_reduce(d_out, x_out, y, mean, invstd, p: float, partial: torch.Tensor) -> torch.Tensor:
    n, K = y.shape
    lib.check(lib.load().b200gnn_bn_act_bwd_reduce_f32(_f32(d_out, "d_out"), _f32(x_out, "x_out"), _f32(y, "y"),
                                                       _f32(mean, "mean"), _f32(invstd, "invstd"), n, K, p,
                                                       _f32(partial, "partial"), partial.shape[0], lib.stream_ptr()),
              "bn_act_bwd_reduce_f32")
    return partial


def bn_act_bwd_apply(d_out, x_out, y, mean, invstd, gamma, sums, n_norm: int, p: float, d_y, d_gamma, d_beta, d_bias,
                     partial, coef):
    n, K = y.shape
    sum_slots = sums.numel() // (2 * K)
    lib.check(lib.load().b200gnn_bn_act_bwd_apply_f32(
        _f32(d_out, "d_out"), _f32(x_out, "x_out"), _f32(y, "y"), _f32(mean, "mean"), _f32(invstd, "invstd"),
        _f32(gamma, "gamma"), _f32(sums, "sums"), sum_slots, n_norm, n, K, p, _f32(d_y, "d_y"), _f32(d_gamma, "d_gamma"),
        _f32(d_beta, "d_beta"), _f32(d_bias, "d_bias"), _f32(partial, "partial"), partial.shape[0], _f32(coef, "coef"),
        lib.stream_ptr()), "bn_act_bwd_apply_f32")
