"""Fused full-batch training step for the GraphSAGE student — BASELINE.json configs[2] (SAGE + G-CRD) and the reference's
``train()`` for ``--gnn sage`` (arxiv_pyg/gnn.py:56-85 ``SAGE``, :102-195 ``train``; SAGEConv semantics SURVEY Appendix A.3).

Per layer (PyG SAGEConv: aggregate first, no self loops, unweighted mean):

    M  = mean_{j in N(i)} X_j                       b200gnn SpMM (mean), TMA kernels at these widths
    Y  = M W_l^T + b_l + X W_r^T                    two tcgen05 GEMMs, the second through the ACCUMULATING epilogue
    X' = dropout(relu(BN(Y)))                       hidden layers; column statistics + the fused pass of dense_rows.cu
backward:
    dM = dY W_l ;  dX = dY W_r + A_mean^T dM        (SpMM on the cached 1/deg-weighted CSC view, GEMM accumulating on top)
    dW_l = dY^T M, dW_r = dY^T X, db_l = colsum dY  split-K tcgen05 weight-gradient GEMMs where the tiling allows
    Adam over one flat parameter buffer.

No autograd tape, no torch BatchNorm / Adam, no cuBLAS on the step where the tensor-core tilings apply (round 1 ran SAGE
through the module path: 25 % of its step was torch BN/elementwise and 12 % cuBLAS fallbacks).  ``train_step(..., aux=)`` adds
an auxiliary distillation loss on ``out_feat`` as every engine.StudentTrainer does (kd + beta*aux; configs[2] = G-CRD).
Parameters use nn.Linear's [out, in] layout and the reference module's state_dict keys (convs.i.lin_l.weight / .bias,
convs.i.lin_r.weight, bns.i.*).
"""
from __future__ import annotations

import math
from typing import List, Optional, Tuple

import torch

from . import lib, ops
from .engine import StudentTrainer
from .sparse import CsrGraph, SparseTensor


class SAGEStudentTrainer(StudentTrainer):
    views = ("Wl", "bl", "Wr", "gamma", "beta")

    def __init__(self, adj: SparseTensor, dims: List[int], dropout: float = 0.5, lr: float = 0.01, seed: int = 0,
                 alpha: float = 0.9, kd_T: float = 4.0, bn_eps: float = 1e-5, bn_momentum: float = 0.1,
                 fuse_row_passes: bool = True):
        assert adj.is_cuda(), "the engine runs on a CUDA device"
        for d in dims:
            assert d % 4 == 0 and d <= 1024, "layer widths must be multiples of 4 (128-bit rows)"
        st = adj.set_value(None).storage                      # SAGEConv drops edge values (A.3)
        self.G: CsrGraph = st.engine_csr_unweighted()         # mean over in-neighbours
        self.Gt: CsrGraph = st.engine_csc("mean")             # transpose with 1/deg(dst) weights: the mean's backward
        self.nnz = self.G.nnz
        super().__init__(adj.device, dims, adj.size(0), dropout, lr, seed, alpha, kd_T, bn_eps, bn_momentum)
        dev, N, L = self.device, self.N, self.L
        buf = lambda k: torch.zeros(N, k, device=dev)
        self.M = [buf(dims[l]) for l in range(L)]                 # mean-aggregated input of layer l
        self.Y = [buf(dims[l + 1]) for l in range(L)]
        self.A = [buf(dims[l + 1]) for l in range(L - 1)]
        self.dY = [buf(dims[l + 1]) for l in range(L)]
        self.dM = [buf(dims[l]) for l in range(L)]
        self.dA = [buf(dims[l + 1]) for l in range(L - 1)]
        self.bn = [torch.empty(4, dims[l + 1], device=dev) for l in range(L - 1)]
        # BatchNorm statistics / backward reductions taken in GEMM epilogues (engine.py, SURVEY §8 f1)
        self._gemm_part = {k: torch.empty(ops.gemm_stat_slots(N, k), 2, k, device=dev)
                           for k in set(self.dims[1:-1]) if fuse_row_passes and ops.gemm_stats_supported(k)}
        self.split = {}
        self.wgrad_ws = self._wgrad_workspace()

    # ------------------------------------------------------------------ parameters
    @staticmethod
    def param_table(dims: List[int]) -> List[Tuple[str, Tuple[int, ...], str]]:
        """Keys of the reference's SAGE module: per layer convs.i.lin_l.weight [out,in] (nn.Linear's layout) and bias,
        convs.i.lin_r.weight [out,in]; per hidden layer bns.i.weight / bias."""
        table = []
        for l in range(len(dims) - 1):
            w = (dims[l + 1], dims[l])
            table += [(f"convs.{l}.lin_l.weight", w, "Wl"), (f"convs.{l}.lin_l.bias", (dims[l + 1],), "bl"),
                      (f"convs.{l}.lin_r.weight", w, "Wr")]
            if l < len(dims) - 2:
                table += StudentTrainer._bn_table(l, dims[l + 1])
        return table

    def _init_weights(self, g: torch.Generator):
        """nn.Linear.reset_parameters: kaiming-uniform(a=sqrt 5) => U(+-1/sqrt(fan_in)) for weight and bias."""
        for l in range(self.L):
            bound = 1.0 / math.sqrt(self.dims[l])
            self.Wl[l].copy_((torch.rand(self.dims[l + 1], self.dims[l], generator=g) * 2 - 1) * bound)
            self.bl[l].copy_((torch.rand(self.dims[l + 1], generator=g) * 2 - 1) * bound)
            self.Wr[l].copy_((torch.rand(self.dims[l + 1], self.dims[l], generator=g) * 2 - 1) * bound)

    # ------------------------------------------------------------------ helpers
    def _split(self, w: torch.Tensor, transpose: bool, key: str):
        shape = (w.shape[1], w.shape[0]) if transpose else tuple(w.shape)
        if key not in self.split:
            self.split[key] = (torch.empty(shape, device=self.device), torch.empty(shape, device=self.device))
        hi, lo = self.split[key]
        return ops.split_tf32(w, transpose=transpose, hi=hi, lo=lo)

    def _wgrad(self, x, g, out_t: torch.Tensor, key: str):
        """out_t [n_out, n_in] = (x^T g)^T = g^T x: the tensor-core kernel produces x^T g [n_in, n_out]; nn.Linear keeps [out,in]."""
        k_in, n_out = x.shape[1], g.shape[1]
        if key not in self._static:
            self._static[key] = torch.empty(k_in, n_out, device=self.device)
        tmp = self._static[key]
        if ops.wgrad_supported(k_in, n_out):
            ops.gemm_wgrad_tf32x3(x, g, out=tmp, workspace=self.wgrad_ws)
        else:
            torch.mm(x.t(), g, out=tmp)
        lib.check(lib.load().b200gnn_transpose_f32(lib.dptr(tmp, torch.float32, "tmp"), k_in, n_out,
                                                   lib.dptr(out_t, torch.float32, "out"), lib.stream_ptr()), "transpose_f32")

    # ------------------------------------------------------------------ forward / backward
    def forward(self, x: torch.Tensor, training: bool = True) -> torch.Tensor:
        inp = x
        for l in range(self.L):
            k = self.dims[l + 1]
            ops.spmm_csr(self.G, inp, "mean", out=self.M[l])
            hi, lo = self._split(self.Wl[l], False, f"wl{l}")            # GEMM wants B as [N_out, K]: nn.Linear's own layout
            ops.gemm_tf32x3(self.M[l], hi, lo, bias=self.bl[l], out=self.Y[l])
            hi, lo = self._split(self.Wr[l], False, f"wr{l}")
            gp = self._gemm_part.get(k) if (training and l < self.L - 1) else None
            if gp is not None:                       # BatchNorm statistics of the layer output from this GEMM's epilogue
                ops.gemm_tf32x3_stats(inp, hi, lo, None, self.Y[l], gp, accumulate=True)
            else:
                ops.gemm_tf32x3(inp, hi, lo, out=self.Y[l], accumulate=True)
            if l == self.L - 1:
                break
            if training:
                part = gp if gp is not None else ops.col_stats(self.Y[l], partial=self._part(k))
                ops.bn_finalize(part, self.N, self.gamma[l], self.beta[l], self.bn_eps, self.bn_momentum, self.running_mean[l],
                                self.running_var[l], out=self.bn[l])
                ops.affine_relu_dropout(self.Y[l], self.bn[l][2], self.bn[l][3], True, self.p, self.seed, l, out=self.A[l],
                                        step_dev=self.step_count, step_mul=self.L)
            else:
                ops.affine_relu_dropout(self.Y[l], *self._bn_eval(l), True, 0.0, out=self.A[l])
            inp = self.A[l]
        return self.Y[-1]

    def backward(self, x: torch.Tensor, d_out_feat: Optional[torch.Tensor] = None):
        for l in range(self.L - 1, -1, -1):
            k = self.dims[l + 1]
            inp = x if l == 0 else self.A[l - 1]
            ops.col_sum(self.dY[l], out=self.gbl[l], partial=self._part(k))
            self._wgrad(self.M[l], self.dY[l], self.gWl[l], f"wg{self.dims[l]}x{k}")
            self._wgrad(inp, self.dY[l], self.gWr[l], f"wg{self.dims[l]}x{k}")
            if l == 0:
                break
            # dM = dY W_l ; dX = dY W_r + A_mean^T dM (+ the auxiliary loss's gradient on out_feat)
            hi, lo = self._split(self.Wl[l], True, f"wlT{l}")
            ops.gemm_tf32x3(self.dY[l], hi, lo, out=self.dM[l])
            d_prev = self.dA[l - 1]
            ops.spmm_csr(self.Gt, self.dM[l], "sum", out=d_prev)
            if d_out_feat is not None and l == self.L - 1:
                d_prev.add_(d_out_feat)
            hi, lo = self._split(self.Wr[l], True, f"wrT{l}")
            kp = self.dims[l]
            gp = self._gemm_part.get(kp)
            if gp is not None:
                # the last contribution to dOut is an accumulating GEMM: its epilogue masks, stores dz and reduces the BatchNorm
                # backward column sums (pass 1 of the block's backward)
                ops.gemm_tf32x3_bnbwd(self.dY[l], hi, lo, d_prev, self.A[l - 1], self.Y[l - 1], self.bn[l - 1][0], self.bn[l - 1][1],
                                      self.p, gp, accumulate=True)
                ops.bn_act_bwd_apply(d_prev, None, self.Y[l - 1], self.bn[l - 1][0], self.bn[l - 1][1], self.gamma[l - 1], gp,
                                     self.N, self.p, self.dY[l - 1], self.ggamma[l - 1], self.gbeta[l - 1], None, self._part(kp),
                                     self._coef(kp))
                continue
            ops.gemm_tf32x3(self.dY[l], hi, lo, out=d_prev, accumulate=True)
            ops.bn_act_bwd(d_prev, self.A[l - 1], self.Y[l - 1], self.bn[l - 1][0], self.bn[l - 1][1], self.gamma[l - 1], self.p,
                           d_y=self.dY[l - 1], d_gamma=self.ggamma[l - 1], d_beta=self.gbeta[l - 1], partial=self._part(kp),
                           coef=self._coef(kp), want_dbias=False)
