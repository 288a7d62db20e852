"""Fused full-batch training step for the GCN student (+ logit-KD) — BASELINE.json configs[1].

Mirrors what one call of the reference's ``train()`` does for ``--gnn gcn --training kd|supervised``
(arxiv_pyg/gnn.py:102-195 with ``GCN.forward`` :45-53, ``kd_criterion`` criterion.py:8-21, Adam :308-315):

    for each layer:  H = X W            (dense GEMM; cuBLAS fp32 through torch.mm — a plain library GEMM)
                     Y = Â H + b        (b200gnn SpMM, bias + BatchNorm statistics fused in the epilogue)
                     X = dropout(relu(BN(Y)))   (one b200gnn pass)
    loss, dlogits = fused CE/KD row kernel over logits[train_idx]
    backward: dH = Âᵀ dY (same SpMM kernel), dW = Xᵀ dH, dX = dH Wᵀ, fused BN/ReLU/dropout backward
    Adam over one flat parameter buffer.

No autograd tape: activations live in preallocated buffers and the whole step (≈40 launches) is captured
into one CUDA graph.  Everything except the three GEMM shapes is hand-written sm_100a code behind the C ABI.

``StudentTrainer`` is the part of the step that does not depend on the model; the GCN engine here, the GraphSAGE engine
(engine_sage.py) and the multi-GPU GCN engines (hybrid.py, dist.py) derive from it.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import torch

from . import lib, ops
from .sparse import CsrGraph, SparseTensor


def gcn_norm(adj: SparseTensor) -> SparseTensor:
    """PyG gcn_norm for a SparseTensor (SURVEY Appendix A.2): Â = D^-1/2 (A + I) D^-1/2, A value-less => ones."""
    if not adj.has_value():
        adj = adj.fill_value(1.0)
    adj = adj.fill_diag(1.0)
    deg = adj.sum(dim=1)
    dis = deg.pow(-0.5)
    dis.masked_fill_(dis == float("inf"), 0.0)
    row, col, val = adj.coo()
    return adj.set_value(dis[row] * val * dis[col])


def _is_symmetric(adj: SparseTensor) -> bool:
    st = adj.storage
    if st.sparse_sizes()[0] != st.sparse_sizes()[1]:
        return False
    perm = st.csr2csc()
    same = torch.equal(st.col()[perm], st.row()) and torch.equal(st.row()[perm], st.col())
    if same and st.value() is not None:
        same = torch.equal(st.value()[perm], st.value())
    return bool(same)


class StudentTrainer:
    """What the fused student engines share: one flat parameter / gradient / Adam buffer laid out by the engine's parameter
    table, the BatchNorm running statistics, reduction scratch, and the step itself (forward, fused KD loss, backward,
    cross-rank gradient reduction, Adam), eager or replayed from a CUDA graph.

    A subclass defines ``views``, ``param_table``, ``_init_weights``, ``forward`` and ``backward``, and calls
    ``StudentTrainer.__init__`` once it knows how many rows its activations have."""

    views: Tuple[str, ...] = ()    # names of the per-layer view lists; the gradient of self.<v>[l] is self.g<v>[l]
    # training rows over all ranks, the KD loss's normaliser (the multi-GPU engines' shard_inputs set it); 0 = the local rows
    n_train_global = 0
    # train_step(aux=) feeds d aux / d out_feat into backward; the multi-GPU engines do not carry that gradient
    aux_loss_supported = True

    def __init__(self, device: torch.device, dims: List[int], n_rows: int, dropout: float, lr: float, seed: int,
                 alpha: float, kd_T: float, bn_eps: float, bn_momentum: float):
        self.device = dev = device
        self.dims, self.L = list(dims), len(dims) - 1
        self.p, self.lr, self.alpha, self.kd_T = float(dropout), float(lr), float(alpha), float(kd_T)
        self.bn_eps, self.bn_momentum, self.seed = bn_eps, bn_momentum, int(seed)
        self.N = n_rows
        layout = self.param_layout(self.dims)
        n_par = sum(math.prod(shape) for _, shape, _ in layout.values())
        self.params = torch.zeros(n_par, device=dev)
        # gradients and the three loss scalars share one buffer (padded to 16 bytes): the multi-GPU engines exchange and
        # reduce both with a single launch
        self.n_par_pad = (n_par + 3) // 4 * 4
        self._grads_buf = torch.zeros(self.n_par_pad + 4, device=dev)
        self.grads = self._grads_buf[:n_par]
        self.loss_out = self._grads_buf[self.n_par_pad:self.n_par_pad + 3]
        self.exp_avg = torch.zeros(n_par, device=dev)
        self.exp_avg_sq = torch.zeros(n_par, device=dev)
        self.step_count = torch.zeros(1, dtype=torch.int32, device=dev)
        for v in self.views:
            setattr(self, v, []); setattr(self, "g" + v, [])
        self._param: Dict[str, torch.Tensor] = {}
        for key, (off, shape, v) in layout.items():
            n = math.prod(shape)
            self._param[key] = self.params[off:off + n].view(shape)
            getattr(self, v).append(self._param[key])
            getattr(self, "g" + v).append(self.grads[off:off + n].view(shape))
        self.running_mean = [torch.zeros(d, device=dev) for d in self.dims[1:-1]]
        self.running_var = [torch.ones(d, device=dev) for d in self.dims[1:-1]]
        self.rs = ops.rows_slots(n_rows)
        self.kd_part = torch.empty(2 * int(lib.load().b200gnn_kd_partials(n_rows)), device=dev)
        self._static: Dict[str, torch.Tensor] = {}
        for k in set(self.dims[1:]):
            self._part(k); self._coef(k)
        self._graph: Dict[int, torch.cuda.CUDAGraph] = {}
        self.loss_aux = None
        self.reset_parameters(seed)

    # ------------------------------------------------------------------ parameters
    @staticmethod
    def param_table(dims: List[int]) -> List[Tuple[str, Tuple[int, ...], str]]:
        """(state-dict key, shape, view list) of every parameter, in the order they are packed into the flat buffers."""
        raise NotImplementedError

    @staticmethod
    def _bn_table(l: int, k: int) -> List[Tuple[str, Tuple[int, ...], str]]:
        return [(f"bns.{l}.weight", (k,), "gamma"), (f"bns.{l}.bias", (k,), "beta")]

    @classmethod
    def param_layout(cls, dims: List[int]) -> Dict[str, Tuple[int, Tuple[int, ...], str]]:
        """state-dict key -> (offset into the flat buffers, shape, view list).  The offsets must stay put: the multi-GPU
        engines exchange the gradient buffer by position and the Adam state is positional."""
        layout, off = {}, 0
        for key, shape, v in cls.param_table(dims):
            layout[key] = (off, shape, v)
            off += math.prod(shape)
        return layout

    def _init_weights(self, g: torch.Generator):
        raise NotImplementedError

    def reset_parameters(self, seed: int = 0):
        """The model's weight initialisation (its own generator order), BatchNorm1d ones / zeros, a fresh Adam."""
        self._init_weights(torch.Generator().manual_seed(seed))
        for l in range(self.L - 1):
            self.gamma[l].fill_(1.0); self.beta[l].zero_()
            self.running_mean[l].zero_(); self.running_var[l].fill_(1.0)
        self.exp_avg.zero_(); self.exp_avg_sq.zero_(); self.step_count.zero_()

    def state_dict(self) -> Dict[str, torch.Tensor]:
        """The reference module's keys: the parameter table's and bns.i.running_mean / running_var."""
        sd = {key: v.detach().clone() for key, v in self._param.items()}
        for l in range(self.L - 1):
            sd[f"bns.{l}.running_mean"] = self.running_mean[l].clone()
            sd[f"bns.{l}.running_var"] = self.running_var[l].clone()
        return sd

    def load_state_dict(self, sd: Dict[str, torch.Tensor]):
        for key, v in self._param.items():
            v.copy_(sd[key])
        for l in range(self.L - 1):
            if f"bns.{l}.running_mean" in sd:
                self.running_mean[l].copy_(sd[f"bns.{l}.running_mean"]); self.running_var[l].copy_(sd[f"bns.{l}.running_var"])

    # ------------------------------------------------------------------ helpers
    def out_feat(self) -> torch.Tensor:
        """The reference's ``model.out_feat`` (arxiv_pyg/gnn.py:51): output of the last hidden layer."""
        return self.A[-1]

    def dropout_offset(self, layer: int, step: int) -> int:
        return layer + step * self.L

    def _bn_eval(self, l: int, cols: slice = slice(None)):
        """Eval-mode BatchNorm of hidden layer l (its columns ``cols``) as y * scale + shift from the running statistics."""
        scale = self.gamma[l][cols] * torch.rsqrt(self.running_var[l][cols] + self.bn_eps)
        shift = self.beta[l][cols] - self.running_mean[l][cols] * scale
        return scale, shift

    def _wgrad_workspace(self) -> Optional[torch.Tensor]:
        """Split-K workspace shared by every layer whose weight gradient the tensor-core kernel can tile (None if none)."""
        floats = [lib.load().b200gnn_wgrad_workspace_floats(k_in, n_out) for k_in, n_out in zip(self.dims, self.dims[1:])
                  if ops.wgrad_supported(k_in, n_out)]
        return torch.empty(max(floats), device=self.device) if floats else None

    def _part(self, k: int) -> torch.Tensor:
        key = f"part{k}"
        if key not in self._static:
            self._static[key] = torch.empty(self.rs, 2, k, device=self.device)
        return self._static[key]

    def _coef(self, k: int) -> torch.Tensor:
        key = f"coef{k}"
        if key not in self._static:
            self._static[key] = torch.empty(3, k, device=self.device)
        return self._static[key]

    # ------------------------------------------------------------------ step
    def _reduce_grads(self):
        """Sums the gradient buffer (with the loss scalars behind it) over ranks; one GPU has nothing to sum."""

    def _step_impl(self, x, y, train_idx, teacher_logits, aux=None, beta: float = 1.0):
        logits = self.forward(x, training=True)
        self.dY[-1].zero_()
        ops.kd_loss_fwd_bwd(logits, y, train_idx, teacher_logits, self.alpha, self.kd_T, d_logits=self.dY[-1],
                            loss_out=self.loss_out, partial=self.kd_part, n_norm=self.n_train_global)
        if aux is None:
            self.backward(x)
        else:
            feat = self.out_feat().detach().requires_grad_(True)
            with torch.enable_grad():
                loss_aux = aux(feat)
                (loss_aux * beta).backward()
            self.loss_aux = loss_aux.detach()
            d_feat = feat.grad if feat.grad is not None else torch.zeros_like(feat)
            self.backward(x, d_out_feat=d_feat.contiguous())
        self._reduce_grads()
        ops.adam_step(self.params, self.grads, self.exp_avg, self.exp_avg_sq, self.step_count, self.lr)

    def train_step(self, x, y, train_idx, teacher_logits=None, aux=None, beta: float = 1.0) -> torch.Tensor:
        """One reference ``train()`` call: kd if teacher_logits is given, else supervised (arxiv_pyg/gnn.py:102-195), and
        with ``aux`` the kd + beta*aux form of gnn_kd_and_aux.py:100-189 — ``aux(out_feat)`` receives the [N, H] output
        of the last hidden layer (the reference's ``model.out_feat``, requires_grad) and returns the auxiliary loss, e.g.
        ``lambda f: criterion.lpw_criterion(z, y, f[idx], t_feat[idx], edge_index, "cosine", 1)[2]`` or a projection head +
        ``nce_criterion``; parameters of such heads get their gradients through torch autograd and stay with the caller's
        optimizer.  Returns the device tensor [loss, loss_cls, loss_kd] (+ beta*aux folded into loss); no host sync."""
        if aux is not None and not self.aux_loss_supported:
            raise NotImplementedError(f"{type(self).__name__} does not take an auxiliary loss (aux=)")
        self._step_impl(x, y, train_idx, teacher_logits, aux, beta)
        if aux is not None:
            self.loss_out[0].add_(self.loss_aux * beta)
        return self.loss_out

    # ------------------------------------------------------------------ CUDA graph
    def capture(self, x, y, train_idx, teacher_logits=None, warmup: int = 2, key: int = 0):
        """Capture the step on static input buffers; afterwards ``replay(key)`` runs one full step.
        Several input-buffer sets can be captured (key = 0, 1, ...) so that uploads of the next step's inputs overlap
        the current step (activations and parameters are shared between the graphs)."""
        self._static.update(x=x, y=y, train_idx=train_idx, teacher=teacher_logits)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(warmup):
                self._step_impl(x, y, train_idx, teacher_logits)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._step_impl(x, y, train_idx, teacher_logits)
        self._graph[key] = g
        return self

    def replay(self, key: int = 0) -> torch.Tensor:
        self._graph[key].replay()
        return self.loss_out

    def launches_per_step(self) -> int:
        """b200gnn kernel launches in one training step (counted, not estimated)."""
        before = lib.launch_count()
        st = self._static
        self._step_impl(st["x"], st["y"], st["train_idx"], st["teacher"])
        return lib.launch_count() - before


class GCNStudentTrainer(StudentTrainer):
    """State + fused step of an L-layer GCN student on one GPU."""

    views = ("W", "b", "gamma", "beta")

    def __init__(self, adj: SparseTensor, dims: List[int], dropout: float = 0.5, lr: float = 0.01, seed: int = 0,
                 alpha: float = 0.9, kd_T: float = 4.0, bn_eps: float = 1e-5, bn_momentum: float = 0.1,
                 aggregate_first: Optional[bool] = None, tensor_core_gemm: bool = True, overlap_wgrad: bool = True,
                 fuse_row_passes: bool = True):
        assert adj.is_cuda(), "the engine runs on a CUDA device"
        for d in dims[1:]:
            assert d % 4 == 0 and d <= 1024, "layer widths must be multiples of 4 (128-bit rows)"
        self.G, self.Gt, rows_alloc = self._prepare_graph(adj)
        self.nnz = self.G.nnz
        super().__init__(adj.device, dims, self.G.n_rows, dropout, lr, seed, alpha, kd_T, bn_eps, bn_momentum)
        dev, N, L = self.device, self.N, self.L
        self.tc_gemm = bool(tensor_core_gemm) and all(d % 4 == 0 for d in dims)
        # Layer 0 may aggregate BEFORE its GEMM: Â(XW) = (ÂX)W.  When the input is narrower than the hidden width
        # the gather runs at the narrow width, and because X needs no gradient the backward aggregation of layer 0
        # disappears altogether: dW0 = (ÂX)ᵀ dY0.  Same mathematics as the reference (PyG transforms first and
        # pays a 256-wide backward SpMM whose result is only used as an intermediate); fp32 reassociation only.
        self.agg_first = (dims[0] < dims[1] and dims[0] % 4 == 0) if aggregate_first is None else bool(aggregate_first)
        if L < 2:
            self.agg_first = False
        # tf32 hi/lo splits of the weights for the tcgen05 GEMM: W^T [out,in] feeds the forward (C = X W),
        # W [in,out] feeds the input gradient (dX = dH W^T); refreshed every step (a few KB).
        self.Wt_split = [(torch.empty(dims[l + 1], dims[l], device=dev), torch.empty(dims[l + 1], dims[l], device=dev))
                         for l in range(L)]
        self.W_split = [(torch.empty(dims[l], dims[l + 1], device=dev), torch.empty(dims[l], dims[l + 1], device=dev))
                        for l in range(L)]
        self.wgrad_ws = self._wgrad_workspace() if self.tc_gemm else None

        # ---- activations / gradients (preallocated; CUDA-graph friendly)
        self._blocks = []

        def buf(k):
            blk = torch.zeros(rows_alloc, k, device=dev)
            self._blocks.append(blk)
            return blk[:N]
        self.H = [buf(dims[l + 1]) for l in range(L)]            # X W
        self.Y = [buf(dims[l + 1]) for l in range(L)]            # Â H + b  (last = logits)
        self.A = [buf(dims[l + 1]) for l in range(L - 1)]        # dropout(relu(BN(Y)))
        self.dY = [buf(dims[l + 1]) for l in range(L)]
        self.dH = [buf(dims[l + 1]) for l in range(L)]
        self.dA = [buf(dims[l + 1]) for l in range(L - 1)]
        self.AX = buf(dims[0]) if self.agg_first else None         # Â X (layer 0, aggregate-first)
        slots_spmm = ops.stat_slots(self.G)
        self.stat_part = [torch.empty(slots_spmm, 2, dims[l + 1], device=dev) for l in range(L - 1)]
        self.bn = [torch.empty(4, dims[l + 1], device=dev) for l in range(L - 1)]   # mean, invstd, scale, shift
        # Row passes fused into GEMM epilogues (SURVEY §8 f1): the layer-0 BatchNorm statistics come out of the layer-0 GEMM
        # and pass 1 of every BatchNorm/ReLU/dropout backward out of the input-gradient GEMM that produces its dOut.
        self.fuse_rows = bool(fuse_row_passes) and self.tc_gemm
        self._gemm_part = {k: torch.empty(ops.gemm_stat_slots(N, k), 2, k, device=dev)
                           for k in set(dims[1:-1]) if self.fuse_rows and ops.gemm_stats_supported(k)}
        # weight gradients only feed Adam: they run on a side stream next to the BN/ReLU backward passes and the next
        # aggregation (parallel branches of the captured graph)
        self.overlap_wgrad = overlap_wgrad
        self._side = torch.cuda.Stream(device=dev) if overlap_wgrad else None
        self._ev_fork, self._ev_join = torch.cuda.Event(), torch.cuda.Event()

    def _prepare_graph(self, adj: SparseTensor) -> Tuple[CsrGraph, CsrGraph, int]:
        """(graph of the forward aggregation, graph of the backward aggregation, rows every activation buffer allocates).
        The multi-GPU engines return their rank's row shard here, with buffers over-allocated to the common block size."""
        norm = gcn_norm(adj)                     # cached=True semantics: normalise once (arxiv_pyg/gnn.py:28)
        G = norm.storage.engine_csr()
        Gt = G if _is_symmetric(norm) else norm.storage.engine_csc("value")
        return G, Gt, G.n_rows

    # ------------------------------------------------------------------ parameters
    @staticmethod
    def param_table(dims: List[int]) -> List[Tuple[str, Tuple[int, ...], str]]:
        """Keys of the reference's GCN module under PyG 1.x: per layer convs.i.weight [in,out] and bias, per hidden layer
        bns.i.weight / bias."""
        table = []
        for l in range(len(dims) - 1):
            table += [(f"convs.{l}.weight", (dims[l], dims[l + 1]), "W"), (f"convs.{l}.bias", (dims[l + 1],), "b")]
            if l < len(dims) - 2:
                table += StudentTrainer._bn_table(l, dims[l + 1])
        return table

    def _init_weights(self, g: torch.Generator):
        """GCNConv: glorot weight, zero bias (SURVEY A.2)."""
        for l in range(self.L):
            fan_in, fan_out = self.dims[l], self.dims[l + 1]
            a = math.sqrt(6.0 / (fan_in + fan_out))
            self.W[l].copy_((torch.rand(fan_in, fan_out, generator=g) * 2 - 1) * a)
            self.b[l].zero_()

    # ------------------------------------------------------------------ forward / backward
    def activation_pattern(self, l: int) -> torch.Tensor:
        """bool [N, dims[l+1]]: ReLU-active AND kept by dropout in the last training forward of hidden layer l."""
        return self.A[l] > 0

    def forward(self, x: torch.Tensor, training: bool = True) -> torch.Tensor:
        """Returns logits [N,C]; hidden activations stay in self.A (self.A[-1] is the reference's model.out_feat)."""
        inp = x
        for l in range(self.L):
            last = l == self.L - 1
            if l == 0 and self.agg_first:
                ops.spmm_csr(self.G, x, "sum", out=self.AX)
                if training:
                    gp = self._gemm_part.get(self.dims[1])
                    if gp is not None:                               # statistics of Y0 from the GEMM epilogue
                        hi, lo = ops.split_tf32(self.W[0], transpose=True, hi=self.Wt_split[0][0], lo=self.Wt_split[0][1])
                        ops.gemm_tf32x3_stats(self.AX, hi, lo, self.b[0], self.Y[0], gp)
                        part = gp
                    else:
                        self._linear(0, self.AX, self.Y[0], bias=self.b[0])
                        part = ops.col_stats(self.Y[0], partial=self._part(self.dims[1]))
                    ops.bn_finalize(part, self.N, self.gamma[0], self.beta[0], self.bn_eps,
                                    self.bn_momentum, self.running_mean[0], self.running_var[0], out=self.bn[0])
                    ops.affine_relu_dropout(self.Y[0], self.bn[0][2], self.bn[0][3], True, self.p, self.seed, 0,
                                            out=self.A[0], step_dev=self.step_count, step_mul=self.L)
                else:
                    self._linear(0, self.AX, self.Y[0], bias=self.b[0])
                    ops.affine_relu_dropout(self.Y[0], *self._bn_eval(0), True, 0.0, out=self.A[0])
                inp = self.A[0]
                continue
            self._linear(l, inp, self.H[l])
            if last:
                ops.spmm_csr(self.G, self.H[l], "sum", bias=self.b[l], out=self.Y[l])
            elif training:
                ops.spmm_csr(self.G, self.H[l], "sum", bias=self.b[l], out=self.Y[l], stat_partial=self.stat_part[l])
                ops.bn_finalize(self.stat_part[l], self.N, self.gamma[l], self.beta[l], self.bn_eps, self.bn_momentum,
                                self.running_mean[l], self.running_var[l], out=self.bn[l])
                ops.affine_relu_dropout(self.Y[l], self.bn[l][2], self.bn[l][3], True, self.p, self.seed, l,
                                        out=self.A[l], step_dev=self.step_count, step_mul=self.L)
                inp = self.A[l]
            else:
                ops.spmm_csr(self.G, self.H[l], "sum", bias=self.b[l], out=self.Y[l])
                ops.affine_relu_dropout(self.Y[l], *self._bn_eval(l), True, 0.0, out=self.A[l])
                inp = self.A[l]
        return self.Y[-1]

    def backward(self, x: torch.Tensor, d_out_feat: Optional[torch.Tensor] = None):
        """Consumes self.dY[-1] (d loss / d logits) and, for the auxiliary distillation losses, d loss / d out_feat
        ([N, H], added to the gradient arriving at the last hidden activation); fills self.grads."""
        for l in range(self.L - 1, -1, -1):
            inp = x if l == 0 else self.A[l - 1]
            if l == self.L - 1:
                ops.col_sum(self.dY[l], out=self.gb[l], partial=self._part(self.dims[l + 1]))
            if l == 0 and self.agg_first:
                self._wgrad_async(0, self.AX, self.dY[0])              # dW0 = (ÂX)ᵀ dY0, no backward aggregation
                continue
            ops.spmm_csr(self.Gt, self.dY[l], "sum", out=self.dH[l])
            d_prev = self.dA[l - 1] if l > 0 else None
            gp = self._gemm_part.get(self.dims[l]) if l > 0 else None
            if l > 0:
                acc = d_out_feat is not None and l == self.L - 1
                if acc:
                    # the auxiliary loss's gradient w.r.t. out_feat is the starting value the input-gradient GEMM adds to
                    d_prev = d_out_feat
                if gp is not None:
                    # dgrad GEMM whose epilogue masks by the ReLU/dropout pattern, stores dz and reduces the two BatchNorm
                    # backward column sums: pass 1 of the block's backward costs no sweep of its own
                    hi, lo = ops.split_tf32(self.W[l], transpose=False, hi=self.W_split[l][0], lo=self.W_split[l][1])
                    ops.gemm_tf32x3_bnbwd(self.dH[l], hi, lo, d_prev, self.A[l - 1], self.Y[l - 1], self.bn[l - 1][0],
                                          self.bn[l - 1][1], self.p, gp, accumulate=acc)
                else:
                    self._linear_dgrad(l, self.dH[l], d_prev, accumulate=acc)
            self._wgrad_async(l, inp, self.dH[l])                      # forks after the dgrad GEMM (both want the whole SM)
            if l > 0:
                k = self.dims[l]
                part = self._part(k)
                if gp is not None:
                    ops.bn_act_bwd_apply(d_prev, None, self.Y[l - 1], self.bn[l - 1][0], self.bn[l - 1][1], self.gamma[l - 1],
                                         gp, self.N, self.p, self.dY[l - 1], self.ggamma[l - 1], self.gbeta[l - 1],
                                         self.gb[l - 1], part, self._coef(k))
                else:
                    ops.bn_act_bwd(d_prev, self.A[l - 1], self.Y[l - 1], self.bn[l - 1][0], self.bn[l - 1][1],
                                   self.gamma[l - 1], self.p, d_y=self.dY[l - 1], d_gamma=self.ggamma[l - 1],
                                   d_beta=self.gbeta[l - 1], d_bias=self.gb[l - 1], partial=part, coef=self._coef(k))
        self._wgrad_join()

    def _wgrad_async(self, l: int, inp: torch.Tensor, d_out: torch.Tensor):
        """grad W_l on the side stream, ordered after everything enqueued so far on the current stream."""
        if self._side is None:
            return self._linear_wgrad(l, inp, d_out)
        self._ev_fork.record(torch.cuda.current_stream())
        self._side.wait_event(self._ev_fork)
        with torch.cuda.stream(self._side):
            self._linear_wgrad(l, inp, d_out)

    def _wgrad_join(self):
        if self._side is not None:
            self._ev_join.record(self._side)
            torch.cuda.current_stream().wait_event(self._ev_join)

    def _linear(self, l: int, inp: torch.Tensor, out: torch.Tensor, bias: Optional[torch.Tensor] = None):
        """out = inp @ W_l (+bias): tcgen05 3xTF32 kernel, or cuBLAS fp32 when disabled."""
        if self.tc_gemm:
            hi, lo = ops.split_tf32(self.W[l], transpose=True, hi=self.Wt_split[l][0], lo=self.Wt_split[l][1])
            ops.gemm_tf32x3(inp, hi, lo, bias=bias, out=out)
        elif bias is not None:
            torch.addmm(bias, inp, self.W[l], out=out)
        else:
            torch.mm(inp, self.W[l], out=out)

    def _linear_dgrad(self, l: int, d_out: torch.Tensor, d_inp: torch.Tensor, accumulate: bool = False):
        """d_inp (+)= d_out @ W_l^T."""
        if self.tc_gemm:
            hi, lo = ops.split_tf32(self.W[l], transpose=False, hi=self.W_split[l][0], lo=self.W_split[l][1])
            ops.gemm_tf32x3(d_out, hi, lo, out=d_inp, accumulate=accumulate)
        elif accumulate:
            d_inp.addmm_(d_out, self.W[l].t())
        else:
            torch.mm(d_out, self.W[l].t(), out=d_inp)

    def _linear_wgrad(self, l: int, inp: torch.Tensor, d_out: torch.Tensor):
        """grad W_l = inp^T @ d_out: split-K tcgen05 kernel where the tiling allows, cuBLAS fp32 otherwise."""
        if self.tc_gemm and ops.wgrad_supported(self.dims[l], self.dims[l + 1]):
            ops.gemm_wgrad_tf32x3(inp, d_out, out=self.gW[l], workspace=self.wgrad_ws)
        else:
            torch.mm(inp.t(), d_out, out=self.gW[l])

    # ------------------------------------------------------------------ accounting
    def aggregations_per_step(self) -> Dict[int, int]:
        """width -> number of SpMM launches of that width in one training step."""
        out: Dict[int, int] = {}
        for l in range(self.L):
            if l == 0 and self.agg_first:
                out[self.dims[0]] = out.get(self.dims[0], 0) + 1
            else:
                out[self.dims[l + 1]] = out.get(self.dims[l + 1], 0) + 2
        return out

    def spmm_algorithmic_bytes(self) -> Dict[int, int]:
        """Compulsory HBM bytes of one aggregation per feature width (SURVEY.md §8d):
        2*N*K*4 (read X, write Y) + nnz*(4 col + 4 val) + (N+1)*4."""
        return {k: 2 * self.N * k * 4 + self.nnz * 8 + (self.N + 1) * 4 for k in set(self.dims)}
