"""Node-parallel full-batch training across P GPUs (SURVEY.md §8e; BASELINE.json north_star).

The reference is single-GPU (one process per `--device`, arxiv_pyg/scripts/run_gcn.sh:24-28); this is the
B200-native extension the north star asks for, and its correctness target is equality with the 1-GPU step.

Partition
    Nodes are relabelled by a degree-balancing permutation (sort by degree, deal out in snake order) so that P
    contiguous, equally sized row blocks carry the same number of non-zeros and rows — hubs spread over the ranks
    instead of piling up on rank 0.  Rank p owns rows [p*B, (p+1)*B) of the relabelled Â, the activations and the
    labels of those nodes.  N is padded to P*B with isolated nodes.  Weights, BatchNorm affine parameters and Adam
    state are replicated.
Exchange (one per aggregation, over NVLink through NCCL)
    Y_p = Â[p,:] · H needs every row of H, so each aggregation is preceded by an all-gather of the local
    [B, K] block into a [P*B, K] buffer.  On a graph without locality (the synthetic ARXIV-shape: src uniform)
    every rank references ~all rows, so gathering whole blocks moves fewer bytes than pulling rows on demand
    (each remote row would be fetched once per referencing edge: ~1.8x the block size at P=8).
    Backward uses the symmetry of Â: dH_p = Â[p,:] · dY (all-gather of dY), no reduce-scatter.
    With aggregate-first layer 0 the input features are replicated and need no exchange at all, so a 3-layer
    GCN step performs 4 all-gathers: [N,256] and [N,40] forward, [N,40] and [N,256] backward.
Reductions
    BatchNorm statistics (forward and backward), the three loss scalars and the flat gradient buffer are
    all-reduced (sum); everything else is local.  Results match the 1-GPU engine up to fp32 reassociation.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List, Optional

import torch
import torch.distributed as dist

from . import lib, ops
from .engine import GCNStudentTrainer, gcn_norm, _is_symmetric
from .sparse import SparseTensor, csr_graph_from


import os as _os
_DIAG_SKIP_COMM = _os.environ.get("B200GNN_DIAG_SKIP_ALLGATHER", "0") == "1"


@dataclass
class ShardPlan:
    """Host-side description of the partition (device-agnostic: also exercised on CPU with gloo)."""
    world: int
    n: int                 # real nodes
    block: int             # rows per rank (B)
    perm: torch.Tensor     # new id -> old id, length n
    inv: torch.Tensor      # old id -> new id, length n

    @property
    def n_pad(self) -> int:
        return self.world * self.block

    def real_rows(self, rank: int) -> int:
        """Real (non-padding) nodes of a rank; they occupy the first slots of its block."""
        full_rounds, rem = divmod(self.n, self.world)
        if rem == 0:
            return full_rounds
        last_round = full_rounds                      # index of the partial round
        k_of_rank = rank if last_round % 2 == 0 else self.world - 1 - rank
        return full_rounds + (1 if k_of_rank < rem else 0)

    def rows_of(self, rank: int):
        return rank * self.block, rank * self.block + self.real_rows(rank)


def make_plan(rowcount: torch.Tensor, world: int) -> ShardPlan:
    """Degree-balancing relabelling: nodes sorted by degree (desc, stable) are dealt to ranks in snake order; each rank's
    nodes then occupy one contiguous block of new ids."""
    n = rowcount.numel()
    block = -(-n // world)
    order = torch.argsort(rowcount.cpu(), descending=True, stable=True)          # old ids, heaviest first
    pos = torch.arange(n)
    rnd, k = pos // world, pos % world
    rank_of = torch.where(rnd % 2 == 0, k, world - 1 - k)                         # snake
    slot = rnd                                                                   # position inside the rank's block
    new_id = rank_of * block + slot
    inv = torch.empty(n, dtype=torch.long)
    inv[order] = new_id
    # ranks may hold fewer than `block` real nodes: the tail ids of a block are padding (isolated, zero features)
    perm = torch.full((world * block,), -1, dtype=torch.long)
    perm[new_id] = order
    return ShardPlan(world, n, block, perm, inv)


def relabel_adjacency(adj: SparseTensor, plan: ShardPlan) -> SparseTensor:
    """P Â Pᵀ on the padded index space (values carried along)."""
    row, col, val = adj.coo()
    inv = plan.inv.to(row.device)
    return SparseTensor(row=inv[row], col=inv[col], value=val, sparse_sizes=(plan.n_pad, plan.n_pad), is_sorted=False)


def shard_rows(adj_relabelled: SparseTensor, plan: ShardPlan, rank: int):
    """(rowptr, col, val) of the real rows of `rank` — a rectangular n_real x n_pad CSR block."""
    rowptr, col, val = adj_relabelled.csr()
    r0, r1 = plan.rows_of(rank)
    e0, e1 = int(rowptr[r0]), int(rowptr[r1])
    return (rowptr[r0:r1 + 1] - e0).contiguous(), col[e0:e1].contiguous(), None if val is None else val[e0:e1].contiguous()


def scatter_rows(t: torch.Tensor, plan: ShardPlan, fill=0) -> torch.Tensor:
    """[n, ...] in original node order -> [n_pad, ...] in relabelled order (padding rows = fill)."""
    out = torch.full((plan.n_pad,) + tuple(t.shape[1:]), fill, dtype=t.dtype, device=t.device)
    out[plan.inv.to(t.device)] = t
    return out


class ShardedGCNTrainer(GCNStudentTrainer):
    """One rank of the node-parallel GCN student; same step semantics as GCNStudentTrainer."""

    aux_loss_supported = False       # out_feat's gradient would need its own route through the row shards

    def __init__(self, adj: SparseTensor, dims: List[int], group=None, **kw):
        assert dist.is_initialized(), "torch.distributed must be initialised (backend nccl)"
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.n_global = adj.size(0)
        super().__init__(adj, dims, **kw)
        dev = self.device
        self.full = {k: torch.empty(self.plan.n_pad, k, device=dev) for k in set(dims[1:])}   # all-gather targets
        self.sum_buf = {k: torch.empty(2, k, device=dev) for k in set(dims[1:])}
        self.row0 = self.rank * self.plan.block

    def _prepare_graph(self, adj: SparseTensor):
        """This rank's rows of the relabelled Â (forward and, Â being symmetric, backward); buffers of the common block size."""
        norm = gcn_norm(adj)
        if not _is_symmetric(norm):
            raise NotImplementedError("node-parallel backward relies on a symmetric normalised adjacency")
        self.plan = make_plan(norm.storage.rowcount(), self.world)
        rel = relabel_adjacency(norm, self.plan)
        rowptr, col, val = shard_rows(rel, self.plan, self.rank)
        shard = csr_graph_from(rowptr, col, val, self.plan.real_rows(self.rank), self.plan.n_pad)
        return shard, shard, self.plan.block

    # -- data placement helpers (original node order -> this rank's block)
    def shard_inputs(self, x, y, train_idx, teacher_logits=None):
        """Replicated padded features (aggregate-first layer 0 gathers from all nodes) + this rank's labels,
        teacher logits and local training rows."""
        plan, dev = self.plan, self.device
        r0, r1 = plan.rows_of(self.rank)
        x_pad = scatter_rows(x.to(dev), plan)
        y_loc = scatter_rows(y.to(dev), plan)[r0:r1].contiguous()
        t_loc = None if teacher_logits is None else scatter_rows(teacher_logits.to(dev), plan)[r0:r1].contiguous()
        new_train = plan.inv.to(dev)[train_idx.to(dev)]
        mine = new_train[(new_train >= r0) & (new_train < r1)] - r0
        self.n_train_global = int(train_idx.numel())
        return x_pad, y_loc, torch.sort(mine).values.contiguous(), t_loc

    def _block_of(self, view: torch.Tensor) -> torch.Tensor:
        """The [block, k] allocation behind a [:N] activation view (padding rows stay zero)."""
        for blk in self._blocks:
            if blk.data_ptr() == view.data_ptr() and blk.shape[1] == view.shape[1]:
                return blk
        raise KeyError("not an engine activation buffer")

    def gather_rows(self, local: torch.Tensor) -> torch.Tensor:
        """local rows of every rank -> [n, k] in ORIGINAL node order (for evaluation / tests)."""
        blk = torch.zeros(self.plan.block, local.shape[1], device=local.device)
        blk[:local.shape[0]] = local
        full = torch.empty(self.plan.n_pad, local.shape[1], device=local.device)
        dist.all_gather_into_tensor(full, blk, group=self.group)
        return full[self.plan.inv.to(local.device)]

    # -- collectives
    def _all_gather(self, local: torch.Tensor) -> torch.Tensor:
        full = self.full[local.shape[1]]
        if _DIAG_SKIP_COMM:            # timing diagnostics only (results are wrong): isolates the compute per rank
            return full
        dist.all_gather_into_tensor(full, self._block_of(local), group=self.group)
        return full

    def _global_stats(self, partial: torch.Tensor, k: int) -> torch.Tensor:
        s = ops.partial_reduce(partial, out=self.sum_buf[k])
        dist.all_reduce(s, group=self.group)
        return s.view(1, 2, k)

    # -- forward / backward with exchanges
    def forward(self, x_pad: torch.Tensor, training: bool = True) -> torch.Tensor:
        r0 = self.row0
        inp = None
        for l in range(self.L):
            last = l == self.L - 1
            k = self.dims[l + 1]
            if l == 0 and self.agg_first:
                ops.spmm_csr(self.G, x_pad, "sum", out=self.AX)
                self._linear(0, self.AX, self.Y[0], bias=self.b[0])
                part = ops.col_stats(self.Y[0], partial=self._part(k)) if training else None
            else:
                src = x_pad[r0:r0 + self.N] if l == 0 else inp
                self._linear(l, src, self.H[l])
                full = self._all_gather(self.H[l])
                if last or not training:
                    ops.spmm_csr(self.G, full, "sum", bias=self.b[l], out=self.Y[l]); part = None
                else:
                    part = self.stat_part[l]
                    ops.spmm_csr(self.G, full, "sum", bias=self.b[l], out=self.Y[l], stat_partial=part)
            if last:
                break
            if training:
                sums = self._global_stats(part, k)
                ops.bn_finalize(sums, self.n_global, self.gamma[l], self.beta[l], self.bn_eps, self.bn_momentum,
                                self.running_mean[l], self.running_var[l], out=self.bn[l])
                ops.affine_relu_dropout(self.Y[l], self.bn[l][2], self.bn[l][3], True, self.p, self.seed, l, out=self.A[l],
                                        step_dev=self.step_count, step_mul=self.L, row_offset=r0)
            else:
                ops.affine_relu_dropout(self.Y[l], *self._bn_eval(l), True, 0.0, out=self.A[l])
            inp = self.A[l]
        return self.Y[-1]

    def backward(self, x_pad: torch.Tensor):
        r0 = self.row0
        for l in range(self.L - 1, -1, -1):
            k_out = self.dims[l + 1]
            inp = x_pad[r0:r0 + self.N] if l == 0 else self.A[l - 1]
            if l == self.L - 1:
                ops.col_sum(self.dY[l], out=self.gb[l], partial=self._part(k_out))
            if l == 0 and self.agg_first:
                self._wgrad_async(0, self.AX, self.dY[0])
                continue
            full = self._all_gather(self.dY[l])
            ops.spmm_csr(self.G, full, "sum", out=self.dH[l])        # Â symmetric: dH_p = Â[p,:] dY
            if l > 0:
                self._linear_dgrad(l, self.dH[l], self.dA[l - 1])
            self._wgrad_async(l, inp, self.dH[l])                    # side stream: hides under BN backward + the next all-gather
            if l > 0:
                k = self.dims[l]
                part, bn = self._part(k), self.bn[l - 1]
                ops.bn_act_bwd_reduce(self.dA[l - 1], self.A[l - 1], self.Y[l - 1], bn[0], bn[1], self.p, part)
                sums = self._global_stats(part, k)
                ops.bn_act_bwd_apply(self.dA[l - 1], self.A[l - 1], self.Y[l - 1], bn[0], bn[1], self.gamma[l - 1], sums,
                                     self.n_global, self.p, self.dY[l - 1], self.ggamma[l - 1], self.gbeta[l - 1],
                                     self.gb[l - 1], part, self._coef(k))
                if self.rank != 0:      # dgamma/dbeta come from GLOBAL sums: count them once in the all-reduce below
                    self.ggamma[l - 1].zero_(); self.gbeta[l - 1].zero_()
        self._wgrad_join()

    def _reduce_grads(self):
        dist.all_reduce(self._grads_buf, group=self.group)      # gradients + the three loss scalars

    def exchange_bytes_per_step(self) -> int:
        """Bytes each rank RECEIVES over NVLink per step in the all-gathers (the data-path collectives)."""
        per = 0
        for l in range(self.L):
            if l == 0 and self.agg_first:
                continue
            per += 2 * self.plan.n_pad * self.dims[l + 1] * 4
        return per * (self.world - 1) // self.world
