"""Hybrid-layout multi-GPU training step (SURVEY.md §8e; BASELINE.json north_star "up to 8 B200s").

Why not plain node parallelism.  Row-sharding Â makes every aggregation all-gather its whole [N, K] operand: on a graph
without locality each rank references ~all rows, so at P = 8 every rank RECEIVES 7/8 of two [N,256] tensors per step
(351 MB, >= 0.46 ms on NVLink) while its compute shrinks to ~0.3 ms — the round-1 engine scaled 0.58 / 0.35 / 0.15.

What this module does instead.  Dense work (GEMMs, loss, optimizer) stays NODE-parallel ("R layout": rank p owns the
rows of its node block, all K columns), but WIDE aggregations run FEATURE-parallel ("C layout": rank p owns columns
[p*K/P, (p+1)*K/P) of ALL nodes and multiplies them by the whole Â, which is 30 MB and replicated):

    R -> C :  H_R [n_p, K]  --exchange-->  H_C [N, K/P]        (each rank sends (P-1)/P of ITS block, split P ways)
    Y_C = Â · H_C                                               (no halo at all)
    BatchNorm statistics of Y_C are LOCAL (whole columns), so is BN/ReLU/dropout and its backward
    C -> R :  A_C [N, K/P]  --exchange-->  A_R [n_p, K]

An exchange moves N·K·4·(P-1)/P² bytes per rank (19 MB at P=8, K=256) instead of the all-gather's N·K·4·(P-1)/P
(152 MB): 8x less at P=8, and the per-layer BatchNorm all-reduces disappear.  Narrow aggregations (the 40 logits,
K % 4P != 0) keep the row-sharded form with an all-gather (27 MB in total).  The backward uses the symmetry of Â the
same way.  Nodes are relabelled by the degree-balancing permutation of dist.make_plan (dense: no padding rows), and
dropout decisions are taken by ORIGINAL node id and GLOBAL feature index (b200gnn_affine_relu_dropout_mapped_f32), so
the P-GPU step reproduces the 1-GPU step's masks and, up to fp32 reassociation, its loss and gradients.

Exchanges: `PeerExchange` — one b200gnn_peer_copy2d_f32 launch that stores this rank's blocks straight into the
consumers' arenas over NVLink (CUDA IPC mappings) plus a flag barrier (csrc/peer.cu; no collective library on the data
path, CUDA-graph capturable); `TorchExchange` — the same primitives on torch.distributed collectives (gloo for the CPU
tests of the host logic, NCCL as the baseline the peer path is measured against).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional

import torch
import torch.distributed as dist

from . import lib, ops
from .engine import GCNStudentTrainer, gcn_norm, _is_symmetric
from .sparse import SparseTensor, csr_graph_from


# ----------------------------------------------------------------------------------------------------- partition plan
@dataclass
class DensePlan:
    """Degree-balanced relabelling without padding: rank p owns new ids [offsets[p], offsets[p+1])."""
    world: int
    n: int
    counts: List[int]
    offsets: List[int]
    perm: torch.Tensor     # new id -> old id
    inv: torch.Tensor      # old id -> new id

    @property
    def block(self) -> int:
        return max(self.counts)

    def rows_of(self, rank: int):
        return self.offsets[rank], self.offsets[rank + 1]


def make_dense_plan(rowcount: torch.Tensor, world: int) -> DensePlan:
    """Nodes sorted by degree (desc, stable) are dealt to the ranks in snake order (as dist.make_plan), then packed:
    every rank gets n//world or n//world+1 nodes and, because hubs are dealt out first, the same share of non-zeros."""
    n = rowcount.numel()
    order = torch.argsort(rowcount.cpu(), descending=True, stable=True)
    pos = torch.arange(n)
    rnd, k = pos // world, pos % world
    rank_of = torch.where(rnd % 2 == 0, k, world - 1 - k)
    counts = torch.bincount(rank_of, minlength=world).tolist()
    offsets = [0]
    for c in counts:
        offsets.append(offsets[-1] + int(c))
    new_id = torch.tensor(offsets[:-1], dtype=torch.long)[rank_of] + rnd
    inv = torch.empty(n, dtype=torch.long)
    inv[order] = new_id
    perm = torch.empty(n, dtype=torch.long)
    perm[new_id] = order
    return DensePlan(world, n, [int(c) for c in counts], offsets, perm, inv)


def relabel(adj: SparseTensor, plan: DensePlan) -> SparseTensor:
    row, col, val = adj.coo()
    inv = plan.inv.to(row.device)
    return SparseTensor(row=inv[row], col=inv[col], value=val, sparse_sizes=(plan.n, plan.n), is_sorted=False)


def row_shard(adj_rel: SparseTensor, plan: DensePlan, rank: int):
    rowptr, col, val = adj_rel.csr()
    r0, r1 = plan.rows_of(rank)
    e0, e1 = int(rowptr[r0]), int(rowptr[r1])
    return (rowptr[r0:r1 + 1] - e0).contiguous(), col[e0:e1].contiguous(), None if val is None else val[e0:e1].contiguous()


# ----------------------------------------------------------------------------------------------------- exchanges
class TorchExchange:
    """R<->C layout exchanges and row all-gathers on torch.distributed collectives (any backend, CPU or CUDA)."""

    def __init__(self, plan: DensePlan, rank: int, group=None):
        self.plan, self.rank, self.world, self.group = plan, rank, plan.world, group
        self.n_p = plan.counts[rank]

    def buffer(self, name: str, shape, device) -> torch.Tensor:
        return torch.zeros(*shape, dtype=torch.float32, device=device)

    def r2c(self, src: torch.Tensor, dst: torch.Tensor, name: str = ""):
        """src [n_p, K] (R layout) -> dst [N, K/P] (C layout)."""
        P, n_p = self.world, self.n_p
        kc = src.shape[1] // P
        packed = src.view(n_p, P, kc).permute(1, 0, 2).reshape(P * n_p, kc).contiguous()
        dist.all_to_all_single(dst, packed, output_split_sizes=self.plan.counts, input_split_sizes=[n_p] * P, group=self.group)

    def c2r(self, src: torch.Tensor, dst: torch.Tensor, name: str = ""):
        """src [N, K/P] (C layout) -> dst [n_p, K] (R layout)."""
        P, n_p = self.world, self.n_p
        kc = src.shape[1]
        tmp = torch.empty(P * n_p, kc, dtype=src.dtype, device=src.device)
        dist.all_to_all_single(tmp, src.contiguous(), output_split_sizes=[n_p] * P, input_split_sizes=self.plan.counts,
                               group=self.group)
        dst.view(n_p, P, kc).copy_(tmp.view(P, n_p, kc).permute(1, 0, 2))

    def allgather_rows(self, src: torch.Tensor, dst: torch.Tensor, name: str = ""):
        """src [n_p, K] -> dst [N, K] (every rank's block at its row offset)."""
        P = self.world
        dist.all_to_all_single(dst, src.repeat(P, 1), output_split_sizes=self.plan.counts,
                               input_split_sizes=[self.n_p] * P, group=self.group)

    def allgather_vec(self, src: torch.Tensor, dst: torch.Tensor, name: str = ""):
        """src [m] -> dst [P, m]."""
        dist.all_gather_into_tensor(dst.view(-1), src.contiguous().view(-1), group=self.group)

    def check(self):
        pass


class NullExchange(TorchExchange):
    """TIMING DIAGNOSTICS ONLY: one rank's share of the compute on a single GPU, exchanges skipped (results are wrong).
    Lets ncu profile what a rank of a P-GPU run executes (ncu must not wrap multi-rank commands)."""

    def r2c(self, src, dst, name=""): pass
    def c2r(self, src, dst, name=""): pass
    def allgather_rows(self, src, dst, name=""): pass
    def allgather_vec(self, src, dst, name=""): pass


class PeerExchange:
    """The same primitives as direct stores into the consumers' buffers (CUDA IPC arena + flag barrier)."""

    def __init__(self, plan: DensePlan, rank: int, arena_bytes: int, group=None):
        from .peer import PeerArena
        self.plan, self.rank, self.world = plan, rank, plan.world
        self.n_p = plan.counts[rank]
        self.arena = PeerArena(arena_bytes, group)
        self._order = [(rank + 1 + i) % self.world for i in range(self.world)]     # start with the next rank: spread NVLink load

    def buffer(self, name: str, shape, device) -> torch.Tensor:
        return self.arena.alloc(name, shape)

    def fused_r2c_targets(self, name: str):
        """Raw addresses of every rank's C-layout buffer `name` (rank order = column-block order): the GEMM epilogue stores
        its tiles there directly (b200gnn_gemm_tf32x3_scatter_f32); follow with barrier()."""
        return [self.arena.peer_ptr(name, q, 0) for q in range(self.world)]

    def barrier(self):
        self.arena.barrier()

    def fused_c2r_targets(self, name: str):
        """Raw addresses of every rank's R-layout buffer `name` ([block, K]); producers store row i of their C-layout result at
        (i - offsets[q], rank*kc ...) of rank q's buffer; follow with barrier()."""
        return [self.arena.peer_ptr(name, q, 0) for q in range(self.world)]

    def r2c(self, src: torch.Tensor, dst: torch.Tensor, name: str):
        from .peer import copy2d
        P, n_p, K = self.world, self.n_p, src.shape[1]
        kc = K // P
        off = self.plan.offsets[self.rank]
        copies = [(self.arena.peer_ptr(name, q, off * kc), src.data_ptr() + 4 * q * kc, kc, src.stride(0), n_p) for q in self._order]
        self.arena.exchange(copies, kc)

    def c2r(self, src: torch.Tensor, dst: torch.Tensor, name: str):
        from .peer import copy2d
        P, kc = self.world, src.shape[1]
        K = kc * P
        copies = [(self.arena.peer_ptr(name, q, self.rank * kc), src.data_ptr() + 4 * self.plan.offsets[q] * src.stride(0), K,
                   src.stride(0), self.plan.counts[q]) for q in self._order]
        self.arena.exchange(copies, kc)

    def allgather_rows(self, src: torch.Tensor, dst: torch.Tensor, name: str):
        from .peer import copy2d
        K = src.shape[1]
        off = self.plan.offsets[self.rank]
        copies = [(self.arena.peer_ptr(name, q, off * K), src.data_ptr(), K, src.stride(0), self.n_p) for q in self._order]
        self.arena.exchange(copies, K)

    def allgather_vec(self, src: torch.Tensor, dst: torch.Tensor, name: str):
        from .peer import copy2d
        m = src.numel()
        assert m % 4 == 0
        copies = [(self.arena.peer_ptr(name, q, self.rank * m), src.data_ptr(), m, m, 1) for q in self._order]
        self.arena.exchange(copies, m)

    def check(self):
        if self.arena.error_flag():
            raise lib.B200GnnError("peer barrier timed out: a rank never arrived")


def _numel(shape) -> int:
    n = 1
    for d in shape:
        n *= int(d)
    return n


# ----------------------------------------------------------------------------------------------------- trainer
class HybridGCNTrainer(GCNStudentTrainer):
    """One rank of the hybrid-layout GCN student; same step semantics as GCNStudentTrainer (engine.py)."""

    aux_loss_supported = False       # out_feat's gradient would need its own route through the R / C layouts

    def __init__(self, adj: SparseTensor, dims: List[int], group=None, exchange: str = "peer", _fake=None, fuse_r2c: bool = True,
                 fuse_c2r: bool = True, fuse_gather: bool = False, **kw):
        self.group = group
        self.fuse_r2c, self.fuse_c2r = bool(fuse_r2c), bool(fuse_c2r)
        # the narrow row all-gather inside the GEMM epilogue (b200gnn_gemm_tf32x3_bcast_f32): measured neutral on 2 GPUs
        # (1.85 vs 1.81 ms/step), P x the stores from a 1-wave GEMM — off unless asked for
        self.fuse_gather = bool(fuse_gather)
        if _fake is not None:                       # (rank, world) of a pretended run: exchange="null" only
            assert exchange == "null"
            self.rank, self.world = _fake
        else:
            assert dist.is_initialized(), "torch.distributed must be initialised"
            self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        P = self.world
        self.n_global = adj.size(0)
        super().__init__(adj, dims, **kw)
        dev = self.device
        N, L = self.n_global, self.L
        self.row0 = self.plan.offsets[self.rank]
        self.rowmap = self.plan.perm[self.row0:self.row0 + self.n_p].to(torch.int32).to(dev)    # local row -> original id
        self.rowmap_full = self.plan.perm.to(torch.int32).to(dev)                                # C layout: new id -> original id
        # aggregation mode per operand width
        self.col_mode = {k: (k % (4 * P) == 0) for k in set(dims)}
        n_par = self.params.numel()
        self.n_par = n_par
        n_red = self._grads_buf.numel()                 # gradients + loss scalars, reduced together
        B = self.plan.block
        kin = dims[0]
        # ---- buffers: ("ex", ...) are destinations of exchanges (peer stores land in them: they live in the arena),
        #      ("loc", ...) are purely local
        specs = []
        if self.agg_first and self.col_mode[kin]:
            specs += [("loc", "AXc", (N, kin // P)), ("ex", "AX_R", (B, kin))]
        for l in range(L):
            k = dims[l + 1]
            if l == 0 and self.agg_first:
                continue
            if self.col_mode[k]:
                specs += [("ex", f"Hc{l}", (N, k // P)), ("loc", f"Yc{l}", (N, k // P))]
                if l < L - 1:
                    specs += [("loc", f"Ac{l}", (N, k // P)), ("ex", f"A_R{l}", (B, k)), ("ex", f"dAc{l}", (N, k // P)),
                              ("loc", f"dYc{l}", (N, k // P))]
                else:
                    specs += [("ex", f"Y_R{l}", (B, k)), ("ex", f"dYc{l}", (N, k // P))]
                specs += [("loc", f"dHc{l}", (N, k // P)), ("ex", f"dH_R{l}", (B, k))]
            else:
                specs += [("ex", f"Hfull{l}", (N, k)), ("ex", f"dYfull{l}", (N, k))]
        for k in sorted(set(dims[1:-1])):
            specs.append(("ex", f"stat_all{k}", (P, 2, k)))
        specs += [("ex", "grads_all", (P, n_red))]
        need = sum((4 * _numel(shape) + 255) // 256 * 256 for kind, _, shape in specs if kind == "ex") + 4096
        if exchange == "peer":
            self.ex = PeerExchange(self.plan, self.rank, need, group)
        elif exchange == "null":
            self.ex = NullExchange(self.plan, self.rank, group)
        else:
            self.ex = TorchExchange(self.plan, self.rank, group)
        self.c: Dict[str, torch.Tensor] = {}
        for kind, name, shape in specs:
            t = self.ex.buffer(name, shape, dev) if kind == "ex" else torch.zeros(*shape, device=dev)
            if name.endswith("_R") or "_R" in name:          # R-layout blocks are allocated at the common block size
                t = t[:self.n_p]
            self.c[name] = t
        kmax = max(dims[1:])
        self.stat_loc = torch.zeros(2 * kmax, device=dev)
        self.stat_all = {k: self.c[f"stat_all{k}"] for k in set(dims[1:-1])}
        self.grads_all = self.c["grads_all"]
        self.bn_c = {l: torch.empty(4, dims[l + 1] // P, device=dev) for l in range(L - 1) if self.col_mode[dims[l + 1]]}
        slots_full = ops.stat_slots(self.Gfull)
        self.stat_part_c = {l: torch.empty(slots_full, 2, dims[l + 1] // P, device=dev)
                            for l in range(L - 1) if self.col_mode[dims[l + 1]]}
        self.rs_full = ops.rows_slots(N)
        self._layer_in: List[Optional[torch.Tensor]] = [None] * L

    def _prepare_graph(self, adj: SparseTensor):
        """This rank's rows of the relabelled Â for the row-sharded aggregations (forward and, Â being symmetric, backward),
        buffers of the common block size; the whole relabelled Â (self.Gfull) for the feature-parallel ones."""
        norm = gcn_norm(adj)
        if not _is_symmetric(norm):
            raise NotImplementedError("the multi-GPU backward relies on a symmetric normalised adjacency")
        self.plan = make_dense_plan(norm.storage.rowcount(), self.world)
        rel = relabel(norm, self.plan)
        rowptr, col, val = row_shard(rel, self.plan, self.rank)
        self.n_p = self.plan.counts[self.rank]
        shard = csr_graph_from(rowptr, col, val, self.n_p, self.n_global)
        frp, fcol, fval = rel.csr()
        self.Gfull = csr_graph_from(frp, fcol, fval, self.n_global, self.n_global)
        return shard, shard, self.plan.block

    # ------------------------------------------------------------------ data placement
    def shard_inputs(self, x, y, train_idx, teacher_logits=None):
        """Original node order -> what this rank holds: its rows of X / labels / teacher logits in relabelled order, the
        column slice of X for all nodes when layer 0 aggregates feature-parallel, its local training rows."""
        plan, dev = self.plan, self.device
        perm = plan.perm.to(dev)
        r0, r1 = plan.rows_of(self.rank)
        mine = perm[r0:r1]
        x = x.to(dev)
        kin, P = self.dims[0], self.world
        if self.agg_first and self.col_mode[kin]:
            kc = kin // P
            x_in = x[:, self.rank * kc:(self.rank + 1) * kc][perm].contiguous()      # [N, kin/P]: C layout
        elif self.agg_first:
            x_in = x[perm].contiguous()                                                # replicated (narrow input)
        else:
            x_in = x[mine].contiguous()                                                # R layout
        y_loc = y.to(dev)[mine].contiguous()
        t_loc = None if teacher_logits is None else teacher_logits.to(dev)[mine].contiguous()
        new_train = plan.inv.to(dev)[train_idx.to(dev)]
        loc = new_train[(new_train >= r0) & (new_train < r1)] - r0
        self.n_train_global = int(train_idx.numel())
        return x_in, y_loc, torch.sort(loc).values.contiguous(), t_loc

    def input_bytes(self, x_in, y_loc, tr_loc, t_loc) -> int:
        return sum(t.numel() * t.element_size() for t in (x_in, y_loc, tr_loc, t_loc) if t is not None)

    def gather_rows(self, local: torch.Tensor) -> torch.Tensor:
        """Every rank's [n_p, k] rows -> [N, k] in ORIGINAL node order (evaluation / tests; torch.distributed)."""
        full = torch.empty(self.n_global, local.shape[1], device=local.device)
        dist.all_to_all_single(full, local.contiguous().repeat(self.world, 1), output_split_sizes=self.plan.counts,
                               input_split_sizes=[self.n_p] * self.world, group=self.group)
        return full[self.plan.inv.to(local.device)]

    def out_feat(self) -> torch.Tensor:
        l = self.L - 2
        return self.c[f"A_R{l}"] if self.col_mode[self.dims[l + 1]] else self.A[l]

    # ------------------------------------------------------------------ pieces
    def _cols(self, v: torch.Tensor, k: int) -> torch.Tensor:
        kc = k // self.world
        return v[self.rank * kc:(self.rank + 1) * kc]

    def _row_stats_allgather(self, partial: torch.Tensor, k: int) -> torch.Tensor:
        """local [slots,2,k] partial sums -> [P,2,k] (one block per rank, summed by the consumer in rank order)."""
        s = ops.partial_reduce(partial, out=self.stat_loc[:2 * k].view(2, k))
        self.ex.allgather_vec(s.view(-1), self.stat_all[k], f"stat_all{k}")
        return self.stat_all[k]

    def _act_R(self, l: int, y: torch.Tensor, bn: torch.Tensor, out: torch.Tensor, training: bool):
        ops.affine_relu_dropout_mapped(y, bn[2], bn[3], True, self.p if training else 0.0, self.seed, l, out=out,
                                       step_dev=self.step_count if training else None, step_mul=self.L, rowmap=self.rowmap)

    # ------------------------------------------------------------------ forward
    def forward(self, x_in: torch.Tensor, training: bool = True) -> torch.Tensor:
        c, P, dims = self.c, self.world, self.dims
        inp = None
        for l in range(self.L):
            last = l == self.L - 1
            k = dims[l + 1]
            if l == 0 and self.agg_first:
                if self.col_mode[dims[0]]:
                    kc0 = dims[0] // P
                    if self._fusable_c2r(kc0):       # aggregation epilogue = the C->R exchange
                        ops.spmm_csr_scatter(self.Gfull, x_in, self.ex.fused_c2r_targets("AX_R"), self.plan.offsets, dims[0],
                                             self.rank * kc0)
                        self.ex.barrier()
                    else:
                        ops.spmm_csr(self.Gfull, x_in, "sum", out=c["AXc"])
                        self.ex.c2r(c["AXc"], c["AX_R"], "AX_R")
                    ax = c["AX_R"]
                else:
                    ax = ops.spmm_csr(self.G, x_in, "sum", out=self.AX)
                self._layer_in[0] = ax
                gp = self._gemm_part.get(k) if training else None
                if gp is not None:                   # this rank's BatchNorm partial sums out of the GEMM epilogue (engine.py)
                    hi, lo = ops.split_tf32(self.W[0], transpose=True, hi=self.Wt_split[0][0], lo=self.Wt_split[0][1])
                    ops.gemm_tf32x3_stats(ax, hi, lo, self.b[0], self.Y[0], gp)
                else:
                    self._linear(0, ax, self.Y[0], bias=self.b[0])
                if training:
                    part = gp if gp is not None else ops.col_stats(self.Y[0], partial=self._part(k))
                    sums = self._row_stats_allgather(part, k)
                    ops.bn_finalize(sums, self.n_global, self.gamma[0], self.beta[0], self.bn_eps, self.bn_momentum,
                                    self.running_mean[0], self.running_var[0], out=self.bn[0])
                    self._act_R(0, self.Y[0], self.bn[0], self.A[0], True)
                else:
                    ops.affine_relu_dropout(self.Y[0], *self._bn_eval(0), True, 0.0, out=self.A[0])
                inp = self.A[0]
                continue
            src = x_in if l == 0 else inp
            self._layer_in[l] = src
            fused_gather = (not self.col_mode[k]) and isinstance(self.ex, PeerExchange) and self.tc_gemm and self.fuse_gather and k % 4 == 0
            if self.col_mode[k] and self._fusable(k):
                self._linear_r2c(l, src, f"Hc{l}")           # GEMM epilogue = the R->C exchange
            elif fused_gather:                              # GEMM epilogue = the row all-gather of the narrow operand
                hi, lo = ops.split_tf32(self.W[l], transpose=True, hi=self.Wt_split[l][0], lo=self.Wt_split[l][1])
                ops.gemm_tf32x3_bcast(src, hi, lo, self.ex.fused_c2r_targets(f"Hfull{l}"), self.row0, k)
                self.ex.barrier()
            else:
                self._linear(l, src, self.H[l])
            if self.col_mode[k]:
                kc = k // P
                if not self._fusable(k):
                    self.ex.r2c(self.H[l], c[f"Hc{l}"], f"Hc{l}")
                bias_c = self._cols(self.b[l], k)
                if last:
                    ops.spmm_csr(self.Gfull, c[f"Hc{l}"], "sum", bias=bias_c, out=c[f"Yc{l}"])
                    self.ex.c2r(c[f"Yc{l}"], c[f"Y_R{l}"], f"Y_R{l}")
                    return c[f"Y_R{l}"]
                if training:
                    if kc <= 64:      # narrow slices: the multi-row-per-warp kernel (no fused statistics) + one small pass
                        ops.spmm_csr(self.Gfull, c[f"Hc{l}"], "sum", bias=bias_c, out=c[f"Yc{l}"])
                        part = ops.col_stats(c[f"Yc{l}"], partial=self._part_c(kc))
                    else:
                        part = self.stat_part_c[l]
                        ops.spmm_csr(self.Gfull, c[f"Hc{l}"], "sum", bias=bias_c, out=c[f"Yc{l}"], stat_partial=part)
                    ops.bn_finalize(part, self.n_global, self._cols(self.gamma[l], k), self._cols(self.beta[l], k), self.bn_eps,
                                    self.bn_momentum, self._cols(self.running_mean[l], k), self._cols(self.running_var[l], k),
                                    out=self.bn_c[l])
                    if isinstance(self.ex, PeerExchange) and self.fuse_c2r:     # activation pass = the C->R exchange of A_l
                        ops.affine_relu_dropout_scatter(c[f"Yc{l}"], self.bn_c[l][2], self.bn_c[l][3], True, self.p, self.seed, l,
                                                        c[f"Ac{l}"], self.step_count, self.L, self.rowmap_full, k, self.rank * kc,
                                                        self.ex.fused_c2r_targets(f"A_R{l}"), self.plan.offsets, k)
                        self.ex.barrier()
                        inp = c[f"A_R{l}"]
                        continue
                    ops.affine_relu_dropout_mapped(c[f"Yc{l}"], self.bn_c[l][2], self.bn_c[l][3], True, self.p, self.seed, l,
                                                   out=c[f"Ac{l}"], step_dev=self.step_count, step_mul=self.L,
                                                   rowmap=self.rowmap_full, k_global=k, col_offset=self.rank * kc)
                else:
                    ops.spmm_csr(self.Gfull, c[f"Hc{l}"], "sum", bias=bias_c, out=c[f"Yc{l}"])
                    cols = slice(self.rank * kc, (self.rank + 1) * kc)
                    ops.affine_relu_dropout(c[f"Yc{l}"], *self._bn_eval(l, cols), True, 0.0, out=c[f"Ac{l}"])
                self.ex.c2r(c[f"Ac{l}"], c[f"A_R{l}"], f"A_R{l}")
                inp = c[f"A_R{l}"]
            else:
                if not fused_gather:
                    self.ex.allgather_rows(self.H[l], c[f"Hfull{l}"], f"Hfull{l}")
                if last:
                    ops.spmm_csr(self.G, c[f"Hfull{l}"], "sum", bias=self.b[l], out=self.Y[l])
                    return self.Y[l]
                if training:
                    part = self.stat_part[l]
                    ops.spmm_csr(self.G, c[f"Hfull{l}"], "sum", bias=self.b[l], out=self.Y[l], stat_partial=part)
                    sums = self._row_stats_allgather(part, k)
                    ops.bn_finalize(sums, self.n_global, self.gamma[l], self.beta[l], self.bn_eps, self.bn_momentum,
                                    self.running_mean[l], self.running_var[l], out=self.bn[l])
                    self._act_R(l, self.Y[l], self.bn[l], self.A[l], True)
                else:
                    ops.spmm_csr(self.G, c[f"Hfull{l}"], "sum", bias=self.b[l], out=self.Y[l])
                    ops.affine_relu_dropout(self.Y[l], *self._bn_eval(l), True, 0.0, out=self.A[l])
                inp = self.A[l]
        raise AssertionError("unreachable")

    def _fusable_c2r(self, kc: int, stats: bool = False) -> bool:
        """C->R exchange performed by the producing kernel: TMA SpMM kernels (kc % 128 == 0) or the narrow kernel (kc <= 64)."""
        return isinstance(self.ex, PeerExchange) and self.fuse_c2r and (kc % 128 == 0 or (kc <= 64 and not stats))

    def _fusable(self, k: int) -> bool:
        """R->C exchange performed by the producing GEMM's epilogue: peer exchange, tensor-core GEMM, 32-column chunks."""
        return isinstance(self.ex, PeerExchange) and self.tc_gemm and self.fuse_r2c and (k // self.world) % 32 == 0 and k > 48

    def _linear_r2c(self, l: int, inp: torch.Tensor, name: str):
        """H = inp @ W_l stored straight into every rank's C-layout buffer `name` (no H_R, no exchange kernel)."""
        hi, lo = ops.split_tf32(self.W[l], transpose=True, hi=self.Wt_split[l][0], lo=self.Wt_split[l][1])
        ops.gemm_tf32x3_scatter(inp, hi, lo, self.ex.fused_r2c_targets(name), self.row0)
        self.ex.barrier()

    def _dgrad_r2c(self, l: int, d_out: torch.Tensor, name: str):
        """dA = d_out @ W_l^T stored straight into every rank's C-layout buffer `name`."""
        hi, lo = ops.split_tf32(self.W[l], transpose=False, hi=self.W_split[l][0], lo=self.W_split[l][1])
        ops.gemm_tf32x3_scatter(d_out, hi, lo, self.ex.fused_r2c_targets(name), self.row0)
        self.ex.barrier()

    def logits_rows(self) -> torch.Tensor:
        l = self.L - 1
        return self.c[f"Y_R{l}"] if self.col_mode[self.dims[l + 1]] else self.Y[l]

    # ------------------------------------------------------------------ backward
    def backward(self, x_in: torch.Tensor):
        """Consumes self.dY[-1] (d loss / d logits of the local rows); fills self.grads with this rank's CONTRIBUTION
        (summed over ranks by the caller).  Parameters whose gradient a rank computes from whole columns
        (feature-parallel BatchNorm: gamma/beta/conv-bias slices) are zero outside its slice."""
        c, P, dims, L = self.c, self.world, self.dims, self.L
        self.grads.zero_()                              # slices a rank does not own stay zero (summed over ranks later)
        d_act = None                                    # d loss / d A_{l-1} in R layout, produced by layer l's dgrad
        fused_prev = False                              # ... or already delivered in C layout by that GEMM's epilogue
        dz_ready = False                                # ... or already masked + reduced by that GEMM's epilogue (R layout)
        for l in range(L - 1, -1, -1):
            k = dims[l + 1]
            last = l == L - 1
            first_agg = l == 0 and self.agg_first
            hidden_in = self._layer_in[l]
            if first_agg:
                # BatchNorm backward in R layout with globally summed statistics, then dW0 = (ÂX)^T dY0
                part, bn = self._part(k), self.bn[0]
                if dz_ready:                            # layer 1's input-gradient GEMM already stored dz and reduced it
                    sums = self._row_stats_allgather(self._gemm_part[k], k)
                    x_out = None
                else:
                    ops.bn_act_bwd_reduce(d_act, self.A[0], self.Y[0], bn[0], bn[1], self.p, part)
                    sums = self._row_stats_allgather(part, k)
                    x_out = self.A[0]
                ops.bn_act_bwd_apply(d_act, x_out, self.Y[0], bn[0], bn[1], self.gamma[0], sums, self.n_global, self.p,
                                     self.dY[0], self.ggamma[0], self.gbeta[0], self.gb[0], part, self._coef(k))
                if self.rank != 0:                      # computed from GLOBAL sums on every rank: count once
                    self.ggamma[0].zero_(); self.gbeta[0].zero_()
                self._wgrad_async(0, hidden_in, self.dY[0])
                continue
            # ---- d loss / d Y_l  ->  dH_l = Â dY_l
            if self.col_mode[k]:
                kc = k // P
                if last:
                    ops.col_sum(self.dY[l], out=self.gb[l], partial=self._part(k))
                    self.ex.r2c(self.dY[l], c[f"dYc{l}"], f"dYc{l}")
                else:
                    if not fused_prev:
                        self.ex.r2c(d_act, c[f"dAc{l}"], f"dAc{l}")
                    bn = self.bn_c[l]
                    pk = self._part_c(kc)
                    ops.bn_act_bwd(c[f"dAc{l}"], c[f"Ac{l}"], c[f"Yc{l}"], bn[0], bn[1], self._cols(self.gamma[l], k), self.p,
                                   d_y=c[f"dYc{l}"], d_gamma=self._cols(self.ggamma[l], k), d_beta=self._cols(self.gbeta[l], k),
                                   d_bias=self._cols(self.gb[l], k), partial=pk, coef=self._coef(kc))
                if self._fusable_c2r(kc):            # aggregation epilogue = the C->R exchange of d H_l
                    ops.spmm_csr_scatter(self.Gfull, c[f"dYc{l}"], self.ex.fused_c2r_targets(f"dH_R{l}"), self.plan.offsets, k,
                                         self.rank * kc)
                    self.ex.barrier()
                else:
                    ops.spmm_csr(self.Gfull, c[f"dYc{l}"], "sum", out=c[f"dHc{l}"])
                    self.ex.c2r(c[f"dHc{l}"], c[f"dH_R{l}"], f"dH_R{l}")
                dH = c[f"dH_R{l}"]
            else:
                if last:
                    ops.col_sum(self.dY[l], out=self.gb[l], partial=self._part(k))
                else:
                    part, bn = self._part(k), self.bn[l]
                    ops.bn_act_bwd_reduce(d_act, self.A[l], self.Y[l], bn[0], bn[1], self.p, part)
                    sums = self._row_stats_allgather(part, k)
                    ops.bn_act_bwd_apply(d_act, self.A[l], self.Y[l], bn[0], bn[1], self.gamma[l], sums, self.n_global, self.p,
                                         self.dY[l], self.ggamma[l], self.gbeta[l], self.gb[l], part, self._coef(k))
                    if self.rank != 0:
                        self.ggamma[l].zero_(); self.gbeta[l].zero_()
                self.ex.allgather_rows(self.dY[l], c[f"dYfull{l}"], f"dYfull{l}")
                ops.spmm_csr(self.G, c[f"dYfull{l}"], "sum", out=self.dH[l])
                dH = self.dH[l]
            fused_prev = False
            if l > 0:
                k_prev = dims[l]
                prev_first_agg = (l - 1 == 0) and self.agg_first
                if (not prev_first_agg) and self.col_mode[k_prev] and (l - 1 < L - 1) and self._fusable(k_prev):
                    self._dgrad_r2c(l, dH, f"dAc{l - 1}")   # input-gradient GEMM epilogue = the R->C exchange of d A_{l-1}
                    fused_prev, d_act = True, None
                elif prev_first_agg and self._gemm_part.get(k_prev) is not None:
                    # layer 0's BatchNorm lives in R layout: pass 1 of its backward in this GEMM's epilogue (engine.py)
                    hi, lo = ops.split_tf32(self.W[l], transpose=False, hi=self.W_split[l][0], lo=self.W_split[l][1])
                    ops.gemm_tf32x3_bnbwd(dH, hi, lo, self.dA[0], self.A[0], self.Y[0], self.bn[0][0], self.bn[0][1], self.p,
                                          self._gemm_part[k_prev])
                    d_act, dz_ready = self.dA[0], True
                else:
                    self._linear_dgrad(l, dH, self.dA[l - 1])
                    d_act = self.dA[l - 1]
            self._wgrad_async(l, hidden_in, dH)
        self._wgrad_join()

    def _part_c(self, kc: int) -> torch.Tensor:
        key = f"partc{kc}"
        if key not in self._static:
            self._static[key] = torch.empty(self.rs_full, 2, kc, device=self.device)
        return self._static[key]

    # ------------------------------------------------------------------ step
    def _reduce_grads(self):
        # gradients and loss scalars (one buffer): every rank's contribution lands in every rank's [P, n] block and is summed
        # in rank order (fp64) -> bit-identical replicas, no all-reduce
        self.ex.allgather_vec(self._grads_buf, self.grads_all, "grads_all")
        ops.partial_reduce(self.grads_all, out=self._grads_buf)

    def exchange_bytes_per_step(self) -> int:
        """Bytes each rank RECEIVES over NVLink per training step (data-path exchanges only)."""
        P, N, dims, L = self.world, self.n_global, self.dims, self.L
        tot = 0
        if self.agg_first and self.col_mode[dims[0]]:
            tot += self.n_p * dims[0] * 4 * (P - 1) // P
        for l in range(L):
            if l == 0 and self.agg_first:
                continue
            k = dims[l + 1]
            if self.col_mode[k]:
                per = self.n_p * k * 4 * (P - 1) // P          # one R<->C exchange
                tot += per * (4 if l < L - 1 else 4)            # H r2c, A/Y c2r, dA/dY r2c, dH c2r
            else:
                tot += 2 * (N - self.n_p) * k * 4
        return tot
