"""R-GCN engines: ``RGCNTrainer`` (the training step, below) and the full-batch ``RGCNInference`` — ``RGCN.inference`` of the reference (mag_pyg/gnn.py:140-171), BASELINE.json configs[4]
("R-GCN teacher ... MAG-shape heterogeneous ... node-parallel 2/4/8×B200").

Per layer and node type t (the reference's loop, :153-169):

    out[t]  = root_lins[t](x[t])                                          one GEMM per node type
    out[t] += rel_lins[r]( mean_{j in N_r(i)} x[src(r)][j] )              per relation r = (src, ·, t): rectangular mean-SpMM,
                                                                          then a GEMM that ACCUMULATES into out[t]
    x = relu(out)  between layers

What differs from the reference's execution (not from its arithmetic): the per-relation CSR is built ONCE by the device
ingestion kernels (the reference re-sorts every relation on every call, :149-151); the relation GEMMs add into ``out[t]``
through the accumulating tcgen05 epilogue (``b200gnn_gemm_tf32x3_acc_f32``) instead of materialising ``rel_lins(tmp)`` and
an ``add_``; aggregation runs before the transform, as in the reference's inference (its training path transforms per EDGE).

Multi-GPU (``exchange`` given): same hybrid layout as hybrid.py, per node type — activations live node-parallel ("R": rank p
owns rows [off_t[p], off_t[p+1]) of every type, contiguous blocks, no relabelling: column-split aggregations are balanced by
construction), every aggregation runs feature-parallel ("C": rank p owns columns [p·F/P, (p+1)·F/P) of ALL nodes of the
source type) on the whole replicated relation graph, one R→C exchange per node type and one C→R exchange per relation per
layer; the GEMMs see only local rows.  Results equal the single-GPU engine up to fp32 reassociation of the column split.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import torch

from . import lib, ops
from .hybrid import DensePlan
from .sparse import SparseTensor


def _block_plan(n: int, world: int) -> DensePlan:
    """Contiguous equal row blocks of one node type (identity relabelling)."""
    base, rem = divmod(n, world)
    counts = [base + (1 if q < rem else 0) for q in range(world)]
    offs = [0]
    for c in counts:
        offs.append(offs[-1] + c)
    ar = torch.arange(n)
    return DensePlan(world, n, counts, offs, ar, ar)


class RGCNInference:
    """state: the reference module's state_dict (``convs.{i}.rel_lins.{r}.weight`` [out,in], ``convs.{i}.root_lins.{t}.weight``
    / ``.bias``, ``emb_dict.{t}``); edge_index_dict: {(src_key, name, dst_key): [2, E] (row 0 = source)}; key2int as the
    reference builds it (node-type keys and relation triples -> ints)."""

    def __init__(self, state: Dict[str, torch.Tensor], num_nodes: Dict[int, int], edge_index_dict, key2int, device="cuda",
                 exchange_factory=None, rank: int = 0, world: int = 1):
        self.dev = torch.device(device)
        self.key2int = key2int
        self.num_nodes = {int(k): int(v) for k, v in num_nodes.items()}
        self.n_layers = 1 + max(int(k.split(".")[1]) for k in state if k.startswith("convs."))
        self.rank, self.world = rank, world
        f32 = lambda t: t.detach().to(self.dev, torch.float32).contiguous()
        self.emb = {int(k.split(".")[1]): f32(v) for k, v in state.items() if k.startswith("emb_dict.")}
        self.layers = []
        for i in range(self.n_layers):
            rel = {int(k.split(".")[3]): f32(v) for k, v in state.items() if k.startswith(f"convs.{i}.rel_lins.") and k.endswith(".weight")}
            root_w = {int(k.split(".")[3]): f32(v) for k, v in state.items() if k.startswith(f"convs.{i}.root_lins.") and k.endswith(".weight")}
            root_b = {int(k.split(".")[3]): f32(v) for k, v in state.items() if k.startswith(f"convs.{i}.root_lins.") and k.endswith(".bias")}
            self.layers.append((rel, root_w, root_b))
        # relation graphs: rows = destination nodes, cols = source nodes, built once (device ingestion kernels)
        self.rels: List[Tuple[int, int, int, SparseTensor]] = []
        for keys, ei in edge_index_dict.items():
            s, d, r = key2int[keys[0]], key2int[keys[-1]], key2int[keys]
            ei = ei.to(self.dev)
            adj = SparseTensor(row=ei[1], col=ei[0], sparse_sizes=(self.num_nodes[d], self.num_nodes[s]), is_sorted=False)
            adj.storage.engine_csr_unweighted()
            self.rels.append((s, d, r, adj))
        self.nnz = sum(a.nnz() for *_, a in self.rels)
        # multi-GPU plumbing
        self.plans = {t: _block_plan(n, world) for t, n in self.num_nodes.items()}
        self.ex = {t: exchange_factory(self.plans[t]) for t in self.num_nodes} if (world > 1 and exchange_factory) else None
        self._bufs: Dict[str, torch.Tensor] = {}

    # ------------------------------------------------------------------ helpers
    def _gemm(self, x: torch.Tensor, w: torch.Tensor, out: torch.Tensor, bias=None, accumulate=False):
        """out (+)= x @ w^T (+bias) on the tcgen05 GEMM; K not a multiple of 4 is zero-padded (exact)."""
        k = x.shape[1]
        if k % 4:
            pad = 4 - k % 4
            x = torch.nn.functional.pad(x, (0, pad)).contiguous()
            w = torch.nn.functional.pad(w, (0, pad)).contiguous()
        hi, lo = ops.split_tf32(w)
        if accumulate:
            ops.gemm_tf32x3(x, hi, lo, out=out, accumulate=True)
        else:
            ops.gemm_tf32x3(x, hi, lo, bias=bias, out=out)

    def _buf(self, key: str, shape, ex=None) -> torch.Tensor:
        b = self._bufs.get(key)
        if b is None or tuple(b.shape) != tuple(shape):
            b = self._bufs[key] = (ex.buffer(key, shape, self.dev) if ex is not None else torch.empty(*shape, device=self.dev))
        return b

    def rows_of(self, t: int):
        return self.plans[t].rows_of(self.rank)

    # ------------------------------------------------------------------ forward
    @torch.no_grad()
    def __call__(self, x_dict: Dict[int, torch.Tensor]) -> Dict[int, torch.Tensor]:
        """x_dict: features of the node types that have them (int keys), FULL matrices; embedding tables fill the rest
        (mag_pyg/gnn.py:145-147).  Returns {type: [n_t, out]} on one GPU, this rank's row blocks on several."""
        x = {int(k): v.to(self.dev, torch.float32).contiguous() for k, v in x_dict.items()}
        x.update(self.emb)
        if self.world > 1:
            x = {t: v[self.rows_of(t)[0]:self.rows_of(t)[1]].contiguous() for t, v in x.items()}
        for i, (rel_w, root_w, root_b) in enumerate(self.layers):
            f_out = next(iter(root_w.values())).shape[0]
            out = {}
            for t, xt in x.items():
                o = self._buf(f"out{i}_{t}", (xt.shape[0], f_out))
                self._gemm(xt, root_w[t], o, bias=root_b[t])
                out[t] = o
            if self.world == 1:
                for s, d, r, adj in self.rels:
                    agg = adj.matmul(x[s], reduce="mean")                            # [n_d, F]
                    self._gemm(agg, rel_w[r], out[d], accumulate=True)
            else:
                P = self.world
                f_in = next(iter(x.values())).shape[1]
                if f_in % (4 * P):
                    raise lib.B200GnnError(f"feature width {f_in} must be a multiple of 4*world for the column layout")
                kc = f_in // P
                xc = {}
                for t, xt in x.items():                                              # R -> C, once per node type
                    dst = self._buf(f"xc{i}_{t}", (self.num_nodes[t], kc), self.ex[t])
                    self.ex[t].r2c(xt, dst, f"xc{i}_{t}")
                    xc[t] = dst
                for s, d, r, adj in self.rels:
                    agg_c = adj.matmul(xc[s], reduce="mean")                         # [n_d, F/P]: my columns, all destinations
                    n_p = self.plans[d].counts[self.rank]
                    dst = self._buf(f"agg{i}_{r}", (self.plans[d].block, f_in), self.ex[d])[:n_p]
                    self.ex[d].c2r(agg_c, dst, f"agg{i}_{r}")                        # C -> R: my destinations, all columns
                    self._gemm(dst, rel_w[r], out[d], accumulate=True)
            if i != self.n_layers - 1:
                for o in out.values():
                    o.relu_()
            x = out
        return x

    def gather(self, x_loc: Dict[int, torch.Tensor]) -> Dict[int, torch.Tensor]:
        """All ranks' row blocks -> full matrices (evaluation / tests; torch.distributed)."""
        import torch.distributed as dist
        if self.world == 1:
            return x_loc
        full = {}
        for t, v in x_loc.items():
            f = torch.empty(self.num_nodes[t], v.shape[1], device=v.device)
            dist.all_to_all_single(f, v.contiguous().repeat(self.world, 1), output_split_sizes=self.plans[t].counts,
                                   input_split_sizes=[v.shape[0]] * self.world)
            full[t] = f
        return full


# ------------------------------------------------------------------------------------------------------ training
def _pad4(k: int) -> int:
    return (k + 3) // 4 * 4


class _Graph:
    """Per-graph preparation of the fused step: type row ranges, the (destination, relation slot) CSR of the aggregation
    and its mean-weighted transpose, the (type, local id) order of the embedding scatter, and the activation buffers."""


class RGCNTrainer:
    """Fused training step of the reference's R-GCN (``RGCN.forward`` mag_pyg/gnn.py:126-138, ``train()`` :174-268 for
    ``--training supervised|kd``, and with ``train_step(aux=)`` the representation losses) on device tensors, aggregate-first:

        M_l[i, s]  = mean over the edges j -> i of the s-th relation into type(i) of x_l[j]     one SpMM per layer
        out_l[t]   = x_l[t] · root_lins[t]ᵀ + b_t                                               one grouped GEMM
        out_l[t]  += M_l[t] · [rel_lins[r_1] | … | rel_lins[r_S_t]]ᵀ                            one grouped GEMM (accumulate)
        x_{l+1}    = dropout(relu(out_l))                                                       (hidden layers)

    which is the reference's per-edge ``rel_lins[r](x_j)`` scatter-mean by linearity (its own ``inference()`` relies on the
    same identity).  The backward mirrors it: dM = dOut · [rel_lins …] (grouped), dx = the transposed mean-weighted SpMM of
    dM, dx += dOut · root_lins (grouped), weight gradients per (type, slot) on the split-K kernel, the typed scatter into the
    embedding tables, Adam over one flat buffer (embedding tables included: rows without gradient still decay their
    moments, as torch Adam over ``model.parameters()`` does).

    Rows must be grouped by node type (``node_type`` non-decreasing: ``group_hetero_graph`` ids and GraphSAINT node sets
    are).  Widths that are not multiples of 4 are zero-padded internally (exact); the padded entries of every parameter
    stay zero.  ``rel_dst_type[r]`` is the destination node type of relation r."""

    def __init__(self, num_nodes_dict, x_types, num_edge_types: int, rel_dst_type, in_channels: int, hidden_channels: int,
                 out_channels: int, num_layers: int, dropout: float = 0.5, lr: float = 0.01, alpha: float = 0.9,
                 kd_T: float = 4.0, seed: int = 0, device="cuda"):
        dev = torch.device(device)
        if dev.type == "cuda" and dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        self.num_nodes = {int(k): int(v) for k, v in num_nodes_dict.items()}
        self.T = len(self.num_nodes)
        if sorted(self.num_nodes) != list(range(self.T)) or self.T > 16:
            raise lib.B200GnnError("node types must be the integers 0..T-1 (T <= 16), as group_hetero_graph numbers them")
        self.x_types = sorted(int(t) for t in x_types)
        self.emb_types = [t for t in range(self.T) if t not in self.x_types]
        self.R = int(num_edge_types)
        self.rel_dst = [int(t) for t in rel_dst_type]
        if len(self.rel_dst) != self.R or any(not 0 <= t < self.T for t in self.rel_dst):
            raise lib.B200GnnError("rel_dst_type needs one destination node type per relation")
        self.rels_of = {t: [r for r in range(self.R) if self.rel_dst[r] == t] for t in range(self.T)}
        self.slot = [self.rels_of[self.rel_dst[r]].index(r) for r in range(self.R)]
        self.S_max = max(1, max(len(v) for v in self.rels_of.values()))
        self.L = int(num_layers)
        self.dims = [int(in_channels)] + [int(hidden_channels)] * (self.L - 1) + [int(out_channels)]
        self.dp = [_pad4(d) for d in self.dims]
        self.p, self.lr, self.alpha, self.kd_T, self.seed = float(dropout), float(lr), float(alpha), float(kd_T), int(seed)

        # flat parameter buffer in the engine's layout: per layer and node type the relation block [S_t·Fi, No] (slot-major
        # rows, i.e. rel_lins[r].weightᵀ stacked), the root block [Fi, No] and the bias [No]; then the embedding tables
        blocks, off = [], 0
        for l in range(self.L):
            fi, no = self.dp[l], self.dp[l + 1]
            for t in range(self.T):
                for name, shape in ((f"rel{l}_{t}", (len(self.rels_of[t]) * fi, no)), (f"root{l}_{t}", (fi, no)),
                                    (f"bias{l}_{t}", (no,))):
                    blocks.append((name, off, shape)); off += math.prod(shape)
        for t in self.emb_types:
            blocks.append((f"emb{t}", off, (self.num_nodes[t], self.dp[0]))); off += self.num_nodes[t] * self.dp[0]
        self.params = torch.zeros(off, device=dev)
        self.grads = torch.zeros(off, device=dev)
        self.exp_avg = torch.zeros(off, device=dev)
        self.exp_avg_sq = torch.zeros(off, device=dev)
        self.step_count = torch.zeros(1, dtype=torch.int32, device=dev)
        self.loss_out = torch.zeros(3, device=dev)
        self.P: Dict[str, torch.Tensor] = {}
        self.G: Dict[str, torch.Tensor] = {}
        for name, o, shape in blocks:
            self.P[name] = self.params[o:o + math.prod(shape)].view(shape)
            self.G[name] = self.grads[o:o + math.prod(shape)].view(shape)
        # reference keys -> views of the flat buffers in the reference's shapes
        self._pview: Dict[str, torch.Tensor] = {}
        self._gview: Dict[str, torch.Tensor] = {}
        for key, _ in self.param_table(self.num_nodes, self.x_types, self.R, *self.dims[:1], hidden_channels, out_channels,
                                       self.L):
            self._pview[key] = self._view(self.P, key)
            self._gview[key] = self._view(self.G, key)
        # tf32 splits of the weights, refreshed every step: forward operands [No, K] and input-gradient operands [N, No]
        self._split: Dict[str, Tuple[torch.Tensor, torch.Tensor]] = {}
        for l in range(self.L):
            fi, no = self.dp[l], self.dp[l + 1]
            for t in range(self.T):
                k = len(self.rels_of[t]) * fi
                if k:
                    self._split[f"rel{l}_{t}"] = (torch.empty(no, k, device=dev), torch.empty(no, k, device=dev))
                    # zero rows past S_t·Fi: the input gradient of the unused slots comes out zero
                    self._split[f"relT{l}_{t}"] = (torch.zeros(self.S_max * fi, no, device=dev),
                                                   torch.zeros(self.S_max * fi, no, device=dev))
                self._split[f"root{l}_{t}"] = (torch.empty(no, fi, device=dev), torch.empty(no, fi, device=dev))
                self._split[f"rootT{l}_{t}"] = (torch.empty(fi, no, device=dev), torch.empty(fi, no, device=dev))
        ws = [lib.load().b200gnn_wgrad_workspace_floats(fi, no) for fi, no in zip(self.dp, self.dp[1:]) if ops.wgrad_supported(fi, no)]
        self.wgrad_ws = torch.empty(max(ws), device=dev) if ws else None
        self._graph: Optional[_Graph] = None
        self._xpad: Dict[int, Tuple[torch.Tensor, torch.Tensor]] = {}
        self._last_p = 0.0
        self._last_inputs = None
        self.loss_aux: Optional[torch.Tensor] = None
        self.reset_parameters(seed)

    # ------------------------------------------------------------------ parameters
    @staticmethod
    def param_table(num_nodes_dict, x_types, num_edge_types: int, in_channels: int, hidden_channels: int, out_channels: int,
                    num_layers: int) -> List[Tuple[str, Tuple[int, ...]]]:
        """(state-dict key, shape) of every parameter of the reference module, in its order."""
        types = sorted(int(t) for t in num_nodes_dict)
        xt = {int(t) for t in x_types}
        dims = [in_channels] + [hidden_channels] * (num_layers - 1) + [out_channels]
        table = [(f"emb_dict.{t}", (int(num_nodes_dict[t]), in_channels)) for t in types if t not in xt]
        for l in range(num_layers):
            table += [(f"convs.{l}.rel_lins.{r}.weight", (dims[l + 1], dims[l])) for r in range(num_edge_types)]
            for t in types:
                table += [(f"convs.{l}.root_lins.{t}.weight", (dims[l + 1], dims[l])), (f"convs.{l}.root_lins.{t}.bias", (dims[l + 1],))]
        return table

    def _view(self, store: Dict[str, torch.Tensor], key: str) -> torch.Tensor:
        """The reference-shaped view of parameter ``key`` inside the engine layout (strided; padding excluded)."""
        f = key.split(".")
        if f[0] == "emb_dict":
            return store[f"emb{f[1]}"][:, :self.dims[0]]
        l = int(f[1])
        fi, fo = self.dims[l], self.dims[l + 1]
        if f[2] == "rel_lins":
            r = int(f[3])
            s, t = self.slot[r], self.rel_dst[r]
            return store[f"rel{l}_{t}"][s * self.dp[l]:s * self.dp[l] + fi, :fo].t()
        t = int(f[3])
        if f[4] == "bias":
            return store[f"bias{l}_{t}"][:fo]
        return store[f"root{l}_{t}"][:fi, :fo].t()

    def reset_parameters(self, seed: int = 0):
        """The reference's initialisation: xavier_uniform embeddings, torch.nn.Linear defaults; a fresh Adam."""
        g = torch.Generator().manual_seed(seed)
        self.params.zero_()
        for key, v in self._pview.items():
            if key.startswith("emb_dict."):
                a = math.sqrt(6.0 / (v.shape[0] + v.shape[1]))
            else:
                a = 1.0 / math.sqrt(self.dims[int(key.split(".")[1])])
            v.copy_((torch.rand(tuple(v.shape), generator=g) * 2 - 1) * a)
        self.exp_avg.zero_(); self.exp_avg_sq.zero_(); self.step_count.zero_()

    def state_dict(self) -> Dict[str, torch.Tensor]:
        """The reference module's keys and shapes (``emb_dict.{t}``, ``convs.{i}.rel_lins.{r}.weight``,
        ``convs.{i}.root_lins.{t}.weight`` / ``.bias``)."""
        return {k: v.detach().clone() for k, v in self._pview.items()}

    def load_state_dict(self, sd: Dict[str, torch.Tensor]):
        for k, v in self._pview.items():
            v.copy_(sd[k])

    def gradients(self) -> Dict[str, torch.Tensor]:
        """The gradient of every parameter after the last backward, under its state-dict key."""
        return {k: v.detach().clone() for k, v in self._gview.items()}

    # ------------------------------------------------------------------ graph preparation
    def _prepare(self, edge_index, edge_type, node_type, local_node_idx) -> _Graph:
        key = (edge_index, edge_type, node_type, local_node_idx)
        G = self._graph
        if G is not None and all(a is b for a, b in zip(G.key, key)) and G.versions == tuple(t._version for t in key):
            return G
        dev = self.device
        n = int(node_type.numel())
        if node_type.device != dev or edge_index.device != dev:
            raise lib.B200GnnError("RGCNTrainer: graph tensors must be on the engine's device (no CPU fallback)")
        if n > 1 and not bool((node_type[1:] >= node_type[:-1]).all()):
            raise lib.B200GnnError("RGCNTrainer: rows must be grouped by node type (node_type non-decreasing), as "
                                   "group_hetero_graph numbers nodes and GraphSAINT batches keep them; the engine does not re-sort")
        counts = torch.bincount(node_type, minlength=self.T).tolist() if n else [0] * self.T
        if len(counts) != self.T or (n and int(node_type[0]) < 0):
            raise lib.B200GnnError(f"RGCNTrainer: node types outside 0..{self.T - 1}")
        G = _Graph()
        G.key, G.versions, G.n = key, tuple(t._version for t in key), n
        G.row0 = [sum(counts[:t]) for t in range(self.T)]
        G.rows = counts
        # rows (destination, relation slot) of the aggregation: viewed as [n, S_max·F] its output is M itself
        slot = torch.tensor(self.slot, dtype=torch.long, device=dev)
        src, dst = edge_index[0], edge_index[1]
        adj = SparseTensor(row=dst * self.S_max + slot[edge_type], col=src, sparse_sizes=(n * self.S_max, n), is_sorted=False)
        G.fwd = adj.storage.engine_csr_unweighted()
        G.bwd = adj.storage.engine_csc("mean")        # weights 1 / count(dst, slot): the mean's transpose
        if self.emb_types and n:
            from .sparse import device_argsort
            big = max(self.num_nodes.values()) + 1
            G.order = device_argsort(node_type, local_node_idx, self.T, big)
        # activations: X[l] input of layer l (X[0] = grouped input), M[l], out[l]; gradients dOut[l], dM[l], dX0
        z = lambda k: torch.zeros(n, k, device=dev)
        G.X = [z(self.dp[0])]
        G.M = [z(self.S_max * self.dp[l]) for l in range(self.L)]
        G.out = [z(self.dp[l + 1]) for l in range(self.L)]
        G.X += [z(self.dp[l + 1]) for l in range(self.L - 1)]
        G.dOut = [z(self.dp[l + 1]) for l in range(self.L)]
        G.dM = [z(self.S_max * self.dp[l]) for l in range(self.L)]
        G.dX0 = z(self.dp[0]) if self.emb_types else None
        G.slots = ops.rows_slots(max(n, 1))               # enough for the column sums of any type's rows
        G.col_part = torch.empty(G.slots * 2 * max(self.dp[1:]), device=dev)
        G.kd_part = torch.empty(2 * int(lib.load().b200gnn_kd_partials(max(n, 1))), device=dev)
        G.err = torch.zeros(1, dtype=torch.int32, device=dev)
        self._graph = G
        return G

    def _table_args(self, x_dict, grads: bool):
        import ctypes as C
        ptrs, rows = (C.c_void_p * self.T)(), (C.c_int64 * self.T)()
        for t in range(self.T):
            rows[t] = self.num_nodes[t]
            if t in self.emb_types:
                ptrs[t] = (self.G if grads else self.P)[f"emb{t}"].data_ptr()
            elif not grads:
                ptrs[t] = self._features(x_dict, t).data_ptr()
        return ptrs, rows

    def _features(self, x_dict, t: int) -> torch.Tensor:
        """Feature table of type t as a contiguous fp32 [n_t, Fi0] (zero-padded to a multiple of 4; cached per tensor)."""
        x = x_dict[t]
        hit = self._xpad.get(t)
        if hit is not None and hit[0] is x and hit[2] == x._version:
            return hit[1]
        if x.shape != (self.num_nodes[t], self.dims[0]) or x.device != self.device:
            raise lib.B200GnnError(f"RGCNTrainer: features of type {t} must be [{self.num_nodes[t]}, {self.dims[0]}] on {self.device}")
        xp = torch.nn.functional.pad(x.float(), (0, self.dp[0] - self.dims[0])).contiguous()
        self._xpad[t] = (x, xp, x._version)
        return xp

    # ------------------------------------------------------------------ forward / backward
    def _groups(self, G: _Graph, names, bias_l: Optional[int] = None):
        """(row0, rows, hi, lo, bias) per node type for the grouped GEMM; names[t] None: K = 0 for that type."""
        out = []
        for t in range(self.T):
            hi, lo = self._split[names[t]] if names[t] in self._split else (None, None)
            out.append((G.row0[t], G.rows[t], hi, lo, None if bias_l is None else self.P[f"bias{bias_l}_{t}"]))
        return out

    def _forward(self, G: _Graph, x_dict, training: bool) -> torch.Tensor:
        L = lib.load()
        p = self.p if training else 0.0
        self._last_p = p
        n = G.n
        if n == 0:
            return G.out[-1][:, :self.dims[-1]]
        ptrs, rows = self._table_args(x_dict, grads=False)
        lib.check(L.b200gnn_typed_gather_f32(ptrs, rows, self.T, G.key[2].data_ptr(), G.key[3].data_ptr(), n, self.dp[0],
                                             G.X[0].data_ptr(), self.dp[0], G.err.data_ptr(), lib.stream_ptr()), "typed_gather_f32")
        for l in range(self.L):
            fi = self.dp[l]
            for t in range(self.T):
                if f"rel{l}_{t}" in self._split:
                    hi, lo = self._split[f"rel{l}_{t}"]
                    ops.split_tf32(self.P[f"rel{l}_{t}"], transpose=True, hi=hi, lo=lo)
                hi, lo = self._split[f"root{l}_{t}"]
                ops.split_tf32(self.P[f"root{l}_{t}"], transpose=True, hi=hi, lo=lo)
            ops.spmm_csr(G.fwd, G.X[l], "mean", out=G.M[l].view(n * self.S_max, fi))
            ops.gemm_tf32x3_grouped(G.X[l], G.out[l], self._groups(G, [f"root{l}_{t}" for t in range(self.T)], bias_l=l))
            ops.gemm_tf32x3_grouped(G.M[l], G.out[l], self._groups(G, [f"rel{l}_{t}" for t in range(self.T)]), accumulate=True)
            if l < self.L - 1:
                ops.affine_relu_dropout(G.out[l], None, None, True, p, self.seed, l, out=G.X[l + 1],
                                        step_dev=self.step_count if training else None, step_mul=self.L)
        return G.out[-1][:, :self.dims[-1]]

    def _wgrad(self, x: torch.Tensor, g: torch.Tensor, out: torch.Tensor):
        """out[Fi, No] = xᵀ g: split-K tcgen05 kernel where its tiling allows, the library GEMM otherwise."""
        if ops.wgrad_supported(x.shape[1], g.shape[1]):
            ops.gemm_wgrad_tf32x3(x, g, out=out, workspace=self.wgrad_ws)
        else:
            torch.mm(x.t(), g, out=out)

    def _backward(self, G: _Graph, d_out_feat: Optional[torch.Tensor] = None):
        """Consumes G.dOut[-1] (d loss / d logits, padded columns zero); fills self.grads.  ``d_out_feat`` [n, hidden] (row
        pitch free) is a gradient w.r.t. ``out_feat()``, added at the last hidden layer's ReLU/dropout backward."""
        L = lib.load()
        n = G.n
        self.grads.zero_()
        if n == 0:
            return
        for l in range(self.L - 1, -1, -1):
            fi, no = self.dp[l], self.dp[l + 1]
            dO = G.dOut[l]
            for t in range(self.T):
                r0, m = G.row0[t], G.rows[t]
                if m == 0:
                    continue
                rows = slice(r0, r0 + m)
                ops.col_sum(dO[rows], out=self.G[f"bias{l}_{t}"], partial=G.col_part[:G.slots * 2 * no].view(G.slots, 2, no))
                self._wgrad(G.X[l][rows], dO[rows], self.G[f"root{l}_{t}"])
                for s in range(len(self.rels_of[t])):
                    self._wgrad(G.M[l][rows, s * fi:(s + 1) * fi], dO[rows], self.G[f"rel{l}_{t}"][s * fi:(s + 1) * fi])
            if l == 0 and not self.emb_types:
                break
            for t in range(self.T):
                if f"relT{l}_{t}" in self._split:
                    hi, lo = self._split[f"relT{l}_{t}"]
                    k = len(self.rels_of[t]) * fi
                    ops.split_tf32(self.P[f"rel{l}_{t}"], hi=hi[:k], lo=lo[:k])
                hi, lo = self._split[f"rootT{l}_{t}"]
                ops.split_tf32(self.P[f"root{l}_{t}"], hi=hi, lo=lo)
            ops.gemm_tf32x3_grouped(dO, G.dM[l], self._groups(G, [f"relT{l}_{t}" for t in range(self.T)]))
            dX = G.dOut[l - 1] if l > 0 else G.dX0
            ops.spmm_csr(G.bwd, G.dM[l].view(n * self.S_max, fi), "sum", out=dX)
            ops.gemm_tf32x3_grouped(dO, dX, self._groups(G, [f"rootT{l}_{t}" for t in range(self.T)]), accumulate=True)
            if l > 0:
                extra = d_out_feat if l == self.L - 1 else None
                ops.relu_dropout_bwd(dX, G.X[l], self._last_p, out=dX, extra=extra)
            else:
                ptrs, rows = self._table_args(None, grads=True)
                lib.check(L.b200gnn_typed_scatter_f32(dX.data_ptr(), dX.stride(0), G.key[2].data_ptr(), G.key[3].data_ptr(),
                                                      G.order.data_ptr(), n, fi, ptrs, rows, self.T, lib.stream_ptr()),
                          "typed_scatter_f32")

    # ------------------------------------------------------------------ public
    def forward(self, x_dict, edge_index, edge_type, node_type, local_node_idx, training: bool = False) -> torch.Tensor:
        """``RGCN.forward``: logits [n, out_channels] (a view into the engine's buffer, valid until the next call).  With
        training=False (the reference's eval mode, e.g. a KD teacher) no dropout is drawn."""
        G = self._prepare(edge_index, edge_type, node_type, local_node_idx)
        return self._forward(G, {int(k): v for k, v in x_dict.items()}, training)

    def logits(self) -> torch.Tensor:
        """Logits [n, out_channels] of the last forward (a training step's forward included)."""
        return self._graph.out[-1][:, :self.dims[-1]]

    def out_feat(self) -> torch.Tensor:
        """The reference's ``model.out_feat``: the last hidden activation (after ReLU and dropout) of the last forward."""
        return self._graph.X[-1][:, :self.dims[-2]]

    def backward(self, d_logits: torch.Tensor):
        """Gradients of every parameter (``gradients()``) for an injected d loss / d logits [n, out_channels], through the
        activations of the last ``forward``."""
        G = self._graph
        G.dOut[-1].zero_()
        G.dOut[-1][:, :self.dims[-1]].copy_(d_logits)
        self._backward(G)

    def _step(self, x_dict, edge_index, edge_type, node_type, local_node_idx, y, train_idx, teacher_logits, aux=None,
              beta: float = 1.0):
        G = self._prepare(edge_index, edge_type, node_type, local_node_idx)
        logits = self._forward(G, x_dict, training=True)
        G.dOut[-1].zero_()
        ops.kd_loss_fwd_bwd(logits, y, train_idx, teacher_logits, self.alpha, self.kd_T,
                            d_logits=G.dOut[-1][:, :self.dims[-1]], loss_out=self.loss_out, partial=G.kd_part)
        d_feat = None
        if aux is not None:
            feat = self.out_feat().detach().requires_grad_(True)
            with torch.enable_grad():
                loss_aux = aux(feat)
                if loss_aux.requires_grad:
                    (loss_aux * beta).backward()
            self.loss_aux = loss_aux.detach()
            d_feat = feat.grad                        # None: the loss does not depend on out_feat, the plain backward
            if d_feat is not None and d_feat.stride(-1) != 1:
                d_feat = d_feat.contiguous()
        self._backward(G, d_feat)
        ops.adam_step(self.params, self.grads, self.exp_avg, self.exp_avg_sq, self.step_count, self.lr)
        if aux is not None:
            self.loss_out[0].add_(self.loss_aux * beta)

    def train_step(self, x_dict, edge_index, edge_type, node_type, local_node_idx, y, train_idx,
                   teacher_logits: Optional[torch.Tensor] = None, aux=None, beta: float = 1.0) -> torch.Tensor:
        """One step of the reference's ``train()`` loop body (mag_pyg/gnn.py:188-257): forward with dropout, cross-entropy
        (supervised) or ``kd_criterion`` against ``teacher_logits`` [n, out_channels] over the rows ``train_idx``, backward,
        Adam.  ``y``: labels per row ([n] or [n, 1], int64).  Returns the device tensor [loss, loss_cls, loss_kd]; no host
        sync for the loss (preparing a new graph reads its type counts and hub plan once).

        Representation distillation (``--training fitnet|at|lpw|gpw|nce``): ``aux(feat)`` receives ``out_feat()`` — the
        last hidden activation after ReLU and dropout, [n, hidden], detached and requiring grad — and returns the
        auxiliary loss, built with ``criterion.*`` and any torch-side projection heads.  Its gradient (autograd) times
        ``beta`` joins the backward at the last hidden layer's ReLU/dropout backward, so the dropout mask applies to it as
        in the reference; ``self.loss_aux`` holds its value and ``loss[0]`` includes ``beta * loss_aux``.  Without
        ``teacher_logits`` this is mag_pyg/gnn.py's ``loss_cls + beta * aux`` (:204-251), with them the ``kd + beta * aux``
        of mag_pyg/gnn_kd_and_aux.py (:204-271).  A loss that does not depend on ``feat`` runs the plain backward.  On MAG:

        * teacher features: a teacher ``RGCNTrainer`` (e.g. 3 x 512) on the same batch, ``forward(..., training=False)``,
          then ``out_feat()[train_idx]`` (clone it: the buffer is reused by the next forward);
        * LSP edges: ``nn.subgraph(train_idx, batch.edge_index, relabel_nodes=True)[0]`` (gnn.py:237);
        * GSP and G-CRD row samples: ``sampled_inds=``, or numpy's global RNG as the reference draws them;
        * the ``student_proj`` / ``teacher_proj`` heads of fitnet and nce (Linear -> BatchNorm1d -> ReLU, proj_dim 128)
          stay torch modules; put their parameters in the caller's torch Adam at the engine's learning rate.  Adam is
          elementwise, so this equals the reference's single optimizer over model and heads.

        ``aux`` needs a hidden layer (num_layers >= 2)."""
        if aux is not None and self.L < 2:
            raise lib.B200GnnError("RGCNTrainer: aux= needs a hidden layer (num_layers >= 2): there is no out_feat")
        x_dict = {int(k): v for k, v in x_dict.items()}
        y = y.reshape(-1).contiguous()
        train_idx = train_idx.contiguous()
        self._last_inputs = (x_dict, edge_index, edge_type, node_type, local_node_idx, y, train_idx, teacher_logits, aux,
                             float(beta))
        self._step(*self._last_inputs)
        return self.loss_out

    def launches_per_step(self) -> int:
        """b200gnn kernel launches in one training step on the last train_step's inputs (counted, not estimated; runs a
        step)."""
        before = lib.launch_count()
        self._step(*self._last_inputs)
        return lib.launch_count() - before
