"""B200-native sparse message-passing engine for the student-GNN distillation
hot path of chaitjo/efficient-gnns (SURVEY.md §8).

Layout
  csrc/        hand-written sm_100a CUDA kernels behind the C ABI in include/b200gnn.h
  lib.py       ctypes binding of libb200gnn.so (fails loudly if it is missing)
  ops.py       autograd-aware operators (spmm, fused BN/ReLU/dropout, losses)
  sparse.py    SparseTensor mirror (storage caches: rowptr/colptr/csr2csc/hub plan)
  nn.py        GCNConv / SAGEConv / MessagePassing mirrors of the PyG surface
  criterion.py fused distillation criteria (same names/arguments as the reference's criterion.py)
  engine.py    graph-captured full training step for the benchmark configs
  engine_sage.py / rgcn.py     fused GraphSAGE step; fused R-GCN training step and full-batch R-GCN inference
  hybrid.py / peer.py / hybrid_gat.py   multi-GPU: node-parallel dense ops + feature-parallel aggregations, peer-memory exchange
  dist.py      round-1 node-parallel engine (all-gather per aggregation), kept as the baseline
  sampling.py  device-side GraphSAINT random-walk sampler, small-graph DataLoader
  torch_ops.py `torch.ops.b200gnn.*` registration (import it to register; the module path does not need it)
  shim/        packages named torch_sparse / torch_scatter / torch_geometric / ogb
               re-exporting the above so the reference's scripts run unmodified

There is no CPU fallback anywhere in this package: CPU tensors raise.
The CPU oracle lives in the top-level ``oracle/`` directory and is test-only.
"""
from . import lib  # noqa: F401

__all__ = ["lib"]
__version__ = "0.1.0"
