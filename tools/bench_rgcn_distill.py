"""Representation distillation on the MAG student: the fused engine (RGCNTrainer.train_step(aux=)) against the module path
(MessagePassing RelNet + torch Adam over model and heads), both with the b200gnn criteria, on GraphSAINT batches.

    python tools/bench_rgcn_distill.py [--steps 5] [--warmup 2] [--scale 1.0] [--out profiles] [--modes fitnet,at,...]

The graph, batches (batch_size 20000, walk_length 2) and module path come from tools/bench_rgcn_train.py.  Each mode runs
at the settings of the reference's mag_pyg/scripts/run.sh (the gnn.py form, loss_cls + beta * aux) with a 3 x 512 eval-mode
teacher (randomly initialised: its cost, not its accuracy, is measured), whose forward is part of every step: the engine
uses a teacher RGCNTrainer, the module path a teacher RelNet.  The engine and the module path run alternately on the same
batches; times are CUDA events after warm-up.  One JSON line per mode (ms/step, b200gnn launches per engine step, train
rows per batch, peak memory of each path), with the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "tools"))

from bench_rgcn_train import gpu_info, mag_graph, module_net, timed  # noqa: E402

import efficient_gnns_b200  # noqa: E402
from efficient_gnns_b200 import criterion as C  # noqa: E402
from efficient_gnns_b200 import lib, sampling  # noqa: E402
from efficient_gnns_b200.rgcn import RGCNTrainer  # noqa: E402

# mode -> (criterion, kernel, beta, max_samples, nce_T, projection heads): mag_pyg/scripts/run.sh
MODES = {
    "fitnet": ("fitnet", None, 100.0, None, None, True),
    "at": ("at", None, 1e4, None, None, False),
    "lpw_rbf": ("lpw", "rbf", 100.0, None, None, False),
    "gpw_cosine": ("gpw", "cosine", 100.0, 24576, None, False),
    "gpw_rbf": ("gpw", "rbf", 100.0, 8192, None, False),
    "nce": ("nce", None, 0.1, 24576, 0.075, True),
}
PROJ = 128


def aux_loss(mode, z, labels, f, t_feat, edges, heads):
    kind, kernel, beta, max_samples, nce_T, _ = MODES[mode]
    if heads:
        f, t_feat = heads[0](f), heads[1](t_feat)
    if kind == "fitnet":
        return C.fitnet_criterion(z, labels, f, t_feat, beta)[2]
    if kind == "at":
        return C.at_criterion(z, labels, f, t_feat, beta)[2]
    if kind == "lpw":
        return C.lpw_criterion(z, labels, f, t_feat, edges, kernel, beta)[2]
    if kind == "gpw":
        return C.gpw_criterion(z, labels, f, t_feat, kernel, beta, max_samples)[2]
    return C.nce_criterion(z, labels, f, t_feat, beta, nce_T, max_samples)[2]


def make_heads(hidden):
    mk = lambda i: torch.nn.Sequential(torch.nn.Linear(i, PROJ), torch.nn.BatchNorm1d(PROJ), torch.nn.ReLU()).cuda()  # noqa: E731
    return mk(hidden), mk(512)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=str(ROOT / "profiles"))
    ap.add_argument("--modes", default=",".join(MODES))
    args = ap.parse_args()
    torch.cuda.set_device(0)
    info = gpu_info()
    homo, num_nodes, rel_dst, x_dict, x_type, classes = mag_graph(args.scale)
    R = len(rel_dst)
    out_dir = Path(args.out)
    out_dir.mkdir(parents=True, exist_ok=True)
    full = homo.to(torch.device("cuda"))
    loader = sampling.GraphSAINTRandomWalkSampler(full, batch_size=20000, walk_length=2, num_steps=args.warmup + args.steps, seed=0)
    batches = list(loader)
    from test_rgcn_gpu import RelConv
    teacher = RGCNTrainer(num_nodes, [x_type], R, rel_dst, 128, 512, classes, 3, dropout=0.5, seed=1)
    tnet = module_net(num_nodes, x_type, R, 512, classes)[0]
    tnet.convs.insert(1, RelConv(512, 512, len(num_nodes), R).cuda())
    tnet.load_state_dict(teacher.state_dict())
    tnet.eval()

    for mode in args.modes.split(","):
        np.random.seed(0)                                     # the GSP / G-CRD row samples (criterion.py:62-64)
        with_heads = MODES[mode][5]
        st = RGCNTrainer(num_nodes, [x_type], R, rel_dst, 128, 32, classes, 2, dropout=0.5, lr=0.005)
        heads_e = make_heads(32) if with_heads else ()
        opt_h = torch.optim.Adam([q for h in heads_e for q in h.parameters()], lr=0.005) if with_heads else None
        net, _ = module_net(num_nodes, x_type, R, 32, classes)
        heads_m = make_heads(32) if with_heads else ()
        opt = torch.optim.Adam(list(net.parameters()) + [q for h in heads_m for q in h.parameters()], lr=0.005)
        t_e, t_m, launches, rows, peak_e, peak_m = [], [], [], [], 0, 0
        for i, b in enumerate(batches):
            tidx = b.train_mask.nonzero().view(-1)
            labels = b.y.view(-1)[tidx]
            gargs = (b.edge_index, b.edge_attr, b.node_type, b.local_node_idx)
            edges = efficient_gnns_b200.nn.subgraph(tidx, b.edge_index, relabel_nodes=True)[0] if MODES[mode][0] == "lpw" else None

            def estep():
                teacher.forward(x_dict, *gargs)
                t_feat = teacher.out_feat()[tidx]
                st.train_step(x_dict, *gargs, b.y, tidx,
                              aux=lambda f: aux_loss(mode, st.logits()[tidx], labels, f[tidx], t_feat, edges, heads_e), beta=MODES[mode][2])
                if opt_h is not None:
                    opt_h.step(); opt_h.zero_grad()

            def mstep():
                opt.zero_grad()
                with torch.no_grad():
                    h = tnet.convs[0](efficient_gnns_b200.nn.group_input(x_dict, tnet.emb_dict, b.node_type, b.local_node_idx, 128),
                                      b.edge_index, b.edge_attr, b.node_type)
                    for conv in tnet.convs[1:-1]:
                        h = conv(F.relu(h), b.edge_index, b.edge_attr, b.node_type)
                    h = F.relu(h)
                    tnet.convs[-1](h, b.edge_index, b.edge_attr, b.node_type)      # teacher logits (gnn.py computes them)
                    t_feat = h[tidx]
                o = net(x_dict, *gargs)[tidx]
                loss = F.cross_entropy(o, labels) + MODES[mode][2] * aux_loss(mode, o.detach(), labels, net.out_feat[tidx], t_feat,
                                                                             edges, heads_m)
                loss.backward()
                opt.step()
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            before = lib.launch_count()
            te = timed(estep)
            launches.append(lib.launch_count() - before)
            peak_e = max(peak_e, torch.cuda.max_memory_allocated())
            torch.cuda.reset_peak_memory_stats()
            tm = timed(mstep)
            peak_m = max(peak_m, torch.cuda.max_memory_allocated())
            if i >= args.warmup:
                t_e.append(te); t_m.append(tm); rows.append(int(tidx.numel()))
        kind, kernel, beta, max_samples, nce_T, _ = MODES[mode]
        rec = dict(workload=f"saint_batch_{mode}", scale=args.scale, **info, batch_size=20000, walk_length=2, criterion=kind,
                   kernel=kernel, beta=beta, max_samples=max_samples, nce_T=nce_T, proj_dim=PROJ if with_heads else None,
                   teacher="3x512 eval", batch_nodes=[int(b.num_nodes) for b in batches[args.warmup:]], train_rows=rows,
                   engine_ms=sorted(t_e)[len(t_e) // 2], engine_ms_all=t_e, module_ms=sorted(t_m)[len(t_m) // 2], module_ms_all=t_m,
                   launches_per_step=launches[-1], engine_peak_mib=round(peak_e / 2 ** 20, 1),
                   module_peak_mib=round(peak_m / 2 ** 20, 1), loss=float(st.loss_out[0]), loss_aux=float(st.loss_aux))
        line = json.dumps(rec)
        print(line, flush=True)
        (out_dir / f"rgcn_distill_{mode}.json").write_text(line + "\n")
        del st, net, opt, heads_e, heads_m, opt_h
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
