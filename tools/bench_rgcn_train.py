"""R-GCN training on the MAG-shaped synthetic (BASELINE configs[4]): the fused engine (rgcn.RGCNTrainer) against the module
path (MessagePassing RelNet + torch Adam), and one grouped GEMM launch against the per-type loop it replaces.

    python tools/bench_rgcn_train.py [--steps 5] [--warmup 2] [--scale 1.0] [--out profiles]

The graph is grouped the way the reference's main() does (mag_pyg/gnn.py:322-346: reverse relations, undirected cites,
group_hetero_graph) through the ogb / torch_geometric shims.  Workloads: the full-graph student step (2 layers x 32 hidden,
349 classes) and a GraphSAINT batch step (batch_size 20000, walk_length 2, as mag_pyg/gnn.py:361-366) with and without a
3 x 512 KD teacher forward (randomly initialised: its cost, not its accuracy, is measured).  Each workload writes one JSON
line, with the GPU name and power limit read in the same run.  Times are CUDA events after warm-up; the batch workloads
include the per-batch graph preparation, and the engine and the module path run alternately on the same batches.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import efficient_gnns_b200  # noqa: E402,F401
from efficient_gnns_b200 import lib, ops, sampling  # noqa: E402
from efficient_gnns_b200.graphdata import Data  # noqa: E402
from efficient_gnns_b200.rgcn import RGCNTrainer  # noqa: E402


def mag_graph(scale: float):
    sys.path.insert(0, str(Path(efficient_gnns_b200.__file__).resolve().parent / "shim"))
    from torch_geometric.utils import to_undirected
    from torch_geometric.utils.hetero import group_hetero_graph
    from efficient_gnns_b200 import synthetic
    ds = synthetic.make_mag_dataset(scale)
    eid = dict(ds["edge_index_dict"])
    r, c = eid[("author", "affiliated_with", "institution")]
    eid[("institution", "to", "author")] = torch.stack([c, r])
    r, c = eid[("author", "writes", "paper")]
    eid[("paper", "to", "author")] = torch.stack([c, r])
    r, c = eid[("paper", "has_topic", "field_of_study")]
    eid[("field_of_study", "to", "paper")] = torch.stack([c, r])
    eid[("paper", "cites", "paper")] = to_undirected(eid[("paper", "cites", "paper")])
    edge_index, edge_type, node_type, local_node_idx, local2global, key2int = group_hetero_graph(eid, ds["num_nodes_dict"])
    n = node_type.numel()
    homo = Data(edge_index=edge_index, edge_attr=edge_type, node_type=node_type, local_node_idx=local_node_idx, num_nodes=n)
    homo.y = node_type.new_full((n, 1), -1)
    homo.y[local2global["paper"]] = ds["y_dict"]["paper"]
    homo.train_mask = torch.zeros(n, dtype=torch.bool)
    homo.train_mask[local2global["paper"][ds["split_idx"]["train"]["paper"]]] = True
    num_nodes = {key2int[k]: v for k, v in ds["num_nodes_dict"].items()}
    rel_dst = [0] * len(eid)
    for k in eid:
        rel_dst[key2int[k]] = key2int[k[-1]]
    x_dict = {key2int["paper"]: ds["x_dict"]["paper"].cuda()}
    return homo, num_nodes, rel_dst, x_dict, key2int["paper"], ds["num_classes"]


def module_net(num_nodes, x_type, n_rels, hidden, classes):
    from test_rgcn_gpu import RelNet
    torch.manual_seed(0)
    net = RelNet(128, hidden, classes, num_nodes, [x_type], n_rels).cuda()
    for p in net.parameters():
        torch.nn.init.normal_(p, std=0.05)
    return net, torch.optim.Adam(net.parameters(), lr=0.005)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(gpu=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.stdout else None)


def grouped_vs_loop(tr: RGCNTrainer, reps: int = 20):
    """One grouped launch against the per-type loop of gemm_tf32x3 at the layer-0 root and the logits relation shapes."""
    G = tr._graph
    out = {}
    for name, a, c, groups, acc in (
            ("layer0_root_N32_K128", G.X[0], G.out[0], tr._groups(G, [f"root0_{t}" for t in range(tr.T)], bias_l=0), False),
            ("logits_rel_N352", G.M[1], G.out[1], tr._groups(G, [f"rel1_{t}" for t in range(tr.T)]), True)):
        def grouped():
            ops.gemm_tf32x3_grouped(a, c, groups, accumulate=acc)

        def loop():
            for r0, m, hi, lo, bias in groups:
                if m and hi is not None:
                    ops.gemm_tf32x3(a[r0:r0 + m, :hi.shape[1]], hi, lo, bias=bias, out=c[r0:r0 + m], accumulate=acc)
        for f in (grouped, loop):
            f()
        t_g, t_l = [], []
        for _ in range(reps):                                  # alternated
            t_g.append(timed(grouped)); t_l.append(timed(loop))
        out[name] = dict(grouped_ms=sorted(t_g)[reps // 2], per_type_loop_ms=sorted(t_l)[reps // 2],
                         loop_launches=sum(1 for _, m, hi, _, _ in groups if m and hi is not None))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=str(ROOT / "profiles"))
    ap.add_argument("--skip-module-full", action="store_true", help="do not time the module path on the whole graph")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    info = gpu_info()
    homo, num_nodes, rel_dst, x_dict, x_type, classes = mag_graph(args.scale)
    R = len(rel_dst)
    out_dir = Path(args.out)
    out_dir.mkdir(parents=True, exist_ok=True)
    dev = torch.device("cuda")
    full = homo.to(dev)
    train_idx = full.train_mask.nonzero().view(-1)

    def emit(name, rec):
        rec = dict(workload=name, scale=args.scale, **info, **rec)
        line = json.dumps(rec)
        print(line, flush=True)
        (out_dir / f"rgcn_train_{name}.json").write_text(line + "\n")

    # ---- full-graph student step
    st = RGCNTrainer(num_nodes, [x_type], R, rel_dst, 128, 32, classes, 2, dropout=0.5, lr=0.005)
    step = lambda: st.train_step(x_dict, full.edge_index, full.edge_attr, full.node_type, full.local_node_idx, full.y, train_idx)
    for _ in range(args.warmup):
        step()
    t_eng = [timed(step) for _ in range(args.steps)]
    rec = dict(n_nodes=full.num_nodes, n_edges=int(full.edge_index.size(1)), engine_ms=sorted(t_eng)[len(t_eng) // 2],
               engine_ms_all=t_eng, launches_per_step=st.launches_per_step(), loss=float(st.loss_out[0]),
               grouped_gemm=grouped_vs_loop(st))
    if not args.skip_module_full:
        try:
            net, opt = module_net(num_nodes, x_type, R, 32, classes)
            tm = train_idx

            def mstep():
                opt.zero_grad()
                o = net(x_dict, full.edge_index, full.edge_attr, full.node_type, full.local_node_idx)[tm]
                F.cross_entropy(o, full.y.view(-1)[tm]).backward()
                opt.step()
            mstep()
            before = lib.launch_count()
            rec["module_ms"] = timed(mstep)
            rec["module_b200gnn_launches"] = lib.launch_count() - before
        except torch.cuda.OutOfMemoryError as e:
            rec["module_ms"] = None
            rec["module_error"] = f"out of memory: {str(e).splitlines()[0]}"
        torch.cuda.empty_cache()
    emit("full_graph_student", rec)
    del st
    torch.cuda.empty_cache()

    # ---- GraphSAINT batches, without and with the KD teacher
    loader = sampling.GraphSAINTRandomWalkSampler(full, batch_size=20000, walk_length=2, num_steps=args.warmup + args.steps, seed=0)
    batches = list(loader)
    for kd in (False, True):
        st = RGCNTrainer(num_nodes, [x_type], R, rel_dst, 128, 32, classes, 2, dropout=0.5, lr=0.005)
        teacher = RGCNTrainer(num_nodes, [x_type], R, rel_dst, 128, 512, classes, 3, dropout=0.5, seed=1) if kd else None
        net, opt = module_net(num_nodes, x_type, R, 32, classes)
        tnet = None
        if kd:
            from test_rgcn_gpu import RelConv
            tnet = module_net(num_nodes, x_type, R, 512, classes)[0]
            tnet.convs.insert(1, RelConv(512, 512, len(num_nodes), R).cuda())
            tnet.load_state_dict(teacher.state_dict())
            tnet.eval()
        t_e, t_m, launches = [], [], []
        for i, b in enumerate(batches):
            tidx = b.train_mask.nonzero().view(-1)

            def estep():
                t = teacher.forward(x_dict, b.edge_index, b.edge_attr, b.node_type, b.local_node_idx) if kd else None
                st.train_step(x_dict, b.edge_index, b.edge_attr, b.node_type, b.local_node_idx, b.y, tidx, teacher_logits=t)

            def mstep():
                opt.zero_grad()
                o = net(x_dict, b.edge_index, b.edge_attr, b.node_type, b.local_node_idx)[b.train_mask]
                lab = b.y[b.train_mask].squeeze(1)
                if kd:
                    with torch.no_grad():
                        h = tnet.convs[0](efficient_gnns_b200.nn.group_input(x_dict, tnet.emb_dict, b.node_type,
                                                                               b.local_node_idx, 128), b.edge_index, b.edge_attr, b.node_type)
                        for conv in tnet.convs[1:]:
                            h = conv(F.relu(h), b.edge_index, b.edge_attr, b.node_type)
                        to = h[b.train_mask]
                    T = 4.0
                    loss_cls = F.cross_entropy(o, lab)
                    loss_kd = F.kl_div(F.log_softmax(o / T, 1), F.softmax(to / T, 1), reduction="batchmean") * T * T
                    (0.1 * loss_cls + 0.9 * loss_kd).backward()
                else:
                    F.cross_entropy(o, lab).backward()
                opt.step()
            before = lib.launch_count()
            te = timed(estep)
            launches.append(lib.launch_count() - before)
            tm = timed(mstep)
            if i >= args.warmup:
                t_e.append(te); t_m.append(tm)
        name = "saint_batch_kd" if kd else "saint_batch_supervised"
        emit(name, dict(batch_size=20000, walk_length=2, batch_nodes=[int(b.num_nodes) for b in batches[args.warmup:]],
                        engine_ms=sorted(t_e)[len(t_e) // 2], engine_ms_all=t_e, module_ms=sorted(t_m)[len(t_m) // 2],
                        module_ms_all=t_m, launches_per_step=launches[-1], loss=float(st.loss_out[0])))
        del st, teacher, net, opt, tnet
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
