"""Fused R-GCN training engine (rgcn.RGCNTrainer) and the node-type-grouped tcgen05 GEMM under it: against the fixture made
by the reference's own RGCN class, a fp64 restatement of one train() step, the inference engine, and the module path."""
import pytest
import torch

import efficient_gnns_b200  # noqa: F401
from conftest import rel_err
from efficient_gnns_b200 import lib, ops, sampling
from efficient_gnns_b200.graphdata import Data
from efficient_gnns_b200.rgcn import RGCNInference, RGCNTrainer
from oracle import rgcn_train as ort

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]


# ------------------------------------------------------------------ grouped GEMM
def _grouped_case(N, groups, strided, seed):
    """groups: [(rows, K, bias)]; A / C row-strided when `strided`."""
    g = torch.Generator().manual_seed(seed)
    Kmax = max(k for _, k, _ in groups)
    n = sum(m for m, _, _ in groups)
    lda = Kmax + (12 if strided else 0)
    ldc = N + (8 if strided else 0)
    A = torch.randn(n, lda, generator=g).cuda()[:, :Kmax]
    C0 = torch.randn(n, ldc, generator=g).cuda()[:, :N]
    Bs = [torch.randn(N, k, generator=g).cuda() * 0.1 for _, k, _ in groups]
    biases = [torch.randn(N, generator=g).cuda() if b else None for _, _, b in groups]
    return A, C0, Bs, biases


@pytest.mark.parametrize("N", [8, 32, 352, 512])
@pytest.mark.parametrize("accumulate", [False, True])
def test_grouped_gemm_bit_identical_to_per_group_launches_and_fp64(N, accumulate):
    spec = [(300, 20, True), (0, 36, True), (129, 128, False), (517, 384, True), (64, 0, True)]   # K=0: no relation
    A, C0, Bs, biases = _grouped_case(N, spec, strided=True, seed=N)
    C = C0.clone()
    groups, r0, want = [], 0, C0.clone()
    for (m, k, _), B, b in zip(spec, Bs, biases):
        bias = None if accumulate else b
        hi, lo = ops.split_tf32(B) if k else (None, None)
        groups.append((r0, m, hi, lo, bias))
        if m and k:                                                   # the plain kernel on contiguous copies
            o = want[r0:r0 + m].contiguous()
            ops.gemm_tf32x3(A[r0:r0 + m, :k].contiguous(), hi, lo, bias=bias, out=o, accumulate=accumulate)
            want[r0:r0 + m] = o
        elif m and not accumulate:
            want[r0:r0 + m] = 0 if bias is None else bias
        r0 += m
    before = lib.launch_count()
    ops.gemm_tf32x3_grouped(A, C, groups, accumulate=accumulate)
    assert lib.launch_count() - before == 1
    torch.cuda.synchronize()
    assert torch.equal(C, want)
    r0 = 0
    for (m, k, _), B, b in zip(spec, Bs, biases):
        ref = (C0[r0:r0 + m].double() if accumulate else 0) + (A[r0:r0 + m, :k].double() @ B.double().t() if k else 0)
        if not accumulate and b is not None:
            ref = ref + b.double()
        if m:
            assert rel_err(C[r0:r0 + m], torch.as_tensor(ref).expand(m, N)) < 1e-5
        r0 += m


# ------------------------------------------------------------------ against the reference class fixture
def _fixture_trainer(G, **kw):
    rel_dst = [d for _, d, _ in G["rels"]]
    tr = RGCNTrainer(G["num_nodes"], [0], len(G["rels"]), rel_dst, 16, 24, 5, 2, dropout=0.0, **kw)
    tr.load_state_dict(G["state"])
    return tr


def _cuda(*ts):
    return [t.cuda() for t in ts]


def test_forward_and_gradients_match_reference_class_fixture(golden_rgcn):
    G = golden_rgcn
    tr = _fixture_trainer(G)
    ei, et, nt, li = _cuda(G["edge_index"], G["edge_type"], G["node_type"], G["local_node_idx"])
    out = tr.forward({0: G["x_paper"].cuda()}, ei, et, nt, li)
    assert rel_err(out, G["out_forward"]) < 1e-5
    assert rel_err(tr.out_feat(), G["out_feat"]) < 1e-5
    tr.backward(G["w"].cuda())
    grads = tr.gradients()
    assert set(grads) == set(G["grads"])
    for k, want in G["grads"].items():
        assert rel_err(grads[k], want) < 5e-5, k


def test_non_grouped_node_type_is_rejected_before_any_launch(golden_rgcn):
    G = golden_rgcn
    tr = _fixture_trainer(G)
    ei, et, nt, li = _cuda(G["edge_index"], G["edge_type"], G["node_type"], G["local_node_idx"])
    perm = torch.randperm(nt.numel(), generator=torch.Generator().manual_seed(0)).cuda()
    before = lib.launch_count()
    with pytest.raises(lib.B200GnnError, match="grouped by node type"):
        tr.train_step({0: G["x_paper"].cuda()}, ei, et, nt[perm], li[perm], torch.zeros_like(nt), torch.arange(5, device="cuda"))
    assert lib.launch_count() == before


def test_inference_engine_reads_the_trained_state_dict(golden_rgcn):
    G = golden_rgcn
    tr = _fixture_trainer(G, lr=0.01)
    tr.p = 0.5
    ei, et, nt, li = _cuda(G["edge_index"], G["edge_type"], G["node_type"], G["local_node_idx"])
    x = {0: G["x_paper"].cuda()}
    y = torch.randint(0, 5, (nt.numel(),), generator=torch.Generator().manual_seed(1)).cuda()
    for _ in range(3):
        tr.train_step(x, ei, et, nt, li, y, torch.arange(60, device="cuda"))
    out = tr.forward(x, ei, et, nt, li).clone()
    inf = RGCNInference(tr.state_dict(), G["num_nodes"], G["edge_index_dict"], G["key2int"])({0: G["x_paper"]})
    off = 0
    for t in range(3):
        n_t = G["num_nodes"][t]
        assert rel_err(out[off:off + n_t], inf[t]) < 1e-5
        off += n_t


# ------------------------------------------------------------------ one step against the fp64 restatement
NODES = {0: 80, 1: 60, 2: 30}
RELS = [(1, 0, 150), (0, 0, 500), (2, 1, 70), (0, 2, 0), (0, 1, 120)]      # (src, dst, edges): relation 3 has no edges


def _small_graph():
    g = torch.Generator().manual_seed(5)
    off = {0: 0, 1: 80, 2: 140}
    eis, ets = [], []
    for r, (s, d, e) in enumerate(RELS):
        src = torch.randint(0, NODES[s], (e,), generator=g)
        dst = torch.randint(0, NODES[d] // 2, (e,), generator=g)   # the upper half of each type gets no edges of r
        if r == 1:
            dst[:300] = 3                                            # a hub destination (> 256 edges)
        eis.append(torch.stack([src + off[s], dst + off[d]]))
        ets.append(torch.full((e,), r, dtype=torch.long))
    nt = torch.cat([torch.full((NODES[t],), t, dtype=torch.long) for t in range(3)])
    li = torch.cat([torch.arange(NODES[t]) for t in range(3)])
    x0 = torch.randn(NODES[0], 10, generator=g)
    y = torch.randint(0, 7, (nt.numel(), 1), generator=g)
    train_idx = torch.randperm(NODES[0], generator=g)[:50].sort().values
    teacher = torch.randn(nt.numel(), 7, generator=g) * 3
    return torch.cat(eis, 1), torch.cat(ets), nt, li, x0, y, train_idx, teacher


@pytest.mark.parametrize("kd", [False, True], ids=["supervised", "kd"])
def test_train_step_matches_fp64_restatement(kd):
    ei, et, nt, li, x0, y, train_idx, teacher = _small_graph()
    L, p, lr, seed = 2, 0.5, 0.01, 3
    tr = RGCNTrainer(NODES, [0], len(RELS), [d for _, d, _ in RELS], 10, 13, 7, L, dropout=p, lr=lr, seed=seed)
    state = tr.state_dict()
    m = {k: torch.zeros_like(v).double().cpu() for k, v in state.items()}
    v = {k: torch.zeros_like(v).double().cpu() for k, v in state.items()}
    ref_state = {k: t.double().cpu() for k, t in state.items()}
    n = nt.numel()
    # step 1 on the whole graph, step 2 on a sub-graph that leaves out part of type 2: its embedding rows get no gradient
    keep = torch.cat([torch.arange(140), torch.arange(140, 170, 2)])
    sub_map = torch.full((n,), -1, dtype=torch.long)
    sub_map[keep] = torch.arange(keep.numel())
    emask = (sub_map[ei[0]] >= 0) & (sub_map[ei[1]] >= 0)
    batches = [(ei, et, nt, li, y, train_idx, teacher),
               (sub_map[ei[:, emask]], et[emask], nt[keep], li[keep], y[keep], train_idx, teacher[keep])]
    x_dict = {0: x0.cuda()}
    after = []
    for step, (bei, bet, bnt, bli, by, btr, bte) in enumerate(batches):
        masks = [ops.dropout_mask(bnt.numel(), tr.dp[l + 1], p, seed, l + step * L).cpu()[:, :13] for l in range(L - 1)]
        loss = tr.train_step(x_dict, *_cuda(bei, bet, bnt, bli, by, btr), teacher_logits=bte.cuda() if kd else None).clone()
        logits, grads = tr.logits().clone(), tr.gradients()
        m_prev = {k: t.clone() for k, t in m.items()}
        rl, rc, rk, rlog, ref_state = ort.train_step(ref_state, m, v, step + 1, {0: x0}, bei, bet, bnt, bli, by, btr, 3, len(RELS),
                                                     L, 10, lr, masks=masks, p=p, teacher_logits=bte if kd else None)
        assert rel_err(loss, torch.stack([rl, rc, rk])) < 1e-5
        assert rel_err(logits, rlog) < 1e-5
        got = tr.state_dict()
        after.append(got)
        for k in state:
            g_ref = (m[k] - 0.9 * m_prev[k]) / 0.1                      # this step's fp64 gradient
            assert rel_err(grads[k], g_ref) < 1e-4, (step, k)
            # Adam moves an element by ~lr·m/sqrt(v): compare where the first moment is above fp32 noise
            big = m[k].abs() > 1e-4 * m[k].abs().max().clamp(min=1e-30)
            if big.any():
                assert (got[k].double().cpu() - ref_state[k])[big].abs().max().item() < 1e-5, (step, k)
    # rows of type 2 outside the second batch had no gradient there, yet moved (their moments decay, as in torch Adam)
    out_rows = torch.arange(1, 30, 2)
    had_grad = (m["emb_dict.2"][out_rows].abs() > 0).any(1)
    assert had_grad.any()
    moved = (after[1]["emb_dict.2"][out_rows] != after[0]["emb_dict.2"][out_rows]).any(1).cpu()
    assert torch.equal(moved, had_grad)


# ------------------------------------------------------------------ against the module path on GraphSAINT batches
def test_tracks_module_path_on_graphsaint_batches_and_learns():
    import torch.nn.functional as F
    from test_rgcn_gpu import RelNet
    g = torch.Generator().manual_seed(0)
    n_paper, n_author = 1500, 900
    n = n_paper + n_author
    node_type = torch.cat([torch.zeros(n_paper, dtype=torch.long), torch.ones(n_author, dtype=torch.long)])
    local_idx = torch.cat([torch.arange(n_paper), torch.arange(n_author)])
    cites = torch.randint(0, n_paper, (2, 6000), generator=g)
    writes = torch.stack([torch.randint(0, n_author, (5000,), generator=g) + n_paper, torch.randint(0, n_paper, (5000,), generator=g)])
    edge_index = torch.cat([cites, writes, writes.flip(0)], 1)
    edge_type = torch.cat([torch.zeros(6000), torch.ones(5000), torch.full((5000,), 2.0)]).long()
    x_paper = torch.randn(n_paper, 16, generator=g)
    y = torch.full((n, 1), -1, dtype=torch.long)
    y[:n_paper, 0] = (x_paper @ torch.randn(16, 5, generator=g)).argmax(1)
    train_mask = torch.zeros(n, dtype=torch.bool)
    train_mask[:n_paper] = torch.rand(n_paper, generator=g) < 0.6
    data = Data(edge_index=edge_index, edge_attr=edge_type, node_type=node_type, local_node_idx=local_idx, y=y, train_mask=train_mask)
    data.num_nodes = n
    loader = sampling.GraphSAINTRandomWalkSampler(data.to("cuda"), batch_size=400, walk_length=2, num_steps=3, seed=1)
    torch.manual_seed(0)
    model = RelNet(16, 32, 5, {0: n_paper, 1: n_author}, [0], 3).cuda()
    for prm in model.parameters():
        torch.nn.init.normal_(prm, std=0.1)
    opt = torch.optim.Adam(model.parameters(), lr=0.01)
    tr = RGCNTrainer({0: n_paper, 1: n_author}, [0], 3, [0, 0, 1], 16, 32, 5, 2, dropout=0.0, lr=0.01)
    tr.load_state_dict(model.state_dict())
    x_dict = {0: x_paper.cuda()}
    batches = list(loader)
    for b in batches:
        train_idx = b.train_mask.nonzero().view(-1)
        loss = tr.train_step(x_dict, b.edge_index, b.edge_attr, b.node_type, b.local_node_idx, b.y, train_idx).clone()
        opt.zero_grad()
        out = model(x_dict, b.edge_index, b.edge_attr, b.node_type, b.local_node_idx)[b.train_mask]
        ref = F.cross_entropy(out, b.y[b.train_mask].squeeze(1))
        ref.backward()
        opt.step()
        assert abs(loss[0].item() - ref.item()) <= 1e-4 * abs(ref.item())
    sd = tr.state_dict()
    for k, prm in model.state_dict().items():
        assert rel_err(sd[k], prm) < 1e-4, k
    losses = []
    for epoch in range(6):
        tot = cnt = 0
        for b in loader:
            train_idx = b.train_mask.nonzero().view(-1)
            tot += tr.train_step(x_dict, b.edge_index, b.edge_attr, b.node_type, b.local_node_idx, b.y, train_idx)[0].item() * train_idx.numel()
            cnt += train_idx.numel()
        losses.append(tot / cnt)
    assert losses[-1] < 0.8 * losses[0], losses
    assert tr.launches_per_step() > 0
