"""Representation distillation (FitNet, AT, LSP, GSP, G-CRD) on the fused R-GCN engine: the ReLU/dropout backward with an
added upstream gradient, RGCNTrainer.train_step(aux=, beta=) against the fixture made by the reference's own MAG train()
loops, against the fp64 restatement with the engine's dropout masks, and against the module path on GraphSAINT batches."""
import numpy as np
import pytest
import torch

import efficient_gnns_b200  # noqa: F401
from conftest import rel_err
from efficient_gnns_b200 import criterion as C
from efficient_gnns_b200 import lib, ops, sampling
from efficient_gnns_b200 import nn as bnn
from efficient_gnns_b200.graphdata import Data
from efficient_gnns_b200.rgcn import RGCNTrainer
from test_rgcn_distill_cpu import (CASES, check_grads, draw_sample, golden_distill, head_params, heads,  # noqa: F401
                                   make_aux, replay_fp64, roundoff_keys, weighted_triple)

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]


# ------------------------------------------------------------------ kernel
@pytest.mark.parametrize("k_extra", [13, 32])
@pytest.mark.parametrize("p", [0.0, 0.5])
def test_relu_dropout_bwd_add_is_the_plain_kernel_on_the_sum(k_extra, p):
    g = torch.Generator().manual_seed(k_extra)
    n, K = 1000, 36
    y = torch.randn(n, K, generator=g)
    keep = (torch.rand(n, K, generator=g) >= p).float()
    x_out = (y.relu() * keep / (1 - p)).cuda()
    d_out = torch.randn(n, K, generator=g).cuda()
    base = torch.randn(n, k_extra + 7, generator=g).cuda()
    extra = base[:, 1:1 + k_extra]                                     # row-strided, not 16-byte aligned
    want = ops.relu_dropout_bwd(d_out + torch.nn.functional.pad(extra, (0, K - k_extra)), x_out, p)
    got = ops.relu_dropout_bwd(d_out, x_out, p, extra=extra)
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    ref = (d_out.double() + torch.nn.functional.pad(extra.double(), (0, K - k_extra))) * (x_out > 0).double() / (1 - p)
    assert rel_err(got, ref) < 1e-6
    inplace = d_out.clone()
    ops.relu_dropout_bwd(inplace, x_out, p, out=inplace, extra=extra)
    assert torch.equal(inplace, want)
    before = lib.launch_count()
    e = torch.empty(0, K, device="cuda")
    ops.relu_dropout_bwd(e, e, p, out=e, extra=torch.empty(0, k_extra, device="cuda"))
    assert lib.launch_count() == before


# ------------------------------------------------------------------ against the reference's train()
def _batch(b):
    return [b[k].cuda() for k in ("edge_index", "edge_attr", "node_type", "local_node_idx", "y", "train_mask")]


def _trainers(G, p=0.0, seed=0):
    d, R = G["dims"], len(G["rels"])
    rel_dst = [dd for _, dd, _ in G["rels"]]
    mk = lambda hid, L: RGCNTrainer(G["num_nodes"], [0], R, rel_dst, d["in_channels"], hid, d["out_channels"], L,  # noqa: E731
                                    dropout=p, lr=G["lr"], alpha=G["alpha"], kd_T=G["kd_T"], seed=seed)
    tr, teacher = mk(d["hidden"], 2), mk(d["teacher_hidden"], 3)
    tr.load_state_dict(G["student"])
    teacher.load_state_dict(G["teacher"])
    return tr, teacher


def replay_engine(G, case, p=0.0, seed=0):
    """The fixture's two batches through the engine, b200gnn criteria, fp32 torch heads and torch Adam on the heads."""
    tr, teacher = _trainers(G, p, seed)
    sp, tp = heads(G, "cuda", torch.float32) if case["heads"] else (None, None)
    opt = torch.optim.Adam([q for _, q in head_params(sp, tp)], lr=G["lr"]) if case["heads"] else None
    x = {0: G["x_paper"].float().cuda()}
    np.random.seed(G["np_seed"])
    steps = []
    for b in G["batches"]:
        ei, et, nt, li, y, mask = _batch(b)
        train_idx = mask.nonzero().view(-1)
        labels = y.view(-1)[train_idx]
        t_logits = teacher.forward(x, ei, et, nt, li).clone()
        t_feat = teacher.out_feat()[train_idx].clone()
        edges = bnn.subgraph(train_idx, ei, relabel_nodes=True)[0] if case["training"] == "lpw" else None
        aux = make_aux(C, case, train_idx, labels, t_feat, edges, draw_sample(case, train_idx.numel()), sp, tp)
        loss = tr.train_step(x, ei, et, nt, li, y, train_idx, teacher_logits=t_logits if case["form"] == "kd_aux" else None,
                             aux=lambda f: aux(f, tr.logits()), beta=case["beta"]).clone()
        grads = tr.gradients()
        if opt is not None:
            grads.update({k: q.grad.detach().clone() for k, q in head_params(sp, tp)})
            opt.step()
            opt.zero_grad()
        steps.append((loss[0], loss[1], loss[2], tr.loss_aux.clone(), grads, train_idx.numel()))
    return steps, tr, (sp, tp)


def _first_moments(grads_per_step):
    m = {k: torch.zeros_like(t) for k, t in grads_per_step[0].items()}
    for g in grads_per_step:
        m = {k: 0.9 * m[k] + 0.1 * g[k] for k in m}
    return m


def _check_states(got, want, m, noise):
    """Adam moves an element by ~lr·m/sqrt(v): compare where the first moment is above fp32 noise."""
    for k, w in want.items():
        if k in noise:
            continue
        big = m[k].abs() > 1e-4 * m[k].abs().max().clamp(min=1e-30)
        if big.any():
            assert (got[k].double().cpu() - w.double())[big].abs().max().item() < 1e-5, k


@pytest.mark.parametrize("name", CASES)
def test_engine_replays_reference_train(golden_distill, name):
    G = golden_distill
    case = G["cases"][name]
    tol = 1e-4 if case["training"] == "nce" else 5e-5
    steps, tr, (sp, tp) = replay_engine(G, case)
    assert rel_err(weighted_triple(steps), case["result"]) < (1e-4 if case["training"] == "nce" else 1e-5)
    noise = roundoff_keys(case["grads"])
    for s, want in enumerate(case["grads"]):
        check_grads(steps[s][4], want, tol, noise)
    m = _first_moments(case["grads"])
    _check_states(tr.state_dict(), case["final"], m, noise)
    if case["heads"]:
        for name_h, mod in (("student_proj", sp), ("teacher_proj", tp)):
            got = {f"{name_h}.{k}": v for k, v in mod.named_parameters()}
            _check_states(got, {k: case["final_heads"][name_h][k.split(".", 1)[1]] for k in got}, m, noise)


# ------------------------------------------------------------------ dropout: the injected gradient goes through the mask
@pytest.mark.parametrize("name", ["gnn/lpw_rbf", "kd_aux/nce"])
def test_aux_gradient_passes_the_engine_dropout_mask(golden_distill, name):
    G = golden_distill
    case = G["cases"][name]
    p, seed = 0.5, 5
    hid = G["dims"]["hidden"]
    masks_of = lambda s: [ops.dropout_mask(G["batches"][s]["node_type"].numel(), (hid + 3) // 4 * 4, p, seed, s * 2)  # noqa: E731
                          .cpu()[:, :hid]]
    got, _, _ = replay_engine(G, case, p=p, seed=seed)
    want, _, _ = replay_fp64(G, case, masks_of=masks_of, p=p)
    tol = 1e-4 if case["training"] == "nce" else 5e-5
    noise = roundoff_keys([w[4] for w in want])
    for (l0, lc, lk, la, g, _), (r0, rc, rk, ra, rg, _) in zip(got, want):
        assert rel_err(torch.stack([l0, lc, lk, la]), torch.stack([r0, rc, rk, ra])) < (1e-4 if case["training"] == "nce" else 1e-5)
        check_grads(g, rg, tol, noise)


# ------------------------------------------------------------------ the plain step is unchanged
def _fixture_step_args(G):
    ei, et, nt, li, y, mask = _batch(G["batches"][0])
    return {0: G["x_paper"].float().cuda()}, ei, et, nt, li, y, mask.nonzero().view(-1)


def test_aux_without_gradient_leaves_the_step_bit_identical(golden_distill):
    G = golden_distill
    args = _fixture_step_args(G)
    a, _ = _trainers(G, p=0.5, seed=2)
    b, _ = _trainers(G, p=0.5, seed=2)
    for _ in range(2):
        la = a.train_step(*args).clone()
        lb = b.train_step(*args, aux=lambda f: 0 * f.sum(), beta=3.0).clone()
        torch.cuda.synchronize()
        assert torch.equal(la, lb)
        assert torch.equal(a.params, b.params) and torch.equal(a.grads, b.grads)
        assert torch.equal(a.exp_avg, b.exp_avg) and torch.equal(a.exp_avg_sq, b.exp_avg_sq)
    assert float(b.loss_aux) == 0.0


def test_aux_needs_a_hidden_layer_and_is_rejected_before_any_launch(golden_distill):
    G = golden_distill
    d, R = G["dims"], len(G["rels"])
    tr = RGCNTrainer(G["num_nodes"], [0], R, [dd for _, dd, _ in G["rels"]], d["in_channels"], d["hidden"], d["out_channels"], 1)
    before = lib.launch_count()
    with pytest.raises(lib.B200GnnError, match="hidden layer"):
        tr.train_step(*_fixture_step_args(G), aux=lambda f: f.sum())
    assert lib.launch_count() == before


def test_launches_per_step_counts_the_aux_step(golden_distill):
    G = golden_distill
    args = _fixture_step_args(G)
    tr, _ = _trainers(G)
    tr.train_step(*args)
    plain = tr.launches_per_step()
    train_idx, labels = args[-1], args[5].view(-1)[args[-1]]
    t_feat = torch.rand(train_idx.numel(), G["dims"]["teacher_hidden"], device="cuda")
    tr.train_step(*args, aux=lambda f: C.at_criterion(tr.logits()[train_idx], labels, f[train_idx], t_feat, 1.0)[2], beta=2.0)
    with_aux = tr.launches_per_step()
    assert with_aux > plain > 0


# ------------------------------------------------------------------ against the module path on GraphSAINT batches
def _saint_setup():
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
    return {0: n_paper, 1: n_author}, {0: x_paper.cuda()}, list(loader)


@pytest.mark.parametrize("mode", ["gpw_poly", "nce"])
def test_tracks_module_path_with_aux_on_graphsaint_batches(mode):
    from test_rgcn_gpu import RelNet
    nodes, x_dict, batches = _saint_setup()
    kd = mode == "nce"                                   # gpw-poly in the gnn.py form, nce in the gnn_kd_and_aux.py form
    beta, lr, alpha, T = (100.0 if mode == "gpw_poly" else 0.5), 0.01, 0.9, 4.0
    torch.manual_seed(0)
    model = RelNet(16, 32, 5, nodes, [0], 3).cuda()
    for prm in model.parameters():
        torch.nn.init.normal_(prm, std=0.1)
    mk = lambda i: torch.nn.Sequential(torch.nn.Linear(i, 24), torch.nn.BatchNorm1d(24), torch.nn.ReLU()).cuda()  # noqa: E731
    heads_m = (mk(32), mk(48)) if kd else ()
    heads_e = (mk(32), mk(48)) if kd else ()
    for a, b in zip(heads_e, heads_m):
        a.load_state_dict(b.state_dict())
    hp = lambda hs: [q for h in hs for q in h.parameters()]  # noqa: E731
    opt = torch.optim.Adam(list(model.parameters()) + hp(heads_m), lr=lr)
    opt_h = torch.optim.Adam(hp(heads_e), lr=lr) if kd else None
    tr = RGCNTrainer(nodes, [0], 3, [0, 0, 1], 16, 32, 5, 2, dropout=0.0, lr=lr, alpha=alpha, kd_T=T)
    tr.load_state_dict(model.state_dict())
    teacher = RGCNTrainer(nodes, [0], 3, [0, 0, 1], 16, 48, 5, 3, dropout=0.0, seed=1)

    def aux_of(f, z, labels, t_feat, hs):
        if mode == "gpw_poly":
            return C.gpw_criterion(z, labels, f, t_feat, "poly", beta, 10 ** 9)[2]
        return C.nce_criterion(z, labels, hs[0](f), hs[1](t_feat), beta, 0.075, 10 ** 9)[2]

    for b in batches:
        train_idx = b.train_mask.nonzero().view(-1)
        labels = b.y.view(-1)[train_idx]
        gargs = (b.edge_index, b.edge_attr, b.node_type, b.local_node_idx)
        t_logits = teacher.forward(x_dict, *gargs).clone()
        t_feat = teacher.out_feat()[train_idx].clone()
        loss = tr.train_step(x_dict, *gargs, b.y, train_idx, teacher_logits=t_logits if kd else None,
                             aux=lambda f: aux_of(f[train_idx], tr.logits()[train_idx], labels, t_feat, heads_e), beta=beta).clone()
        if kd:
            opt_h.step(); opt_h.zero_grad()
        opt.zero_grad()
        out = model(x_dict, *gargs)[train_idx]
        cls = C.kd_criterion(out, labels, t_logits[train_idx], alpha, T)[0] if kd else C.cross_entropy(out, labels)
        ref = cls + beta * aux_of(model.out_feat[train_idx], out.detach(), labels, t_feat, heads_m)
        ref.backward()
        opt.step()
        assert abs(loss[0].item() - ref.item()) <= 1e-4 * abs(ref.item())
    # Adam scales every element by its own gradient history: compare where the module path's first moment is above fp32
    # noise.  InfoNCE at T = 0.075 multiplies logit differences by 13; as in test_engine_gpu.py its tolerance is twice the
    # others'.  Parameters that no training row reaches (zero moments) must not move at all.
    sd = tr.state_dict()
    tol = 2e-4 if mode == "nce" else 1e-4
    for k, prm in model.named_parameters():
        m = opt.state[prm]["exp_avg"]
        big = m.abs() > 1e-4 * m.abs().max().clamp(min=1e-30)
        if big.any():
            assert rel_err(sd[k][big], prm.detach()[big]) < tol, k
        else:
            assert torch.equal(sd[k], prm.detach()), k
    for he, hm in zip(heads_e, heads_m):
        for (k, a), (_, b) in zip(he.named_parameters(), hm.named_parameters()):
            if k != "0.bias":                             # round-off gradient before BatchNorm: Adam moves it by lr·sign
                assert rel_err(a, b) < 1e-4, k
