"""Representation distillation on the R-GCN student, the parts that need no GPU: the fp64 restatement of one step with an
auxiliary loss (oracle/rgcn_distill.distill_step) against the fixture made by the reference's own MAG train() loops
(tests/golden/make_golden_rgcn_distill.py), and its reduction to the plain step at beta = 0."""
import math
from pathlib import Path

import numpy as np
import pytest
import torch

import efficient_gnns_b200  # noqa: F401
from conftest import rel_err
from oracle import criterion as oc
from oracle import graph as og
from oracle import rgcn_distill as odi
from oracle import rgcn_train as ort

GOLDEN = Path(__file__).resolve().parent / "golden" / "rgcn_distill_mag.pt"
CASES = sorted(torch.load(GOLDEN, weights_only=False)["cases"])


def _unflatten(vec, layout):
    out, o = {}, 0
    for k, shape in layout:
        n = math.prod(shape)
        out[k] = vec[o:o + n].view(shape).double()
        o += n
    return out


def load_fixture():
    """The fixture with each case's flat fp32 vectors expanded into {key: tensor} per step (gradients, heads included),
    ``final`` {key: tensor} and ``final_heads`` {head: state dict}."""
    G = torch.load(GOLDEN, weights_only=False)
    for case in G["cases"].values():
        steps = [_unflatten(g, G["layout"]) for g in case["grads"]]
        if case["heads"]:
            for st, hg in zip(steps, case["head_grads"]):
                st.update(_unflatten(hg, G["head_layout"]))
            hs = _unflatten(case["final_heads"], G["head_state_layout"])
            case["final_heads"] = {h: {k.split(".", 1)[1]: v for k, v in hs.items() if k.startswith(h + ".")}
                                   for h in ("student_proj", "teacher_proj")}
        case["grads"] = steps
        case["final"] = _unflatten(case["final"], G["layout"])
    return G


@pytest.fixture(scope="session")
def golden_distill():
    return load_fixture()


def heads(G, device="cpu", dtype=torch.float64):
    """The reference's student_proj / teacher_proj (Linear -> BatchNorm1d -> ReLU) at the fixture's initial state."""
    d = G["dims"]
    mk = lambda i: torch.nn.Sequential(torch.nn.Linear(i, d["proj_dim"]), torch.nn.BatchNorm1d(d["proj_dim"]),  # noqa: E731
                                       torch.nn.ReLU()).to(device, dtype)
    sp, tp = mk(d["hidden"]), mk(d["teacher_hidden"])
    sp.load_state_dict(G["heads"]["student_proj"]); tp.load_state_dict(G["heads"]["teacher_proj"])
    return sp.train(), tp.train()


def head_params(sp, tp):
    return [(f"student_proj.{k}", p) for k, p in sp.named_parameters()] + [(f"teacher_proj.{k}", p) for k, p in tp.named_parameters()]


def draw_sample(case, m: int):
    """The row sample gpw / nce draw from numpy's global RNG when max_samples < m (criterion.py:62-64, 134-136)."""
    if case["training"] in ("gpw", "nce") and case["max_samples"] < m:
        return torch.as_tensor(np.random.choice(m, case["max_samples"], replace=False), dtype=torch.long)
    return None


def make_aux(crit, case, train_idx, labels, t_feat, edges=None, sampled=None, sp=None, tp=None):
    """aux(feat, logits) of one train() branch (mag_pyg/gnn.py:204-251) on the criterion module ``crit`` (oracle.criterion in
    fp64, efficient_gnns_b200.criterion on the device): the auxiliary loss on feat[train_idx], through the heads if any."""
    kind, beta = case["training"], case["beta"]

    def aux(feat, logits):
        f, z, tf = feat[train_idx], logits[train_idx].detach(), t_feat
        if case["heads"]:
            f, tf = sp(f), tp(tf)
        if kind == "fitnet":
            return crit.fitnet_criterion(z, labels, f, tf, beta)[2]
        if kind == "at":
            return crit.at_criterion(z, labels, f, tf, beta)[2]
        if kind == "lpw":
            return crit.lpw_criterion(z, labels, f, tf, edges, case["kernel"], beta)[2]
        if kind == "gpw":
            return crit.gpw_criterion(z, labels, f, tf, case["kernel"], beta, case["max_samples"], sampled)[2]
        return crit.nce_criterion(z, labels, f, tf, beta, case["nce_T"], case["max_samples"], sampled)[2]
    return aux


def _oracle_args(G, b):
    return {0: G["x_paper"]}, b["edge_index"], b["edge_attr"], b["node_type"], b["local_node_idx"]


def replay_fp64(G, case, masks_of=None, p: float = 0.0):
    """Both fixture batches through distill_step + fp64 heads under torch Adam.  Returns per step (loss, loss_cls, loss_kd,
    loss_aux, grads incl. heads), the final state and heads."""
    d, R = G["dims"], len(G["rels"])
    state = {k: v.clone() for k, v in G["student"].items()}
    m = {k: torch.zeros_like(v) for k, v in state.items()}
    v = {k: torch.zeros_like(t) for k, t in state.items()}
    sp, tp = heads(G) if case["heads"] else (None, None)
    opt = torch.optim.Adam([q for _, q in head_params(sp, tp)], lr=G["lr"]) if case["heads"] else None
    np.random.seed(G["np_seed"])
    steps = []
    for s, b in enumerate(G["batches"]):
        args = _oracle_args(G, b)
        train_idx = b["train_mask"].nonzero().view(-1)
        labels = b["y"].view(-1)[train_idx]
        with torch.no_grad():
            t_logits, t_feat = ort.rgcn_forward(G["teacher"], *args, 3, R, 3, d["in_channels"])
        edges = torch.from_numpy(og.subgraph(train_idx.numpy(), b["edge_index"].numpy(), True)[0]) if case["training"] == "lpw" else None
        aux = make_aux(oc, case, train_idx, labels, t_feat[train_idx], edges, draw_sample(case, train_idx.numel()), sp, tp)
        kd = case["form"] == "kd_aux"
        loss, lc, lk, la, _, state, grads = odi.distill_step(
            state, m, v, s + 1, *args, b["y"], train_idx, 3, R, 2, d["in_channels"], G["lr"], aux, case["beta"],
            masks=masks_of(s) if masks_of else None, p=p, teacher_logits=t_logits if kd else None, alpha=G["alpha"], T=G["kd_T"])
        grads = dict(grads)
        if opt is not None:
            grads.update({k: q.grad.detach().clone() for k, q in head_params(sp, tp)})
            opt.step()
            opt.zero_grad()
        steps.append((loss, lc, lk, la, grads, train_idx.numel()))
    return steps, state, (sp, tp)


def roundoff_keys(grads_per_step):
    """Parameters whose gradient is zero up to round-off in every step: the bias of a Linear that feeds a train-mode
    BatchNorm1d (the heads' first layer; Adam moves it by lr * sign(round-off)), and weights that no training row reaches."""
    keys = set(grads_per_step[0])
    for g in grads_per_step:
        scale = max(t.abs().max().item() for t in g.values())
        keys &= {k for k, t in g.items() if t.abs().max().item() < 1e-9 * scale}
    return keys


def check_grads(got, want, tol, noise):
    """rel_err per parameter; a round-off-only gradient must stay round-off (1e-5 of the step's largest gradient)."""
    assert set(got) == set(want)
    scale = max(t.abs().max().item() for t in want.values())
    for k in want:
        if k in noise:
            assert got[k].abs().max().item() < 1e-5 * scale, k
        else:
            assert rel_err(got[k], want[k]) < tol, k


def weighted_triple(steps):
    """train()'s return value: (loss, loss_cls, loss_aux) averaged over batches weighted by their train-row counts."""
    n = sum(s[5] for s in steps)
    return torch.tensor([sum(float(s[i]) * s[5] for s in steps) / n for i in (0, 1, 3)], dtype=torch.float64)


@pytest.mark.parametrize("name", CASES)
def test_distill_step_reproduces_reference_train(golden_distill, name):
    G = golden_distill
    case = G["cases"][name]
    steps, state, (sp, tp) = replay_fp64(G, case)
    assert rel_err(weighted_triple(steps), case["result"]) < 1e-10
    noise = roundoff_keys(case["grads"])
    assert not case["heads"] or {"student_proj.0.bias", "teacher_proj.0.bias"} <= noise
    # gradients and states are stored rounded to fp32: 1e-6 is that rounding, not the fp64 agreement
    for s, want in enumerate(case["grads"]):
        check_grads(steps[s][4], want, 1e-6, noise)
    for k, want in case["final"].items():
        assert rel_err(state[k], want) < 1e-6, k
    if case["heads"]:
        for name_h, mod in (("student_proj", sp), ("teacher_proj", tp)):
            for k, want in case["final_heads"][name_h].items():
                if f"{name_h}.{k}" not in noise:
                    assert rel_err(mod.state_dict()[k], want) < 1e-6, (name_h, k)


def test_distill_step_with_beta_zero_is_the_plain_step(golden_distill):
    G = golden_distill
    d, R = G["dims"], len(G["rels"])
    b = G["batches"][0]
    args = _oracle_args(G, b)
    train_idx = b["train_mask"].nonzero().view(-1)
    with torch.no_grad():
        t_logits, _ = ort.rgcn_forward(G["teacher"], *args, 3, R, 3, d["in_channels"])
    aux = lambda f, z: f[train_idx].pow(2).mean()  # noqa: E731
    for teacher in (None, t_logits):
        zeros = lambda: {k: torch.zeros_like(t) for k, t in G["student"].items()}  # noqa: E731
        m1, v1, m2, v2 = zeros(), zeros(), zeros(), zeros()
        a = ort.train_step(G["student"], m1, v1, 1, *args, b["y"], train_idx, 3, R, 2, d["in_channels"], G["lr"],
                           teacher_logits=teacher)
        bb = odi.distill_step(G["student"], m2, v2, 1, *args, b["y"], train_idx, 3, R, 2, d["in_channels"], G["lr"], aux, 0.0,
                              teacher_logits=teacher)
        for x, y in zip(a[:3], bb[:3]):
            assert torch.equal(x, y)
        assert float(bb[3]) > 0
        assert torch.equal(a[3], bb[4])
        for k in a[4]:
            assert torch.equal(a[4][k], bb[5][k]) and torch.equal(m1[k], m2[k]) and torch.equal(v1[k], v2[k]), k
