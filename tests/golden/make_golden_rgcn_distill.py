"""Generate rgcn_distill_mag.pt by running the REFERENCE's own MAG training loops, unmodified:

    python tests/golden/make_golden_rgcn_distill.py        (needs the reference checkout; not run on the GPU box)

`train()` of mag_pyg/gnn.py (``loss_cls + beta * aux``, :174-268) and of mag_pyg/gnn_kd_and_aux.py (``kd + beta * aux``)
is called for the five representation losses (fitnet, at, lpw, gpw, nce) on a small 3-type / 5-relation graph, with a
2-layer student, a 3-layer eval-mode teacher and, for fitnet and nce, the reference's projection heads (Linear ->
BatchNorm1d -> ReLU).  The only stand-ins are those of make_golden.install_mag_stubs() plus:
  * a list of hand-built batch objects with ``.to()`` for the GraphSAINT loader (two batches: the whole graph, then a
    sub-graph that leaves out part of one embedding table);
  * an ``args`` namespace and a dummy ``tqdm``;
  * an optimizer wrapper that records every parameter's ``.grad`` before torch Adam's ``step()``;
  * the module global ``F`` swapped for a proxy whose ``dropout`` is the identity: ``RGCN.forward`` hard-codes p = 0.5
    under ``model.train()``, and torch's dropout RNG cannot be replayed elsewhere.
Everything runs in fp64 (default dtype), so the fixture pins the arithmetic, not fp32 rounding.  numpy's global RNG is
seeded before each train() call: the GSP case with max_samples below the train-row count draws its row sample from it.
The initial states, batches and train()'s returned triples are stored in fp64; each case's per-step gradients and final
states are stored as flat fp32 vectors in the order of ``layout`` / ``head_layout`` / ``head_state_layout`` (rounding
them keeps the file small and costs nothing against the fp32 engine's tolerances).
"""
from __future__ import annotations

import importlib.util
import sys
import types
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE))
import make_golden as mg  # noqa: E402

REF = mg.REF
OUT = HERE / "rgcn_distill_mag.pt"

NODES = {0: 24, 1: 12, 2: 8}                                   # type 0 carries features, 1 / 2 get embedding tables
RELS = [(1, 0, 60), (0, 0, 90), (2, 1, 30), (0, 1, 50), (1, 2, 24)]     # (src type, dst type, #edges)
IN, HID, OUT_C, T_HID, PROJ = 5, 6, 3, 7, 6                    # widths not multiples of 4
LR, ALPHA, KD_T, NP_SEED = 0.01, 0.9, 4.0, 7

# (name, training, kernel, beta, max_samples, nce_T, heads)
CASES = [
    ("fitnet", "fitnet", None, 100.0, 8192, 0.075, True),
    ("at", "at", None, 1000.0, 8192, 0.075, False),
    ("lpw_rbf", "lpw", "rbf", 100.0, 8192, 0.075, False),
    ("lpw_cosine", "lpw", "cosine", 100.0, 8192, 0.075, False),
    ("lpw_poly", "lpw", "poly", 100.0, 8192, 0.075, False),
    ("gpw_cosine", "gpw", "cosine", 100.0, 8192, 0.075, False),
    ("gpw_poly", "gpw", "poly", 100.0, 8192, 0.075, False),
    ("gpw_rbf", "gpw", "rbf", 100.0, 10, 0.075, False),           # 10 < train rows: np.random.choice draws the sample
    ("nce", "nce", None, 0.5, 8192, 0.075, True),
]
FORMS = {"gnn": "gnn.py", "kd_aux": "gnn_kd_and_aux.py"}


def graph():
    g = torch.Generator().manual_seed(31)
    off = {0: 0, 1: NODES[0], 2: NODES[0] + NODES[1]}
    eis, ets = [], []
    for r, (s, d, e) in enumerate(RELS):
        src = torch.randint(0, NODES[s], (e,), generator=g)
        dst = torch.randint(0, NODES[d], (e,), generator=g)
        eis.append(torch.stack([src + off[s], dst + off[d]]))
        ets.append(torch.full((e,), r, dtype=torch.long))
    ei, et = torch.cat(eis, 1), torch.cat(ets)
    nt = torch.cat([torch.full((NODES[t],), t, dtype=torch.long) for t in range(3)])
    li = torch.cat([torch.arange(NODES[t]) for t in range(3)])
    n = nt.numel()
    x_paper = torch.randn(NODES[0], IN, generator=g, dtype=torch.float64)
    y = torch.full((n, 1), -1, dtype=torch.long)
    y[:NODES[0], 0] = torch.randint(0, OUT_C, (NODES[0],), generator=g)
    train_mask = torch.zeros(n, dtype=torch.bool)
    train_mask[:NODES[0]] = torch.rand(NODES[0], generator=g) < 0.65
    batches = [dict(edge_index=ei, edge_attr=et, node_type=nt, local_node_idx=li, y=y, train_mask=train_mask)]
    # the second batch leaves out every other row of type 2: those embedding rows get no gradient
    keep = torch.cat([torch.arange(off[2]), torch.arange(off[2], n, 2)])
    sub = torch.full((n,), -1, dtype=torch.long)
    sub[keep] = torch.arange(keep.numel())
    em = (sub[ei[0]] >= 0) & (sub[ei[1]] >= 0)
    batches.append(dict(edge_index=sub[ei[:, em]], edge_attr=et[em], node_type=nt[keep], local_node_idx=li[keep], y=y[keep],
                        train_mask=train_mask[keep]))
    return x_paper, batches


class _Batch:
    def __init__(self, d):
        self.__dict__.update(d)

    def to(self, device):
        return self


class _Pbar:
    def __init__(self, *a, **k):
        pass

    def update(self, *a):
        pass

    def close(self):
        pass


class _RecordingAdam:
    """torch Adam over named parameters; records every .grad right before each step()."""

    def __init__(self, named, lr):
        self.named = list(named)
        self.opt = torch.optim.Adam([p for _, p in self.named], lr=lr)
        self.grads = []

    def zero_grad(self):
        self.opt.zero_grad()

    def step(self):
        self.grads.append({k: (p.grad if p.grad is not None else torch.zeros_like(p)).detach().clone() for k, p in self.named})
        self.opt.step()


def _no_dropout_F():
    import torch.nn.functional as F
    proxy = types.ModuleType("F_without_dropout")
    proxy.__dict__.update({k: getattr(F, k) for k in dir(F) if not k.startswith("__")})
    proxy.dropout = lambda x, p=0.5, training=True, inplace=False: x
    return proxy


def _load(name, file):
    spec = importlib.util.spec_from_file_location(name, REF / "mag_pyg" / file)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.F = _no_dropout_F()
    mod.tqdm = _Pbar
    return mod


def _heads():
    mk = lambda i: torch.nn.Sequential(torch.nn.Linear(i, PROJ), torch.nn.BatchNorm1d(PROJ), torch.nn.ReLU())  # noqa: E731
    return mk(HID), mk(T_HID)


def _clone(sd):
    return {k: v.detach().clone() for k, v in sd.items()}


def _layout(named):
    return [(k, tuple(v.shape)) for k, v in named]


def _flat(d, layout):
    """The tensors of ``d`` in ``layout`` order, concatenated into one fp32 vector."""
    return torch.cat([d[k].detach().reshape(-1).to(torch.float32) for k, _ in layout])


def main():
    assert REF.exists(), "the reference checkout is needed to regenerate this fixture"
    mg.install_mag_stubs()
    sys.path.insert(0, str(REF / "mag_pyg"))
    torch.set_default_dtype(torch.float64)
    mods = {form: _load(f"mag_{form}", file) for form, file in FORMS.items()}
    x_paper, batches = graph()
    x_dict = {0: x_paper}
    R = len(RELS)
    torch.manual_seed(0)
    student0 = _clone(mods["gnn"].RGCN(IN, HID, OUT_C, 2, 0.5, NODES, [0], R).state_dict())
    teacher = _clone(mods["gnn"].RGCN(IN, T_HID, OUT_C, 3, 0.5, NODES, [0], R).state_dict())
    sp, tp = _heads()
    heads0 = dict(student_proj=_clone(sp.state_dict()), teacher_proj=_clone(tp.state_dict()))
    layout = _layout(student0.items())
    head_layout = _layout([(f"student_proj.{k}", p) for k, p in sp.named_parameters()] +
                          [(f"teacher_proj.{k}", p) for k, p in tp.named_parameters()])
    head_state_layout = _layout([(f"student_proj.{k}", v) for k, v in sp.state_dict().items()] +
                                [(f"teacher_proj.{k}", v) for k, v in tp.state_dict().items()])

    cases = {}
    for form, mod in mods.items():
        for name, training, kernel, beta, max_samples, nce_T, heads in CASES:
            model = mod.RGCN(IN, HID, OUT_C, 2, 0.5, NODES, [0], R)
            model.load_state_dict(student0)
            tm = mod.RGCN(IN, T_HID, OUT_C, 3, 0.5, NODES, [0], R)
            tm.load_state_dict(teacher)
            tm.eval()
            named = list(model.named_parameters())
            sp = tp = None
            if heads:
                sp, tp = _heads()
                sp.load_state_dict(heads0["student_proj"]); tp.load_state_dict(heads0["teacher_proj"])
                named += [(f"student_proj.{k}", p) for k, p in sp.named_parameters()]
                named += [(f"teacher_proj.{k}", p) for k, p in tp.named_parameters()]
            opt = _RecordingAdam(named, LR)
            args = types.SimpleNamespace(training=training, alpha=ALPHA, kd_T=KD_T, beta=beta, kernel=kernel,
                                         max_samples=max_samples, nce_T=nce_T, num_steps=len(batches), batch_size=1)
            np.random.seed(NP_SEED)
            triple = mod.train(model, [_Batch(b) for b in batches], x_dict, opt, args, "cpu", tm, sp, tp)
            head_state = ({**{f"student_proj.{k}": v for k, v in sp.state_dict().items()},
                           **{f"teacher_proj.{k}": v for k, v in tp.state_dict().items()}} if heads else None)
            cases[f"{form}/{name}"] = dict(
                form=form, training=training, kernel=kernel, beta=beta, max_samples=max_samples, nce_T=nce_T, heads=heads,
                result=torch.tensor(triple, dtype=torch.float64),
                grads=torch.stack([_flat(g, layout) for g in opt.grads]),
                head_grads=torch.stack([_flat(g, head_layout) for g in opt.grads]) if heads else None,
                final=_flat(model.state_dict(), layout),
                final_heads=_flat(head_state, head_state_layout) if heads else None)
    torch.save(dict(num_nodes=NODES, rels=RELS, dims=dict(in_channels=IN, hidden=HID, out_channels=OUT_C, teacher_hidden=T_HID,
                                                         proj_dim=PROJ),
                    lr=LR, alpha=ALPHA, kd_T=KD_T, np_seed=NP_SEED, x_paper=x_paper, batches=batches,
                    student=student0, teacher=teacher, heads=heads0, layout=layout, head_layout=head_layout,
                    head_state_layout=head_state_layout, cases=cases), OUT)
    print("wrote", OUT.name, len(cases), "cases")


if __name__ == "__main__":
    main()
