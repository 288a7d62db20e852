"""R-GCN training engine, the parts that need no GPU: its parameter table against the reference-shaped module, and the fp64
restatement of the training step (oracle/rgcn_train.py) against the fixture made by the reference's own RGCN class."""
import pytest
import torch

import efficient_gnns_b200  # noqa: F401
from conftest import rel_err
from efficient_gnns_b200.rgcn import RGCNTrainer
from oracle import rgcn_train as ort

MAG_NODES = {0: 736_389, 1: 1_134_649, 2: 8_740, 3: 59_965}


class _RefShapedRGCN(torch.nn.Module):
    """The module tree of the reference's RGCN (mag_pyg/gnn.py:71-103) with meta tensors: names and shapes only."""

    def __init__(self, in_channels, hidden, out_channels, num_layers, num_nodes_dict, x_types, num_edge_types):
        super().__init__()
        lin = lambda i, o, b: torch.nn.Linear(i, o, bias=b, device="meta")
        self.emb_dict = torch.nn.ParameterDict({f"{k}": torch.nn.Parameter(torch.empty(num_nodes_dict[k], in_channels, device="meta"))
                                                for k in set(num_nodes_dict).difference(set(x_types))})
        dims = [in_channels] + [hidden] * (num_layers - 1) + [out_channels]
        self.convs = torch.nn.ModuleList()
        for i in range(num_layers):
            conv = torch.nn.Module()
            conv.rel_lins = torch.nn.ModuleList([lin(dims[i], dims[i + 1], False) for _ in range(num_edge_types)])
            conv.root_lins = torch.nn.ModuleList([lin(dims[i], dims[i + 1], True) for _ in num_nodes_dict])
            self.convs.append(conv)


@pytest.mark.parametrize("hidden,layers", [(32, 2), (512, 3)], ids=["student", "teacher"])
def test_parameter_table_matches_the_reference_module(hidden, layers):
    ref = _RefShapedRGCN(128, hidden, 349, layers, MAG_NODES, [0], 7).state_dict()
    table = RGCNTrainer.param_table(MAG_NODES, [0], 7, 128, hidden, 349, layers)
    assert {k: tuple(v.shape) for k, v in ref.items()} == dict(table)
    assert len(table) == len(ref)


def test_fp64_oracle_step_reproduces_reference_fixture(golden_rgcn):
    G = golden_rgcn
    st = {k: v.double().clone().requires_grad_(True) for k, v in G["state"].items()}
    out, feat = ort.rgcn_forward(st, {0: G["x_paper"].double()}, G["edge_index"], G["edge_type"], G["node_type"],
                                 G["local_node_idx"], 3, len(G["rels"]), 2, 16)
    assert rel_err(out, G["out_forward"]) < 1e-6 and rel_err(feat, G["out_feat"]) < 1e-6
    (out * G["w"].double()).sum().backward()
    for k, t in st.items():
        assert rel_err(t.grad, G["grads"][k]) < 1e-5, k


def test_oracle_adam_matches_torch_adam():
    g = torch.Generator().manual_seed(0)
    p = {"a": torch.randn(5, 3, generator=g, dtype=torch.float64), "b": torch.randn(4, generator=g, dtype=torch.float64)}
    tp = {k: torch.nn.Parameter(v.clone()) for k, v in p.items()}
    opt = torch.optim.Adam(tp.values(), lr=0.01)
    m = {k: torch.zeros_like(v) for k, v in p.items()}
    v2 = {k: torch.zeros_like(v) for k, v in p.items()}
    for step in (1, 2, 3):
        grads = {k: torch.randn(v.shape, generator=g, dtype=torch.float64) * (0 if step == 2 and k == "b" else 1) for k, v in p.items()}
        for k in tp:
            tp[k].grad = grads[k].clone()
        opt.step()
        ort.adam_update(p, grads, m, v2, step, 0.01)
        for k in p:
            assert torch.allclose(p[k], tp[k].detach(), rtol=1e-12, atol=1e-14)
