"""One training step of the reference's R-GCN, restated in fp64 on the CPU: ``RGCN.forward`` (mag_pyg/gnn.py:126-138, the
per-edge message-passing form of oracle.nn.rgcn_conv), the supervised or ``kd_criterion`` loss over the training rows
(mag_pyg/gnn.py:191-203), autograd, and torch.optim.Adam's update (dense over every parameter, embedding tables included).

Dropout is not drawn here: ``masks[l]`` ([n, hidden] keep-masks, 0/1) are injected, so the step can be compared with an
engine that draws its own.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from . import criterion as oc
from . import nn as onn


def rgcn_forward(state: Dict[str, torch.Tensor], x_dict, edge_index, edge_type, node_type, local_node_idx, num_types: int,
                 num_edge_types: int, num_layers: int, in_channels: int, masks: Optional[List[torch.Tensor]] = None,
                 p: float = 0.5):
    """(logits, out_feat) of RGCN.forward on the given state (tensors keep their dtype and autograd)."""
    emb = {k.split(".")[1]: v for k, v in state.items() if k.startswith("emb_dict.")}
    h = onn.rgcn_group_input(x_dict, emb, node_type, local_node_idx, in_channels)
    out_feat = None
    for i in range(num_layers):
        rel = [state[f"convs.{i}.rel_lins.{r}.weight"] for r in range(num_edge_types)]
        root_w = [state[f"convs.{i}.root_lins.{t}.weight"] for t in range(num_types)]
        root_b = [state[f"convs.{i}.root_lins.{t}.bias"] for t in range(num_types)]
        h = onn.rgcn_conv(h, edge_index, edge_type, node_type, rel, root_w, root_b)
        if i != num_layers - 1:
            h = torch.relu(h)
            if masks is not None:
                h = h * masks[i].to(h.dtype) / (1.0 - p)
            out_feat = h
    return h, out_feat


def adam_update(params: Dict[str, torch.Tensor], grads: Dict[str, torch.Tensor], exp_avg, exp_avg_sq, step: int, lr: float,
                betas=(0.9, 0.999), eps: float = 1e-8):
    """torch.optim.Adam (no weight decay, no amsgrad) for step number ``step`` (1-based); updates every dict in place."""
    b1, b2 = betas
    for k in params:
        g = grads[k]
        exp_avg[k] = b1 * exp_avg[k] + (1 - b1) * g
        exp_avg_sq[k] = b2 * exp_avg_sq[k] + (1 - b2) * g * g
        bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
        params[k] = params[k] - lr * (exp_avg[k] / bc1) / ((exp_avg_sq[k] / bc2).sqrt() + eps)


def train_step(state, exp_avg, exp_avg_sq, step: int, x_dict, edge_index, edge_type, node_type, local_node_idx, y, train_idx,
               num_types: int, num_edge_types: int, num_layers: int, in_channels: int, lr: float, masks=None, p: float = 0.5,
               teacher_logits=None, alpha: float = 0.9, T: float = 4.0):
    """One reference train() step in fp64.  Returns (loss, loss_cls, loss_kd, logits, new state); exp_avg / exp_avg_sq are
    updated in place."""
    st = {k: v.detach().double().clone().requires_grad_(True) for k, v in state.items()}
    xd = {k: v.double() for k, v in x_dict.items()}
    logits, _ = rgcn_forward(st, xd, edge_index, edge_type, node_type, local_node_idx, num_types, num_edge_types, num_layers,
                             in_channels, masks, p)
    out, labels = logits[train_idx], y.view(-1)[train_idx]
    if teacher_logits is None:
        loss = oc.cross_entropy(out, labels)
        loss_cls, loss_kd = loss, loss * 0
    else:
        loss, loss_cls, loss_kd = oc.kd_criterion(out, labels, teacher_logits.double()[train_idx], alpha, T)
    loss.backward()
    params = {k: v.detach() for k, v in st.items()}
    grads = {k: v.grad if v.grad is not None else torch.zeros_like(v) for k, v in st.items()}
    adam_update(params, grads, exp_avg, exp_avg_sq, step, lr)
    return loss.detach(), loss_cls.detach(), loss_kd.detach(), logits.detach(), params
