"""One training step of the reference's R-GCN with a representation-distillation loss, restated in fp64 on the CPU: the
``fitnet|at|lpw|gpw|nce`` branches of mag_pyg/gnn.py ``train()`` (:204-251, ``loss_cls + beta * aux``) and of
mag_pyg/gnn_kd_and_aux.py (:204-271, ``kd + beta * aux``).  Forward, losses and torch.optim.Adam's update come from
oracle.rgcn_train; dropout masks are injected, as there.
"""
from __future__ import annotations

import torch

from . import criterion as oc
from .rgcn_train import adam_update, rgcn_forward


def distill_step(state, exp_avg, exp_avg_sq, step: int, x_dict, edge_index, edge_type, node_type, local_node_idx, y,
                 train_idx, num_types: int, num_edge_types: int, num_layers: int, in_channels: int, lr: float, aux,
                 beta: float = 1.0, masks=None, p: float = 0.5, teacher_logits=None, alpha: float = 0.9, T: float = 4.0):
    """``loss_cls + beta * aux`` without ``teacher_logits``, ``kd + beta * aux`` with them.  ``aux(out_feat, logits)`` gets
    the fp64 last hidden activation (after ReLU and the injected dropout) and the logits of ALL rows and returns the
    auxiliary loss; parameters it owns (projection heads) receive their ``.grad`` from the same backward.  Returns
    (loss, loss_cls, loss_kd, loss_aux, logits, new state, gradients); exp_avg / exp_avg_sq are updated in place."""
    st = {k: v.detach().double().clone().requires_grad_(True) for k, v in state.items()}
    xd = {k: v.double() for k, v in x_dict.items()}
    logits, out_feat = rgcn_forward(st, xd, edge_index, edge_type, node_type, local_node_idx, num_types, num_edge_types,
                                    num_layers, in_channels, masks, p)
    out, labels = logits[train_idx], y.view(-1)[train_idx]
    if teacher_logits is None:
        loss = oc.cross_entropy(out, labels)
        loss_cls, loss_kd = loss, loss * 0
    else:
        loss, loss_cls, loss_kd = oc.kd_criterion(out, labels, teacher_logits.double()[train_idx], alpha, T)
    loss_aux = aux(out_feat, logits)
    loss = loss + beta * loss_aux
    loss.backward()
    params = {k: v.detach() for k, v in st.items()}
    grads = {k: v.grad if v.grad is not None else torch.zeros_like(v) for k, v in st.items()}
    adam_update(params, grads, exp_avg, exp_avg_sq, step, lr)
    return loss.detach(), loss_cls.detach(), loss_kd.detach(), loss_aux.detach(), logits.detach(), params, grads
