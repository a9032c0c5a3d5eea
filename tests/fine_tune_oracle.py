"""fp64 reference of fine-tuning with a frozen trunk (sc_trunk_features, sc_head_train_forward_backward), built on the
unchanged deterministic and training oracles of ``oracle/network.py``.

* trunk = conv1..conv5 with BatchNorm (stored statistics) and PReLU of every view; its output per sample and view is the
  flattened conv5 activation [540] (k = c*9 + h*3 + w), the input of ``<view>_d1`` before dropout.
* head = every other array; one training step is fp64 autograd over the head arrays only, with the dropout, loss and Lasagne
  Adam of ``oracle.network.train_step``.  The trunk arrays are copied through unchanged.
"""
from collections import OrderedDict

import numpy as np
import torch

from oracle import network as on


def is_trunk(name):
    return "_ch_conv" in name or "_ch_prelu" in name


def trunk_features(P, in1, in2, in3, dtype=torch.float64):
    """[N,1,32,32] x3 -> [N,3,540] trunk features in deterministic mode"""
    out = []
    with torch.no_grad():
        for b, x in zip(on.BRANCHES, (in1, in2, in3)):
            taps = {}
            on.branch_forward(P, b, torch.as_tensor(np.ascontiguousarray(x)), dtype, taps=taps)
            out.append(taps["%s_c5" % b].flatten(1))
    return torch.stack(out, 1).numpy()


def _head(T, feats, in4, masks, dtype):
    """head forward on torch parameters T from features [N,3,540] -> logits; masks as for oracle.network.train_forward"""
    f = torch.as_tensor(np.ascontiguousarray(feats)).to(dtype)
    d1 = []
    for v, b in enumerate(on.BRANCHES):
        x = f[:, v]
        if masks is not None:
            x = x * masks["%s_l1drop" % b].reshape(x.shape[0], 540).to(dtype) * 2.0
        d1.append(on._prelu(x @ T["%s_d1" % b][0] + T["%s_d1" % b][1], T["%s_prelu_d1" % b][0]))
    x = torch.cat(d1, dim=1)
    if masks is not None:
        x = x * masks["f1_drop"].to(dtype) * 2.0
    x = on._prelu(x @ T["FC1"][0] + T["FC1"][1], T["prelu_f1"][0])
    if masks is not None:
        x = x * masks["f2_drop"].to(dtype) * 2.0
    x = torch.cat([x, torch.as_tensor(np.ascontiguousarray(in4)).to(dtype)], dim=1)
    x = on._prelu(x @ T["fc_2"][0] + T["fc_2"][1], T["prelu_f2"][0])
    return x @ T["out_layer"][0] + T["out_layer"][1]


def head_forward(P, feats, in4, dtype=torch.float64):
    """deterministic softmax [N,15] from trunk features"""
    with torch.no_grad():
        return torch.softmax(_head(on.to_torch(P, dtype, requires_grad=False), feats, in4, None, dtype), dim=1).numpy()


def head_names(P):
    return [(n, k) for n, k in on.trainable_names(P) if not is_trunk(n)]


def _masks(masks):
    return None if masks is None else {k: torch.as_tensor(np.ascontiguousarray(v)) for k, v in masks.items()}


def head_loss(P, feats, in4, y, masks=None, dtype=torch.float64):
    """mean cross-entropy of the training-mode head (finite-difference checks)"""
    with torch.no_grad():
        z = _head(on.to_torch(P, dtype, requires_grad=False), feats, in4, _masks(masks), dtype)
        logp = torch.log_softmax(z, dim=1)
        return float(-logp[torch.arange(z.shape[0]), torch.as_tensor(np.asarray(y).astype(np.int64))].mean())


def head_train_step(P, feats, in4, y, masks=None, state=None, lr=1e-3, dtype=torch.float64):
    """One head-only minibatch update from trunk features.  Returns (loss, grads{(name,k): ndarray} of the head arrays, new P,
    new state) like oracle.network.train_step; the trunk arrays of the new P are copies of P's."""
    T = on.to_torch(P, dtype, requires_grad=False)
    names = head_names(P)
    for n, k in names:
        T[n][k].requires_grad_(True)
    z = _head(T, feats, in4, _masks(masks), dtype)
    logp = torch.log_softmax(z, dim=1)
    loss = -logp[torch.arange(z.shape[0]), torch.as_tensor(np.asarray(y).astype(np.int64))].mean()
    grads = torch.autograd.grad(loss, [T[n][k] for n, k in names])
    if state is None:
        state = {"t": 0, "m": {}, "v": {}}
    t = state["t"] + 1
    newP = OrderedDict((n, [np.array(a, copy=True) for a in arrs]) for n, arrs in P.items())
    new_state = {"t": t, "m": {}, "v": {}}
    G = {}
    for (n, k), g in zip(names, grads):
        p = T[n][k].detach()
        m = state["m"].get((n, k), torch.zeros_like(p))
        v = state["v"].get((n, k), torch.zeros_like(p))
        p2, m2, v2 = on.adam_update(p, g, m, v, t, lr=lr)
        newP[n][k] = p2.numpy().astype(np.float32)
        new_state["m"][(n, k)], new_state["v"][(n, k)] = m2, v2
        G[(n, k)] = g.numpy()
    return float(loss.detach()), G, newP, new_state
