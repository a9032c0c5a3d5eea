"""Monte-Carlo dropout oracle (sc_segment_volume_mc): T stochastic passes of the head, restated in fp64 on torch-CPU.

TEST INFRASTRUCTURE, like ``oracle/``: built from the unchanged deterministic oracle ``oracle/network.py`` (same layer
semantics, stored BatchNorm statistics).  The dropout masks are applied to the ACTIVATIONS, as ``train_forward`` does,
while the device masks weight rows; the parity tests therefore check the device's row mappings independently.
"""
import numpy as np
import torch
import torch.nn.functional as F

from oracle.network import BRANCHES, _bn_affine, _prelu, _t

DROP_UNITS = 2700   # keep bits per pass: [3][540] *_l1drop (c, h, w) | [540] f1_drop | [540] f2_drop


def hash3(seed, idx):
    """``hash3`` of csrc/common.cuh (splitmix64 finaliser, top bits) in wrapping uint64 arithmetic; idx may be an array."""
    u = np.uint64
    with np.errstate(over="ignore"):
        z = u(seed) + u(0x9E3779B97F4A7C15) * (np.asarray(idx, dtype=u) + u(1))
        z = (z ^ (z >> u(30))) * u(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> u(27))) * u(0x94D049BB133111EB)
        return ((z ^ (z >> u(31))) >> u(16)).astype(np.uint32)


def mc_keep_masks(seed, T):
    """uint8 [T, 2700]: pass t keeps unit j when hash3(seed, t * 2700 + j) & 1 -- the mask the training step gives sample t."""
    return (hash3(seed, np.arange(T * DROP_UNITS, dtype=np.uint64)) & 1).astype(np.uint8).reshape(T, DROP_UNITS)


def _branch_flat(P, b, x, dtype):
    """conv1..conv5 of one view in deterministic mode -> the flattened [N, 540] input of d1 (c, h, w order)."""
    x = x.to(dtype)
    for i in range(1, 6):
        w = torch.flip(_t(P["%s_ch_conv%d" % (b, i)][0], dtype), dims=[2, 3])
        x = F.conv2d(x, w)
        scale, shift = _bn_affine(P, "%s_ch_conv%d_bn" % (b, i), dtype)
        x = _prelu(x * scale.view(1, -1, 1, 1) + shift.view(1, -1, 1, 1), _t(P["%s_ch_prelu%d" % (b, i)][0], dtype))
        if i in (2, 4):
            x = F.max_pool2d(x, 2)
    return x.flatten(1)


def _head_dropout(P, flats, atlas, keep, dtype):
    """d1 x3 and the FC head with the keep mask applied to the ACTIVATIONS at the three dropout sites (x 2, as train_forward)."""
    k = torch.as_tensor(np.asarray(keep, np.float64)).to(dtype) * 2.0
    feats = []
    for i, b in enumerate(BRANCHES):
        W, bias = (_t(a, dtype) for a in P["%s_d1" % b])
        feats.append(_prelu((flats[i] * k[i * 540:(i + 1) * 540]) @ W + bias, _t(P["%s_prelu_d1" % b][0], dtype)))
    x = torch.cat(feats, dim=1) * k[1620:2160]
    W, bias = (_t(a, dtype) for a in P["FC1"])
    x = _prelu(x @ W + bias, _t(P["prelu_f1"][0], dtype)) * k[2160:2700]
    x = torch.cat([x, atlas.to(dtype)], dim=1)
    W, bias = (_t(a, dtype) for a in P["fc_2"])
    x = _prelu(x @ W + bias, _t(P["prelu_f2"][0], dtype))
    W, bias = (_t(a, dtype) for a in P["out_layer"])
    return torch.softmax(x @ W + bias, dim=1)


def _inputs(in1, in2, in3, in4):
    return [torch.as_tensor(np.ascontiguousarray(a)) for a in (in1, in2, in3, in4)]


def forward_dropout(P, in1, in2, in3, in4, keep, dtype=torch.float64):
    """One dropout pass: the deterministic forward (stored BN statistics) with the [2700] keep mask applied to the
    activations at *_l1drop, f1_drop and f2_drop, kept units scaled by 2.  -> softmax [N, 15]."""
    xs = _inputs(in1, in2, in3, in4)
    with torch.no_grad():
        flats = [_branch_flat(P, b, x, dtype) for b, x in zip(BRANCHES, xs[:3])]
        return _head_dropout(P, flats, xs[3], keep, dtype).numpy()


def mc_predict(P, in1, in2, in3, in4, seed, T, dtype=torch.float64):
    """Monte-Carlo dropout over T passes (masks of mc_keep_masks) -> (mean softmax [N, 15], predictive entropy H [N],
    mutual information max(0, H - mean_t H(p_t)) [N]); entropies in nats with 0 ln 0 = 0."""
    xs = _inputs(in1, in2, in3, in4)
    keep = mc_keep_masks(seed, T)
    with torch.no_grad():
        flats = [_branch_flat(P, b, x, dtype) for b, x in zip(BRANCHES, xs[:3])]
        psum, hsum = 0.0, 0.0
        for t in range(T):
            p = _head_dropout(P, flats, xs[3], keep[t], dtype)
            psum = psum + p
            hsum = hsum - torch.xlogy(p, p).sum(1)
        pbar = psum / T
        H = -torch.xlogy(pbar, pbar).sum(1)
        mi = torch.clamp(H - hsum / T, min=0.0)
    return pbar.numpy(), H.numpy(), mi.numpy()
