"""fp64 numpy restatement of the resampling rules of include/subcort_b200.h (sc_resample_volume, sc_map_proba_back) and of the
nearest-neighbour label rule of the training set, for the parity tests of the kernels."""
import numpy as np


def target_dims(shape, spacing, resample_mm):
    """m = max(1, floor(n s / t + 0.5)) per axis"""
    return tuple(max(1, int(np.floor(n * s / resample_mm + 0.5))) for n, s in zip(shape[:3], spacing))


def weight_matrix(n, m):
    """[m, n]: row j holds the normalised weights w_ij = max(0, 1 - |i - x_j| / h), x_j = (j + 0.5) r - 0.5, h = max(r, 1)"""
    r = n / m
    h = max(r, 1.0)
    x = (np.arange(m) + 0.5) * r - 0.5
    W = np.maximum(0.0, 1.0 - np.abs(np.arange(n)[None, :] - x[:, None]) / h)
    return W / W.sum(1, keepdims=True)


def resample(vol, out_shape):
    """[X,Y,Z] or [X,Y,Z,C] -> out_shape[:3] (+ C), separable, fp64"""
    out = np.asarray(vol, np.float64)
    for a in range(3):
        W = weight_matrix(out.shape[a], int(out_shape[a]))
        out = np.moveaxis(np.tensordot(W, out, axes=([1], [a])), 0, a)
    return out


def backmap_axis(n, m):
    """native -> (lower target neighbour i0, weight f of the upper one) for an axis of n native and m target voxels"""
    r = n / m
    y = np.clip((np.arange(n) + 0.5) / r - 0.5, 0.0, m - 1.0)
    i0 = np.minimum(np.floor(y), m - 2).astype(np.int64) if m > 1 else np.zeros(n, np.int64)
    return i0, y - i0


def map_proba_back(proba, cand, native_shape, native_mask=None):
    """target probabilities [m0,m1,m2,15] and candidates -> (native proba [X,Y,Z,15], first arg-max labels, written mask, top-two
    gap).  Neighbours with zero trilinear weight or no candidate are dropped and the rest renormalised; a voxel is written when
    one neighbour remains and native_mask (if given) is non-zero."""
    proba = np.asarray(proba, np.float64)
    cand = np.asarray(cand) != 0
    tshape = proba.shape[:3]
    axes = [backmap_axis(n, m) for n, m in zip(native_shape, tshape)]
    acc = np.zeros(tuple(native_shape) + (15,))
    wsum = np.zeros(tuple(native_shape))
    for dx in (0, 1):
        for dy in (0, 1):
            for dz in (0, 1):
                idx, wts = [], []
                for (i0, f), d, m in zip(axes, (dx, dy, dz), tshape):
                    idx.append(np.minimum(i0 + d, m - 1))
                    wts.append(f if d else 1.0 - f)
                w = wts[0][:, None, None] * wts[1][None, :, None] * wts[2][None, None, :]
                ix = np.ix_(*idx)
                w = np.where(cand[ix], w, 0.0)
                wsum += w
                acc += w[..., None] * proba[ix]
    written = wsum > 0
    if native_mask is not None:
        written &= np.asarray(native_mask) != 0
    p = np.where(written[..., None], acc / np.where(wsum > 0, wsum, 1.0)[..., None], 0.0)
    srt = np.sort(p, -1)
    return p, np.argmax(p, -1).astype(np.uint8), written, srt[..., -1] - srt[..., -2]


def nearest_index(n, m):
    x = (np.arange(m) + 0.5) * (n / m) - 0.5
    return np.clip(np.floor(x + 0.5), 0, n - 1).astype(np.int64)


def nearest_labels(lab, out_shape):
    return np.asarray(lab)[np.ix_(*[nearest_index(n, int(m)) for n, m in zip(lab.shape[:3], out_shape)])]
