"""Oracle: per-structure segmentation metrics (Dice, volumes, surface distances), restated with numpy + scipy.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  The usual host evaluation (scipy / medpy style) written out as the
definition that ``sc_evaluate_segmentation`` is checked against, number for number:

* labels 0..15, 15 counts as background (0) in both volumes (training does the same, ``base.py`` ``y[y == 15] = 0``);
  any value above 15 is an error;
* per structure l = 1..14, A = (seg == l), B = (ref == l): counts, Dice (NaN when both are empty), volumes in mm^3;
* surface S(M) = M & ~binary_erosion(M, 6-connected, border_value=0); d_AB = distance from each voxel of S(A) to the
  nearest voxel of S(B) in mm (exact Euclidean distance with the voxel spacing), d_BA the other way round;
  hd = max of both, hd95 = np.percentile(hstack(d_AB, d_BA), 95), assd = (mean d_AB + mean d_BA) / 2; NaN when A or B
  is empty;
* confusion[r][s] = voxels with reference class r and segmentation class s (after 15 -> 0).

The distance transforms run on the bounding box of S(A) | S(B): every feature and every query voxel lies inside it, so
the result equals the whole-volume transform.
"""
import numpy as np
from scipy import ndimage

FIELDS = ("n_seg", "n_ref", "n_both", "dice", "vol_seg_mm3", "vol_ref_mm3", "hd_mm", "hd95_mm", "assd_mm")
_STRUCT = ndimage.generate_binary_structure(3, 1)


def surface(m):
    """voxels of m with a 6-neighbour outside m or outside the volume"""
    return m & ~ndimage.binary_erosion(m, structure=_STRUCT)


def _labels(a, name):
    a = np.asarray(a)
    if a.ndim != 3:
        raise ValueError("%s must be a 3-D label volume, got shape %s" % (name, a.shape))
    if a.size and (a.min() < 0 or a.max() > 15):
        raise ValueError("%s holds a label outside 0..15" % name)
    a = a.astype(np.int64)
    a[a == 15] = 0
    return a


def surface_distances(sa, sb, spacing):
    """(d_AB, d_BA) of two non-empty surface masks"""
    box = tuple(slice(i.min(), i.max() + 1) for i in np.nonzero(sa | sb))
    sa, sb = sa[box], sb[box]
    d_ab = ndimage.distance_transform_edt(~sb, sampling=spacing)[sa]
    d_ba = ndimage.distance_transform_edt(~sa, sampling=spacing)[sb]
    return d_ab, d_ba


def evaluate(seg, ref, spacing=(1.0, 1.0, 1.0)):
    """-> ({l: {field: value}} for l = 1..14, confusion int64 [15, 15])"""
    seg, ref = _labels(seg, "seg"), _labels(ref, "ref")
    if seg.shape != ref.shape:
        raise ValueError("seg and ref shapes differ: %s vs %s" % (seg.shape, ref.shape))
    sx, sy, sz = (float(s) for s in spacing)
    confusion = np.bincount((ref * 15 + seg).ravel(), minlength=225).reshape(15, 15).astype(np.int64)
    out = {}
    for l in range(1, 15):
        a, b = seg == l, ref == l
        na, nb, nab = int(a.sum()), int(b.sum()), int((a & b).sum())
        r = dict(n_seg=na, n_ref=nb, n_both=nab, dice=2 * nab / (na + nb) if na + nb else float("nan"),
                 vol_seg_mm3=na * sx * sy * sz, vol_ref_mm3=nb * sx * sy * sz,
                 hd_mm=float("nan"), hd95_mm=float("nan"), assd_mm=float("nan"))
        if na and nb:
            d_ab, d_ba = surface_distances(surface(a), surface(b), (sx, sy, sz))
            r.update(hd_mm=float(max(d_ab.max(), d_ba.max())), hd95_mm=float(np.percentile(np.hstack((d_ab, d_ba)), 95)),
                     assd_mm=float((d_ab.mean() + d_ba.mean()) / 2))
        out[l] = r
    return out, confusion
