"""oracle/evaluate.py on hand-computed cases: the definitions sc_evaluate_segmentation is checked against."""
import math

import numpy as np
import pytest

from oracle import evaluate as oe


def _cube_pair(axis, k, shape=(20, 18, 16), lo=4, size=5, label=5):
    seg = np.zeros(shape, np.uint8)
    ref = np.zeros_like(seg)
    sl = [slice(lo, lo + size)] * 3
    seg[tuple(sl)] = label
    sl[axis] = slice(lo + k, lo + k + size)
    ref[tuple(sl)] = label
    return seg, ref


@pytest.mark.parametrize("axis", [0, 1, 2])
@pytest.mark.parametrize("k", [1, 3])
def test_shifted_cube_hausdorff_is_shift_times_spacing(axis, k):
    spacing = (2.0, 0.7, 1.3)
    seg, ref = _cube_pair(axis, k)
    m, _ = oe.evaluate(seg, ref, spacing)
    r = m[5]
    assert r["hd_mm"] == pytest.approx(k * spacing[axis], rel=1e-12)
    assert r["n_seg"] == r["n_ref"] == 125 and r["n_both"] == 25 * (5 - k)
    assert r["dice"] == pytest.approx(2 * 25 * (5 - k) / 250)
    assert r["vol_seg_mm3"] == pytest.approx(125 * 2.0 * 0.7 * 1.3)
    assert 0 < r["assd_mm"] <= r["hd95_mm"] <= r["hd_mm"]


def test_identical_volumes():
    rng = np.random.RandomState(0)
    seg = rng.randint(0, 16, (12, 10, 9)).astype(np.uint8)
    m, conf = oe.evaluate(seg, seg, (1.0, 0.7, 1.3))
    for l in range(1, 15):
        r = m[l]
        assert r["n_seg"] == r["n_ref"] == r["n_both"] == int(((seg == l)).sum())
        assert r["dice"] == 1.0
        assert r["hd_mm"] == r["hd95_mm"] == r["assd_mm"] == 0.0
    assert (conf == np.diag(np.diag(conf))).all()


def test_empty_and_nan_conventions():
    seg = np.zeros((8, 8, 8), np.uint8)
    ref = np.zeros_like(seg)
    seg[1:3, 1:3, 1:3] = 2          # only in seg
    ref[5:7, 5:7, 5:7] = 3          # only in ref
    m, conf = oe.evaluate(seg, ref)
    assert m[2]["dice"] == 0.0 and m[3]["dice"] == 0.0
    assert math.isnan(m[4]["dice"])                       # in neither
    for l in (2, 3, 4):
        assert all(math.isnan(m[l][f]) for f in ("hd_mm", "hd95_mm", "assd_mm"))
    assert m[4]["n_seg"] == m[4]["n_ref"] == 0 and m[4]["vol_seg_mm3"] == 0.0
    assert conf[0, 2] == 8 and conf[3, 0] == 8 and conf.sum() == 512


def test_fifteen_counts_as_background():
    seg = np.zeros((6, 6, 6), np.uint8)
    ref = np.zeros_like(seg)
    seg[1:4, 1:4, 1:4] = 1
    ref[1:4, 1:4, 1:4] = 1
    seg[0] = 15                      # a background ring in one volume only changes nothing
    ref[:, 0] = 15
    m, conf = oe.evaluate(seg, ref)
    m0, conf0 = oe.evaluate(np.where(seg == 15, 0, seg), np.where(ref == 15, 0, ref))
    for l in range(1, 15):
        assert np.array_equal([m[l][f] for f in oe.FIELDS], [m0[l][f] for f in oe.FIELDS], equal_nan=True)
    assert (conf == conf0).all()
    assert m[1]["dice"] == 1.0 and m[1]["hd_mm"] == 0.0


def test_label_above_fifteen_is_an_error():
    seg = np.zeros((4, 4, 4), np.uint8)
    bad = seg.copy()
    bad[1, 2, 3] = 16
    with pytest.raises(ValueError, match="ref"):
        oe.evaluate(seg, bad)
    with pytest.raises(ValueError, match="seg"):
        oe.evaluate(bad, seg)


def test_surface_touching_the_border():
    m = np.ones((3, 4, 5), bool)
    assert oe.surface(m).sum() == m.size - 1 * 2 * 3    # only the interior voxels are not on the surface


def test_percentile_on_a_tiny_list():
    # S(A) = one voxel, S(B) = a 2-voxel bar: d_AB = [1], d_BA = [1, 2]; hstack = [1, 1, 2]
    # numpy linear percentile 95: h = 0.95 * 2 = 1.9 -> 1 + 0.9 * (2 - 1) = 1.9
    seg = np.zeros((1, 1, 6), np.uint8)
    ref = np.zeros_like(seg)
    seg[0, 0, 1] = 7
    ref[0, 0, 2:4] = 7
    m, _ = oe.evaluate(seg, ref)
    assert m[7]["hd_mm"] == 2.0
    assert m[7]["hd95_mm"] == pytest.approx(1.9, rel=1e-12)
    assert m[7]["assd_mm"] == pytest.approx((1.0 + 1.5) / 2)
