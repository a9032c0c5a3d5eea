"""sc_evaluate_segmentation (csrc/evaluate.cu) against oracle/evaluate.py: counts, volumes and the confusion matrix exact,
Dice to 1e-12, hd / hd95 / assd to 1e-9 relative, NaN in the same places."""
import ctypes
import math
import os

import numpy as np
import pytest
import torch

from oracle import evaluate as oe
from gpu_util import cuda_ctx, dev

pytestmark = pytest.mark.gpu
ANISO = (1.0, 0.7, 1.3)


@pytest.fixture(scope="module")
def ctx():
    c = cuda_ctx()
    yield c
    c.close()


def _assert_equal_metrics(got, want):
    """got: {l: {field: value}} or METRICS_DTYPE rows; want: the oracle's {l: {field: value}}"""
    for l in range(1, 15):
        g = got[l] if isinstance(got, dict) else got[l - 1]
        w = want[l]
        for f in ("n_seg", "n_ref", "n_both", "vol_seg_mm3", "vol_ref_mm3"):
            assert g[f] == w[f], (l, f, g[f], w[f])
        for f in ("dice", "hd_mm", "hd95_mm", "assd_mm"):
            gv, wv = float(g[f]), float(w[f])
            if math.isnan(wv):
                assert math.isnan(gv), (l, f, gv)
            else:
                tol = 1e-12 if f == "dice" else 1e-9 * wv + 1e-12
                assert abs(gv - wv) <= tol, (l, f, gv, wv)


def _check(ctx, seg, ref, spacing):
    want, wconf = oe.evaluate(seg, ref, spacing)
    rows, conf = ctx.evaluate_segmentation(dev(seg), dev(ref), spacing, confusion=True)
    _assert_equal_metrics(rows, want)
    assert np.array_equal(conf, wconf)
    return rows


def _blobs(shape, rng, n_blobs, classes, noise=0.02):
    ref = np.zeros(shape, np.uint8)
    for _ in range(n_blobs):
        c = [rng.randint(0, s) for s in shape]
        r = [rng.randint(1, 6) for _ in shape]
        ref[tuple(slice(max(0, ci - ri), min(s, ci + ri + 1)) for ci, ri, s in zip(c, r, shape))] = classes[rng.randint(len(classes))]
    seg = ref.copy()
    shift = rng.randint(-1, 2, size=3)                          # a slightly displaced segmentation ...
    seg = np.roll(seg, tuple(shift), axis=(0, 1, 2))
    for a in (seg, ref):                                         # ... and scattered labels (15 included) in both
        m = rng.rand(*shape) < noise
        a[m] = rng.randint(0, 16, size=int(m.sum()))
    return seg, ref


@pytest.mark.parametrize("spacing", [(1.0, 1.0, 1.0), ANISO])
@pytest.mark.parametrize("shape,seed", [((40, 36, 30), 0), ((33, 17, 9), 1), ((1, 24, 20), 2), ((27, 1, 31), 3), ((64, 50, 47), 4)])
def test_random_blobs_equal_oracle(ctx, shape, seed, spacing):
    rng = np.random.RandomState(seed)
    seg, ref = _blobs(shape, rng, 40, list(range(1, 15)))
    rows = _check(ctx, seg, ref, spacing)
    assert np.isfinite(rows["hd_mm"]).sum() >= 3                 # the distance path ran for several classes


def test_edge_cases(ctx):
    shape = (20, 18, 16)
    seg = np.zeros(shape, np.uint8)
    ref = np.zeros_like(seg)
    seg[2:5, 2:5, 2:5] = 1                # only in seg
    ref[10:13, 2:5, 2:5] = 2              # only in ref; class 3 in neither
    ref[0:20, 0:18, 12:16] = 4            # touches every face but z = 0 ...
    seg[0:20, 0:18, 11:16] = 4            # ... and its segmentation one plane thicker
    seg[7, 9, 3] = 5                      # single voxels
    ref[7, 9, 5] = 5
    seg[15, 3, 8] = 6
    ref[15, 3, 8] = 6
    ref[0, 0, 0] = 7                      # a corner voxel against a far one
    seg[19, 17, 10] = 7
    rows = _check(ctx, seg, ref, ANISO)
    assert np.isnan(rows[0]["hd_mm"]) and rows[0]["dice"] == 0.0
    assert np.isnan(rows[2]["dice"])
    assert rows[4]["hd_mm"] == rows[4]["hd95_mm"] == pytest.approx(2 * 1.3) and rows[4]["n_both"] == 0
    assert rows[5]["hd_mm"] == 0.0 and rows[5]["dice"] == 1.0


def test_whole_volume_one_class_and_full_faces(ctx):
    full = np.full((9, 7, 5), 3, np.uint8)
    rows = _check(ctx, full, full, ANISO)
    assert rows[2]["dice"] == 1.0 and rows[2]["hd_mm"] == 0.0
    other = full.copy()
    other[4:, :, :] = 8                   # two classes filling the volume, each touching five faces
    _check(ctx, full, other, ANISO)
    _check(ctx, other, full, (2.0, 1.0, 0.5))


def test_same_pointer(ctx):
    rng = np.random.RandomState(7)
    seg, _ = _blobs((30, 26, 22), rng, 30, list(range(1, 15)))
    d = dev(seg)
    want, wconf = oe.evaluate(seg, seg, ANISO)
    rows, conf = ctx.evaluate_segmentation(d, d, ANISO, confusion=True)
    _assert_equal_metrics(rows, want)
    assert np.array_equal(conf, wconf)
    assert all(rows[l - 1]["hd_mm"] == 0.0 for l in range(1, 15) if rows[l - 1]["n_seg"])


def test_bad_input_is_rejected_and_the_next_call_succeeds(ctx):
    from cnn_cort import _native
    rng = np.random.RandomState(3)
    seg, ref = _blobs((16, 14, 12), rng, 12, [1, 2, 3])
    for which in ("seg", "ref"):
        bad = (seg if which == "seg" else ref).copy()
        bad[3, 4, 5] = 16
        args = (dev(bad), dev(ref)) if which == "seg" else (dev(seg), dev(bad))
        with pytest.raises(_native.NativeError, match=which):
            ctx.evaluate_segmentation(*args, ANISO)
        _check(ctx, seg, ref, ANISO)
    for sp in ((0.0, 1.0, 1.0), (1.0, -1.0, 1.0), (1.0, 1.0, float("nan")), (float("inf"), 1.0, 1.0)):
        with pytest.raises(_native.NativeError, match="spacing"):
            ctx.evaluate_segmentation(dev(seg), dev(ref), sp)
    lib, d_seg, d_ref = ctx.lib, dev(seg), dev(ref)
    dims = (ctypes.c_int32 * 3)(*seg.shape)
    sp = (ctypes.c_double * 3)(1.0, 1.0, 1.0)
    out = np.zeros(14, _native.METRICS_DTYPE)
    for args in ((None, d_ref.data_ptr(), dims, sp, out.ctypes.data), (d_seg.data_ptr(), None, dims, sp, out.ctypes.data),
                 (d_seg.data_ptr(), d_ref.data_ptr(), None, sp, out.ctypes.data), (d_seg.data_ptr(), d_ref.data_ptr(), dims, None, out.ctypes.data),
                 (d_seg.data_ptr(), d_ref.data_ptr(), dims, sp, None), (d_seg.data_ptr(), d_ref.data_ptr(), (ctypes.c_int32 * 3)(0, 4, 4), sp, out.ctypes.data)):
        assert lib.sc_evaluate_segmentation(ctx.h, *args, None, None) == -2
    assert not out.view(np.uint8).any()   # outputs untouched on an error
    assert lib.sc_evaluate_segmentation(None, d_seg.data_ptr(), d_ref.data_ptr(), dims, sp, out.ctypes.data, None, None) == -2
    _check(ctx, seg, ref, ANISO)


def test_host_arrays_of_any_label_dtype(ctx):
    from cnn_cort import base
    rng = np.random.RandomState(11)
    seg, ref = _blobs((22, 20, 18), rng, 20, list(range(1, 15)))
    want, wconf = oe.evaluate(seg, ref, ANISO)
    for s, r in ((seg.astype(np.float32), ref.astype(np.int16)), (np.asfortranarray(seg.astype(np.float64)), torch.from_numpy(ref).cuda())):
        got, conf = base.evaluate_segmentation(s, r, ANISO, device=0)
        _assert_equal_metrics(got, want)
        assert np.array_equal(conf, wconf)
    with pytest.raises(ValueError, match="non-integral"):
        base.evaluate_segmentation(seg + np.float32(0.5), ref, device=0)
    with pytest.raises(ValueError, match="negative"):
        base.evaluate_segmentation(seg.astype(np.int32) - 1, ref, device=0)
    big = seg.astype(np.int32)
    big[0, 0, 0] = 300                    # above 15, whatever the width: rejected by the library, naming the input
    from cnn_cort import _native
    with pytest.raises(_native.NativeError, match="seg"):
        base.evaluate_segmentation(big, ref, device=0)


def test_segmented_subject_256_with_scattered_false_positives(ctx, tmp_path, weights_path):
    """A synthetic 256^3 subject with manual labels and 1.2 mm voxels, segmented by segment_arrays, plus scattered false
    positives so that the class boxes span the volume; scored from the device label volume and through evaluate_scan."""
    from cnn_cort import base, nets, nifti, synthetic
    from oracle import network as on
    ctx.load_weights(nets.pack_params(on.load_params(weights_path)))
    zoom = 1.2
    d = synthetic.write_subject(str(tmp_path), "s01", shape=(256, 256, 256), seed=1234, with_labels=True, zoom=zoom)
    t1 = nifti.load(os.path.join(d, "T1.nii.gz")).get_data()
    atlas = nifti.load(os.path.join(d, "tmp", "MNI_sub_probabilities.nii.gz")).get_data()
    mask = nifti.load(os.path.join(d, "tmp", "MNI_subcortical_mask.nii.gz")).get_data()
    lab, _, _ = base.segment_arrays(ctx, t1, atlas, crop_mask=mask)
    seg = np.array(lab)
    rng = np.random.RandomState(0)
    noise = rng.rand(*seg.shape) < 1e-4
    seg[noise] = rng.randint(1, 15, size=int(noise.sum()))
    ref_path = os.path.join(d, "gt_15_classes.nii.gz")
    ref_nii = nifti.load(ref_path)
    ref = ref_nii.get_data()
    spacing = tuple(float(s) for s in np.sqrt((ref_nii.affine[:3, :3] ** 2).sum(0)))    # 1.2 as the header stores it
    assert spacing[0] == pytest.approx(zoom)
    want, wconf = oe.evaluate(seg, ref, spacing)
    assert sum(want[l]["n_both"] for l in range(1, 15)) > 0
    assert min(want[l]["n_seg"] for l in range(1, 15)) > 0
    rows, conf = ctx.evaluate_segmentation(dev(seg), dev(ref), spacing, confusion=True)
    _assert_equal_metrics(rows, want)
    assert np.array_equal(conf, wconf)
    seg_path = os.path.join(d, "out_subcortical_rawseg.nii.gz")
    nifti.Nifti1Image(seg.astype(t1.dtype), affine=np.diag([zoom, zoom, zoom, 1.0])).to_filename(seg_path)
    got, conf = base.evaluate_scan(seg_path, ref_path, device=0)
    _assert_equal_metrics(got, want)
    assert np.array_equal(conf, wconf)
