"""Host-side logic of the device-resident training set (base.load_scan_training_set / ScanTrainingSet), no GPU needed:
its row order and contents follow load_data + generate_training_set for the same seeds, and malformed sample tables
are rejected before anything reaches the device."""
import os
import random

import numpy as np
import pytest

from cnn_cort import base, nifti, synthetic
from oracle import gather as og

OPTIONS = {'t1_name': 'T1.nii.gz', 'roi_name': 'gt_15_classes.nii.gz', 'patch_size': [32, 32], 'debug': 'False'}


def _cpu_centres(mask, device, balance_neg=True):
    """base._training_centres on the host: oracle.get_mask_voxels consumes Python's ``random`` exactly as
    base.get_mask_voxels does (one shuffle of range(N))"""
    pos = og.get_mask_voxels(np.logical_and(mask > 0, mask < 15))
    neg = og.get_mask_voxels(mask == 15, size=len(pos) if balance_neg else None)
    return np.concatenate([pos, neg]).astype(np.int32)


class _Captured(object):
    def __init__(self, volumes, samples, atlas_rows, labels, names=(), device=None):
        base.check_sample_table([v.shape for v in volumes], samples, atlas_rows, labels)
        self.volumes, self.samples, self.atlas_rows, self.labels, self.names = volumes, samples, atlas_rows, labels, names


class _Ctx(object):
    device = 0


def test_scan_set_rows_follow_generate_training_set(tmp_path, monkeypatch):
    root = str(tmp_path)
    for i, (name, dt) in enumerate((("s01", np.float32), ("s02", np.int16))):
        synthetic.write_subject(root, name, shape=(30 + 4 * i, 28, 26), seed=40 + i, with_labels=True, t1_dtype=dt)
    options = dict(OPTIONS, train_folder=root)
    monkeypatch.setattr(base, "_training_centres", _cpu_centres)
    monkeypatch.setattr(base, "get_context", lambda device=None: _Ctx())
    monkeypatch.setattr(base, "_dev", lambda a, device, dtype=None: np.asarray(a, dtype))
    monkeypatch.setattr(base, "ScanTrainingSet", _Captured)

    # the materialised path, built from the same host pieces: per-subject patches, labels, atlas rows
    random.seed(3)
    np.random.seed(5)
    xa, xc, xs, xat, ys = [], [], [], [], []
    vols = []
    for name in ("s01", "s02"):
        d = os.path.join(root, name)
        vol = base._train_normalise(nifti.load(os.path.join(d, "T1.nii.gz")).get_data())
        lab = nifti.load(os.path.join(d, "gt_15_classes.nii.gz")).get_data()
        atlas = nifti.load(os.path.join(d, "tmp", "MNI_sub_probabilities.nii.gz")).get_data()
        cen = _cpu_centres(lab, 0)
        for out, mode in zip((xa, xc, xs), og.VIEWS):
            out.append(og.get_patches(vol, cen, (32, 32), mode))
        yp = np.zeros((len(cen), 32, 32), np.uint8)
        yp[:, 16, 16] = lab[cen[:, 0], cen[:, 1], cen[:, 2]]
        ys.append(yp)
        xat.append(og.atlas_vectors_train(atlas, cen))
        vols.append(vol)
    ref = base.generate_training_set(xa, xc, xs, xat, ys, options)

    random.seed(3)
    np.random.seed(5)
    got = base.load_scan_training_set(options)
    n = len(ref[4])
    assert got.samples.shape == (n, 4) and got.samples.dtype == np.int32 and 0 < n
    assert np.array_equal(got.labels, ref[4]) and np.array_equal(got.atlas_rows, ref[3])
    assert [os.path.basename(os.path.dirname(p)) for p in got.names] == ["s01", "s02"]
    assert all(np.array_equal(a, b) for a, b in zip(got.volumes, vols))
    assert set(np.unique(got.samples[:, 0])) == {0, 1}
    for k in (0, 1):                      # every row's patches, cut from its own scan, are the reference's row
        rows = np.nonzero(got.samples[:, 0] == k)[0]
        for view, mode in enumerate(og.VIEWS):
            assert np.array_equal(og.get_patches(vols[k], got.samples[rows, 1:], (32, 32), mode), ref[view][rows, 0]), (k, mode)
    # randomize=False: concatenation order, positives of the first subject first
    random.seed(3)
    np.random.seed(5)
    plain = base.load_scan_training_set(options, randomize=False)
    assert (plain.samples[:len(xa[0]), 0] == 0).all() and np.array_equal(np.sort(plain.labels), np.sort(ref[4]))


def _table(n=4):
    s = np.array([[0, 1, 2, 3], [1, 0, 0, 0], [1, 6, 4, 2], [0, 4, 5, 6]][:n], np.int32)
    return s, np.zeros((n, 15), np.float32), np.zeros(n, np.uint8)


@pytest.mark.parametrize("case,match", [
    ("scan_high", "scan index 2 out of range"), ("scan_negative", "scan index -1 out of range"),
    ("centre_high", "centre .* outside scan 1"), ("centre_negative", "centre .* outside scan 0"),
    ("atlas_rows", "atlas rows must be"), ("labels", "labels must be"), ("table_shape", "sample table must be")])
def test_malformed_tables_are_rejected_before_any_device_call(case, match):
    shapes = [(5, 6, 7), (7, 5, 3)]
    vols = [np.zeros(s, np.float32) for s in shapes]
    s, a, y = _table()
    if case == "scan_high":
        s[2, 0] = 2
    elif case == "scan_negative":
        s[1, 0] = -1
    elif case == "centre_high":
        s[2, 1:] = (6, 4, 3)             # z == Z of scan 1
    elif case == "centre_negative":
        s[0, 2] = -1
    elif case == "atlas_rows":
        a = a[:3]
    elif case == "labels":
        y = np.zeros(5, np.uint8)
    else:
        s = s[:, :3]
    with pytest.raises(ValueError, match=match):
        base.check_sample_table(shapes, s, a, y)
    # the constructor validates first: on a box without a GPU any device call would raise something else
    with pytest.raises(ValueError, match=match):
        base.ScanTrainingSet(vols, s, a, y)


def test_well_formed_table_passes():
    s, a, y = _table()
    base.check_sample_table([(5, 6, 7), (7, 5, 3)], s, a, y)
    base.check_sample_table([(5, 6, 7)], np.zeros((0, 4), np.int32), np.zeros((0, 15), np.float32), np.zeros(0, np.uint8))
