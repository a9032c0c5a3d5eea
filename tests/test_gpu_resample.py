"""Resampling to the network's grid: sc_resample_volume / sc_map_proba_back against the fp64 oracle (tests/resample_oracle.py),
the identity of the option on a 1 mm scan, segment_arrays and the training set end to end on an anisotropic subject, and the
argument errors."""
import os
import random

import numpy as np
import pytest
import torch

from gpu_util import cuda_ctx, dev
import resample_oracle as ro

pytestmark = pytest.mark.gpu

OPTIONS = {'experiment': 'miccai2012_v1', 'patch_size': [32, 32], 'mode': 'cuda0', 'device': 0, 'load_weights': 'True',
           'net_verbose': 0, 'train_split': 0.25, 'max_epochs': 1, 'patience': 1, 'batch_size': 128, 'test_batch_size': 5000,
           'debug': 'False', 'out_probabilities': 'True', 'post_process': 'False', 't1_name': 'T1.nii.gz',
           'roi_name': 'gt_15_classes.nii.gz', 'mc_samples': 0, 'mc_seed': 0, 'resample_mm': None, 'crop': 'True',
           'crop_bool': True}


@pytest.fixture(scope="module")
def ctx():
    c = cuda_ctx()
    yield c
    c.close()


@pytest.fixture(scope="module")
def net(weights_path):
    from cnn_cort import nets
    cuda_ctx().close()                   # skips without a GPU
    return nets.build_model(os.path.dirname(os.path.dirname(weights_path)), dict(OPTIONS))


# ---- kernels against the oracle ------------------------------------------------------------------------------------------
RESAMPLE_CASES = [
    ((37, 29, 41), (26, 20, 29)),        # down on every axis, odd non-cubic
    ((17, 23, 9), (29, 31, 13)),         # up on every axis
    ((40, 7, 13), (13, 19, 13)),         # mixed: down, up, r = 1
    ((21, 6, 11), (1, 6, 4)),            # m = 1
    ((320, 5, 3), (224, 5, 3)),          # 0.7 mm -> 1 mm along a long axis
]


@pytest.mark.parametrize("channels", [1, 15])
@pytest.mark.parametrize("shape,out_shape", RESAMPLE_CASES)
def test_resample_vs_oracle(ctx, shape, out_shape, channels):
    rng = np.random.RandomState(sum(shape) + channels)
    if channels == 1:
        vol = (rng.randn(*shape) * 100 + 20).astype(np.float32)
    else:
        vol = rng.dirichlet(np.ones(15) * 0.3, size=shape).astype(np.float32)
    d = dev(vol)
    out = ctx.resample_volume(d, out_shape)
    ref = ro.resample(vol.astype(np.float64), out_shape)
    got = out.cpu().numpy()
    assert got.shape == ref.shape
    assert np.abs(got - ref).max() <= 2e-6 * np.abs(vol).max()
    again = ctx.resample_volume(d, out_shape)
    assert torch.equal(out.view(torch.int32), again.view(torch.int32))          # byte-identical
    if channels == 15:
        assert got.min() >= 0 and np.abs(got.sum(-1) - 1).max() < 1e-5


@pytest.mark.parametrize("channels", [1, 15])
def test_resample_identity_is_exact(ctx, channels):
    shape = (19, 8, 27) + ((15,) if channels == 15 else ())
    vol = torch.randn(shape, device="cuda")
    assert torch.equal(ctx.resample_volume(vol, shape[:3]).view(torch.int32), vol.view(torch.int32))


MAP_CASES = [((26, 20, 29), (37, 29, 41)), ((29, 31, 13), (17, 23, 9)), ((13, 19, 13), (40, 7, 13)), ((1, 6, 4), (21, 6, 11))]


@pytest.mark.parametrize("use_mask", [False, True])
@pytest.mark.parametrize("tshape,nshape", MAP_CASES)
def test_map_proba_back_vs_oracle(ctx, tshape, nshape, use_mask):
    rng = np.random.RandomState(sum(tshape) + sum(nshape) + use_mask)
    proba = rng.dirichlet(np.ones(15) * 0.5, size=tshape).astype(np.float32)
    cand = (rng.rand(*tshape) < 0.7).astype(np.uint8)
    nmask = (rng.rand(*nshape) < 0.8).astype(np.uint8) if use_mask else None
    p_ref, l_ref, written, gap = ro.map_proba_back(proba.astype(np.float64), cand, nshape, nmask)
    d_proba, d_cand, d_mask = dev(proba), dev(cand), (dev(nmask) if use_mask else None)
    outs = []
    for _ in range(2):
        lab = torch.full(nshape, 99, dtype=torch.uint8, device="cuda")
        prob = torch.full(nshape + (15,), -1.0, device="cuda")
        ctx.map_proba_back(d_proba, d_cand, nshape, native_mask=d_mask, label_out=lab, proba_out=prob)
        outs.append((lab.cpu().numpy(), prob.cpu().numpy()))
    (lab, prob), (lab2, prob2) = outs
    assert np.array_equal(lab, lab2) and np.array_equal(prob.view(np.int32), prob2.view(np.int32))
    assert written.any()
    assert (lab[~written] == 99).all() and (prob[~written] == -1.0).all()
    assert (lab[written] != 99).all()
    assert np.abs(prob[written] - p_ref[written]).max() < 1e-6
    sure = written & (gap > 1e-5)
    assert np.array_equal(lab[sure], l_ref[sure])
    # labels only: the probability output is optional
    lab3, none = ctx.map_proba_back(d_proba, d_cand, nshape, native_mask=d_mask)
    assert none is None and np.array_equal(lab3.cpu().numpy()[written], lab[written])


def test_argument_errors(ctx):
    from cnn_cort._native import NativeError, _dims
    lib, h = ctx.lib, ctx.h
    vol = torch.full((6, 5, 4), 7.0, device="cuda")
    out = torch.full((3, 5, 4), -1.0, device="cuda")
    p, c = vol.data_ptr(), out.data_ptr()

    def err(status, name):
        assert status == -2, status
        assert name in lib.sc_last_error().decode()

    err(lib.sc_resample_volume(h, None, _dims(vol.shape), 1, _dims(out.shape), c, None), "in_dev")
    err(lib.sc_resample_volume(h, p, _dims(vol.shape), 1, _dims(out.shape), None, None), "out_dev")
    err(lib.sc_resample_volume(h, p, _dims((6, 0, 4)), 1, _dims(out.shape), c, None), "in_dims")
    err(lib.sc_resample_volume(h, p, _dims(vol.shape), 1, _dims((3, 5, 0)), c, None), "out_dims")
    err(lib.sc_resample_volume(h, p, _dims(vol.shape), 3, _dims(out.shape), c, None), "channels")
    err(lib.sc_resample_volume(h, p, _dims(vol.shape), 1, _dims(vol.shape), p, None), "out_dev == in_dev")
    assert bool((out == -1.0).all()) and bool((vol == 7.0).all())
    proba = torch.full((3, 5, 4, 15), 1.0 / 15, device="cuda")
    cand = torch.ones((3, 5, 4), dtype=torch.uint8, device="cuda")
    lab = torch.full((6, 5, 4), 99, dtype=torch.uint8, device="cuda")
    po = torch.full((6, 5, 4, 15), -1.0, device="cuda")
    pp, cp, lp, op = proba.data_ptr(), cand.data_ptr(), lab.data_ptr(), po.data_ptr()
    td, nd = _dims(cand.shape), _dims(lab.shape)
    err(lib.sc_map_proba_back(h, None, cp, td, None, nd, lp, op, None), "proba_dev")
    err(lib.sc_map_proba_back(h, pp, None, td, None, nd, lp, op, None), "cand_dev")
    err(lib.sc_map_proba_back(h, pp, cp, td, None, nd, None, op, None), "label_dev")
    err(lib.sc_map_proba_back(h, pp, cp, _dims((0, 5, 4)), None, nd, lp, op, None), "target_dims")
    err(lib.sc_map_proba_back(h, pp, cp, td, None, _dims((6, 5, -1)), lp, op, None), "native_dims")
    err(lib.sc_map_proba_back(h, pp, cp, td, None, nd, lp, pp, None), "proba_out_dev == proba_dev")
    err(lib.sc_map_proba_back(h, pp, cp, td, None, nd, cp, op, None), "label_dev == cand_dev")
    assert bool((lab == 99).all()) and bool((po == -1.0).all())
    with pytest.raises(NativeError, match="channels"):
        ctx.resample_volume(torch.zeros((4, 4, 4, 3), device="cuda"), (2, 2, 2))


# ---- the option on a 1 mm scan changes nothing ---------------------------------------------------------------------------
def _read_outputs(d):
    from cnn_cort import nifti
    out = {}
    for f in sorted(os.listdir(d)):
        if f.startswith('out_'):
            img = nifti.load(os.path.join(d, f))
            out[f] = (np.asarray(img.get_data()).copy(), np.asarray(img.affine).copy())
    return out


@pytest.mark.parametrize("crop", [False, True])
def test_test_scan_identity_at_1mm(net, tmp_path, crop):
    from cnn_cort import base, synthetic
    root = str(tmp_path)
    d = synthetic.write_subject(root, "s01", shape=(48, 44, 40), seed=5)
    results = []
    for mm in (None, 1.0):
        options = dict(OPTIONS, test_folder=root, crop=str(crop), crop_bool=crop, resample_mm=mm)
        t1_names, _ = base.load_test_names(options)
        base.test_scan(net, t1_names[0], options)
        results.append(_read_outputs(d))
    a, b = results
    assert sorted(a) == sorted(b) == ['out_subcortical_prob.nii.gz', 'out_subcortical_rawseg.nii.gz']
    for k in a:
        assert a[k][0].dtype == b[k][0].dtype and np.array_equal(a[k][0], b[k][0]) and np.array_equal(a[k][1], b[k][1]), k


def test_training_set_identity_at_1mm(tmp_path):
    from cnn_cort import base, synthetic
    cuda_ctx().close()
    root = str(tmp_path)
    for k in range(2):
        synthetic.write_subject(root, "s%02d" % k, shape=(40, 36, 32), seed=10 + k, with_labels=True)
    arrays = []
    for mm in (None, 1.0):
        random.seed(3)
        np.random.seed(3)
        scans = base.load_scan_training_set(dict(OPTIONS, train_folder=root, resample_mm=mm))
        arrays.append(scans.to_arrays())
    for x, y in zip(*arrays):
        assert x.dtype == y.dtype and np.array_equal(x.view(np.uint8), y.view(np.uint8))


# ---- end to end on an anisotropic subject ---------------------------------------------------------------------------------
SPACING = (0.8, 0.8, 1.2)
NSHAPE = (80, 72, 64)


def _aniso_subject(root, name="a01", seed=21):
    """a synthetic subject on an (0.8, 0.8, 1.2) mm grid: T1 with per-structure contrast, priors, registered mask and labels"""
    from cnn_cort import nifti, synthetic
    d = os.path.join(root, name)
    os.makedirs(os.path.join(d, "tmp"), exist_ok=True)
    aff = np.diag(list(SPACING) + [1.0])
    atlas, _, _ = synthetic.make_atlas(NSHAPE, seed)
    labels = synthetic.make_labels(atlas)
    t1 = synthetic.make_t1(NSHAPE, seed) + np.float32(120.0) * (labels % 4).astype(np.float32)
    mask = synthetic.make_mask(atlas)
    nifti.Nifti1Image(t1.astype(np.float32), aff).to_filename(os.path.join(d, "T1.nii.gz"))
    nifti.Nifti1Image(atlas, aff).to_filename(os.path.join(d, "tmp", "MNI_sub_probabilities.nii.gz"))
    nifti.Nifti1Image(mask, aff).to_filename(os.path.join(d, "tmp", "MNI_subcortical_mask.nii.gz"))
    nifti.Nifti1Image(labels, aff).to_filename(os.path.join(d, "gt_15_classes.nii.gz"))
    return d, t1.astype(np.float32), atlas, mask, labels


@pytest.mark.parametrize("crop", [False, True])
def test_segment_arrays_vs_composition(net, tmp_path, crop):
    from cnn_cort import base
    ctx = net.ctx
    _, t1, atlas, mask, _ = _aniso_subject(str(tmp_path))
    tshape = ro.target_dims(NSHAPE, SPACING, 1.0)
    assert tshape == (64, 58, 77)
    # the composition: oracle resampling, the existing device pass on the target grid, oracle back-mapping
    t1r = dev(ro.resample(t1, tshape).astype(np.float32))
    raw = t1r.view(-1).view(torch.uint8)
    vol, _, _ = ctx.normalise_volume(raw, np.float32, tshape)
    if crop:
        rm = dev(ro.resample(mask, tshape).astype(np.float32))
        cand = ctx.dilate_mask(ctx.candidate_mask(rm.view(-1).view(torch.uint8), np.float32, tshape), 10)
    else:
        cand = ctx.candidate_mask(raw, np.float32, tshape)
    box, _ = ctx.mask_bbox(cand)
    tl = torch.zeros(tshape, dtype=torch.uint8, device="cuda")
    tp = torch.zeros(tshape + (15,), dtype=torch.float32, device="cuda")
    ctx.segment_volume(vol, dev(ro.resample(atlas, tshape).astype(np.float32)), box=box, cand_mask=cand, label_vol=tl, proba_vol=tp)
    p_ref, l_ref, written, gap = ro.map_proba_back(tp.cpu().numpy(), cand.cpu().numpy(), NSHAPE, None if crop else t1 != 0)
    lab, prob, n_cand = base.segment_arrays(ctx, t1, atlas, crop_mask=mask if crop else None, want_proba=True, spacing=SPACING,
                                            resample_mm=1.0)
    lab, prob = lab.copy(), prob.copy()
    assert lab.shape == NSHAPE and prob.shape == NSHAPE + (15,)
    assert n_cand == int(cand.sum())
    assert written.sum() > 1000 and (lab[~written] == 0).all() and (prob[~written] == 0).all()
    agree = lab[written] == l_ref[written]
    assert agree.mean() >= 0.999, agree.mean()
    assert (gap[written][~agree] < 2e-2).all(), gap[written][~agree].max()
    assert np.array_equal(lab[written], prob[written].argmax(-1))


def test_training_set_on_target_grid(tmp_path):
    from cnn_cort import base
    ctx = cuda_ctx()
    ctx.close()
    root = str(tmp_path)
    _, t1, atlas, _, labels = _aniso_subject(root)
    tshape = ro.target_dims(NSHAPE, SPACING, 1.0)
    random.seed(7)
    scans = base.load_scan_training_set(dict(OPTIONS, train_folder=root, resample_mm=1.0), randomize=False)
    assert tuple(scans.volumes[0].shape) == tshape
    lab_t = ro.nearest_labels(labels, tshape)
    s = scans.samples.cpu().numpy()
    x, y, z = s[:, 1], s[:, 2], s[:, 3]
    assert (s[:, 0] == 0).all()
    pos = int(((lab_t > 0) & (lab_t < 15)).sum())
    assert pos > 0 and len(s) == pos + min(pos, int((lab_t == 15).sum()))
    expect = lab_t[x, y, z].astype(np.uint8)
    expect[expect == 15] = 0
    assert np.array_equal(scans.y, expect)
    pri = ro.resample(atlas, tshape)[x, y, z]
    assert np.abs(scans.atlas.cpu().numpy() - pri).max() <= 2e-6
    vol = ro.resample(t1, tshape).astype(np.float32)
    assert np.allclose(scans.volumes[0].cpu().numpy(), base._train_normalise(vol), rtol=0, atol=1e-4)


# ---- what the option does not cover -----------------------------------------------------------------------------------------
def test_unsupported_combinations_raise(net, tmp_path):
    from cnn_cort import base, synthetic
    root = str(tmp_path)
    synthetic.write_subject(root, "s01", shape=(40, 36, 32), seed=4, with_labels=True)
    options = dict(OPTIONS, test_folder=root, train_folder=root, crop='True', crop_bool=True, resample_mm=1.0)
    t1_names, _ = base.load_test_names(options)
    with pytest.raises(ValueError, match="resample_mm"):
        base.test_scan(net, t1_names[0], dict(options, inference='patchwise'))
    with pytest.raises(ValueError, match="resample_mm"):
        base.test_scan(net, t1_names[0], dict(options, mc_samples=4))
    with pytest.raises(ValueError, match="resample_mm"):
        base.load_data(options)
    with pytest.raises(ValueError, match="spacing"):
        base.segment_arrays(net.ctx, np.ones((8, 8, 8), np.float32), np.zeros((8, 8, 8, 15), np.float32), resample_mm=1.0)
