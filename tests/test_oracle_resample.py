"""The resampling oracle (tests/resample_oracle.py) against torch's antialiased interpolation, its invariants, the target-grid rule
of cnn_cort.base.resample_dims and the parsing of [model] resample_mm.  CPU only."""
import configparser

import numpy as np
import pytest
import torch

import resample_oracle as ro

SHAPES = [((17, 23, 9), (11, 31, 9)), ((40, 7, 13), (13, 19, 1)), ((5, 6, 7), (10, 3, 7)), ((1, 8, 12), (1, 5, 12))]


def _torch_antialias(vol, out_shape):
    """torch.nn.functional.interpolate(mode='bilinear', antialias=True, align_corners=False) over (x, y), then over (y, z)"""
    F = torch.nn.functional
    t = torch.from_numpy(np.asarray(vol, np.float64)).permute(2, 0, 1)[None]          # [1, Z, X, Y]
    t = F.interpolate(t, size=(out_shape[0], out_shape[1]), mode='bilinear', antialias=True, align_corners=False)
    t = t[0].permute(1, 2, 0)[None]                                                    # [1, X', Y', Z]
    t = F.interpolate(t, size=(out_shape[1], out_shape[2]), mode='bilinear', antialias=True, align_corners=False)
    return t[0].numpy()


@pytest.mark.parametrize("shape,out_shape", SHAPES)
def test_oracle_equals_torch_antialias(shape, out_shape):
    vol = np.random.RandomState(sum(shape)).randn(*shape)
    ref = _torch_antialias(vol, out_shape)
    got = ro.resample(vol, out_shape)
    assert got.shape == tuple(out_shape)
    assert np.abs(got - ref).max() < 1e-12


def test_identity_is_exact():
    vol = np.random.RandomState(1).randn(9, 10, 11)
    assert np.array_equal(ro.resample(vol, vol.shape), vol)
    assert np.array_equal(ro.weight_matrix(10, 10), np.eye(10))


@pytest.mark.parametrize("shape,out_shape", SHAPES)
def test_constants_and_prior_sums_are_kept(shape, out_shape):
    c = np.full(shape, 3.25)
    assert np.allclose(ro.resample(c, out_shape), 3.25, rtol=0, atol=1e-12)
    pri = np.random.RandomState(2).dirichlet(np.ones(15) * 0.3, size=shape)
    rp = ro.resample(pri, out_shape)
    assert rp.shape == tuple(out_shape) + (15,)
    assert rp.min() >= 0 and rp.max() <= 1 + 1e-12
    assert np.allclose(rp.sum(-1), 1.0, rtol=0, atol=1e-12)


def test_backmap_and_nearest_rules():
    i0, f = ro.backmap_axis(7, 7)
    assert np.array_equal(i0 + f, np.arange(7))
    i0, f = ro.backmap_axis(5, 1)
    assert (i0 == 0).all() and (f == 0).all()
    assert np.array_equal(ro.nearest_index(6, 6), np.arange(6))
    assert np.array_equal(ro.nearest_index(6, 3), [1, 3, 5])        # x_j = 0.5, 2.5, 4.5 rounded half up
    proba = np.random.RandomState(3).dirichlet(np.ones(15), size=(4, 5, 6))
    p, lab, written, _ = ro.map_proba_back(proba, np.ones((4, 5, 6)), (4, 5, 6))
    assert written.all() and np.allclose(p, proba, rtol=0, atol=1e-15) and np.array_equal(lab, proba.argmax(-1))


@pytest.mark.parametrize("shape,spacing,mm,expect", [
    ((320, 320, 320), (0.7, 0.7, 0.7), 1.0, (224, 224, 224)),
    ((256, 256, 256), (1.0, 1.0, 1.0), 1.0, (256, 256, 256)),
    ((176, 176, 176), (1.2, 1.2, 1.2), 1.0, (211, 211, 211)),
    ((160, 160, 160), (0.8, 0.8, 0.8), 1.0, (128, 128, 128)),
    ((1, 1, 1), (0.3, 0.3, 0.3), 1.0, (1, 1, 1)),
    ((80, 72, 64), (0.8, 0.8, 1.2), 1.0, (64, 58, 77)),
])
def test_resample_dims(shape, spacing, mm, expect):
    from cnn_cort import base
    dims, r = base.resample_dims(shape, spacing, mm)
    assert dims == expect == ro.target_dims(shape, spacing, mm)
    assert r == tuple(n / m for n, m in zip(shape, expect))


def test_nearest_index_matches_oracle():
    from cnn_cort import base
    for n, m in ((10, 7), (7, 10), (320, 224), (1, 1), (5, 1)):
        assert np.array_equal(base.nearest_index(n, m), ro.nearest_index(n, m))


def _config(**model):
    cfg = configparser.RawConfigParser()
    cfg.read_dict({
        'database': {'train_folder': 't', 'inference_folder': 'i', 't1_name': 'T1.nii.gz', 'roi_name': 'gt.nii.gz',
                     'save_tmp': 'True'},
        'model': dict({'name': 'x', 'mode': 'cuda0', 'patch_size': '32', 'train_split': '0.25', 'max_epochs': '1',
                       'patience': '1', 'batch_size': '128', 'test_batch_size': '100', 'net_verbose': '0',
                       'load_weights': 'True', 'debug': 'False', 'out_probabilities': 'False', 'post_process': 'True',
                       'speedup_segmentation': 'True'}, **model)})
    return cfg


def test_load_options_resample_mm():
    from cnn_cort.load_options import load_options
    assert load_options(_config())['resample_mm'] is None
    assert load_options(_config(resample_mm=''))['resample_mm'] is None
    assert load_options(_config(resample_mm=' 1.0 '))['resample_mm'] == 1.0
    assert load_options(_config(resample_mm='0.75'))['resample_mm'] == 0.75
    for bad in ('0', '-1', 'nan', 'inf', 'one'):
        with pytest.raises(ValueError, match="resample_mm"):
            load_options(_config(resample_mm=bad))
