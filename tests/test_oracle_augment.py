"""The augmented-gather oracle (tests/augment_oracle.py) against the plain gather oracle, exact geometry, its random
distributions and row keying, and the [model] augment_* option parsing.  CPU only."""
import configparser

import numpy as np
import pytest

import augment_oracle as ao
from oracle import gather as og

SHAPES = [(40, 36, 33), (21, 50, 28), (7, 5, 6)]     # the last one is smaller than a patch on every axis
ALL = dict(rotation_deg=30.0, scale=0.2, intensity=0.3, noise=0.1, seed=11, epoch=3)


def _table(seed=0):
    rng = np.random.RandomState(seed)
    vols = [rng.randn(*s) for s in SHAPES]
    rows = []
    for k, s in enumerate(SHAPES):
        corners = np.array([(x, y, z) for x in (0, s[0] - 1) for y in (0, s[1] - 1) for z in (0, s[2] - 1)])
        edges = np.array([(0, s[1] // 2, s[2] // 2), (s[0] - 1, 0, s[2] // 2), (s[0] // 2, s[1] - 1, 0)])
        interior = np.stack([rng.randint(0, d, 8) for d in s], 1)
        c = np.concatenate([corners, edges, interior])
        rows.append(np.concatenate([np.full((len(c), 1), k), c], 1))
    return vols, np.concatenate(rows).astype(np.int32)


def test_zero_ranges_equal_get_patches():
    vols, samples = _table()
    rows = np.random.RandomState(1).permutation(len(samples))
    for aug in ({}, dict(seed=5, epoch=7)):
        got = ao.gather(vols, samples, rows, aug)
        for v, mode in enumerate(og.VIEWS):
            for k, vol in enumerate(vols):
                m = samples[rows, 0] == k
                assert np.array_equal(got[v][m], og.get_patches(vol, samples[rows[m], 1:], (32, 32), mode)), (mode, k)


def test_linear_volume_is_sampled_at_c_plus_M_o():
    """Trilinear interpolation reproduces a linear function exactly wherever all 8 corners lie inside, so the oracle must
    equal V(c + M o) there; o is written out per view here, independently of the oracle's axis table."""
    shape = (90, 96, 84)
    coef = np.array([0.7, -1.3, 0.45])
    X, Y, Z = np.meshgrid(*[np.arange(n, dtype=np.float64) for n in shape], indexing="ij")
    vol = coef[0] * X + coef[1] * Y + coef[2] * Z + 2.0
    rng = np.random.RandomState(2)
    cen = np.stack([rng.randint(35, n - 35, 20) for n in shape], 1)
    samples = np.concatenate([np.zeros((20, 1)), cen], 1).astype(np.int32)
    aug = dict(rotation_deg=180.0, scale=0.25, intensity=0.5, seed=3, epoch=1)
    got = ao.gather([vol], samples, np.arange(20), aug)
    prm = ao.parameters(aug, np.arange(20))
    M = prm["M"]
    assert np.allclose(np.einsum("nij,nkj->nik", M, M), (prm["s"] ** 2)[:, None, None] * np.eye(3), atol=1e-12)
    assert np.allclose(np.linalg.det(M), prm["s"] ** 3, atol=1e-12)
    i = np.arange(32.0)[:, None] - 16
    j = np.arange(32.0)[None, :] - 16
    e = np.eye(3)
    rows_cols = {0: (e[0], e[1]), 1: (e[0], e[2]), 2: (e[1], e[2])}        # axial (x, y), coronal (x, z), saggital (y, z)
    for v in range(3):
        er, ec = rows_cols[v]
        for n in range(20):
            o = i[..., None] * er + j[..., None] * ec                       # [32, 32, 3]
            p = cen[n] + o @ M[n].T
            want = prm["a"][n] * (p @ coef + 2.0) + prm["b"][n]
            assert np.abs(got[v][n] - want).max() < 1e-10, (v, n)


def test_parameter_and_noise_distributions():
    aug = dict(rotation_deg=25.0, scale=0.15, intensity=0.2, noise=0.3, seed=9, epoch=2)
    rows = np.arange(100000)
    prm = ao.parameters(aug, rows)
    assert np.abs(prm["theta"]).max() <= 25.0 and np.abs(prm["theta"]).max() > 24.9
    assert prm["s"].min() >= 1 / 1.15 and prm["s"].max() <= 1.15
    assert np.abs(prm["a"] - 1).max() <= 0.2 and np.abs(prm["b"]).max() <= 0.2
    assert np.allclose(np.linalg.norm(prm["axis"], axis=1), 1.0)
    assert np.abs(prm["axis"].mean(0)).max() < 0.01                        # uniform on the sphere: mean 0, E[k k^T] = I / 3
    assert np.abs(prm["axis"].T @ prm["axis"] / len(rows) - np.eye(3) / 3).max() < 0.01
    assert abs(prm["theta"].mean()) < 0.1 and abs(np.log(prm["s"]).mean()) < 1e-3
    g = ao.noise(aug, rows[:40]).ravel()                                  # 122 880 draws
    assert abs(g.mean()) < 0.02 and abs(g.std() - 1.0) < 0.02
    vol = np.zeros((64, 64, 64))
    samples = np.array([[0, 32, 32, 32]] * 40, np.int32)
    out = np.stack(ao.gather([vol], samples, np.arange(40), dict(noise=0.3, seed=9, epoch=2)))
    assert abs(out.mean()) < 0.01 and abs(out.std() - 0.3) < 0.01


def test_rows_not_positions_key_the_draws():
    vols, samples = _table(3)
    rows = np.arange(len(samples))
    perm = np.random.RandomState(4).permutation(len(samples))
    a = ao.gather(vols, samples, rows, ALL)
    b = ao.gather(vols, samples, perm, ALL)
    for v in range(3):
        assert np.array_equal(a[v][perm], b[v])
    c = ao.gather(vols, samples, rows, dict(ALL, epoch=4))
    d = ao.gather(vols, samples, rows, dict(ALL, seed=12))
    assert not np.allclose(a[0], c[0]) and not np.allclose(a[0], d[0])


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


def test_load_options_augment():
    from cnn_cort.load_options import load_options
    assert load_options(_config())['augment'] is None
    zero = {'augment_rotation_deg': '0', 'augment_scale': '0.0', 'augment_intensity': '', 'augment_noise': '0', 'augment_seed': '5'}
    assert load_options(_config(**zero))['augment'] is None
    got = load_options(_config(augment_rotation_deg=' 10 ', augment_noise='0.05'))['augment']
    assert got == dict(rotation_deg=10.0, scale=0.0, intensity=0.0, noise=0.05, seed=0)
    got = load_options(_config(augment_rotation_deg='180', augment_scale='0.15', augment_intensity='0.99',
                               augment_seed='18446744073709551615'))['augment']
    assert got == dict(rotation_deg=180.0, scale=0.15, intensity=0.99, noise=0.0, seed=2 ** 64 - 1)
    bad = [('rotation_deg', '-1'), ('rotation_deg', '180.5'), ('rotation_deg', 'nan'), ('scale', '-0.1'), ('scale', 'inf'),
           ('intensity', '1'), ('intensity', '-0.2'), ('noise', '-1'), ('noise', 'nan'), ('noise', 'lots'), ('seed', '-1'),
           ('seed', '1.5'), ('seed', str(2 ** 64))]
    for key, value in bad:
        with pytest.raises(ValueError, match="augment_" + key):
            load_options(_config(**{'augment_' + key: value, 'augment_noise': '0.1'} if key != 'noise' else
                                 {'augment_noise': value}))
