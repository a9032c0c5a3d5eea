"""Oracle gather vs. the golden vectors produced by executing the reference's own
get_patches / get_mask_voxels / generate_training_set text (tests/golden/make_golden.py)."""

import numpy as np
import pytest

from oracle import gather


@pytest.fixture(scope="module")
def G(gather_golden):
    return gather_golden


@pytest.mark.parametrize("mode", gather.VIEWS)
def test_patches_match_reference_float64(G, mode):
    got = gather.get_patches(G["A_vol"], G["A_centers"], (32, 32), mode)
    assert got.dtype == np.float64
    assert np.array_equal(got, G["A_" + mode])
    loop = np.array(gather.get_patches_loop(G["A_vol"], G["A_centers"], (32, 32), mode))
    assert np.array_equal(loop, G["A_" + mode])


@pytest.mark.parametrize("mode", gather.VIEWS)
def test_patches_match_reference_float32_and_labels(G, mode):
    assert np.array_equal(gather.get_patches(G["B_vol"], G["B_sel"], (32, 32), mode), G["B_x_" + mode])
    assert np.array_equal(gather.get_patches(G["B_lab"], G["B_sel"], (32, 32), mode), G["B_y_" + mode])


def test_patch_geometry():
    vol = np.arange(20 * 22 * 24, dtype=np.float64).reshape(20, 22, 24) + 1
    c = np.array([[17, 18, 19]])
    ax = gather.get_patches(vol, c, (32, 32), "axial")[0]
    co = gather.get_patches(vol, c, (32, 32), "coronal")[0]
    sa = gather.get_patches(vol, c, (32, 32), "saggital")[0]
    assert ax[16, 16] == co[16, 16] == sa[16, 16] == vol[17, 18, 19]
    assert ax[0, 0] == vol[1, 2, 19] and co[0, 0] == vol[1, 18, 3] and sa[0, 0] == vol[17, 2, 3]
    assert ax[31, 16] == 0 and ax[18, 16] == vol[19, 18, 19]  # x = 17+15 = 32 is outside
    z = gather.get_patches(vol, np.array([[0, 0, 0]]), (32, 32), "axial")[0]
    assert not z[:16].any() and not z[:, :16].any() and z[16, 16] == vol[0, 0, 0]


def test_mask_voxels_order(G):
    assert np.array_equal(gather.get_mask_voxels(G["C_mask"]), G["C_vox"])
    lab = G["B_lab"]
    assert np.array_equal(gather.get_mask_voxels(np.logical_and(lab > 0, lab < 15)), G["B_pos_centers"])
    import random
    sub = gather.get_mask_voxels(G["C_mask"], size=10, rng=random.Random(3))
    assert sub.shape == (10, 3) and len({tuple(r) for r in sub}) == 10


def test_generate_training_set(G):
    n0 = 10
    xa = [G["B_x_axial"][:n0], G["B_x_axial"][n0:]]
    xc = [G["B_x_coronal"][:n0], G["B_x_coronal"][n0:]]
    xs = [G["B_x_saggital"][:n0], G["B_x_saggital"][n0:]]
    ya = [G["B_y_axial"][:n0], G["B_y_axial"][n0:]]
    at = [G["T_atlas0"], G["T_atlas1"]]
    r = gather.generate_training_set(xa, xc, xs, at, ya, randomize=False)
    for k, v in zip(("xa", "xc", "xs", "at", "y"), r):
        assert v.dtype == G["T_plain_" + k].dtype and np.array_equal(v, G["T_plain_" + k]), k
    assert r[4].max() <= 14
    np.random.seed(77)
    r = gather.generate_training_set(xa, xc, xs, at, ya, randomize=True)
    for k, v in zip(("xa", "xc", "xs", "at", "y"), r):
        assert np.array_equal(v, G["T_shuf_" + k]), k


def test_atlas_vectors_bg_fix():
    rng = np.random.RandomState(0)
    atlas = rng.rand(6, 5, 4, 15).astype(np.float32)
    atlas[1, 2, 3] = 0
    c = np.array([[1, 2, 3], [0, 0, 0]])
    v = gather.atlas_vectors_test(atlas, c)
    assert v.dtype == np.float32 and v[0, 14] == 1 and v[0, :14].sum() == 0
    assert np.array_equal(v[1], atlas[0, 0, 0])
    assert gather.atlas_vectors_train(atlas, c)[0].sum() == 0  # quirk Q4: no fix at train time


def test_normalise_dtype_rules_of_the_reference_numpy():
    """numpy 1.12 (requirements.txt:18): float32 array (op) float64 scalar stays float32 -> the train path (base.py:146) is
    float32 arithmetic; an integer array (op) float64 scalar is float64 -> the test path (base.py:358) on an int16 T1."""
    rng = np.random.RandomState(4)
    vol = rng.randint(0, 1500, size=(9, 8, 7)).astype(np.int16)
    nz = vol[vol != 0]
    tr = gather.normalise(vol, np.float32)
    assert tr.dtype == np.float32
    assert np.array_equal(tr, (vol.astype(np.float32) - np.float32(nz.mean())) / np.float32(nz.std()))
    te = gather.normalise(vol)
    assert te.dtype == np.float64 and np.array_equal(te, (vol.astype(np.float64) - nz.mean()) / nz.std())
    # the float64-promoted result (what NumPy 2 would compute for the train path) differs in the last bit somewhere
    wide = ((vol.astype(np.float32) - nz.mean()) / nz.std()).astype(np.float32)
    assert np.abs(wide - tr).max() < 1e-6


def test_patch_batches_and_candidates():
    rng = np.random.RandomState(1)
    vol = rng.rand(12, 10, 9) + 0.5
    vol[3, 3, 3] = 0
    cen = gather.candidates(vol)
    assert len(cen) == vol.size - 1
    atlas = rng.rand(12, 10, 9, 15).astype(np.float32)
    norm = gather.normalise(vol)
    assert abs(norm[vol != 0].mean()) < 1e-12
    tot = 0
    for ax, co, sa, av, c in gather.patch_batches(norm, atlas, cen, 500):
        assert ax.shape == (len(c), 1, 32, 32) and ax.dtype == np.float32 and av.shape == (len(c), 15)
        tot += len(c)
    assert tot == len(cen)
    m = np.zeros((40, 40, 40), np.float32)
    m[20, 20, 20] = 1
    assert len(gather.candidates(vol, crop_mask=m)) == 1561  # 6-connected ball of radius 10
