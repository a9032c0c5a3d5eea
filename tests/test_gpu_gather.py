"""K1 parity (bit-exact): CUDA gather / candidate indexing / scatter through the C-ABI vs the
reference-generated golden vectors and the oracle."""

import numpy as np
import pytest

from oracle import gather as og
from gpu_util import cuda_ctx, dev

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = cuda_ctx()
    yield c
    c.close()


@pytest.fixture(scope="module")
def G(gather_golden):
    return gather_golden


def _gather(ctx, vol, cen, atlas=None, bg_fix=True):
    out = ctx.gather_patches(dev(vol.astype(np.float32)), dev(np.asarray(cen, np.int32).reshape(-1, 3)),
                             atlas=None if atlas is None else dev(atlas), bg_fix=bg_fix)
    return [o.cpu().numpy() if o is not None else None for o in out]


def test_patches_vs_reference_golden(ctx, G):
    ax, co, sa, _ = _gather(ctx, G["A_vol"], G["A_centers"])
    for got, mode in zip((ax, co, sa), og.VIEWS):
        assert got.shape == (len(G["A_centers"]), 1, 32, 32)
        assert np.array_equal(got[:, 0], G["A_" + mode].astype(np.float32)), mode
    ax, co, sa, _ = _gather(ctx, G["B_vol"], G["B_sel"])
    for got, mode in zip((ax, co, sa), og.VIEWS):
        assert np.array_equal(got[:, 0], G["B_x_" + mode]), mode
    ax, co, sa, _ = _gather(ctx, G["B_lab"], G["B_sel"])  # label volumes: exact in float32
    for got, mode in zip((ax, co, sa), og.VIEWS):
        assert np.array_equal(got[:, 0].astype(np.uint8), G["B_y_" + mode]), mode


@pytest.mark.parametrize("shape,n", [((33, 47, 29), 257), ((64, 64, 64), 1000), ((5, 6, 7), 31), ((40, 8, 90), 1)])
def test_patches_vs_oracle_random(ctx, shape, n):
    rng = np.random.RandomState(sum(shape) + n)
    vol = rng.randn(*shape).astype(np.float32)
    atlas = rng.rand(*shape, 15).astype(np.float32)
    cen = np.stack([rng.randint(0, s, n) for s in shape], 1)
    cen[0] = 0
    cen[-1] = np.array(shape) - 1
    ax, co, sa, at = _gather(ctx, vol, cen, atlas)
    for got, mode in zip((ax, co, sa), og.VIEWS):
        assert np.array_equal(got[:, 0], og.get_patches(vol, cen, (32, 32), mode)), mode
    assert np.array_equal(at, og.atlas_vectors_test(atlas, cen))


def test_consecutive_candidates_full_volume_order(ctx):
    rng = np.random.RandomState(4)
    vol = rng.randn(20, 21, 40).astype(np.float32)
    cen = og.get_mask_voxels(np.ones(vol.shape, bool))[5000:5000 + 999]  # runs of consecutive z
    ax, co, sa, _ = _gather(ctx, vol, cen)
    for got, mode in zip((ax, co, sa), og.VIEWS):
        assert np.array_equal(got[:, 0], og.get_patches(vol, cen, (32, 32), mode)), mode


def test_empty_and_partial_outputs(ctx):
    vol = np.ones((8, 8, 8), np.float32)
    ax, co, sa, at = _gather(ctx, vol, np.zeros((0, 3), np.int32), np.zeros((8, 8, 8, 15), np.float32))
    assert ax.shape == (0, 1, 32, 32) and at.shape == (0, 15)
    out = ctx.gather_patches(dev(vol), dev(np.array([[1, 2, 3]], np.int32)), views=(False, True, False))
    assert out[0] is None and out[2] is None and out[1].shape == (1, 1, 32, 32)


def test_atlas_background_fix_is_numpy_exact(ctx):
    rng = np.random.RandomState(8)
    atlas = rng.rand(6, 6, 6, 15).astype(np.float32)
    atlas[0, 0, 0] = 0                       # all-zero row -> [14] = 1
    atlas[1, 1, 1] = 0
    atlas[1, 1, 1, 3], atlas[1, 1, 1, 9] = 0.25, -0.25   # cancels exactly -> fix applies (np.sum == 0)
    row = (rng.rand(15).astype(np.float32) - 0.5)
    atlas[2, 2, 2] = row                     # mixed signs: whatever np.sum says
    atlas[3, 3, 3] = 0
    atlas[3, 3, 3, 0], atlas[3, 3, 3, 8] = 1e-8, -1e-8
    cen = og.get_mask_voxels(np.ones((6, 6, 6), bool))
    vol = np.zeros((6, 6, 6), np.float32)
    at = _gather(ctx, vol, cen, atlas)[3]
    assert np.array_equal(at, og.atlas_vectors_test(atlas, cen))
    at_train = _gather(ctx, vol, cen, atlas, bg_fix=False)[3]
    assert np.array_equal(at_train, og.atlas_vectors_train(atlas, cen))


@pytest.mark.parametrize("shape", [(9, 7, 11), (31, 33, 17), (64, 64, 65), (1, 1, 1)])
def test_nonzero_coords_order(ctx, shape, G):
    rng = np.random.RandomState(sum(shape))
    for dens in (0.0, 0.3, 1.0):
        m = (rng.rand(*shape) < dens)
        got = ctx.nonzero_coords(dev(m.view(np.uint8))).cpu().numpy()
        assert got.dtype == np.int32 and np.array_equal(got, og.get_mask_voxels(m))
    img = rng.randn(*shape).astype(np.float32)
    img[rng.rand(*shape) < 0.5] = 0
    img.flat[0] = -0.0
    assert np.array_equal(ctx.nonzero_coords(dev(img)).cpu().numpy(), og.get_mask_voxels(img.astype(bool)))
    assert np.array_equal(ctx.nonzero_coords(dev(G["C_mask"].view(np.uint8))).cpu().numpy(), G["C_vox"])


def test_nonzero_full_size_is_sorted_and_complete(ctx):
    import torch
    g = torch.Generator(device="cuda").manual_seed(1)
    vol = (torch.rand((256, 256, 256), device="cuda", generator=g) < 0.37).to(torch.uint8)
    xyz = ctx.nonzero_coords(vol).long()
    assert xyz.shape[0] == int(vol.sum())
    lin = (xyz[:, 0] * 256 + xyz[:, 1]) * 256 + xyz[:, 2]
    assert bool((lin[1:] > lin[:-1]).all())                 # strictly increasing == C-order, no duplicates
    assert bool(vol.view(-1)[lin].all())


def test_scatter_and_center_labels(ctx):
    import torch
    rng = np.random.RandomState(2)
    shape = (12, 10, 9)
    cen = og.get_mask_voxels(rng.rand(*shape) < 0.4)
    lab = rng.randint(0, 15, len(cen)).astype(np.int32)
    pr = rng.rand(len(cen), 15).astype(np.float32)
    lv = torch.zeros(shape, dtype=torch.uint8, device="cuda")
    pv = torch.zeros(shape + (15,), dtype=torch.float32, device="cuda")
    ctx.scatter(dev(cen.astype(np.int32)), shape, label=dev(lab), proba=dev(pr), label_vol=lv, proba_vol=pv)
    ref_l = np.zeros(shape, np.uint8)
    ref_p = np.zeros(shape + (15,), np.float32)
    ref_l[cen[:, 0], cen[:, 1], cen[:, 2]] = lab
    ref_p[cen[:, 0], cen[:, 1], cen[:, 2]] = pr
    assert np.array_equal(lv.cpu().numpy(), ref_l) and np.array_equal(pv.cpu().numpy(), ref_p)
    labels = rng.randint(0, 16, shape).astype(np.uint8)
    y = ctx.gather_center_labels(dev(labels), dev(cen.astype(np.int32))).cpu().numpy()
    assert np.array_equal(y, labels[cen[:, 0], cen[:, 1], cen[:, 2]])


def test_base_helpers_match_reference_semantics(ctx, G):
    from cnn_cort import base
    vox = base.get_mask_voxels(G["C_mask"])
    assert isinstance(vox, list) and isinstance(vox[0], tuple) and np.array_equal(np.array(vox), G["C_vox"])
    p = base.get_patches(G["A_vol"], [tuple(c) for c in G["A_centers"]], (32, 32), mode='coronal')
    assert np.array_equal(p, G["A_coronal"].astype(np.float32))
    sub = base.get_mask_voxels(G["C_mask"], size=7)
    assert len(sub) == 7 and set(sub) <= set(vox)


@pytest.mark.parametrize("shape,it", [((40, 40, 40), 10), ((17, 23, 9), 3), ((8, 8, 8), 1), ((30, 12, 50), 0)])
def test_dilate_mask_equals_scipy(ctx, shape, it):
    from scipy import ndimage
    rng = np.random.RandomState(sum(shape) + it)
    m = rng.rand(*shape) < 0.01
    m[0, 0, 0] = True                       # border behaviour (border_value = 0)
    m[-1, -1, -1] = True
    got = ctx.dilate_mask(dev(m.view(np.uint8)), it).cpu().numpy().astype(bool)
    ref = ndimage.binary_dilation(m, iterations=it) if it else m
    assert np.array_equal(got, ref)


def test_error_codes_not_exceptions(ctx):
    """bad arguments come back as negative status codes with a message (no exception crosses the C boundary)"""
    import ctypes
    from cnn_cort import _native
    lib = ctx.lib
    dims = (ctypes.c_int32 * 3)(4, 4, 4)
    assert lib.sc_gather_patches(ctx.h, None, dims, None, 0, None, 5, None, None, None, None, None) == -2
    assert b"sc_gather_patches" in lib.sc_last_error()
    assert lib.sc_set_option(ctx.h, b"no_such_key", 1) == -2
    assert lib.sc_forward(ctx.h, None, None, None, None, 4, None, None, None) in (-2, -3)   # no weights / null input
    bad = (ctypes.c_int32 * 3)(0, 4, 4)
    assert lib.sc_nonzero_coords(ctx.h, ctypes.c_void_p(1), 1, bad, None, 0, None, None) == -2
    with pytest.raises(_native.NativeError):
        ctx.load_weights(np.zeros(10, np.float32))
