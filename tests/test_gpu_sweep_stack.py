"""Strip-sweep convolutions with the stacked filter-row issue order (conv_sweep.cu): every input row feeds three output rows
through one MMA pass into a ring of S accumulator slots (S = 14 / 8 / 6 for 32 / 48 / 64 output columns) plus two spill
slots; output class row n lands in slot (n + 2) mod S, and an item that does not follow on from the previous item's slots
jumps the slot counter ahead.  Small boxes of 24 consecutive extents (12 .. 33) give maps of many row counts, cut into
items of one, two and more rows; a wider volume leaves the small-map item cut, so every CTA runs several items and hands
its slots over between them; a scattered sparse mask leaves consecutive computed items of a CTA non-adjacent.  Tolerances
are those of the other oracle tests."""
import numpy as np
import pytest
import torch

from oracle import gather as og, network as on
from gpu_util import cuda_ctx, dev

pytestmark = pytest.mark.gpu
TOL = 1e-3


@pytest.fixture(scope="module")
def P(weights_path):
    return on.load_params(weights_path)


@pytest.fixture(scope="module")
def ctx(P):
    from cnn_cort import nets
    c = cuda_ctx()
    c.load_weights(nets.pack_params(P))
    if c.counter("gemm") != 1:
        c.close()
        pytest.skip("tcgen05 back-end not selected")
    yield c
    c.close()


def _atlas(rng, shape):
    return rng.dirichlet(np.ones(15) * 0.3, size=shape).astype(np.float32)


def _vs_oracle(P, vol, atlas, pick, got, what):
    x = [og.get_patches(vol, pick, (32, 32), m)[:, None] for m in og.VIEWS]
    ref = on.forward(P, *x, og.atlas_vectors_test(atlas, pick), dtype=torch.float64)
    err = np.abs(got - ref).max()
    agree = (np.argmax(got, 1) == np.argmax(ref, 1)).mean()
    assert err < TOL, "%s: max|dp| = %g" % (what, err)
    assert agree >= 0.999, "%s: argmax agreement %g" % (what, agree)


@pytest.mark.parametrize("dims", [(12, 19, 26), (13, 20, 27), (14, 21, 28), (15, 22, 29), (16, 23, 30), (17, 24, 31), (18, 25, 32),
                                  (33, 12, 21)])
def test_dense_row_counts_vs_oracle(ctx, P, dims):
    rng = np.random.RandomState(1000 + sum(dims) * 7 + dims[0])
    shape = tuple(d + 3 for d in dims)
    box = (1, 1 + dims[0], 2, 2 + dims[1], 0, dims[2])
    vol = rng.randn(*shape).astype(np.float32)
    atlas = _atlas(rng, shape)
    prob = torch.full(shape + (15,), -1.0, dtype=torch.float32, device="cuda")
    lab = torch.full(shape, 99, dtype=torch.uint8, device="cuda")
    ctx.segment_volume(dev(vol), dev(atlas), box=box, label_vol=lab, proba_vol=prob)
    inside = np.zeros(shape, bool)
    inside[box[0]:box[1], box[2]:box[3], box[4]:box[5]] = True
    L, Pv = lab.cpu().numpy(), prob.cpu().numpy()
    assert (L[~inside] == 99).all() and (Pv[~inside] == -1.0).all()
    cen = og.get_mask_voxels(inside)
    pick = cen[rng.choice(len(cen), size=240, replace=False)]
    got = Pv[pick[:, 0], pick[:, 1], pick[:, 2]]
    _vs_oracle(P, vol, atlas, pick, got, "dense box %s" % (dims,))
    assert np.array_equal(L[pick[:, 0], pick[:, 1], pick[:, 2]], np.argmax(got, 1))


def test_several_items_per_cta_vs_oracle(ctx, P):
    """A volume wide enough for the regular item cut (12 - 96 class rows per item, more items than CTAs in every sweep, CTA
    pairs included): every CTA hands its accumulator slots over from one item to the next."""
    rng = np.random.RandomState(46)
    shape = (50, 76, 76)
    vol = rng.randn(*shape).astype(np.float32)
    atlas = _atlas(rng, shape)
    prob = torch.full(shape + (15,), -1.0, dtype=torch.float32, device="cuda")
    lab = torch.full(shape, 99, dtype=torch.uint8, device="cuda")
    ctx.segment_volume(dev(vol), dev(atlas), label_vol=lab, proba_vol=prob)
    L, Pv = lab.cpu().numpy(), prob.cpu().numpy()
    cen = og.get_mask_voxels(np.ones(shape, bool))
    pick = cen[rng.choice(len(cen), size=300, replace=False)]
    got = Pv[pick[:, 0], pick[:, 1], pick[:, 2]]
    _vs_oracle(P, vol, atlas, pick, got, "wide volume")
    assert np.array_equal(L[pick[:, 0], pick[:, 1], pick[:, 2]], np.argmax(got, 1))


def test_scattered_mask_vs_oracle(ctx, P):
    """Isolated candidates far apart: the sweeps compute a few short items per CTA with skipped items between them, so the
    slot counter jumps: the halo slots of one item are flushed and the next item claims fresh leading slots."""
    rng = np.random.RandomState(44)
    shape = (70, 64, 58)
    vol = rng.randn(*shape).astype(np.float32)
    atlas = _atlas(rng, shape)
    cand = np.zeros(shape, bool)
    pts = np.stack([rng.randint(0, s, 90) for s in shape], 1)
    pts = np.concatenate([pts, [[0, 0, 0], [69, 63, 57], [0, 63, 57], [35, 0, 29]]])
    cand[pts[:, 0], pts[:, 1], pts[:, 2]] = True
    prob = torch.full(shape + (15,), -1.0, dtype=torch.float32, device="cuda")
    lab = torch.full(shape, 99, dtype=torch.uint8, device="cuda")
    ctx.segment_volume(dev(vol), dev(atlas), cand_mask=dev(cand.view(np.uint8)), label_vol=lab, proba_vol=prob)
    L, Pv = lab.cpu().numpy(), prob.cpu().numpy()
    assert (L[~cand] == 99).all() and (Pv[~cand] == -1.0).all()
    pick = og.get_mask_voxels(cand)
    got = Pv[pick[:, 0], pick[:, 1], pick[:, 2]]
    _vs_oracle(P, vol, atlas, pick, got, "scattered mask")
    assert np.array_equal(L[pick[:, 0], pick[:, 1], pick[:, 2]], np.argmax(got, 1))


def test_patchwise_odd_batch_vs_oracle(ctx, P):
    """Patchwise maps (conv2 with the fused stride-2 pool, conv3, and the CTA-pair conv4 / conv5) over an odd number of
    patches: several items per sweep, the last strip pair half outside the map."""
    rng = np.random.RandomState(45)
    vol = rng.randn(40, 36, 44).astype(np.float32)
    atlas = _atlas(rng, vol.shape)
    cen = og.get_mask_voxels(np.ones(vol.shape, bool))
    pick = cen[rng.choice(len(cen), size=333, replace=False)]
    ax, co, sa, at = ctx.gather_patches(dev(vol), dev(pick.astype(np.int32)), atlas=dev(atlas), bg_fix=True)
    proba, label = ctx.forward(ax, co, sa, at)
    got = proba.cpu().numpy()
    ref = on.forward(P, ax.cpu().numpy(), co.cpu().numpy(), sa.cpu().numpy(), at.cpu().numpy(), dtype=torch.float64)
    assert np.abs(got - ref).max() < TOL
    assert (np.argmax(got, 1) == np.argmax(ref, 1)).mean() >= 0.999
    assert np.array_equal(label.cpu().numpy(), np.argmax(got, 1))
