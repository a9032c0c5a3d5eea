"""The FC head's tail on the tensor cores: fc_2 computes the out_layer, softmax and argmax in its epilogue (one CTA pair
owns every n-tile of a 256-row block), so there is no h2 buffer and no separate out_softmax launch."""
import numpy as np
import pytest
import torch

from oracle import gather as og, network as on
from gpu_util import cuda_ctx, dev

pytestmark = pytest.mark.gpu
SHAPE = (10, 16, 32)            # x-planes of 512 voxels
CHUNK = 1024                    # the smallest slab the library takes: two x-planes -> 5 slabs
SLAB_COUNTS = [1, 255, 256, 257, 0]


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


def _inputs(seed):
    rng = np.random.RandomState(seed)
    vol = rng.randn(*SHAPE).astype(np.float32)
    atlas = rng.dirichlet(np.ones(15) * 0.3, size=SHAPE).astype(np.float32)
    atlas[1, 1, 1] = 0
    cand = np.zeros(SHAPE, np.uint8)
    per_slab = CHUNK // (SHAPE[1] * SHAPE[2])
    for s, n in enumerate(SLAB_COUNTS):     # compacted rows per slab: one, a partial block, a full one, one row past it, none
        flat = cand[s * per_slab:(s + 1) * per_slab].reshape(-1)
        flat[rng.choice(flat.size, size=n, replace=False)] = 1
    return vol, atlas, cand


def test_partial_blocks_under_compaction(ctx, P):
    vol, atlas, cand = _inputs(7)
    ctx.set_option("chunk_voxels", CHUNK)
    try:
        lab = torch.full(SHAPE, 99, dtype=torch.uint8, device="cuda")
        prob = torch.full(SHAPE + (15,), -1.0, dtype=torch.float32, device="cuda")
        ctx.segment_volume(dev(vol), dev(atlas), cand_mask=dev(cand), label_vol=lab, proba_vol=prob)
    finally:
        ctx.set_option("chunk_voxels", 1 << 20)
    L, Pv = lab.cpu().numpy(), prob.cpu().numpy()
    sel = cand.astype(bool)
    assert (L[~sel] == 99).all() and (Pv[~sel] == -1.0).all()
    cen = og.get_mask_voxels(sel)
    assert len(cen) == sum(SLAB_COUNTS)
    x = [og.get_patches(vol, cen, (32, 32), m)[:, None] for m in og.VIEWS]
    ref = on.forward(P, *x, og.atlas_vectors_test(atlas, cen), dtype=torch.float64)
    got = Pv[cen[:, 0], cen[:, 1], cen[:, 2]]
    err = np.abs(got - ref).max()
    assert err < 1e-3, "max|dp| = %g" % err
    assert np.array_equal(L[cen[:, 0], cen[:, 1], cen[:, 2]], np.argmax(got, 1))


def test_one_fc2_launch_per_slab_and_no_out_softmax(ctx):
    vol, atlas, cand = _inputs(8)
    lab = torch.zeros(SHAPE, dtype=torch.uint8, device="cuda")
    ctx.set_option("chunk_voxels", CHUNK)
    ctx.set_option("profile", 1)
    try:
        ctx.profile_read()
        ctx.segment_volume(dev(vol), dev(atlas), label_vol=lab)        # every voxel a candidate: 5 slabs, no compaction
        torch.cuda.synchronize()
        prof = ctx.profile_read()
    finally:
        ctx.set_option("profile", 0)
        ctx.set_option("chunk_voxels", 1 << 20)
    assert "out_softmax" not in prof, prof
    assert prof["gemm_fc2"][1] == len(SLAB_COUNTS), prof
