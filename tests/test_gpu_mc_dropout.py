"""Monte-Carlo dropout over the dense path (sc_segment_volume_mc) against the fp64 oracle (tests/mc_dropout_oracle.py:mc_predict),
and its write set, determinism, compaction, argument checks and the test_scan outputs."""
import os

import numpy as np
import pytest
import torch

from oracle import gather as og, network as on
from gpu_util import cuda_ctx, dev
import mc_dropout_oracle as mco

pytestmark = pytest.mark.gpu
LN15 = float(np.log(15.0))


@pytest.fixture(scope="module")
def P(weights_path):
    return on.load_params(weights_path)


@pytest.fixture(scope="module")
def ctx(P):
    from cnn_cort import nets
    c = cuda_ctx()
    c.load_weights(nets.pack_params(P))
    yield c
    c.close()


def _soft_atlas(rng, n):
    return rng.dirichlet(np.ones(15) * 0.3, size=n).astype(np.float32)


def _outputs(shape):
    return (torch.full(shape, 99, dtype=torch.uint8, device="cuda"), torch.full(shape + (15,), -1.0, device="cuda"),
            torch.full(shape, -2.0, device="cuda"), torch.full(shape, -3.0, device="cuda"))


def _run_mc(ctx, vol, atlas, T, seed, shape, box=None, cand=None):
    lab, prob, ent, mi = _outputs(shape)
    ctx.segment_volume_mc(vol, atlas, T, seed, box=box, cand_mask=cand, label_vol=lab, proba_vol=prob, entropy_vol=ent, mi_vol=mi)
    return lab, prob, ent, mi


def _untouched(outs, sel):
    lab, prob, ent, mi = outs
    return (bool((lab[~sel] == 99).all()) and bool((prob[~sel] == -1.0).all()) and bool((ent[~sel] == -2.0).all())
            and bool((mi[~sel] == -3.0).all()))


@pytest.mark.parametrize("T,seed", [(1, 0), (8, 0), (1, 5), (8, 5)])
@pytest.mark.parametrize("shape,box", [((20, 24, 18), None), ((37, 29, 41), (5, 30, 0, 29, 7, 33))])
def test_mc_vs_oracle(ctx, P, shape, box, T, seed):
    rng = np.random.RandomState(sum(shape) + T + seed)
    vol = rng.randn(*shape).astype(np.float32)
    atlas = _soft_atlas(rng, vol.size).reshape(shape + (15,))
    atlas[1, 1, 1] = 0                                          # background fix of an all-zero prior row
    cand = rng.rand(*shape) < 0.8
    inside = np.zeros(shape, bool)
    b = box or (0, shape[0], 0, shape[1], 0, shape[2])
    inside[b[0]:b[1], b[2]:b[3], b[4]:b[5]] = True
    sel = inside & cand
    outs = _run_mc(ctx, dev(vol), dev(atlas), T, seed, shape, box=box, cand=dev(cand.view(np.uint8)))
    assert _untouched(outs, torch.from_numpy(sel).cuda())
    L, Pv, H, MI = (o.cpu().numpy() for o in outs)
    assert np.array_equal(L[sel], np.argmax(Pv[sel], 1))      # labels: first arg-max of the device mean, everywhere
    if T == 1:
        assert (MI[sel] == 0).all()
    cen = og.get_mask_voxels(sel)
    pick = cen[rng.choice(len(cen), size=min(300, len(cen)), replace=False)]
    x = [og.get_patches(vol, pick, (32, 32), m)[:, None] for m in og.VIEWS]
    pbar, h, mi = mco.mc_predict(P, *x, og.atlas_vectors_test(atlas, pick), seed=seed, T=T)
    i = (pick[:, 0], pick[:, 1], pick[:, 2])
    what = "%s T=%d seed=%d" % (shape, T, seed)
    assert np.abs(Pv[i] - pbar).max() < 1e-3, what
    assert np.abs(H[i] - h).max() < 2e-3, what
    assert np.abs(MI[i] - mi).max() < 4e-3, what
    assert (L[i] == np.argmax(pbar, 1)).mean() >= 0.999, what


def test_mc_deterministic_and_seeded(ctx):
    g = torch.Generator(device="cuda").manual_seed(3)
    shape = (30, 26, 34)
    vol = torch.randn(shape, device="cuda", generator=g)
    atlas = torch.rand(shape + (15,), device="cuda", generator=g) ** 6
    atlas = atlas / atlas.sum(-1, keepdim=True)
    a = _run_mc(ctx, vol, atlas, 5, 17, shape)
    b = _run_mc(ctx, vol, atlas, 5, 17, shape)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    c = _run_mc(ctx, vol, atlas, 5, 18, shape)
    assert not torch.equal(a[2], c[2])
    H, MI = a[2], a[3]
    assert float(H.min()) >= -1e-6 and float(H.max()) <= LN15 + 1e-5 and bool((MI >= 0).all()) and bool((MI <= H).all())
    assert float(MI.max()) > 0


def test_mc_candidate_compaction(ctx):
    """Several slabs (one without candidates), the compacted and the dense FC rows: same statistics, same write set."""
    g = torch.Generator(device="cuda").manual_seed(21)
    shape = (40, 48, 36)
    vol = torch.randn(shape, device="cuda", generator=g)
    atlas = torch.rand(shape + (15,), device="cuda", generator=g) ** 6
    atlas = atlas / atlas.sum(-1, keepdim=True)
    cand = torch.rand(shape, device="cuda", generator=g) < 0.35
    cand[20:26] = False
    cand = cand.to(torch.uint8).contiguous()
    ctx.set_option("chunk_voxels", 6000)
    out = []
    try:
        for on_ in (1, 0):
            ctx.set_option("tc_compact", on_)
            out.append(_run_mc(ctx, vol, atlas, 4, 9, shape, cand=cand))
    finally:
        ctx.set_option("tc_compact", 1)
        ctx.set_option("chunk_voxels", 1 << 20)
    sel = cand.bool()
    assert _untouched(out[0], sel) and _untouched(out[1], sel)
    for k in (1, 2, 3):
        assert float((out[0][k][sel] - out[1][k][sel]).abs().max()) < 1e-5
    assert float((out[0][0][sel] == out[1][0][sel]).float().mean()) >= 0.9999


def test_mc_leaves_segment_volume_alone(ctx):
    g = torch.Generator(device="cuda").manual_seed(7)
    shape = (28, 32, 30)
    vol = torch.randn(shape, device="cuda", generator=g)
    atlas = torch.rand(shape + (15,), device="cuda", generator=g) ** 6
    atlas = atlas / atlas.sum(-1, keepdim=True)
    cand = (torch.rand(shape, device="cuda", generator=g) < 0.5).to(torch.uint8)

    def deterministic():
        lab = torch.zeros(shape, dtype=torch.uint8, device="cuda")
        prob = torch.zeros(shape + (15,), device="cuda")
        n0 = ctx.counter("launches")
        ctx.segment_volume(vol, atlas, cand_mask=cand, label_vol=lab, proba_vol=prob)
        return lab, prob, ctx.counter("launches") - n0

    before = deterministic()
    n0 = ctx.counter("launches")
    _run_mc(ctx, vol, atlas, 3, 1, shape, cand=cand)
    assert ctx.counter("launches") - n0 > before[2]
    after = deterministic()
    assert torch.equal(before[0], after[0]) and torch.equal(before[1], after[1]) and before[2] == after[2]


def test_mc_argument_errors(ctx):
    from cnn_cort._native import NativeError
    shape = (16, 18, 20)
    vol = torch.randn(shape, device="cuda")
    atlas = torch.full(shape + (15,), 1.0 / 15, device="cuda")
    outs = _outputs(shape)
    lab, prob, ent, mi = outs
    kw = dict(label_vol=lab, proba_vol=prob, entropy_vol=ent, mi_vol=mi)
    with pytest.raises(NativeError, match="samples"):
        ctx.segment_volume_mc(vol, atlas, 0, 0, **kw)
    with pytest.raises(NativeError, match="samples"):
        ctx.segment_volume_mc(vol, atlas, 1025, 0, **kw)
    with pytest.raises(NativeError, match="NULL"):
        ctx.segment_volume_mc(vol, atlas, 4, 0)
    with pytest.raises(NativeError, match="box"):
        ctx.segment_volume_mc(vol, atlas, 4, 0, box=(0, 17, 0, 18, 0, 20), **kw)
    default = ctx.counter("gemm")
    ctx.set_option("gemm", 0)
    try:
        with pytest.raises(NativeError, match="gemm"):
            ctx.segment_volume_mc(vol, atlas, 4, 0, **kw)
    finally:
        ctx.set_option("gemm", default)
    assert _untouched(outs, torch.ones(shape, dtype=torch.bool, device="cuda"))


def test_test_scan_mc_outputs(ctx, tmp_path, weights_path):
    from cnn_cort import base, nets, nifti, synthetic
    root = str(tmp_path)
    d = synthetic.write_subject(root, "s01", shape=(48, 44, 40), seed=3)
    options = {'experiment': 'miccai2012_v1', 'patch_size': [32, 32], 'mode': 'cuda0', 'device': 0, 'load_weights': 'True',
               'net_verbose': 0, 'train_split': 0.25, 'max_epochs': 1, 'patience': 1, 'batch_size': 128,
               'test_batch_size': 5000, 'debug': 'False', 'out_probabilities': 'True', 'post_process': 'False',
               'crop': 'True', 'crop_bool': True, 'test_folder': root, 't1_name': 'T1.nii.gz', 'mc_samples': 4, 'mc_seed': 1}
    net = nets.build_model(os.path.dirname(os.path.dirname(weights_path)), options)
    t1_names, _ = base.load_test_names(options)
    base.test_scan(net, t1_names[0], options)
    t1 = nifti.load(t1_names[0])
    vols = {}
    for key, f in (('H', 'out_subcortical_entropy.nii.gz'), ('MI', 'out_subcortical_mi.nii.gz')):
        img = nifti.load(os.path.join(d, f))
        assert img.get_data().dtype == np.float32 and img.shape == (48, 44, 40)
        assert np.allclose(img.affine, t1.affine)
        vols[key] = img.get_data()
    H, MI = vols['H'], vols['MI']
    assert H.min() >= -1e-6 and H.max() <= LN15 + 1e-5 and (MI >= 0).all() and (MI <= H).all() and H.max() > 0
    seg = nifti.load(os.path.join(d, 'out_subcortical_rawseg.nii.gz')).get_data()
    prob = nifti.load(os.path.join(d, 'out_subcortical_prob.nii.gz')).get_data()
    nz = prob.sum(-1) > 0
    assert np.array_equal(seg[nz], np.argmax(prob[nz], -1)) and np.allclose(prob[nz].sum(-1), 1, atol=1e-4)
    unc = base.structure_uncertainty(seg, H, MI)
    for l in range(1, 15):
        m = seg == l
        assert unc[l]['voxels'] == int(m.sum())
        if m.any():
            assert abs(unc[l]['entropy'] - H[m].astype(np.float64).mean()) < 1e-6
            assert abs(unc[l]['mutual_info'] - MI[m].astype(np.float64).mean()) < 1e-6
    options['inference'] = 'patchwise'
    with pytest.raises(ValueError, match="mc_samples"):
        base.test_scan(net, t1_names[0], options)
