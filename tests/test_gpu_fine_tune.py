"""Fine-tuning with a frozen trunk on the device: sc_trunk_features, sc_head_train_forward_backward, sc_head_eval_batch and
sc_freeze_trunk against the fp64 reference (tests/fine_tune_oracle.py) and the full training step, and Net.fine_tune end to
end."""
import ctypes
import os
import pickle

import numpy as np
import pytest
import torch

import fine_tune_oracle as fto
from oracle import network as on
from gpu_util import cuda_ctx, dev

pytestmark = pytest.mark.gpu

# head gradients: the tensor-core bounds of test_gpu_train.py (max-norm relative to the tensor's largest entry, relative L2)
TOL = dict(maxnorm=5e-2, l2=3e-2)
# Trunk features: five split-bf16 tensor-core convolutions.  Each product keeps ~2^-16 of relative precision (the lo*lo term is
# dropped, activations are stored as bf16 hi + lo, 2^-17), so after five layers a feature is expected within ~1e-4 of its
# scale; a pre-activation within that distance of a PReLU kink or a max-pool tie may take the other branch and move one
# feature further, which the max-norm bound (2e-3 of the largest feature) allows while the relative L2 bound (5e-4) keeps the
# table as a whole tight.  A wrong layout or tap order is an O(1) error.
FEAT_TOL = dict(maxnorm=2e-3, l2=5e-4)


def _batch(n, seed):
    rng = np.random.RandomState(seed)
    x = [rng.randn(n, 1, 32, 32).astype(np.float32) for _ in range(3)]
    at = rng.dirichlet(np.ones(15) * 0.3, size=n).astype(np.float32)
    y = rng.randint(0, 15, n).astype(np.uint8)
    masks = {"%s_l1drop" % b: (rng.rand(n, 60, 3, 3) < 0.5).astype(np.uint8) for b in on.BRANCHES}
    masks["f1_drop"] = (rng.rand(n, 540) < 0.5).astype(np.uint8)
    masks["f2_drop"] = (rng.rand(n, 540) < 0.5).astype(np.uint8)
    packed = np.concatenate([masks["%s_l1drop" % b].reshape(n, 540) for b in on.BRANCHES] +
                            [masks["f1_drop"], masks["f2_drop"]], axis=1)
    return x, at, y, masks, np.ascontiguousarray(packed)


def _params(source, weights_path):
    return on.load_params(weights_path) if source == "committed" else on.init_params(3)


def _ctx(P):
    from cnn_cort import nets
    ctx = cuda_ctx()
    ctx.load_weights(nets.pack_params(P))
    return ctx


def _trunk_mask():
    """bool [SC_PARAM_FLOATS]: the trunk entries of the flat parameter / gradient layout"""
    from cnn_cort import nets
    m = []
    for name, shapes in nets.layer_table():
        for s in shapes:
            m.append(np.full(int(np.prod(s)), fto.is_trunk(name)))
    return np.concatenate(m)


def _assert_grads(G, G_ref, tol=TOL):
    for (name, k), g_ref in G_ref.items():
        g = G[name][k].astype(np.float64)
        denom = max(np.abs(g_ref).max(), 1e-6)
        err = np.abs(g - g_ref).max() / denom
        l2 = np.linalg.norm(g - g_ref) / max(np.linalg.norm(g_ref), 1e-6)
        assert err < tol["maxnorm"], "%s[%d]: rel err %g (|g|max %g)" % (name, k, err, denom)
        assert l2 < tol["l2"], "%s[%d]: relative L2 err %g" % (name, k, l2)


@pytest.mark.parametrize("source", ["committed", "random"])
def test_trunk_features_match_oracle(weights_path, source):
    P = _params(source, weights_path)
    ctx = _ctx(P)
    x, _, _, _, _ = _batch(37, 1)
    got = ctx.trunk_features(*[dev(a) for a in x]).cpu().numpy().astype(np.float64)
    ref = fto.trunk_features(P, *x)
    err = np.abs(got - ref).max() / np.abs(ref).max()
    l2 = np.linalg.norm(got - ref) / np.linalg.norm(ref)
    assert err < FEAT_TOL["maxnorm"] and l2 < FEAT_TOL["l2"], (err, l2)
    ctx.close()


@pytest.mark.parametrize("source,n", [("committed", 24), ("random", 17)])
def test_head_step_matches_oracle(weights_path, source, n):
    from cnn_cort import nets
    P = _params(source, weights_path)
    ctx = _ctx(P)
    x, at, y, masks, packed = _batch(n, 5)
    feats = fto.trunk_features(P, *x).astype(np.float32)           # one feature table for both sides
    loss_ref, G_ref, _, _ = fto.head_train_step(P, feats.astype(np.float64), at, y, masks=masks)
    ctx.grad_tensor().fill_(1.0)                                   # every entry must be rewritten
    loss = ctx.head_train_forward_backward(dev(feats), dev(at), dev(y), drop_masks=dev(packed))
    assert abs(float(loss.item()) - loss_ref) < 1e-4 * max(1.0, abs(loss_ref)), (float(loss.item()), loss_ref)
    g = ctx.grad_tensor().cpu().numpy()
    assert (g[_trunk_mask()] == 0).all()
    _assert_grads(nets.unpack_params(g), G_ref)
    ctx.close()


def test_idx_and_kernel_by_kernel_agree(weights_path):
    P = on.load_params(weights_path)
    ctx = _ctx(P)
    N, n = 300, 130
    rng = np.random.RandomState(3)
    x, at, y, _, packed = _batch(N, 8)
    feats = ctx.trunk_features(*[dev(a) for a in x])
    d_at, d_y = dev(at), dev(y)
    perm = rng.permutation(N)[:n]
    masks = dev(packed[:n])
    loss_a = float(ctx.head_train_forward_backward(feats, d_at, d_y, idx=dev(perm.astype(np.int64)), drop_masks=masks).item())
    ga = ctx.grad_tensor().clone()
    sel = torch.from_numpy(perm).cuda()
    loss_b = float(ctx.head_train_forward_backward(feats[sel].contiguous(), d_at[sel].contiguous(), d_y[sel].contiguous(),
                                                   drop_masks=masks).item())
    gb = ctx.grad_tensor().clone()
    ctx.set_option("train_graph", 0)
    loss_c = float(ctx.head_train_forward_backward(feats, d_at, d_y, idx=dev(perm.astype(np.int64)), drop_masks=masks).item())
    gc = ctx.grad_tensor().clone()
    scale = float(ga.abs().max())
    for loss, g in ((loss_b, gb), (loss_c, gc)):     # the bias / slope sums are float atomics: equal up to their order
        assert abs(loss - loss_a) < 1e-6 * max(1.0, abs(loss_a))
        assert float((g - ga).abs().max()) < 1e-5 * scale
    # generated masks: same seed -> same step, another seed -> another step
    ctx.set_option("train_graph", 1)
    l1 = float(ctx.head_train_forward_backward(feats, d_at, d_y, idx=dev(perm.astype(np.int64)), seed=4).item())
    l2 = float(ctx.head_train_forward_backward(feats, d_at, d_y, idx=dev(perm.astype(np.int64)), seed=4).item())
    l3 = float(ctx.head_train_forward_backward(feats, d_at, d_y, idx=dev(perm.astype(np.int64)), seed=5).item())
    assert abs(l1 - l2) < 1e-6 * max(1.0, abs(l1)) and l1 != l3 and np.isfinite(l3)
    ctx.close()


def test_freeze_keeps_the_trunk_and_moves_the_head(weights_path):
    from cnn_cort import nets, _native
    P = on.load_params(weights_path)
    ctx = _ctx(P)
    tmask = _trunk_mask()
    p0 = ctx.get_params()
    x, at, y, masks, packed = _batch(24, 11)
    feats = fto.trunk_features(P, *x).astype(np.float32)
    ctx.freeze_trunk(True)
    # first step against the oracle's Adam (test_gpu_train.py criteria)
    _, G_ref, P_ref, _ = fto.head_train_step(P, feats.astype(np.float64), at, y, masks=masks, lr=1e-3)
    ctx.head_train_forward_backward(dev(feats), dev(at), dev(y), drop_masks=dev(packed))
    ctx.adam_step(lr=1e-3)
    P1 = nets.unpack_params(ctx.get_params())
    for name, arrs in P_ref.items():
        if fto.is_trunk(name):
            continue
        for k, a in enumerate(arrs):
            diff = np.abs(P1[name][k] - a)
            g_ref = np.abs(G_ref[(name, k)])
            ok = g_ref > 0.05 * g_ref.max()
            assert ok.any() and diff[ok].max() < 5e-5, "%s[%d]: %g" % (name, k, diff[ok].max())
            assert diff.max() < 2.1e-3
    # more steps with generated masks: the trunk, BatchNorm running statistics included, stays bit-identical
    for s in range(3):
        ctx.head_train_forward_backward(dev(feats), dev(at), dev(y), seed=s)
        ctx.adam_step(lr=1e-3)
    p1 = ctx.get_params()
    assert np.array_equal(p1[tmask], p0[tmask])
    assert not np.array_equal(p1[~tmask], p0[~tmask])
    d = [dev(a) for a in x] + [dev(at), dev(y)]
    with pytest.raises(_native.NativeError, match="frozen"):
        ctx.train_forward_backward(*d)
    # unfrozen: the full step and Adam (trunk entries and BatchNorm statistics updated again) match the oracle on the case and
    # within the bounds of test_gpu_train.py (committed weights, its seed-5 batch of 24).  The trunk gradients of the tensor-core
    # step carry single-term flips of ~1 / sqrt(N) of a tensor's norm, so they are checked on the batch those bounds were set on.
    ctx.freeze_trunk(False)
    ctx.load_weights(nets.pack_params(P))
    ctx.reset_optimizer()
    x, at, y, masks, packed = _batch(24, 5)
    loss_ref, G_ref, P_ref, _ = on.train_step(P, *x, at, y, masks=masks, lr=1e-3)
    loss = ctx.train_forward_backward(*[dev(a) for a in x], dev(at), dev(y), drop_masks=dev(packed))
    assert abs(float(loss.item()) - loss_ref) < 1e-4 * max(1.0, abs(loss_ref))
    _assert_grads(nets.unpack_params(ctx.grad_tensor().cpu().numpy()), G_ref)
    ctx.adam_step(lr=1e-3)
    P2 = nets.unpack_params(ctx.get_params())
    for name, arrs in P_ref.items():
        for k, a in enumerate(arrs):
            diff = np.abs(P2[name][k] - a)
            if name.endswith("_bn") and k >= 2:
                assert diff.max() < 2e-5 + 2e-4 * np.abs(a).max(), "%s[%d]: %g" % (name, k, diff.max())
            else:
                g_ref = np.abs(G_ref[(name, k)])
                ok = g_ref > 0.05 * g_ref.max()
                assert ok.any() and diff[ok].max() < 5e-5, "%s[%d]: %g" % (name, k, diff[ok].max())
                assert diff.max() < 2.1e-3
    ctx.close()


@pytest.mark.parametrize("source", ["committed", "random"])
def test_head_eval_matches_eval_batch(weights_path, source):
    ctx = _ctx(_params(source, weights_path))
    x, at, y, _, _ = _batch(600, 13)
    d = [dev(a) for a in x]
    feats = ctx.trunk_features(*d)
    ref = ctx.eval_batch(*d, dev(at), dev(y)).cpu().numpy()
    got = ctx.head_eval_batch(feats, dev(at), dev(y)).cpu().numpy()
    assert abs(got[0] - ref[0]) < 1e-4 * abs(ref[0]) and got[1] == ref[1], (got, ref)
    perm = np.random.RandomState(0).permutation(600)[:250].astype(np.int64)
    sel = torch.from_numpy(perm).cuda()
    ref = ctx.eval_batch(*[a[sel].contiguous() for a in d], dev(at[perm]), dev(y[perm])).cpu().numpy()
    got = ctx.head_eval_batch(feats, dev(at), dev(y), idx=dev(perm)).cpu().numpy()
    assert abs(got[0] - ref[0]) < 1e-4 * abs(ref[0]) and got[1] == ref[1], (got, ref)
    ctx.close()


def test_fine_tune_end_to_end(tmp_path, weights_path):
    from cnn_cort import base, nets, synthetic
    root = str(tmp_path / "train")
    for i, name in enumerate(("s01", "s02")):
        synthetic.write_subject(root, name, shape=(44, 40, 36), seed=20 + i, with_labels=True,
                                contrast={l: 40.0 * ((l * 7) % 5 - 2) for l in range(1, 16)})
    options = {'train_folder': root, 't1_name': 'T1.nii.gz', 'roi_name': 'gt_15_classes.nii.gz', 'patch_size': [32, 32],
               'debug': 'False', 'device': 0, 'experiment': 'ft', 'mode': 'cuda0', 'load_weights': 'False', 'net_verbose': 0,
               'train_split': 0.25, 'max_epochs': 4, 'patience': 10, 'batch_size': 128, 'seed': 1}
    np.random.seed(3)
    scans = base.load_scan_training_set(options)
    net = nets.build_model(str(tmp_path), options)
    net.load_params_from(weights_path)
    net.fine_tune(scans)
    H = net.train_history_
    assert len(H) == 4 and set(H[0]) == {'epoch', 'train_loss', 'valid_loss', 'valid_accuracy', 'train_loss_best',
                                         'valid_loss_best', 'dur'}
    assert H[-1]['train_loss'] < H[0]['train_loss'], [h['train_loss'] for h in H]
    wfile = os.path.join(str(tmp_path), 'ft', 'ft.pkl')
    assert os.path.exists(wfile) and os.path.exists(os.path.join(str(tmp_path), 'ft', 'ft_history.pkl'))
    with open(wfile, 'rb') as f:
        W = pickle.load(f)
    C = on.load_params(weights_path)
    for name in C:
        if fto.is_trunk(name):
            for a, b in zip(W[name], C[name]):
                assert np.array_equal(a, np.asarray(b, np.float32)), name
    assert not np.array_equal(W['FC1'][0], np.asarray(C['FC1'][0], np.float32))      # the head did move
    net.fit(scans, epochs=1)                     # the trunk is unfrozen again
    assert len(net.train_history_) == 5 and np.isfinite(net.train_history_[-1]['train_loss'])


def test_argument_errors(weights_path):
    from cnn_cort import _native
    P = on.load_params(weights_path)
    ctx = _ctx(P)
    lib, h, st = ctx.lib, ctx.h, torch.cuda.current_stream().cuda_stream
    x, at, y, _, _ = _batch(8, 2)
    d = [dev(a) for a in x]
    feats = ctx.trunk_features(*d)
    d_at, d_y = dev(at), dev(y)
    loss = torch.zeros(1, device="cuda")
    out2 = torch.zeros(2, device="cuda")
    p = lambda t: t.data_ptr()

    def err(status, name):
        assert status == -2, status
        assert name in lib.sc_last_error().decode(), (name, lib.sc_last_error())

    err(lib.sc_trunk_features(h, None, p(d[1]), p(d[2]), 8, p(feats), st), "in1_dev")
    err(lib.sc_trunk_features(h, p(d[0]), p(d[1]), p(d[2]), 8, None, st), "feats_dev")
    err(lib.sc_trunk_features(h, p(d[0]), p(d[1]), p(d[2]), 0, p(feats), st), "n =")
    err(lib.sc_head_train_forward_backward(h, None, p(d_at), p(d_y), None, 8, 8, 0, None, p(loss), st), "feats_dev")
    err(lib.sc_head_train_forward_backward(h, p(feats), None, p(d_y), None, 8, 8, 0, None, p(loss), st), "atlas_rows_dev")
    err(lib.sc_head_train_forward_backward(h, p(feats), p(d_at), None, None, 8, 8, 0, None, p(loss), st), "labels_dev")
    err(lib.sc_head_train_forward_backward(h, p(feats), p(d_at), p(d_y), None, 8, 8, 0, None, None, st), "loss_dev")
    for n in (0, -3, 16385):
        err(lib.sc_head_train_forward_backward(h, p(feats), p(d_at), p(d_y), None, n, 20000, 0, None, p(loss), st), "n =")
    err(lib.sc_head_eval_batch(h, p(feats), p(d_at), None, None, 8, p(out2), st), "labels_dev")
    err(lib.sc_head_eval_batch(h, p(feats), p(d_at), p(d_y), None, 8, None, st), "out2_dev")
    err(lib.sc_head_eval_batch(h, p(feats), p(d_at), p(d_y), None, 0, p(out2), st), "n =")
    ctx.set_option("gemm", 0)
    for call in (lambda: ctx.trunk_features(*d), lambda: ctx.head_train_forward_backward(feats, d_at, d_y),
                 lambda: ctx.head_eval_batch(feats, d_at, d_y), lambda: ctx.freeze_trunk(True)):
        with pytest.raises(_native.NativeError, match="gemm"):
            call()
    ctx.freeze_trunk(False)                      # unfreezing is always allowed
    ctx.close()
