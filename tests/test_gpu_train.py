"""K4/K5 parity: one training step (training-mode forward, loss, every gradient tensor, Lasagne Adam,
BN running statistics) through the C-ABI vs the fp64 autograd oracle with injected dropout masks;
then the nolearn-style fit loop."""
import os
import pickle

import numpy as np
import pytest
import torch

from oracle import network as on
from gpu_util import cuda_ctx, dev

pytestmark = pytest.mark.gpu


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


# Gradient tolerances per back-end, relative to the largest entry of each tensor.  The exact-fp32 SIMT cross-check agrees with
# the fp64 oracle to 2e-3.  The tensor-core path stores activations as bf16 hi+lo pairs (2^-17 relative) and the network is
# piecewise linear: a pre-activation within ~1e-5 of a PReLU kink or a max-pool tie may take the other branch, which moves ONE
# term of a sum of ~10^4 terms by its full size; such rare single-element flips are allowed for by the looser max-norm bound,
# while the relative L2 bound keeps the tensor as a whole within 3e-2: the terms of a weight gradient have random signs, so with
# N ~ 10^4 terms (17 .. 24 samples) ONE flipped term is ~ 1 / sqrt(N) = 1 % of the tensor's norm; runs with one to three flips
# have been observed (1.8e-2 on saggital_ch_conv1), a wrong kernel shows up as tens of per cent.
# (which elements flip varies from run to run: the BatchNorm sums are accumulated with floating-point atomics)
TOL = {0: dict(maxnorm=2e-3, l2=2e-3, well=1e-5), 1: dict(maxnorm=5e-2, l2=3e-2, well=None)}


@pytest.mark.parametrize("backend", [1, 0])
@pytest.mark.parametrize("source,n", [("committed", 24), ("random", 17)])
def test_train_step_matches_autograd_oracle(weights_path, source, n, backend):
    from cnn_cort import nets
    P = on.load_params(weights_path) if source == "committed" else on.init_params(3)
    ctx = cuda_ctx()
    ctx.load_weights(nets.pack_params(P))
    ctx.set_option("gemm", backend)
    tol = TOL[backend]
    x, at, y, masks, packed = _batch(n, 5)
    loss_ref, G_ref, P_ref, state = on.train_step(P, *x, at, y, masks=masks, lr=1e-3)
    loss = ctx.train_forward_backward(*[dev(a) for a in x], dev(at), dev(y), drop_masks=dev(packed))
    assert abs(float(loss.item()) - loss_ref) < 1e-4 * max(1.0, abs(loss_ref)), (float(loss.item()), loss_ref)
    G = nets.unpack_params(ctx.grad_tensor().cpu().numpy())
    worst = 0.0
    for (name, k), g_ref in G_ref.items():
        g = G[name][k].astype(np.float64)
        denom = max(np.abs(g_ref).max(), 1e-6)
        err = np.abs(g - g_ref).max() / denom
        l2 = np.linalg.norm(g - g_ref) / max(np.linalg.norm(g_ref), 1e-6)
        worst = max(worst, err)
        assert err < tol["maxnorm"], "%s[%d]: rel err %g (|g|max %g)" % (name, k, err, denom)
        assert l2 < tol["l2"], "%s[%d]: relative L2 err %g" % (name, k, l2)
    # BN batch statistics ride in the gradient slots of the running statistics
    ctx.adam_step(lr=1e-3)
    P_new = nets.unpack_params(ctx.get_params())
    for name, arrs in P_ref.items():
        for k, a in enumerate(arrs):
            diff = np.abs(P_new[name][k] - a)
            if name.endswith("_bn") and k >= 2:      # running mean / inv_std: 0.9 s + 0.1 batch
                assert diff.max() < 2e-5 + 2e-4 * np.abs(a).max(), "%s[%d]: %g" % (name, k, diff.max())
            else:
                # Adam's first step is lr*g/(|g| + 3.2e-7): only entries with |g| >> 3e-7 are well conditioned
                g_ref = np.abs(G_ref[(name, k)])
                ok = g_ref > (tol["well"] if tol["well"] else 0.05 * g_ref.max())
                assert ok.any() and diff[ok].max() < 5e-5, "%s[%d]: %g" % (name, k, diff[ok].max())
                assert diff.max() < 2.1e-3
    assert ctx.counter("adam_t") == 1
    # the refreshed inference layouts see the new parameters
    proba, _ = ctx.forward(*[dev(a) for a in x], dev(at))
    ref = on.forward(P_new, *x, at, dtype=torch.float64)
    assert np.abs(proba.cpu().numpy() - ref).max() < 1e-3
    ctx.close()


def test_generated_masks_and_eval(weights_path):
    from cnn_cort import nets
    P = on.load_params(weights_path)
    ctx = cuda_ctx()
    ctx.load_weights(nets.pack_params(P))
    x, at, y, _, _ = _batch(40, 9)
    d = [dev(a) for a in x] + [dev(at), dev(y)]
    l1 = float(ctx.train_forward_backward(*d, seed=1).item())
    g1 = ctx.grad_tensor().clone()
    l1b = float(ctx.train_forward_backward(*d, seed=1).item())
    l2 = float(ctx.train_forward_backward(*d, seed=2).item())
    assert abs(l1 - l1b) < 1e-5 * max(1, abs(l1)) and l1 != l2 and np.isfinite(l1) and np.isfinite(l2)
    assert torch.isfinite(g1).all() and float(g1.abs().max()) > 0
    lh = float(ctx.train_forward_backward(*d, n_global=80, seed=1).item())   # DP shard of a global batch of 80
    assert abs(lh - 0.5 * l1) < 1e-5 * max(1, abs(l1))
    out = ctx.eval_batch(*d).cpu().numpy()
    ref = on.forward(P, *x, at, dtype=torch.float64)
    ce = -np.log(ref[np.arange(40), y]).sum()
    assert abs(out[0] - ce) < 1e-3 * max(1.0, ce) and out[1] == (np.argmax(ref, 1) == y).sum()
    ctx.close()


def test_fit_loop_history_checkpoint_and_early_stopping(tmp_path):
    from cnn_cort import nets
    rng = np.random.RandomState(0)
    n = 96
    y = np.repeat(np.arange(3), n // 3).astype(np.uint8)
    x = [rng.randn(n, 1, 32, 32).astype(np.float32) * 0.5 for _ in range(3)]
    for c in range(3):                      # class-dependent mean makes the problem learnable
        for a in x:
            a[y == c] += c - 1
    at = np.zeros((n, 15), np.float32)
    at[np.arange(n), (y + 14) % 15] = 1     # atlas channel j <-> class j+1
    perm = rng.permutation(n)
    x = [a[perm] for a in x]; at = at[perm]; y = y[perm]
    options = {'experiment': 'unit', 'patch_size': [32, 32], 'mode': 'cuda0', 'device': 0, 'load_weights': 'False',
               'net_verbose': 0, 'train_split': 0.25, 'max_epochs': 6, 'patience': 2, 'batch_size': 32, 'seed': 1}
    net = nets.build_model(str(tmp_path), options)
    net.fit({'in1': x[0], 'in2': x[1], 'in3': x[2], 'in4': at}, y)
    H = net.train_history_
    assert 1 <= len(H) <= 6 and set(H[0]) == {'epoch', 'train_loss', 'valid_loss', 'valid_accuracy', 'train_loss_best',
                                               'valid_loss_best', 'dur'}
    assert H[-1]['train_loss'] < H[0]['train_loss'] and np.isfinite(H[-1]['valid_loss'])
    wfile = os.path.join(str(tmp_path), 'unit', 'unit.pkl')
    assert os.path.exists(wfile) and os.path.exists(os.path.join(str(tmp_path), 'unit', 'unit_history.pkl'))
    with open(wfile, 'rb') as f:
        W = pickle.load(f)
    assert list(W.keys()) == [n_ for n_, _ in nets.layer_table()] and W['fc_2'][0].shape == (555, 270)
    options2 = dict(options, load_weights='True')
    net2 = nets.build_model(str(tmp_path), options2)          # resume = load_params_from (weights + BN statistics only)
    p = net2.predict_proba({'in1': x[0], 'in2': x[1], 'in3': x[2], 'in4': at})
    assert p.shape == (n, 15) and np.allclose(p.sum(1), 1, atol=1e-4)
    assert net2.predict({'in1': x[0], 'in2': x[1], 'in3': x[2], 'in4': at}).dtype == np.int64


@pytest.mark.parametrize("t1_dtype", [np.float32, np.int16])
def test_load_data_and_generate_training_set(tmp_path, t1_dtype):
    """a-8: load_data -> generate_training_set on synthetic subjects (boundary-restricted sampling) vs the oracle.
    int16 T1: the train-path normalisation is float32 arithmetic under the reference's numpy 1.12 (base.py:146)."""
    from cnn_cort import base, nifti, synthetic
    from oracle import gather as og
    root = str(tmp_path)
    for i, name in enumerate(("s01", "s02")):
        synthetic.write_subject(root, name, shape=(44, 40, 36), seed=20 + i, with_labels=True, t1_dtype=t1_dtype)
    options = {'train_folder': root, 't1_name': 'T1.nii.gz', 'roi_name': 'gt_15_classes.nii.gz', 'patch_size': [32, 32],
               'debug': 'False', 'device': 0}
    x_axial, x_cor, x_sag, y_axial, x_atlas, names = base.load_data(options)
    assert len(x_axial) == len(x_cor) == len(x_sag) == len(y_axial) == len(x_atlas) == len(names) == 2
    for s, name in enumerate(("s01", "s02")):
        t1 = nifti.load(os.path.join(root, name, "T1.nii.gz")).get_data()
        lab = nifti.load(os.path.join(root, name, "gt_15_classes.nii.gz")).get_data()
        atlas = nifti.load(os.path.join(root, name, "tmp", "MNI_sub_probabilities.nii.gz")).get_data()
        norm = og.normalise(t1, np.float32)
        assert t1.dtype == t1_dtype and norm.dtype == np.float32
        pos = og.get_mask_voxels(np.logical_and(lab > 0, lab < 15))
        n_pos = len(pos)
        n_neg = min(n_pos, int((lab == 15).sum()))          # shuffled list truncated to len(positives), base.py:327-329
        assert x_axial[s].shape == (n_pos + n_neg, 32, 32) and x_axial[s].dtype == np.float32
        # positives: all of them, in np.nonzero order, bit-exact patches and labels
        for got, mode in zip((x_axial[s], x_cor[s], x_sag[s]), og.VIEWS):
            assert np.array_equal(got[:n_pos], og.get_patches(norm, pos, (32, 32), mode))
        assert np.array_equal(y_axial[s][:n_pos, 16, 16], lab[pos[:, 0], pos[:, 1], pos[:, 2]])
        assert np.array_equal(x_atlas[s][:n_pos], og.atlas_vectors_train(atlas, pos))
        # negatives: n_pos distinct label-15 voxels (random subset)
        assert (y_axial[s][n_pos:, 16, 16] == 15).all()
    xa, xc, xs, xat, y = base.generate_training_set(x_axial, x_cor, x_sag, x_atlas, y_axial, options)
    n = sum(len(a) for a in x_axial)
    assert xa.shape == (n, 1, 32, 32) and xat.shape == (n, 15) and y.shape == (n,) and y.dtype == np.uint8
    assert y.max() <= 14 and 0 < (y == 0).sum() <= n // 2       # label 15 -> class 0
