"""Training from device-resident scans: sc_gather_samples bit-exact against the oracle, load_scan_training_set equal to
load_data + generate_training_set, the same training step and fit loop as on the materialised arrays, and data-parallel
fit on a scan set (tests/dp_scans_check.py under torchrun)."""
import ctypes
import os
import pickle
import random
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import gather as og
from gpu_util import cuda_ctx, dev

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))

SHAPES = [(40, 36, 33), (21, 50, 28), (7, 5, 6)]     # the last one is smaller than a patch on every axis


@pytest.fixture(scope="module")
def ctx():
    c = cuda_ctx()
    yield c
    c.close()


def _table():
    rng = np.random.RandomState(0)
    vols = [rng.randn(*s).astype(np.float32) for s in SHAPES]
    rows = []
    for k, s in enumerate(SHAPES):
        corners = np.array([(x, y, z) for x in (0, s[0] - 1) for y in (0, s[1] - 1) for z in (0, s[2] - 1)])
        interior = np.stack([rng.randint(0, d, 24) for d in s], 1)
        c = np.concatenate([corners, interior])
        rows.append(np.concatenate([np.full((len(c), 1), k), c], 1))
    samples = np.ascontiguousarray(np.concatenate(rows), dtype=np.int32)
    atlas = rng.rand(len(samples), 15).astype(np.float32)
    labels = rng.randint(0, 15, len(samples)).astype(np.uint8)
    per = [np.nonzero(samples[:, 0] == k)[0] for k in range(3)]
    idx = np.stack([p[:32] for p in per], 1).reshape(-1)                # subjects interleaved
    idx = np.concatenate([idx, idx[::-3], [5, 5, 5, 40, 40]]).astype(np.int64)   # repeated rows
    return vols, samples, atlas, labels, idx


def _expected(vols, samples, rows, mode):
    out = np.empty((len(rows), 32, 32), np.float32)
    for k, v in enumerate(vols):
        m = samples[rows, 0] == k
        if m.any():
            out[m] = og.get_patches(v, samples[rows[m], 1:], (32, 32), mode)
    return out


def test_gather_samples_bit_exact(ctx):
    vols, samples, atlas, labels, idx = _table()
    d_vols = [dev(v) for v in vols]
    table = ctx.scan_table(d_vols)
    ds, da, dy = dev(samples), dev(atlas), dev(labels)
    for ix in (idx, None):
        rows = ix if ix is not None else np.arange(len(samples))
        got = ctx.gather_samples(table, 3, ds, da, dy, idx=None if ix is None else dev(ix))
        for t, mode in zip(got[:3], og.VIEWS):
            assert t.shape == (len(rows), 1, 32, 32)
            assert np.array_equal(t[:, 0].cpu().numpy(), _expected(vols, samples, rows, mode)), mode
        assert np.array_equal(got[3].cpu().numpy(), atlas[rows]) and np.array_equal(got[4].cpu().numpy(), labels[rows])
    # every output NULL on its own: the others are still exact
    full = [t.cpu().numpy() for t in ctx.gather_samples(table, 3, ds, da, dy, idx=dev(idx))]
    for off in range(5):
        views = tuple(v != off for v in range(3))
        got = ctx.gather_samples(table, 3, ds, da, dy, idx=dev(idx), views=views, want_atlas=off != 3, want_y=off != 4)
        assert got[off] is None
        for k, t in enumerate(got):
            if k != off:
                assert np.array_equal(t.cpu().numpy(), full[k]), (off, k)
    # n == 0 is a no-op
    got = ctx.gather_samples(table, 3, ds, da, dy, idx=dev(np.zeros(0, np.int64)))
    assert got[0].shape == (0, 1, 32, 32) and got[4].shape == (0,)
    torch.cuda.synchronize()


def test_gather_samples_bad_arguments(ctx):
    vols, samples, atlas, labels, idx = _table()
    d_vols = [dev(v) for v in vols]
    table = ctx.scan_table(d_vols)
    ds, da, dy = dev(samples), dev(atlas), dev(labels)
    out = torch.empty((4, 1, 32, 32), device="cuda")
    at = torch.empty((4, 15), device="cuda")
    y = torch.empty(4, dtype=torch.uint8, device="cuda")
    P = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None      # noqa: E731
    lib = ctx.lib

    def call(table_=table, n_scans=3, samples_=ds, atlas_=da, labels_=dy, n=4, at_out=at, y_out=y):
        return lib.sc_gather_samples(ctx.h, P(table_), n_scans, P(samples_), P(atlas_), P(labels_), None, n,
                                     P(out), P(out), P(out), P(at_out), P(y_out), None)

    assert call() == 0
    assert call(n=0, table_=None, samples_=None) == 0                       # no-op
    assert call(n=-1) == -2 and b"sc_gather_samples" in lib.sc_last_error()
    assert call(n_scans=-1) == -2 and call(n_scans=0) == -2
    assert call(table_=None) == -2 and call(samples_=None) == -2
    assert call(atlas_=None) == -2 and call(labels_=None) == -2           # output requested without its source
    assert call(atlas_=None, at_out=None) == 0 and call(labels_=None, y_out=None) == 0
    assert lib.sc_gather_samples(None, P(table), 3, P(ds), None, None, None, 4, P(out), None, None, None, None, None) == -2
    torch.cuda.synchronize()


def _write_subjects(root, t1_dtype, shape=(44, 40, 36)):
    from cnn_cort import synthetic
    for i, name in enumerate(("s01", "s02")):
        synthetic.write_subject(root, name, shape=shape, seed=20 + i, with_labels=True, t1_dtype=t1_dtype)
    return {'train_folder': root, 't1_name': 'T1.nii.gz', 'roi_name': 'gt_15_classes.nii.gz', 'patch_size': [32, 32],
            'debug': 'False', 'device': 0}


def _both_sets(options, seed=7):
    from cnn_cort import base
    random.seed(seed)
    np.random.seed(seed)
    x_axial, x_cor, x_sag, y_axial, x_atlas, _ = base.load_data(options)
    arrays = base.generate_training_set(x_axial, x_cor, x_sag, x_atlas, y_axial, options)
    random.seed(seed)
    np.random.seed(seed)
    return arrays, base.load_scan_training_set(options)


@pytest.mark.parametrize("t1_dtype", [np.float32, np.int16])
def test_scan_set_equals_reference_pipeline(tmp_path, t1_dtype):
    arrays, scans = _both_sets(_write_subjects(str(tmp_path), t1_dtype))
    got = scans.to_arrays()
    assert len(scans) == len(arrays[4]) > 0 and len(scans.names) == 2
    for a, b, what in zip(got, arrays, ("axial", "coronal", "saggital", "atlas", "y")):
        assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b), what
    assert scans.device_bytes() < sum(a.nbytes for a in arrays) // 10


@pytest.fixture(scope="module")
def sets(tmp_path_factory):
    return _both_sets(_write_subjects(str(tmp_path_factory.mktemp("scans")), np.float32))


def test_train_step_on_gathered_batch_matches_arrays(sets, weights_path):
    from cnn_cort import nets
    from oracle import network as on
    from test_gpu_train import TOL, _batch
    arrays, scans = sets
    ctx = cuda_ctx()
    ctx.load_weights(nets.pack_params(on.load_params(weights_path)))
    rows = np.random.RandomState(1).choice(len(scans), 24, replace=False)
    packed = dev(_batch(24, 5)[4])
    ref_in = [dev(a[rows]) for a in arrays]
    got_in = scans.gather(rows, ctx=ctx)
    for a, b in zip(ref_in, got_in):
        assert torch.equal(a, b)
    res = []
    for inputs in (ref_in, got_in):
        loss = float(ctx.train_forward_backward(*inputs, drop_masks=packed).item())
        res.append((loss, nets.unpack_params(ctx.grad_tensor().cpu().numpy())))
    (l0, G0), (l1, G1) = res
    assert abs(l0 - l1) < 1e-4 * max(1.0, abs(l0))
    tol = TOL[ctx.counter("gemm")]                 # run-to-run noise of the BatchNorm atomics, test_gpu_train.py
    for name, arrs in G0.items():
        for k, g in enumerate(arrs):
            g, h = g.astype(np.float64), G1[name][k].astype(np.float64)
            assert np.abs(g - h).max() <= tol["maxnorm"] * max(np.abs(g).max(), 1e-6), (name, k)
            assert np.linalg.norm(g - h) <= tol["l2"] * max(np.linalg.norm(g), 1e-6), (name, k)
    ctx.close()


def _record_minibatches(ctx, log):
    """wrap the context's training / evaluation calls so that every minibatch fit feeds them is logged as CRCs of its
    tensors plus the step's global batch size and dropout seed"""
    import zlib

    def digest(ts):
        return tuple(zlib.crc32(t.contiguous().cpu().numpy().tobytes()) for t in ts)

    train, evaluate = ctx.train_forward_backward, ctx.eval_batch

    def train_rec(*b, **kw):
        log.append(("train", digest(b), kw.get("n_global"), kw.get("seed")))
        return train(*b, **kw)

    def eval_rec(*b):
        log.append(("eval", digest(b)))
        return evaluate(*b)

    ctx.train_forward_backward, ctx.eval_batch = train_rec, eval_rec


def test_fit_on_scans_matches_fit_on_arrays(sets, tmp_path):
    """fit(scans) runs the loop of fit(arrays) with another minibatch source: from the same initialisation and seeds, every
    training and validation minibatch (inputs, labels, global batch size, dropout seed) must be bit-identical, in the same
    order.  The losses then differ only by the run-to-run noise of the training step itself: its kernels reduce with
    floating-point atomics, so two fits of the SAME arrays already differ in the last bits, which flips PReLU / max-pool
    decisions and grows over the steps (0.4 - 3.4 % of the validation loss after two epochs here).  The losses are held to 5 %;
    a minibatch source that misaligned inputs and labels would give a loss near chance (ln 15 = 2.7)."""
    from cnn_cort import nets
    arrays, scans = sets
    H, logs = [], []
    for arm in ("arrays", "scans"):
        options = {'experiment': arm, 'patch_size': [32, 32], 'mode': 'cuda0', 'device': 0, 'load_weights': 'False',
                   'net_verbose': 0, 'train_split': 0.25, 'max_epochs': 2, 'patience': 5, 'batch_size': 1024, 'seed': 1}
        net = nets.build_model(str(tmp_path), options)
        logs.append([])
        _record_minibatches(net.ctx, logs[-1])
        if arm == "scans":
            net.fit(scans)
            with pytest.raises(ValueError):
                net.fit(scans, scans.y)
        else:
            xa, xc, xs, xat, y = arrays
            net.fit({'in1': xa, 'in2': xc, 'in3': xs, 'in4': xat}, y)
        H.append(net.train_history_)
        with open(os.path.join(str(tmp_path), arm, arm + '.pkl'), 'rb') as f:
            assert nets.pack_params(pickle.load(f)).size == nets._native.PARAM_FLOATS
    n_train = -(-len(nets.TrainSplit(0.25).indices(scans.y)[0]) // 1024)
    assert sum(e[0] == "train" for e in logs[0]) == 2 * n_train
    assert logs[0] == logs[1]
    assert len(H[0]) == len(H[1]) == 2
    for a, b in zip(*H):
        for k in ('train_loss', 'valid_loss'):
            assert np.isfinite(a[k]) and np.isfinite(b[k]) and abs(a[k] - b[k]) <= 0.05 * abs(a[k]), (k, a[k], b[k])


def _free_port():
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _run_dp(tmp_path, extra):
    root = str(tmp_path)
    _write_subjects(root, np.float32, shape=(36, 32, 30))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(HERE, "dp_scans_check.py"), "--data=" + root] + extra
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "dp_scans_check ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_dp_fit_on_scans_two_ranks_nccl(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _run_dp(tmp_path, ["--backend=nccl"])


def test_dp_fit_on_scans_two_ranks_sharing_one_gpu_gloo(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    _run_dp(tmp_path, ["--backend=gloo", "--same-device"])
