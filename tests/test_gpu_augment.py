"""Augmented minibatch gather on the device: sc_gather_samples_augmented against the fp64 oracle (tests/augment_oracle.py), its
identity with sc_gather_samples at zero ranges, determinism and row keying, argument errors, and the augmented training paths
of Net.fit and Net.fine_tune on a ScanTrainingSet."""
import ctypes

import numpy as np
import pytest
import torch

import augment_oracle as ao
from gpu_util import cuda_ctx, dev

pytestmark = pytest.mark.gpu

SHAPES = [(40, 36, 33), (21, 50, 28), (7, 5, 6)]     # the last one is smaller than a patch on every axis
CONFIGS = {
    "rotation": dict(rotation_deg=40.0),
    "scale": dict(scale=0.3),
    "intensity": dict(intensity=0.4),
    "noise": dict(noise=0.2),
    "all": dict(rotation_deg=180.0, scale=0.2, intensity=0.3, noise=0.1),
}
U = 2.0 ** -24          # float32 unit roundoff


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
    idx = rng.permutation(len(samples))
    idx = np.concatenate([idx, idx[::-3], [5, 5, 5, 40, 40]]).astype(np.int64)   # shuffled, then repeated rows
    return vols, samples, atlas, labels, idx


def _device(vols, samples, atlas, labels, ctx):
    d_vols = [dev(v) for v in vols]
    return d_vols, ctx.scan_table(d_vols), dev(samples), dev(atlas), dev(labels)


def _tolerance(aug, rows, samples, vmax):
    """bound of |device - oracle| from float32 rounding: the position p = c + (i-16) M e_row + (j-16) M e_col is computed from
    M rounded to float32 with two fused multiply-adds, so each coordinate is off by at most U (2 |c| + 96 s); the trilinear
    interpolant of the zero-extended volume is Lipschitz with constant 2 max|v| per axis; weights, the 8-term sum and the
    intensity transform add a few U of the value; the float32 Box-Muller draw is within 2e-6 (1 + |g|)."""
    prm = ao.parameters(aug, rows)
    cmax = float(np.abs(samples[rows, 1:]).max())
    dp = U * (2 * cmax + 96 * prm["s"].max())
    interp = 3 * dp * 2 * vmax + 16 * U * vmax
    g = np.abs(ao.noise(aug, rows)).max() if aug.get("noise") else 0.0
    return 2 * (prm["a"].max() * interp + 8 * U * (prm["a"].max() * vmax + 1) + aug.get("noise", 0.0) * 2e-6 * (1 + g))


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_kernel_matches_oracle(ctx, name):
    vols, samples, atlas, labels, idx = _table()
    _, table, ds, da, dy = _device(vols, samples, atlas, labels, ctx)
    aug = dict(CONFIGS[name], seed=123, epoch=4)
    got = ctx.gather_samples(table, 3, ds, da, dy, idx=dev(idx), augment=aug)
    want = ao.gather(vols, samples, idx, aug)
    tol = _tolerance(aug, idx, samples, max(float(np.abs(v).max()) for v in vols))
    for v in range(3):
        err = np.abs(got[v][:, 0].cpu().numpy().astype(np.float64) - want[v]).max()
        assert err <= tol, (name, v, err, tol)
    plain = ctx.gather_samples(table, 3, ds, da, dy, idx=dev(idx))
    assert torch.equal(got[3], plain[3]) and torch.equal(got[4], plain[4])
    torch.cuda.synchronize()


def test_linear_volume_to_float32_rounding(ctx):
    """trilinear interpolation is exact on a linear volume, so away from the edges the kernel equals V(c + M o) up to the float32
    rounding of the position and of the values"""
    shape = (90, 96, 84)
    coef = np.array([0.7, -1.3, 0.45])
    X, Y, Z = np.meshgrid(*[np.arange(n, dtype=np.float64) for n in shape], indexing="ij")
    vol = (coef[0] * X + coef[1] * Y + coef[2] * Z + 2.0).astype(np.float32)
    rng = np.random.RandomState(2)
    cen = np.stack([rng.randint(35, n - 35, 64) for n in shape], 1)
    samples = np.ascontiguousarray(np.concatenate([np.zeros((64, 1)), cen], 1), dtype=np.int32)
    d_vol = dev(vol)
    table = ctx.scan_table([d_vol])
    aug = dict(rotation_deg=180.0, scale=0.25, intensity=0.5, seed=3, epoch=1)
    got = ctx.gather_samples(table, 1, dev(samples), augment=aug)
    want = ao.gather([vol.astype(np.float64)], samples, np.arange(64), aug)
    prm = ao.parameters(aug, np.arange(64))
    vmax = float(np.abs(vol).max())
    dp = U * (2 * float(cen.max()) + 96 * prm["s"].max())
    tol = 2 * prm["a"].max() * (np.abs(coef).sum() * dp + 16 * U * vmax) + 8 * U * (prm["a"].max() * vmax + 1)
    for v in range(3):
        err = np.abs(got[v][:, 0].cpu().numpy().astype(np.float64) - want[v]).max()
        assert err <= tol, (v, err, tol)


def test_zero_ranges_equal_plain_gather(ctx):
    vols, samples, atlas, labels, idx = _table()
    _, table, ds, da, dy = _device(vols, samples, atlas, labels, ctx)
    for ix in (dev(idx), None):
        plain = ctx.gather_samples(table, 3, ds, da, dy, idx=ix)
        for aug in (dict(), dict(seed=2 ** 64 - 1, epoch=-5)):
            got = ctx.gather_samples(table, 3, ds, da, dy, idx=ix, augment=aug)
            for a, b in zip(got, plain):
                assert torch.equal(a, b)
    torch.cuda.synchronize()


def test_deterministic_and_keyed_by_row(ctx):
    vols, samples, atlas, labels, idx = _table()
    _, table, ds, da, dy = _device(vols, samples, atlas, labels, ctx)
    aug = dict(CONFIGS["all"], seed=7, epoch=2)
    a = ctx.gather_samples(table, 3, ds, da, dy, idx=dev(idx), augment=aug)
    b = ctx.gather_samples(table, 3, ds, da, dy, idx=dev(idx), augment=aug)
    for x, y in zip(a, b):
        assert np.array_equal(x.cpu().numpy().view(np.uint8), y.cpu().numpy().view(np.uint8))
    for other in (dict(aug, epoch=3), dict(aug, seed=8)):
        c = ctx.gather_samples(table, 3, ds, da, dy, idx=dev(idx), augment=other)
        for v in range(3):
            assert not torch.equal(a[v], c[v])
    # every row's patches depend on the row only: the identity order, a permutation and repeats agree
    full = ctx.gather_samples(table, 3, ds, da, dy, augment=aug)
    for v in range(3):
        assert torch.equal(a[v], full[v][dev(idx)])
    torch.cuda.synchronize()


def test_bad_arguments(ctx):
    from cnn_cort import _native
    vols, samples, atlas, labels, _ = _table()
    _, table, ds, da, dy = _device(vols, samples, atlas, labels, ctx)
    out = torch.empty((4, 1, 32, 32), device="cuda")
    at = torch.empty((4, 15), device="cuda")
    y = torch.empty(4, dtype=torch.uint8, device="cuda")
    P = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None      # noqa: E731
    lib = ctx.lib

    def call(aug=_native.Augment(rotation_deg=10.0), table_=table, n_scans=3, samples_=ds, atlas_=da, labels_=dy, n=4, at_out=at,
             y_out=y):
        return lib.sc_gather_samples_augmented(ctx.h, P(table_), n_scans, P(samples_), P(atlas_), P(labels_), None, n,
                                               None if aug is None else ctypes.byref(aug), P(out), P(out), P(out), P(at_out),
                                               P(y_out), None)

    def err(status, field):
        assert status == -2, (field, status)
        msg = lib.sc_last_error().decode()
        assert "sc_gather_samples_augmented" in msg and field in msg, (field, msg)

    assert call() == 0
    assert call(n=0, table_=None, samples_=None) == 0                       # no-op
    err(call(aug=None), "aug")
    for field, bad in (("rotation_deg", -1.0), ("rotation_deg", 181.0), ("rotation_deg", float("nan")), ("scale", -0.5),
                       ("scale", float("inf")), ("intensity", 1.0), ("intensity", -0.1), ("noise", -1.0), ("noise", float("nan"))):
        err(call(aug=_native.Augment(**{field: bad})), field)
        err(call(aug=_native.Augment(**{field: bad}), n=0, table_=None, samples_=None), field)
    err(call(n=-1), "negative")
    err(call(n_scans=0), "scan list")
    err(call(table_=None), "scan list")
    err(call(samples_=None), "sample table")
    err(call(atlas_=None), "atlas")
    err(call(labels_=None), "label")
    assert call(atlas_=None, at_out=None) == 0 and call(labels_=None, y_out=None) == 0
    with pytest.raises(ValueError, match="unknown"):
        ctx.gather_samples(table, 3, ds, augment=dict(rotation=5.0))
    torch.cuda.synchronize()


AUG = dict(rotation_deg=12.0, scale=0.15, intensity=0.2, noise=0.05, seed=5)


def _scan_set(root, contrast=None):
    from cnn_cort import base, synthetic
    for i, name in enumerate(("s01", "s02")):
        synthetic.write_subject(root, name, shape=(44, 40, 36), seed=20 + i, with_labels=True, contrast=contrast)
    options = {'train_folder': root, 't1_name': 'T1.nii.gz', 'roi_name': 'gt_15_classes.nii.gz', 'patch_size': [32, 32],
               'debug': 'False', 'device': 0}
    np.random.seed(3)
    return base.load_scan_training_set(options)


def _options(name, **kw):
    return dict({'experiment': name, 'patch_size': [32, 32], 'mode': 'cuda0', 'device': 0, 'load_weights': 'False',
                 'net_verbose': 0, 'train_split': 0.25, 'max_epochs': 2, 'patience': 5, 'batch_size': 1024, 'seed': 1,
                 'augment': AUG}, **kw)


def test_fit_gathers_training_minibatches_augmented(tmp_path):
    from cnn_cort import nets
    scans = _scan_set(str(tmp_path / "train"))
    log = []
    gather = scans.gather

    def spy(idx=None, ctx=None, augment=None, epoch=None):
        log.append((augment, epoch))
        return gather(idx, ctx=ctx, augment=augment, epoch=epoch)

    scans.gather = spy
    net = nets.build_model(str(tmp_path), _options("fit_aug"))
    net.fit(scans)
    tr, va = nets.TrainSplit(0.25).indices(scans.y)
    n_tr, n_va = -(-len(tr) // 1024), -(-len(va) // 1024)
    expect = []
    for ep in (1, 2):
        expect += [(AUG, ep)] * n_tr + [(None, None)] * n_va
    assert log == expect
    H = net.train_history_
    assert len(H) == 2 and all(np.isfinite(h['train_loss']) and np.isfinite(h['valid_loss']) for h in H)
    del log[:]
    net.fit(scans, epochs=1)                    # a resumed fit continues the epoch numbers
    assert log[0] == (AUG, 3)
    with pytest.raises(ValueError, match="ScanTrainingSet"):
        xa, xc, xs, xat, y = scans.to_arrays()
        net.fit({'in1': xa, 'in2': xc, 'in3': xs, 'in4': xat}, y)


def test_fine_tune_rebuilds_training_features_per_epoch(tmp_path, weights_path):
    from cnn_cort import nets
    import fine_tune_oracle as fto
    scans = _scan_set(str(tmp_path / "train"), contrast={l: 40.0 * ((l * 7) % 5 - 2) for l in range(1, 16)})
    net = nets.build_model(str(tmp_path), _options("ft_aug", max_epochs=2, batch_size=512))
    net.load_params_from(weights_path)
    ctx = net.ctx
    before = ctx.get_params()
    tr, va = nets.TrainSplit(0.25).indices(scans.y)
    snaps = {}
    step = ctx.head_train_forward_backward

    def spy(feats, *a, **kw):
        snaps.setdefault(len(net.train_history_) + 1, feats.clone())
        return step(feats, *a, **kw)

    ctx.head_train_forward_backward = spy
    net.fine_tune(scans)
    assert sorted(snaps) == [1, 2] and all(np.isfinite(h['train_loss']) for h in net.train_history_)
    after = ctx.get_params()
    mask = np.concatenate([np.full(int(np.prod(s)), fto.is_trunk(name)) for name, shapes in nets.layer_table() for s in shapes])
    assert np.array_equal(before[mask].view(np.uint32), after[mask].view(np.uint32))
    assert not np.array_equal(before[~mask], after[~mask])
    # the frozen trunk's features of the gathers fine_tune fed it, in its chunks (trunk arrays unchanged: recomputing is exact)
    C, n = nets.FEATURE_CHUNK, len(scans)
    plain = torch.cat([ctx.trunk_features(*scans.gather(np.arange(s, min(n, s + C)), ctx=ctx)[:3]) for s in range(0, n, C)])
    d_tr, d_va = dev(tr.astype(np.int64)), dev(va.astype(np.int64))
    for ep, feats in snaps.items():
        assert torch.equal(feats[d_va], plain[d_va]), ep
        want = torch.cat([ctx.trunk_features(*scans.gather(d_tr[s:s + C], ctx=ctx, augment=AUG, epoch=ep)[:3])
                          for s in range(0, len(tr), C)])
        assert torch.equal(feats[d_tr], want), ep
        assert not torch.equal(feats[d_tr], plain[d_tr]), ep
    assert not torch.equal(snaps[1][d_tr], snaps[2][d_tr])
    with pytest.raises(ValueError, match="ScanTrainingSet"):
        xa, xc, xs, xat, y = scans.to_arrays()
        net.fine_tune({'in1': xa, 'in2': xc, 'in3': xs, 'in4': xat}, y)
