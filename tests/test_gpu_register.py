"""Atlas registration on the device (csrc/register.cu) against oracle/register.py: kernel parity at a fixed transform,
recovery of known transforms on synthetic pairs, determinism, the mask, the test_scan pipeline and argument errors."""
import os

import numpy as np
import pytest
import torch

from oracle import register as orr
from gpu_util import cuda_ctx, dev
from cnn_cort import _native, base, nifti, synthetic

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = cuda_ctx()
    yield c
    c.close()


def _oblique(spacing, deg, axis, origin):
    M = np.eye(4)
    M[:3, :3] = synthetic._rotation(deg, axis) @ np.diag(spacing)
    M[:3, 3] = origin
    return M


@pytest.fixture(scope="module")
def fixed():
    """non-cubic pair, oblique matrices on both sides, a transform that leaves part of the subject outside the template"""
    rng = np.random.RandomState(5)
    from scipy import ndimage
    flo = (ndimage.gaussian_filter(rng.randn(41, 37, 33), 2.0) * 100 + 500).astype(np.float32)
    MF = _oblique((1.5, 1.4, 1.6), 7.0, (0.2, 1.0, 0.3), (-30.0, -25.0, -26.0))
    ref = (ndimage.gaussian_filter(rng.randn(45, 38, 29), 2.0) * 80 + 300).astype(np.float32)
    ref[:4] = 0
    ref[:, :, -3:] = 0
    MR = _oblique((1.0, 1.1, 1.2), 5.0, (1.0, 1.0, 0.0), (-22.0, -20.0, -17.0))
    A = np.eye(4)
    A[:3, :3] += 0.03 * rng.randn(3, 3)
    A[:3, 3] = rng.randn(3) * 2 + (12.0, 0.0, 0.0)      # part of the subject maps outside the template
    grid = (rng.randn(*orr.grid_dims(ref.shape), 3) * 1.0).astype(np.float32)
    pri = rng.rand(41, 37, 33, 15).astype(np.float32)
    return ref, MR, flo, MF, A, grid, pri


def test_warp_parity(ctx, fixed):
    ref, MR, flo, MF, A, grid, pri = fixed
    for vol in (flo, pri):
        for g in (None, grid):
            got = ctx.warp_volume(dev(vol), MF, A, None if g is None else dev(g), ref.shape, MR).cpu().numpy()
            want = orr.warp(vol, MF, A, None if g is None else g.astype(np.float64), ref.shape, MR)
            assert got.shape == want.shape
            assert (want == 0).any() and (want != 0).any()
            assert np.abs(got - want).max() <= 1e-5 * np.abs(vol).max()


def test_objective_and_gradient_parity(ctx, fixed):
    ref, MR, flo, MF, A, grid, _ = fixed
    g64 = grid.astype(np.float64)
    for g in (None, grid):
        nmi, be, J, ga, gg = ctx.register_objective(dev(ref), MR, dev(flo), MF, A, None if g is None else dev(g), want_grad=True)
        o = orr.objective(ref, MR, flo.astype(np.float64), MF, A, None if g is None else g64, want_grad=True)
        assert abs(nmi - o['nmi']) <= 1e-6 * o['nmi'], (nmi, o['nmi'])
        assert abs(be - o['be']) <= 1e-6 * max(o['be'], 1e-30)
        assert abs(J - o['j']) <= 1e-6 * abs(o['j'])
        assert np.linalg.norm(ga - o['grad_A']) <= 1e-4 * np.linalg.norm(o['grad_A'])
        if g is not None:
            got = gg.cpu().numpy()
            assert np.linalg.norm(got - o['grad_grid']) <= 1e-4 * np.linalg.norm(o['grad_grid'])


def _errors(P, A, grid):
    m = P['t1'] != 0
    ph = orr.phi(P['t1'].shape, P['t1_affine'], A, None if grid is None else grid.astype(np.float64))
    return np.sqrt(((ph - P['phi']) ** 2).sum(-1))[m]


def _register(ctx, P, ffd=True):
    ref, flo = dev(P['t1']), dev(P['template'])
    A = ctx.register_affine(ref, P['t1_affine'], flo, P['template_affine'])
    grid = ctx.register_ffd(ref, P['t1_affine'], flo, P['template_affine'], A) if ffd else None
    return A, grid


def test_recovers_identity(ctx):
    P = synthetic.make_registration_pair((128, 128, 128), identity=True)
    A, _ = _register(ctx, P, ffd=False)
    e = _errors(P, A, None)
    assert e.mean() < 0.05 and e.max() < 0.25, (e.mean(), e.max())


def test_recovers_affine(ctx):
    P = synthetic.make_registration_pair((128, 128, 128), seed=1, deform_mm=0.0)
    A, _ = _register(ctx, P, ffd=False)
    e = _errors(P, A, None)
    assert e.mean() < 0.3 and np.percentile(e, 95) < 0.6, (e.mean(), np.percentile(e, 95))


def test_recovers_affine_and_deformation(ctx):
    P = synthetic.make_registration_pair((128, 128, 128), seed=2, deform_mm=4.0)
    A, grid = _register(ctx, P)
    g = grid.cpu().numpy()
    ea, e = _errors(P, A, None), _errors(P, A, g)
    assert e.mean() < 0.7 and np.percentile(e, 95) < 1.5, (e.mean(), np.percentile(e, 95))
    assert e.mean() < ea.mean()
    m = P['t1'] != 0
    assert orr.jacobian_det_min(P['t1'].shape, P['t1_affine'], A, g.astype(np.float64), m) > 0
    got = ctx.warp_volume(dev(P['priors']), P['template_affine'], A, grid, P['t1'].shape, P['t1_affine']).cpu().numpy()
    truth = P['truth_priors']
    for c in range(14):
        t = truth[..., c] > 0.5
        if t.sum() >= 500:
            r = got[..., c] > 0.5
            dice = 2.0 * (t & r).sum() / (t.sum() + r.sum())
            assert dice >= 0.9, (c, dice)


def test_deterministic_and_mask(ctx):
    P = synthetic.make_registration_pair((96, 96, 96), seed=4, deform_mm=3.0)
    runs = []
    for _ in range(2):
        A, grid, pri, mask = base.register_arrays(ctx, P['t1'], P['t1_affine'], P['template'], P['template_affine'], P['priors'])
        runs.append((A.cpu().numpy(), grid.cpu().numpy(), pri.cpu().numpy(), mask.cpu().numpy()))
    for a, b in zip(runs[0], runs[1]):
        assert a.tobytes() == b.tobytes()
    from scipy.ndimage import binary_dilation
    pri, mask = runs[0][2], runs[0][3]
    want = binary_dilation(pri[..., 0:13].sum(-1) > 0, iterations=5)
    assert mask.dtype == np.float32 and set(np.unique(mask)) <= {0.0, 1.0}
    assert np.array_equal(mask.astype(bool), want)


def _options(test_folder, template=None, priors=None, crop='True'):
    return {'test_folder': test_folder, 't1_name': 'T1.nii.gz', 'out_probabilities': 'False', 'post_process': 'True',
            'crop': crop, 'crop_bool': crop == 'True', 'debug': 'False', 'device': 0, 'test_batch_size': 100000,
            'atlas_template': template, 'atlas_priors': priors}


def test_pipeline(ctx, tmp_path, weights_path):
    from cnn_cort import nets
    from oracle import network as on
    P = synthetic.make_registration_pair((96, 96, 96), seed=6, deform_mm=3.0)
    atl = tmp_path / "atlas"
    atl.mkdir()
    nifti.Nifti1Image(P['template'], P['template_affine']).to_filename(str(atl / "MNI.nii.gz"))
    nifti.Nifti1Image(P['priors'], P['template_affine']).to_filename(str(atl / "priors.nii.gz"))
    subj = tmp_path / "test" / "s1"
    subj.mkdir(parents=True)
    t1 = str(subj / "T1.nii.gz")
    nifti.Nifti1Image(P['t1'], P['t1_affine']).to_filename(t1)
    class _Net(object):          # test_scan's dense path only reads net.ctx
        pass
    net = _Net()
    net.ctx = ctx
    ctx.load_weights(nets.pack_params(on.load_params(weights_path)))
    opts = _options(str(tmp_path / "test"), str(atl / "MNI.nii.gz"), str(atl / "priors.nii.gz"))
    base.test_scan(net, t1, opts)
    names = ['transf.txt', 'rT1d_template.nii.gz', 'MNI_sub_probabilities.nii.gz', 'MNI_subcortical_mask.nii.gz']
    for n in names:
        assert os.path.exists(str(subj / "tmp" / n)), n
    seg = str(subj / "out_subcortical_seg_prec.nii.gz")
    first = nifti.load(seg).get_data().copy()
    mt = {n: os.path.getmtime(str(subj / "tmp" / n)) for n in names}
    base.test_scan(net, t1, opts)                    # reads the files written by the first call
    assert {n: os.path.getmtime(str(subj / "tmp" / n)) for n in names} == mt
    assert np.array_equal(nifti.load(seg).get_data(), first)
    A = np.loadtxt(str(subj / "tmp" / "transf.txt"))
    assert A.shape == (4, 4) and np.array_equal(A[3], [0, 0, 0, 1])
    aff = nifti.load(str(subj / "tmp" / "MNI_sub_probabilities.nii.gz")).affine
    assert np.allclose(aff, P['t1_affine'], atol=1e-5)
    # without a template a missing registration is the same IOError as before
    subj2 = tmp_path / "test2" / "s1"
    subj2.mkdir(parents=True)
    nifti.Nifti1Image(P['t1'], P['t1_affine']).to_filename(str(subj2 / "T1.nii.gz"))
    with pytest.raises(IOError, match="MNI_sub_probabilities.nii.gz is missing"):
        base.test_scan(net, str(subj2 / "T1.nii.gz"), _options(str(tmp_path / "test2")))


def test_errors(ctx, fixed):
    ref, MR, flo, MF, A, grid, pri = fixed
    r, f = dev(ref), dev(flo)
    lib, h, s = ctx.lib, ctx.h, _native._stream()
    D, M = _native._dims, _native._mat
    out = (_native.ctypes.c_double * 16)()

    def err(status):
        assert status == -2          # SC_ERR_ARG
        return lib.sc_last_error().decode()

    assert "ref_dev" in err(lib.sc_register_affine(h, None, D(ref.shape), M(MR), f.data_ptr(), D(flo.shape), M(MF), out, s))
    assert "flo_dev" in err(lib.sc_register_affine(h, r.data_ptr(), D(ref.shape), M(MR), None, D(flo.shape), M(MF), out, s))
    small = dev(np.ones((6, 20, 20), np.float32))
    assert "below 8" in err(lib.sc_register_affine(h, small.data_ptr(), D((6, 20, 20)), M(MR), f.data_ptr(), D(flo.shape), M(MF), out, s))
    sing = MR.copy()
    sing[0, :3] = 0
    assert "ref_vox2mm" in err(lib.sc_register_affine(h, r.data_ptr(), D(ref.shape), M(sing), f.data_ptr(), D(flo.shape), M(MF), out, s))
    nan = MF.copy()
    nan[1, 1] = np.nan
    assert "flo_vox2mm" in err(lib.sc_register_affine(h, r.data_ptr(), D(ref.shape), M(MR), f.data_ptr(), D(flo.shape), M(nan), out, s))
    o = dev(np.zeros(ref.shape + (3,), np.float32))
    assert "channels" in err(lib.sc_warp_volume(h, f.data_ptr(), D(flo.shape), 3, M(MF), M(A), None, D(ref.shape), M(MR), o.data_ptr(), s))
    z = dev(np.zeros(ref.shape, np.float32))
    assert "mask" in err(lib.sc_register_affine(h, z.data_ptr(), D(ref.shape), M(MR), f.data_ptr(), D(flo.shape), M(MF), out, s))
    far = A.copy()
    far[:3, 3] += 1e4
    val = (_native.ctypes.c_double * 3)()
    assert "overlap" in err(lib.sc_register_objective(h, r.data_ptr(), D(ref.shape), M(MR), f.data_ptr(), D(flo.shape), M(MF), M(far),
                                                      None, val, None, None, s))
    with pytest.raises(_native.NativeError, match="ref_vox2mm"):
        ctx.register_affine(r, sing, f, MF)
    ctx.register_objective(r, MR, f, MF, A)          # the next call succeeds
