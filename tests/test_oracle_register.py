"""oracle/register.py on its own (CPU): the NMI gradients against finite differences, exact subdivision, the warp against
scipy, affine recovery by the oracle optimiser, and the configuration keys of the registration."""
import configparser

import numpy as np
import pytest
from scipy import ndimage

from oracle import register as orr
from cnn_cort import synthetic
from cnn_cort.load_options import load_options

MR = np.array([[1.0, 0.1, 0.0, -11.0], [0.0, 1.05, 0.0, -10.0], [0.05, 0.0, 0.95, -9.0], [0, 0, 0, 1.0]])
MF = np.array([[1.1, 0.05, 0.0, -20.0], [0.0, 1.0, 0.1, -18.0], [0.02, 0.0, 1.2, -17.0], [0, 0, 0, 1.0]])


def _pair(seed=0):
    """24^3-ish subject inside a larger template, related by a known transform; evaluated away from it"""
    rng = np.random.RandomState(seed)
    flo = ndimage.gaussian_filter(rng.randn(36, 34, 32), 2.0) * 100 + 500
    A = np.eye(4)
    A[:3, :3] += 0.02 * rng.randn(3, 3)
    A[:3, 3] = rng.randn(3)
    gd = orr.grid_dims((24, 22, 20))
    grid = rng.randn(*gd, 3) * 0.5
    ref = orr.warp(flo, MF, A, grid, (24, 22, 20), MR) * 0.8 + 20
    ref[:3] = 0
    A2 = A.copy()
    A2[:3, :3] += 0.01 * rng.randn(3, 3)
    A2[:3, 3] += 0.3 * rng.randn(3)
    return ref, flo, A2, grid + 0.2 * rng.randn(*grid.shape)


def test_nmi_gradient_matches_finite_differences():
    ref, flo, A, grid = _pair()
    rng_ = orr.ranges(ref, flo)
    o = orr.objective(ref, MR, flo, MF, A, grid, want_grad=True, rng=rng_)
    assert o['n'] == int((ref != 0).sum())        # every masked voxel lands inside the template
    eps = 1e-6
    fd = np.zeros((3, 4))
    for i in range(3):
        for j in range(4):
            Ap, Am = A.copy(), A.copy()
            Ap[i, j] += eps
            Am[i, j] -= eps
            fd[i, j] = (orr.objective(ref, MR, flo, MF, Ap, grid, rng=rng_)['nmi'] - orr.objective(ref, MR, flo, MF, Am, grid, rng=rng_)['nmi']) / (2 * eps)
    assert np.linalg.norm(fd - o['grad_A']) <= 1e-3 * np.linalg.norm(o['grad_A'])
    r = np.random.RandomState(1)
    idx = [tuple(r.randint(0, d) for d in grid.shape[:3]) + (r.randint(3),) for _ in range(40)]
    an, fdv = [], []
    for ix in idx:
        gp, gm = grid.copy(), grid.copy()
        gp[ix] += eps
        gm[ix] -= eps
        fdv.append((orr.objective(ref, MR, flo, MF, A, gp, rng=rng_)['j'] - orr.objective(ref, MR, flo, MF, A, gm, rng=rng_)['j']) / (2 * eps))
        an.append(o['grad_grid'][ix])
    an, fdv = np.array(an), np.array(fdv)
    assert np.linalg.norm(fdv - an) <= 1e-3 * np.linalg.norm(an)
    # the NMI part alone (no bending energy): d NMI / d grid from the adjoint
    g_nmi = (o['grad_grid'] + orr.LAMBDA * orr.bending_energy(grid)[1]) / (1 - orr.LAMBDA)
    fdn = []
    for ix in idx[:15]:
        gp, gm = grid.copy(), grid.copy()
        gp[ix] += eps
        gm[ix] -= eps
        fdn.append((orr.objective(ref, MR, flo, MF, A, gp, rng=rng_)['nmi'] - orr.objective(ref, MR, flo, MF, A, gm, rng=rng_)['nmi']) / (2 * eps))
    an = np.array([g_nmi[ix] for ix in idx[:15]])
    assert np.linalg.norm(np.array(fdn) - an) <= 1e-3 * np.linalg.norm(an)


def test_subdivision_reproduces_the_coarse_field():
    fine_dims = (37, 30, 41)
    coarse_dims = tuple((d + 1) // 2 for d in fine_dims)
    rng = np.random.RandomState(2)
    coarse = rng.randn(*orr.grid_dims(coarse_dims), 3)
    fine = orr.subdivide(coarse, fine_dims)
    assert fine.shape[:3] == orr.grid_dims(fine_dims)
    uc = orr.field(coarse, coarse_dims)
    uf = orr.field(fine, fine_dims)
    assert np.abs(uf[::2, ::2, ::2] - uc).max() < 1e-9


def test_warp_equals_map_coordinates():
    rng = np.random.RandomState(3)
    flo = rng.randn(20, 18, 16)
    A = np.eye(4)
    A[:3, :3] += 0.05 * rng.randn(3, 3)
    A[:3, 3] = rng.randn(3) * 4
    grid = rng.randn(*orr.grid_dims((14, 15, 13)), 3)
    dims = (14, 15, 13)
    got = orr.warp(flo, MF, A, grid, dims, MR)
    p = orr.phi(dims, MR, A, grid)
    w = (p - MF[:3, 3]) @ np.linalg.inv(MF[:3, :3]).T
    inside = ((w >= 0) & (w <= np.array(flo.shape) - 1)).all(-1)
    want = ndimage.map_coordinates(flo, np.moveaxis(w, -1, 0), order=1, cval=0.0)
    assert 0.1 < inside.mean() < 1.0
    assert np.allclose(np.where(inside, want, 0.0), got, atol=1e-12)


def test_oracle_recovers_a_known_affine():
    P = synthetic.make_registration_pair((40, 40, 40), seed=3, subject_spacing=(2.0, 2.0, 2.4), template_spacing=3.0, deform_mm=0.0,
                                         translation_mm=8.0)
    A, _ = orr.register_affine(P['t1'], P['t1_affine'], P['template'], P['template_affine'])
    m = P['t1'] != 0
    err = np.sqrt(((orr.phi(P['t1'].shape, P['t1_affine'], A) - P['phi']) ** 2).sum(-1))[m]
    A0 = orr.init_affine(P['t1'].astype(np.float64), P['t1_affine'], P['template'].astype(np.float64), P['template_affine'])
    err0 = np.sqrt(((orr.phi(P['t1'].shape, P['t1_affine'], A0) - P['phi']) ** 2).sum(-1))[m]
    assert err0.mean() > 2.0
    assert err.mean() < 0.5, err.mean()


def _cfg(extra=""):
    cfg = configparser.RawConfigParser()
    cfg.read_string("""[database]
train_folder = /t
inference_folder = /i
t1_name = T1.nii.gz
roi_name = gt.nii.gz
save_tmp = True
%s
[model]
name = m
mode = cuda0
patch_size = 32
batch_size = 256
patience = 20
net_verbose = 1
max_epochs = 100
train_split = 0.25
test_batch_size = 100000
load_weights = True
out_probabilities = False
speedup_segmentation = True
post_process = True
debug = True
""" % extra)
    return cfg


@pytest.mark.parametrize("extra,want", [("", (None, None)),
                                        ("atlas_template = /a/MNI.nii.gz\natlas_priors = /a/priors.nii.gz", ("/a/MNI.nii.gz", "/a/priors.nii.gz"))])
def test_config_registration_keys(extra, want):
    o = load_options(_cfg(extra))
    assert (o['atlas_template'], o['atlas_priors']) == want
    assert o['t1_name'] == 'T1.nii.gz' and o['device'] == 0
