"""Synthetic subjects for benchmarks and tests (SURVEY.md 8d): a strictly positive smooth
T1, a 15-channel atlas prior made of Gaussian blobs (with all-zero rows far from every
blob, to exercise the background fix), the registered-mask file the crop path reads and
a 15-class label volume for training.  Not part of the reference; it only pre-creates the
files whose existence makes the reference skip registration (base.py:201,362).
"""
import os

import numpy as np

from . import nifti


def make_t1(shape, seed=1234):
    from scipy.ndimage import gaussian_filter
    rng = np.random.RandomState(seed)
    f = gaussian_filter(rng.standard_normal(shape).astype(np.float32), 3.0)
    f /= f.std()
    f += 0.15 * rng.standard_normal(shape).astype(np.float32)
    return np.maximum(f * 150.0 + 600.0, 1.0).astype(np.float32)


def make_atlas(shape, seed=1234):
    """-> (atlas [X,Y,Z,15] float32, blob centres [14,3], sigmas [14])"""
    rng = np.random.RandomState(seed + 7)
    X, Y, Z = shape
    atlas = np.zeros(shape + (15,), np.float32)
    box = np.array([min(96, X), min(96, Y), min(64, Z)]) // 2
    mid = np.array(shape) // 2
    cen = np.stack([rng.randint(mid[a] - box[a], mid[a] + box[a] + 1, size=14) for a in range(3)], 1)
    sig = rng.uniform(6.0, 12.0, size=14) * min(1.0, min(shape) / 128.0 + 0.25)
    near = np.zeros(shape, bool)
    for j in range(14):
        g = [np.exp(-0.5 * ((np.arange(shape[a]) - cen[j, a]) / sig[j]) ** 2).astype(np.float32) for a in range(3)]
        lo = [max(0, int(cen[j, a] - 4 * sig[j])) for a in range(3)]
        hi = [min(shape[a], int(cen[j, a] + 4 * sig[j]) + 1) for a in range(3)]
        sl = tuple(slice(l, h) for l, h in zip(lo, hi))
        blob = g[0][sl[0], None, None] * g[1][None, sl[1], None] * g[2][None, None, sl[2]]
        blob[blob < 1e-3] = 0
        atlas[sl + (j,)] = blob
        r = int(40 * min(1.0, min(shape) / 128.0 + 0.25))
        nl = [max(0, cen[j, a] - r) for a in range(3)]
        nh = [min(shape[a], cen[j, a] + r + 1) for a in range(3)]
        near[tuple(slice(l, h) for l, h in zip(nl, nh))] = True
    s = atlas[..., :14].sum(-1)
    big = s > 1.0
    atlas[big, :14] /= s[big, None]
    atlas[..., 14] = np.clip(1.0 - atlas[..., :14].sum(-1), 0.0, 1.0)
    atlas[~near] = 0.0
    return atlas, cen, sig


def make_mask(atlas):
    from scipy.ndimage import binary_dilation
    m = atlas[..., 0:13].sum(-1) > 0.01
    return binary_dilation(m, iterations=5).astype(np.float32)


def make_labels(atlas):
    """labels 1..14 where a structure prior > 0.5, a 2-voxel ring of 15 around them, else 0"""
    from scipy.ndimage import binary_dilation
    best = atlas[..., :14].argmax(-1)
    val = atlas[..., :14].max(-1)
    lab = np.where(val > 0.5, best + 1, 0).astype(np.uint8)
    ring = binary_dilation(lab > 0, iterations=2) & (lab == 0)
    lab[ring] = 15
    return lab


def _rotation(deg, axis):
    a = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    t = np.deg2rad(deg)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(t) * K + (1 - np.cos(t)) * K @ K


def _bspline_field(coef, dims, s):
    """cubic B-spline displacement [X,Y,Z,3] of control points [gx,gy,gz,3] spaced s voxels, cp i at voxel (i - 1) s"""
    mats = []
    for n, g in zip(dims, coef.shape[:3]):
        v = np.arange(n)
        a = v // s
        f = (v - a * s) / float(s)
        w = np.stack([(1 - f) ** 3 / 6, (3 * f ** 3 - 6 * f ** 2 + 4) / 6, (-3 * f ** 3 + 3 * f ** 2 + 3 * f + 1) / 6, f ** 3 / 6], 1)
        B = np.zeros((n, g))
        for k in range(4):
            B[v, a + k] = w[:, k]
        mats.append(B)
    return np.einsum('xi,yj,zk,ijkc->xyzc', mats[0], mats[1], mats[2], coef, optimize=True)


def _trilinear(vol, w):
    """vol [X,Y,Z(,C)] at voxel coordinates w [...,3]; 0 where w leaves [0, d-1] on any axis"""
    d = np.array(vol.shape[:3])
    inside = ((w >= 0) & (w <= d - 1)).all(-1)
    wc = np.clip(w, 0, d - 1)
    i0 = np.minimum(np.floor(wc).astype(np.int64), d - 2)
    f = wc - i0
    out = 0.0
    for dx in (0, 1):
        for dy in (0, 1):
            for dz in (0, 1):
                wt = (f[..., 0] if dx else 1 - f[..., 0]) * (f[..., 1] if dy else 1 - f[..., 1]) * (f[..., 2] if dz else 1 - f[..., 2])
                c = vol[i0[..., 0] + dx, i0[..., 1] + dy, i0[..., 2] + dz]
                out = out + (wt[..., None] * c if c.ndim > wt.ndim else wt * c)
    return np.where(inside[..., None] if np.ndim(out) > inside.ndim else inside, out, 0.0)


def make_registration_pair(subject_shape=(128, 128, 128), template_shape=None, seed=0, subject_spacing=(1.0, 1.0, 1.2),
                           template_spacing=1.5, oblique_deg=5.0, rotation_deg=8.0, scale=0.1, shear=0.03,
                           translation_mm=12.0, deform_mm=4.0, intensity=(0.8, 40.0), noise=0.01, identity=False):
    """A subject made from a template through a known transform, for registration tests and benchmarks.

    Template: make_t1 texture plus the make_atlas structures, inside an ellipsoidal head (0 outside), on a
    template_spacing mm grid centred on the origin; its priors are make_atlas's.  Subject: subject_shape voxels of
    subject_spacing mm with an oblique_deg sform rotation, intensities a * T(phi_true(x)) + b plus Gaussian noise (noise x
    the template's standard deviation) where T(phi_true(x)) > 0, else 0.  phi_true(x) = A_true [x; 1] + u_true(x) (subject mm
    -> template mm): A_true rotates by rotation_deg, scales each axis by up to +-scale, shears by up to shear and
    translates by translation_mm; u_true is a cubic B-spline on a grid of 10 subject voxels with random coefficients,
    scaled to max |u| = deform_mm.  identity=True returns the template itself as the subject (phi_true = identity).

    -> dict: t1, t1_affine (4x4 vox -> mm), template, template_affine, priors (template grid, [X,Y,Z,15]),
    truth_priors (the priors warped through phi_true, trilinear), phi (template mm, [X,Y,Z,3]), affine (A_true 4x4)."""
    rng = np.random.RandomState(seed + 11)
    subject_shape = tuple(int(s) for s in subject_shape)
    fov = max(n * sp for n, sp in zip(subject_shape, subject_spacing))
    if template_shape is None:
        template_shape = (int(np.ceil(fov * 1.15 / template_spacing)),) * 3
    template_shape = tuple(int(s) for s in template_shape)
    MF = np.diag([template_spacing] * 3 + [1.0])
    MF[:3, 3] = -template_spacing * (np.array(template_shape) - 1) / 2.0
    atlas, _, _ = make_atlas(template_shape, seed)
    tex = make_t1(template_shape, seed)
    tex = tex + 300.0 * (atlas[..., :14] * (np.arange(14) % 3 - 1.0)).sum(-1)
    x = np.stack(np.meshgrid(*[np.arange(n, dtype=np.float64) for n in template_shape], indexing='ij'), -1) @ MF[:3, :3].T + MF[:3, 3]
    radii = np.array([0.40, 0.36, 0.33]) * np.array(template_shape) * template_spacing
    head = ((x / radii) ** 2).sum(-1) <= 1.0
    template = np.where(head, np.maximum(tex, 1.0), 0.0).astype(np.float32)
    if identity:
        phi = x
        return {'t1': template.copy(), 't1_affine': MF.copy(), 'template': template, 'template_affine': MF,
                'priors': atlas, 'truth_priors': atlas.copy(), 'phi': phi, 'affine': np.eye(4)}
    MR = np.eye(4)
    MR[:3, :3] = _rotation(oblique_deg, (1.0, 1.0, 0.0)) @ np.diag(subject_spacing)
    MR[:3, 3] = -MR[:3, :3] @ ((np.array(subject_shape) - 1) / 2.0)
    A = np.eye(4)
    S = np.diag(1.0 + rng.uniform(-scale, scale, 3))
    Sh = np.eye(3) + np.triu(rng.uniform(-shear, shear, (3, 3)), 1)
    A[:3, :3] = _rotation(rotation_deg, rng.randn(3)) @ Sh @ S
    t = rng.randn(3)
    A[:3, 3] = translation_mm * t / np.linalg.norm(t)
    xs = np.stack(np.meshgrid(*[np.arange(n, dtype=np.float64) for n in subject_shape], indexing='ij'), -1) @ MR[:3, :3].T + MR[:3, 3]
    phi = xs @ A[:3, :3].T + A[:3, 3]
    if deform_mm > 0:
        g = tuple((n - 1) // 10 + 4 for n in subject_shape)
        u = _bspline_field(rng.randn(*(g + (3,))), subject_shape, 10)
        phi = phi + u * (deform_mm / np.sqrt((u ** 2).sum(-1)).max())
    w = (phi - MF[:3, 3]) @ np.linalg.inv(MF[:3, :3]).T
    warped = _trilinear(template.astype(np.float64), w)
    a, b = intensity
    t1 = np.where(warped > 0, a * warped + b + noise * template[head].std() * rng.standard_normal(subject_shape), 0.0)
    return {'t1': t1.astype(np.float32), 't1_affine': MR, 'template': template, 'template_affine': MF, 'priors': atlas,
            'truth_priors': _trilinear(atlas, w).astype(np.float32), 'phi': phi, 'affine': A}


def write_subject(root, name, shape=(256, 256, 256), seed=1234, with_labels=False, t1_name="T1.nii.gz",
                  roi_name="gt_15_classes.nii.gz", zoom=1.0, t1_dtype=np.float32, contrast=None):
    """contrast: None, or per-label mean intensities {label: value} (or a sequence indexed by label 0..15) added to the T1
    inside each labelled structure, so that the image carries its structures; two tables make two "scanner" domains.  None
    writes exactly what it always did."""
    d = os.path.join(root, name)
    os.makedirs(os.path.join(d, "tmp"), exist_ok=True)
    aff = np.diag([zoom, zoom, zoom, 1.0])
    t1 = make_t1(shape, seed)
    atlas, _, _ = make_atlas(shape, seed)
    if contrast is not None:
        table = np.zeros(16, np.float32)
        for l, v in (contrast.items() if isinstance(contrast, dict) else enumerate(contrast)):
            table[int(l)] = v
        t1 = (t1 + table[make_labels(atlas)]).astype(t1.dtype)
    if np.dtype(t1_dtype).kind in "iu":       # scanner-style integer intensities (the usual on-disk type of a T1)
        t1 = np.rint(t1).astype(t1_dtype)
    nifti.Nifti1Image(t1, aff).to_filename(os.path.join(d, t1_name))
    nifti.Nifti1Image(atlas, aff).to_filename(os.path.join(d, "tmp", "MNI_sub_probabilities.nii.gz"))
    nifti.Nifti1Image(make_mask(atlas), aff).to_filename(os.path.join(d, "tmp", "MNI_subcortical_mask.nii.gz"))
    if with_labels:
        nifti.Nifti1Image(make_labels(atlas), aff).to_filename(os.path.join(d, roi_name))
    return d
