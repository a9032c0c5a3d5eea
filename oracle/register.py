"""Oracle: atlas registration (affine + cubic B-spline FFD, NMI), restated in float64 numpy / scipy.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  Every step of ``csrc/register.cu`` written out as the definition the
device is checked against; the conventions are those of the registration section of ``include/subcort_b200.h``:

* reference = subject T1 (mask: voxels != 0), floating = template; both with a row-major voxel -> mm 4x4 matrix;
* phi(x) = A [x; 1] + u(v): subject mm -> template mm, A 3x4, u a cubic B-spline displacement in template mm whose
  control point (i, j, k) sits at subject voxel ((i-1) s, (j-1) s, (k-1) s), grid dims floor((d-1)/s) + 4;
* trilinear sampling; a point is inside the floating image when its voxel coordinate lies in [0, d-1] on every axis,
  outside it samples 0 and the subject voxel does not count towards the similarity;
* NMI = (H_R + H_F) / H_RF over a 64 x 64 joint histogram with cubic B-spline Parzen windows on both axes, intensities
  mapped linearly to [2, 61] (reference: min / max over its mask; floating: over every voxel, so that an interpolated
  value can never leave the range);
* bending energy BE = mean over the interior control points of the squared second derivatives of u with respect to the
  grid coordinates, cross terms doubled, evaluated analytically at the control points; J = (1 - lambda) NMI - lambda BE.
"""
import numpy as np
from scipy import ndimage

BINS = 64
SPACING = 5                  # control-point spacing in voxels of the level's subject image
LAMBDA = 0.001               # bending-energy weight of the FFD objective
MIN_LEVEL_DIM = 16           # a pyramid level is used only when every subject dim is at least this
AFF_LEVELS, AFF_ITERS, AFF_ALPHA0, AFF_ALPHA_MAX = 4, 50, 1.0, 4.0     # alphas in level voxels (max corner move)
FFD_LEVELS, FFD_ITERS, FFD_ALPHA0, FFD_ALPHA_MAX = 3, 150, 0.5, 2.0    # alphas in level voxels (max control-point move)
ALPHA_MIN = 0.01


# ---------------------------------------------------------------------------------------------
# pyramid and geometry
# ---------------------------------------------------------------------------------------------
def downsample(vol):
    """[1/4, 1/2, 1/4] along each axis (edge voxels repeated), then every second voxel: dims (d + 1) // 2"""
    v = np.asarray(vol, np.float64)
    for ax in range(3):
        v = ndimage.correlate1d(v, [0.25, 0.5, 0.25], axis=ax, mode='nearest')
    return v[::2, ::2, ::2]


def pyramid(vol, levels):
    out = [np.asarray(vol, np.float64)]
    for _ in range(1, levels):
        out.append(downsample(out[-1]))
    return out


def level_vox2mm(M, level):
    return np.asarray(M, np.float64) @ np.diag([2.0 ** level] * 3 + [1.0])


def used_levels(ref_dims, flo_dims, n):
    """coarsest first: level 0 and the levels l < n at which both images have every dim >= MIN_LEVEL_DIM"""
    d, ok = np.concatenate([ref_dims, flo_dims]).astype(np.int64), []
    for l in range(n):
        if (d >= MIN_LEVEL_DIM).all() or l == 0:
            ok.append(l)
        d = (d + 1) // 2
    return ok[::-1]


def grid_dims(dims, s=SPACING):
    return tuple(int((d - 1) // s + 4) for d in dims)


def bspline_basis(f):
    f = np.asarray(f, np.float64)
    return np.stack([(1 - f) ** 3 / 6, (3 * f ** 3 - 6 * f ** 2 + 4) / 6, (-3 * f ** 3 + 3 * f ** 2 + 3 * f + 1) / 6, f ** 3 / 6], -1)


def bspline_matrix(n, s, g):
    """[n, g]: weight of control point i at voxel v (cps floor(v/s) .. floor(v/s) + 3)"""
    v = np.arange(n)
    a = v // s
    w = bspline_basis((v - a * s) / float(s))
    B = np.zeros((n, g))
    for k in range(4):
        B[v, a + k] = w[:, k]
    return B


def field(grid, dims, s=SPACING):
    """u [X, Y, Z, 3] of a control-point grid [gx, gy, gz, 3]"""
    Bx, By, Bz = (bspline_matrix(d, s, g) for d, g in zip(dims, grid.shape[:3]))
    return np.einsum('xi,yj,zk,ijkc->xyzc', Bx, By, Bz, grid, optimize=True)


def field_adjoint(g, gdims, s=SPACING):
    """transpose of field(): [X, Y, Z, 3] voxel values -> [gx, gy, gz, 3] (z pass, then y, then x)"""
    Bx, By, Bz = (bspline_matrix(d, s, n) for d, n in zip(g.shape[:3], gdims))
    t = np.einsum('zk,xyzc->xykc', Bz, g)
    t = np.einsum('yj,xykc->xjkc', By, t)
    return np.einsum('xi,xjkc->ijkc', Bx, t)


def subdivide(grid, fine_dims, s=SPACING):
    """exact cubic B-spline refinement to the next finer level (half the spacing in subject voxels): fine cp j sits on
    coarse cp (j + 1) / 2 when j is odd, between coarse cps j / 2 and j / 2 + 1 when j is even"""
    out = np.asarray(grid, np.float64)
    for ax, gf in enumerate(grid_dims(fine_dims, s)):
        c = np.moveaxis(out, ax, 0)
        j = np.arange(gf)
        i = (j + 1) // 2
        odd = (j % 2 == 1)[(slice(None),) + (None,) * (c.ndim - 1)]
        im, ip = np.clip(i - 1, 0, None), np.minimum(i + 1, c.shape[0] - 1)
        vo = (c[im] + 6 * c[i] + c[ip]) / 8
        ie = j // 2
        ve = (c[ie] + c[np.minimum(ie + 1, c.shape[0] - 1)]) / 2
        out = np.moveaxis(np.where(odd, vo, ve), 0, ax)
    return out


def ref_mm(dims, M):
    """subject voxel centres in mm [X, Y, Z, 3]"""
    v = np.stack(np.meshgrid(*[np.arange(d, dtype=np.float64) for d in dims], indexing='ij'), -1)
    return v @ M[:3, :3].T + M[:3, 3]


def phi(dims, M, A, grid=None, s=SPACING):
    """phi(x) in template mm [X, Y, Z, 3]"""
    p = ref_mm(dims, M) @ A[:3, :3].T + A[:3, 3]
    if grid is not None:
        p = p + field(grid, dims, s)
    return p


def trilinear(vol, w):
    """sample vol [X, Y, Z(, C)] at voxel coordinates w [..., 3] -> (values, voxel gradient [..., 3] (1 channel only),
    inside); 0 outside"""
    vol = np.asarray(vol, np.float64)
    d = np.array(vol.shape[:3])
    inside = ((w >= 0) & (w <= d - 1)).all(-1)
    wc = np.clip(w, 0, d - 1)
    i0 = np.minimum(np.floor(wc).astype(np.int64), np.maximum(d - 2, 0))
    f = wc - i0
    val, grad = 0.0, np.zeros(w.shape)
    for dx in (0, 1):
        for dy in (0, 1):
            for dz in (0, 1):
                c = vol[i0[..., 0] + dx, i0[..., 1] + dy, i0[..., 2] + dz]
                wx = f[..., 0] if dx else 1 - f[..., 0]
                wy = f[..., 1] if dy else 1 - f[..., 1]
                wz = f[..., 2] if dz else 1 - f[..., 2]
                if c.ndim > w.ndim - 1:
                    val = val + (wx * wy * wz)[..., None] * c
                    continue
                val = val + wx * wy * wz * c
                grad[..., 0] += (1 if dx else -1) * wy * wz * c
                grad[..., 1] += wx * (1 if dy else -1) * wz * c
                grad[..., 2] += wx * wy * (1 if dz else -1) * c
    ins = inside[..., None] if np.ndim(val) > inside.ndim else inside
    return np.where(ins, val, 0.0), np.where(inside[..., None], grad, 0.0), inside


def warp(flo, MF, A, grid, ref_dims, MR, s=SPACING):
    """floating volume [X, Y, Z(, C)] resampled on the subject grid through phi (0 outside)"""
    p = phi(ref_dims, MR, A, grid, s)
    w = (p - MF[:3, 3]) @ np.linalg.inv(MF[:3, :3]).T
    return trilinear(flo, w)[0]


# ---------------------------------------------------------------------------------------------
# similarity
# ---------------------------------------------------------------------------------------------
def parzen(t):
    """cubic B-spline beta3(t) and its derivative"""
    a = np.abs(t)
    b = np.where(a < 1, 2 / 3 - a * a + a ** 3 / 2, np.where(a < 2, (2 - a) ** 3 / 6, 0.0))
    db = np.where(a < 1, -2 * t + 1.5 * t * a, np.where(a < 2, -0.5 * np.sign(t) * (2 - a) ** 2, 0.0))
    return b, db


def ranges(ref, flo):
    """(rmin, rscale, fmin, fscale): bin = 2 + (v - min) * scale, [min, max] -> [2, 61]"""
    rm = ref[ref != 0]
    rmin, rmax = float(rm.min()), float(rm.max())
    fmin, fmax = float(flo.min()), float(flo.max())
    return rmin, 59.0 / max(rmax - rmin, 1e-30), fmin, 59.0 / max(fmax - fmin, 1e-30)


def objective(ref, MR, flo, MF, A, grid=None, s=SPACING, want_grad=False, rng=None):
    """-> dict(nmi, be, j, grad_A [3, 4] (d NMI / d A), grad_grid [gx, gy, gz, 3] (d J / d grid)).  J = NMI without a grid."""
    ref = np.asarray(ref, np.float64)
    dims = ref.shape
    rmin, rs, fmin, fs = rng or ranges(ref, flo)
    x = ref_mm(dims, MR)
    p = x @ A[:3, :3].T + A[:3, 3]
    if grid is not None:
        p = p + field(grid, dims, s)
    Qi = np.linalg.inv(MF[:3, :3])
    w = (p - MF[:3, 3]) @ Qi.T
    F, gF, inside = trilinear(flo, w)
    sel = (ref != 0) & inside
    n = int(sel.sum())
    if n == 0:
        raise ValueError("the reference mask does not overlap the template")
    r = 2 + (ref[sel] - rmin) * rs
    f = 2 + (F[sel] - fmin) * fs
    ra, fa = np.floor(r).astype(np.int64), np.floor(f).astype(np.int64)
    H = np.zeros(BINS * BINS)
    wr = [parzen(ra + i - 1 - r)[0] for i in range(4)]
    wf = [parzen(fa + k - 1 - f) for k in range(4)]
    for i in range(4):
        for k in range(4):
            H += np.bincount((ra + i - 1) * BINS + fa + k - 1, wr[i] * wf[k][0], BINS * BINS)
    P = H.reshape(BINS, BINS) / n
    pr, pf = P.sum(1), P.sum(0)

    def ent(q):
        q = q[q > 0]
        return -(q * np.log(q)).sum()

    HR, HF, HRF = ent(pr), ent(pf), ent(P.ravel())
    nmi = (HR + HF) / HRF
    be, gbe = (0.0, None) if grid is None else bending_energy(grid)
    lam = 0.0 if grid is None else LAMBDA
    out = {'nmi': nmi, 'be': be, 'j': (1 - lam) * nmi - lam * be, 'n': n}
    if not want_grad:
        return out
    with np.errstate(divide='ignore', invalid='ignore'):
        T = np.where(P > 0, (nmi * np.log(P) - np.log(pf)[None, :]) / HRF, 0.0)
    dF = np.zeros(n)
    for i in range(4):
        for k in range(4):
            dF += T[ra + i - 1, fa + k - 1] * wr[i] * wf[k][1]
    dF *= -fs / n                          # -(1/N) sum T beta3(a - r) beta3'(b - f), times the bin scale
    g = np.zeros(dims + (3,))
    g[sel] = dF[:, None] * (gF[sel] @ Qi)
    gx = np.concatenate([x, np.ones(dims + (1,))], -1)
    out['grad_A'] = np.einsum('xyzi,xyzj->ij', g, gx)
    if grid is not None:
        out['grad_grid'] = (1 - lam) * field_adjoint(g, grid.shape[:3], s) - lam * gbe
    return out


# ---------------------------------------------------------------------------------------------
# bending energy
# ---------------------------------------------------------------------------------------------
_B = np.array([1 / 6, 4 / 6, 1 / 6])
_D1 = np.array([-0.5, 0.0, 0.5])
_D2 = np.array([1.0, -2.0, 1.0])
# (x, y, z) 1-D stencils and weight of the six second derivatives: xx, yy, zz, xy, xz, yz
BE_TERMS = [((_D2, _B, _B), 1.0), ((_B, _D2, _B), 1.0), ((_B, _B, _D2), 1.0),
            ((_D1, _D1, _B), 2.0), ((_D1, _B, _D1), 2.0), ((_B, _D1, _D1), 2.0)]


def _stencil(st):
    return st[0][:, None, None] * st[1][None, :, None] * st[2][None, None, :]


def bending_energy(grid):
    """-> (BE, dBE/dgrid) over the interior control points (1 .. g-2 on every axis)"""
    g = np.asarray(grid, np.float64)
    gx, gy, gz = g.shape[:3]
    ncp = (gx - 2) * (gy - 2) * (gz - 2)
    be, grad = 0.0, np.zeros_like(g)
    for st, wt in BE_TERMS:
        K = _stencil(st)
        D = np.zeros((gx - 2, gy - 2, gz - 2, 3))
        for a in range(3):
            for b in range(3):
                for c in range(3):
                    D += K[a, b, c] * g[a:a + gx - 2, b:b + gy - 2, c:c + gz - 2]
        be += wt * (D * D).sum()
        for a in range(3):
            for b in range(3):
                for c in range(3):
                    grad[a:a + gx - 2, b:b + gy - 2, c:c + gz - 2] += 2 * wt * K[a, b, c] * D
    return be / ncp, grad / ncp


# ---------------------------------------------------------------------------------------------
# optimiser
# ---------------------------------------------------------------------------------------------
def ascend(value, grad, x0, norm, alpha0, alpha_max, alpha_min, max_iter):
    """Polak-Ribiere conjugate directions with a backtracking step: the direction is scaled so that norm(step) = alpha;
    a step that raises the objective is taken and alpha <- min(1.5 alpha, alpha_max), otherwise alpha is halved.  Ends
    when alpha < alpha_min or after max_iter accepted steps.  -> (x, accepted steps)"""
    x = x0.copy()
    J = value(x)
    g = grad(x)
    d = g.copy()
    alpha, it = alpha0, 0
    while it < max_iter and alpha >= alpha_min:
        n = norm(d)
        if not n > 0:
            break
        xt = x + (alpha / n) * d
        Jt = value(xt)
        if Jt > J:
            x, J, it = xt, Jt, it + 1
            alpha = min(1.5 * alpha, alpha_max)
            gn = grad(x)
            gg = (g * g).sum()
            beta = max(0.0, (gn * (gn - g)).sum() / gg) if gg > 0 else 0.0
            d = gn + beta * d
            g = gn
        else:
            alpha *= 0.5
    return x, it


def mask_box(ref):
    """half-open voxel box of ref != 0"""
    nz = np.nonzero(ref)
    return [(int(a.min()), int(a.max()) + 1) for a in nz]


def _centre_of_mass(vol, M, weights):
    x = ref_mm(vol.shape, M)
    w = weights.astype(np.float64)
    return (x * w[..., None]).reshape(-1, 3).sum(0) / w.sum()


def init_affine(ref, MR, flo, MF):
    """translation that aligns the intensity centres of mass (reference: over its mask)"""
    A = np.eye(4)
    A[:3, 3] = _centre_of_mass(flo, MF, flo) - _centre_of_mass(ref, MR, np.where(ref != 0, ref, 0))
    return A


def affine_frame(ref_l, MR_l):
    """(corners [8, 3] in mm of the mask's box, centre c, R^2): the step is normalised by the largest corner move; the
    search runs in theta = (L R, A (c; 1)) so that a unit of every parameter moves the box by about the same"""
    box = mask_box(ref_l)
    cs = np.array([[bx, by, bz] for bx in (box[0][0], box[0][1] - 1) for by in (box[1][0], box[1][1] - 1)
                   for bz in (box[2][0], box[2][1] - 1)], np.float64)
    corners = cs @ MR_l[:3, :3].T + MR_l[:3, 3]
    c = corners.mean(0)
    R2 = max(((corners - c) ** 2).sum(1).mean() / 3.0, 1e-12)
    return corners, c, R2


def register_affine(ref, MR, flo, MF, levels=AFF_LEVELS, iters=AFF_ITERS, verbose=False):
    ref, flo = np.asarray(ref, np.float64), np.asarray(flo, np.float64)
    MR, MF = np.asarray(MR, np.float64), np.asarray(MF, np.float64)
    A = init_affine(ref, MR, flo, MF)
    rp, fp = pyramid(ref, levels), pyramid(flo, levels)
    h0 = np.sqrt((MR[:3, :3] ** 2).sum(0)).min()
    stats = []
    for l in used_levels(ref.shape, flo.shape, levels):
        ref_l, flo_l = rp[l], fp[l]
        MR_l, MF_l = level_vox2mm(MR, l), level_vox2mm(MF, l)
        rng = ranges(ref_l, flo_l)
        corners, c, R2 = affine_frame(ref_l, MR_l)
        R = np.sqrt(R2)

        def to_A(th):
            B = np.eye(4)
            B[:3, :3] = th[:9].reshape(3, 3) / R
            B[:3, 3] = th[9:] - B[:3, :3] @ c
            return B

        def to_theta(B):
            return np.concatenate([(B[:3, :3] * R).ravel(), B[:3, :3] @ c + B[:3, 3]])

        def value(th):
            return objective(ref_l, MR_l, flo_l, MF_l, to_A(th), rng=rng)['nmi']

        def grad(th):
            G = objective(ref_l, MR_l, flo_l, MF_l, to_A(th), rng=rng, want_grad=True)['grad_A']
            gl = G[:, :3] - np.outer(G[:, 3], c)      # gradient w.r.t. L with t' = L c + t held
            return np.concatenate([(gl / R).ravel(), G[:, 3]])

        def norm(d):
            dL = d[:9].reshape(3, 3) / R
            return np.sqrt((((corners - c) @ dL.T + d[9:]) ** 2).sum(1)).max()

        h = h0 * 2.0 ** l
        th, it = ascend(value, grad, to_theta(A), norm, AFF_ALPHA0 * h, AFF_ALPHA_MAX * h, ALPHA_MIN * h, iters)
        A = to_A(th)
        stats.append((l, it))
        if verbose:
            print("affine level %d: %d steps, nmi %.5f" % (l, it, value(th)))
    return A, stats


def register_ffd(ref, MR, flo, MF, A, levels=FFD_LEVELS, iters=FFD_ITERS, verbose=False):
    ref, flo = np.asarray(ref, np.float64), np.asarray(flo, np.float64)
    MR, MF = np.asarray(MR, np.float64), np.asarray(MF, np.float64)
    rp, fp = pyramid(ref, levels), pyramid(flo, levels)
    h0 = np.sqrt((MR[:3, :3] ** 2).sum(0)).min()
    grid, stats = None, []
    for l in used_levels(ref.shape, flo.shape, levels):
        ref_l, flo_l = rp[l], fp[l]
        MR_l, MF_l = level_vox2mm(MR, l), level_vox2mm(MF, l)
        rng = ranges(ref_l, flo_l)
        grid = np.zeros(grid_dims(ref_l.shape) + (3,)) if grid is None else subdivide(grid, ref_l.shape)
        shape = grid.shape

        def value(x):
            return objective(ref_l, MR_l, flo_l, MF_l, A, x.reshape(shape), rng=rng)['j']

        def grad(x):
            return objective(ref_l, MR_l, flo_l, MF_l, A, x.reshape(shape), rng=rng, want_grad=True)['grad_grid'].ravel()

        def norm(d):
            return np.sqrt((d.reshape(-1, 3) ** 2).sum(1)).max()

        h = h0 * 2.0 ** l
        x, it = ascend(value, grad, grid.ravel(), norm, FFD_ALPHA0 * h, FFD_ALPHA_MAX * h, ALPHA_MIN * h, iters)
        grid = x.reshape(shape)
        stats.append((l, it))
        if verbose:
            print("ffd level %d: %d steps, J %.5f" % (l, it, value(x)))
    return grid, stats


def jacobian_det_min(dims, M, A, grid, mask=None, s=SPACING):
    """smallest determinant of d phi / d x (central differences of phi on the subject grid, in mm / mm) over mask"""
    p = phi(dims, M, A, grid, s)
    J = np.stack([np.gradient(p[..., c], axis=a) for c in range(3) for a in range(3)], -1).reshape(dims + (3, 3))
    J = J @ np.linalg.inv(M[:3, :3])          # per voxel -> per mm
    det = np.linalg.det(J)
    return float(det[mask].min() if mask is not None else det.min())
