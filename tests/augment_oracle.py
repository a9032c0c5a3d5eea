"""Augmented minibatch gather oracle (sc_gather_samples_augmented): the header's definition restated in fp64 numpy.

TEST INFRASTRUCTURE, like ``oracle/``.  Random numbers come from ``mc_dropout_oracle.hash3``, which is pinned against the C++
``hash3`` of csrc/common.cuh.  Everything else is computed in float64: the transform M (not rounded to float32), the sample
positions, the trilinear weights and the intensity transform, so the device result differs from it only by float32 rounding.
"""
import numpy as np

from mc_dropout_oracle import hash3

EPOCH_MIX = 0xD1B54A32D192ED03
SLOTS = 8192            # hash slots per table row
NOISE_SLOT = 1024
# (row axis, column axis) of each view, get_patches's windows: axial rows x, cols y; coronal rows x, cols z; saggital rows y, cols z
VIEW_AXES = ((0, 1), (0, 2), (1, 2))


def epoch_seed(seed, epoch):
    """s_e = seed ^ (epoch * 0xD1B54A32D192ED03) in wrapping uint64 arithmetic"""
    return (int(seed) ^ ((int(epoch) * EPOCH_MIX) & (2 ** 64 - 1))) & (2 ** 64 - 1)


def uniform(se, rows, slot):
    """u(row, slot) = (hash3(s_e, row * 8192 + slot) + 0.5) * 2^-32, float64; rows and slot broadcast"""
    key = np.asarray(rows, dtype=np.uint64) * np.uint64(SLOTS) + np.asarray(slot, dtype=np.uint64)
    return (hash3(se, key).astype(np.float64) + 0.5) * 2.0 ** -32


def parameters(aug, rows):
    """-> dict of float64 arrays per row: axis [n, 3], theta (degrees), s, a, b, and M = s R(axis, theta) [n, 3, 3]"""
    se = epoch_seed(aug.get("seed", 0), aug.get("epoch", 0))
    rows = np.asarray(rows, dtype=np.int64)
    u = [uniform(se, rows, k) for k in range(6)]
    z = 2.0 * u[0] - 1.0
    r = np.sqrt(np.maximum(0.0, 1.0 - z * z))
    phi = 2.0 * np.pi * u[1]
    k = np.stack([r * np.cos(phi), r * np.sin(phi), z], axis=1)
    theta = float(aug.get("rotation_deg", 0.0)) * (2.0 * u[2] - 1.0)
    s = (1.0 + float(aug.get("scale", 0.0))) ** (2.0 * u[3] - 1.0)
    si = float(aug.get("intensity", 0.0))
    a = 1.0 + si * (2.0 * u[4] - 1.0)
    b = si * (2.0 * u[5] - 1.0)
    t = np.deg2rad(theta)
    c, sn = np.cos(t), np.sin(t)
    K = np.zeros((len(rows), 3, 3))
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 2] = -k[:, 2], k[:, 1], -k[:, 0]
    K[:, 1, 0], K[:, 2, 0], K[:, 2, 1] = k[:, 2], -k[:, 1], k[:, 0]
    R = (c[:, None, None] * np.eye(3) + sn[:, None, None] * K + (1.0 - c)[:, None, None] * k[:, :, None] * k[:, None, :])
    return dict(axis=k, theta=theta, s=s, a=a, b=b, M=s[:, None, None] * R)


def noise(aug, rows):
    """Box-Muller g [n, 3, 32, 32] of pixel (view, i, j): slots 1024 + 2 (view * 1024 + i * 32 + j) + {0, 1}"""
    se = epoch_seed(aug.get("seed", 0), aug.get("epoch", 0))
    rows = np.asarray(rows, dtype=np.int64)[:, None]
    n = NOISE_SLOT + 2 * np.arange(3 * 1024, dtype=np.int64)[None, :]
    u1, u2 = uniform(se, rows, n), uniform(se, rows, n + 1)
    return (np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)).reshape(-1, 3, 32, 32)


def positions(M, centres, view):
    """p = c + (i - 16) M e_row + (j - 16) M e_col -> float64 [n, 32, 32, 3]"""
    ar, ac = VIEW_AXES[view]
    o = np.arange(32, dtype=np.float64) - 16.0
    c = np.asarray(centres, dtype=np.float64)
    return (c[:, None, None, :] + o[None, :, None, None] * M[:, None, None, :, ar] + o[None, None, :, None] * M[:, None, None, :, ac])


def trilinear(vol, p):
    """trilinear interpolation of the zero-extended volume at points p [..., 3] (a corner outside contributes 0)"""
    f = np.floor(p)
    t = p - f
    i = f.astype(np.int64)
    out = np.zeros(p.shape[:-1])
    for dx in (0, 1):
        for dy in (0, 1):
            for dz in (0, 1):
                d = (dx, dy, dz)
                w = np.ones(p.shape[:-1])
                ok = np.ones(p.shape[:-1], bool)
                idx = []
                for ax in range(3):
                    q = i[..., ax] + d[ax]
                    w = w * (t[..., ax] if d[ax] else 1.0 - t[..., ax])
                    ok &= (q >= 0) & (q < vol.shape[ax])
                    idx.append(np.clip(q, 0, vol.shape[ax] - 1))
                out += w * np.where(ok, vol[tuple(idx)], 0.0)
    return out


def gather(vols, samples, rows, aug):
    """-> (axial, coronal, saggital) float64 [n, 32, 32] of table rows `rows` (samples int [N, 4]: scan, x, y, z) under the
    augmentation dict aug (rotation_deg, scale, intensity, noise, seed, epoch; absent = 0)"""
    rows = np.asarray(rows, dtype=np.int64)
    prm = parameters(aug, rows)
    g = noise(aug, rows) if aug.get("noise", 0.0) else np.zeros((len(rows), 3, 32, 32))
    out = [np.empty((len(rows), 32, 32)) for _ in range(3)]
    scan, cen = samples[rows, 0], samples[rows, 1:]
    for v in range(3):
        for k, vol in enumerate(vols):
            m = scan == k
            if m.any():
                out[v][m] = trilinear(np.asarray(vol, np.float64), positions(prm["M"][m], cen[m], v))
        out[v] = prm["a"][:, None, None] * out[v] + prm["b"][:, None, None] + float(aug.get("noise", 0.0)) * g[:, v]
    return tuple(out)
