#!/usr/bin/env python
"""Generate the committed golden fixtures from a checkout of the original project:

    python tests/golden/make_golden.py /path/to/original/project

Nothing in the test-suite reads the original project -- only this script does, and its
outputs are committed.  To keep each fixture under 1 MB, every voxel of a stored volume
that no patch around a stored centre reads is set to zero (a patch is a copy of the
voxels it reads, so the stored patches are still the original's output for the stored
volume).

gather_golden.npz  -- produced by EXECUTING the reference's own source text of
    ``get_patches`` (cnn_cort/base.py:272-308), ``get_mask_voxels`` (:310-331) and
    ``generate_training_set`` (:53-117).  The reference is Python 2; the function text
    is sliced out of base.py and three mechanical token fixes are applied so that it
    parses/runs on Python 3 + numpy 2 (nothing else is altered):
      1. ``idx/2`` and ``.shape[k] / 2``  ->  ``//``           (py2 integer division)
      2. ``map(add, ...)``               ->  ``list(map(...))`` (py2 map returns a list)
      3. ``new_image[idx]`` (list of slices) -> ``new_image[tuple(idx)]`` (numpy>=1.23)
      4. the two-line ``print "..."`` debug block in generate_training_set is dropped.
    The patch arrays of generate_training_set's output are the B_x_* patches (unshuffled)
    and those rows in the order T_shuf_perm (shuffled); tests/conftest.py rebuilds them.
forward_golden.npz -- oracle/network.py (fp64 and fp32) on the committed weights and
    seeded inputs: a regression pin of the restatement (the Theano stack is absent, so
    this part is NOT reference output; see oracle/__init__.py "parity unpinned").
"""
import os
import re
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
def read_mask(shape, centres):
    """the voxels that the axial, coronal and saggital (32, 32) patches around ``centres`` read"""
    m = np.zeros(shape, bool)
    for x, y, z in np.asarray(centres).tolist():
        sx, sy, sz = (slice(max(c - 16, 0), c + 16) for c in (x, y, z))
        m[sx, sy, z] = m[sx, y, sz] = m[x, sy, sz] = True
    return m


def restrict(vol, centres):
    vol = vol.copy()
    vol[~read_mask(vol.shape, centres)] = 0
    return vol


def shrink_gather(out):
    """zero the unread voxels, store the shuffle of generate_training_set as a permutation"""
    out = dict(out)
    out["A_vol"] = restrict(out["A_vol"], out["A_centers"])
    out["B_vol"] = restrict(out["B_vol"], out["B_sel"])
    rows = [r.tobytes() for r in out["T_plain_xa"]]
    perm = np.array([rows.index(r.tobytes()) for r in out["T_shuf_xa"]], dtype=np.int64)
    for k, mode in (("xa", "axial"), ("xc", "coronal"), ("xs", "saggital")):
        plain, shuf = out.pop("T_plain_" + k), out.pop("T_shuf_" + k)
        assert plain.dtype == out["B_x_" + mode].dtype and np.array_equal(plain, out["B_x_" + mode][:, None]), k
        assert np.array_equal(shuf, plain[perm]), k
    assert np.array_equal(out["T_shuf_at"], out["T_plain_at"][perm]) and np.array_equal(out["T_shuf_y"], out["T_plain_y"][perm])
    out["T_shuf_perm"] = perm
    return out


def shrink_forward(out):
    return dict(out, vol=restrict(out["vol"], out["centers"]))


def _slice_def(src, name):
    m = re.search(r"^def %s\(.*?(?=^def |\Z)" % name, src, flags=re.S | re.M)
    return m.group(0)


def reference_functions(ref_root):
    src = open(os.path.join(ref_root, "cnn_cort", "base.py")).read()
    gp = _slice_def(src, "get_patches")
    gp = gp.replace("idx/2", "idx//2")
    gp = gp.replace("[map(add, center, patch_half) for center in centers]",
                    "[list(map(add, center, patch_half)) for center in centers]")
    gp = gp.replace("np.squeeze(new_image[idx])", "np.squeeze(new_image[tuple(idx)])")
    gm = _slice_def(src, "get_mask_voxels")
    gt = _slice_def(src, "generate_training_set")
    gt = gt.replace("y_train.shape[1] / 2, y_train.shape[2] / 2", "y_train.shape[1] // 2, y_train.shape[2] // 2")
    gt = "\n".join(l for l in gt.split("\n") if not l.strip().startswith("print "))
    gt = gt.replace("    if options['debug'] == 'True':\n", "    if options['debug'] == 'True':\n        pass\n")
    ns = {"np": np}
    exec("from operator import add\n" + gp + "\n" + gm + "\n" + gt, ns)
    return ns["get_patches"], ns["get_mask_voxels"], ns["generate_training_set"]


def make_gather(ref_root):
    get_patches, get_mask_voxels, generate_training_set = reference_functions(ref_root)
    rng = np.random.RandomState(20121)
    out = {}
    # case A: non-cubic volume smaller than a patch in one axis, float64 (test-path dtype)
    volA = rng.randn(40, 36, 20)
    cenA = [(0, 0, 0), (39, 35, 19), (16, 16, 16), (15, 17, 3), (39, 0, 10), (0, 35, 0), (20, 18, 19)]
    cenA += [tuple(int(v) for v in c) for c in
             np.stack([rng.randint(0, 40, 25), rng.randint(0, 36, 25), rng.randint(0, 20, 25)], 1)]
    out["A_vol"] = volA
    out["A_centers"] = np.array(cenA, dtype=np.int64)
    for mode in ("axial", "coronal", "saggital"):
        out["A_" + mode] = np.array(get_patches(volA, cenA, [32, 32], mode=mode))
    # case B: float32 volume (train-path dtype) and a uint8 label volume, 48^3
    volB = rng.randn(48, 48, 48).astype(np.float32)
    labB = np.zeros((48, 48, 48), np.uint8)
    labB[20:28, 18:30, 22:27] = rng.randint(1, 15, size=(8, 12, 5))
    labB[18:20, 18:30, 22:27] = 15
    labB[28:30, 18:30, 22:27] = 15
    maskB = np.logical_and(labB > 0, labB < 15)
    cenB = get_mask_voxels(maskB)
    out["B_vol"] = volB
    out["B_lab"] = labB
    out["B_pos_centers"] = np.array(cenB, dtype=np.int64)
    sel = cenB[::17]
    out["B_sel"] = np.array(sel, dtype=np.int64)
    for mode in ("axial", "coronal", "saggital"):
        out["B_x_" + mode] = np.array(get_patches(volB, sel, (32, 32), mode=mode))
        out["B_y_" + mode] = np.array(get_patches(labB, sel, (32, 32), mode=mode))
    # mask ordering on an irregular mask
    maskC = rng.rand(9, 7, 11) > 0.6
    out["C_mask"] = maskC
    out["C_vox"] = np.array(get_mask_voxels(maskC), dtype=np.int64)
    # generate_training_set (no shuffle + fixed-seed shuffle)
    xa = [out["B_x_axial"][:10], out["B_x_axial"][10:]]
    xc = [out["B_x_coronal"][:10], out["B_x_coronal"][10:]]
    xs = [out["B_x_saggital"][:10], out["B_x_saggital"][10:]]
    at = [rng.rand(10, 15), rng.rand(len(sel) - 10, 15)]
    ya = [out["B_y_axial"][:10], out["B_y_axial"][10:]]
    out["T_atlas0"], out["T_atlas1"] = at
    r = generate_training_set(xa, xc, xs, at, ya, {"debug": "False"}, randomize=False)
    for k, v in zip(("xa", "xc", "xs", "at", "y"), r):
        out["T_plain_" + k] = v
    np.random.seed(77)  # the reference draws its seed from the global stream (:93)
    r = generate_training_set(xa, xc, xs, at, ya, {"debug": "False"}, randomize=True)
    for k, v in zip(("xa", "xc", "xs", "at", "y"), r):
        out["T_shuf_" + k] = v
    out = shrink_gather(out)
    np.savez_compressed(os.path.join(HERE, "gather_golden.npz"), **out)
    print("gather_golden.npz:", {k: v.shape for k, v in out.items()})


def make_forward():
    import torch
    from oracle import network as net
    P = net.load_params(os.path.join(ROOT, "nets", "miccai2012_v1", "miccai2012_v1.pkl"))
    rng = np.random.RandomState(4242)
    n = 48
    from scipy.ndimage import gaussian_filter
    vol = gaussian_filter(rng.randn(72, 72, 72), 3)
    vol = (vol / vol.std() + 0.15 * rng.randn(72, 72, 72)).astype(np.float32)
    from oracle import gather
    cen = np.stack([rng.randint(0, 72, n) for _ in range(3)], 1)
    cen[0] = (0, 0, 0)
    cen[1] = (71, 71, 71)
    x1, x2, x3 = (gather.get_patches(vol, cen, (32, 32), m).astype(np.float32)[:, None] for m in gather.VIEWS)
    at = rng.rand(n, 15).astype(np.float32) ** 4
    at /= at.sum(1, keepdims=True)
    at[5] = 0
    at[5, 14] = 1
    p64 = net.forward(P, x1, x2, x3, at, dtype=torch.float64)
    p32 = net.forward(P, x1, x2, x3, at, dtype=torch.float32)
    np.savez_compressed(os.path.join(HERE, "forward_golden.npz"), **shrink_forward(dict(
        vol=vol, centers=cen.astype(np.int64), atlas=at, proba64=p64, proba32=p32)))
    print("forward_golden.npz: max|p64-p32| =", np.abs(p64 - p32).max(), "labels", np.argmax(p64, 1)[:16])


if __name__ == "__main__":
    make_gather(sys.argv[1])
    make_forward()
