"""Cost and effect of running the network on a 1 mm grid ([model] resample_mm = 1.0) for scans of other voxel sizes.

1. Cost.  The synthetic 0.7 mm 320^3 volume of bench.py's volume_320_proba section (synthetic.make_t1 / make_atlas, seed 4321),
   segmented with base.segment_arrays on its native grid and with resample_mm = 1.0 (224^3 target grid), in two modes:
     full   every non-zero T1 voxel is a candidate
     crop   the registered-style prior mask (synthetic.make_mask), dilated 10 times on the grid the network runs on
   The priors and the mask are device-resident CUDA tensors; the T1 is a host array (segment_arrays uploads it) and the labels
   come back to the host, as in test_scan.  Every arm is warmed up; the arms then alternate for --rounds rounds of --calls calls,
   each timed with CUDA events.  Per arm: median of the round means, max - min spread, and the per-class split of one profiled
   call (a run of its own).  The resampling kernels are also timed alone (--reps launches between two events): the T1
   (1 channel) and the priors (15 channels) 320^3 -> 224^3, and the back-mapping 224^3 -> 320^3 with a native mask; their bytes
   are computed from the shapes (every element read once and written once per axis pass; the back-mapping reads the target
   probabilities and candidates once and the native mask, and writes the labels), over the kernel time.
2. Accuracy demo, reported and not asserted.  A 1 mm synthetic subject (synthetic.write_subject's volumes with the `contrast`
   table below, 160^3) is resampled to 0.75 mm (213^3; T1 cubic, priors linear, labels and mask nearest, scipy.ndimage.zoom).
   The 0.75 mm scan is segmented on its native grid and with resample_mm = 1.0 (crop mode); the mean Dice over the 14
   structures against the 0.75 mm labels is reported for both, beside the 1 mm original's Dice against its own labels.

The GPU name and power limit are read in the same run.
usage: python scripts/exp_resample.py [--rounds 3] [--calls 2] [--reps 10] [--out profiles/r9_exp_resample.jsonl]
One JSON line per measurement is printed and appended to --out."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "sub-cortical_segmentation_b200"))

import torch  # noqa: E402
from cnn_cort import base, nets, synthetic  # noqa: E402
from cnn_cort._native import Context  # noqa: E402
from oracle import network as on  # noqa: E402

SIZE, SPACING, SEED = 320, 0.7, 4321
CONTRAST = {l: 60.0 * (l % 5) - 90.0 for l in range(1, 15)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    name, pl = [s.strip() for s in q.stdout.strip().split(",")][:2]
    return name, float(pl)


def emit(line, out):
    print(json.dumps(line), flush=True)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "a") as f:
            f.write(json.dumps(line) + "\n")


def timed(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def cost(ctx, args, gpu):
    shape = (SIZE,) * 3
    spacing = (SPACING,) * 3
    t1 = synthetic.make_t1(shape, SEED)
    atlas_h = synthetic.make_atlas(shape, SEED)[0]
    atlas = torch.from_numpy(np.ascontiguousarray(atlas_h, dtype=np.float32)).cuda()
    mask = torch.from_numpy(synthetic.make_mask(atlas_h)).cuda()
    del atlas_h
    tshape, _ = base.resample_dims(shape, spacing, 1.0)
    for mode in ("full", "crop"):
        crop = mask if mode == "crop" else None
        arms = {"native": {}, "resample_1mm": {"spacing": spacing, "resample_mm": 1.0}}

        def call(kw):
            return base.segment_arrays(ctx, t1, atlas, crop_mask=crop, **kw)

        res = {}
        for arm, kw in arms.items():
            call(kw)
            n0 = ctx.counter("launches")
            _, _, n_cand = call(kw)
            res[arm] = {"launches_per_call": ctx.counter("launches") - n0, "candidates": n_cand, "round_means_ms": []}
        for _ in range(args.rounds):
            for arm, kw in arms.items():
                ms = []
                for _ in range(args.calls):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    call(kw)
                    b.record()
                    torch.cuda.synchronize()
                    ms.append(a.elapsed_time(b))
                res[arm]["round_means_ms"].append(float(np.mean(ms)))
        for arm in arms:
            m = res[arm]["round_means_ms"]
            res[arm]["median_ms"] = float(np.median(m))
            res[arm]["spread_ms"] = max(m) - min(m)
        ctx.set_option("profile", 1)
        for arm, kw in arms.items():
            ctx.profile_read()
            call(kw)
            res[arm]["profile_ms"] = {k: round(v[0], 3) for k, v in ctx.profile_read().items()}
        ctx.set_option("profile", 0)
        lab_native = call({})[0].copy()
        lab_rs = call(arms["resample_1mm"])[0].copy()
        sel = t1 != 0 if crop is None else lab_native > 0
        emit({"exp": "resample_cost", "gpu": gpu[0], "power_limit_w": gpu[1], "mode": mode, "shape": list(shape),
              "spacing_mm": SPACING, "target_shape": list(tshape), "rounds": args.rounds, "calls_per_round": args.calls,
              "arms": res, "speedup": res["native"]["median_ms"] / res["resample_1mm"]["median_ms"],
              "label_agreement_native_vs_1mm": float((lab_native[sel] == lab_rs[sel]).mean())}, args.out)
    # the kernels alone
    d_t1 = torch.from_numpy(t1).cuda()
    out1 = torch.empty(tshape, dtype=torch.float32, device="cuda")
    out15 = torch.empty(tshape + (15,), dtype=torch.float32, device="cuda")
    kernels = {}

    def passes_bytes(ch):
        b, cur = 0, list(shape)
        for a in range(3):
            n_in = int(np.prod(cur)) * ch
            cur[a] = tshape[a]
            b += 4 * (n_in + int(np.prod(cur)) * ch)
        return b

    for key, src, dst, ch in (("resample_t1", d_t1, out1, 1), ("resample_priors", atlas, out15, 15)):
        ms = timed(lambda: ctx.resample_volume(src, tshape, out=dst), args.reps)
        kernels[key] = {"ms": ms, "bytes": passes_bytes(ch), "gb_per_s": passes_bytes(ch) / ms / 1e6}
    proba = out15
    cand = torch.ones(tshape, dtype=torch.uint8, device="cuda")
    nmask = torch.ones(shape, dtype=torch.uint8, device="cuda")
    lab = torch.zeros(shape, dtype=torch.uint8, device="cuda")
    ms = timed(lambda: ctx.map_proba_back(proba, cand, shape, native_mask=nmask, label_out=lab), args.reps)
    nb = int(np.prod(tshape)) * (60 + 1) + int(np.prod(shape)) * 2
    kernels["map_proba_back"] = {"ms": ms, "bytes": nb, "gb_per_s": nb / ms / 1e6}
    emit({"exp": "resample_kernels", "gpu": gpu[0], "power_limit_w": gpu[1], "shape": list(shape), "target_shape": list(tshape),
          "reps": args.reps, "kernels": kernels}, args.out)


def accuracy(ctx, args, gpu):
    from scipy import ndimage
    shape = (160, 160, 160)
    atlas, _, _ = synthetic.make_atlas(shape, 99)
    labels = synthetic.make_labels(atlas)
    table = np.zeros(16, np.float32)
    for l, v in CONTRAST.items():
        table[l] = v
    t1 = (synthetic.make_t1(shape, 99) + table[labels]).astype(np.float32)
    mask = synthetic.make_mask(atlas)
    z = 1.0 / 0.75
    t1_f = np.maximum(ndimage.zoom(t1, z, order=3), 1.0).astype(np.float32)
    atlas_f = np.clip(ndimage.zoom(atlas, (z, z, z, 1), order=1), 0, 1).astype(np.float32)
    labels_f = ndimage.zoom(labels, z, order=0)
    mask_f = ndimage.zoom(mask, z, order=0)

    def dice(seg, ref):
        m, _ = base.evaluate_segmentation(seg, ref, device=ctx.device)
        d = [m[l]['dice'] for l in range(1, 15) if not np.isnan(m[l]['dice'])]
        return float(np.mean(d)), {l: m[l]['dice'] for l in range(1, 15)}

    res = {}
    res["1mm_original"] = dice(base.segment_arrays(ctx, t1, atlas, crop_mask=mask)[0].copy(), labels)
    res["0.75mm_native_grid"] = dice(base.segment_arrays(ctx, t1_f, atlas_f, crop_mask=mask_f)[0].copy(), labels_f)
    res["0.75mm_resample_1mm"] = dice(base.segment_arrays(ctx, t1_f, atlas_f, crop_mask=mask_f, spacing=(0.75,) * 3,
                                                          resample_mm=1.0)[0].copy(), labels_f)
    emit({"exp": "resample_accuracy", "gpu": gpu[0], "power_limit_w": gpu[1], "shape_1mm": list(shape),
          "shape_0.75mm": list(t1_f.shape), "contrast": CONTRAST, "mode": "crop",
          "mean_dice": {k: v[0] for k, v in res.items()}, "dice": {k: v[1] for k, v in res.items()}}, args.out)


def main(args):
    if not torch.cuda.is_available():
        sys.exit("exp_resample.py measures on the GPU; no CUDA device found")
    torch.cuda.set_device(0)
    gpu = gpu_info()
    ctx = Context(0)
    ctx.load_weights(nets.pack_params(on.load_params(os.path.join(ROOT, "nets", "miccai2012_v1", "miccai2012_v1.pkl"))))
    cost(ctx, args, gpu)
    accuracy(ctx, args, gpu)
    ctx.close()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--calls", type=int, default=2)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r9_exp_resample.jsonl"))
    main(ap.parse_args())
