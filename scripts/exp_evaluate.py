"""Device time of sc_evaluate_segmentation on a 256^3 label pair against the scipy oracle: prints ONE JSON line.

The pair is the synthetic subject's manual labels (cnn_cort.synthetic, seed 1234) as the reference and, as the
segmentation, the same structures grown by one voxel along x, with and without scattered false positives (1e-4 of the
voxels set to a random structure, which stretches every class box over the whole volume).  Spacing (1.0, 0.9, 1.2) mm.
Per pair: the median of --calls CUDA-event timed calls after warm-up, the "evaluate" profile class of one call, the
per-kernel device times of one call (torch.profiler), the oracle's host seconds (timed once) and whether all metrics agree.

usage: python scripts/exp_evaluate.py [--calls 30]
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "sub-cortical_segmentation_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402
from scipy import ndimage  # noqa: E402

from cnn_cort import _native, synthetic  # noqa: E402
from oracle import evaluate as oe  # noqa: E402

SPACING = (1.0, 0.9, 1.2)


def agree(rows, conf, want, wconf):
    ok = bool(np.array_equal(conf, wconf))
    for l in range(1, 15):
        g, w = rows[l - 1], want[l]
        ok &= all(int(g[f]) == w[f] for f in ("n_seg", "n_ref", "n_both")) and all(float(g[f]) == w[f] for f in ("vol_seg_mm3", "vol_ref_mm3"))
        for f in ("dice", "hd_mm", "hd95_mm", "assd_mm"):
            gv, wv = float(g[f]), float(w[f])
            ok &= (np.isnan(gv) and np.isnan(wv)) or abs(gv - wv) <= (1e-12 if f == "dice" else 1e-9 * wv + 1e-12)
    return bool(ok)


def main():
    calls = int(sys.argv[sys.argv.index("--calls") + 1]) if "--calls" in sys.argv else 30
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    gpu_name, power = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else (torch.cuda.get_device_name(0), "unknown")
    ctx = _native.Context(0)
    shape = (256, 256, 256)
    ref = synthetic.make_labels(synthetic.make_atlas(shape, 1234)[0])
    grown = ndimage.grey_dilation(np.where(ref == 15, 0, ref), size=(2, 1, 1))
    rng = np.random.RandomState(0)
    noisy = grown.copy()
    m = rng.rand(*shape) < 1e-4
    noisy[m] = rng.randint(1, 15, size=int(m.sum()))
    out = {"gpu": gpu_name, "power_limit": power, "shape": list(shape), "spacing": list(SPACING), "calls": calls, "pairs": {}}
    d_ref = torch.from_numpy(ref).cuda()
    for name, seg in (("clean", grown), ("false_positives", noisy)):
        d_seg = torch.from_numpy(seg).cuda()
        for _ in range(3):
            ctx.evaluate_segmentation(d_seg, d_ref, SPACING, confusion=True)
        times = []
        for _ in range(calls):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rows, conf = ctx.evaluate_segmentation(d_seg, d_ref, SPACING, confusion=True)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        ctx.set_option("profile", 1)
        l0 = ctx.counter("launches")
        ctx.evaluate_segmentation(d_seg, d_ref, SPACING)
        prof = ctx.profile_read()
        launches = ctx.counter("launches") - l0
        ctx.set_option("profile", 0)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as p:
            ctx.evaluate_segmentation(d_seg, d_ref, SPACING)
            torch.cuda.synchronize()
        kernels = {}
        for e in p.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            if t > 0:
                kernels[e.key] = {"ms": round(t / 1000.0, 4), "count": e.count}
        t0 = time.time()
        want, wconf = oe.evaluate(seg, ref, SPACING)
        host_s = time.time() - t0
        out["pairs"][name] = {
            "median_ms": float(np.median(times)), "min_ms": float(np.min(times)), "max_ms": float(np.max(times)),
            "profile_evaluate": {k: [round(v[0], 4), v[1]] for k, v in prof.items()}, "launches": launches,
            "kernels": kernels, "classes_with_distances": int(sum(int(r["n_seg"] > 0 and r["n_ref"] > 0) for r in rows)),
            "oracle_host_s": round(host_s, 2), "speedup_vs_oracle": round(host_s * 1000.0 / float(np.median(times)), 1),
            "agree": agree(rows, conf, want, wconf)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
