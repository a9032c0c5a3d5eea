"""Cost and effect of Monte-Carlo dropout (sc_segment_volume_mc) against the deterministic dense pass (sc_segment_volume).

Input: the synthetic 256^3 subject of bench.py (synthetic.make_t1 / make_atlas, seed 1234), device-resident, in two modes:
  full   every non-zero T1 voxel is a candidate, the box is their bounding box (bench.py's workload)
  crop   the registered-style prior mask dilated 10 times (test_scan's default crop mode) and its bounding box
Arms per mode: the deterministic call and T = 1, 8, 20 passes.  Every arm is warmed up; the arms then alternate for
--rounds rounds of --calls calls each, timed one by one with CUDA events.  Per arm: the median of the round means and their
max - min spread, launches per call and the per-class split of one profiled call (sc_set_option("profile", 1), a run of
its own).  Per mode: label agreement of the T = 20 mean with the deterministic labels and the mean entropy / mutual
information over the candidates.  The GPU name and power limit are read in the same run.

usage: python scripts/exp_mc_dropout.py [--rounds 3] [--calls 2] [--out profiles/r7_exp_mc_dropout.jsonl]
One JSON line per mode is printed and appended to --out."""
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
from cnn_cort import nets, synthetic  # noqa: E402
from cnn_cort._native import Context  # noqa: E402
from oracle import network as on  # noqa: E402

SIZE, SEED, SAMPLES, MC_SEED = 256, 1234, (1, 8, 20), 7


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    name, pl = [s.strip() for s in q.stdout.strip().split(",")][:2]
    return name, float(pl)


def main(args):
    if not torch.cuda.is_available():
        sys.exit("exp_mc_dropout.py measures on the GPU; no CUDA device found")
    torch.cuda.set_device(0)
    name, power = gpu_info()
    ctx = Context(0)
    ctx.load_weights(nets.pack_params(on.load_params(os.path.join(ROOT, "nets", "miccai2012_v1", "miccai2012_v1.pkl"))))
    shape = (SIZE,) * 3
    t1 = synthetic.make_t1(shape, SEED)
    nz = t1[np.nonzero(t1)]
    vol = torch.from_numpy(((t1 - nz.mean()) / nz.std()).astype(np.float32)).cuda()
    atlas_h = synthetic.make_atlas(shape, SEED)[0]
    atlas = torch.from_numpy(np.ascontiguousarray(atlas_h, dtype=np.float32)).cuda()
    masks = {"full": torch.from_numpy((t1 != 0).view(np.uint8)).cuda(),
             "crop": ctx.dilate_mask(torch.from_numpy(np.ascontiguousarray(synthetic.make_mask(atlas_h) != 0).view(np.uint8)).cuda(), 10)}
    del t1, atlas_h
    lab = torch.zeros(shape, dtype=torch.uint8, device="cuda")
    ent = torch.zeros(shape, dtype=torch.float32, device="cuda")
    mi = torch.zeros(shape, dtype=torch.float32, device="cuda")
    for mode, cand in masks.items():
        box, n_cand = ctx.mask_bbox(cand)
        arms = [("det", 0)] + [("mc%d" % T, T) for T in SAMPLES]

        def call(T):
            if T == 0:
                ctx.segment_volume(vol, atlas, box=box, cand_mask=cand, label_vol=lab)
            else:
                ctx.segment_volume_mc(vol, atlas, T, MC_SEED, box=box, cand_mask=cand, label_vol=lab, entropy_vol=ent, mi_vol=mi)

        res = {}
        for arm, T in arms:                                    # warm-up, launches per call
            call(T)
            torch.cuda.synchronize()
            n0 = ctx.counter("launches")
            call(T)
            torch.cuda.synchronize()
            res[arm] = {"samples": T, "launches_per_call": ctx.counter("launches") - n0, "round_means_ms": []}
        for _ in range(args.rounds):
            for arm, T in arms:
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.calls)]
                for a, b in ev:
                    a.record()
                    call(T)
                    b.record()
                torch.cuda.synchronize()
                res[arm]["round_means_ms"].append(float(np.mean([a.elapsed_time(b) for a, b in ev])))
        for arm, T in arms:
            m = res[arm]["round_means_ms"]
            res[arm]["median_ms"] = float(np.median(m))
            res[arm]["spread_ms"] = max(m) - min(m)
            res[arm]["vs_det"] = res[arm]["median_ms"] / float(np.median(res["det"]["round_means_ms"]))
        ctx.set_option("profile", 1)
        for arm, T in arms:
            ctx.profile_read()
            call(T)
            torch.cuda.synchronize()
            res[arm]["profile_ms"] = {k: round(v[0], 3) for k, v in ctx.profile_read().items()}
        ctx.set_option("profile", 0)
        sel = cand.bool()
        call(0)
        det = lab[sel].clone()
        call(SAMPLES[-1])
        torch.cuda.synchronize()
        line = {"exp": "mc_dropout", "gpu": name, "power_limit_w": power, "mode": mode, "shape": list(shape), "box": list(box),
                "candidates": n_cand, "rounds": args.rounds, "calls_per_round": args.calls, "mc_seed": MC_SEED, "arms": res,
                "label_agreement_T%d_vs_det" % SAMPLES[-1]: float((lab[sel] == det).float().mean()),
                "mean_entropy_T%d" % SAMPLES[-1]: float(ent[sel].double().mean()),
                "mean_mutual_info_T%d" % SAMPLES[-1]: float(mi[sel].double().mean())}
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "a") as f:
                f.write(json.dumps(line) + "\n")
    ctx.close()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--calls", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_exp_mc_dropout.jsonl"))
    main(ap.parse_args())
