"""A/B of two library builds on the bench.py workload (dense 256^3 pass, every voxel a candidate): the strip-sweep
convolutions (conv2 .. conv5) of a baseline tree against this tree.  Each tree has one lib/ path, so every (round, arm)
runs in a child process of its own; the arms alternate for --rounds rounds so that clock and power drift hit both alike.

Each child records the GPU name and power limit, warms up, times --passes passes one by one with CUDA events, takes the
per-class profile split of one more pass (sc_set_option("profile", 1)), the per-role cycle counters of each sweep class
(sc_set_option("tc_timing", cls), one more pass each) and writes the labels of its last timed pass at the voxel sample
of `bench.py --dump-outputs`.  The parent prints and writes (JSON lines) each arm's per-round means, their median and
max - min spread, the mean profile split with the conv2 .. conv5 sum, the counters, and the label agreement of the arms.

usage: python scripts/exp_sweep_stack.py --baseline DIR [--rounds 6] [--passes 10] [--out FILE.jsonl]
(DIR: a built checkout of the baseline commit, e.g. a git worktree)"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZE, SEED, DUMP_VOXELS = 256, 1234, 1 << 22         # bench.py: synthetic_volume(256, 1234), DUMP_VOXELS
SWEEP_CLASSES = [(5, "conv2"), (6, "conv3"), (7, "conv4"), (8, "conv5")]   # profile classes of the sweeps


def child(root, data, out_labels):
    sys.path[:0] = [root, os.path.join(root, "sub-cortical_segmentation_b200")]
    import pickle
    import torch
    from cnn_cort import _native, nets
    torch.cuda.set_device(0)
    ctx = _native.Context(0)
    with open(os.path.join(root, "nets", "miccai2012_v1", "miccai2012_v1.pkl"), "rb") as f:
        ctx.load_weights(nets.pack_params(pickle.load(f, encoding="latin1")))
    vol = torch.from_numpy(np.load(os.path.join(data, "norm.npy"))).cuda()
    atlas = torch.from_numpy(np.load(os.path.join(data, "atlas.npy"))).cuda()
    mask = torch.from_numpy(np.load(os.path.join(data, "mask.npy"))).cuda()
    lab = torch.zeros(vol.shape, dtype=torch.uint8, device="cuda")

    def step():
        ctx.segment_volume(vol, atlas, cand_mask=mask, label_vol=lab)

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.passes)]
    l0 = ctx.counter("launches")
    for e0, e1 in ev:
        e0.record()
        step()
        e1.record()
    torch.cuda.synchronize()
    launches = (ctx.counter("launches") - l0) / args.passes
    ms = [e0.elapsed_time(e1) for e0, e1 in ev]
    idx = np.load(os.path.join(data, "label_index.npy"))
    np.save(out_labels, lab.view(-1).cpu().numpy()[idx])
    ctx.set_option("profile", 1)
    ctx.profile_read()
    step()
    torch.cuda.synchronize()
    prof = {k: v[0] for k, v in ctx.profile_read().items()}
    ctx.set_option("profile", 0)
    # per-role cycle counters, averaged over sampled CTAs and given per output row of the sweep: MMA-warp busy (total minus
    # its waits for a ring row and for a free accumulator) and epilogue busy (total minus its waits for a full accumulator).
    # A kernel without counters leaves the buffer as the previous class wrote it: such a class is reported as null.
    timing, prev = {}, None
    for cls, nm in SWEEP_CLASSES:
        ctx.set_option("tc_timing", cls)
        step()
        torch.cuda.synchronize()
        v = np.array([[ctx.counter("tc_timing:%d" % (c * 8 + k)) for k in range(8)] for c in range(0, 74, 18)], dtype=np.float64)
        m = v.mean(0)
        timing[nm] = None if (prev is not None and np.array_equal(v, prev)) or m[7] == 0 else {
            "rows_per_cta": m[7], "mma_busy_clk_per_row": (m[4] - m[2] - m[3]) / m[7], "mma_wait_ring_clk_per_row": m[2] / m[7],
            "mma_wait_acc_clk_per_row": m[3] / m[7], "epi_busy_clk_per_row": (m[6] - m[5]) / m[7], "epi_wait_clk_per_row": m[5] / m[7]}
        prev = v
    ctx.set_option("tc_timing", -1)
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    print(json.dumps({"gpu": torch.cuda.get_device_name(0), "power_limit": q.stdout.strip() or None, "ms": ms,
                      "launches_per_pass": launches, "profile_ms": prof, "tc_timing": timing}))


def main():
    data = tempfile.mkdtemp(prefix="exp_sweep_stack_")
    sys.path[:0] = [ROOT, os.path.join(ROOT, "sub-cortical_segmentation_b200")]
    from cnn_cort import synthetic
    shape = (SIZE,) * 3
    t1 = synthetic.make_t1(shape, SEED)
    nz = t1[np.nonzero(t1)]
    np.save(os.path.join(data, "norm.npy"), ((t1 - nz.mean()) / nz.std()).astype(np.float32))
    np.save(os.path.join(data, "atlas.npy"), synthetic.make_atlas(shape, SEED)[0])
    np.save(os.path.join(data, "mask.npy"), (t1 != 0).view(np.uint8))
    n = t1.size
    np.save(os.path.join(data, "label_index.npy"), np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_VOXELS), replace=False)))
    arms = [("baseline", os.path.abspath(args.baseline)), ("this", ROOT)]
    res = {a: [] for a, _ in arms}
    labels = {}
    for r in range(args.rounds):
        for arm, root in arms:
            lf = os.path.join(data, "labels_%s_%d.npy" % (arm, r))
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", root, "--data", data, "--labels", lf,
                                "--passes", str(args.passes)], capture_output=True, text=True)
            if p.returncode != 0:
                sys.exit("child %s round %d failed:\n%s" % (arm, r, p.stderr[-3000:]))
            d = json.loads(p.stdout.strip().splitlines()[-1])
            d["round"], d["arm"], d["mean_ms"] = r, arm, float(np.mean(d["ms"]))
            res[arm].append(d)
            labels.setdefault(arm, np.load(lf))
            print("round %d %-8s mean %.2f ms (min %.2f max %.2f)  %s %s" % (r, arm, d["mean_ms"], min(d["ms"]), max(d["ms"]),
                                                                           d["gpu"], d["power_limit"]), flush=True)
    summary = {"gpu": res["this"][0]["gpu"], "power_limit": res["this"][0]["power_limit"], "rounds": args.rounds, "passes": args.passes}
    for arm, _ in arms:
        m = [d["mean_ms"] for d in res[arm]]
        classes = sorted({k for d in res[arm] for k in d["profile_ms"]})
        summary[arm] = {"round_means_ms": m, "median_ms": float(np.median(m)), "spread_ms": max(m) - min(m),
                        "launches_per_pass": res[arm][0]["launches_per_pass"],
                        "profile_ms": {k: float(np.mean([d["profile_ms"].get(k, 0.0) for d in res[arm]])) for k in classes},
                        "tc_timing_round0": res[arm][0]["tc_timing"]}
        summary[arm]["sweeps_ms"] = sum(summary[arm]["profile_ms"].get(nm, 0.0) for _, nm in SWEEP_CLASSES)
    summary["gain_ms"] = summary["baseline"]["median_ms"] - summary["this"]["median_ms"]
    summary["sweeps_ratio"] = summary["this"]["sweeps_ms"] / summary["baseline"]["sweeps_ms"]
    shutil.rmtree(data)
    same = int((labels["baseline"] == labels["this"]).sum())
    summary["labels"] = {"sampled": int(labels["this"].size), "equal": same, "differ": int(labels["this"].size) - same,
                         "agreement": same / labels["this"].size}
    print(json.dumps(summary, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            for arm, _ in arms:
                for d in res[arm]:
                    f.write(json.dumps(d) + "\n")
            f.write(json.dumps(summary) + "\n")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline", help="root of the built baseline tree")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--passes", type=int, default=10)
    ap.add_argument("--out")
    ap.add_argument("--child")
    ap.add_argument("--data")
    ap.add_argument("--labels")
    args = ap.parse_args()
    if args.child:
        child(args.child, args.data, args.labels)
    else:
        if not args.baseline:
            ap.error("--baseline is required")
        main()
