"""Training data path: materialised patch arrays vs device-resident scans.

    python scripts/exp_train_scans.py [--ks 2,8] [--shape 256] [--reps 2] [--batch 1024]

Writes max(K) synthetic subjects with labels (cnn_cort.synthetic) to a temporary directory, then for every K runs two
arms, each in a child process of its own, alternately, --reps times each:
  arrays  load_data + generate_training_set + Net.fit on the arrays
  scans   load_scan_training_set + Net.fit on the scan set
Same seeds, one epoch.  One JSON line per run on stdout: samples, set-up seconds, peak host RSS of the child
(ru_maxrss), device bytes of the training set, epoch seconds, and, from a second epoch with per-kernel profiling on
(kernel-by-kernel launches: the profiler turns the training step's CUDA graph off), the total and per-step time of
the gather kernel class next to the training step's kernels.  The GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import random
import resource
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "sub-cortical_segmentation_b200")]


def gpu_info():
    import torch
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or "not read"
    except (OSError, subprocess.SubprocessError):
        power = "not read"
    return {"gpu": torch.cuda.get_device_name(0), "power_limit": power}


def child(arm, data, batch):
    import numpy as np
    import torch
    from cnn_cort import base, nets
    options = {'train_folder': data, 't1_name': 'T1.nii.gz', 'roi_name': 'gt_15_classes.nii.gz', 'patch_size': [32, 32],
               'debug': 'False', 'device': 0, 'mode': 'cuda0', 'load_weights': 'False', 'net_verbose': 0,
               'train_split': 0.25, 'max_epochs': 1, 'patience': 20, 'batch_size': batch, 'seed': 1}
    torch.cuda.set_device(0)
    random.seed(1)
    np.random.seed(1)
    t0 = time.time()
    if arm == "arrays":
        x_axial, x_cor, x_sag, y_axial, x_atlas, _ = base.load_data(options)
        del _
        xa, xc, xs, xat, y = base.generate_training_set(x_axial, x_cor, x_sag, x_atlas, y_axial, options)
        del x_axial, x_cor, x_sag, y_axial, x_atlas
        X = {'in1': xa, 'in2': xc, 'in3': xs, 'in4': xat}
        fit_args = (X, y)
        n = len(y)
        dev_bytes = sum(a.nbytes for a in (xa, xc, xs, xat, y))      # what fit holds on the device (resident case)
    else:
        scans = base.load_scan_training_set(options)
        fit_args = (scans,)
        n = len(scans)
        dev_bytes = scans.device_bytes()
    torch.cuda.synchronize()
    setup_s = time.time() - t0
    net = nets.Net(options, None, None, seed=1)
    t1 = time.time()
    net.fit(*fit_args, epochs=1)
    torch.cuda.synchronize()
    fit_s = time.time() - t1
    epoch_s = net.train_history_[-1]['dur']
    ctx = net.ctx
    ctx.set_option("profile", 1)
    ctx.profile_read()
    net.fit(*fit_args, epochs=1)
    prof = ctx.profile_read()
    ctx.set_option("profile", 0)
    tr, va = net.train_split.indices(fit_args[-1] if arm == "arrays" else scans.y)
    steps = -(-len(tr) // batch)
    g_ms, g_launches = prof.get("gather", (0.0, 0))
    step_ms = sum(prof.get(k, (0.0, 0))[0] for k in ("train_fwd", "train_bwd", "adam"))
    out = {"arm": arm, "subjects": len([d for d in os.listdir(data) if os.path.isdir(os.path.join(data, d))]),
           "samples": n, "batch": batch, "setup_s": round(setup_s, 2),
           "peak_rss_mb": round(resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1024.0, 1),
           "device_set_bytes": int(dev_bytes), "epoch_s": round(epoch_s, 3), "fit_s": round(fit_s, 3),
           "train_steps": steps, "gather_ms_total": round(g_ms, 3), "gather_launches": g_launches,
           "gather_ms_per_batch": round(g_ms / max(1, g_launches), 4) if g_launches else None,
           "train_kernels_ms_per_step": round(step_ms / steps, 4),
           "final_train_loss": net.train_history_[-1]['train_loss']}
    if g_launches:
        out["gather_share_of_step"] = round((g_ms / g_launches) / (g_ms / g_launches + step_ms / steps), 4)
    out.update(gpu_info())
    print(json.dumps(out), flush=True)


def _write(args):
    from cnn_cort import synthetic
    root, i, shape = args
    synthetic.write_subject(root, "s%02d" % i, shape=(shape,) * 3, seed=100 + i, with_labels=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="2,8")
    ap.add_argument("--shape", type=int, default=256)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--child", choices=("arrays", "scans"))
    ap.add_argument("--data")
    a = ap.parse_args()
    if a.child:
        return child(a.child, a.data, a.batch)
    ks = [int(k) for k in a.ks.split(",")]
    tmp = tempfile.mkdtemp(prefix="exp_train_scans_")
    try:
        subj = os.path.join(tmp, "subjects")
        t0 = time.time()
        from concurrent.futures import ProcessPoolExecutor
        with ProcessPoolExecutor(min(max(ks), os.cpu_count() or 1)) as pool:
            list(pool.map(_write, [(subj, i, a.shape) for i in range(max(ks))]))
        sys.stderr.write("wrote %d subjects of %d^3 in %.0f s\n" % (max(ks), a.shape, time.time() - t0))
        for k in ks:
            data = os.path.join(tmp, "k%d" % k)
            os.makedirs(data)
            for i in range(k):
                os.symlink(os.path.join(subj, "s%02d" % i), os.path.join(data, "s%02d" % i))
            for rep in range(a.reps):
                for arm in ("arrays", "scans"):
                    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", arm, "--data", data,
                                        "--batch", str(a.batch)], capture_output=True, text=True)
                    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
                    if r.returncode != 0 or not lines:
                        sys.stderr.write(r.stdout[-2000:] + r.stderr[-4000:])
                        raise SystemExit("arm %s (K=%d) failed" % (arm, k))
                    d = json.loads(lines[-1])
                    d["rep"] = rep
                    print(json.dumps(d), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
