"""Cost and effect of fine-tuning the head with a frozen trunk (Net.fine_tune) against full training (Net.fit).

Arms, each printed as one JSON line with the GPU name and power limit read in the same run:
  features  sc_trunk_features over the training set of 2 synthetic 256^3 subjects (synthetic.write_subject, labels on):
            samples/s of the table build (gather of the patches + trunk) and of the trunk alone, and the table's device bytes
  step      head step (sc_head_train_forward_backward on rows of the table) against the full step (sc_train_forward_backward on
            the gathered patches) at batch 256 and 1 024: CUDA events around --steps graph-launched steps per round after a
            warm-up, the two arms alternated for --rounds rounds in this process; median of the rounds and the spread
  epoch     one epoch of fine_tune against one epoch of fit on the same set (history 'dur')
  adapt     source = the committed weights, target = synthetic subjects with a per-label contrast table: mean Dice
            (evaluate_segmentation) on a held-out target subject for the starting weights, after fine_tune on ONE labelled
            target subject for --epochs epochs, and after fit for the same epochs.  Reported, not asserted.

usage: python scripts/exp_fine_tune.py [--rounds 3] [--steps 200] [--epochs 5] [--out profiles/r8_exp_fine_tune.jsonl]"""
import argparse
import json
import os
import random
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "sub-cortical_segmentation_b200"))

import torch  # noqa: E402
from cnn_cort import base, nets, nifti, synthetic  # noqa: E402

WEIGHTS = os.path.join(ROOT, "nets", "miccai2012_v1", "miccai2012_v1.pkl")
# target domain: per-label mean intensities added inside the structures (T1 units; the synthetic T1 is ~600 +- 150)
CONTRAST = {l: 60.0 * (((l * 5) % 7) - 3) for l in range(1, 16)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    name, pl = [s.strip() for s in q.stdout.strip().split(",")][:2]
    return name, float(pl)


def options(root, name, **kw):
    o = {'train_folder': root, 't1_name': 'T1.nii.gz', 'roi_name': 'gt_15_classes.nii.gz', 'patch_size': [32, 32],
         'debug': 'False', 'device': 0, 'experiment': name, 'mode': 'cuda0', 'load_weights': 'False', 'net_verbose': 0,
         'train_split': 0.25, 'max_epochs': 1, 'patience': 1000, 'batch_size': 128, 'seed': 1}
    o.update(kw)
    return o


def scan_set(root, seeds, shape, contrast=None):
    for i, s in enumerate(seeds):
        synthetic.write_subject(root, "s%02d" % i, shape=shape, seed=s, with_labels=True, contrast=contrast)
    random.seed(1)
    np.random.seed(1)
    return base.load_scan_training_set(options(root, "x"))


def net_from(weights_dir, name, **kw):
    net = nets.build_model(weights_dir, options("", name, **kw))
    net.load_params_from(WEIGHTS)
    return net


def events_ms(fn, k):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(k):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / k


def arm_features(net, S, gpu):
    ctx, n = net.ctx, len(S)
    torch.cuda.synchronize()
    t0 = time.time()
    feats, _, _, _ = net._feature_table(S, None, torch.device('cuda', 0))
    torch.cuda.synchronize()
    build_s = time.time() - t0
    chunk, trunk_ms = 16384, 0.0
    for s in range(0, n, chunk):
        in1, in2, in3, _, _ = S.gather(np.arange(s, min(n, s + chunk)), ctx=ctx)
        trunk_ms += events_ms(lambda: ctx.trunk_features(in1, in2, in3, out=feats[s:s + len(in1)]), 1)
    return dict(arm="features", gpu=gpu[0], power_limit_w=gpu[1], samples=n, table_bytes=feats.numel() * 4,
                build_s=round(build_s, 3), build_samples_per_s=round(n / build_s), trunk_ms=round(trunk_ms, 1),
                trunk_samples_per_s=round(n / (trunk_ms / 1e3))), feats


def arm_step(net, S, feats, gpu, rounds, steps):
    ctx = net.ctx
    out = []
    for bs in (256, 1024):
        idx = torch.from_numpy(np.random.RandomState(bs).permutation(len(S))[:bs].astype(np.int64)).cuda()
        batch = S.gather(idx, ctx=ctx)
        loss = torch.zeros(1, device='cuda')
        full = lambda: ctx.train_forward_backward(*batch, seed=3, loss_out=loss)
        head = lambda: ctx.head_train_forward_backward(feats, S.atlas, S.labels, idx=idx, seed=3, loss_out=loss)
        for fn in (full, head):
            events_ms(fn, 20)
        res = {"full": [], "head": []}
        for _ in range(rounds):
            for name, fn in (("full", full), ("head", head)):
                res[name].append(events_ms(fn, steps))
        line = dict(arm="step", gpu=gpu[0], power_limit_w=gpu[1], batch=bs, steps_per_round=steps, rounds=rounds)
        for name, v in res.items():
            line[name + "_ms"] = round(float(np.median(v)), 4)
            line[name + "_spread_ms"] = round(float(max(v) - min(v)), 4)
        line["head_over_full"] = round(line["head_ms"] / line["full_ms"], 4)
        out.append(line)
    return out


def arm_epoch(S, gpu, tmp):
    a = net_from(tmp, "ep_ft")
    torch.cuda.synchronize()
    t0 = time.time()
    a.fine_tune(S, epochs=1)
    torch.cuda.synchronize()
    ft_total = time.time() - t0
    b = net_from(tmp, "ep_fit")
    b.fit(S, epochs=1)
    return dict(arm="epoch", gpu=gpu[0], power_limit_w=gpu[1], samples=len(S), batch=128,
                fine_tune_epoch_s=round(a.train_history_[-1]['dur'], 3), fine_tune_total_s=round(ft_total, 3),
                fit_epoch_s=round(b.train_history_[-1]['dur'], 3))


def mean_dice(net, subj_dir):
    t1 = nifti.load(os.path.join(subj_dir, "T1.nii.gz")).get_data()
    atlas = nifti.load(os.path.join(subj_dir, "tmp", "MNI_sub_probabilities.nii.gz")).get_data()
    mask = nifti.load(os.path.join(subj_dir, "tmp", "MNI_subcortical_mask.nii.gz")).get_data()
    ref = nifti.load(os.path.join(subj_dir, "gt_15_classes.nii.gz")).get_data()
    lab, _, _ = base.segment_arrays(net.ctx, t1, atlas, crop_mask=mask)
    m, _ = base.evaluate_segmentation(lab.copy(), ref)
    d = [v['dice'] for v in m.values() if v['dice'] == v['dice']]
    return float(np.mean(d))


def arm_adapt(gpu, tmp, epochs, shape):
    train_root, test_root = os.path.join(tmp, "target_train"), os.path.join(tmp, "target_test")
    S = scan_set(train_root, [41], shape, CONTRAST)                    # ONE labelled target subject
    synthetic.write_subject(test_root, "held_out", shape=shape, seed=42, with_labels=True, contrast=CONTRAST)
    held = os.path.join(test_root, "held_out")
    src = net_from(tmp, "adapt_src")
    start = mean_dice(src, held)
    ft = net_from(tmp, "adapt_ft")
    ft.fine_tune(S, epochs=epochs)
    ft_dice = mean_dice(ft, held)
    fit = net_from(tmp, "adapt_fit")
    fit.fit(S, epochs=epochs)
    fit_dice = mean_dice(fit, held)
    return dict(arm="adapt", gpu=gpu[0], power_limit_w=gpu[1], shape=list(shape), contrast=CONTRAST, train_samples=len(S),
                epochs=epochs, dice_start=round(start, 4), dice_fine_tune=round(ft_dice, 4), dice_fit=round(fit_dice, 4),
                fine_tune_s=round(sum(h['dur'] for h in ft.train_history_), 2),
                fit_s=round(sum(h['dur'] for h in fit.train_history_), 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--epochs", type=int, default=5)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--adapt-size", type=int, default=160)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu = gpu_info()
    torch.cuda.set_device(0)
    lines = []
    with tempfile.TemporaryDirectory() as tmp:
        S = scan_set(os.path.join(tmp, "source"), [1234, 1235], (a.size,) * 3)
        probe = net_from(tmp, "probe")
        line, feats = arm_features(probe, S, gpu)
        lines.append(line)
        lines += arm_step(probe, S, feats, gpu, a.rounds, a.steps)
        del feats
        lines.append(arm_epoch(S, gpu, tmp))
        del S
        lines.append(arm_adapt(gpu, tmp, a.epochs, (a.adapt_size,) * 3))
    for line in lines:
        print(json.dumps(line), flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
