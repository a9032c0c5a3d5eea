"""Cost and effect of training-time augmentation in the minibatch gather (sc_gather_samples_augmented).

Arms, each printed as one JSON line with the GPU name and power limit read in the same run:
  gather  plain (sc_gather_samples) against augmented gather (rotation 15 deg, scale 0.15, intensity 0.2, noise 0.05) of
          shuffled minibatches of 256 and 1 024 rows from 8 synthetic 256^3 scans (512 MB of volumes, beyond the 126 MB L2),
          and the full training step (sc_train_forward_backward) on such a minibatch: CUDA events around --launches launches
          per round (each launch a different minibatch of 64), the three arms alternated for --rounds rounds; median of the
          rounds and the spread; the augmented gather as a share of the step
  epoch   one epoch of fit and of fine_tune on the training set of 2 synthetic 256^3 subjects, with and without augmentation
          (history 'dur' of the second of two epochs; fine_tune's includes the per-epoch rebuild of the training rows' features)
  adapt   source = the committed weights; target = synthetic subjects with a per-label contrast table, rotated by 10 degrees and
          zoomed by 1.15 on the host (scipy.ndimage.affine_transform of T1, labels, priors and mask): mean Dice
          (evaluate_segmentation) on a held-out target subject after fine_tune on ONE labelled target subject for --epochs
          epochs, with and without augmentation.  Reported, not asserted.

usage: python scripts/exp_augment.py [--rounds 5] [--launches 200] [--epochs 5] [--out profiles/r10_exp_augment.jsonl]"""
import argparse
import json
import os
import random
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "sub-cortical_segmentation_b200"))

import torch  # noqa: E402
from cnn_cort import base, nets, nifti, synthetic  # noqa: E402

WEIGHTS = os.path.join(ROOT, "nets", "miccai2012_v1", "miccai2012_v1.pkl")
AUG = dict(rotation_deg=15.0, scale=0.15, intensity=0.2, noise=0.05, seed=1)
# target domain of the demo: per-label intensities (as scripts/exp_fine_tune.py), a 10 degree rotation and a 1.15 zoom
CONTRAST = {l: 60.0 * (((l * 5) % 7) - 3) for l in range(1, 16)}
ROT_DEG, ZOOM = 10.0, 1.15


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


def scan_set(root, seeds, shape, contrast=None, warp=False):
    for i, s in enumerate(seeds):
        d = synthetic.write_subject(root, "s%02d" % i, shape=shape, seed=s, with_labels=True, contrast=contrast)
        if warp:
            warp_subject(d)
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
    for i in range(k):
        fn(i)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / k


def arm_gather(gpu, rounds, launches, size):
    """8 synthetic scans of unit Gaussian noise (normalised intensities) and 50 000 training centres per scan, drawn from the
    central half of each axis as training centres lie inside the head"""
    g = torch.Generator(device="cuda").manual_seed(0)
    vols = [torch.randn((size,) * 3, device="cuda", generator=g) for _ in range(8)]
    rng = np.random.RandomState(0)
    per = 50000
    cen = rng.randint(size // 4, 3 * size // 4, size=(8 * per, 3))
    samples = np.concatenate([np.repeat(np.arange(8), per)[:, None], cen], 1)
    S = base.ScanTrainingSet(vols, samples, rng.rand(len(samples), 15), rng.randint(0, 15, len(samples)))
    ctx = nets.Net(options("", "probe"), None, None, seed=0).ctx
    out = []
    for bs in (256, 1024):
        perm = rng.permutation(len(S))
        batches = [torch.from_numpy(perm[i * bs:(i + 1) * bs].astype(np.int64)).cuda() for i in range(64)]
        step_in = S.gather(batches[0], ctx=ctx)
        loss = torch.zeros(1, device="cuda")
        arms = {"plain": lambda i: S.gather(batches[i % 64], ctx=ctx),
                "augmented": lambda i: S.gather(batches[i % 64], ctx=ctx, augment=AUG, epoch=1),
                "step": lambda i: ctx.train_forward_backward(*step_in, seed=3, loss_out=loss)}
        for fn in arms.values():
            events_ms(fn, 20)
        res = {k: [] for k in arms}
        for _ in range(rounds):
            for name, fn in arms.items():
                res[name].append(events_ms(fn, launches if name != "step" else max(20, launches // 4)))
        line = dict(arm="gather", gpu=gpu[0], power_limit_w=gpu[1], batch=bs, scans=8, scan_size=size, rows=len(S),
                    launches_per_round=launches, rounds=rounds, augment=AUG)
        for name, v in res.items():
            line[name + "_ms"] = round(float(np.median(v)), 4)
            line[name + "_spread_ms"] = round(float(max(v) - min(v)), 4)
        line["augmented_over_plain"] = round(line["augmented_ms"] / line["plain_ms"], 2)
        line["augmented_share_of_step"] = round(line["augmented_ms"] / line["step_ms"], 4)
        # the kernels alone (the library's per-class events around each launch), without the host side of the Python call
        ctx.set_option("profile", 1)
        ctx.profile_read()
        for i in range(launches):
            arms["plain"](i)
            arms["augmented"](i)
        prof = ctx.profile_read()
        ctx.set_option("profile", 0)
        line["plain_kernel_ms"] = round(prof["gather"][0] / prof["gather"][1], 4)
        line["augment_kernel_ms"] = round(prof["augment"][0] / prof["augment"][1], 4)
        line["augment_kernel_share_of_step"] = round(line["augment_kernel_ms"] / line["step_ms"], 4)
        out.append(line)
    del S, vols
    return out


def arm_epoch(gpu, tmp, size):
    S = scan_set(os.path.join(tmp, "source"), [1234, 1235], (size,) * 3)
    line = dict(arm="epoch", gpu=gpu[0], power_limit_w=gpu[1], samples=len(S), batch=128, augment=AUG)
    for method in ("fit", "fine_tune"):
        for tag, aug in (("plain", None), ("augmented", AUG)):
            net = net_from(tmp, "ep_%s_%s" % (method, tag), augment=aug)
            getattr(net, method)(S, epochs=2)
            line["%s_%s_epoch_s" % (method, tag)] = round(net.train_history_[-1]['dur'], 3)
            del net
    return line


def warp_subject(d):
    """rotate by ROT_DEG about the axis (1, 1, 1) / sqrt(3) and zoom by ZOOM about the volume centre, in place: T1 and priors
    linear, labels and mask nearest"""
    from scipy import ndimage
    k = np.ones(3) / np.sqrt(3)
    t = np.deg2rad(ROT_DEG)
    K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    R = np.cos(t) * np.eye(3) + np.sin(t) * K + (1 - np.cos(t)) * np.outer(k, k)
    A = R.T / ZOOM                                       # output voxel x reads input c + A (x - c): structures grow by ZOOM
    for rel, order in (("T1.nii.gz", 1), ("gt_15_classes.nii.gz", 0), ("tmp/MNI_subcortical_mask.nii.gz", 0),
                       ("tmp/MNI_sub_probabilities.nii.gz", 1)):
        path = os.path.join(d, rel)
        img = nifti.load(path)
        v = np.asarray(img.get_data())
        c = (np.array(v.shape[:3]) - 1) / 2.0
        off = c - A @ c
        if v.ndim == 4:
            w = np.stack([ndimage.affine_transform(v[..., ch], A, off, order=order) for ch in range(v.shape[3])], -1)
        else:
            w = ndimage.affine_transform(v, A, off, order=order)
        nifti.Nifti1Image(w.astype(v.dtype), img.affine).to_filename(path)


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
    S = scan_set(train_root, [41], shape, CONTRAST, warp=True)           # ONE labelled target subject
    held = synthetic.write_subject(test_root, "held_out", shape=shape, seed=42, with_labels=True, contrast=CONTRAST)
    warp_subject(held)
    line = dict(arm="adapt", gpu=gpu[0], power_limit_w=gpu[1], shape=list(shape), rotation_deg=ROT_DEG, zoom=ZOOM,
                train_samples=len(S), epochs=epochs, augment=AUG, dice_start=round(mean_dice(net_from(tmp, "adapt_src"), held), 4))
    for tag, aug in (("plain", None), ("augmented", AUG)):
        net = net_from(tmp, "adapt_" + tag, augment=aug)
        net.fine_tune(S, epochs=epochs)
        line["dice_fine_tune_" + tag] = round(mean_dice(net, held), 4)
        line["fine_tune_%s_s" % tag] = round(sum(h['dur'] for h in net.train_history_), 2)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--epochs", type=int, default=5)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--adapt-size", type=int, default=160)
    ap.add_argument("--arms", default="gather,epoch,adapt")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu = gpu_info()
    torch.cuda.set_device(0)
    arms = a.arms.split(",")
    with tempfile.TemporaryDirectory() as tmp:
        for arm in arms:
            if arm == "gather":
                lines = arm_gather(gpu, a.rounds, a.launches, a.size)
            elif arm == "epoch":
                lines = [arm_epoch(gpu, tmp, a.size)]
            else:
                lines = [arm_adapt(gpu, tmp, a.epochs, (a.adapt_size,) * 3)]
            for line in lines:
                print(json.dumps(line), flush=True)
                if a.out:
                    with open(a.out, "a") as f:
                        f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
