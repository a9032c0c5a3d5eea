#!/usr/bin/env python
"""Atlas registration on one GPU: a synthetic 256^3 1 mm subject made from a 182 x 218 x 182 1 mm template through a known
affine + B-spline transform (cnn_cort.synthetic.make_registration_pair).  Prints one JSON line:

  gpu, power_limit_w          the card, read in the same run
  affine_ms, ffd_ms           CUDA-event time of sc_register_affine / sc_register_ffd; iterations (accepted steps) per level
  warp_priors_ms, mask_ms     sc_warp_volume of the 15-channel priors, sc_prior_mask
  nmi, disp_mean_mm, disp_p95_mm   final NMI and the displacement error against phi_true over the subject's mask
  test_scan_*_s               test_scan on a fresh subject folder: registration, writing tmp/, segmentation (wall clock)
  dice                        per structure, labels segmented with the registered priors against those with the true priors

    python scripts/exp_register.py [--out FILE] [--size 256]
"""
import argparse
import json
import os
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
from oracle import network as on, register as orr  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    name, pl = [s.strip() for s in q.stdout.strip().split(",")][:2]
    return name, float(pl)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return out, a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--size", type=int, default=256)
    args = ap.parse_args()
    name, pl = gpu_info()
    torch.cuda.set_device(0)
    ctx = base.get_context(0)
    n = args.size
    tshape = (182, 218, 182) if n == 256 else (int(n * 0.71),) * 3
    P = synthetic.make_registration_pair((n, n, n), template_shape=tshape, seed=7, subject_spacing=(1.0, 1.0, 1.0),
                                         template_spacing=1.0, deform_mm=4.0)
    ref, flo, pri = base._cuda_f32(P['t1'], 0), base._cuda_f32(P['template'], 0), base._cuda_f32(P['priors'], 0)
    MR, MF = P['t1_affine'], P['template_affine']
    ctx.register_objective(ref, MR, flo, MF, np.eye(4))          # warm-up: module load, workspace
    A, t_aff = timed(lambda: ctx.register_affine(ref, MR, flo, MF))
    grid, t_ffd = timed(lambda: ctx.register_ffd(ref, MR, flo, MF, A))
    iters = {"affine": [ctx.counter("reg_iters:%d" % l) for l in range(4)], "ffd": [ctx.counter("reg_iters:%d" % (4 + l)) for l in range(3)]}
    warped, t_warp = timed(lambda: ctx.warp_volume(pri, MF, A, grid, ref.shape, MR))
    mask, t_mask = timed(lambda: ctx.prior_mask(warped, 5))
    nmi = ctx.register_objective(ref, MR, flo, MF, A, grid)[0]
    g = grid.cpu().numpy().astype(np.float64)
    m = P['t1'] != 0
    err = np.sqrt(((orr.phi(P['t1'].shape, MR, A, g) - P['phi']) ** 2).sum(-1))[m]
    err_aff = np.sqrt(((orr.phi(P['t1'].shape, MR, A) - P['phi']) ** 2).sum(-1))[m]
    # the pipeline: test_scan on a fresh subject folder
    ctx.load_weights(nets.pack_params(on.load_params(os.path.join(ROOT, "nets", "miccai2012_v1", "miccai2012_v1.pkl"))))
    with tempfile.TemporaryDirectory() as tmp:
        nifti.Nifti1Image(P['template'], MF).to_filename(os.path.join(tmp, "MNI.nii.gz"))
        nifti.Nifti1Image(P['priors'], MF).to_filename(os.path.join(tmp, "priors.nii.gz"))
        subj = os.path.join(tmp, "test", "s1")
        os.makedirs(subj)
        t1p = os.path.join(subj, "T1.nii.gz")
        nifti.Nifti1Image(P['t1'], MR).to_filename(t1p)
        opts = {'test_folder': os.path.dirname(subj), 't1_name': 'T1.nii.gz', 'out_probabilities': 'False', 'post_process': 'True',
                'crop': 'True', 'crop_bool': True, 'debug': 'False', 'device': 0, 'test_batch_size': 100000,
                'atlas_template': os.path.join(tmp, "MNI.nii.gz"), 'atlas_priors': os.path.join(tmp, "priors.nii.gz")}
        rt = {}
        t0 = time.time()
        priors, rmask = base.register_masks(t1p, opts, timings=rt)
        torch.cuda.synchronize()

        class _N(object):
            pass
        net = _N()
        net.ctx = ctx
        t1s = time.time()
        seg_reg, _, _ = base.segment_arrays(ctx, P['t1'], priors, rmask, post_mask=rmask)
        seg_reg = seg_reg.copy()
        t_seg = time.time() - t1s
        truth_mask = synthetic.make_mask(P['truth_priors'])
        seg_true, _, _ = base.segment_arrays(ctx, P['t1'], P['truth_priors'], truth_mask, post_mask=truth_mask)
        metrics, _ = base.evaluate_segmentation(seg_reg, seg_true.copy())
        t_total = time.time() - t0
    rec = {"exp": "register", "gpu": name, "power_limit_w": pl, "subject": [n] * 3, "template": list(tshape),
           "affine_ms": t_aff, "ffd_ms": t_ffd, "iterations": iters, "warp_priors_ms": t_warp, "mask_ms": t_mask,
           "nmi": nmi, "disp_mean_mm": float(err.mean()), "disp_p95_mm": float(np.percentile(err, 95)),
           "disp_affine_only_mean_mm": float(err_aff.mean()),
           "test_scan_register_s": rt['register_s'], "test_scan_write_tmp_s": rt['write_s'], "test_scan_segment_s": t_seg,
           "dice": {int(l): (None if v['dice'] != v['dice'] else round(v['dice'], 4)) for l, v in metrics.items()},
           "truth_voxels": {int(l): v['n_ref'] for l, v in metrics.items()}}
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
