#!/usr/bin/env python
"""bench.py -- the reference's headline metric on B200 (BASELINE.json).

Workload (configs[1]): miccai2012_v1 inference of one synthetic 256^3 T1 + synthetic 15-channel
atlas priors, full brain (speedup_segmentation=False: every voxel is a candidate).  One "step" =
one whole volume from "volume + atlas resident in HBM" to "label volume resident in HBM"
(sc_segment_volume: dense dilated formulation of the three-branch CNN + atlas-fused FC head).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--size 256] [--dump-outputs DIR]

--dump-outputs DIR: after the timed steps, rank 0 writes the label volume of its last step as DIR/labels.npy (float32
labels at a fixed, seeded sample of at most DUMP_VOXELS voxels) and DIR/label_index.npy (their flat C-order indices,
float64).  The inputs are seeded, so two builds run with the same arguments can be compared output for output.

N > 1 (launched by torchrun, one rank per GPU): every rank segments its own volume (configs[2]:
volumes sharded across GPUs, no collective) -> weak scaling; value = N * voxels * K / max-over-ranks time.
--impl reference: the reference's CPU path (oracle restatement: numpy gather + torch-CPU forward in
nolearn-sized minibatches of 128) timed on this box's host cores on a bounded sample of the same volume.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os

# stdout carries exactly ONE JSON line: everything libraries print (NCCL's version banner ...) is rerouted to stderr
_JSON_FD = os.dup(1)
os.dup2(2, 1)


def _plain(o):
    """numpy scalars / arrays (a float32 from a parity check ...) -> plain Python for json"""
    if hasattr(o, "tolist"):
        return o.tolist()
    return str(o)


def emit_json(obj):
    os.write(_JSON_FD, (json.dumps(obj, default=_plain) + "\n").encode())

import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "sub-cortical_segmentation_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

METRIC = "voxels_per_sec_full_volume_inference"
UNIT = "voxels/s"
WEIGHTS = os.path.join(ROOT, "nets", "miccai2012_v1", "miccai2012_v1.pkl")
FLOP_PATCHWISE = 35407800       # SURVEY.md 8(d): algorithmic forward FLOPs per voxel, patchwise form
# dense-form algorithmic FLOPs per voxel per kernel class (2 x MAC, three views), SURVEY.md 8f-1
FLOP_DENSE = {"conv1": 3 * 2 * 180, "conv2": 3 * 2 * 3600, "conv3": 3 * 2 * 7200, "conv4": 3 * 2 * 14400,
              "conv5": 3 * 2 * 21600, "gemm_d1": 3 * 2 * 97200, "gemm_fc1": 2 * 291600, "gemm_fc2": 2 * 149850,
              "out_softmax": 2 * 4050}
DUMP_VOXELS = 1 << 22           # 16 MB of float32 labels + 32 MB of float64 indices at most


def dump_labels(lab, out_dir):
    """a fixed, seeded sample of the uint8 label volume (all of it when it has <= DUMP_VOXELS voxels) -> out_dir/*.npy"""
    n = lab.numel()
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_VOXELS), replace=False))
    vals = lab.view(-1).cpu().numpy()[idx]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "labels.npy"), vals.astype(np.float32))
    np.save(os.path.join(out_dir, "label_index.npy"), idx.astype(np.float64))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "tflops_burst": d["bf16_tflops"], "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "tflops_burst": 1590.0, "source": "fallback"}


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled every 100 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def synthetic_volume(size, seed):
    """strictly positive T1 (every voxel a candidate, SURVEY quirk Q3) normalised like base.py:358, + atlas."""
    from cnn_cort import synthetic
    shape = (size, size, size)
    t1 = synthetic.make_t1(shape, seed)
    nz = t1[np.nonzero(t1)]
    norm = ((t1 - nz.mean()) / nz.std()).astype(np.float32)
    atlas, _, _ = synthetic.make_atlas(shape, seed)
    return t1, norm, atlas


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle restatement of the reference's mode=cpu path (test infrastructure used
# here ONLY as the thing timed for the baseline, never on the product path).
# ------------------------------------------------------------------------------------------------
def cpu_reference_rate(norm, atlas, n_voxels, repeats=1, seed=0):
    import torch
    from oracle import gather as og, network as on
    torch.set_num_threads(os.cpu_count() or 1)
    P = on.load_params(WEIGHTS)
    rng = np.random.RandomState(seed)
    shape = norm.shape
    start = rng.randint(0, norm.size - n_voxels)
    lin = np.arange(start, start + n_voxels)                       # consecutive C-order candidates, as test_scan sees them
    cen = np.stack(np.unravel_index(lin, shape), 1)
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        for ax, co, sa, av, _c in og.patch_batches(norm, atlas, cen, 100000):
            on.predict(P, ax, co, sa, av, dtype=torch.float32, minibatch=128)
        times.append(time.perf_counter() - t0)
    return n_voxels / min(times), times


def run_reference(args, rank, world):
    if rank != 0:
        return
    size = args.size
    _, norm, atlas = synthetic_volume(size, 1234)
    sample = args.ref_sample
    for _ in range(args.warmup):
        cpu_reference_rate(norm, atlas, min(256, sample))
    t0 = time.perf_counter()
    rates = [cpu_reference_rate(norm, atlas, sample, seed=s)[0] for s in range(args.steps)]
    total = time.perf_counter() - t0
    value = sample * args.steps / total
    cores = os.cpu_count() or 1
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "miccai2012_v1 inference, one synthetic %d^3 T1 + atlas priors, full brain" % size,
                      "note": "oracle port of the reference's mode=cpu path (Theano stack absent); each step = %d consecutive "
                              "candidate voxels (numpy gather + torch-CPU fp32 forward, minibatch 128), extrapolates linearly" % sample},
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                            "sample": "%d steps x %d voxels of the %d^3 volume" % (args.steps, sample, size)},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0, "per_step_rates": rates}
    emit_json(out)


# ------------------------------------------------------------------------------------------------
# secondary sections (BASELINE.json configs[3], [4] and the N > 1 paths); none of them may cost the headline line
# ------------------------------------------------------------------------------------------------
FLOP_TRAIN_SAMPLE = 3 * FLOP_PATCHWISE       # SURVEY.md 8(d): forward + backward ~ 3 x forward = 106.2 MFLOP per sample


def bench_train(ctx, torch, dist, rank, world, peaks, steps=20, warmup=5):
    """configs[3] (global batch 256 split over the ranks, strong scaling) and configs[4] (1024 samples per GPU, i.e. global
    batch 8192 at 8 GPUs): one training step = forward + backward + gradient all-reduce + Adam, timed on the device."""
    from cnn_cort import parallel
    out = {}
    grads = ctx.grad_tensor()
    if world > 1:
        ctx.fused_attach()          # CUDA IPC handles of the gradient / parameter buffers: the fused all-reduce + Adam kernel
    for name, per_gpu in (("global_batch_256", max(1, 256 // world)), ("per_gpu_batch_1024", 1024)):
        gb = per_gpu * world
        g = torch.Generator(device="cuda").manual_seed(100 + rank)
        x = [torch.randn((per_gpu, 1, 32, 32), device="cuda", generator=g) for _ in range(3)]
        at = torch.softmax(3 * torch.randn((per_gpu, 15), device="cuda", generator=g), 1)
        y = torch.randint(0, 15, (per_gpu,), device="cuda", generator=g, dtype=torch.uint8)
        hx = [t.cpu().pin_memory() for t in x] + [at.cpu().pin_memory(), y.cpu().pin_memory()]
        loss = torch.zeros(1, device="cuda")

        def step(i, from_host=False):
            d = [t.cuda(non_blocking=True) for t in hx] if from_host else x + [at, y]
            ctx.train_forward_backward(*d, n_global=gb, seed=i, loss_out=loss)
            parallel.allreduce_gradients(grads, loss)
            ctx.adam_step(lr=1e-3, stat_scale=1.0 / world)

        def sync():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        for i in range(warmup):
            step(i)
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.counter("launches")
        e0.record()
        for i in range(steps):
            step(i)
        e1.record()
        sync()
        launches = (ctx.counter("launches") - l0) / steps
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        for i in range(2):                      # the first copy out of a fresh page-locked buffer costs tens of ms once
            step(i, from_host=True)
        sync()
        e0.record()
        for i in range(steps):
            step(i, from_host=True)
            float(loss.item())
        e1.record()
        sync()
        ms2 = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        ar_ms = None
        fused_ms = None
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
            sync()
            e0.record()
            for _ in range(50):
                dist.all_reduce(grads)
            e1.record()
            sync()
            ar_ms = e0.elapsed_time(e1) / 50
            # the same step with the gradient all-reduce fused into the Adam kernel over NVLink peer memory (sc_allreduce_adam_step)
            def fstep(i):
                ctx.train_forward_backward(*(x + [at, y]), n_global=gb, seed=i, loss_out=loss)
                ctx.allreduce_adam_step(lr=1e-3)
            for i in range(warmup):
                fstep(i)
            sync()
            e0.record()
            for i in range(steps):
                fstep(i)
            e1.record()
            sync()
            t = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            fused_ms = float(t) / steps
        per = float(ms) / steps
        tfl = gb * FLOP_TRAIN_SAMPLE / (per * 1e-3) / 1e12
        hbm = None           # the step is bound by the element-wise BatchNorm passes: DRAM bytes per step from the committed ncu capture
        tpath = os.path.join(ROOT, "profiles", "r2_train_traffic.json")
        if os.path.exists(tpath):
            byt = json.load(open(tpath))["dram_bytes_per_step"].get(str(per_gpu))
            if byt:
                gbs = byt / (per * 1e-3) / 1e9
                hbm = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                       "traffic": byt, "note": "per GPU; DRAM bytes of one step measured with ncu (profiles/r2_train_traffic_1024.txt)"}
        out[name] = {"global_batch": gb, "per_gpu_batch": per_gpu, "ms_per_step": per, "samples_per_s": gb / (per * 1e-3),
                     "e2e_samples_per_s": gb / (float(ms2) / steps * 1e-3), "h2d_bytes_per_step": int(per_gpu * (3 * 4096 + 60 + 1)),
                     "allreduce_ms": ar_ms, "allreduce_bytes": 883455 * 4, "ms_per_step_fused_allreduce_adam": fused_ms,
                     "samples_per_s_fused": (gb / (fused_ms * 1e-3)) if fused_ms else None, "gpu_launches_per_step": launches, "loss": float(loss.item()),
                     "roofline": {"bound": "tensor", "achieved": tfl, "peak": peaks["tflops"] * world, "unit": "TFLOP/s",
                                  "frac": tfl / (peaks["tflops"] * world), "flops_per_sample": FLOP_TRAIN_SAMPLE},
                     "roofline_hbm": hbm}
    out["scaling"] = {"global_batch_256": "strong (256 / N samples per GPU)", "per_gpu_batch_1024": "weak"}
    out["bn"] = "per-GPU batch statistics"
    return out


def bench_single_volume_sharded(ctx, torch, dist, rank, world, d_vol, d_atlas, d_mask, nvox, steps=3):
    """the metric's 'seconds per 256^3 volume at N GPUs': ONE volume, every rank segments its x-slab of the candidate box
    (parallel.segment_volume_sharded: no collective on the data path), the label slabs are gathered to rank 0 by
    NCCL point-to-point copies over NVLink.  The volume / atlas are rank 0's, broadcast once outside the timed region."""
    from cnn_cort import parallel
    vol, atlas, mask = d_vol.clone(), d_atlas.clone(), d_mask.clone()
    dist.broadcast(vol, 0); dist.broadcast(atlas, 0); dist.broadcast(mask, 0)
    shape = tuple(vol.shape)
    lab = torch.zeros(shape, dtype=torch.uint8, device="cuda")
    box = (0, shape[0], 0, shape[1], 0, shape[2])

    def one():
        lab.zero_()
        mine = parallel.segment_volume_sharded(ctx, vol, atlas, box=box, cand_mask=mask, label_vol=lab)
        reqs = []
        if rank == 0:
            for r in range(1, world):
                s = parallel.shard_box(box, r, world)
                if s is not None:
                    reqs.append(dist.irecv(lab[s[0]:s[1]], src=r))
        elif mine is not None:
            reqs.append(dist.isend(lab[mine[0]:mine[1]], dst=0))
        for q in reqs:
            q.wait()

    one()
    dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        one()
    e1.record()
    dist.barrier(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    # union check against the unsharded result on rank 0
    ok = None
    if rank == 0:
        ref = torch.zeros(shape, dtype=torch.uint8, device="cuda")
        ctx.segment_volume(vol, atlas, cand_mask=mask, label_vol=ref)
        ok = bool((ref == lab).all())
    ms = float(t.item())
    return {"ms_per_volume": ms, "seconds_per_volume": ms * 1e-3, "voxels_per_s": nvox / (ms * 1e-3), "union_equals_unsharded": ok,
            "note": "x-slab split of one %s volume over %d GPUs, each slab recomputes a 16-plane halo in the saggital view and the full "
                    "planes of the axial / coronal views' conv phase is restricted to its slab +- 16; labels gathered to rank 0" % (shape, world)}


def bench_test_scan_hot(ctx, torch, t1, atlas, steps=3):
    """the drop-in call's timed part (cnn_cort.base.segment_arrays = test_scan minus NIfTI I/O): raw T1 + atlas priors in
    page-locked Fortran-ordered host arrays (what nifti.load(pinned=True) yields) -> label volume on the host; device-side
    import, normalisation, candidate mask, bounding box, dense network pass."""
    from cnn_cort import base, synthetic
    def pinned_f(a):
        t = torch.empty(a.size * a.itemsize, dtype=torch.uint8, pin_memory=True)
        v = t.numpy().view(a.dtype).reshape(a.shape, order="F")
        v[...] = a
        return t, v
    keep1, t1f = pinned_f(t1)
    keep2, atf = pinned_f(atlas)
    keep3, mkf = pinned_f(synthetic.make_mask(atlas))
    out = {}
    for name, crop in (("full_brain", None), ("crop", mkf)):
        tm = {}
        base.segment_arrays(ctx, t1f, atf, crop, False, tm)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            base.segment_arrays(ctx, t1f, atf, crop, False, tm)
        wall = (time.perf_counter() - t0) / steps
        out[name] = {"wall_ms": wall * 1e3, "candidates": tm["n_candidates"], "candidate_voxels_per_s": tm["n_candidates"] / wall,
                     "box": list(tm["box"]) if tm["box"] else None}
    out["call"] = ("cnn_cort.base.segment_arrays (the body of test_scan between reading the NIfTI files into page-locked memory and "
                   "writing the outputs), host wall clock")
    return out


def bench_volume_320_proba(ctx, torch, dist, rank, world, steps=2):
    """configs[4]: out_probabilities=True over a 0.7 mm 320^3 volume per GPU (32 768 000 voxels, 1.97 GB probability volume)"""
    _, norm, atlas = synthetic_volume(320, 4321 + rank)
    dv, da = torch.from_numpy(norm).cuda(), torch.from_numpy(atlas).cuda()
    lab = torch.zeros(norm.shape, dtype=torch.uint8, device="cuda")
    prob = torch.zeros(norm.shape + (15,), dtype=torch.float32, device="cuda")
    ctx.segment_volume(dv, da, label_vol=lab, proba_vol=prob)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        ctx.segment_volume(dv, da, label_vol=lab, proba_vol=prob)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    n = norm.size
    del dv, da, lab, prob
    torch.cuda.empty_cache()
    return {"ms_per_volume": ms, "voxels_per_s": world * n / (ms * 1e-3), "voxels_per_volume": n, "proba_volume_bytes": n * 60,
            "volumes": world, "workspace_bytes": ctx.counter("workspace_bytes")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--gemm", type=int, default=-1, help="-1 library default, 0 SIMT fp32, 1 tcgen05 TF32")
    ap.add_argument("--ref-sample", type=int, default=16384)
    ap.add_argument("--cpu-sample", type=int, default=65536)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="headline + e2e only (skip train / sharded / 320^3 / dp_check sections)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the labels of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist
    from cnn_cort import _native, nets
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import datetime     # a rank that leaves a collective section early must cost minutes, not the default ten
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=180))
    peaks = load_peaks()
    size = args.size
    nvox = size ** 3
    t1, norm, atlas = synthetic_volume(size, 1234 + rank)
    ctx = _native.Context(local_rank)
    import pickle
    with open(WEIGHTS, "rb") as f:
        ctx.load_weights(nets.pack_params(pickle.load(f, encoding="latin1")))
    if args.gemm >= 0:
        ctx.set_option("gemm", args.gemm)
    backend = "tcgen05-bf16x3" if ctx.counter("gemm") == 1 else "simt-fp32"

    d_vol = torch.from_numpy(norm).cuda()
    d_atlas = torch.from_numpy(atlas).cuda()
    d_mask = torch.from_numpy((t1 != 0).view(np.uint8)).cuda()      # base.py:372 candidates = non-zero voxels of the raw T1
    d_lab = torch.zeros((size,) * 3, dtype=torch.uint8, device="cuda")
    n_cand = int(d_mask.sum())

    def step():
        ctx.segment_volume(d_vol, d_atlas, cand_mask=d_mask, label_vol=d_lab)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    ctx.set_option("profile", 1)
    ctx.profile_read()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    l0 = ctx.counter("launches")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ctx.counter("launches") - l0
    prof = ctx.profile_read()
    ctx.set_option("profile", 0)
    clk = clocks.stop() if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * n_cand * args.steps / (ms_max * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_labels(d_lab, args.dump_outputs)       # before the sections below overwrite d_lab

    # ---- end to end through the host-buffer C-ABI call: pinned host volume + atlas in, labels out ----
    h_vol = torch.from_numpy(norm).pin_memory()
    h_atlas = torch.from_numpy(atlas).pin_memory()
    h_mask = torch.from_numpy((t1 != 0).view(np.uint8)).pin_memory()
    h_lab = torch.zeros((size,) * 3, dtype=torch.uint8).pin_memory()
    e2e_steps = max(1, min(args.steps, 3))

    def e2e_step():
        ctx.segment_volume_host(h_vol.numpy(), h_atlas.numpy(), cand_mask=h_mask.numpy(), label_out=h_lab.numpy())

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for _ in range(e2e_steps):
        e2e_step()
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    t = torch.tensor([e2e_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * n_cand * e2e_steps / (float(t.item()) * 1e-3)
    agree = float((torch.from_numpy(h_lab.numpy()).cuda() == d_lab).float().mean())

    # ---- secondary measurements on rank 0: K1 gather bandwidth and the patchwise (predict_proba) path ----
    extra = {}
    if rank == 0:
        try:
            nb = 100000                                   # one reference test batch (test_batch_size, configuration.cfg:19)
            time.sleep(2.0)                               # the secondary kernels are timed alone: let the power-capped clocks of the volume passes recover
            xyz = ctx.nonzero_coords(d_mask)[5000000:5000000 + nb].contiguous()
            bufs = [torch.empty((nb, 1, 32, 32), device="cuda") for _ in range(3)] + [torch.empty((nb, 15), device="cuda")]
            import ctypes
            def gather():
                _native._check(ctx.lib.sc_gather_patches(ctx.h, d_vol.data_ptr(), _native._dims(d_vol.shape), d_atlas.data_ptr(), 1,
                                                         xyz.data_ptr(), nb, bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr(),
                                                         bufs[3].data_ptr(), torch.cuda.current_stream().cuda_stream))
            for _ in range(3):
                gather()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(20):
                gather()
            e1.record()
            torch.cuda.synchronize()
            g_ms = e0.elapsed_time(e1) / 20
            gbs = nb * 12424 / (g_ms * 1e-3) / 1e9       # SURVEY 8(d): 12 424 algorithmic bytes per voxel
            extra["gather"] = {"kernel": "gather_patches_kernel", "voxels_per_call": nb, "ms_per_call": g_ms, "voxels_per_s": nb / (g_ms * 1e-3),
                               "bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                               "note": "3 x [n,1,32,32] fp32 patches + [n,15] atlas vectors written per call; outputs (1.2 GB) exceed L2"}
            ctx.forward_from_volume(d_vol, d_atlas, xyz)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(3):
                ctx.forward_from_volume(d_vol, d_atlas, xyz)
            e1.record()
            torch.cuda.synchronize()
            p_ms = e0.elapsed_time(e1) / 3
            extra["patchwise"] = {"call": "sc_forward_from_volume (gather + predict_proba on patches, one 100 000-voxel test batch)",
                                  "ms_per_batch": p_ms, "voxels_per_s": nb / (p_ms * 1e-3),
                                  "algorithmic_tflops": nb * FLOP_PATCHWISE / (p_ms * 1e-3) / 1e12}
            # brain-like candidate mask (a centred ball holding 35 % of the voxels, its bounding box passed as test_scan does):
            # the conv phase runs on the box, d1 skips tiles without candidates, the FC head runs on the compacted candidate rows
            axr = torch.arange(size, device="cuda", dtype=torch.float32) - (size - 1) / 2
            rad = size * (3 * 0.35 / (4 * np.pi)) ** (1.0 / 3.0)
            ball = ((axr[:, None, None] ** 2 + axr[None, :, None] ** 2 + axr[None, None, :] ** 2) < rad * rad).to(torch.uint8).contiguous()
            lo, hi = int(np.floor((size - 1) / 2 - rad)) , int(np.ceil((size - 1) / 2 + rad)) + 1
            lo, hi = max(lo, 0), min(hi, size)
            bbox = (lo, hi, lo, hi, lo, hi)
            n_ball = int(ball.sum())
            time.sleep(1.0)
            for _ in range(2):
                ctx.segment_volume(d_vol, d_atlas, box=bbox, cand_mask=ball, label_vol=d_lab)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(3):
                ctx.segment_volume(d_vol, d_atlas, box=bbox, cand_mask=ball, label_vol=d_lab)
            e1.record()
            torch.cuda.synchronize()
            m_ms = e0.elapsed_time(e1) / 3
            extra["masked_volume"] = {"call": "sc_segment_volume with a candidate mask (centred ball, %.0f %% of the 256^3 voxels) and its bounding box" % (100.0 * n_ball / size ** 3),
                                      "candidates": n_ball, "ms_per_volume": m_ms, "candidate_voxels_per_s": n_ball / (m_ms * 1e-3)}
            del ball
            del bufs
        except Exception as exc:          # the secondary sections must never cost the headline line
            extra["secondary_error"] = repr(exc)[:300]

    # ---- sections every rank takes part in: training (configs[3], [4]), the N > 1 checks, one volume sharded over the ranks,
    # the 320^3 probability sweep (configs[4]) ----
    if not args.no_secondary:
        del h_vol, h_atlas, h_mask, h_lab
        def section(name, fn):
            try:
                extra[name] = fn()
            except Exception as exc:
                extra[name] = {"error": repr(exc)[:300]}
                sys.stderr.write("bench.py: section %s failed on rank %d: %r\n" % (name, rank, exc))
        time.sleep(1.0)
        section("train", lambda: bench_train(ctx, torch, dist, rank, world, peaks))
        ctx.load_weights(nets.pack_params(pickle.load(open(WEIGHTS, "rb"), encoding="latin1")))   # the steps above moved the weights
        if world > 1:
            def dp():
                sys.path.insert(0, os.path.join(ROOT, "tests"))
                import dp_check
                res = dp_check.run_checks(ctx, rank, world, local_rank, fit=True)
                res["result"] = "ok"
                return res
            section("dp_check", dp)
            ctx.load_weights(nets.pack_params(pickle.load(open(WEIGHTS, "rb"), encoding="latin1")))
            section("single_volume_sharded", lambda: bench_single_volume_sharded(ctx, torch, dist, rank, world, d_vol, d_atlas, d_mask, nvox))
        if rank == 0:
            section("test_scan_hot", lambda: bench_test_scan_hot(ctx, torch, t1, atlas))
            if "wall_ms" in extra["test_scan_hot"].get("full_brain", {}):
                extra["test_scan_hot"]["full_brain"]["vs_e2e"] = extra["test_scan_hot"]["full_brain"]["wall_ms"] / (1e3 * n_cand * world / e2e_value)
        del d_vol, d_atlas, d_mask, d_lab
        torch.cuda.empty_cache()
        section("volume_320_proba", lambda: bench_volume_320_proba(ctx, torch, dist, rank, world))

    if rank != 0:
        if world > 1:
            dist.barrier()            # rank 0 is still measuring its CPU baseline
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel class (CUDA-event times measured over the timed region) ----
    table = {}
    for name, (kms, cnt) in prof.items():
        fl = FLOP_DENSE.get(name, 0) * nvox * args.steps
        table[name] = {"ms_per_step": kms / args.steps, "launches_per_step": cnt / args.steps,
                       "share": kms / max(ms, 1e-9), "algorithmic_tflops": fl / (kms * 1e-3) / 1e12 if kms > 0 and fl else None}
    dom = max(table, key=lambda k: table[k]["ms_per_step"])
    dk = table[dom]
    flops_per_launch = FLOP_DENSE.get(dom, 0) * nvox / max(dk["launches_per_step"], 1e-9)
    dur_s = dk["ms_per_step"] * 1e-3 / max(dk["launches_per_step"], 1e-9)
    achieved = flops_per_launch / dur_s / 1e12 if dur_s > 0 else 0.0
    # executed tensor work of the bf16x3 split: 3 MMAs per algorithmic product, plus K / N padding of the tile
    pad = {"gemm_d1": 3 * (576 / 540.0) * (192 / 180.0), "gemm_fc1": 3 * (576 / 540.0) * (576 / 540.0),
           "gemm_fc2": 3 * (576 / 555.0) * (288 / 270.0)}.get(dom)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")     # dram bytes per launch from the committed ncu --set full capture
    if os.path.exists(tpath) and size == 256 and backend.startswith("tcgen05"):
        traffic = json.load(open(tpath))["bytes_per_launch"].get(dom)
    roofline = {"kernel": dom, "bound": "tensor", "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s",
                "frac": achieved / peaks["tflops"], "traffic": traffic,
                "executed_over_algorithmic": pad,
                "tensor_pipe_frac_executed": (achieved * pad / peaks["tflops"]) if (pad and backend.startswith("tcgen05")) else None,
                "peak_source": "%s bf16 sustained (MEASURED_PEAKS.json); the kernel issues 3 bf16 MMAs per algorithmic product "
                               "(split-precision, needed for the 1e-3 tolerance), so frac <= 1/3 by construction" % peaks["source"],
                "algorithmic_flops_per_launch": flops_per_launch, "avg_launch_ms": dur_s * 1e3,
                "patchwise_equivalent_tflops": value * FLOP_PATCHWISE / 1e12,
                "dense_executed_tflops": value * sum(FLOP_DENSE.values()) / 1e12}

    cpu_base = None
    if world == 1 and not args.no_cpu_baseline:
        rate, times = cpu_reference_rate(norm, atlas, args.cpu_sample)
        cpu_base = {"value": rate, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                    "sample": "%d consecutive candidate voxels of the same %d^3 volume: numpy gather + torch-CPU fp32 forward, "
                              "minibatch 128 (%.1f s); extrapolates linearly to the volume" % (args.cpu_sample, size, min(times))}

    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
           "ms_per_step": ms_max / args.steps, "seconds_per_volume": ms_max / args.steps * 1e-3, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if backend.startswith("tcgen05") else "f32",
           "data": "synthetic",
           "config": {"workload": "miccai2012_v1 inference on B200, one synthetic %d^3 T1 + synthetic atlas priors per GPU, full brain "
                                  "(speedup_segmentation=False, all %d voxels)" % (size, n_cand),
                      "path": "sc_segment_volume (dense dilated formulation == patchwise network at every voxel)",
                      "gemm_backend": backend, "l2": "inputs + activations (>> 126 MB) exceed L2; no explicit flush",
                      "parallelism": "volumes sharded across %d GPU(s), no collective" % world},
           "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(norm.nbytes + atlas.nbytes + nvox),
                   "d2h_bytes_per_step": int(nvox), "steps": e2e_steps, "label_agreement_with_device_path": agree,
                   "call": "sc_segment_volume_host (pinned host volume + atlas + mask in, uint8 label volume out)"},
           "gpu_launches": int(launches), "clocks": clk, "roofline": roofline, "kernels": table}
    out.update(extra)
    if cpu_base:
        out["cpu_baseline"] = cpu_base
    emit_json(out)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
