"""Data-parallel Net.fit on a ScanTrainingSet, run by every rank of a torchrun job (test infrastructure, launched by
tests/test_gpu_train_scans.py): NCCL on >= 2 GPUs, or two gloo ranks sharing one GPU.

  1. fit(scans) from different per-rank initialisations: the replicas end bit-identical
  2. a rank whose scan set differs (other negatives, drawn from another seed) makes every rank raise
"""
import os
import random
import sys

import numpy as np
import torch
import torch.distributed as dist

from dp_check import _agree        # tests/ is the script's directory; dp_check puts the package on sys.path
from cnn_cort import base, nets    # noqa: E402


def check_fit_on_scans(rank, world, device, data):
    options = {'experiment': 'dp_scans', 'patch_size': [32, 32], 'mode': 'cuda%d' % device, 'device': device,
               'load_weights': 'False', 'net_verbose': 0, 'train_split': 0.25, 'max_epochs': 2, 'patience': 5,
               'batch_size': 512, 'seed': None, 'train_folder': data, 't1_name': 'T1.nii.gz',
               'roi_name': 'gt_15_classes.nii.gz', 'debug': 'False'}
    random.seed(11)
    np.random.seed(11)
    scans = base.load_scan_training_set(options, device=device)
    net = nets.Net(options, None, None, seed=1000 + rank)         # per-rank initialisation differs on purpose
    net.fit(scans)
    p = net.ctx.param_tensor().clone()
    ref = p.clone()
    if dist.get_backend() == "nccl":
        dist.broadcast(ref, 0)
    else:
        h = ref.cpu()
        dist.broadcast(h, 0)
        ref = h.to(p.device)
    errs = []
    if not torch.equal(p, ref):
        errs.append("Net.fit(scans) replicas diverged")
    if not (len(net.train_history_) == 2 and np.isfinite(net.train_history_[-1]['train_loss'])):
        errs.append("Net.fit(scans) history incomplete")
    random.seed(11 + (rank == world - 1))                        # the last rank draws other negatives
    np.random.seed(11)
    other = base.load_scan_training_set(options, device=device)
    try:
        net.fit(other, epochs=1)
    except ValueError:
        pass
    else:
        errs.append("a rank with a different scan set was not detected")
    net.ctx.close()
    return errs


def main():
    backend, same_device, data = "nccl", False, None
    for a in sys.argv[1:]:
        if a.startswith("--backend="):
            backend = a.split("=", 1)[1]
        elif a == "--same-device":
            same_device = True
        elif a.startswith("--data="):
            data = a.split("=", 1)[1]
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    device = 0 if same_device else local
    torch.cuda.set_device(device)
    import datetime
    if backend == "nccl":
        dist.init_process_group("nccl", device_id=torch.device("cuda", device), timeout=datetime.timedelta(seconds=180))
    else:
        dist.init_process_group(backend, timeout=datetime.timedelta(seconds=180))
    _agree(check_fit_on_scans(rank, world, device, data), "Net.fit on scans")
    dist.barrier()
    if rank == 0:
        print("dp_scans_check ok: world=%d backend=%s" % (world, backend))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
