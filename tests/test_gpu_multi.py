"""N > 1 on real GPUs: torchrun-launched checks of sharded inference and DP training (tests/dp_check.py).
Two ranks over NCCL when the box has >= 2 GPUs; two gloo ranks sharing GPU 0 otherwise, so the single-GPU test box
exercises the data-parallel host logic (param broadcast, gradient all-reduce, dataset check, Net.fit) on real kernels."""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _free_port():
    """a port no other job on a shared machine is listening on (a fixed port may be taken)"""
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _run(extra):
    port = _free_port()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(HERE, "dp_check.py")] + extra
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "dp_check ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_two_ranks_nccl():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _run(["--backend=nccl"])


def test_two_ranks_sharing_one_gpu_gloo():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    _run(["--backend=gloo", "--same-device"])
