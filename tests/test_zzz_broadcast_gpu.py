"""dmnd_block_broadcast (csrc/cuda/comm.cu): the resident, masked reference block from rank 0 to every rank over NCCL, device to
device, through the C ABI -- needs two GPUs (skipped on a machine with one)."""
import os, subprocess, sys
import pytest
from conftest import ROOT

pytestmark = pytest.mark.gpu


def test_block_broadcast_two_ranks():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port", "29577",
                        os.path.join(ROOT, "tests", "_bcast_worker.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "broadcast ok on 2 ranks" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
