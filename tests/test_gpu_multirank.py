"""GPU, >= 2 devices: one process per GPU under torchrun (NCCL) -- SURVEY 4(iv): the sharded projection (gather fused into
the kernel over peer memory, NCCL fallback, ragged module helper) equals the unsharded run bit for bit, and the data-parallel
trainer step equals the single-process step.  Skipped on a machine with fewer than 2 GPUs."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs on one node")
def test_sharded_equals_unsharded_two_ranks():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "multirank_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    print(out.stdout[-4000:], out.stderr[-4000:])
    assert out.returncode == 0 and "MULTIRANK OK" in out.stdout
