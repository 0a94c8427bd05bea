"""Row-sharded mixed loss with shared context frames against the fp64 oracle of the whole problem: one rank always,
two ranks over NCCL + peer mailboxes under torch.distributed.run when the box has two GPUs."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tests", "sharded_nccl_ctx_worker.py")


def _run(cmd, timeout):
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    sys.stdout.write(r.stdout[-3000:])
    sys.stderr.write(r.stderr[-3000:])
    return r


def test_sharded_ctx_single_rank_vs_oracle():
    r = _run([sys.executable, WORKER, "256", "5", "6", "10", "1", "2"], 300)
    assert r.returncode == 0 and "SHARDED_CTX_OK" in r.stdout


def test_sharded_ctx_nccl_vs_oracle():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
              "127.0.0.1", "--master-port", "29633", WORKER, "1024", "4", "16", "16", "1", "2"], 600)
    assert r.returncode == 0 and "SHARDED_CTX_OK" in r.stdout
