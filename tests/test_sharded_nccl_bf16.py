"""Row-sharded mixed loss on bf16 videos over 2 and 4 GPUs (NCCL + peer mailboxes), run under torch.distributed.run:
on every rank the bf16 evaluation equals the evaluation on the widened fp32 videos, and the gathered gradient meets
the fp64 oracle bounds.  Skipped on boxes with fewer GPUs."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tests", "sharded_nccl_bf16_worker.py")


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_nccl_bf16(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", str(29621 + world), WORKER, "1024", "4", "16",
                        "16", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    sys.stdout.write(r.stdout[-3000:])
    sys.stderr.write(r.stderr[-3000:])
    assert r.returncode == 0 and "SHARDED_BF16_OK" in r.stdout
