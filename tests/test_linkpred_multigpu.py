"""Query-sharded link-prediction evaluation over two GPUs with NCCL, as a -m gpu test: skipped on a one-GPU box, run
under torchrun on two GPUs otherwise (tests/multigpu/check_nccl_linkpred.py: the 2-rank result equals the single-rank
one)."""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_nccl_linkpred_two_gpus():
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29538", os.path.join(ROOT, "tests", "multigpu", "check_nccl_linkpred.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "nccl linkpred check ok on 2 GPUs" in r.stdout
