"""2-rank NCCL parity of the data-parallel step through the real engine (SURVEY §8 row a9): skipped on a 1-GPU box."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_step_equals_single_rank_on_concatenated_batch():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29533",
           os.path.join(ROOT, "tests", "ddp_parity_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0 and "DDP_PARITY_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-6000:]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_recipe_loop_under_ddp(tmp_path):
    """finetune.main with enable_ddp on 2 ranks (NCCL): the reference's DDP recipe mode end to end (sampler shards, broadcast, async all-reduce
    + deferred AdamW inside train(), epoch metric all-reduces); replicas stay bit-identical."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29534",
           os.path.join(ROOT, "tests", "ddp_recipe_worker.py"), str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0 and "DDP_RECIPE_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-6000:]
