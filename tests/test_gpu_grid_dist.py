"""Grid layout of LightGCNEngine on 4 and 8 GPUs (tests/dist_check_grid.py under torchrun): tables, forward table and
loss rows against the single-GPU engine, identical loss rows on every rank, user-sharded top-K, 200 replayed steps."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_GPUS = torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("world", [4, 8])
def test_grid_layout_matches_single_gpu(world):
    if N_GPUS < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(29541 + world), os.path.join(ROOT, "tests", "dist_check_grid.py")]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    shapes = 1 if world == 4 else 2
    assert res.returncode == 0 and res.stdout.count("GRID_DIST_OK") == shapes, res.stdout[-4000:]
