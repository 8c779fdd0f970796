"""Row-partitioned NGCF on 2 to 8 GPUs (tests/dist_check_ngcf.py under torchrun): bit-identical replicas across ranks,
deterministic eager and graph-replayed steps, and the single-GPU engine's results, with NVSwitch multicast stores and
with per-peer stores."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("multicast", ["1", "0"])
def test_row_partitioned_ngcf_matches_single_gpu(multicast):
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
           "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tests", "dist_check_ngcf.py")]
    env = dict(os.environ, ARLIB_B200_MULTICAST=multicast)
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900, env=env)
    assert res.returncode == 0 and "NGCF_DIST_CHECK_OK" in res.stdout, res.stdout[-3000:]
