"""The grid layout (R row blocks x C column slices) of LightGCNEngine and its column-group hand-off kernel on ONE GPU,
ranks as threads (tests/grid_one_device_check.py): the training step against the single-GPU engine -- E0 and the
forward table within 2e-6 after 5 steps (2 eager, 3 replayed from a CUDA graph), loss rows bit-identical on
all ranks, the E0 slice bit-identical across each column group -- and the hand-off alone on 2 to 8 streams: 1 000
captured hand-offs replayed twice, stamps counting up one by one, the error word untouched.

Each case runs in a process of its own with CUDA_DEVICE_MAX_CONNECTIONS=32 (every rank's stream gets its own hardware
queue) and CUDA_MODULE_LOADING=EAGER (no kernel is loaded, which synchronises the context, while a rank spins)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    env = dict(os.environ, CUDA_DEVICE_MAX_CONNECTIONS="32", CUDA_MODULE_LOADING="EAGER")
    cmd = [sys.executable, os.path.join(ROOT, "tests", "grid_one_device_check.py")] + [str(a) for a in args]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900, env=env)
    assert res.returncode == 0, res.stdout[-4000:]
    return res.stdout


@pytest.mark.parametrize("grid", ["2x2", "2x4"])
def test_grid_layout_matches_single_gpu(grid):
    out = _run("engine", "--grid", grid, "--d", 64, 128, "--layers", 1, 2, 3)
    assert out.count("GRID_OK") == 6, out[-4000:]


def test_group_handoff_replayed_on_two_to_eight_streams():
    out = _run("handoff", "--ranks", 2, 3, 4, 5, 6, 7, 8)
    assert out.count("HANDOFF_OK") == 7, out[-4000:]
