import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="module")
def one_cpu_thread():
    """CPU torch on one thread: with several, the sparse backward of the oracle trainers sums in a different order
    from run to run, and over an epoch of Adam (SimGCL's sign() perturbation above all) that drift can exceed the
    tolerances the trainers are pinned to."""
    import torch
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


@pytest.fixture(scope="session")
def golden():
    import numpy as np
    return np.load(os.path.join(ROOT, "tests", "golden", "ml100k_lightgcn.npz"), allow_pickle=False)


@pytest.fixture(scope="session")
def golden_rows(golden):
    """(train_rows, test_rows) as the reference's [user, item, weight] string rows."""
    names_u = [str(x) for x in golden["user_names"]]
    names_i = [str(x) for x in golden["item_names"]]
    train = [[names_u[u], names_i[i], 1.0] for u, i in zip(golden["train_u"], golden["train_i"])]
    test = [[str(u), str(i), 1.0] for u, i in zip(golden["test_user_names"], golden["test_item_names"])]
    return train, test
