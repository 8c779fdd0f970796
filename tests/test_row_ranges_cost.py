"""Row ranges that balance a * nnz + b * rows (graph.balanced_row_ranges with cost): contiguous, covering every row,
and without the argument exactly the nnz-balanced ranges."""
import numpy as np
import pytest
import torch

from arlib_b200.graph import balanced_row_ranges


def _power_law_indptr(n=5000, seed=0):
    deg = np.random.default_rng(seed).zipf(1.8, n).clip(1, 4000)
    return np.concatenate([[0], np.cumsum(deg)])


def _nnz_only_reference(indptr, world):
    nnz = int(indptr[-1])
    b = [0]
    for p in range(1, world):
        b.append(min(max(int(np.searchsorted(indptr, nnz * p // world, side="left")), b[-1]), len(indptr) - 1))
    return b + [len(indptr) - 1]


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_weighted_ranges_are_contiguous_and_cover_all_rows(world):
    ip = _power_law_indptr()
    n = len(ip) - 1
    assert balanced_row_ranges(ip, world) == _nnz_only_reference(ip, world)
    for cost in [(1.0, 0.0), (0.0, 1.0), (0.5, 40.0), (2e-3, 1.3)]:
        b = balanced_row_ranges(ip, world, cost)
        assert len(b) == world + 1 and b[0] == 0 and b[-1] == n
        assert all(b[k] <= b[k + 1] for k in range(world))


def test_row_weight_moves_boundaries_towards_equal_rows():
    ip = _power_law_indptr()
    n = len(ip) - 1
    by_nnz = balanced_row_ranges(ip, 4)
    by_rows = balanced_row_ranges(ip, 4, (0.0, 1.0))
    assert by_rows == [0, n // 4, n // 2, 3 * n // 4, n]
    rows = lambda b: max(b[k + 1] - b[k] for k in range(4))
    mixed = balanced_row_ranges(ip, 4, (1.0, float(ip[-1]) / n))
    assert rows(by_rows) <= rows(mixed) <= rows(by_nnz)


def test_bad_cost_weights_are_rejected():
    with pytest.raises(ValueError):
        balanced_row_ranges(_power_law_indptr(), 2, (0.0, 0.0))


def test_ngcf_engine_refuses_column_sharding():
    from arlib_b200.engine import NGCFEngine
    table, W = torch.zeros(10, 64), torch.zeros(2, 128, 64)
    with pytest.raises(ValueError, match="column"):
        NGCFEngine(None, table, W, 4, 0.001, 1e-4, 8, 8, mode="dshard")
