"""Host logic of the grid layout of LightGCNEngine (R row blocks x C column slices), no GPU: validation of the grid,
the rank <-> (row block, column slice) mapping, and what each rank of a fake process group ends up with -- its row
range, its column range, the column-group partners its layer rows and Adam rows go to, the row group's exchange
buffers of the loss, and the hand-off flags it publishes to."""
import types

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from arlib_b200.dist import DistContext
from arlib_b200.engine import LightGCNEngine, dshard_columns, grid_groups, grid_shape
from arlib_b200.graph import DeviceGraph
from arlib_b200.util.synth import synth_edges


def _engine(**kw):
    table = torch.zeros(10, kw.pop("d", 64))
    args = dict(comm=types.SimpleNamespace(world=kw.pop("world", 8), rank=0), mode="grid")
    args.update(kw)
    return LightGCNEngine(None, table, 4, 2, 0.01, 1e-4, 64, 64, **args)


@pytest.mark.parametrize("grid, world", [((1, 8), 8), ((8, 1), 8), ((2, 1), 2), ((3, 2), 8), ((2, 2), 8),
                                         ((2, 4), 4), (None, 8), ((2, 2, 2), 8), ("2x4", 8)])
def test_grid_shapes_outside_the_rule_are_rejected(grid, world):
    with pytest.raises(ValueError, match="grid"):
        grid_shape(grid, world)
    with pytest.raises(ValueError, match="grid"):
        _engine(grid=grid, world=world)


def test_grid_without_a_process_group_is_rejected():
    with pytest.raises(ValueError, match="R \\* C"):
        LightGCNEngine(None, torch.zeros(10, 64), 4, 2, 0.01, 1e-4, 64, 64, mode="grid", grid=(2, 2))


def test_grid_slice_width_must_be_compiled():
    assert grid_shape((2, 4), 8) == (2, 4) and grid_shape([4, 2], 8) == (4, 2)
    with pytest.raises(ValueError, match="slices of 8, 16"):
        _engine(grid=(2, 4), d=16)                # 4-column slices
    with pytest.raises(ValueError, match="not divisible"):
        _engine(grid=(2, 4), d=66)


def test_rank_maps_to_row_block_and_column_slice():
    for R, C in ((2, 2), (2, 4), (4, 2), (2, 3)):
        seen = set()
        for rank in range(R * C):
            r, c, col, row = grid_groups(R, C, rank)
            assert r * C + c == rank and 0 <= r < R and 0 <= c < C
            seen.add((r, c))
            assert col == [q * C + c for q in range(R)] and rank in col
            assert row == [r * C + q for q in range(C)] and rank in row
            assert all(grid_groups(R, C, q)[1] == c for q in col) and all(grid_groups(R, C, q)[0] == r for q in row)
        assert len(seen) == R * C


class _FakeComm(DistContext):
    """DistContext over a fake arena: rank q's buffers start at (q + 1) << 40, so every pointer names its rank"""

    def __init__(self, rank, world):
        self.rank, self.world, self.group = rank, world, None
        self._off = {}
        self.hdl = types.SimpleNamespace(buffer_ptrs=[(q + 1) << 40 for q in range(world)])
        self.use_multicast = False
        self.subgroup_calls = []

    def allocate(self, specs):
        out, off = {}, 0
        for name, (shape, dtype) in specs.items():
            out[name] = torch.zeros(shape, dtype=dtype)
            self._off[name] = off
            off += (out[name].numel() * out[name].element_size() + 255) // 256 * 256
        return out

    def subgroups(self, groups):
        self.subgroup_calls.append([list(g) for g in groups])
        return "row group %d" % (self.rank // len(groups[0]))

    def barrier(self):
        pass


@pytest.mark.parametrize("R, C", [(2, 2), (2, 4), (4, 2)])
def test_each_rank_gets_its_rows_columns_and_partners(monkeypatch, R, C):
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(LightGCNEngine, "_refresh_adam_coefs", lambda self: None)
    monkeypatch.setenv("ARLIB_B200_COEF_STREAM", "0")
    U, I, E, d, L = 120, 180, 3000, 64, 3
    tu, ti, _, _ = synth_edges(U, I, E, seed=5)
    N = U + I
    half = sp.csr_matrix((np.ones(E, dtype=np.float32), (tu, ti + U)), shape=(N, N), dtype=np.float32)
    g = DeviceGraph.from_scipy(half + half.T, "cpu")
    table = torch.randn(N, d)
    bounds = g.row_ranges(R)
    world = R * C
    for rank in range(world):
        comm = _FakeComm(rank, world)
        eng = LightGCNEngine(g, table, U, L, 0.01, 1e-4, 64, 64, comm=comm, mode="grid", grid=(R, C))
        r, c = divmod(rank, C)
        c0, c1 = dshard_columns(d, C, c)
        assert (eng.grid_r, eng.grid_c, eng.col0, eng.col1, eng.d) == (r, c, c0, c1, d // C)
        assert (eng.r0, eng.r1) == (bounds[r], bounds[r + 1]) and (eng.g.r0, eng.g.r1) == (eng.r0, eng.r1)
        assert tuple(eng.E0.shape) == (N, d // C) and torch.equal(eng.E0, table[:, c0:c1])
        assert tuple(eng.G.shape) == tuple(eng.m.shape) == (N, d // C)
        base = lambda q, name: ((q + 1) << 40) + comm._off[name]
        partners = [q * C + c for q in range(R) if q * C + c != rank]
        # layer rows and Adam rows go to the column group only, never by multicast
        for name in ("E0", "F", "fw0", "fw1", "bw0", "bw1"):
            assert eng._peers(name) == [base(q, name) for q in partners]
            assert eng._mcast(name) == 0
        assert eng._peer_E0_rows == [base(q, "E0") + eng.r0 * (d // C) * 4 for q in partners]
        assert eng._handoff_peers == [base(q, "handoff") for q in partners]
        # the loss exchange spans the row group, in column-slice order, this rank at position c
        assert eng._xchg_all == [base(r * C + q, "xchg") for q in range(C)] and eng.xchg_rank == c
        assert comm.subgroup_calls == [[[q * C + k for k in range(C)] for q in range(R)]]
        assert eng.row_pg == "row group %d" % r
        assert not eng.fuse_adam and eng.launches_per_step == 4 * L + 6
