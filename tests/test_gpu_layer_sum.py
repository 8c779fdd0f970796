"""GPU parity of the batch-rows layer sum of the LightGCN step: forward layers 1 .. L-1 write only their tables and the
last layer forms ((E0 + E1) + ... + E_{L-1} + t) / (L + 1) at the batch's rows (acc_terms).  It must equal the running
layer sum of forward_table bit for bit on those rows, and a training epoch must not change by a bit."""
import gc

import numpy as np
import pytest
import torch

from oracle import port

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _graph(U, I, E, seed, hub=0):
    from arlib_b200.graph import DeviceGraph
    rng = np.random.default_rng(seed)
    u = rng.integers(0, U, E)
    i = rng.integers(0, I, E)
    if hub:                                                  # one user and one item row with `hub` entries each
        u[:hub] = 0
        i[:hub] = rng.permutation(I)[:hub]
        i[hub:2 * hub] = 1
        u[hub:2 * hub] = rng.permutation(U)[:hub]
    key = np.unique(u.astype(np.int64) * I + i)
    u, i = key // I, key % I
    return DeviceGraph.from_dataloader_adj(port.bipartite_adjacency(u, i, U, I), DEV), u, i


def _bits(t):
    return t.cpu().numpy().view(np.uint32)


@pytest.mark.parametrize("d", [16, 64, 128])
@pytest.mark.parametrize("L", [1, 2, 3, 6])
def test_acc_terms_equal_running_layer_sum(d, L):
    from arlib_b200 import ops
    U, I = 500, 700
    g0, _, _ = _graph(U, I, 12000, 3, hub=400)
    g = g0.replan(64, 64)                                    # hub rows cut into several segments
    n = U + I
    sel = np.random.default_rng(1).choice(n, 300, replace=False)
    flags = np.zeros(((n + 31) // 32) * 32, dtype=np.uint8)
    flags[sel] = 1
    mask = torch.from_numpy(np.packbits(flags, bitorder="little").view(np.int32).copy()).to(DEV)
    rows = torch.from_numpy(sel).to(DEV)
    E = [torch.randn(n, d, device=DEV)]
    for _ in range(L - 1):
        E.append(torch.empty(n, d, device=DEV))
        ops.spmm(g, E[-2], Y=E[-1])
    # reference: the running sum of forward_table
    ref = torch.empty(n, d, device=DEV)
    x = E[0]
    for k in range(1, L + 1):
        last = k == L
        y = None if last else torch.empty(n, d, device=DEV)
        ops.spmm(g, x, Y=y, acc_in=E[0] if k == 1 else ref, acc_out=ref, acc_div=float(L + 1) if last else 1.0,
                 row_mask=mask if last else None)
        x = y
    out = torch.full((n, d), 7.0, device=DEV)
    ops.spmm(g, E[-1], acc_out=out, acc_div=float(L + 1), acc_terms=E, row_mask=mask)
    assert np.array_equal(_bits(out[rows]), _bits(ref[rows]))
    others = torch.ones(n, dtype=torch.bool, device=DEV)
    others[rows] = False
    assert bool((out[others] == 7.0).all())                  # rows outside the mask are not written


def _engine(L, worklists, batch_rows_sum):
    from arlib_b200.engine import LightGCNEngine, DeviceTrainSet

    class RunningSumEngine(LightGCNEngine):
        """the running layer sum at every row in every layer (forward_table), as before the batch-rows sum"""
        def _forward_batch(self, row_mask, worklist):
            return self.forward_table(row_mask=row_mask, worklist=worklist)

    U, I = 600, 800
    g, u, i = _graph(U, I, 12000, 5, hub=400)
    gen = torch.Generator().manual_seed(7)
    table = ((torch.rand(U + I, 64, generator=gen) - 0.5) * 0.2).to(DEV)
    eng = (LightGCNEngine if batch_rows_sum else RunningSumEngine)(g, table, U, L, 0.01, 1e-4, 512, len(u))
    if not worklists:
        eng.wl = None
    eng.sample_epoch(DeviceTrainSet.from_arrays(u, i, U, I, DEV), seed=11, epoch=0)
    return eng


@pytest.mark.parametrize("L", [1, 2, 3, 4, 9])
@pytest.mark.parametrize("use_graph", [False, True])
@pytest.mark.parametrize("worklists", [False, True])
def test_engine_epoch_equals_running_layer_sum_step(L, use_graph, worklists):
    res = []
    for batch_rows_sum in (False, True):
        eng = _engine(L, worklists, batch_rows_sum)
        out = eng.run_steps(0, eng.n_batches, use_graph=use_graph).clone()
        torch.cuda.synchronize()
        res.append([out, eng.E0.clone(), eng.m.clone(), eng.v.clone()])
        assert len(eng.fw) == (max(2, L - 1) if L > 1 else 0)
        assert int(eng.G.count_nonzero()) == 0
        del eng                                              # its captured graph is released before the next capture
        gc.collect()
        torch.cuda.synchronize()
    for a, b in zip(*res):
        assert np.array_equal(_bits(a), _bits(b))
