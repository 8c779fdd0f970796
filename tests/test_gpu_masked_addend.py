"""GPU parity of the gradient reads gated by the batch bitmap (addend_mask): the backward layers of the LightGCN step read
G only at the batch's rows, add +0.0f elsewhere, and the fused optimizer puts every batch row of G back to +0.0f.  Outputs
must equal the unmasked launch bit for bit, and a training epoch must not change by a bit."""
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


def _mask(n, sel):
    flags = np.zeros(((n + 31) // 32) * 32, dtype=np.uint8)
    flags[sel] = 1
    return torch.from_numpy(np.packbits(flags, bitorder="little").view(np.int32).copy()).to(DEV)


def _sparse_table(n, d, sel, gen):
    """rows `sel` random (some of them -0.0 / +0.0 exactly), every other row +0.0"""
    G = torch.zeros(n, d, device=DEV)
    rows = torch.from_numpy(sel).to(DEV)
    G[rows] = torch.randn(len(sel), d, generator=gen).to(DEV)
    G[rows[:7]] = -0.0
    G[rows[7:11], :d // 2] = -0.0
    return G, rows


@pytest.mark.parametrize("d", [16, 64, 128])
@pytest.mark.parametrize("col_masked", [False, True])
def test_masked_addend_equals_unmasked(d, col_masked):
    """the middle backward layer (Y = A H + G) and the first one (column-masked): same bits with and without the mask,
    also at rows of G that hold -0.0 and where every gathered row of X is -0.0"""
    from arlib_b200 import ops
    U, I = 500, 700
    g0, _, _ = _graph(U, I, 12000, 3, hub=400)
    g = g0.replan(64, 64)                                    # hub rows cut into several segments
    n = U + I
    gen = torch.Generator().manual_seed(d)
    sel = np.random.default_rng(2).choice(n, 150, replace=False)
    sel[0] = 0                                               # a hub row in the bitmap
    mask = _mask(n, sel)
    G, _ = _sparse_table(n, d, sel, gen)
    H = G.clone() if col_masked else torch.randn(n, d, generator=gen).to(DEV)
    H[: n // 2] = -0.0
    cm = mask if col_masked else None
    ref = torch.full((n, d), 7.0, device=DEV)
    out = torch.full((n, d), 7.0, device=DEV)
    ops.spmm(g, H, Y=ref, addend=G, col_mask=cm)
    ops.spmm(g, H, Y=out, addend=G, col_mask=cm, addend_mask=mask)
    assert np.array_equal(_bits(out), _bits(ref))


@pytest.mark.parametrize("d", [16, 64, 128])
@pytest.mark.parametrize("col_masked", [False, True])
def test_masked_acc_in_fused_adam_equals_unmasked(d, col_masked):
    """the last backward layer: (acc_in + A H) / (L + 1) into the fused Adam update, acc_in read only at the bitmap's rows;
    p / m / v bit-identical to the unmasked launch, and every row of the bitmap of acc_in is +0.0 afterwards"""
    from arlib_b200 import ops
    U, I = 500, 700
    g0, _, _ = _graph(U, I, 12000, 4, hub=400)
    g = g0.replan(64, 64)
    n = U + I
    gen = torch.Generator().manual_seed(100 + d)
    sel = np.random.default_rng(3).choice(n, 150, replace=False)
    mask = _mask(n, sel)
    G, rows = _sparse_table(n, d, sel, gen)
    H = G.clone() if col_masked else torch.randn(n, d, generator=gen).to(DEV)
    cm = mask if col_masked else None
    p0 = torch.randn(n, d, generator=gen).to(DEV)
    m0 = torch.randn(n, d, generator=gen).to(DEV) * 0.01
    v0 = torch.rand(n, d, generator=gen).to(DEV) * 0.01
    coefs = torch.zeros(2, device=DEV)
    step = torch.zeros(1, dtype=torch.int32, device=DEV)
    ops.adam_coefs(step, coefs, 0.01)
    res = []
    for amask in (None, mask):
        p, m, v, Gk = p0.clone(), m0.clone(), v0.clone(), G.clone()
        X = Gk if col_masked else H                          # column-masked: the gathered table is G itself (L = 1)
        ops.spmm(g, X, acc_in=Gk, acc_div=4.0, col_mask=cm, adam=(p, m, v, coefs, 0.9, 0.999, 1e-8),
                 zero_acc_in=not col_masked, addend_mask=amask)
        res.append((p, m, v, Gk))
    for a, b in zip(res[0][:3], res[1][:3]):
        assert np.array_equal(_bits(a), _bits(b))
    if not col_masked:
        assert np.array_equal(_bits(res[1][3]), np.zeros((n, d), np.uint32))   # +0.0 everywhere, -0.0 rows included


def _engine(L, worklists, addend_mask):
    from arlib_b200 import ops
    from arlib_b200.engine import LightGCNEngine, DeviceTrainSet

    class UnmaskedEngine(LightGCNEngine):
        """G read at every row and separate backward tables, as before the batch bitmap gated the gradient reads"""
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            self.bw = [torch.empty_like(self.E0), torch.empty_like(self.E0)] if self.L > 1 else []

        def _launch_step(self, b):
            spmm = ops.spmm

            def unmasked(*a, **k):
                k.pop("addend_mask", None)
                return spmm(*a, **k)
            ops.spmm = unmasked
            try:
                super()._launch_step(b)
            finally:
                ops.spmm = spmm

    U, I = 600, 800
    g, u, i = _graph(U, I, 12000, 5, hub=400)
    gen = torch.Generator().manual_seed(7)
    table = ((torch.rand(U + I, 64, generator=gen) - 0.5) * 0.2).to(DEV)
    eng = (LightGCNEngine if addend_mask else UnmaskedEngine)(g, table, U, L, 0.01, 1e-4, 100, len(u))
    assert 12 * eng.B <= eng.N                               # the step reads G at the batch's rows only
    if not worklists:
        eng.wl = None
    eng.sample_epoch(DeviceTrainSet.from_arrays(u, i, U, I, DEV), seed=11, epoch=0)
    return eng


@pytest.mark.parametrize("L", [1, 2, 3, 4])
@pytest.mark.parametrize("use_graph", [False, True])
@pytest.mark.parametrize("worklists", [False, True])
def test_engine_epoch_equals_unmasked_step(L, use_graph, worklists):
    res = []
    for addend_mask in (False, True):
        eng = _engine(L, worklists, addend_mask)
        if addend_mask and L > 1:
            assert eng.bw[0] is eng.fw[1] and eng.bw[1] is eng.fw[0]
        if use_graph:
            out = eng.run_steps(0, eng.n_batches, use_graph=True).clone()
            torch.cuda.synchronize()
            assert int(eng.G.count_nonzero()) == 0
        else:
            for b in range(eng.n_batches):                   # G is all zero after every step (all +0.0 when masked)
                eng.run_steps(b, 1, use_graph=False)
                torch.cuda.synchronize()
                assert int(eng.G.count_nonzero()) == 0
                assert not addend_mask or not _bits(eng.G).any()
            out = eng.out4[:eng.n_batches].clone()
        res.append([out, eng.E0.clone(), eng.m.clone(), eng.v.clone(), eng.forward_table().clone()])
        del eng                                              # its captured graph is released before the next capture
        gc.collect()
        torch.cuda.synchronize()
    for a, b in zip(*res):
        assert np.array_equal(_bits(a), _bits(b))
