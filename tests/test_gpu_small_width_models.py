"""The four drop-in recommenders at emb_size 8 and 16 on the ml-100k golden rows: one epoch on the fused path and on the
reference-shaped loop (``fused=False``), against the oracle trainers in float64 from the same initial tables, the same
host-sampled triples (the reference's, frozen in the golden file) and, for SimGCL / XSimGCL, the same noise tables."""
import copy
import io
import os
import random
import types

import numpy as np
import pytest
import torch

from oracle import port

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
WIDTHS = [8, 16]


def _args(**kw):
    base = dict(topK="50", emb_size=64, n_layers=2, batch_size=2048, lRate=0.005, reg=1e-4, maxEpoch=1, seed=2018,
                sampler="host", model_name="LightGCN")
    base.update(kw)
    return types.SimpleNamespace(**base)


def _rec(name, golden_rows, d, **kw):
    import importlib
    from arlib_b200.util.DataLoader import DataLoader
    train, test = golden_rows
    random.seed(2018); np.random.seed(2018); torch.manual_seed(2018)
    data = DataLoader.from_rows([list(r) for r in train], (), test)
    cls = getattr(importlib.import_module("arlib_b200.recommender." + name), name)
    return cls(_args(model_name=name, emb_size=d, **kw), data)


def _adj(golden):
    U, I = golden["user_names"].shape[0], golden["item_names"].shape[0]
    return port.normalize_graph_mat(port.bipartite_adjacency(golden["train_u"].astype(np.int64),
                                                             golden["train_i"].astype(np.int64), U, I))


def _batches(golden):
    off = np.concatenate([[0], np.cumsum(golden["batch_len"])])
    for b in range(len(off) - 1):
        sl = slice(off[b], off[b + 1])
        yield golden["batch_u"][sl].tolist(), golden["batch_i"][sl].tolist(), golden["batch_j"][sl].tolist()


def _f64(tr):
    """an oracle trainer built from float64 tables runs its propagation in float64 too"""
    tr.adj = tr.adj.double()
    return tr


def _init(rec):
    e = rec.model.embedding_dict
    return e["user_emb"].detach().cpu().clone(), e["item_emb"].detach().cpu().clone()


def _noise(n, d, seed):
    gen = torch.Generator().manual_seed(seed)
    return lambda: torch.rand(n, d, generator=gen)


def _assert_close_to_fp64(got_u, got_i, want_u, want_i, what):
    """1e-4 relative; Adam's 1 / (sqrt(v) + 1e-8) amplifies rounding on elements with gradients below ~1e-8 (see
    test_gpu_golden_models.py), so failing that, the bulk of the table within 1e-4 and no element beyond 1e-3"""
    got = torch.cat([got_u, got_i]).double().cpu()
    want = torch.cat([want_u, want_i]).double().cpu()
    diff = (got - want).abs() / float(want.abs().max())
    frac_off, worst = float((diff > 1e-4).double().mean()), float(diff.max())
    print("%s vs the float64 oracle: worst %.2e, %.2e of the table beyond 1e-4" % (what, worst, frac_off))
    assert worst < 1e-4 or (frac_off < 1e-3 and worst < 1e-3), (worst, frac_off)


def _check_metrics_and_sets(rec, fu, fi):
    """metrics of the trained drop-in (our evaluator) vs the oracle's full-rank test on the oracle's final tables
    within 1e-3; top-50 sets equal except at counted boundary near-ties"""
    rec_list, measure = rec.test()
    ref_list, ref_measure = port.full_rank_test(rec.data, fu.float(), fi.float(), 50, [50])
    for a, b in zip(measure[1:], ref_measure[1:]):
        assert a.split(":")[0] == b.split(":")[0]
        assert abs(float(a.split(":")[1]) - float(b.split(":")[1])) < 1e-3, (a, b)
    near = 0
    for u, items in ref_list.items():
        got, want = set(p[0] for p in rec_list[u]), set(p[0] for p in items)
        if got == want:
            continue
        near += 1
        kth = min(s for _, s in items)
        uid = rec.data.user[u]
        s = (fu[uid].double() @ fi.double().T).numpy()
        tol = 1e-4 * max(1e-30, abs(kth)) + 1e-6
        for name in got ^ want:
            assert abs(s[rec.data.item[name]] - kth) <= tol, "user %s: item %s is not a boundary near-tie" % (u, name)
    print("top-50 sets: %d of %d users differ at a boundary near-tie" % (near, len(ref_list)))
    assert near <= 0.02 * len(ref_list)


@pytest.mark.parametrize("d", WIDTHS)
@pytest.mark.parametrize("fused", [True, False])
def test_lightgcn_epoch(golden, golden_rows, d, fused):
    rec = _rec("LightGCN", golden_rows, d, fused=fused)
    iu, ii = _init(rec)
    tr = _f64(port.LightGCNTrainer(_adj(golden), iu.double(), ii.double(), 2, 0.005, 1e-4))
    for b in _batches(golden):
        tr.step(*b)
    rec.train()
    e = rec.model.embedding_dict
    _assert_close_to_fp64(e["user_emb"].detach(), e["item_emb"].detach(), tr.user_emb.detach(), tr.item_emb.detach(),
                          "LightGCN d=%d fused=%s" % (d, fused))
    with torch.no_grad():
        fu, fi = tr.forward()
    _check_metrics_and_sets(rec, fu, fi)


@pytest.mark.parametrize("d", WIDTHS)
def test_lightgcn_callers_adam_is_handed_over(golden, golden_rows, d):
    """the caller's torch.optim.Adam drives the fused engine and gets its state back: a second epoch continues it"""
    rec = _rec("LightGCN", golden_rows, d, maxEpoch=2)
    iu, ii = _init(rec)
    opt = torch.optim.Adam(rec.model.parameters(), lr=0.005)
    tr = _f64(port.LightGCNTrainer(_adj(golden), iu.double(), ii.double(), 2, 0.005, 1e-4))
    for b in _batches(golden):
        tr.step(*b)
    rec.train(optimizer=opt, Epoch=1)
    e = rec.model.embedding_dict
    _assert_close_to_fp64(e["user_emb"].detach(), e["item_emb"].detach(), tr.user_emb.detach(), tr.item_emb.detach(),
                          "LightGCN d=%d caller's Adam" % d)
    n_batches = len(golden["batch_len"])
    st = opt.state[e["user_emb"]]
    assert int(st["step"]) == n_batches and float(st["exp_avg_sq"].abs().max()) > 0
    # the state the optimizer holds now is the engine's: one more plain torch step moves from it like Adam does
    ou = tr.opt.state[tr.user_emb]
    assert torch.allclose(st["exp_avg"].double().cpu(), ou["exp_avg"], rtol=1e-3, atol=1e-9)


@pytest.mark.parametrize("d", WIDTHS)
def test_lightgcn_adjgrad_deepcopy_and_save(golden_rows, d):
    rec = _rec("LightGCN", golden_rows, d)
    mat = rec.train(requires_adjgrad=True)
    assert mat.shape == (rec.data.user_num, rec.data.item_num)
    assert float(mat.abs().max()) > 0
    rec2 = copy.deepcopy(rec)
    assert torch.equal(rec2.user_emb.cpu(), rec.user_emb.cpu())
    buf = io.BytesIO()
    torch.save(rec, buf)
    buf.seek(0)
    rec3 = torch.load(buf, weights_only=False)
    assert torch.equal(rec3.item_emb.cpu(), rec.item_emb.cpu())


@pytest.mark.parametrize("d", WIDTHS)
@pytest.mark.parametrize("fused", [True, False])
def test_ngcf_epoch(golden, golden_rows, d, fused):
    rec = _rec("NGCF", golden_rows, d, fused=fused)
    m = rec.model
    iu, ii = _init(rec)
    w1 = [m.W["w1_%d" % k].detach().cpu().double() for k in range(2)]
    w2 = [m.W["w2_%d" % k].detach().cpu().double() for k in range(2)]
    tr = _f64(port.NGCFTrainer(_adj(golden), iu.double(), ii.double(), w1, w2, 0.005, 1e-4))
    for b in _batches(golden):
        tr.step(*b)
    rec.train()
    e = m.embedding_dict
    _assert_close_to_fp64(e["user_emb"].detach(), e["item_emb"].detach(), tr.user_emb.detach(), tr.item_emb.detach(),
                          "NGCF d=%d fused=%s" % (d, fused))
    wg = torch.cat([m.W["w%d_%d" % (a, k)].detach().cpu().double().reshape(-1) for a in (1, 2) for k in range(2)])
    ww = torch.cat([w.detach().reshape(-1) for w in (tr.w1[0], tr.w1[1], tr.w2[0], tr.w2[1])])
    assert float((wg - ww).abs().max() / ww.abs().max()) < 1e-4
    with torch.no_grad():
        fu, fi = tr.forward()
    _check_metrics_and_sets(rec, fu, fi)


def _contrastive_oracle(kind, golden, iu, ii, d, seed):
    U, I = iu.shape[0], ii.shape[0]
    draw = _noise(U + I, d, seed)
    if kind == "simgcl":
        tr = port.SimGCLTrainer(_adj(golden), iu, ii, 2, 0.1, 0.2, 0.005, 1e-4, draw, tau=0.2, dtype=torch.float64)
    else:
        tr = port.XSimGCLTrainer(_adj(golden), iu, ii, 2, 0.1, 0.2, 1, 0.005, 1e-4, draw, tau=0.1, dtype=torch.float64)
    for b in _batches(golden):
        tr.step(*b)
    return tr


@pytest.mark.parametrize("d", WIDTHS)
@pytest.mark.parametrize("name", ["SimGCL", "XSimGCL"])
def test_contrastive_reference_loop_epoch(golden, golden_rows, d, name):
    rec = _rec(name, golden_rows, d, fused=False)
    iu, ii = _init(rec)
    draw = _noise(iu.shape[0] + ii.shape[0], d, 77 + d)
    rec.model.noise_source = lambda k, like: draw().to(like.device)
    rec.train()
    tr = _contrastive_oracle(name.lower(), golden, iu, ii, d, 77 + d)
    e = rec.model.embedding_dict
    _assert_close_to_fp64(e["user_emb"].detach(), e["item_emb"].detach(), tr.user_emb.detach(), tr.item_emb.detach(),
                          "%s d=%d reference-shaped loop" % (name, d))
    with torch.no_grad():
        out = tr.forward()
    _check_metrics_and_sets(rec, out[0], out[1])


@pytest.mark.parametrize("d", WIDTHS)
@pytest.mark.parametrize("kind", ["simgcl", "xsimgcl"])
def test_contrastive_fused_engine_epoch(golden, golden_rows, d, kind):
    """the fused engine (shared first layer, one backward propagation, Adam in the last SpMM) with injected noise
    tables, stepped through the golden triples"""
    from arlib_b200.engine import ContrastiveEngine
    from arlib_b200.graph import DeviceGraph
    U, I = golden["user_names"].shape[0], golden["item_names"].shape[0]
    gen = torch.Generator().manual_seed(1000 + d)
    iu = torch.nn.init.xavier_uniform_(torch.empty(U, d), generator=gen)
    ii = torch.nn.init.xavier_uniform_(torch.empty(I, d), generator=gen)
    adj = port.bipartite_adjacency(golden["train_u"].astype(np.int64), golden["train_i"].astype(np.int64), U, I)
    graph = DeviceGraph.from_dataloader_adj(adj, DEV)
    table = torch.cat([iu, ii]).to(DEV)
    T = golden["batch_u"].shape[0]
    draw = _noise(U + I, d, 5 + d)
    passes = (0,) if kind == "xsimgcl" else (1, 2)
    tabs = {(p, k): torch.empty((U + I, d), device=DEV) for p in passes for k in (1, 2)}
    eng = ContrastiveEngine(graph, table, U, kind, 2, 0.1, 0.2, 0.1 if kind == "xsimgcl" else 0.2, 0.005, 1e-4, 2048, T,
                            layer_cl=1, noise_tables=tabs)
    eng.set_triples(golden["batch_u"], golden["batch_i"], golden["batch_j"])
    for b in range(eng.n_batches):
        for p in passes:                          # reference order: pass 1 layers 1..L, then pass 2 layers 1..L
            for k in (1, 2):
                tabs[(p, k)].copy_(draw())
        eng.run_steps(b, 1, use_graph=False)
    tr = _contrastive_oracle(kind, golden, iu, ii, d, 5 + d)
    _assert_close_to_fp64(table[:U], table[U:], tr.user_emb.detach(), tr.item_emb.detach(),
                          "%s d=%d fused engine" % (kind, d))
    with torch.no_grad():
        out = tr.forward()
    F = eng.forward_table(out=torch.empty_like(table)).cpu().double()
    assert float((F - torch.cat([out[0], out[1]])).abs().max() / torch.cat([out[0], out[1]]).abs().max()) < 5e-4


@pytest.mark.parametrize("d", WIDTHS)
@pytest.mark.parametrize("name", ["SimGCL", "XSimGCL"])
def test_contrastive_class_fused_path_trains(golden_rows, d, name):
    """the class's fused path (Philox noise drawn in the SpMM epilogue) at the small widths: it trains and evaluates"""
    rec = _rec(name, golden_rows, d)
    iu, _ = _init(rec)
    rec.train()
    moved = rec.model.embedding_dict["user_emb"].detach().cpu()
    assert torch.isfinite(moved).all() and not torch.equal(moved, iu)
    _, measure = rec.test()
    assert float(measure[1].split(":")[1]) > 0.0                    # hit ratio after one epoch
