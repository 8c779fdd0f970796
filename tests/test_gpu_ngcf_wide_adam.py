"""NGCF at d = 128 and 256 on the fused dense layer kernels (csrc/ngcf.cu) and NGCFEngine, and NGCF.train() with the
caller's torch.optim.Adam at every width: against float64 autograd of the layer expression, and one ml-100k epoch against
the float64 oracle trainer (oracle.port.NGCFTrainer) on the reference's frozen triples."""
import copy
import os
import random
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import port

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ALL_WIDTHS = [8, 16, 32, 64, 128, 256]
WIDE = [128, 256]
LR, BETAS, EPS = 0.003, (0.8, 0.99), 1e-7          # not Adam's defaults: the engine must take the caller's


# ---- helpers copied from test_gpu_small_width_models.py
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


def _assert_close_to_fp64(got_u, got_i, want_u, want_i, what):
    """1e-4 relative; Adam's 1 / (sqrt(v) + 1e-8) amplifies rounding on elements with gradients below ~1e-8 (see
    test_gpu_golden_models.py), so failing that, the bulk of the table within 1e-4 and no element beyond 1e-3"""
    got = torch.cat([got_u, got_i]).double().cpu()
    want = torch.cat([want_u, want_i]).double().cpu()
    diff = (got - want).abs() / float(want.abs().max())
    frac_off, worst = float((diff > 1e-4).double().mean()), float(diff.max())
    print("%s vs the float64 oracle: worst %.2e, %.2e of the table beyond 1e-4" % (what, worst, frac_off))
    assert worst < 1e-4 or (frac_off < 1e-3 and worst < 1e-3), (worst, frac_off)


# ---- this file's own
def _rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / b.abs().max())


def _flat_w(ws):
    return torch.cat([w.detach().reshape(-1).double().cpu() for w in ws])


@pytest.mark.parametrize("n", [1, 64, 333, 1000])
@pytest.mark.parametrize("d", WIDE)
def test_wide_dense_layer_matches_autograd(d, n):
    """E' = leaky_relu([P + E | P * E] [W1 ; W2]) and its gradients w.r.t. P, E (direct) and W, vs torch autograd in
    float64 of the same expression, as tests/test_gpu_ngcf.py does at d <= 64.  Its bounds (2e-6 forward, 3e-6 backward)
    are scaled by sqrt(d / 64): the forward chains are K = 2d long, those of dP / dE_direct K = d, and the rounding
    error of a K-term fp32 dot product grows like sqrt(K)."""
    from arlib_b200 import ops
    from arlib_b200.engine import NGCFEngine
    gen = torch.Generator().manual_seed(n + d)
    P = torch.randn(n, d, generator=gen) * 0.3
    E = torch.randn(n, d, generator=gen) * 0.3
    W = torch.randn(2 * d, d, generator=gen) / d ** 0.5
    dOut = torch.randn(n, d, generator=gen)
    acc = torch.randn(n, d, generator=gen)
    Pd, Ed, Wd = (t.double().requires_grad_(True) for t in (P, E, W))
    Z = (Pd + Ed) @ Wd[:d] + (Pd * Ed) @ Wd[d:]
    Y = F.leaky_relu(Z, 0.01)
    Y.backward(dOut.double())
    s = (d / 64) ** 0.5
    Pc, Ec, Wc = P.to(DEV), E.to(DEV), W.to(DEV)
    Yc = torch.empty_like(Pc)
    mean = torch.empty_like(Pc)
    ops.ngcf_dense_forward(Pc, Ec, Wc, Yc, acc_in=acc.to(DEV), acc_out=mean, acc_div=3.0)
    errs = {"fwd": _rel(Yc, Y.detach()), "mean": _rel(mean, (acc.double() + Y.detach()) / 3.0)}
    dP, dE = torch.empty_like(Pc), torch.empty_like(Pc)
    part = torch.empty((NGCFEngine.N_PARTIALS[d], 2 * d * d), device=DEV)
    dW = torch.empty((2 * d, d), device=DEV)
    WT = Wc.t().contiguous()
    ops.ngcf_dense_backward(dOut.to(DEV), Yc, Pc, Ec, WT, dP, dE, part, dW)
    errs.update(dP=_rel(dP, Pd.grad), dE=_rel(dE, Ed.grad), dW=_rel(dW, Wd.grad))
    print("d=%d n=%d:" % (d, n), {k: "%.2e" % v for k, v in errs.items()})
    assert errs["fwd"] < 2e-6 * s and errs["mean"] < 2e-6 * s
    assert errs["dP"] < 3e-6 * s and errs["dE"] < 3e-6 * s
    assert errs["dW"] < 3e-6                             # K = n: the chains of the d = 64 test
    dW2 = torch.empty_like(dW)
    ops.ngcf_dense_backward(dOut.to(DEV), Yc, Pc, Ec, WT, dP, dE, part, dW2)
    assert torch.equal(dW, dW2)                          # partials are reduced in slice order
    # another slice count changes only where the dW chains restart
    part3 = torch.empty((3, 2 * d * d), device=DEV)
    dW3 = torch.empty_like(dW)
    ops.ngcf_dense_backward(dOut.to(DEV), Yc, Pc, Ec, WT, dP, dE, part3, dW3)
    assert _rel(dW3, Wd.grad) < 3e-6


def _engine_and_oracle(golden, golden_rows, d, eps=1e-8):
    """NGCFEngine on the recommender's own initial tables and weights at width d (those of test_ngcf_epoch), and the
    float64 oracle trainer from the same values, both with Adam's eps = ``eps``"""
    from arlib_b200.engine import NGCFEngine
    from arlib_b200.graph import DeviceGraph
    rec = _rec("NGCF", golden_rows, d)
    m = rec.model
    iu, ii = _init(rec)
    w1 = [m.W["w1_%d" % k].detach().cpu() for k in range(2)]
    w2 = [m.W["w2_%d" % k].detach().cpu() for k in range(2)]
    U, I = golden["user_names"].shape[0], golden["item_names"].shape[0]
    adj = port.bipartite_adjacency(golden["train_u"].astype(np.int64), golden["train_i"].astype(np.int64), U, I)
    table = torch.cat([iu, ii]).to(DEV)
    W = torch.stack([torch.cat([w1[k], w2[k]], 0) for k in range(2)], 0).contiguous().to(DEV)
    eng = NGCFEngine(DeviceGraph.from_dataloader_adj(adj, DEV), table, W, U, 0.005, 1e-4, 2048, golden["batch_u"].shape[0],
                     adam_eps=eps)
    eng.set_triples(golden["batch_u"], golden["batch_i"], golden["batch_j"])
    tr = _f64(port.NGCFTrainer(_adj(golden), iu.double(), ii.double(), [w.double() for w in w1], [w.double() for w in w2],
                               0.005, 1e-4))
    tr.opt = torch.optim.Adam([tr.user_emb, tr.item_emb] + [w for k in range(2) for w in (tr.w1[k], tr.w2[k])], lr=0.005,
                              eps=eps)
    return eng, table, W, tr, U


@pytest.mark.parametrize("use_graph", [False, True])
@pytest.mark.parametrize("d", WIDE)
def test_wide_engine_epoch_matches_the_fp64_oracle(golden, golden_rows, d, use_graph):
    """one epoch of NGCFEngine on the reference's ml-100k triples against oracle.port.NGCFTrainer in float64 from the
    same initial tables and weights; G is all zero afterwards.  Adam's eps is 1e-7 here.  With the default 1e-8, an
    element whose gradient stays near 1e-8 moves by up to lr per step in a direction set by rounding, and at these
    widths enough elements sit there that a free-running epoch is not a well-conditioned quantity: measured 1.7e-2
    (d = 128) and 1.0e-3 (d = 256) from float64 with per-batch losses within 1.7e-7, and the same fused formulation in
    fp32 on the CPU also leaves the 1e-4 rule at d = 128 from another starting point.  The default eps is checked step
    by step (test_wide_engine_steps_match_fp64_steps)."""
    eng, table, W, tr, U = _engine_and_oracle(golden, golden_rows, d, eps=1e-7)
    losses = eng.run_steps(0, use_graph=use_graph)[:, 0].cpu().numpy()
    want = np.array([tr.step(*b) for b in _batches(golden)])
    print("d=%d per-batch loss: worst relative difference %.2e" % (d, float(np.max(np.abs(losses / want - 1)))))
    np.testing.assert_allclose(losses, want, rtol=2e-5)
    _assert_close_to_fp64(table[:U], table[U:], tr.user_emb.detach(), tr.item_emb.detach(),
                          "NGCFEngine d=%d graph=%s tables" % (d, use_graph))
    got_w = _flat_w([W[k, :d] for k in range(2)] + [W[k, d:] for k in range(2)])
    want_w = _flat_w(tr.w1 + tr.w2)
    _assert_close_to_fp64(got_w, got_w[:0], want_w, want_w[:0], "NGCFEngine d=%d graph=%s weights" % (d, use_graph))
    assert int(eng.step_dev) == len(golden["batch_len"])
    assert int((eng.G != 0).sum()) == 0


@pytest.mark.parametrize("d", WIDE)
def test_wide_engine_steps_match_fp64_steps(golden, golden_rows, d):
    """teacher-forced: before every step of the epoch, a float64 oracle starts from the engine's own parameters and Adam
    moments and takes the same step.  One step is well conditioned where an epoch need not be.  The looser bound of the
    first steps is Adam's: while v is small, m / (sqrt(v) + eps) is close to sign(g) on elements with gradients near eps
    (measured: up to 3.6e-5 at step 0, below 1e-6 from step 3 on)."""
    eng, table, W, _, U = _engine_and_oracle(golden, golden_rows, d)
    nadj = _adj(golden)
    for b, bt in enumerate(_batches(golden)):
        tb, Wb = table.cpu().double(), W.cpu().double()
        m, v, Wm, Wv = (x.cpu().double() for x in (eng.m, eng.v, eng.Wm, eng.Wv))
        step = int(eng.step_dev)
        tr = _f64(port.NGCFTrainer(nadj, tb[:U], tb[U:], [Wb[k, :d] for k in range(2)], [Wb[k, d:] for k in range(2)],
                                   0.005, 1e-4))
        ps = [tr.user_emb, tr.item_emb, tr.w1[0], tr.w2[0], tr.w1[1], tr.w2[1]]
        mv = [(m[:U], v[:U]), (m[U:], v[U:])] + [(Wm[k, h * d:(h + 1) * d], Wv[k, h * d:(h + 1) * d])
                                                 for k in range(2) for h in range(2)]
        if step:
            for p, (a, c) in zip(ps, mv):
                tr.opt.state[p] = {'step': torch.tensor(float(step)), 'exp_avg': a.clone(), 'exp_avg_sq': c.clone()}
        want_loss = tr.step(*bt)
        loss = float(eng.run_steps(b, 1, use_graph=False)[0, 0])
        errs = {"loss": abs(loss / want_loss - 1),
                "table": _rel(table, torch.cat([tr.user_emb.detach(), tr.item_emb.detach()])),
                "W": _rel(W, torch.stack([torch.cat([tr.w1[k].detach(), tr.w2[k].detach()], 0) for k in range(2)])),
                "m": _rel(eng.m, torch.cat([tr.opt.state[tr.user_emb]["exp_avg"], tr.opt.state[tr.item_emb]["exp_avg"]]))}
        assert errs["loss"] < 1e-6 and errs["m"] < 1e-5, (b, errs)
        bound = 1e-4 if b < 3 else 1e-5
        assert errs["table"] < bound and errs["W"] < bound, (b, errs)
    assert int((eng.G != 0).sum()) == 0


def _spy(monkeypatch):
    from arlib_b200.recommender.NGCF import NGCF
    calls = []
    orig = NGCF._train_fused
    monkeypatch.setattr(NGCF, "_train_fused", lambda self, *a, **k: (calls.append(self), orig(self, *a, **k))[1])
    return calls


def _pairs(rec, tr):
    """(model parameter, the oracle's parameter) for all 2 + 2L parameters"""
    m, L = rec.model, rec.model.layers
    out = [(m.embedding_dict["user_emb"], tr.user_emb), (m.embedding_dict["item_emb"], tr.item_emb)]
    for k in range(L):
        out += [(m.W["w1_%d" % k], tr.w1[k]), (m.W["w2_%d" % k], tr.w2[k])]
    return out


@pytest.mark.parametrize("d", ALL_WIDTHS)
def test_callers_adam_drives_the_unified_fused_loop(golden, golden_rows, monkeypatch, d):
    """attack/White/CLeaR.py:145-146 on an NGCF victim: ``train(Epoch=1, optimizer=torch.optim.Adam(model.parameters(),
    ...))`` runs on the fused engine with the optimizer's lr / betas / eps, ends one epoch within the float64 oracle's
    rule, and hands every parameter's Adam state back: a second call continues it, and the caller's own step after that
    works.  Only one epoch is compared: NGCF parameters after many steps are not well conditioned (test_gpu_ngcf.py)."""
    calls = _spy(monkeypatch)
    rec = _rec("NGCF", golden_rows, d)
    m = rec.model
    iu, ii = _init(rec)
    w1 = [m.W["w1_%d" % k].detach().cpu().double() for k in range(2)]
    w2 = [m.W["w2_%d" % k].detach().cpu().double() for k in range(2)]
    opt = torch.optim.Adam(m.parameters(), lr=LR, betas=BETAS, eps=EPS)
    tr = _f64(port.NGCFTrainer(_adj(golden), iu.double(), ii.double(), w1, w2, LR, 1e-4))
    tr.opt = torch.optim.Adam([q for _, q in _pairs(rec, tr)], lr=LR, betas=BETAS, eps=EPS)
    for b in _batches(golden):
        tr.step(*b)
    rec.train(Epoch=1, optimizer=opt)
    assert calls == [rec]
    e = m.embedding_dict
    _assert_close_to_fp64(e["user_emb"].detach(), e["item_emb"].detach(), tr.user_emb.detach(), tr.item_emb.detach(),
                          "NGCF d=%d caller's Adam, tables" % d)
    pairs = _pairs(rec, tr)
    got_w, want_w = _flat_w([p for p, _ in pairs[2:]]), _flat_w([q for _, q in pairs[2:]])
    _assert_close_to_fp64(got_w, got_w[:0], want_w, want_w[:0], "NGCF d=%d caller's Adam, weights" % d)
    n_batches = len(golden["batch_len"])
    assert len(opt.state) == 2 + 2 * m.layers
    for p, q in pairs:
        st, so = opt.state[p], tr.opt.state[q]
        assert float(st["step"]) == n_batches
        assert _rel(st["exp_avg"], so["exp_avg"]) < 1e-3, _rel(st["exp_avg"], so["exp_avg"])
    rec.train(Epoch=1, optimizer=opt)                      # continues from the handed-back state
    assert len(calls) == 2
    assert all(float(opt.state[p]["step"]) == 2 * n_batches for p, _ in pairs)
    assert all(p is q for p, q in zip(opt.param_groups[0]["params"], m.parameters()))
    fu, fi = m()                                           # the caller keeps using its optimizer
    opt.zero_grad(); (fu.sum() + fi.sum()).backward(); opt.step()
    assert all(float(opt.state[p]["step"]) == 2 * n_batches + 1 for p, _ in pairs)
    assert all(torch.isfinite(p).all() for p, _ in pairs)


@pytest.mark.parametrize("d", [64, 256])
def test_other_optimizers_keep_the_reference_shaped_loop(golden_rows, monkeypatch, d):
    """a stale optimizer (built on tensors that are not the model's, as PGA.py:59-67 does), SGD, or Adam over the two
    tables only: the reference-shaped loop, which steps exactly what the optimizer holds"""
    calls = _spy(monkeypatch)
    rec = _rec("NGCF", golden_rows, d)
    m = rec.model
    e = m.embedding_dict
    stale = torch.optim.Adam([torch.nn.Parameter(torch.zeros(3, d, device=DEV)),
                              torch.nn.Parameter(torch.zeros(3, d, device=DEV))], lr=0.01)
    sgd = torch.optim.SGD(m.parameters(), lr=0.01)
    tables = torch.optim.Adam([e["user_emb"], e["item_emb"]], lr=0.01)
    for opt in (stale, sgd, tables):
        w0 = m.W["w1_0"].detach().clone()
        rec.train(Epoch=1, optimizer=opt)
        assert calls == []
        assert torch.equal(m.W["w1_0"].detach(), w0) == (opt is not sgd)   # only SGD holds the weights
    assert float(tables.state[e["user_emb"]]["step"]) == (len(rec.data.training_data) + 2047) // 2048
    assert all(p is not m.W["w1_0"] for p in tables.state)


def test_deepcopy_then_callers_adam_repacks_the_weights_on_the_engine(golden_rows, monkeypatch):
    """a deepcopy un-packs the weight views; the fused path re-packs them (weight_table) and the optimizer's parameter
    objects stay the model's, so the trained values and the handed-back state are on them"""
    calls = _spy(monkeypatch)
    rec = copy.deepcopy(_rec("NGCF", golden_rows, 128))
    m = rec.model
    opt = torch.optim.Adam(m.parameters(), lr=LR, betas=BETAS, eps=EPS)
    before = [p.detach().clone() for p in m.parameters()]
    rec.train(Epoch=1, optimizer=opt)
    assert calls == [rec]
    params = list(m.parameters())
    assert all(p is q for p, q in zip(opt.param_groups[0]["params"], params))
    assert all(not torch.equal(p.detach(), b) for p, b in zip(params, before))
    W = m.weight_table()
    assert W.data_ptr() == m.W["w1_0"].data_ptr() and torch.equal(W[1, 128:], m.W["w2_1"].detach())
    assert all(p in opt.state and float(opt.state[p]["step"]) > 0 for p in params)
