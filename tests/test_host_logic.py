"""CPU-side checks of host logic that needs no device: the util functions' CPU-tensor behaviour (the reference's
own torch expressions), the no-CPU-fallback guards of the fused entry points, and the header <-> ctypes mirror
of struct agcf_spmm_args."""
import ctypes
import os
import re
import types

import numpy as np
import pytest
import torch

from oracle import port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_losses_refuse_cpu_tensors():
    """VERDICT r1: util/loss.py's CPU branch of InfoNCE contradicted "no CPU fallback" -- it now raises like every
    other entry point; so does the fused BPR + L2 op.  (The plain torch expressions bpr_loss / l2_reg_loss stay
    device-agnostic: attacks import them for their own tensors, attack/Black/GTA.py:205.)"""
    from arlib_b200.util.loss import InfoNCE, bpr_l2_fused, bpr_loss, l2_reg_loss
    g = torch.Generator().manual_seed(0)
    a, b = torch.randn(40, 64, generator=g), torch.randn(40, 64, generator=g)
    with pytest.raises(RuntimeError):
        InfoNCE(a, b, 0.2)
    with pytest.raises(RuntimeError):
        bpr_l2_fused(a, b, [0, 1], [2, 3], [4, 5], 1e-4)
    assert torch.equal(bpr_loss(a, b, a), port.bpr_loss(a, b, a)) and torch.equal(l2_reg_loss(0.1, a, b), port.l2_reg_loss(0.1, a, b))


def test_device_only_entry_points_refuse_cpu_tensors():
    """No CPU fallback: the fused helpers raise instead of silently computing on the host."""
    from arlib_b200.util.algorithm import masked_score_topk
    from arlib_b200.util.metrics import AttackMetric
    with pytest.raises(TypeError):
        masked_score_topk(torch.randn(4, 64), torch.randn(9, 64), 3)
    rec = types.SimpleNamespace(user_emb=torch.randn(4, 64), item_emb=torch.randn(9, 64),
                                data=types.SimpleNamespace(user={"a": 0}, item={"x": 0}))
    with pytest.raises(TypeError):
        AttackMetric(rec, ["x"], [3]).hitRate()


def test_spmm_args_struct_mirrors_the_header_field_for_field():
    from arlib_b200 import _lib
    text = open(os.path.join(ROOT, "include", "agcf.h")).read()
    body = re.search(r"typedef struct agcf_spmm_args \{(.*?)\} agcf_spmm_args;", text, re.S).group(1)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        m = re.search(r"(\w+)(\[\d+\])?$", decl)
        names.append(m.group(1))
    assert names == [f[0] for f in _lib.SpmmArgs._fields_]
    # natural C alignment on LP64: pointers and uint64 8 bytes, int32 / float 4 bytes
    a = _lib.SpmmArgs()
    assert ctypes.sizeof(a) % 8 == 0
    assert _lib.SpmmArgs.noise_seed.offset % 8 == 0 and _lib.SpmmArgs.aux_Y.offset % 8 == 0


def test_fused_path_selection_and_sample_epoch_counter():
    from arlib_b200.recommender._base import GraphRecommender
    rec = GraphRecommender.__new__(GraphRecommender)
    rec.args = types.SimpleNamespace(batch_size=2048)
    assert rec._fused_ok()
    rec.args = types.SimpleNamespace(batch_size=6000)            # 3 B > 16384: the single-CTA grouping cannot sort it
    assert not rec._fused_ok()
    rec.args = types.SimpleNamespace(batch_size=2048, fused=False)
    assert not rec._fused_ok()
    assert [rec._next_sample_epoch() for _ in range(3)] == [0, 1, 2]      # keeps counting across train() calls


def test_unique_ids_like_reference_round_trips_through_float32():
    from arlib_b200.encoder import unique_ids_like_reference
    ids = [5, 3, 5, 2 ** 24 + 1, 3]
    want = torch.unique(torch.Tensor(ids).type(torch.long))          # recommender/SimGCL.py:213
    assert torch.equal(unique_ids_like_reference(ids, "cpu"), want)
    assert torch.equal(unique_ids_like_reference(torch.tensor(ids), "cpu"), want)
    assert int(want[-1]) == 2 ** 24                                    # the reference's float32 rounding is kept


def test_fusable_adam_recognises_exactly_the_plain_optimizer_over_the_models_parameters():
    """attack/White/CLeaR.py:59,145-146: ``torch.optim.Adam(model.parameters(), lr)`` handed to train().  Note that
    nn.ParameterDict sorts its keys, so model.parameters() yields item_emb BEFORE user_emb."""
    from arlib_b200.recommender._base import GraphRecommender
    m = torch.nn.Module()
    m.embedding_dict = torch.nn.ParameterDict({'user_emb': torch.nn.Parameter(torch.zeros(3, 4)),
                                               'item_emb': torch.nn.Parameter(torch.zeros(5, 4))})
    f = GraphRecommender._fusable_adam
    got = f(torch.optim.Adam(m.parameters(), lr=0.003, betas=(0.8, 0.99), eps=1e-7), m)
    assert got == {"lr": 0.003, "betas": (0.8, 0.99), "eps": 1e-7}
    assert f(torch.optim.Adam([m.embedding_dict['user_emb'], m.embedding_dict['item_emb']], lr=0.1), m) is not None
    for bad in (torch.optim.SGD(m.parameters(), lr=0.1),
                torch.optim.AdamW(m.parameters(), lr=0.1),
                torch.optim.Adam(m.parameters(), lr=0.1, amsgrad=True),
                torch.optim.Adam(m.parameters(), lr=0.1, weight_decay=1e-4),
                torch.optim.Adam(m.parameters(), lr=0.1, maximize=True),
                torch.optim.Adam([m.embedding_dict['user_emb']], lr=0.1),                      # not all parameters
                torch.optim.Adam([{'params': [m.embedding_dict['user_emb']]}, {'params': [m.embedding_dict['item_emb']]}], lr=0.1),
                torch.optim.Adam([torch.nn.Parameter(torch.zeros(3, 4)), torch.nn.Parameter(torch.zeros(5, 4))], lr=0.1)):  # stale
        assert f(bad, m) is None, type(bad).__name__
    # the two tables alone are not all parameters of a model with more (NGCF's weight matrices)
    m2 = torch.nn.Module()
    m2.embedding_dict = m.embedding_dict
    m2.W = torch.nn.Parameter(torch.zeros(4, 4))
    assert f(torch.optim.Adam([m.embedding_dict['user_emb'], m.embedding_dict['item_emb']], lr=0.1), m2) is None
    # state handover helpers on CPU tensors: a half-initialised state (one parameter stepped) is refused
    opt = torch.optim.Adam(m.parameters(), lr=0.1)
    opt.state[m.embedding_dict['user_emb']] = {'step': torch.tensor(3.0), 'exp_avg': torch.zeros(3, 4), 'exp_avg_sq': torch.zeros(3, 4)}
    assert f(opt, m) is None


def test_device_edge_builders_equal_the_scipy_path():
    """The scale-stress builders (device generator -> CSR -> train set; bench.py --workload c5b) on the CPU device at a
    small shape: the CSR built from edge tensors is bit-identical to the DataLoader formula on scipy
    (util/DataLoader.py:57-87), and the train set read off the CSR equals the one built from edge arrays."""
    from arlib_b200.engine import DeviceTrainSet
    from arlib_b200.graph import DeviceGraph
    from arlib_b200.util.synth import synth_edges_device
    U, I, E = 700, 300, 9000
    u, i = synth_edges_device(U, I, E, seed=3, device="cpu")
    assert u.numel() == E and int(torch.unique(u * I + i).numel()) == E
    assert int(torch.unique(u).numel()) == U and int(torch.unique(i).numel()) == I       # coverage edges
    g = DeviceGraph.from_device_edges(u, i, U, I)
    adj = port.bipartite_adjacency(u.numpy(), i.numpy(), U, I)
    ref = port.normalize_graph_mat(adj).tocsr()
    ref.sort_indices()
    assert np.array_equal(g.rowptr.numpy(), ref.indptr) and np.array_equal(g.col.numpy(), ref.indices)
    assert np.array_equal(g.val.numpy().view(np.uint32), ref.data.astype(np.float32).view(np.uint32))
    ts = DeviceTrainSet.from_graph(g, U, I)
    ts2 = DeviceTrainSet.from_arrays(u.numpy(), i.numpy(), U, I, "cpu")
    assert ts.n_edges == E and torch.equal(ts.rej_rowptr, ts2.rej_rowptr) and torch.equal(ts.rej_items, ts2.rej_items)
    pairs = set(zip(ts.e_user.tolist(), ts.e_item.tolist()))
    assert pairs == set(zip(u.tolist(), i.tolist()))
    sub = DeviceTrainSet.from_graph(g, U, I, epoch_edges=500, seed=1)
    assert sub.n_edges == 500 and set(zip(sub.e_user.tolist(), sub.e_item.tolist())) <= pairs


def test_evaluation_user_chunk_follows_the_workspace_budget():
    """users per agcf_score_topk call = what a ~4 GB workspace holds for the item table (evaluator.user_chunk): every named
    shape in one call, a 1 M-item table in ~10 k-user calls; bounded below and above; the workspace of a chunk fits the budget."""
    from arlib_b200 import _lib
    from arlib_b200.evaluator import user_chunk, WS_BUDGET_BYTES
    lib = _lib.load()
    sizes = [(1682, 64), (3706, 64), (40981, 64), (38048, 64), (91599, 128), (1000000, 128)]
    chunks = [user_chunk(i, d, 50) for i, d in sizes]
    assert all(4096 <= c <= 131072 and c % 1024 == 0 for c in chunks)
    assert chunks[2] >= 29858 and chunks[4] >= 52643          # Gowalla / Amazon-book: all users in one call
    assert chunks[5] < chunks[4] < chunks[2] <= chunks[0]      # more items -> fewer users per call
    for (i, d), c in zip(sizes, chunks):
        if c > 4096:
            assert lib.agcf_score_topk_ws_bytes(c, i, d, 50) <= WS_BUDGET_BYTES * 1.02
