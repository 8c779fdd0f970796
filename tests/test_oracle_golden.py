"""oracle/port.py against the golden vectors frozen from the LIVE reference
(oracle/make_golden.py): this is what pins the oracle (SURVEY.md 8c)."""
import random

import numpy as np
import pytest
import torch

from oracle import port

pytestmark = pytest.mark.usefixtures("one_cpu_thread")


@pytest.fixture(scope="module")
def pdata(golden_rows):
    train, test = golden_rows
    return port.PortData([list(r) for r in train], (), test)


def test_ids_and_adjacency_bit_exact(golden, pdata):
    assert pdata.user_num == golden["user_names"].shape[0]
    assert pdata.item_num == golden["item_names"].shape[0]
    adj = pdata.norm_adj.tocsr()
    adj.sort_indices()
    assert np.array_equal(adj.indptr, golden["adj_indptr"])
    assert np.array_equal(adj.indices, golden["adj_indices"])
    assert np.array_equal(adj.data.astype(np.float32).view(np.uint32), golden["adj_data"].view(np.uint32))


def test_init_uiadj_formula_bit_exact(golden, pdata):
    coo = port.to_torch_coo(port.init_uiadj_norm(pdata.ui_adj)).coalesce()
    assert np.array_equal(coo.indices()[0].numpy(), golden["uiadj_row"])
    assert np.array_equal(coo.indices()[1].numpy(), golden["uiadj_col"])
    assert np.array_equal(coo.values().numpy().view(np.uint32), golden["uiadj_data"].view(np.uint32))
    # the two normalizations are NOT bit-identical (np.power(x,-0.5) vs 1/np.sqrt(x)): both must be kept
    assert not np.array_equal(golden["uiadj_data"].view(np.uint32), golden["adj_data"].view(np.uint32))


def test_host_sampler_consumes_rng_like_reference(golden, golden_rows):
    train, test = golden_rows
    d = port.PortData([list(r) for r in train], (), test)
    random.seed(2018)
    got = list(port.next_batch_pairwise(d, 2048))
    assert [len(b[0]) for b in got] == golden["batch_len"].tolist()
    assert np.array_equal(np.concatenate([b[0] for b in got]), golden["batch_u"])
    assert np.array_equal(np.concatenate([b[1] for b in got]), golden["batch_i"])
    assert np.array_equal(np.concatenate([b[2] for b in got]), golden["batch_j"])


def test_first_loss_bit_exact_and_epoch_within_tolerance(golden, pdata):
    tr = port.LightGCNTrainer(pdata.norm_adj, torch.from_numpy(golden["init_user_emb"]),
                              torch.from_numpy(golden["init_item_emb"]), 2, 0.005, 1e-4)
    off = np.concatenate([[0], np.cumsum(golden["batch_len"])])
    losses = []
    for b in range(len(off) - 1):
        sl = slice(off[b], off[b + 1])
        losses.append(tr.step(golden["batch_u"][sl].tolist(), golden["batch_i"][sl].tolist(),
                              golden["batch_j"][sl].tolist()))
    assert losses[0] == golden["batch_loss"][0]
    np.testing.assert_allclose(losses, golden["batch_loss"], rtol=1e-6)
    # CPU torch backward is not run-to-run deterministic (~1e-7): tolerance, not bits
    assert np.abs(tr.user_emb.detach().numpy() - golden["param_user_emb"]).max() < 2e-6
    assert np.abs(tr.item_emb.detach().numpy() - golden["param_item_emb"]).max() < 2e-6


def test_forward_topk_metrics_bit_exact(golden, pdata):
    fu, fi = port.lightgcn_forward(port.to_torch_coo(pdata.norm_adj), torch.from_numpy(golden["param_user_emb"]),
                                   torch.from_numpy(golden["param_item_emb"]), 2)
    assert np.array_equal(fu.numpy().view(np.uint32), golden["final_user_emb"].view(np.uint32))
    assert np.array_equal(fi.numpy().view(np.uint32), golden["final_item_emb"].view(np.uint32))
    rec, measure = port.full_rank_test(pdata, fu, fi, 50, [50])
    assert list(measure) == list(golden["measure"])
    assert [int(u) for u in rec] == golden["topk_users"].tolist()
    for k, u in enumerate(rec):
        assert set(int(p[0]) for p in rec[u]) == set(golden["topk_items"][k].tolist())
