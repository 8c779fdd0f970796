"""oracle/port.py against the golden vectors frozen from the LIVE reference for NGCF / SimGCL / XSimGCL / InfoNCE
(oracle/make_golden_models.py).  This is what pins those oracle functions (SURVEY.md 8c): recommender/NGCF.py:31-79,
197-212; SimGCL.py:36-85,198-219; XSimGCL.py:39-95,205-223; util/loss.py:42-49."""
import os

import numpy as np
import pytest
import torch

from oracle import port

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NOISE_SEED = 20180

pytestmark = pytest.mark.usefixtures("one_cpu_thread")


def _meta(g):
    out = {}
    for s in g["meta"]:
        k, v = str(s).split("=", 1)
        out[k] = v
    return out


@pytest.fixture(scope="module")
def pdata(golden_rows):
    train, test = golden_rows
    return port.PortData([list(r) for r in train], (), test)


def _batches(golden):
    off = np.concatenate([[0], np.cumsum(golden["batch_len"])])
    return [(golden["batch_u"][off[b]:off[b + 1]].tolist(), golden["batch_i"][off[b]:off[b + 1]].tolist(),
             golden["batch_j"][off[b]:off[b + 1]].tolist()) for b in range(len(off) - 1)]


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _check_eval(pdata, g, fu, fi):
    assert np.array_equal(_bits(fu.numpy()), _bits(g["final_user_emb"]))
    assert np.array_equal(_bits(fi.numpy()), _bits(g["final_item_emb"]))
    rec, measure = port.full_rank_test(pdata, fu, fi, 50, [50])
    assert list(measure) == list(g["measure"])
    assert [int(u) for u in rec] == g["topk_users"].tolist()
    for k, u in enumerate(rec):
        assert set(int(p[0]) for p in rec[u]) == set(g["topk_items"][k].tolist())


def test_ngcf_epoch_and_forward(golden, pdata):
    g = np.load(os.path.join(GOLD, "ml100k_ngcf.npz"), allow_pickle=False)
    m = _meta(g)
    L = int(m["n_layers"])
    # nn.ParameterDict built from a plain dict registers its keys SORTED; Adam is element-wise, the order is immaterial
    assert sorted(g["param_order"].tolist()) == sorted(["embedding_dict.user_emb", "embedding_dict.item_emb",
                                                        "W.w1_0", "W.w2_0", "W.w1_1", "W.w2_1"])
    tr = port.NGCFTrainer(pdata.norm_adj, torch.from_numpy(golden["init_user_emb"]), torch.from_numpy(golden["init_item_emb"]),
                          [torch.from_numpy(g["init_w1_%d" % k]) for k in range(L)],
                          [torch.from_numpy(g["init_w2_%d" % k]) for k in range(L)], float(m["lr"]), float(m["reg"]))
    losses = [tr.step(*b) for b in _batches(golden)]
    assert losses[0] == g["batch_loss"][0]
    np.testing.assert_allclose(losses, g["batch_loss"], rtol=2e-6)
    assert np.abs(tr.user_emb.detach().numpy() - g["param_user_emb"]).max() < 5e-5
    assert np.abs(tr.w1[1].detach().numpy() - g["param_w1_1"]).max() < 5e-6
    adj = port.to_torch_coo(pdata.norm_adj)
    fu, fi = port.ngcf_forward(adj, torch.from_numpy(g["param_user_emb"]), torch.from_numpy(g["param_item_emb"]),
                               [torch.from_numpy(g["param_w1_%d" % k]) for k in range(L)],
                               [torch.from_numpy(g["param_w2_%d" % k]) for k in range(L)])
    _check_eval(pdata, g, fu, fi)


@pytest.mark.parametrize("name", ["simgcl", "xsimgcl"])
def test_contrastive_epoch_and_forward(name, golden, pdata):
    g = np.load(os.path.join(GOLD, "ml100k_%s.npz" % name), allow_pickle=False)
    m = _meta(g)
    L, eps, cl_rate = int(m["n_layers"]), float(m["eps"]), float(m["cl_rate"])
    N = pdata.user_num + pdata.item_num
    torch.manual_seed(NOISE_SEED)
    drawn = []

    def noise():
        t = torch.rand(N, 64)
        drawn.append(float(t.double().sum()))
        return t

    iu, ii = torch.from_numpy(golden["init_user_emb"]), torch.from_numpy(golden["init_item_emb"])
    if name == "simgcl":
        tr = port.SimGCLTrainer(pdata.norm_adj, iu, ii, L, eps, cl_rate, float(m["lr"]), float(m["reg"]), noise)
        per_batch = 2 * L
    else:
        tr = port.XSimGCLTrainer(pdata.norm_adj, iu, ii, L, eps, cl_rate, int(m["layer_cl"]), float(m["lr"]),
                                 float(m["reg"]), noise, tau=float(m["temp"]))
        per_batch = L
    parts = [tr.step(*b) for b in _batches(golden)]
    assert len(g["noise_sum"]) == per_batch * len(parts)
    assert drawn == g["noise_sum"].tolist()              # the reference's rand_like stream, regenerated bit for bit
    assert parts[0][0] == g["rec_loss"][0]
    np.testing.assert_allclose([p[0] for p in parts], g["rec_loss"], rtol=2e-6)
    np.testing.assert_allclose([p[1] for p in parts], cl_rate * g["nce_loss"].sum(1), rtol=2e-5)
    assert np.abs(tr.user_emb.detach().numpy() - g["param_user_emb"]).max() < 5e-5
    assert np.abs(tr.item_emb.detach().numpy() - g["param_item_emb"]).max() < 5e-5
    fu, fi = port.simgcl_forward(port.to_torch_coo(pdata.norm_adj), torch.from_numpy(g["param_user_emb"]),
                                 torch.from_numpy(g["param_item_emb"]), L, eps, None)
    _check_eval(pdata, g, fu, fi)


def test_infonce_known_answers():
    """The vectors were frozen on one CPU model, where the port matched the reference bit for bit.  Torch's CPU
    matrix and vector-math kernels round differently on other CPU models (on some the loss moves by one float32 ulp
    and gradient elements by up to 5e-7 of the gradient's largest magnitude), so the check is held at float32
    rounding level: the loss to 5e-7 relative, every gradient value to 2e-6 of the largest one of its case."""
    g = np.load(os.path.join(GOLD, "infonce_kat.npz"), allow_pickle=False)

    def close(got, want):
        np.testing.assert_allclose(got, want, rtol=0, atol=2e-6 * np.abs(want).max())

    for n, d, tau, seed in g["cases"]:
        n, d, seed = int(n), int(d), int(seed)
        gen = torch.Generator().manual_seed(seed)
        v1 = (torch.rand(n, d, generator=gen) - 0.5).requires_grad_(True)
        v2 = (torch.rand(n, d, generator=gen) - 0.3).requires_grad_(True)
        loss = port.infonce(v1, v2, float(tau))
        loss.backward()
        key = "n%d_d%d_s%d" % (n, d, seed)
        np.testing.assert_allclose(float(loss), float(g[key + "_loss"][0]), rtol=5e-7, atol=0)
        if key + "_g1" in g:
            close(v1.grad.numpy(), g[key + "_g1"])
            close(v2.grad.numpy(), g[key + "_g2"])
        else:
            close(v1.grad.double().sum(1).numpy(), g[key + "_g1rows"])
            close(v2.grad.double().sum(1).numpy(), g[key + "_g2rows"])
