"""GPU parity of every kernel family at the embedding sizes 8 and 16: full-rank top-K (both stage-1 GEMMs x the three
stage-2 implementations), the TF32 group maxima, InfoNCE, the SDDMM of the adjacency gradient, the SimGCL perturbation
epilogue (noise tables and Philox, main and aux outputs), the NGCF dense layer and BPR on a full-width table."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from _util import assert_topk_matches
from oracle import port

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
WIDTHS = [8, 16]


def _rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / b.abs().max())


def _mask_csr(U, lists):
    rp = np.zeros(U + 1, dtype=np.int32)
    rp[1:] = np.cumsum([len(x) for x in lists])
    flat = np.concatenate([np.sort(np.asarray(x, dtype=np.int32)) for x in lists]) if rp[-1] else np.zeros(1, np.int32)
    return torch.from_numpy(rp).to(DEV), torch.from_numpy(flat.astype(np.int32)).to(DEV)


def _all_variants(monkeypatch, ue, ie, K, **kw):
    """top-K of every stage-1 GEMM (0: fp32 CUDA cores, 1: tcgen05) x stage-2 implementation; all must be bit-identical"""
    from arlib_b200 import ops
    outs = {}
    for s2 in ("2", "1", "0"):
        monkeypatch.setenv("AGCF_STAGE2_IMPL", s2)
        for impl in (0, 1):
            v, i = ops.score_topk(ue, ie, K, impl=impl, **kw)
            outs[(impl, s2)] = (v.cpu(), i.cpu())
    monkeypatch.delenv("AGCF_STAGE2_IMPL")
    v0, i0 = outs[(0, "2")]
    for key, (v, i) in outs.items():
        assert torch.equal(i, i0) and torch.equal(v.view(torch.int32), v0.view(torch.int32)), key
    return v0.numpy(), i0.numpy()


@pytest.mark.parametrize("d", WIDTHS)
@pytest.mark.parametrize("U,I,K,masked", [(70, 1000, 50, True), (130, 333, 10, True), (40, 5000, 20, False),
                                          (5, 31, 3, True), (17, 90, 50, True), (33, 2049, 100, False)])
def test_topk_sets_equal_the_reference_rule(monkeypatch, d, U, I, K, masked):
    """(I < 2K: the plain group-major stage 2; 90 items, K = 50: fewer unmasked items than K for some users)"""
    from arlib_b200 import ops
    rng = np.random.default_rng(U + I + d)
    ue, ie = torch.randn(U, d), torch.randn(I, d)
    kw = {}
    lists = [np.zeros(0, np.int64)] * U
    if masked:
        lists = [rng.choice(I, size=int(rng.integers(0, min(I, 60))), replace=False) for _ in range(U)]
        kw["mask_rowptr"], kw["mask_items"] = _mask_csr(U, lists)
    vals, idx = _all_variants(monkeypatch, ue.to(DEV), ie.to(DEV), K, **kw)
    exact = ops.score_rows(ue.to(DEV), torch.arange(U, dtype=torch.int32, device=DEV), ie.to(DEV)).cpu().numpy()
    ref = (ue.double() @ ie.double().T).numpy()
    assert np.abs(exact - ref).max() < 1e-4
    for r in range(U):
        s = exact[r].copy()
        s[lists[r]] = -10e8
        Keff = min(K, I)
        assert set(idx[r][:Keff].tolist()) == port.topk_reference_set(Keff, s)
        assert np.array_equal(vals[r][:Keff], s[idx[r][:Keff]])
        assert np.all(idx[r][Keff:] == -1)
        s64 = ref[r].copy(); s64[lists[r]] = -10e8
        assert_topk_matches(idx[r][:Keff], s64, Keff, 1e-4)


@pytest.mark.parametrize("d", WIDTHS)
def test_topk_tie_rule_known_answer(monkeypatch, d):
    """integer-valued embeddings: many exactly tied scores; the set follows the reference heap's rule"""
    from arlib_b200 import ops
    rng = np.random.default_rng(d)
    U, I, K = 40, 300, 20
    ue = torch.from_numpy(rng.integers(-1, 2, (U, d)).astype(np.float32))
    ie = torch.from_numpy(rng.integers(-1, 2, (I, d)).astype(np.float32))
    lists = [rng.choice(I, size=int(rng.integers(0, 30)), replace=False) for _ in range(U)]
    mrp, mit = _mask_csr(U, lists)
    vals, idx = _all_variants(monkeypatch, ue.to(DEV), ie.to(DEV), K, mask_rowptr=mrp, mask_items=mit)
    s_all = (ue @ ie.T).numpy()
    for r in range(U):
        s = s_all[r].copy()
        s[lists[r]] = -10e8
        assert set(idx[r].tolist()) == port.topk_reference_set(K, s)


@pytest.mark.parametrize("d", WIDTHS)
def test_group_max_within_the_tf32_bound(d):
    """stage 1 on the tensor cores at K = d: |a - e| <= delta = 1.01 2^-9 |u| max|v| (csrc/score.cu header)"""
    from arlib_b200 import ops
    rng = np.random.default_rng(5 + d)
    U, I = 300, 3000
    ue, ie = torch.randn(U, d, device=DEV), torch.randn(I, d, device=DEV) * (1 + 3 * torch.rand(I, 1, device=DEV))
    lists = [rng.choice(I, size=int(rng.integers(0, 50)), replace=False) for _ in range(U)]
    mrp, mit = _mask_csr(U, lists)
    exact = ops.score_group_max(ue, ie, mask_rowptr=mrp, mask_items=mit, impl=0)
    tc = ops.score_group_max(ue, ie, mask_rowptr=mrp, mask_items=mit, impl=1)
    s = (ue.double() @ ie.double().T).cpu().numpy()
    for r in range(U):
        s[r, lists[r]] = -10e8
    pad = (-I) % 32
    want = np.pad(s, ((0, 0), (0, pad)), constant_values=-np.inf).reshape(U, -1, 32).max(2)
    np.testing.assert_allclose(exact.cpu().numpy(), want, rtol=1e-5, atol=1e-5)
    delta = 1.01 * 2.0 ** -9 * ue.norm(dim=1, keepdim=True) * ie.norm(dim=1).max()
    err = (tc - exact).abs() / delta
    assert float(err.max()) <= 1.0, float(err.max())
    assert float(err.max()) > 0.0                                   # it really ran in TF32


@pytest.mark.parametrize("d", WIDTHS)
@pytest.mark.parametrize("n", [1, 5, 63, 64, 65, 300, 2048])
@pytest.mark.parametrize("tau", [0.2, 0.1])
def test_infonce_matches_float64_autograd(d, n, tau):
    from arlib_b200.util.loss import InfoNCE
    g = torch.Generator().manual_seed(n * 7 + d)
    a = torch.randn(n, d, generator=g)
    b = a + 0.3 * torch.randn(n, d, generator=g)
    ar, br = a.double().requires_grad_(True), b.double().requires_grad_(True)
    ref = port.infonce(ar, br, tau)
    (ref * 0.2).backward()
    outs = []
    for _ in range(2):
        ag, bg = a.to(DEV).requires_grad_(True), b.to(DEV).requires_grad_(True)
        got = InfoNCE(ag, bg, tau)
        (got * 0.2).backward()
        outs.append((got.detach().clone(), ag.grad.clone(), bg.grad.clone()))
    got, ga, gb = outs[0]
    assert abs(float(got) - float(ref)) <= 1e-5 * max(1.0, abs(float(ref)))
    for g_, r_ in ((ga.cpu(), ar.grad), (gb.cpu(), br.grad)):
        scale = float(r_.abs().max()) + 1e-30
        assert float((g_.double() - r_).abs().max()) <= 1e-4 * scale + 1e-7
    for x, y in zip(outs[0], outs[1]):
        assert torch.equal(x, y)                                    # fixed slice order: the same bits every call


def _graph(U, I, E, seed):
    from arlib_b200.graph import DeviceGraph
    rng = np.random.default_rng(seed)
    u, i = rng.integers(0, U, E), rng.integers(0, I, E)
    hub = min(300, I)                                               # a hub row longer than the short-row path
    u[:hub], i[:hub] = 0, rng.permutation(I)[:hub]
    key = np.unique(u.astype(np.int64) * I + i)
    u, i = key // I, key % I
    adj = port.bipartite_adjacency(u, i, U, I)
    return adj, DeviceGraph.from_dataloader_adj(adj, DEV)


@pytest.mark.parametrize("d", WIDTHS)
def test_sddmm_matches_torch_sparse_gradient(d):
    """d loss / d values of A for loss = sum(W * (A X)): torch's sparse gradient is <W_i, X_j> on the pattern"""
    from arlib_b200 import ops
    U, I = 200, 400
    adj, g = _graph(U, I, 5000, d)
    csr = port.normalize_graph_mat(adj).tocsr(); csr.sort_indices()
    coo = csr.tocoo()
    A = torch.sparse_coo_tensor(np.vstack([coo.row, coo.col]), torch.from_numpy(coo.data.astype(np.float64)),
                                (U + I, U + I)).coalesce().requires_grad_(True)
    H, X = torch.randn(U + I, d), torch.randn(U + I, d)
    (torch.sparse.mm(A, X.double()) * H.double()).sum().backward()
    ref = A.grad.coalesce()
    ref_vals = torch.sparse_coo_tensor(ref.indices(), ref.values(), ref.shape).to_dense()[coo.row, coo.col]
    gval = torch.zeros(g.nnz, device=DEV)
    ops.sddmm(g, H.to(DEV), X.to(DEV), gval)
    torch.testing.assert_close(gval.cpu().double(), ref_vals, rtol=1e-5, atol=1e-5)
    ops.sddmm(g, H.to(DEV), X.to(DEV), gval, accumulate=True)
    torch.testing.assert_close(gval.cpu().double(), 2 * ref_vals, rtol=1e-5, atol=1e-5)


def _philox_uniform(seed, n_slots, ctr_hi):
    """host Philox4x32-10 of csrc/common.cuh: counter (float4 slot, ctr_hi), key seed -> U[0,1) with 24 bits"""
    m32 = np.uint64(0xFFFFFFFF)
    slot = np.arange(n_slots, dtype=np.uint64)
    c = [slot & m32, slot >> np.uint64(32), np.full(n_slots, ctr_hi & 0xFFFFFFFF, np.uint64),
         np.full(n_slots, ctr_hi >> 32, np.uint64)]
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & m32, (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1), p0 & m32]
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    r = np.stack(c, 1).astype(np.uint32)                            # [slot][4]
    return torch.from_numpy(((r >> 8).astype(np.float32) * np.float32(2.0 ** -24)).reshape(-1))


def _perturbed(t, noise, eps):
    """E + sign(E) * normalize(noise) * eps (recommender/SimGCL.py:204-205), float64"""
    t, noise = t.double(), noise.double()
    return t + torch.sign(t) * F.normalize(noise, dim=-1) * eps


@pytest.mark.parametrize("d", WIDTHS)
def test_noise_epilogue_tables_and_philox_with_aux_outputs(d):
    from arlib_b200 import ops
    U, I = 150, 250
    N = U + I
    _, g = _graph(U, I, 3000, 11 + d)
    X = torch.randn(N, d, device=DEV) * 0.1
    clean = torch.empty_like(X)
    ops.spmm(g, X, Y=clean)
    eps = 0.1
    # noise tables: main output and both aux outputs, each with its own table
    tabs = [torch.rand(N, d, device=DEV) for _ in range(3)]
    y, a1, a2 = (torch.empty_like(X) for _ in range(3))
    ops.spmm(g, X, Y=y, noise=tabs[0], eps=eps)
    torch.testing.assert_close(y.cpu().double(), _perturbed(clean.cpu(), tabs[0].cpu(), eps), rtol=1e-5, atol=1e-6)
    y2 = torch.empty_like(X)
    ops.spmm(g, X, Y=y2, aux=[(a1, tabs[1], 0), (a2, tabs[2], 0)], eps=eps, philox=(5, None, None))
    assert torch.equal(y2, clean)                                   # no main perturbation: Y is A X itself
    for a_, t_ in ((a1, tabs[1]), (a2, tabs[2])):
        torch.testing.assert_close(a_.cpu().double(), _perturbed(clean.cpu(), t_.cpu(), eps), rtol=1e-5, atol=1e-6)
    # Philox: main stream 3 at step 7, aux streams 65 and 129 at the same step
    seed = 0x5eed5eed
    step = torch.full((1,), 7, dtype=torch.int32, device=DEV)
    ops.spmm(g, X, Y=y, eps=eps, philox=(seed, 3, step), aux=[(a1, None, 65), (a2, None, 129)])
    for out, stream in ((y, 3), (a1, 65), (a2, 129)):
        nz = _philox_uniform(seed, N * d // 4, (7 << 32) | stream).view(N, d)
        torch.testing.assert_close(out.cpu().double(), _perturbed(clean.cpu(), nz, eps), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("d,n", [(8, 1000), (16, 1000), (8, 1), (16, 129), (8, 50000)])
def test_ngcf_dense_layer_matches_autograd(d, n):
    from arlib_b200 import ops
    gen = torch.Generator().manual_seed(n + d)
    P = torch.randn(n, d, generator=gen) * 0.3
    E = torch.randn(n, d, generator=gen) * 0.3
    W = torch.randn(2 * d, d, generator=gen) / d ** 0.5
    dOut = torch.randn(n, d, generator=gen)
    acc = torch.randn(n, d, generator=gen)
    Pd, Ed, Wd = (t.double().requires_grad_(True) for t in (P, E, W))
    Y = F.leaky_relu((Pd + Ed) @ Wd[:d] + (Pd * Ed) @ Wd[d:], 0.01)
    Y.backward(dOut.double())
    Pc, Ec, Wc = P.to(DEV), E.to(DEV), W.to(DEV)
    Yc, mean = torch.empty_like(Pc), torch.empty_like(Pc)
    ops.ngcf_dense_forward(Pc, Ec, Wc, Yc, acc_in=acc.to(DEV), acc_out=mean, acc_div=3.0)
    assert _rel(Yc, Y.detach()) < 2e-6
    assert _rel(mean, (acc.double() + Y.detach()) / 3.0) < 2e-6
    dP, dE = torch.empty_like(Pc), torch.empty_like(Pc)
    part = torch.empty((296, 2 * d * d), device=DEV)
    dW = torch.empty((2 * d, d), device=DEV)
    ops.ngcf_dense_backward(dOut.to(DEV), Yc, Pc, Ec, Wc.t().contiguous(), dP, dE, part, dW)
    assert _rel(dP, Pd.grad) < 3e-6 and _rel(dE, Ed.grad) < 3e-6
    assert _rel(dW, Wd.grad) < 3e-6
    dW2 = torch.empty_like(dW)
    ops.ngcf_dense_backward(dOut.to(DEV), Yc, Pc, Ec, Wc.t().contiguous(), dP, dE, part, dW2)
    assert torch.equal(dW, dW2)                                     # partials reduced in CTA order


@pytest.mark.parametrize("d", WIDTHS)
def test_bpr_forward_backward_on_a_full_width_table(d):
    from arlib_b200 import ops
    rng = np.random.default_rng(d)
    U, I, nb, B = 200, 300, 777, 1024
    Ft = torch.randn(U + I, d) * 0.3
    u = rng.integers(0, U, nb).astype(np.int32)
    i = rng.integers(0, 40, nb).astype(np.int32)
    j = rng.integers(0, I, nb).astype(np.int32)
    Fr = Ft.double().requires_grad_(True)
    ue, pe, ne = Fr[torch.from_numpy(u).long()], Fr[U + torch.from_numpy(i).long()], Fr[U + torch.from_numpy(j).long()]
    loss = port.bpr_loss(ue, pe, ne) + port.l2_reg_loss(1e-2, ue, pe)
    loss.backward()
    dv = lambda a: torch.from_numpy(a).to(DEV)
    Fd = Ft.to(DEV)
    out4 = torch.zeros(4, device=DEV)
    coef = torch.empty(B, device=DEV)
    ws = torch.zeros(ops.bpr_ws_bytes(B), dtype=torch.uint8, device=DEV)
    du, di, dj = dv(u), dv(i), dv(j)
    ops.bpr_forward(Fd, du, di, dj, nb, U, 1e-2, out4, coef, ws)
    assert abs(out4[0].item() - loss.item()) <= 2e-6 * abs(loss.item())
    occ = torch.empty(3 * B, dtype=torch.int32, device=DEV)
    seg_off = torch.empty(3 * B + 1, dtype=torch.int32, device=DEV)
    seg_node = torch.empty(3 * B, dtype=torch.int32, device=DEV)
    n_seg = torch.zeros(1, dtype=torch.int32, device=DEV)
    ops.bpr_group_batches(du, di, dj, nb, B, U, occ, seg_off, seg_node, n_seg)
    G = torch.zeros_like(Fd)
    ops.bpr_backward(Fd, du, di, dj, nb, U, 1e-2, 1.0, out4, coef, occ, seg_off, seg_node, n_seg, G)
    torch.testing.assert_close(G.cpu().double(), Fr.grad, rtol=1e-4, atol=1e-7)
