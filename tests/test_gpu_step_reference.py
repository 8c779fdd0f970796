"""A float64 reference of one LightGCN training step (recommender/LightGCN.py:46-64), and teacher-forced checks of the
optimized step against it.

ref_step runs the step in float64: the oracle's forward and losses on the graph's own fp32 values (upcast), autograd for
the gradient, and the Adam update of include/agcf.h.  The GPU tests read the engine's state, run ONE step, and compare
every output with ref_step from that state: the reference never drifts, so step 5 is held as tightly as step 1.  Each
element is compared against a running-error bound derived from the fp32 arithmetic (step_bounds), not a tuned
tolerance, and the bounds are shown to reject four small reference-side perturbations.

The cases switch each fast path of the step on and off: the batch bitmap gating G (12 B <= N) or not, per-batch work
lists, Adam fused into the last backward SpMM, persistent CTAs, the Adam coefficients on a side stream, 64- and
256-entry segments, eager launches and graph replay, L = 1 .. 9 layers (L >= 4: L - 1 forward tables; L > 8: the
forward_table path), d = 8 .. 256 columns, partial batches, and the benchmark shapes.  The d-sharded loss exchange
(bpr_partial / bpr_finish) is checked on one GPU by emulating its ranks."""
import collections
import math

import numpy as np
import pytest
import torch

from oracle import port

DEV = "cuda:0"
UNIT = 2.0 ** -24                 # unit roundoff of fp32: every correctly rounded operation is within UNIT relative
LR, REG, BETAS, EPS = 0.005, 1e-4, (0.9, 0.999), 1e-8

# the CSR the kernels read (device or host tensors) and the number of user rows
RefCSR = collections.namedtuple("RefCSR", "rowptr col val n_users")


# ------------------------------------------------------------------------------------------------ float64 reference
def _adj64(csr):
    rp = csr.rowptr.long()
    n = rp.numel() - 1
    rows = torch.repeat_interleave(torch.arange(n, device=rp.device), rp[1:] - rp[:-1])
    return torch.sparse_coo_tensor(torch.stack([rows, csr.col.long().to(rp.device)]), csr.val.double().to(rp.device),
                                   (n, n)).coalesce()


def adam_scalars(t, lr, betas, eps):
    """(b1, b2, lr / (1 - b1^t), sqrt(1 - b2^t), eps) from lr, b1, b2 and eps rounded to float32, as the ABI takes them"""
    f32 = lambda x: float(np.float32(x))
    lr, b1, b2, eps = f32(lr), f32(betas[0]), f32(betas[1]), f32(eps)
    return b1, b2, lr / (1.0 - b1 ** t), math.sqrt(1.0 - b2 ** t), eps


def ref_step(csr, E0, m, v, t, u, i, j, L, reg, lr, betas=BETAS, eps=EPS):
    """One training step in float64 from parameters E0 and moments m, v (any dtype), Adam step t (1 for the first
    step), triples (u, i, j) (user ids, item ids).  Returns a dict: loss4 = (loss, bpr term, ||F[u]||_F, ||F[U+i]||_F),
    F = the propagated table, g = d loss / d E0, the updated m, v, p, and the Adam scalars c1, c2 that were used."""
    A = _adj64(csr)
    U = csr.n_users
    E = E0.detach().double().clone().requires_grad_(True)
    ru, ri = port.lightgcn_forward(A, E[:U], E[U:], L)
    ue, pe, ne = ru[u], ri[i], ri[j]
    bpr = port.bpr_loss(ue, pe, ne)
    loss = bpr + port.l2_reg_loss(reg, ue, pe)
    g, = torch.autograd.grad(loss, E)
    b1, b2, c1, c2, eps = adam_scalars(t, lr, betas, eps)
    m1 = b1 * m.double() + (1 - b1) * g
    v1 = b2 * v.double() + (1 - b2) * g * g
    p1 = E0.double() - c1 * m1 / (v1.sqrt() / c2 + eps)
    with torch.no_grad():
        loss4 = torch.stack([loss, bpr, ue.norm(), pe.norm()])
        F = torch.cat([ru, ri])
    return dict(loss4=loss4, F=F, g=g, m=m1, v=v1, p=p1, c1=c1, c2=c2, eps=eps, b1=b1, b2=b2, A=A)


# ------------------------------------------------------------------------------------------------ error bounds
def _mean_powers(A, X, L):
    """mean_k A^k X, k = 0 .. L (A >= 0 elementwise: applied to magnitudes it bounds the same sums of |terms|)"""
    acc, Y = X.clone(), X
    for _ in range(L):
        Y = torch.sparse.mm(A, Y)
        acc += Y
    return acc / (L + 1)


def loss_grad_bounds(Fa, cF, F, u, i, j, U, reg, eF=None):
    """Bounds of the fp32 loss row, the coefficients coef_t = d loss / d x_t and G = d loss / d F, when the fp32 table
    the kernels read is within eF of the float64 table F elementwise (default eF = cF * UNIT * Fa; Fa >= |F|).  First
    order in UNIT.  Returns loss4 (bound per entry), coef (bound per triple), Gabs (a magnitude >= |G|) and G (bound
    per element)."""
    d, nb, N = F.shape[1], u.numel(), F.shape[0]
    iu, ii, ij = u, U + i, U + j
    if eF is None:
        eF = cF * UNIT * Fa
    Pu, Pi, Pj = Fa[iu], Fa[ii], Fa[ij]
    Eu, Ei, Ej = eF[iu], eF[ii], eF[ij]
    # x_t = <F_u, F_i> - <F_u, F_j>: two d-term dot products (d UNIT of the sum of |products| in any summation order)
    # and a difference; each factor carries its error eF
    Px = (Pu * (Pi + Pj)).sum(1)
    dx = (d + 1) * UNIT * Px + (Eu * (Pi + Pj) + Pu * (Ei + Ej)).sum(1)
    x = (F[iu] * (F[ii] - F[ij])).sum(1)
    s = torch.sigmoid(x)
    dl = s * (1 - s) / (1e-7 + s)                     # |d l_t / d x_t| <= 1
    lt = -torch.log(1e-7 + s)
    # l_t = -logf(1e-7 + 1 / (1 + expf(-x))): expf and logf are within 2 ulp, four more roundings: 8 UNIT of l_t and,
    # where l_t ~ 0, 8 UNIT absolute (the error of s relative to s); the batch mean is taken in double
    bpr_b = (dl * dx).mean() + 8 * UNIT * (lt.mean() + 1)
    nu, ni = F[iu].norm(), F[ii].norm()
    # ||F[u_.]||_F: the table's error (||eF[u_.]||), d + 4 UNIT for the sums of squares and the square root
    nu_b = Eu.norm() + (d + 4) * UNIT * nu
    ni_b = Ei.norm() + (d + 4) * UNIT * ni
    loss = lt.mean() + reg * (nu + ni)
    loss4 = torch.stack([bpr_b + reg * (nu_b + ni_b) + 2 * UNIT * loss, bpr_b, nu_b, ni_b])
    # coef_t = -s (1 - s) / ((1e-7 + s) nb): |d coef / d x| <= 1 / (4 nb); expf and 7 roundings: 16 UNIT
    cu = dl / nb
    ec = dx / (4 * nb) + 16 * UNIT * cu
    # rows of G: user  sum_t coef_t (F_i - F_j) + reg F_u / nu, positive item  coef_t F_u + reg F_i / ni, negative item
    # -coef_t F_u.  Per term: the coefficient's error times |F|, |coef| times the table's error, three roundings
    U3 = 3 * UNIT
    Gabs, Gerr = torch.zeros_like(F), torch.zeros_like(F)
    Gabs.index_add_(0, iu, cu[:, None] * (Pi + Pj) + reg * Pu / nu)
    Gerr.index_add_(0, iu, ec[:, None] * (Pi + Pj) + cu[:, None] * (Ei + Ej + U3 * (Pi + Pj))
                    + reg * ((Eu + U3 * Pu) / nu + Pu * nu_b / nu ** 2))
    Gabs.index_add_(0, ii, cu[:, None] * Pu + reg * Pi / ni)
    Gerr.index_add_(0, ii, ec[:, None] * Pu + cu[:, None] * (Eu + U3 * Pu) + reg * ((Ei + U3 * Pi) / ni + Pi * ni_b / ni ** 2))
    Gabs.index_add_(0, ij, cu[:, None] * Pu)
    Gerr.index_add_(0, ij, ec[:, None] * Pu + cu[:, None] * (Eu + U3 * Pu))
    # a node's occurrences are summed in fp32: (occurrences) UNIT of its magnitude
    occ = torch.bincount(torch.cat([iu, ii, ij]), minlength=N).double()
    Gerr += occ[:, None] * UNIT * Gabs
    return dict(loss4=loss4, coef=ec, Gabs=Gabs, G=Gerr)


def run_length(g, extra_segments=()):
    """Longest chain of fp32 adds in one SpMM output element: a row of deg entries is summed as segments of at most
    `segment` entries (rows of at most split_above entries: one segment), and the segments' partials are then added,
    so its summation tree is at most segment + ceil(deg / segment) deep.  Max over the plans the step uses."""
    deg = int((g.rowptr[1:] - g.rowptr[:-1]).max())
    run = 1
    for split, seg in [(g.split_above, g.segment)] + [(s, s) for s in extra_segments]:
        run = max(run, min(deg, split), seg + -(-deg // seg) if deg > split else 0)
    return run


def step_bounds(ref, E0, u, i, j, L, reg, run, U):
    """Elementwise error bounds of the fp32 step against ref (first order in UNIT).

    Forward: a layer's output element sums at most `run` deep, so it is within (run + 1) UNIT of A |X| (the product's
    rounding included) plus A times the input's error: layer k is within k (run + 1) UNIT of A^k |E0|.  The layer mean
    adds L + 1 roundings, so F is within cF UNIT of F_abs = mean_k A^k |E0|, cF = L (run + 1) + L + 2.
    Backward: dE0 = mean_k A^k G, as H_{k-1} = A H_k + G: each level adds (run + 2) UNIT of its magnitude, so
    dE0 is within mean_k A^k (G's error + cB UNIT |G|), cB = L (run + 2) + 2."""
    A = ref["A"]
    Fa = _mean_powers(A, E0.double().abs(), L)
    cF = L * (run + 1) + L + 2
    lg = loss_grad_bounds(Fa, cF, ref["F"], u, i, j, U, reg)
    cB = L * (run + 2) + 2
    g = _mean_powers(A, lg["G"] + cB * UNIT * lg["Gabs"], L)
    # rows more than L hops from every batch node: the gradient is exactly zero there
    seed = torch.zeros(E0.shape[0], 1, dtype=torch.float64, device=E0.device)
    seed[torch.cat([u, U + i, U + j])] = 1.0
    far = _mean_powers(A, seed, L)[:, 0] == 0
    return dict(loss4=lg["loss4"], F=cF * UNIT * Fa, g=g, far=far)


def _ulp32(x):
    _, e = torch.frexp(x.float())
    return torch.ldexp(torch.ones_like(x, dtype=torch.float64), (e - 24).clamp_min(-149))


def _ratio(err, tol):
    """max of err / tol; an element with tol == 0 must be exact"""
    err, tol = err.double(), tol.double()
    if bool(((tol == 0) & (err != 0)).any()):
        return math.inf
    nz = tol > 0
    return float((err[nz] / tol[nz]).max()) if bool(nz.any()) else 0.0


def check_step(got, ref, bnd, p0, m0, v0, rows):
    """max(error / bound) per output of one step; > 1 is a failure.  got: the kernel's loss4, F (valid at ``rows``, the
    batch's nodes), m, v, p after the step and, when the step writes it, g = dE0; p0 / m0 / v0: the state before it."""
    g, eg = ref["g"], bnd["g"]
    r = {"loss": _ratio((got["loss4"].double() - ref["loss4"]).abs(), bnd["loss4"]),
         "F": _ratio((got["F"][rows].double() - ref["F"][rows]).abs(), bnd["F"][rows])}
    if "g" in got:                                           # the unfused step writes dE0
        r["g"] = _ratio((got["g"].double() - g).abs(), eg)
    r.update(adam_ratios(ref, g, eg, ref["m"], ref["v"], p0, m0, v0, got["m"], got["v"], got["p"]))
    r["exact"] = 0.0 if far_exact(g, bnd["far"], p0, m0, v0, got["m"], got["v"], got["p"]) else math.inf
    return r


def adam_ratios(s, g, eg, m_ref, v_ref, p0, m0, v0, m, v, p):
    """max(error / bound) of one Adam update of parameters p0 with moments m0, v0 by a gradient within eg of the float64
    g: the kernel's m, v against the float64 m_ref, v_ref, and its p against the update of its own m, v.  s holds the
    scalars b1, b2, c1, c2, eps the update used."""
    b1, b2, c1, c2, eps = s["b1"], s["b2"], s["c1"], s["c2"], s["eps"]
    gm = g.abs() + eg
    m0d, v0d = m0.double(), v0.double()
    md, vd, pd = m.double(), v.double(), p.double()
    r = {}
    # m' = m + (1 - b1) (g - m): three roundings; v' = fma((1 - b2) g, g, b2 v): three roundings
    r["m"] = _ratio((md - m_ref).abs(), (1 - b1) * eg + 3 * UNIT * ((1 - b1) * gm + m0d.abs()))
    r["v"] = _ratio((vd - v_ref).abs(), (1 - b2) * (2 * g.abs() + eg) * eg + 3 * UNIT * (b2 * v0d + (1 - b2) * gm * gm))
    # p' from the kernel's own m', v': c1, c2 rounded to float, sqrt, two divisions, + eps, the product: 8 UNIT of the
    # update, and the final subtraction rounds to p' (a few ulps of p)
    upd = c1 * md / (vd.sqrt() / c2 + eps)
    r["p"] = _ratio((pd - (p0.double() - upd)).abs(), 2 * _ulp32(p) + 8 * UNIT * upd.abs())
    return r


def far_exact(g, far, p0, m0, v0, m, v, p):
    """far from the batch the gradient is zero; where the moments are zero too nothing may change, to the bit"""
    fresh = far & (m0 == 0).all(1) & (v0 == 0).all(1)
    return bool((g[far] == 0).all()) and not _bits(m[fresh]).any() and not _bits(v[fresh]).any() \
        and np.array_equal(_bits(p[fresh]), _bits(p0[fresh]))


def _bits(t):
    return t.detach().contiguous().cpu().numpy().view(np.uint32)


RATIOS = collections.defaultdict(dict)


def _record(group, r):
    for k, x in r.items():
        RATIOS[group][k] = max(RATIOS[group].get(k, 0.0), x)


@pytest.fixture(scope="module", autouse=True)
def _report_ratios():
    yield
    for group, r in sorted(RATIOS.items()):
        print("\nlargest error / bound [%s]: %s" % (group, ", ".join("%s %.3g" % kv for kv in sorted(r.items()))))


# ------------------------------------------------------------------------------------------------ CPU: the reference
def test_ref_step_matches_the_oracle_trainer_with_torch_adam(one_cpu_thread):
    """ref_step against port.LightGCNTrainer with float64 parameters and torch.optim.Adam, three steps"""
    U, I, d, L = 40, 60, 8, 3
    rng = np.random.default_rng(0)
    key = np.unique(rng.integers(0, U, 300) * I + rng.integers(0, I, 300))
    adj = port.bipartite_adjacency(key // I, key % I, U, I)
    norm = port.normalize_graph_mat(adj).tocsr()
    norm.sort_indices()
    csr = RefCSR(torch.from_numpy(norm.indptr.astype(np.int64)), torch.from_numpy(norm.indices.astype(np.int64)),
                 torch.from_numpy(norm.data.astype(np.float32)), U)
    gen = torch.Generator().manual_seed(1)
    E = ((torch.rand(U + I, d, generator=gen) - 0.5) * 0.2).double()
    b1, b2, _, _, eps = adam_scalars(1, LR, BETAS, EPS)
    lr = float(np.float32(LR))
    tr = port.LightGCNTrainer(norm, E[:U], E[U:], L, lr, REG)
    tr.adj = tr.adj.double()
    tr.opt = torch.optim.Adam([tr.user_emb, tr.item_emb], lr=lr, betas=(b1, b2), eps=eps)
    m, v = torch.zeros_like(E), torch.zeros_like(E)
    for t in (1, 2, 3):
        u = torch.from_numpy(rng.integers(0, U, 50))
        i = torch.from_numpy(rng.integers(0, I, 50))
        j = torch.from_numpy(rng.integers(0, I, 50))
        ref = ref_step(csr, E, m, v, t, u, i, j, L, REG, LR)
        loss = tr.step(u, i, j)
        assert abs(loss - float(ref["loss4"][0])) <= 1e-12 * abs(loss)
        st = [tr.opt.state[p] for p in (tr.user_emb, tr.item_emb)]
        for name, want in (("p", torch.cat([tr.user_emb.detach(), tr.item_emb.detach()])),
                           ("m", torch.cat([s["exp_avg"] for s in st])), ("v", torch.cat([s["exp_avg_sq"] for s in st]))):
            scale = float(want.abs().max())
            torch.testing.assert_close(ref[name], want, rtol=1e-12, atol=1e-12 * scale, msg=lambda s: name + ": " + s)
        E, m, v = ref["p"], ref["m"], ref["v"]


# ------------------------------------------------------------------------------------------------ GPU: the engine
def _edges(U, I, E, seed, hub=750):
    """random user-item edges; user 0 and item 1 have `hub` entries each; user U - 1 and items I - 5 .. I - 1 none"""
    rng = np.random.default_rng(seed)
    u = rng.integers(0, U - 1, E)
    i = rng.integers(0, I - 5, E)
    u[:hub] = 0
    i[:hub] = rng.permutation(I - 5)[:hub]
    i[hub:2 * hub] = 1
    u[hub:2 * hub] = rng.permutation(U - 1)[:hub]
    key = np.unique(u.astype(np.int64) * I + i)
    return key // I, key % I


def _triples(eu, ei, U, I, B, T, seed):
    """T triples from the edges; every batch names the hub user and item, the user without edges, items without edges as
    negatives and as a positive, an item that is positive in one triple and negative in another, a repeated user"""
    rng = np.random.default_rng(seed)
    pick = rng.integers(0, eu.shape[0], T)
    tu, ti, tj = eu[pick].copy(), ei[pick].copy(), rng.integers(0, I, T)
    for s in range(0, T, B):
        if T - s < 10:
            continue
        tu[s], ti[s + 1], tu[s + 2] = 0, 1, U - 1
        tj[s + 3], tj[s + 4], ti[s + 5] = I - 1, I - 2, I - 3
        tj[s + 6] = ti[s + 7]
        tu[s + 9] = tu[s + 8]
    return [a.astype(np.int32) for a in (tu, ti, tj)]


def _small_engine(L, d, B, T, seed=0):
    from arlib_b200.engine import LightGCNEngine
    from arlib_b200.graph import DeviceGraph
    U, I = 800, 1000
    eu, ei = _edges(U, I, 12000, seed)
    g = DeviceGraph.from_dataloader_adj(port.bipartite_adjacency(eu, ei, U, I), DEV)
    gen = torch.Generator().manual_seed(seed + d)
    table = ((torch.rand(U + I, d, generator=gen) - 0.5) * 0.2).to(DEV)
    eng = LightGCNEngine(g, table, U, L, LR, REG, B, T)
    return eng, eu, ei


def teacher_forced(eng, steps, use_graph, group):
    """For each step b: read E0 / m / v / step_dev, run the step, compare with ref_step from what was read."""
    csr = RefCSR(eng.g.rowptr, eng.g.col, eng.g.val, eng.U)
    run = run_length(eng.g, [eng.wl_segment] if eng.wl is not None else [])
    for b in steps:
        p0, m0, v0 = eng.E0.clone(), eng.m.clone(), eng.v.clone()
        t = int(eng.step_dev) + 1
        eng.run_steps(b, 1, use_graph=use_graph)
        torch.cuda.synchronize()
        assert int(eng.step_dev) == t
        assert not _bits(eng.G).any(), "G is not all +0.0 after step %d" % b       # the next step accumulates into it
        s0 = b * eng.B
        nb = min(eng.B, eng.T - s0)
        u, i, j = (x[s0:s0 + nb].long() for x in (eng.tu, eng.ti, eng.tj))
        ref = ref_step(csr, p0, m0, v0, t, u, i, j, eng.L, eng.reg, eng.lr, eng.betas, eng.adam_eps)
        bnd = step_bounds(ref, p0, u, i, j, eng.L, eng.reg, run, eng.U)
        rows = torch.unique(torch.cat([u, eng.U + i, eng.U + j]))
        got = dict(loss4=eng.out4[b], F=eng.F, m=eng.m, v=eng.v, p=eng.E0)
        if not eng.fuse_adam:
            got["g"] = eng.dE0
        r = check_step(got, ref, bnd, p0, m0, v0, rows)
        _record(group, r)
        assert max(r.values()) <= 1.0, (b, t, r)
    return csr, run


def _set_triples(eng, eu, ei, seed=1):
    U, I = eng.U, eng.N - eng.U
    eng.set_triples(*_triples(eu, ei, U, I, eng.B, eng.cap, seed))


@pytest.mark.gpu
@pytest.mark.parametrize("L", [1, 2, 3, 4, 9])
@pytest.mark.parametrize("g_mask", [True, False])
def test_step_matches_reference_over_layers(L, g_mask):
    """d = 64; 12 B <= N: the batch bitmap gates G in the backward layers; 12 B > N: G is read at every row.  A partial
    last batch (T = 4 B + 37)."""
    B = 128 if g_mask else 256
    eng, eu, ei = _small_engine(L, 64, B, 4 * B + 37, seed=L)
    assert (12 * eng.B <= eng.N) == g_mask
    _set_triples(eng, eu, ei)
    teacher_forced(eng, range(eng.n_batches), True, "L=%d %s" % (L, "masked G" if g_mask else "full G"))


@pytest.mark.gpu
@pytest.mark.parametrize("d", [8, 16, 32, 128, 256])
def test_step_matches_reference_over_widths(d):
    """L = 3.  d = 8: 32-entry work-list segments, the first backward layer without the column mask"""
    eng, eu, ei = _small_engine(3, d, 128, 4 * 128 + 37, seed=d)
    if d == 8:
        assert eng.wl_segment == 32
    _set_triples(eng, eu, ei)
    teacher_forced(eng, range(eng.n_batches), True, "d=%d" % d)


@pytest.mark.gpu
@pytest.mark.parametrize("use_graph", [False, True])
@pytest.mark.parametrize("segment", ["64", "256"])
@pytest.mark.parametrize("coef_stream", ["0", "1"])
@pytest.mark.parametrize("persistent", ["0", "1"])
@pytest.mark.parametrize("fuse_adam", ["0", "1"])
@pytest.mark.parametrize("worklists", ["0", "1"])
def test_step_matches_reference_flag_product(monkeypatch, worklists, fuse_adam, persistent, coef_stream, segment,
                                             use_graph):
    """L = 3, d = 64, G gated by the batch bitmap; segment 256 runs the plan of the large graphs on a small one"""
    import arlib_b200.graph as graphmod
    monkeypatch.setenv("ARLIB_B200_WORKLISTS", worklists)
    monkeypatch.setenv("ARLIB_B200_FUSE_ADAM", fuse_adam)
    monkeypatch.setenv("ARLIB_B200_COEF_STREAM", coef_stream)
    monkeypatch.setattr(graphmod, "PERSISTENT_ENV", persistent)
    monkeypatch.setattr(graphmod, "SEGMENT_ENV", segment)
    eng, eu, ei = _small_engine(3, 64, 128, 4 * 128 + 37, seed=3)
    assert eng.g.segment == int(segment) and eng.g.persistent == (persistent == "1")
    assert (eng.wl is not None) == (worklists == "1") and eng.fuse_adam == (fuse_adam == "1")
    assert (eng._coef_stream is not None) == (coef_stream == "1")
    _set_triples(eng, eu, ei)
    teacher_forced(eng, range(eng.n_batches), use_graph, "flags")


@pytest.mark.gpu
@pytest.mark.parametrize("g_mask", [True, False])
def test_step_matches_reference_single_partial_batch(g_mask):
    B = 128 if g_mask else 256
    eng, eu, ei = _small_engine(2, 64, B, B - 19, seed=5)
    _set_triples(eng, eu, ei)
    assert eng.n_batches == 1
    for _ in range(4):
        teacher_forced(eng, [0], True, "nb=1")


@pytest.mark.gpu
def test_step_matches_reference_with_the_device_sampler():
    from arlib_b200.engine import DeviceTrainSet
    U, I = 800, 1000
    eu, ei = _edges(U, I, 12000, 7)
    eng, _, _ = _small_engine(3, 64, 128, eu.shape[0], seed=7)
    eng.sample_epoch(DeviceTrainSet.from_arrays(eu, ei, U, I, DEV), seed=11, epoch=0)
    assert eng.T % eng.B
    teacher_forced(eng, [0, 1, 2, 3, eng.n_batches - 1], True, "sampler")


@pytest.mark.gpu
def test_bounds_reject_perturbed_references():
    """the comparison catches (a) one edge of the hub row dropped from A, (b) one triple's negative item replaced,
    (c) the Adam step off by one and (d) one row's momentum not decayed, on real kernel output"""
    eng, eu, ei = _small_engine(2, 64, 128, 4 * 128 + 37, seed=11)
    _set_triples(eng, eu, ei)
    csr, run = teacher_forced(eng, [0], True, "perturbations")
    b = 1
    p0, m0, v0 = eng.E0.clone(), eng.m.clone(), eng.v.clone()
    t = int(eng.step_dev) + 1
    eng.run_steps(b, 1, use_graph=True)
    torch.cuda.synchronize()
    got = dict(loss4=eng.out4[b], F=eng.F, m=eng.m, v=eng.v, p=eng.E0)
    s0, nb = b * eng.B, eng.B
    u, i, j = (x[s0:s0 + nb].long() for x in (eng.tu, eng.ti, eng.tj))
    rows = torch.unique(torch.cat([u, eng.U + i, eng.U + j]))
    assert int(u[0]) == 0                                    # the hub user is in the batch

    def check(csr_, t_, j_, edit=None):
        ref = ref_step(csr_, p0, m0, v0, t_, u, i, j_, eng.L, REG, LR)
        if edit:
            edit(ref)
        bnd = step_bounds(ref, p0, u, i, j_, eng.L, REG, run, eng.U)
        return check_step(got, ref, bnd, p0, m0, v0, rows)

    r = check(csr, t, j)
    _record("perturbations", r)
    assert max(r.values()) <= 1.0, r
    rp, col, val = csr.rowptr.clone(), csr.col, csr.val
    k = int(rp[0]) + 5                                      # one entry of row 0 (the hub user, > 700 entries)
    assert int(rp[1]) - int(rp[0]) > 700
    rp[1:] -= 1
    dropped = RefCSR(rp, torch.cat([col[:k], col[k + 1:]]), torch.cat([val[:k], val[k + 1:]]), csr.n_users)
    j2 = j.clone()
    j2[17] = (j2[17] + 1) % (eng.N - eng.U)
    # a row with momentum, and no gradient this step if there is one (more than L hops from the batch)
    g0 = ref_step(csr, p0, m0, v0, t, u, i, j, eng.L, REG, LR)["g"]
    moving = (m0 != 0).any(1)
    idle = torch.nonzero(moving & (g0 == 0).all(1)).flatten()
    row = int(idle[0]) if idle.numel() else int(torch.nonzero(moving).flatten()[0])

    def not_decayed(ref):
        ref["m"][row] = m0[row].double() + (1 - ref["b1"]) * ref["g"][row]

    caught = {}
    for name, r in (("(a) edge dropped", check(dropped, t, j)), ("(b) negative replaced", check(csr, t, j2)),
                    ("(c) step off by one", check(csr, t + 1, j)), ("(d) momentum not decayed", check(csr, t, j, not_decayed))):
        caught[name] = sorted(k for k, x in r.items() if x > 1.0)
        assert caught[name], (name, r)
    print("\nperturbations rejected by: %s" % caught)


def _bench_graph(name):
    import scipy.sparse as sp
    from bench import make_data
    from arlib_b200.graph import DeviceGraph
    D = make_data(name, 0.5)
    U, I, E = D["U"], D["I"], D["E"]
    N = U + I
    half = sp.csr_matrix((np.ones(E, dtype=np.float32), (D["tu"], D["ti"] + U)), shape=(N, N), dtype=np.float32)
    return D, DeviceGraph.from_dataloader_adj(half + half.T, DEV)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["gowalla", "amazon-book"])
def test_benchmark_shape_steps_match_reference(name):
    """the configuration bench.py measures: steps 0, 1, 2 and the epoch's last, partial, batch, replayed"""
    from bench import xavier_tables
    from arlib_b200.engine import DeviceTrainSet, LightGCNEngine
    D, g = _bench_graph(name)
    U, I, E, d, B, L = D["U"], D["I"], D["E"], D["d"], D["B"], D["L"]
    ue, ie = xavier_tables(U, I, d)
    eng = LightGCNEngine(g, torch.cat([ue, ie]).to(DEV), U, L, LR, REG, B, E)
    assert 12 * B <= eng.N and eng.wl is not None and eng.fuse_adam
    eng.sample_epoch(DeviceTrainSet.from_arrays(D["tu"], D["ti"], U, I, DEV), 7, 0)
    assert eng.T % B
    teacher_forced(eng, [0, 1, 2, eng.n_batches - 1], True, name)


# ------------------------------------------------------------------------------------------------ d-sharded exchange
def _exchange(F, slices, u, i, j, nb, U, cap, xchg, ctr):
    """every emulated rank's bpr_partial, then every rank's bpr_finish, on one stream"""
    from arlib_b200 import ops
    world = len(slices)
    Fs = [F[:, c0:c1].contiguous() for c0, c1 in slices]
    ptrs = [x.data_ptr() for x in xchg]
    out4 = [torch.zeros(4, device=DEV) for _ in range(world)]
    coef = [torch.zeros(cap, device=DEV) for _ in range(world)]
    ws = [torch.zeros(ops.bpr_ws_bytes(cap), dtype=torch.uint8, device=DEV) for _ in range(world)]
    for r in range(world):
        ops.bpr_partial(Fs[r], u, i, j, nb, U, r, cap, ctr[r], ptrs)
    for r in range(world):
        ops.bpr_finish(xchg[r], world, cap, nb, REG, ctr[r], out4[r], coef[r], ws[r])
    return Fs, out4, coef


@pytest.mark.gpu
@pytest.mark.parametrize("d_full", [64, 128])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_dshard_loss_exchange_emulated_on_one_gpu(world, d_full):
    """bpr_partial / bpr_finish of `world` ranks on one device: out4 and coef equal on every rank and within the bounds of
    the float64 loss, the concatenated bpr_backward slices within those of its gradient; 4 rounds with new tables cover
    both halves of the double buffer twice (stale words would show), nb < cap and nb = cap; a single use without a
    counter"""
    from arlib_b200 import ops
    from arlib_b200.engine import dshard_columns
    U, I, cap = 500, 700, 384
    N = U + I
    slices = [dshard_columns(d_full, world, r) for r in range(world)]
    rng = np.random.default_rng(world * 1000 + d_full)
    gen = torch.Generator(device=DEV).manual_seed(world + d_full)
    xchg = [torch.zeros(ops.bpr_xchg_bytes(cap), dtype=torch.uint8, device=DEV) for _ in range(world)]
    ctr = [torch.zeros(1, dtype=torch.int32, device=DEV) for _ in range(world)]
    occ = torch.empty(3 * cap, dtype=torch.int32, device=DEV)
    seg_off = torch.empty(3 * cap + 1, dtype=torch.int32, device=DEV)
    seg_node = torch.empty(3 * cap, dtype=torch.int32, device=DEV)
    n_seg = torch.zeros(1, dtype=torch.int32, device=DEV)
    rounds = [(cap - 77, True), (cap, True), (129, True), (cap, True), (cap - 5, False)]
    for k, (nb, counted) in enumerate(rounds):
        if not counted:                                      # a single use of fresh zeroed buffers, no counter
            xchg = [torch.zeros_like(x) for x in xchg]
        F = torch.randn(N, d_full, device=DEV, generator=gen) * 0.3
        tu = rng.integers(0, 60, nb)                         # repeated users
        ti, tj = rng.integers(0, I, nb), rng.integers(0, I, nb)
        tj[5] = ti[6]
        u, i, j = (torch.from_numpy(a.astype(np.int32)).to(DEV) for a in (tu, ti, tj))
        Fs, out4, coef = _exchange(F, slices, u, i, j, nb, U, cap, xchg, ctr if counted else [None] * world)
        ops.bpr_group_batches(u, i, j, nb, cap, U, occ, seg_off, seg_node, n_seg)
        Gs = []
        for r in range(world):
            Gs.append(torch.zeros_like(Fs[r]))
            ops.bpr_backward(Fs[r], u, i, j, nb, U, REG, 1.0, out4[r], coef[r], occ, seg_off, seg_node, n_seg, Gs[r])
        torch.cuda.synchronize()
        if counted:
            assert [int(c) for c in ctr] == [k + 1] * world      # each finish advanced its counter by exactly one
        for r in range(1, world):
            assert torch.equal(out4[r], out4[0]) and torch.equal(coef[r][:nb], coef[0][:nb])
        # float64 reference on the fp32 table (no propagation: cF = 0)
        ul, il, jl = u.long(), i.long(), j.long()
        F64 = F.double().requires_grad_(True)
        ue, pe, ne = F64[ul], F64[U + il], F64[U + jl]
        bpr = port.bpr_loss(ue, pe, ne)
        loss = bpr + port.l2_reg_loss(REG, ue, pe)
        grad, = torch.autograd.grad(loss, F64)
        s = torch.sigmoid((ue * (pe - ne)).sum(1)).detach()
        dx = -s * (1 - s) / ((1e-7 + s) * nb)                # d loss / d x_t
        bnd = loss_grad_bounds(F.double().abs(), 0, F.double(), ul, il, jl, U, REG)
        want4 = torch.stack([loss, bpr, ue.norm(), pe.norm()]).detach()
        r = {"loss": _ratio((out4[0].double() - want4).abs(), bnd["loss4"]),
             "coef": _ratio((coef[0][:nb].double() - dx).abs(), bnd["coef"]),
             "G": _ratio((torch.cat(Gs, 1).double() - grad).abs(), bnd["G"])}
        _record("dshard world=%d d=%d" % (world, d_full), r)
        assert max(r.values()) <= 1.0, (k, r)
