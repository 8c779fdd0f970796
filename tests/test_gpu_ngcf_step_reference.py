"""A float64 reference of one NGCF training step (recommender/NGCF.py:48-66 with the encoder of :197-212), and
teacher-forced checks of arlib_b200.engine.NGCFEngine and the dense kernels of csrc/ngcf.cu against it.

ref_ngcf_step runs the step in float64 on the graph's own fp32 values (upcast): the reference expression per layer
(P = A E, Z = [P + E | P * E] [W1 ; W2], E' = leaky_relu(Z, 0.01)), the BPR + L2 loss on F = mean_k E_k, a hand-written
backward that keeps every intermediate the engine keeps (pinned to autograd and to port.NGCFTrainer on the CPU), and
the Adam of include/agcf.h on the table and on W at the same step t.  ngcf_fwd_bounds / ngcf_bwd_bounds derive an
elementwise bound of every fp32 output from the arithmetic the kernels do (SpMM chains, one rounding per element-wise
operation, 2d- and d-long fmaf chains, the dW chain of the persistent CTAs or split-K slices): no tuned tolerance.

leaky_relu's branch: an element whose |Z| lies within Z's forward bound is ambiguous -- the fp32 kernel may take either
branch.  The backward then takes the branch the kernel took (E_k > 0, read from the engine); everywhere else the
kernel's branch must equal the reference's.  The ambiguous elements are counted and printed.

The GPU cases: the dense kernels alone at every width and at the row counts where their tiles, persistent loops and
split-K slices change shape; the engine over layers, widths, batch edges, eager launches and graph replay, the device
sampler, the benchmark shapes (Gowalla, Amazon-book) and the row-partitioned layout on one GPU.  The bounds are shown to
reject six small reference-side perturbations."""
import collections
import math
import threading

import numpy as np
import pytest
import torch
import torch.nn.functional as Fn

from oracle import port
from test_gpu_ngcf_rows_one_device import _Ranks, _ThreadComm
from test_gpu_step_reference import (BETAS, DEV, EPS, LR, REG, UNIT, RefCSR, _adj64, _bench_graph, _bits, _edges,
                                     _ratio, _triples, _ulp32, adam_ratios, adam_scalars, far_exact, loss_grad_bounds,
                                     run_length)

SLOPE = 0.01
# the kernels multiply by 0.01f: |fl(0.01f z) - 0.01 z| <= DSLOPE |z|
DSLOPE = abs(float(np.float32(SLOPE)) - SLOPE) + SLOPE * UNIT
N_PARTIALS = {8: 296, 16: 296, 32: 296, 64: 296, 128: 74, 256: 37}       # NGCFEngine.N_PARTIALS (asserted on the GPU)


# ------------------------------------------------------------------------------------------------ float64 reference
def _pick(c, a, b):
    """float64 a where c, else b (torch.where of two Python scalars would round them to float32)"""
    one = torch.ones(c.shape, dtype=torch.float64, device=c.device)
    return torch.where(c, a * one, b * one)


def ngcf_forward64(A, E0, W, f_div=None):
    """layers of the reference expression in float64: P_k = A E_{k-1}, Z_k, E_k = leaky_relu(Z_k); F = mean of
    E_0 .. E_L (f_div: a wrong divisor, for the perturbation test)"""
    L, d = W.shape[0], W.shape[2]
    X = E0.double() if not E0.requires_grad else E0
    Wd = W.double() if not W.requires_grad else W
    Xs, Ps, Zs = [X], [], []
    for k in range(L):
        P = torch.sparse.mm(A, X)
        Z = (P + X) @ Wd[k, :d] + (P * X) @ Wd[k, d:]
        X = Fn.leaky_relu(Z, SLOPE)
        Ps.append(P), Zs.append(Z), Xs.append(X)
    F = sum(Xs) / (L + 1 if f_div is None else f_div)
    return dict(X=Xs, P=Ps, Z=Zs, F=F)


def _loss(F, u, i, j, U, reg):
    ue, pe, ne = F[u], F[U + i], F[U + j]
    bpr = port.bpr_loss(ue, pe, ne)
    return bpr + port.l2_reg_loss(reg, ue, pe), bpr, ue, pe


def ngcf_backward64(A, fw, W, G, pos, slope=SLOPE, swap=None, drop_rows=None):
    """hand-written backward of the step from G = d loss / d F / (L + 1), with leaky_relu's branch `pos` per layer:
    dZ_k, dP_k, dE_direct_k, dW_k and dE_k = d loss / d E_k (dE_0: the gradient of the table).  swap = k: W1 and W2 of
    layer k exchanged here only; drop_rows: rows left out of every dW (both for the perturbation test)."""
    L, d = W.shape[0], W.shape[2]
    Wd = W.double()
    AT = A.t().coalesce()
    out = dict(dZ=[None] * L, dP=[None] * L, dEdir=[None] * L, dW=[None] * L, dE=[None] * (L + 1))
    dE = G
    out["dE"][L] = G
    for k in range(L, 0, -1):
        X, P = fw["X"][k - 1], fw["P"][k - 1]
        dZ = dE * _pick(pos[k - 1], 1.0, slope)
        W1, W2 = (Wd[k - 1, d:], Wd[k - 1, :d]) if swap == k else (Wd[k - 1, :d], Wd[k - 1, d:])
        dA, dB = dZ @ W1.T, dZ @ W2.T
        dP = dA + dB * X
        dEdir = dA + dB * P
        dZw = dZ
        if drop_rows is not None:
            dZw = dZ.clone()
            dZw[drop_rows] = 0.0
        dW = torch.cat([(P + X).T @ dZw, (P * X).T @ dZw])
        dE = torch.sparse.mm(AT, dP) + dEdir + G
        out["dZ"][k - 1], out["dP"][k - 1], out["dEdir"][k - 1], out["dW"][k - 1] = dZ, dP, dEdir, dW
        out["dE"][k - 1] = dE
    return out


def adam64(p, g, m, v, t, lr, betas, eps):
    b1, b2, c1, c2, eps = adam_scalars(t, lr, betas, eps)
    m1 = b1 * m.double() + (1 - b1) * g
    v1 = b2 * v.double() + (1 - b2) * g * g
    p1 = p.double() - c1 * m1 / (v1.sqrt() / c2 + eps)
    return dict(m=m1, v=v1, p=p1, b1=b1, b2=b2, c1=c1, c2=c2, eps=eps)


def ref_ngcf_step(csr, E0, W, m, v, Wm, Wv, t, u, i, j, reg=REG, lr=LR, betas=BETAS, eps=EPS, branch=None, A=None,
                  slope_bwd=SLOPE, f_div=None, swap_bwd=None, w_step=None, drop_rows=None):
    """One NGCF step in float64 from the table E0, W [L, 2d, d], the moments m, v, Wm, Wv and the Adam step t (both
    optimizers use t, as agcf_adam_coefs and agcf_adam_step_f32 read the same counter), on triples (u, i, j).
    branch(fw) -> [bool [N, d]] per layer: leaky_relu's branch in the backward (default Z > 0).  The last five
    arguments perturb the reference (the bounds must reject them)."""
    A = _adj64(csr) if A is None else A
    U, L = csr.n_users, W.shape[0]
    fw = ngcf_forward64(A, E0, W, f_div)
    Fl = fw["F"].detach().clone().requires_grad_(True)
    loss, bpr, ue, pe = _loss(Fl, u, i, j, U, reg)
    gF, = torch.autograd.grad(loss, Fl)
    G = gF / (L + 1 if f_div is None else f_div)
    pos = [Z > 0 for Z in fw["Z"]] if branch is None else branch(fw)
    bw = ngcf_backward64(A, fw, W, G, pos, slope_bwd, swap_bwd, drop_rows)
    tab = adam64(E0, bw["dE"][0], m, v, t, lr, betas, eps)
    dW = torch.stack(bw["dW"])
    wad = adam64(W, dW, Wm, Wv, t if w_step is None else w_step, lr, betas, eps)
    with torch.no_grad():
        loss4 = torch.stack([loss, bpr, ue.norm(), pe.norm()])
    return dict(A=A, U=U, L=L, fw=fw, F=fw["F"], G=G, gF=gF, pos=pos, bw=bw, loss4=loss4, g=bw["dE"][0], dW=dW,
                tab=tab, wad=wad)


# ------------------------------------------------------------------------------------------------ error bounds
def dw_chain(n, d, n_partials):
    """longest fp32 chain of one dW element: the rows one CTA (d <= 64: 128-row tiles at d <= 16, 64-row tiles above)
    or one split-K slice (d >= 128: 64-row chunks) accumulates, then the partials summed in order"""
    tile = 128 if d <= 16 else 64
    per = -(-(-(-n // tile)) // n_partials)
    return per * tile + n_partials


def dense_fwd_bounds(P, X, eP, eX, W):
    """Z = [P + X | P * X] W from fp32 P, X within eP, eX of the float64 P, X: P + X and P * X one rounding each, Z a
    2d-long fmaf chain (2d UNIT of the sum of |terms|).  Then E' = leaky_relu(Z): 1-Lipschitz, the slope product one
    rounding of 0.01f (DSLOPE); ambiguous where |Z| <= eZ."""
    d = X.shape[1]
    Wa = W.double().abs()
    Pa, Xa = P.abs() + eP, X.abs() + eX
    S, M = P + X, P * X
    eS = eP + eX + UNIT * (S.abs() + eP + eX)
    eM = eP * Xa + Pa * eX + UNIT * M.abs()
    Sa, Ma = S.abs() + eS, M.abs() + eM
    Z = S @ W.double()[:d] + M @ W.double()[d:]
    eZ = eS @ Wa[:d] + eM @ Wa[d:] + 2 * d * UNIT * (Sa @ Wa[:d] + Ma @ Wa[d:])
    Y = Fn.leaky_relu(Z, SLOPE)
    amb = Z.abs() <= eZ
    eY = torch.where(Z > eZ, eZ, torch.where(Z < -eZ, SLOPE * eZ + DSLOPE * Z.abs(), eZ + DSLOPE * (Z.abs() + eZ)))
    return dict(S=S, M=M, eS=eS, eM=eM, Sa=Sa, Ma=Ma, Z=Z, eZ=eZ, Y=Y, eY=eY, amb=amb)


def dense_bwd_bounds(dE, edE, pos, P, X, eP, eX, fb, W, chain):
    """the dense backward from fp32 dE' within edE: dZ one rounding on the slope branch (pos = the kernel's branch),
    [dA | dB] = dZ W^T d-long chains, dP = fmaf(dB, X, dA) and dE_direct = fmaf(dB, P, dA) one rounding each, dW =
    A'^T dZ a chain of `chain` roundings over the magnitudes [|P + X| | |P * X|]^T |dZ|"""
    d = X.shape[1]
    Wa = W.double().abs()
    s = _pick(pos, 1.0, SLOPE)
    dZ = dE * s
    edZ = s * edE + _pick(pos, 0.0, DSLOPE) * (dE.abs() + edE)
    dZa = dZ.abs() + edZ
    W1a, W2a = Wa[:d], Wa[d:]
    dA, dB = dZ @ W.double()[:d].T, dZ @ W.double()[d:].T
    edA = edZ @ W1a.T + d * UNIT * (dZa @ W1a.T)
    edB = edZ @ W2a.T + d * UNIT * (dZa @ W2a.T)
    dAa, dBa = dA.abs() + edA, dB.abs() + edB
    Pa, Xa = P.abs() + eP, X.abs() + eX
    edP = edA + edB * Xa + dBa * eX + UNIT * (dAa + dBa * Xa)
    edEdir = edA + edB * Pa + dBa * eP + UNIT * (dAa + dBa * Pa)
    Aa = torch.cat([fb["Sa"], fb["Ma"]], 1)
    eAp = torch.cat([fb["eS"], fb["eM"]], 1)
    edW = eAp.T @ dZa + Aa.T @ edZ + chain * UNIT * (Aa.T @ dZa)
    return dict(dZ=edZ, dP=edP, dEdir=edEdir, dW=edW, dPa=(dA + dB * X).abs() + edP, dEdira=(dA + dB * P).abs() + edEdir)


def ngcf_fwd_bounds(A, fw, W, run):
    """per layer: P_k a SpMM chain ((run + 1) UNIT of A |E_{k-1}| plus A times the input's error), then
    dense_fwd_bounds; F = ((E_0 + E_1) + ... + E_L) / (L + 1): L adds and the division"""
    L = W.shape[0]
    e = torch.zeros_like(fw["X"][0])
    eX, eP, lay = [e], [], []
    for k in range(L):
        X = fw["X"][k]
        Pabs = torch.sparse.mm(A, X.abs() + e)
        ep = torch.sparse.mm(A, e) + (run + 1) * UNIT * Pabs
        fb = dense_fwd_bounds(fw["P"][k], X, ep, e, W[k])
        e = fb["eY"]
        eP.append(ep), lay.append(fb), eX.append(e)
    Sa = sum(x.abs() + ex for x, ex in zip(fw["X"], eX))
    eF = (sum(eX) + L * UNIT * Sa) / (L + 1) + UNIT * fw["F"].abs()
    return dict(eP=eP, eX=eX, lay=lay, eF=eF)


def ngcf_bwd_bounds(ref, fb, W, run, chain, u, i, j, reg):
    """G from loss_grad_bounds (the fp32 F within eF; scaled by fl(1 / (L + 1)): two more roundings), then per layer
    dense_bwd_bounds and dE_{k-1} = A dP + dE_direct + G: the SpMM chain and two additions.  Rows more than L hops
    from the batch have a zero gradient (far)."""
    A, U, L, fw = ref["A"], ref["U"], ref["L"], ref["fw"]
    F = fw["F"]
    lg = loss_grad_bounds(F.abs() + fb["eF"], 0, F, u, i, j, U, reg, eF=fb["eF"])
    s = 1.0 / (L + 1)
    eG = s * lg["G"] + 2 * UNIT * s * lg["Gabs"]
    Ga = s * lg["Gabs"] + eG
    out = dict(loss4=lg["loss4"], F=fb["eF"], dZ=[None] * L, dP=[None] * L, dEdir=[None] * L, dW=[None] * L,
               dE=[None] * (L + 1))
    edE = eG
    out["dE"][L] = eG
    for k in range(L, 0, -1):
        b = dense_bwd_bounds(ref["bw"]["dE"][k], edE, ref["pos"][k - 1], fw["P"][k - 1], fw["X"][k - 1],
                             fb["eP"][k - 1], fb["eX"][k - 1], fb["lay"][k - 1], W[k - 1], chain)
        tA = torch.sparse.mm(A, b["dPa"])
        edE = torch.sparse.mm(A, b["dP"]) + (run + 1) * UNIT * tA + b["dEdir"] + eG \
            + 2 * UNIT * (tA + b["dEdira"] + Ga)
        for key in ("dZ", "dP", "dEdir", "dW"):
            out[key][k - 1] = b[key]
        out["dE"][k - 1] = edE
    seed = torch.zeros(F.shape[0], 1, dtype=torch.float64, device=F.device)
    seed[torch.cat([u, U + i, U + j])] = 1.0
    far = seed[:, 0] == 0
    for _ in range(L):
        seed = torch.sparse.mm(A, seed)
        far &= seed[:, 0] == 0
    out["far"] = far
    return out


# ------------------------------------------------------------------------------------------------ comparison
RATIOS = collections.defaultdict(dict)
AMBIGUOUS = collections.defaultdict(lambda: [0, 0])


def _record(group, r):
    for k, x in r.items():
        RATIOS[group][k] = max(RATIOS[group].get(k, 0.0), x)


@pytest.fixture(scope="module", autouse=True)
def _report_ratios():
    yield
    for group, r in sorted(RATIOS.items()):
        amb = AMBIGUOUS.get(group)
        extra = "; ambiguous branches %d of %d" % tuple(amb) if amb else ""
        print("\nlargest error / bound [%s]: %s%s" % (group, ", ".join("%s %.3g" % kv for kv in sorted(r.items())), extra))


def _r(got, want, bound, rows=None):
    if rows is not None:
        got, want, bound = got[rows], want[rows], bound[rows]
    return _ratio((got.double() - want).abs(), bound)


def kernel_branch(gotE, fb_of, group=None):
    """branch(fw) for ref_ngcf_step: the kernel's branch (E_k > 0).  The holder it returns keeps the forward bounds
    (fb_of(fw) -> ngcf_fwd_bounds) and the number of elements whose branch differs from the reference's although |Z_k|
    exceeds its forward bound (must be 0)."""
    held = {"wrong": 0}

    def branch(fw):
        fb = fb_of(fw)
        held["fb"] = fb
        pos = []
        for k, lay in enumerate(fb["lay"]):
            kp = gotE[k] > 0
            amb = lay["amb"]
            held["wrong"] += int(((kp != (lay["Z"] > 0)) & ~amb).sum())
            if group is not None:
                AMBIGUOUS[group][0] += int(amb.sum())
                AMBIGUOUS[group][1] += amb.numel()
            pos.append(kp)
        return pos

    return branch, held


def compare_step(got, ref, fb, bb, st0, rows=None):
    """max(error / bound) per output of one engine step.  got / st0: the engine's tables after / before the step (see
    _got); rows: the rows each table holds (row-partitioned: every rank's own rows assembled, so all of them)."""
    L, bw = ref["L"], ref["bw"]
    fw = ref["fw"]
    r = {"loss": _ratio((got["out4"].double() - ref["loss4"]).abs(), bb["loss4"]),
         "F": _r(got["F"], ref["F"], bb["F"])}
    r["P"] = max(_r(got["P"][k], fw["P"][k], fb["eP"][k]) for k in range(L))
    r["E"] = max(_r(got["E"][k], fw["X"][k + 1], fb["eX"][k + 1]) for k in range(L))
    r["dE"] = max([_r(x, bw["dE"][k], bb["dE"][k]) for k, x in got["dE"].items()] + [0.0])
    r["dP"] = max(_r(x, bw["dP"][k - 1], bb["dP"][k - 1]) for k, x in got["dP"].items())
    r["dEdir"] = _r(got["dEdir1"], bw["dEdir"][0], bb["dEdir"][0])
    dW = ref["dW"]
    edW = torch.stack(bb["dW"])
    r["dW"] = _r(got["dW"], dW, edW)
    tab, wad = ref["tab"], ref["wad"]
    for name, x in adam_ratios(tab, ref["g"], bb["dE"][0], tab["m"], tab["v"], st0["E0"], st0["m"], st0["v"],
                               got["m"], got["v"], got["E0"]).items():
        r["table " + name] = x
    W0 = st0["W"]
    for name, x in adam_ratios(wad, dW.flatten(1), edW.flatten(1), wad["m"].flatten(1), wad["v"].flatten(1),
                               W0.flatten(1), st0["Wm"].flatten(1), st0["Wv"].flatten(1), got["Wm"].flatten(1),
                               got["Wv"].flatten(1), got["W"].flatten(1)).items():
        r["W " + name] = x
    exact = far_exact(ref["g"], bb["far"], st0["E0"], st0["m"], st0["v"], got["m"], got["v"], got["E0"])
    r["exact"] = 0.0 if exact else math.inf
    return r


def _state(eng):
    return {k: getattr(eng, k).clone() for k in ("E0", "m", "v", "W", "Wm", "Wv")}


def _got(eng, b):
    """the single-GPU engine's outputs of step b: every table it keeps.  dOut holds dE_1 (L >= 2) and dE_2 (L >= 3);
    dPs[0] and dEdir layer 1's"""
    L = eng.L
    dE = {}
    if L >= 2:
        dE[1] = eng.dOut[0]
    if L >= 3:
        dE[2] = eng.dOut[1]
    return dict(out4=eng.out4[b], F=eng.F, P=eng.P, E=eng.Ek, dE=dE, dP={1: eng.dPs[0]}, dEdir1=eng.dEdir, dW=eng.dW,
                W=eng.W, Wm=eng.Wm, Wv=eng.Wv, E0=eng.E0, m=eng.m, v=eng.v)


def _batch(eng, b):
    s0 = b * eng.B
    nb = min(eng.B, eng.T - s0)
    return tuple(x[s0:s0 + nb].long() for x in (eng.tu, eng.ti, eng.tj))


def check_against_reference(csr, A, st0, t, u, i, j, got, run, chain, group, **perturb):
    """ref_ngcf_step from st0 with the kernel's branch, the bounds, compare_step"""
    fb_of = lambda fw: ngcf_fwd_bounds(A, fw, st0["W"], run)
    branch, held = kernel_branch(got["E"], fb_of, group)
    ref = ref_ngcf_step(csr, st0["E0"], st0["W"], st0["m"], st0["v"], st0["Wm"], st0["Wv"], t, u, i, j, branch=branch,
                        A=A, **perturb)
    fb = held["fb"]
    bb = ngcf_bwd_bounds(ref, fb, st0["W"], run, chain, u, i, j, REG)
    r = compare_step(got, ref, fb, bb, st0)
    r["branch"] = math.inf if held["wrong"] else 0.0
    return r


def ngcf_teacher_forced(eng, steps, use_graph, group):
    """For each step b: read the state, run the step, compare every output with ref_ngcf_step from what was read."""
    assert eng.N_PARTIALS == N_PARTIALS
    csr = RefCSR(eng.g.rowptr, eng.g.col, eng.g.val, eng.U)
    A = _adj64(csr)
    run = run_length(eng.g)
    chain = dw_chain(eng.N, eng.d, eng.dW_partial.shape[0])
    for b in steps:
        st0 = _state(eng)
        t = int(eng.step_dev) + 1
        eng.run_steps(b, 1, use_graph=use_graph)
        torch.cuda.synchronize()
        assert int(eng.step_dev) == t, "step_dev did not advance by one"
        assert not _bits(eng.G).any(), "G is not all +0.0 after step %d" % b
        u, i, j = _batch(eng, b)
        r = check_against_reference(csr, A, st0, t, u, i, j, _got(eng, b), run, chain, group)
        _record(group, r)
        assert max(r.values()) <= 1.0, (group, b, t, r)
    return csr, A, run, chain


def _init_params(N, d, L, seed):
    """xavier-uniform table and W (the reference's initializer, recommender/NGCF.py:176-183)"""
    gen = torch.Generator().manual_seed(seed)
    a = (6.0 / (N + d)) ** 0.5
    table = (torch.rand(N, d, generator=gen) * 2 - 1) * a
    W = (torch.rand(L, 2 * d, d, generator=gen) * 2 - 1) * (6.0 / (2 * d)) ** 0.5
    return table.to(DEV), W.to(DEV).contiguous()


def _graph(U, I, n_edges, seed):
    from arlib_b200.graph import DeviceGraph
    eu, ei = _edges(U, I, n_edges, seed)
    return DeviceGraph.from_dataloader_adj(port.bipartite_adjacency(eu, ei, U, I), DEV), eu, ei


def _ngcf_engine(L, d, B, T, seed=0, U=800, I=1000, n_edges=12000):
    from arlib_b200.engine import NGCFEngine
    g, eu, ei = _graph(U, I, n_edges, seed)
    table, W = _init_params(U + I, d, L, seed + d)
    return NGCFEngine(g, table, W, U, LR, REG, B, T), eu, ei


def _set_triples(eng, eu, ei, seed=1):
    eng.set_triples(*_triples(eu, ei, eng.U, eng.N - eng.U, eng.B, eng.cap, seed))


# ------------------------------------------------------------------------------------------------ CPU
def _cpu_problem(L, d=8, U=40, I=60, seed=0):
    rng = np.random.default_rng(seed)
    key = np.unique(rng.integers(0, U, 300) * I + rng.integers(0, I, 300))
    adj = port.bipartite_adjacency(key // I, key % I, U, I)
    norm = port.normalize_graph_mat(adj).tocsr()
    norm.sort_indices()
    csr = RefCSR(torch.from_numpy(norm.indptr.astype(np.int64)), torch.from_numpy(norm.indices.astype(np.int64)),
                 torch.from_numpy(norm.data.astype(np.float32)), U)
    gen = torch.Generator().manual_seed(seed + 1)
    a = (6.0 / (U + I + d)) ** 0.5
    E = ((torch.rand(U + I, d, generator=gen) * 2 - 1) * a).double()
    W = ((torch.rand(L, 2 * d, d, generator=gen) * 2 - 1) * (6.0 / (2 * d)) ** 0.5).double()
    return norm, csr, E, W, rng


@pytest.mark.parametrize("L", [1, 2, 3])
def test_ref_ngcf_step_matches_the_oracle_trainer_with_torch_adam(one_cpu_thread, L):
    """ref_ngcf_step against port.NGCFTrainer in float64 under torch.optim.Adam (scalars rounded to fp32 as the ABI takes
    them), three steps: loss, table, W and every moment to 1e-12"""
    U, I, d = 40, 60, 8
    norm, csr, E, W, rng = _cpu_problem(L, d, U, I, seed=L)
    b1, b2, _, _, eps = adam_scalars(1, LR, BETAS, EPS)
    lr = float(np.float32(LR))
    tr = port.NGCFTrainer(norm, E[:U], E[U:], [W[k, :d] for k in range(L)], [W[k, d:] for k in range(L)], lr, REG)
    tr.adj = tr.adj.double()
    params = [tr.user_emb, tr.item_emb] + tr.w1 + tr.w2
    tr.opt = torch.optim.Adam(params, lr=lr, betas=(b1, b2), eps=eps)
    m, v = torch.zeros_like(E), torch.zeros_like(E)
    Wm, Wv = torch.zeros_like(W), torch.zeros_like(W)
    for t in (1, 2, 3):
        u = torch.from_numpy(rng.integers(0, U, 50))
        i = torch.from_numpy(rng.integers(0, I, 50))
        j = torch.from_numpy(rng.integers(0, I, 50))
        ref = ref_ngcf_step(csr, E, W, m, v, Wm, Wv, t, u, i, j)
        loss = tr.step(u, i, j)
        assert abs(loss - float(ref["loss4"][0])) <= 1e-12 * abs(loss)
        st = lambda ps, key: [tr.opt.state[p][key] for p in ps]
        Wcat = lambda ws: torch.stack([torch.cat([a, b]) for a, b in zip(ws[:L], ws[L:])])
        ws = tr.w1 + tr.w2
        for name, got, want in (
                ("p", ref["tab"]["p"], torch.cat([tr.user_emb.detach(), tr.item_emb.detach()])),
                ("m", ref["tab"]["m"], torch.cat(st([tr.user_emb, tr.item_emb], "exp_avg"))),
                ("v", ref["tab"]["v"], torch.cat(st([tr.user_emb, tr.item_emb], "exp_avg_sq"))),
                ("W", ref["wad"]["p"], Wcat([w.detach() for w in ws])),
                ("Wm", ref["wad"]["m"], Wcat(st(ws, "exp_avg"))), ("Wv", ref["wad"]["v"], Wcat(st(ws, "exp_avg_sq")))):
            scale = float(want.abs().max())
            torch.testing.assert_close(got, want, rtol=1e-12, atol=1e-12 * scale, msg=lambda s: name + ": " + s)
        E, W, m, v, Wm, Wv = ref["tab"]["p"], ref["wad"]["p"], ref["tab"]["m"], ref["tab"]["v"], ref["wad"]["m"], \
            ref["wad"]["v"]


@pytest.mark.parametrize("L", [1, 2, 3])
def test_hand_written_backward_equals_autograd(one_cpu_thread, L):
    """every intermediate of ngcf_backward64 -- dE_k, dP_k, dZ_k, dW_k, the table's gradient -- equals autograd's
    gradient of the loss with respect to that node, to 1e-12"""
    U, I, d = 40, 60, 8
    _, csr, E, W, rng = _cpu_problem(L, d, U, I, seed=10 + L)
    A = _adj64(csr)
    u, i, j = (torch.from_numpy(rng.integers(0, n, 50)) for n in (U, I, I))
    E0 = E.clone().requires_grad_(True)
    Wg = W.clone().requires_grad_(True)
    fw = ngcf_forward64(A, E0, Wg)
    loss = _loss(fw["F"], u, i, j, U, REG)[0]
    nodes = [E0, Wg] + fw["X"][1:] + fw["P"] + fw["Z"]
    grads = torch.autograd.grad(loss, nodes)
    gE0, gW, gX, gP, gZ = grads[0], grads[1], grads[2:2 + L], grads[2 + L:2 + 2 * L], grads[2 + 2 * L:]
    ref = ref_ngcf_step(csr, E, W, torch.zeros_like(E), torch.zeros_like(E), torch.zeros_like(W), torch.zeros_like(W),
                        1, u, i, j)
    bw = ref["bw"]
    close = lambda a, b: torch.testing.assert_close(a, b, rtol=1e-12, atol=1e-12 * float(b.abs().max()))
    close(bw["dE"][0], gE0)
    close(ref["dW"], gW)
    for k in range(L):
        close(bw["dE"][k + 1], gX[k])
        close(bw["dP"][k], gP[k])
        close(bw["dZ"][k], gZ[k])


def _fp32_step(csr, E0, W, m, v, Wm, Wv, t, u, i, j):
    """the fused formulation in fp32 on the CPU: P = A E, Z = [P + E | P * E] W, the loss and its gradient by fp32
    autograd of the oracle's loss, the dense backward with fmaf emulated (exact product, one rounding), dE = A dP +
    dE_direct + G, the Adam of include/agcf.h"""
    A32 = _adj64(csr).float()
    L, d = W.shape[0], W.shape[2]
    f = lambda x: x.float()
    fma = lambda a, b, c: (a.double() * b.double() + c.double()).float()
    X = f(E0)
    W32 = f(W)
    Xs, Ps = [X], []
    for k in range(L):
        P = torch.sparse.mm(A32, X)
        Z = torch.cat([P + X, P * X], 1) @ W32[k]
        X = torch.where(Z > 0, Z, np.float32(SLOPE) * Z)
        Ps.append(P), Xs.append(X)
    F = Xs[0]
    for x in Xs[1:]:
        F = F + x
    F = F / np.float32(L + 1)
    Fl = F.clone().requires_grad_(True)
    loss, bpr, ue, pe = _loss(Fl, u, i, j, csr.n_users, np.float32(REG))
    gF, = torch.autograd.grad(loss, Fl)
    G = gF * np.float32(1.0 / (L + 1))
    dE, dWs, got = G, [None] * L, {}
    for k in range(L, 0, -1):
        P, X = Ps[k - 1], Xs[k - 1]
        dZ = torch.where(Xs[k] > 0, dE, np.float32(SLOPE) * dE)
        dA, dB = dZ @ W32[k - 1, :d].T, dZ @ W32[k - 1, d:].T
        dP, dEdir = fma(dB, X, dA), fma(dB, P, dA)
        dWs[k - 1] = torch.cat([P + X, P * X], 1).T @ dZ
        dE = (torch.sparse.mm(A32, dP) + dEdir) + G
        got["dP%d" % k], got["dEdir%d" % k], got["dE%d" % (k - 1)] = dP, dEdir, dE
    b1, b2, c1, c2, eps = (np.float32(x) for x in adam_scalars(t, LR, BETAS, EPS))

    def adam(p, g, m_, v_):
        m1 = m_ + (np.float32(1) - b1) * (g - m_)
        v1 = fma((np.float32(1) - b2) * g, g, v_ * b2)
        return p - c1 * (m1 / (v1.sqrt() / c2 + eps)), m1, v1

    dW = torch.stack(dWs)
    got.update(out4=torch.stack([loss, bpr, ue.norm(), pe.norm()]).detach(), F=F, P=Ps, E=Xs[1:], dW=dW)
    got["E0"], got["m"], got["v"] = adam(f(E0), dE, f(m), f(v))
    got["W"], got["Wm"], got["Wv"] = adam(W32, dW, f(Wm), f(Wv))
    return got


@pytest.mark.parametrize("L", [1, 2, 3])
def test_fp32_cpu_step_lies_within_the_bounds(one_cpu_thread, L):
    """an fp32 restatement of the fused step on the CPU, two steps, is within ngcf_step's bounds with run = the largest
    row degree (any summation order of a row) and the dW chain = N: the bounds are not too tight"""
    U, I, d = 40, 60, 8
    _, csr, E, W, rng = _cpu_problem(L, d, U, I, seed=20 + L)
    E, W = E.float(), W.float()
    m, v, Wm, Wv = torch.zeros_like(E), torch.zeros_like(E), torch.zeros_like(W), torch.zeros_like(W)
    A = _adj64(csr)
    run = int((csr.rowptr[1:] - csr.rowptr[:-1]).max())
    for t in (1, 2):
        u, i, j = (torch.from_numpy(rng.integers(0, n, 50)) for n in (U, I, I))
        i[3] = j[4]
        st0 = dict(E0=E, m=m, v=v, W=W, Wm=Wm, Wv=Wv)
        got32 = _fp32_step(csr, E, W, m, v, Wm, Wv, t, u, i, j)
        got = dict(out4=got32["out4"], F=got32["F"], P=got32["P"], E=got32["E"],
                   dE={k: got32["dE%d" % k] for k in range(L)}, dP={k: got32["dP%d" % k] for k in range(1, L + 1)},
                   dEdir1=got32["dEdir1"], dW=got32["dW"], W=got32["W"], Wm=got32["Wm"], Wv=got32["Wv"],
                   E0=got32["E0"], m=got32["m"], v=got32["v"])
        r = check_against_reference(csr, A, st0, t, u, i, j, got, run, U + I, "cpu fp32 L=%d" % L)
        _record("cpu fp32 L=%d" % L, r)
        assert max(r.values()) <= 1.0, (L, t, r)
        E, W, m, v, Wm, Wv = got32["E0"], got32["W"], got32["m"], got32["v"], got32["Wm"], got32["Wv"]


def test_dw_chain_follows_the_persistent_loop():
    """a CTA (slice) reaches a second tile (chunk) only past N_PARTIALS tiles"""
    assert dw_chain(18944, 64, 296) == 64 + 296 and dw_chain(18945, 64, 296) == 128 + 296
    assert dw_chain(37888, 16, 296) == 128 + 296 and dw_chain(37889, 8, 296) == 256 + 296
    assert dw_chain(70839, 128, 74) == 15 * 64 + 74 and dw_chain(70839, 256, 37) == 30 * 64 + 37
    assert dw_chain(0, 64, 296) == 296 and dw_chain(1, 64, 1) == 65


# ------------------------------------------------------------------------------------------------ GPU: dense kernels
def _dense_rows(d):
    """row counts where the kernels change shape: the forward's row tile, the backward's tile (d >= 128: split-K chunk),
    one tile per persistent CTA (slice) and past it, three rounds of the persistent loop, the Gowalla table"""
    tf = 64 if d in (32, 64) else 128
    tb = 128 if d <= 16 else 64
    C = N_PARTIALS[d]
    ns = {1, tf - 1, tf, tf + 1, tb - 1, tb + 1, 5 * tb + 3, C * tb - 1, C * tb + 1, 3 * C * tb + 37, 70839}
    cases = [(n, C) for n in sorted(ns)]
    cases += [(3 * C * tb + 37, 1), (3 * C * tb + 37, 3), (tb + 1, 3)]
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("d", [8, 16, 32, 64, 128, 256])
def test_dense_kernels_match_float64(d):
    """agcf_ngcf_dense_forward / backward / reduce_wgrad elementwise against float64 within dense_fwd_bounds /
    dense_bwd_bounds: n = 1 .. 3 rounds of the persistent loop (and 70 839), n_partials = 1, 3, N_PARTIALS[d] and more
    partials than tiles; rows with Z = 0 and with P + E = 0; acc_in aliasing acc_out; dW bit-equal across two runs;
    n = 0 gives dW = +0.0"""
    from arlib_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(d)
    worst = collections.defaultdict(float)
    amb, total = 0, 0
    for n, n_part in _dense_rows(d):
        P = torch.randn(n, d, device=DEV, generator=gen) * 0.5
        X = torch.randn(n, d, device=DEV, generator=gen) * 0.5
        W = torch.randn(2 * d, d, device=DEV, generator=gen) / (2 * d) ** 0.5
        dOut = torch.randn(n, d, device=DEV, generator=gen)
        P[:2], X[:2] = 0.0, 0.0                               # Z = 0 exactly: the slope branch on both sides
        if n > 3:
            P[2] = -X[2]                                      # P + E = 0
        acc = torch.randn(n, d, device=DEV, generator=gen)
        div = 4.0 if n % 2 else 1.0
        Y = torch.full_like(P, float("nan"))
        mean = acc.clone()
        ops.ngcf_dense_forward(P, X, W, Y, acc_in=mean, acc_out=mean, acc_div=div)      # in place, as layers k >= 2
        WT = W.t().contiguous()
        dP, dEdir = torch.full_like(P, float("nan")), torch.full_like(P, float("nan"))
        part = torch.full((n_part, 2 * d * d), float("nan"), device=DEV)
        dW, dW2 = torch.full((2 * d, d), float("nan"), device=DEV), torch.full((2 * d, d), float("nan"), device=DEV)
        ops.ngcf_dense_backward(dOut, Y, P, X, WT, dP, dEdir, part, dW)
        ops.ngcf_dense_backward(dOut, Y, P, X, WT, dP, dEdir, part, dW2)
        torch.cuda.synchronize()
        assert np.array_equal(_bits(dW), _bits(dW2)), (d, n, n_part)
        P64, X64, z = P.double(), X.double(), torch.zeros(n, d, dtype=torch.float64, device=DEV)
        fb = dense_fwd_bounds(P64, X64, z, z, W)
        pos = Y > 0
        wrong = (pos != (fb["Z"] > 0)) & ~fb["amb"]
        assert not bool(wrong.any()), (d, n, int(wrong.sum()))
        amb, total = amb + int(fb["amb"].sum()), total + fb["amb"].numel()
        want_m = (acc.double() + fb["Y"]) / div
        em = (fb["eY"] + UNIT * (acc.double().abs() + fb["Y"].abs() + fb["eY"])) / div + UNIT * want_m.abs()
        bb = dense_bwd_bounds(dOut.double(), z, pos, P64, X64, z, z, fb, W, dw_chain(n, d, n_part))
        s = _pick(pos, 1.0, SLOPE)
        dZ = dOut.double() * s
        W64 = W.double()
        dA, dB = dZ @ W64[:d].T, dZ @ W64[d:].T
        wantW = torch.cat([fb["S"].T @ dZ, fb["M"].T @ dZ])
        r = {"E'": _r(Y, fb["Y"], fb["eY"]), "mean": _r(mean, want_m, em), "dP": _r(dP, dA + dB * X64, bb["dP"]),
             "dEdir": _r(dEdir, dA + dB * P64, bb["dEdir"]), "dW": _r(dW, wantW, bb["dW"])}
        for k, x in r.items():
            worst[k] = max(worst[k], x)
        assert max(r.values()) <= 1.0, (d, n, n_part, r)
    # no rows: the weight gradient is +0.0 (the partials of CTAs without a tile are zero-initialised accumulators).
    # Through the C ABI: an empty tensor's data_ptr() is null, which the ABI rejects
    from arlib_b200 import _lib
    rows, outs = torch.zeros(4, d, device=DEV), torch.zeros(2, 4, d, device=DEV)
    WT = torch.zeros(d, 2 * d, device=DEV)
    part = torch.full((N_PARTIALS[d], 2 * d * d), float("nan"), device=DEV)
    dW = torch.full((2 * d, d), float("nan"), device=DEV)
    _lib.check(_lib.load().agcf_ngcf_dense_backward(rows.data_ptr(), rows.data_ptr(), rows.data_ptr(), rows.data_ptr(),
                                                    WT.data_ptr(), outs[0].data_ptr(), outs[1].data_ptr(),
                                                    part.data_ptr(), part.shape[0], 0, d, _lib.stream_ptr()),
               "agcf_ngcf_dense_backward")
    ops.ngcf_reduce_wgrad(part, dW)
    torch.cuda.synchronize()
    assert not _bits(outs).any(), "n = 0 wrote rows"
    assert not _bits(dW).any(), "n = 0: dW is not +0.0"
    _record("dense d=%d" % d, dict(worst))
    AMBIGUOUS["dense d=%d" % d][0] += amb
    AMBIGUOUS["dense d=%d" % d][1] += total


# ------------------------------------------------------------------------------------------------ GPU: the engine
@pytest.mark.gpu
@pytest.mark.parametrize("L", [1, 2, 3, 4])
def test_ngcf_step_matches_reference_over_layers(L):
    """d = 64, B = 128, a partial last batch (T = 4 B + 37), replayed"""
    eng, eu, ei = _ngcf_engine(L, 64, 128, 4 * 128 + 37, seed=L)
    _set_triples(eng, eu, ei)
    ngcf_teacher_forced(eng, range(eng.n_batches), True, "L=%d" % L)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [8, 16, 32, 64, 128, 256])
def test_ngcf_step_matches_reference_over_widths(d):
    """L = 3, two full batches and a partial one, eager launches"""
    eng, eu, ei = _ngcf_engine(3, d, 128, 2 * 128 + 37, seed=d)
    _set_triples(eng, eu, ei)
    ngcf_teacher_forced(eng, range(eng.n_batches), False, "d=%d" % d)


@pytest.mark.gpu
@pytest.mark.parametrize("use_graph", [False, True])
def test_ngcf_step_matches_reference_single_partial_batch(use_graph):
    """one batch of B - 19 triples (every edge case of _triples) stepped four times"""
    eng, eu, ei = _ngcf_engine(2, 64, 128, 128 - 19, seed=5)
    _set_triples(eng, eu, ei)
    assert eng.n_batches == 1
    ngcf_teacher_forced(eng, [0, 0, 0, 0], use_graph, "nb=1")


@pytest.mark.gpu
def test_ngcf_step_matches_reference_with_the_device_sampler():
    from arlib_b200.engine import DeviceTrainSet
    eng, eu, ei = _ngcf_engine(3, 64, 128, 12000, seed=7)
    eng.sample_epoch(DeviceTrainSet.from_arrays(eu, ei, eng.U, eng.N - eng.U, DEV), seed=11, epoch=0)
    assert eng.T % eng.B
    ngcf_teacher_forced(eng, [0, 1, eng.n_batches - 1], True, "sampler")


BENCH_SHAPES = [("gowalla", 64), ("gowalla", 128), ("gowalla", 256), ("amazon-book", 128)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,d", BENCH_SHAPES)
def test_benchmark_shape_ngcf_steps_match_reference(name, d):
    """the shapes of tools/ngcf_bench.py (L = 3, B = 2048): steps 0, 1, 2 and the epoch's last, partial, batch,
    replayed.  At d = 64 every CTA of the persistent dW loop runs 3 or 4 tiles, at d = 128 / 256 every split-K
    slice 15 to 31 chunks."""
    from arlib_b200.engine import DeviceTrainSet, NGCFEngine
    D, g = _bench_graph(name)
    U, I, E, B, L = D["U"], D["I"], D["E"], D["B"], D["L"]
    table, W = _init_params(U + I, d, L, 2018)
    eng = NGCFEngine(g, table, W, U, LR, REG, B, E)
    eng.sample_epoch(DeviceTrainSet.from_arrays(D["tu"], D["ti"], U, I, DEV), 7, 0)
    assert eng.T % B and dw_chain(eng.N, d, N_PARTIALS[d]) >= 3 * 64 + N_PARTIALS[d]
    ngcf_teacher_forced(eng, [0, 1, 2, eng.n_batches - 1], True, "%s d=%d" % (name, d))


# ------------------------------------------------------------------------------------------------ GPU: row layout
class _RowRanks:
    """P row-partitioned NGCFEngines on one GPU, ranks as threads (tests/test_gpu_ngcf_rows_one_device.py)"""

    def __init__(self, world, g, table, W, U, B, T, triples):
        self.world = world
        self.ranks = _Ranks(world)
        self.streams = [torch.cuda.Stream(device=DEV) for _ in range(world)]
        self.engs = [None] * world
        torch.cuda.synchronize()

        def build(r):
            from arlib_b200.engine import NGCFEngine
            eng = NGCFEngine(g, table.clone(), W.clone(), U, LR, REG, B, T, comm=_ThreadComm(self.ranks, r))
            assert eng.mode == "rows"
            eng.set_triples(*triples)
            self.engs[r] = eng

        self.each(build)

    def each(self, fn):
        errors = []
        torch.cuda.synchronize()                      # what the caller queued (state copies) precedes the ranks' work

        def main(r):
            try:
                with torch.cuda.stream(self.streams[r]):
                    fn(r)
                    torch.cuda.current_stream().synchronize()
            except BaseException as e:          # noqa: BLE001 -- reported by the main thread
                errors.append(e)
                self.ranks.sync.abort()

        threads = [threading.Thread(target=main, args=(r,)) for r in range(self.world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        torch.cuda.synchronize()
        if errors:
            raise errors[0]

    def own(self, pick):
        """the table whose rows [r0, r1) come from rank r's pick(eng)"""
        out = torch.empty_like(pick(self.engs[0]))
        for e in self.engs:
            out[e.r0:e.r1] = pick(e)[e.r0:e.r1]
        return out

    def same(self, pick, what):
        x = pick(self.engs[0])
        for e in self.engs[1:]:
            assert np.array_equal(_bits(pick(e)), _bits(x)), "%s differs across ranks" % what
        return x

    def state(self):
        st = {k: self.same(lambda e: getattr(e, k), k) for k in ("E0", "W", "Wm", "Wv")}
        st.update(m=self.own(lambda e: e.m), v=self.own(lambda e: e.v))
        return {k: x.clone() for k, x in st.items()}

    def got(self, b):
        """dP_1 in dPs[1], dP_2 in dPs[0] (by layer parity, every row); dOut, dEdir, dE0, P_k, E_L, m, v: own rows"""
        e0, L = self.engs[0], self.engs[0].L
        dE = {0: self.own(lambda e: e.dE0)}
        if L >= 2:
            dE[1] = self.own(lambda e: e.dOut[0])
        if L >= 3:
            dE[2] = self.own(lambda e: e.dOut[1])
        dP = {1: self.same(lambda e: e.dPs[1], "dP_1")}
        if L >= 2:
            dP[2] = self.same(lambda e: e.dPs[0], "dP_2")
        return dict(out4=self.same(lambda e: e.out4[b], "loss row"), F=self.same(lambda e: e.F, "F"),
                    P=[self.own(lambda e: e.P[k]) for k in range(L)], E=[self.own(lambda e: e.Ek[k]) for k in range(L)],
                    dE=dE, dP=dP, dEdir1=self.own(lambda e: e.dEdir), dW=self.same(lambda e: e.dW, "dW"),
                    W=self.same(lambda e: e.W, "W"), Wm=self.same(lambda e: e.Wm, "Wm"), Wv=self.same(lambda e: e.Wv, "Wv"),
                    E0=self.same(lambda e: e.E0, "E0"), m=self.own(lambda e: e.m), v=self.own(lambda e: e.v))


@pytest.mark.gpu
@pytest.mark.parametrize("world,d,L", [(2, 64, 2), (2, 128, 2), (3, 64, 3)])
def test_row_partitioned_ngcf_steps_match_reference(world, d, L):
    """the row-partitioned layout emulated on one GPU against the float64 reference directly, step by step: every
    output including the unfused dE0; E0, F, W, dW, dP and the loss row hold the same bits on every rank"""
    g, eu, ei = _graph(1500, 2000, 30000, 31 + d)
    U, I, B = 1500, 2000, 512
    T = 3 * B + 41
    table, W = _init_params(U + I, d, L, 31 + d)
    triples = _triples(eu, ei, U, I, B, T, 3)
    rr = _RowRanks(world, g, table, W, U, B, T, triples)
    e0 = rr.engs[0]
    csr = RefCSR(e0.g.rowptr, e0.g.col, e0.g.val, U)
    A = _adj64(csr)
    run = max(run_length(e.g) for e in rr.engs)
    chain = max(dw_chain(e.r1 - e.r0, d, e.dW_partial.shape[0]) for e in rr.engs) + world
    group = "rows P=%d d=%d L=%d" % (world, d, L)
    for b in range(e0.n_batches):
        st0 = rr.state()
        t = int(e0.step_dev) + 1
        rr.each(lambda r: rr.engs[r].run_steps(b, 1, use_graph=False))
        for e in rr.engs:
            assert int(e.step_dev) == t and not _bits(e.G).any(), "step counter or G after step %d" % b
        u, i, j = _batch(e0, b)
        got = rr.got(b)
        r = check_against_reference(csr, A, st0, t, u, i, j, got, run, chain, group)
        _record(group, r)
        assert max(r.values()) <= 1.0, (group, b, r)


# ------------------------------------------------------------------------------------------------ GPU: the bounds
@pytest.mark.gpu
def test_bounds_reject_perturbed_references():
    """on real kernel output at a shape where the persistent dW loop wraps (N = 25 000 > 296 x 64), the comparison
    catches: (a) one edge of the hub row dropped from A, (b) slope 0.02 in the backward, (c) F divided by L, (d) dW
    without one tile of batch rows from a CTA's second tile, (e) W's Adam at t + 1, (f) one layer's W1 and W2 swapped in
    the backward only"""
    L, d, B = 3, 64, 256
    U, I = 10000, 15000
    eng, eu, ei = _ngcf_engine(L, d, B, 3 * B, seed=41, U=U, I=I, n_edges=150000)
    assert eng.N > N_PARTIALS[d] * 64
    _set_triples(eng, eu, ei)
    csr, A, run, chain = ngcf_teacher_forced(eng, [0], True, "perturbations")
    b = 1
    st0 = _state(eng)
    t = int(eng.step_dev) + 1
    eng.run_steps(b, 1, use_graph=True)
    torch.cuda.synchronize()
    got = _got(eng, b)
    u, i, j = _batch(eng, b)
    assert int(u[0]) == 0                                    # the hub user is in the batch

    def check(csr_=csr, A_=A, **perturb):
        return check_against_reference(csr_, A_, st0, t, u, i, j, got, run, chain, None, **perturb)

    r = check()
    _record("perturbations", r)
    assert max(r.values()) <= 1.0, r
    rp, col, val = csr.rowptr.clone(), csr.col, csr.val
    k = int(rp[0]) + 5                                      # one entry of row 0 (the hub user, > 700 entries)
    assert int(rp[1]) - int(rp[0]) > 700
    rp[1:] -= 1
    dropped = RefCSR(rp, torch.cat([col[:k], col[k + 1:]]), torch.cat([val[:k], val[k + 1:]]), csr.n_users)
    # a 64-row tile past the first 296 (a CTA's second tile) that holds batch nodes
    nodes = torch.unique(torch.cat([u, U + i, U + j]))
    tile = int(nodes[nodes >= N_PARTIALS[d] * 64][0]) // 64
    drop = torch.arange(tile * 64, min(tile * 64 + 64, eng.N), device=DEV)
    cases = {"(a) hub edge dropped": dict(csr_=dropped, A_=_adj64(dropped)), "(b) slope 0.02 in the backward":
             dict(slope_bwd=0.02), "(c) F divided by L": dict(f_div=L), "(d) dW without a second-round tile":
             dict(drop_rows=drop), "(e) W's Adam at t + 1": dict(w_step=t + 1), "(f) W1, W2 of layer 2 swapped":
             dict(swap_bwd=2)}
    caught = {}
    for name, kw in cases.items():
        r = check(**kw)
        caught[name] = sorted(k for k, x in r.items() if x > 1.0)
        assert caught[name], (name, r)
    print("\nperturbations rejected by: %s" % caught)
