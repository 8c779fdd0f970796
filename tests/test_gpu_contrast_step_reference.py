"""A float64 reference of one SimGCL / XSimGCL training step under the engine's own Philox noise, and teacher-forced
checks of arlib_b200.engine.ContrastiveEngine against it.

The perturbation noise is drawn in the SpMM epilogue by Philox4x32-10 (key = seed, counter = (float4 slot,
step << 32 | stream)); engine_noise restates that draw on the host bit for bit, so the reference sees the very noise
the kernels drew, at the step the device counter held.  ref_cl_step runs the step in float64 (the oracle's forward,
losses and InfoNCE, autograd, the Adam of include/agcf.h); cl_step_bounds derives an elementwise bound of every fp32
output from the arithmetic the kernels do (no tuned tolerance), nce_bounds does so for the InfoNCE kernels alone.  The
elements whose sign() the fp32 kernel may legitimately decide differently (|E_k| within its forward bound) are counted
and their perturbation treated as unknown.  The bounds are shown to reject six small reference-side perturbations.

Helpers shared with the LightGCN step (Adam scalars, bounds of the BPR loss, run lengths, the graph and batch makers,
the comparison of the Adam outputs) come from test_gpu_step_reference.py."""
import collections
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as Fn

from oracle import port
from test_gpu_step_reference import (BETAS, DEV, EPS, LR, REG, UNIT, RefCSR, _adj64, _bench_graph, _bits, _edges,
                                     _ratio, _small_engine, _triples, _ulp32, adam_scalars, check_step,
                                     loss_grad_bounds, run_length)

NOISE_EPS = 0.1
SEED = 0x9e3779b97f4a7c15            # both key words non-zero


def f32(x):
    return float(np.float32(x))


# ------------------------------------------------------------------------------------------------ host Philox
def philox4x32(key, ctr_lo, ctr_hi):
    """Philox::gen of csrc/common.cuh, vectorised over ctr_lo: counter words 0, 1 are ctr_lo (low half first), words
    2, 3 ctr_hi; key word 0 is the low half of the 64-bit key.  10 rounds, 64-bit products.  Returns uint32 [..., 4]."""
    m, s = np.uint64(0xFFFFFFFF), np.uint64(32)
    lo = np.asarray(ctr_lo, dtype=np.uint64)
    hi = np.broadcast_to(np.asarray(ctr_hi, dtype=np.uint64), lo.shape)
    c0, c1, c2, c3 = lo & m, lo >> s, hi & m, hi >> s
    k0, k1 = int(key) & 0xFFFFFFFF, (int(key) >> 32) & 0xFFFFFFFF
    M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = (p1 >> s) ^ c1 ^ np.uint64(k0), p1 & m, (p0 >> s) ^ c3 ^ np.uint64(k1), p0 & m
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return np.stack([c0, c1, c2, c3], -1).astype(np.uint32)


def engine_noise(seed, stream, step, N, d):
    """The U[0,1) table the SpMM epilogue draws: element 4 s + c (row-major) is word c of gen(seed, s, step << 32 |
    stream), as (w >> 8) 2^-24 (exact in fp32).  float64 [N, d]."""
    ctr_hi = ((int(step) & 0xFFFFFFFF) << 32) | int(stream)
    w = philox4x32(seed, np.arange(N * d // 4, dtype=np.uint64), ctr_hi)
    return (w >> 8).astype(np.float64).reshape(N, d) * 2.0 ** -24


def step_noises(kind, seed, step, N, d, L, device):
    """{(pass, layer): table} of one step: XSimGCL's pass 0 draws stream k at layer k, SimGCL's perturbed passes 1 and 2
    streams 64 + k and 128 + k (layer 1 of both: the aux outputs of the shared first launch)"""
    passes = (0,) if kind == "xsimgcl" else (1, 2)
    return {(p, k): torch.from_numpy(engine_noise(seed, 64 * p + k, step, N, d)).to(device)
            for p in passes for k in range(1, L + 1)}


# ------------------------------------------------------------------------------------------------ float64 reference
def _grad_scale(x, s):
    """x in the forward, s * (d / dx) in the backward"""
    return x if s == 1.0 else x * s + x.detach() * (1.0 - s)


def _infonce(a, b, temp, temp_bwd=None):
    x = port.infonce(a, b, temp)
    if temp_bwd is None:
        return x
    y = port.infonce(a, b, temp_bwd)
    return x.detach() + (y - y.detach())


def ref_cl_step(csr, E0, m, v, t, u, i, j, kind, L, layer_cl, noises, eps, cl_rate, tau, reg, lr, betas=BETAS,
                adam_eps=EPS, tau_bwd_factor=None, gcl_scale=1.0, drop_user=None):
    """One SimGCL / XSimGCL step in float64 from E0, m, v (Adam step t) on the graph's fp32 values, with the noise tables
    `noises` ({(pass, layer): U[0,1) table}).  eps, cl_rate, reg and tau are rounded to fp32 as the ABI takes them and
    InfoNCE divides by 1 / fl(1 / tau), the kernels' multiplier.  The last three arguments perturb the reference (the
    bounds must reject them): tau scaled in the backward only, the CL view's gradient scaled, one CL user dropped."""
    A = _adj64(csr)
    U, dev = csr.n_users, csr.rowptr.device
    eps, cl_rate, reg = f32(eps), f32(cl_rate), f32(reg)
    inv_t = f32(1.0 / np.float32(tau))
    temp = 1.0 / inv_t
    E = E0.detach().double().clone().requires_grad_(True)
    nz = lambda p: [noises[(p, k)] for k in range(1, L + 1)]
    if kind == "xsimgcl":
        ru, ri, cu, ci = port.xsimgcl_forward(A, E[:U], E[U:], L, eps, layer_cl, nz(0))
        v1, v2 = torch.cat([ru, ri]), _grad_scale(torch.cat([cu, ci]), gcl_scale)
    else:
        ru, ri = port.simgcl_forward(A, E[:U], E[U:], L, eps, None)
        v1 = torch.cat(port.simgcl_forward(A, E[:U], E[U:], L, eps, nz(1)))
        v2 = torch.cat(port.simgcl_forward(A, E[:U], E[U:], L, eps, nz(2)))
    F = torch.cat([ru, ri])
    uu = port.unique_ids_f32(u.cpu()).to(dev)
    ii = port.unique_ids_f32(i.cpu()).to(dev) + U
    if drop_user is not None:
        uu = uu[uu != drop_user]
    tb = None if tau_bwd_factor is None else temp * tau_bwd_factor
    cl2 = torch.stack([_infonce(v1[r], v2[r], temp, tb) for r in (uu, ii)])
    ue, pe, ne = F[u], F[U + i], F[U + j]
    bpr = port.bpr_loss(ue, pe, ne)
    rec = bpr + port.l2_reg_loss(reg, ue, pe)
    g, = torch.autograd.grad(rec + cl_rate * cl2.sum(), E)
    b1, b2, c1, c2, aeps = adam_scalars(t, lr, betas, adam_eps)
    m1 = b1 * m.double() + (1 - b1) * g
    v1_ = b2 * v.double() + (1 - b2) * g * g
    p1 = E0.double() - c1 * m1 / (v1_.sqrt() / c2 + aeps)
    with torch.no_grad():
        loss4 = torch.stack([rec, bpr, ue.norm(), pe.norm()])
    return dict(loss4=loss4, cl2=cl2.detach(), F=F.detach(), g=g, m=m1, v=v1_, p=p1, c1=c1, c2=c2, eps=aeps, b1=b1,
                b2=b2, A=A, uu=uu, ii=ii, kind=kind, L=L, layer_cl=layer_cl, noises=noises, noise_eps=eps,
                cl_rate=cl_rate, reg=reg, inv_t=inv_t, U=U)


# ------------------------------------------------------------------------------------------------ error bounds
def pass_bounds(A, E0, L, noises, eps, run):
    """float64 layers E_1 .. E_L of one propagation pass (perturbed with noises[k - 1] if given) and elementwise bounds
    e_k of the fp32 layers, magnitudes Xa_k >= |E_k|, F = mean_k E_k with its bound eF.

    t_k = A E_{k-1} sums at most `run` deep: within A e_{k-1} + (run + 1) UNIT A Xa_{k-1}.  The perturbation
    sign(t) fl(fl(n / ||n||) eps) carries the norm's d / 2 + 1 UNIT (d squares summed, a square root), the division and
    the product with eps; t + p one more rounding.  Where |t_k| is within t_k's bound the kernel may choose another
    sign, or 0: that element's perturbation is unknown, 2 eps n^ is added to its error (counted in `amb`)."""
    d = E0.shape[1]
    X = E0.double()
    Xa, e = X.abs(), torch.zeros_like(X)
    Es, es, Xas, amb = [], [], [], 0
    for k in range(L):
        t = torch.sparse.mm(A, X)
        ta = torch.sparse.mm(A, Xa)
        et = torch.sparse.mm(A, e) + (run + 1) * UNIT * ta
        if noises is None:
            X, Xa, e = t, ta, et
        else:
            p = eps * Fn.normalize(noises[k], dim=-1)
            ambiguous = (t.abs() <= et) & (et > 0)
            amb += int(ambiguous.sum())
            live = (t != 0) | ambiguous
            X = t + torch.sign(t) * p
            Xa = ta + p * live
            e = et + UNIT * Xa + (d / 2 + 3) * UNIT * p * live + 2 * p * ambiguous
        Es.append(X), es.append(e), Xas.append(Xa)
    # the running layer sum (L - 1 adds) and the division by L: L roundings of at most sum_k Xa_k
    Sa = sum(Xas)
    return dict(E=Es, e=es, Xa=Xas, amb=amb, n=L * X.numel(), F=sum(Es) / L, Fa=Sa / L,
                eF=(sum(es) + L * UNIT * Sa) / L)


def nce_split(n, d):
    """(split, tile) of csrc/contrast.cu for a grid sized for n rows"""
    tile = 64 if d <= 64 else 32
    nt = -(-n // tile)
    return max(1, min(-(-2 * 148 // nt), nt, 16)), tile


def nce_bounds(V1, V2, e1, e2, inv_t, scale1, scale2, cap):
    """InfoNCE of views V1, V2 ([n, d] float64) with 1 / tau = inv_t, when the fp32 views the kernels read are within
    e1, e2 of them (elementwise), on a grid sized for `cap` rows.  First order in UNIT and in the input errors.
    Returns the loss and the gradients scale_k * d loss / d V_k with their bounds (loss_b, g1_b, g2_b)."""
    n, d = V1.shape
    split, tile = nce_split(cap, d)
    n_tiles = -(-n // tile)
    per = -(-n_tiles // split)                              # tiles one slice walks
    depth_ttl = (tile // 16) * per + 4 + split              # a thread's terms, 16 lanes, the slices
    depth_pv = tile * per + split                           # P.V: a tile's rows per tile, the slices

    def normalize(V, e):
        # h = v / max(||v||, 1e-12): ||v||^2 summed d deep, the square root, the division: d / 2 + 2 UNIT of |h|; the
        # input error: |dv| / ||v|| + |h| ||dv|| / ||v||, over 1 - ||dv|| / ||v|| (the kernel's norm is the one divided by)
        nv = V.norm(dim=1, keepdim=True).clamp_min(1e-12)
        rel = e.norm(dim=1, keepdim=True) / nv
        h = V / nv
        assert float(rel.max()) < 0.5, "a view row's error bound is not small against its norm"
        eh = (e / nv + h.abs() * (rel + (d / 2 + 2) * UNIT)) / (1 - rel)
        return h, eh, nv, rel

    H1, eH1, n1, r1 = normalize(V1, e1)
    H2, eH2, n2, r2 = normalize(V2, e2)
    S = H1 @ H2.T
    # logit error ||dh1|| + ||dh2|| + d UNIT (unit vectors); exp(S / t): that over t, the product with 1 / t, expf's
    # 2 ulp -- as a relative error of X = exp(S / t)
    eS = eH1.norm(dim=1)[:, None] + eH2.norm(dim=1)[None, :] + d * UNIT
    rho = torch.expm1(eS * inv_t + UNIT * S.abs() * inv_t) + 4 * UNIT
    X = torch.exp(S * inv_t)
    ttl = X.sum(1)
    dT = (X * rho).sum(1) / ttl + depth_ttl * UNIT          # relative error of the row sum (positive terms)
    rowloss = torch.log(ttl) - S.diagonal() * inv_t
    # -logf(pos / ttl): the relative errors of pos and ttl, the division, logf's ulp
    e_row = rho.diagonal() + dT + UNIT + 2 * UNIT * rowloss.abs()
    loss = rowloss.mean()
    loss_b = e_row.mean() + UNIT * loss.abs()
    P = X / ttl[:, None]
    eP = P * (rho + dT[:, None] + UNIT)                     # P = fl(X / ttl)

    def side(Pm, ePm, Ho, eHo, Hr, eHr, nv, rel, scale):
        # acc = P Hr (depth_pv deep), q = acc - partner, Dh = coef q (coef = fl(fl(scale / t) / n)), then
        # through F.normalize: (Dh - h <h, Dh>) * fl(1 / ||v||)
        acc_a = Pm @ Hr.abs()
        e_acc = ePm @ Hr.abs() + Pm @ eHr + depth_pv * UNIT * acc_a
        q = Pm @ Hr - Hr
        qa = acc_a + Hr.abs()
        c = scale * inv_t / n
        Dh = c * q
        eDh = abs(c) * (e_acc + eHr + UNIT * qa + 4 * UNIT * qa)
        dot = (Ho * Dh).sum(1, keepdim=True)
        edot = (eHo * Dh.abs() + Ho.abs() * eDh).sum(1, keepdim=True) + d * UNIT * (Ho * Dh).abs().sum(1, keepdim=True)
        r = Dh - Ho * dot
        gv = r / nv
        inv_rel = rel / (1 - rel) + (d / 2 + 3) * UNIT
        e_gv = (eDh + eHo * dot.abs() + Ho.abs() * edot + 2 * UNIT * (Dh.abs() + (Ho * dot).abs())) / nv \
            + r.abs() / nv * inv_rel + UNIT * gv.abs()
        return gv, e_gv

    g1, g1_b = side(P, eP, H1, eH1, H2, eH2, n1, r1, scale1)
    g2, g2_b = side(P.T, eP.T, H2, eH2, H1, eH1, n2, r2, scale2)
    return dict(loss=loss, loss_b=loss_b, g1=g1, g1_b=g1_b, g2=g2, g2_b=g2_b)


def backprop_bounds(A, eG, aG, eGcl, aGcl, L, layer_cl, run):
    """bound of dE0 = A D_1 / L, D_L = G, D_{k-1} = A D_k + G (+ Gcl where k - 1 = layer_cl), when G / Gcl are within
    eG / eGcl of their float64 values (magnitudes aG, aGcl): each SpMM level adds (run + 1) UNIT of A |D|, each addend
    one rounding, the division by L one more"""
    eD, aD = eG, aG
    for k in range(L, 1, -1):
        tD = torch.sparse.mm(A, aD)
        eD = torch.sparse.mm(A, eD) + (run + 1) * UNIT * tD + eG + UNIT * (tD + aG)
        aD = tD + aG
        if k - 1 == layer_cl:
            eD = eD + eGcl + UNIT * (aD + aGcl)
            aD = aD + aGcl
    return (torch.sparse.mm(A, eD) + (run + 2) * UNIT * torch.sparse.mm(A, aD)) / L


def cl_step_bounds(ref, E0, u, i, j, run, cap):
    """Elementwise bounds of every fp32 output of the step against ref_cl_step's `ref`.  The rec view's bounds feed the
    BPR bounds (loss_grad_bounds), the views' bounds nce_bounds; the gradient rows of both (XSimGCL's CL view scaled
    by L into Gcl) go through the one backward propagation."""
    A, U, L, kind, lcl = ref["A"], ref["U"], ref["L"], ref["kind"], ref["layer_cl"]
    nz = lambda p: [ref["noises"][(p, k)] for k in range(1, L + 1)]
    eps = ref["noise_eps"]
    if kind == "xsimgcl":
        P0 = pass_bounds(A, E0, L, nz(0), eps, run)
        passes, rec = {"x": P0}, P0
        V1, V2 = (P0["F"], P0["eF"]), (P0["E"][lcl - 1], P0["e"][lcl - 1])
    else:
        rec = pass_bounds(A, E0, L, None, eps, run)
        Pa, Pb = pass_bounds(A, E0, L, nz(1), eps, run), pass_bounds(A, E0, L, nz(2), eps, run)
        passes = {"clean": rec, "a": Pa, "b": Pb}
        V1, V2 = (Pa["F"], Pa["eF"]), (Pb["F"], Pb["eF"])
    lg = loss_grad_bounds(rec["Fa"] + rec["eF"], 0, rec["F"], u, i, j, U, ref["reg"], eF=rec["eF"])
    eG, aG = lg["G"].clone(), lg["Gabs"].clone()
    eGcl, aGcl = torch.zeros_like(eG), torch.zeros_like(eG)
    s1 = ref["cl_rate"]
    s2 = f32(s1 * L) if kind == "xsimgcl" else s1
    cl_b = []
    for rows in (ref["uu"], ref["ii"]):
        nb = nce_bounds(V1[0][rows], V2[0][rows], V1[1][rows], V2[1][rows], ref["inv_t"], s1, s2, cap)
        cl_b.append(nb["loss_b"])
        eG[rows] += nb["g1_b"]
        aG[rows] += nb["g1"].abs() + nb["g1_b"]
        e2, a2 = (eGcl, aGcl) if kind == "xsimgcl" else (eG, aG)
        e2[rows] += nb["g2_b"]
        a2[rows] += nb["g2"].abs() + nb["g2_b"]
    eG += 2 * UNIT * aG                                       # the InfoNCE gradients accumulate into G's rows
    g = backprop_bounds(A, eG, aG, eGcl, aGcl, L, lcl if kind == "xsimgcl" else None, run)
    seed = torch.zeros(E0.shape[0], 1, dtype=torch.float64, device=E0.device)
    seed[torch.cat([u, U + i, U + j])] = 1.0
    far = seed[:, 0] == 0
    for _ in range(L):
        seed = torch.sparse.mm(A, seed)
        far &= seed[:, 0] == 0
    return dict(loss4=lg["loss4"], F=rec["eF"], g=g, far=far, cl=torch.stack(cl_b), passes=passes)


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
        extra = "; ambiguous signs %d of %d" % tuple(amb) if amb else ""
        print("\nlargest error / bound [%s]: %s%s" % (group, ", ".join("%s %.3g" % kv for kv in sorted(r.items())), extra))


def _r(got, want, bound, rows=None):
    if rows is not None:
        got, want, bound = got[rows], want[rows], bound[rows]
    return _ratio((got.double() - want).abs(), bound)


def check_cl_step(eng, b, ref, bnd, p0, m0, v0):
    """max(error / bound) per output of one engine step"""
    u, i, j = _batch(eng, b)
    rows = torch.unique(torch.cat([u, eng.U + i, eng.U + j]))
    got = dict(loss4=eng.out4[b], F=eng.F, m=eng.m, v=eng.v, p=eng.E0)
    r = check_step(got, ref, bnd, p0, m0, v0, rows)
    r["cl"] = _r(eng.cl_out[b], ref["cl2"], bnd["cl"])
    cl_rows = torch.cat([ref["uu"], ref["ii"]])
    ps = bnd["passes"]
    if eng.kind == "xsimgcl":
        k = eng.layer_cl - 1
        r["Ecl"] = _r(eng.Ecl, ps["x"]["E"][k], ps["x"]["e"][k])
    else:
        r["V"] = max(_r(eng.Va, ps["a"]["F"], ps["a"]["eF"], cl_rows), _r(eng.Vb, ps["b"]["F"], ps["b"]["eF"], cl_rows))
        if eng.L > 1:
            r["E1"] = max(_r(t, ps[name]["E"][0], ps[name]["e"][0])
                          for t, name in ((eng.E1, "clean"), (eng.E1a, "a"), (eng.E1b, "b")))
    return r


def _batch(eng, b):
    s0 = b * eng.B
    nb = min(eng.B, eng.T - s0)
    return tuple(x[s0:s0 + nb].long() for x in (eng.tu, eng.ti, eng.tj))


def ref_for_step(eng, csr, b, p0, m0, v0, s, **perturb):
    """ref_cl_step of batch b from the state (p0, m0, v0) with the noise of device step s"""
    u, i, j = _batch(eng, b)
    noise_step = perturb.pop("noise_step", s)
    noises = perturb.pop("noises", None) or step_noises(eng.kind, eng.noise_seed, noise_step, eng.N, eng.d, eng.L, DEV)
    layer_cl = perturb.pop("layer_cl", eng.layer_cl)
    return ref_cl_step(csr, p0, m0, v0, s + 1, u, i, j, eng.kind, eng.L, layer_cl, noises, eng.eps, eng.cl_rate,
                       eng.tau, eng.reg, eng.lr, eng.betas, eng.adam_eps, **perturb)


def _step_once(eng, b, use_graph):
    p0, m0, v0 = eng.E0.clone(), eng.m.clone(), eng.v.clone()
    s = int(eng.step_dev)
    eng.run_steps(b, 1, use_graph=use_graph)
    torch.cuda.synchronize()
    assert int(eng.step_dev) == s + 1
    assert not _bits(eng.G).any(), "G is not all +0.0 after step %d" % b
    if eng.kind == "xsimgcl":
        assert not _bits(eng.Gcl).any(), "Gcl is not all +0.0 after step %d" % b
    return p0, m0, v0, s


def cl_teacher_forced(eng, steps, use_graph, group):
    """For each step b: read E0 / m / v / step_dev, run the step, compare with ref_cl_step from what was read."""
    csr = RefCSR(eng.g.rowptr, eng.g.col, eng.g.val, eng.U)
    run = run_length(eng.g, [eng.wl_segment] if eng.wl is not None else [])
    for b in steps:
        p0, m0, v0, s = _step_once(eng, b, use_graph)
        ref = ref_for_step(eng, csr, b, p0, m0, v0, s)
        u, i, j = _batch(eng, b)
        bnd = cl_step_bounds(ref, p0, u, i, j, run, eng.B)
        for pb in bnd["passes"].values():
            AMBIGUOUS[group][0] += pb["amb"]
            AMBIGUOUS[group][1] += pb["n"]
            assert pb["amb"] <= 0.01 * pb["n"], (b, pb["amb"], pb["n"])
        r = check_cl_step(eng, b, ref, bnd, p0, m0, v0)
        _record(group, r)
        assert max(r.values()) <= 1.0, (group, b, s, r)
    return csr, run


def _cl_engine(kind, L, d, B, T, layer_cl=1, cl_rate=0.2, tau=None, seed=0):
    from arlib_b200.engine import ContrastiveEngine
    from arlib_b200.graph import DeviceGraph
    U, I = 800, 1000
    eu, ei = _edges(U, I, 12000, seed)
    g = DeviceGraph.from_dataloader_adj(port.bipartite_adjacency(eu, ei, U, I), DEV)
    gen = torch.Generator().manual_seed(seed + d)
    table = ((torch.rand(U + I, d, generator=gen) - 0.5) * 0.2).to(DEV)
    tau = tau or (0.1 if kind == "xsimgcl" else 0.2)
    eng = ContrastiveEngine(g, table, U, kind, L, NOISE_EPS, cl_rate, tau, LR, REG, B, T, layer_cl=layer_cl,
                            noise_seed=SEED)
    assert eng.noise_tables is None                         # the production path: Philox in the epilogue
    return eng, eu, ei


def _set_triples(eng, eu, ei, seed=1):
    eng.set_triples(*_triples(eu, ei, eng.U, eng.N - eng.U, eng.B, eng.cap, seed))


# ------------------------------------------------------------------------------------------------ CPU
def test_philox_reproduces_the_random123_known_answers():
    """philox4x32-10 known-answer vectors of Random123 (counter words, key words -> output words)"""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for c, k, want in kat:
        got = philox4x32(k[0] | k[1] << 32, [c[0] | c[1] << 32], c[2] | c[3] << 32)[0]
        assert [int(x) for x in got] == list(want), ["%08x" % x for x in got]


def test_engine_noise_layout():
    """element 4 s + c of the table is word c of slot s, the counter's high word the step, its low word the stream"""
    N, d = 7, 8
    tab = engine_noise(SEED, 129, 2 ** 31 + 3, N, d)
    for s in (0, 5, N * d // 4 - 1):
        w = philox4x32(SEED, [s], ((2 ** 31 + 3) << 32) | 129)[0]
        for c in range(4):
            r, col = divmod(4 * s + c, d)
            assert tab[r, col] == float(np.float32((int(w[c]) >> 8) * 2.0 ** -24))
    assert (tab >= 0).all() and (tab < 1).all()
    assert not np.array_equal(tab, engine_noise(SEED, 129, 3, N, d))


@pytest.mark.parametrize("kind,L,layer_cl", [("simgcl", 2, 1), ("xsimgcl", 3, 2)])
def test_ref_cl_step_matches_the_oracle_trainer_with_torch_adam(one_cpu_thread, kind, L, layer_cl):
    """ref_cl_step against port.SimGCLTrainer / XSimGCLTrainer in float64 under torch.optim.Adam, three steps, with the
    engine's noise of steps 0, 1, 2 injected into both"""
    U, I, d = 40, 60, 8
    rng = np.random.default_rng(0)
    key = np.unique(rng.integers(0, U, 300) * I + rng.integers(0, I, 300))
    adj = port.bipartite_adjacency(key // I, key % I, U, I)
    norm = port.normalize_graph_mat(adj).tocsr()
    norm.sort_indices()
    csr = RefCSR(torch.from_numpy(norm.indptr.astype(np.int64)), torch.from_numpy(norm.indices.astype(np.int64)),
                 torch.from_numpy(norm.data.astype(np.float32)), U)
    gen = torch.Generator().manual_seed(1)
    E = ((torch.rand(U + I, d, generator=gen) - 0.5) * 0.2).double()
    tau, cl_rate = (0.2 if kind == "simgcl" else 0.1), 0.2
    b1, b2, _, _, eps = adam_scalars(1, LR, BETAS, EPS)
    lr, temp = f32(LR), 1.0 / f32(1.0 / np.float32(tau))
    queue = []
    if kind == "simgcl":
        tr = port.SimGCLTrainer(norm, E[:U], E[U:], L, f32(NOISE_EPS), f32(cl_rate), lr, f32(REG), queue.pop,
                                tau=temp, dtype=torch.float64)
    else:
        tr = port.XSimGCLTrainer(norm, E[:U], E[U:], L, f32(NOISE_EPS), f32(cl_rate), layer_cl, lr, f32(REG),
                                 queue.pop, tau=temp, dtype=torch.float64)
    tr.opt = torch.optim.Adam([tr.user_emb, tr.item_emb], lr=lr, betas=(b1, b2), eps=eps)
    m, v = torch.zeros_like(E), torch.zeros_like(E)
    for t in (1, 2, 3):
        noises = step_noises(kind, SEED, t - 1, U + I, d, L, "cpu")
        passes = (0,) if kind == "xsimgcl" else (1, 2)
        queue[:] = [noises[(p, k)] for p in passes for k in range(1, L + 1)][::-1]     # pop() takes them in order
        u, i, j = (torch.from_numpy(rng.integers(0, n, 50)) for n in (U, I, I))
        i[:5] = i[5]                                          # repeated positives: fewer unique items than triples
        ref = ref_cl_step(csr, E, m, v, t, u, i, j, kind, L, layer_cl, noises, NOISE_EPS, cl_rate, tau, REG, LR)
        rec, cl = tr.step(u, i, j)
        assert not queue
        assert abs(rec - float(ref["loss4"][1])) <= 1e-12 * abs(rec)
        assert abs(cl - ref["cl_rate"] * float(ref["cl2"].sum())) <= 1e-12 * abs(cl)
        st = [tr.opt.state[p] for p in (tr.user_emb, tr.item_emb)]
        for name, want in (("p", torch.cat([tr.user_emb.detach(), tr.item_emb.detach()])),
                           ("m", torch.cat([s["exp_avg"] for s in st])), ("v", torch.cat([s["exp_avg_sq"] for s in st]))):
            scale = float(want.abs().max())
            torch.testing.assert_close(ref[name], want, rtol=1e-12, atol=1e-12 * scale, msg=lambda s: name + ": " + s)
        E, m, v = ref["p"], ref["m"], ref["v"]


# ------------------------------------------------------------------------------------------------ GPU: the noise
@pytest.mark.gpu
@pytest.mark.parametrize("d", [8, 16, 32, 64, 128, 256])
def test_philox_noise_is_the_host_table(d):
    """Philox output minus the same launch without noise equals sign(t) eps n / ||n|| of the host table within a few
    ulps: the main stream and both aux outputs, steps 0, 1 and >= 2^31, the full plan, a row bitmap, a batch work list
    and persistent CTAs; the hub rows (> split_above entries) run their epilogue after the partials are combined."""
    from arlib_b200 import ops
    eng, eu, ei = _small_engine(2, d, 128, 128, seed=d)
    _set_triples_lgcn(eng, eu, ei)
    g, X, N = eng.g, eng.E0, eng.N
    deg = g.rowptr[1:] - g.rowptr[:-1]
    hubs = torch.tensor([0, eng.U + 1], device=DEV)         # the hub user and item of _edges, named by every batch
    assert bool((deg[hubs] > g.split_above).all())
    mask = eng.node_mask[:eng.mask_words]
    bits = (mask.long()[:, None] >> torch.arange(32, device=DEV)) & 1
    live_rows = bits.flatten()[:N].bool()
    assert bool(live_rows[hubs].all())                      # so the masked plans compute them too
    eps32 = f32(NOISE_EPS)
    plans = {"full": ({}, None), "row_mask": ({"row_mask": mask}, live_rows), "persistent": ({"persistent": True}, None)}
    if eng.wl is not None:
        plans["worklist"] = ({"worklist": eng._worklist(0)}, live_rows)
    assert "worklist" in plans
    step = torch.zeros(1, dtype=torch.int32, device=DEV)
    worst = 0.0
    for s in (0, 1, 2 ** 31 + 5):
        step.fill_(s if s < 2 ** 31 else s - 2 ** 32)
        tabs = {q: torch.from_numpy(engine_noise(SEED, q, s, N, d)).to(DEV) for q in (7, 65, 129)}
        for name, (kw, rows) in plans.items():
            nan = lambda: torch.full_like(X, float("nan"))
            clean, main, y0, ya, yb = nan(), nan(), nan(), nan(), nan()
            ops.spmm(g, X, Y=clean, **kw)
            ops.spmm(g, X, Y=main, eps=NOISE_EPS, philox=(SEED, 7, step), **kw)
            ops.spmm(g, X, Y=y0, aux=[(ya, None, 65), (yb, None, 129)], eps=NOISE_EPS, philox=(SEED, None, step), **kw)
            torch.cuda.synchronize()
            sel = slice(None) if rows is None else rows
            c = clean[sel].double()
            assert torch.equal(y0[sel], clean[sel])             # no main perturbation when only aux streams are drawn
            for q, y in ((7, main), (65, ya), (129, yb)):
                p = eps32 * Fn.normalize(tabs[q][sel], dim=-1)
                want = torch.sign(c) * p
                # t + fl(fl(n / nrm) eps): nrm within d / 2 + 1 UNIT, the division and the product; the final add
                tol = 2 * _ulp32(y[sel]) + (d / 2 + 3) * UNIT * p
                r = _ratio((y[sel].double() - c - want).abs(), tol)
                worst = max(worst, r)
                assert r <= 1.0, (d, s, name, q, r)
    _record("philox d=%d" % d, {"noise": worst})


def _set_triples_lgcn(eng, eu, ei):
    eng.set_triples(*_triples(eu, ei, eng.U, eng.N - eng.U, eng.B, eng.cap, 1))


# ------------------------------------------------------------------------------------------------ GPU: InfoNCE alone
@pytest.mark.gpu
@pytest.mark.parametrize("d", [8, 16, 32, 64, 128, 256])
def test_infonce_kernels_match_float64(d):
    """agcf_infonce_forward / backward against float64 autograd through the oracle's InfoNCE, elementwise within
    nce_bounds: grids sized for 2048 / 1024 / 64 rows (split 1, 16 and uneven tiles per slice) read n_dev = 1 .. cap
    rows gathered from a table; the first gradient accumulates into a non-zero table, the second overwrites one, rows
    outside the gather keep their bits; zero rows hit the normalize clamp; tau = 0.05 .. 0.2."""
    from arlib_b200 import ops
    R = 2600
    gen = torch.Generator(device=DEV).manual_seed(d)
    T1 = torch.randn(R, d, device=DEV, generator=gen) * 0.3
    T2 = T1 + 0.3 * torch.randn(R, d, device=DEV, generator=gen)
    T1[[5, 9]] = 0.0
    T2[[5, 9]] = 0.0
    worst = collections.defaultdict(float)
    splits = set()
    for cap, ns, tau, scale in ((2048, [1, 2, 63, 64, 65, 2047, 2048], 0.05, 0.2), (1024, [1024, 700], 0.2, 5.0),
                                (64, [64, 33], 0.1, 1.0)):
        split, tile = nce_split(cap, d)
        splits.add(split)
        perm = torch.randperm(R, device=DEV, generator=gen)
        perm = perm[(perm != 5) & (perm != 9)]
        rows = torch.cat([torch.tensor([5], device=DEV), perm[:30], torch.tensor([9], device=DEV), perm[30:cap - 2]])
        rows = rows.to(torch.int32).contiguous()
        ws = ops.infonce_ws(cap, d, DEV)
        inv_t = f32(1.0 / np.float32(tau))
        for n in ns:
            n_dev = torch.tensor([n], dtype=torch.int32, device=DEV)
            loss, _ = ops.infonce_forward(T1, T2, tau, rows=rows, n=cap, n_dev=n_dev, ws=ws)
            G1 = torch.randn(R, d, device=DEV, generator=gen)
            G2 = torch.randn(R, d, device=DEV, generator=gen)
            G1_0, G2_0 = G1.clone(), G2.clone()
            ops.infonce_backward(cap, d, tau, ws, scale=scale, n_dev=n_dev, grad1=G1, rows1=rows, acc1=True,
                                 grad2=G2, rows2=rows, acc2=False)
            torch.cuda.synchronize()
            r = rows[:n].long()
            V1 = T1[r].double().requires_grad_(True)
            V2 = T2[r].double().requires_grad_(True)
            want = port.infonce(V1, V2, 1.0 / inv_t)
            g1, g2 = torch.autograd.grad(want, (V1, V2))
            sc = f32(scale)
            nb = nce_bounds(V1.detach(), V2.detach(), torch.zeros_like(V1), torch.zeros_like(V2), inv_t, sc, sc, cap)
            s1, s2 = sc * g1, sc * g2
            res = {"loss": _ratio((loss.double() - want.detach()).abs().reshape(1), nb["loss_b"].reshape(1)),
                   "g2": _ratio((G2[r].double() - s2).abs(), nb["g2_b"])}
            # accumulated: one more rounding of the sum
            acc_want = G1_0[r].double() + s1
            res["g1"] = _ratio((G1[r].double() - acc_want).abs(),
                               nb["g1_b"] + UNIT * (acc_want.abs() + nb["g1_b"]))
            for k, x in res.items():
                worst[k] = max(worst[k], x)
            assert max(res.values()) <= 1.0, (cap, n, res)
            out = torch.ones(R, dtype=torch.bool, device=DEV)
            out[r] = False
            assert np.array_equal(_bits(G1[out]), _bits(G1_0[out])) and np.array_equal(_bits(G2[out]), _bits(G2_0[out]))
    assert 1 in splits and 16 in splits or d > 64              # split 16 needs 64-row tiles at cap 1024
    _record("infonce d=%d" % d, dict(worst))


# ------------------------------------------------------------------------------------------------ GPU: the engine
@pytest.mark.gpu
@pytest.mark.parametrize("use_graph", [False, True])
@pytest.mark.parametrize("kind,L,layer_cl", [("simgcl", 1, 1), ("simgcl", 2, 1), ("simgcl", 3, 1), ("xsimgcl", 2, 1),
                                             ("xsimgcl", 3, 1), ("xsimgcl", 3, 2)])
def test_cl_step_matches_reference_over_layers(kind, L, layer_cl, use_graph):
    """d = 64, B = 128, a partial last batch (T = 4 B + 37)"""
    eng, eu, ei = _cl_engine(kind, L, 64, 128, 4 * 128 + 37, layer_cl=layer_cl, seed=L + layer_cl)
    _set_triples(eng, eu, ei)
    cl_teacher_forced(eng, range(eng.n_batches), use_graph, "%s L=%d layer_cl=%d" % (kind, L, layer_cl))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["simgcl", "xsimgcl"])
@pytest.mark.parametrize("d", [8, 16, 32, 128, 256])
def test_cl_step_matches_reference_over_widths(kind, d):
    eng, eu, ei = _cl_engine(kind, 2, d, 128, 2 * 128 + 37, seed=d)
    _set_triples(eng, eu, ei)
    cl_teacher_forced(eng, range(eng.n_batches), True, "%s d=%d" % (kind, d))


@pytest.mark.gpu
@pytest.mark.parametrize("kind,cl_rate,tau", [("xsimgcl", 0.0, 0.1), ("xsimgcl", 0.2, 0.05), ("xsimgcl", 5.0, 0.2),
                                              ("simgcl", 0.0, 0.2), ("simgcl", 0.2, 0.1), ("simgcl", 5.0, 0.05)])
def test_cl_step_matches_reference_over_cl_rate_and_tau(kind, cl_rate, tau):
    eng, eu, ei = _cl_engine(kind, 2, 64, 128, 2 * 128 + 37, cl_rate=cl_rate, tau=tau, seed=7)
    _set_triples(eng, eu, ei)
    cl_teacher_forced(eng, range(eng.n_batches), True, "%s cl_rate=%g tau=%g" % (kind, cl_rate, tau))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["simgcl", "xsimgcl"])
@pytest.mark.parametrize("segment", ["64", "256"])
@pytest.mark.parametrize("persistent", ["0", "1"])
@pytest.mark.parametrize("worklists", ["0", "1"])
def test_cl_step_matches_reference_flag_product(monkeypatch, worklists, persistent, segment, kind):
    """L = 3 (XSimGCL: layer_cl = 2), d = 64: per-batch work lists or the row bitmap in the last forward layers,
    persistent CTAs, 64- and 256-entry segments"""
    import arlib_b200.graph as graphmod
    monkeypatch.setenv("ARLIB_B200_WORKLISTS", worklists)
    monkeypatch.setattr(graphmod, "PERSISTENT_ENV", persistent)
    monkeypatch.setattr(graphmod, "SEGMENT_ENV", segment)
    eng, eu, ei = _cl_engine(kind, 3, 64, 128, 2 * 128 + 37, layer_cl=2, seed=3)
    assert eng.g.segment == int(segment) and eng.g.persistent == (persistent == "1")
    assert (eng.wl is not None) == (worklists == "1")
    _set_triples(eng, eu, ei)
    cl_teacher_forced(eng, range(eng.n_batches), True, "flags")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["simgcl", "xsimgcl"])
def test_cl_step_matches_reference_at_batch_edges(kind):
    """batch 0: one unique user; batch 1: B distinct users and B distinct positive items (n_cl = capacity); batch 2:
    the edgeless user and items among the CL rows (zero views: the normalize clamp); batch 3: a single triple of
    the edgeless user and an edgeless item (n_cl = [1, 1])"""
    B = 128
    eng, eu, ei = _cl_engine(kind, 2, 64, B, 3 * B + 1, seed=13)
    U, I = eng.U, eng.N - eng.U
    rng = np.random.default_rng(13)
    pick = rng.integers(0, eu.shape[0], 3 * B)
    tu, ti, tj = eu[pick].astype(np.int32), ei[pick].astype(np.int32), rng.integers(0, I, 3 * B + 1).astype(np.int32)
    tu[:B] = tu[0]
    tu[B:2 * B] = rng.permutation(U - 1)[:B]
    ti[B:2 * B] = rng.permutation(I - 5)[:B]
    tu[2 * B:2 * B + 4] = U - 1
    ti[2 * B + 4:2 * B + 8] = np.arange(I - 4, I)
    tu, ti = np.append(tu, U - 1).astype(np.int32), np.append(ti, I - 1).astype(np.int32)
    eng.set_triples(tu, ti, tj)
    torch.cuda.synchronize()
    assert eng.n_cl[0, 0] == 1 and eng.n_cl[1].tolist() == [B, B] and eng.n_cl[3].tolist() == [1, 1]
    cl_teacher_forced(eng, range(4), True, "%s batch edges" % kind)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["simgcl", "xsimgcl"])
def test_one_captured_step_draws_the_noise_of_the_current_step(kind):
    """batch 0 replayed three times from ONE capture: each replay must draw the noise of steps 0, 1, 2"""
    eng, eu, ei = _cl_engine(kind, 2, 64, 128, 128, seed=17)
    _set_triples(eng, eu, ei)
    cl_teacher_forced(eng, [0, 0, 0], True, "%s replay" % kind)
    assert len(eng._graphs) == 1


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["xsimgcl", "simgcl"])
def test_yelp2018_shape_steps_match_reference(kind):
    """the configuration of tools/contrast_bench.py: steps 0, 1, 2 and the epoch's last, partial, batch, replayed"""
    from bench import xavier_tables
    from arlib_b200.engine import ContrastiveEngine, DeviceTrainSet
    D, g = _bench_graph("yelp2018")
    U, I, E = D["U"], D["I"], D["E"]
    ue, ie = xavier_tables(U, I, 64)
    eng = ContrastiveEngine(g, torch.cat([ue, ie]).to(DEV), U, kind, 2, NOISE_EPS, 0.2, 0.1 if kind == "xsimgcl" else 0.2,
                            LR, REG, 2048, E, noise_seed=SEED)
    eng.sample_epoch(DeviceTrainSet.from_arrays(D["tu"], D["ti"], U, I, DEV), 7, 0)
    assert eng.T % eng.B
    cl_teacher_forced(eng, [0, 1, 2, eng.n_batches - 1], True, "yelp2018 %s" % kind)


# ------------------------------------------------------------------------------------------------ GPU: the bounds
@pytest.mark.gpu
def test_bounds_reject_perturbed_references():
    """on real kernel output the comparison catches: the noise of step t - 1, SimGCL's two perturbed passes swapped,
    layer_cl off by one, one unique CL user dropped, Gcl not scaled by L, tau x 1.05 in the backward only"""
    caught = {}
    for kind, L in (("xsimgcl", 3), ("simgcl", 2)):
        eng, eu, ei = _cl_engine(kind, L, 64, 128, 4 * 128 + 37, layer_cl=1, seed=21)
        _set_triples(eng, eu, ei)
        csr, run = cl_teacher_forced(eng, [0], True, "perturbations")
        b = 1
        p0, m0, v0, s = _step_once(eng, b, True)
        u, i, j = _batch(eng, b)

        def check(**perturb):
            ref = ref_for_step(eng, csr, b, p0, m0, v0, s, **perturb)
            bnd = cl_step_bounds(ref, p0, u, i, j, run, eng.B)
            return check_cl_step(eng, b, ref, bnd, p0, m0, v0)

        r = check()
        _record("perturbations", r)
        assert max(r.values()) <= 1.0, r
        cases = {"noise of step t-1": dict(noise_step=s - 1)}
        if kind == "simgcl":
            nz = step_noises(kind, eng.noise_seed, s, eng.N, eng.d, eng.L, DEV)
            cases["perturbed passes swapped"] = dict(noises={(3 - p, k): x for (p, k), x in nz.items()})
        else:
            uu = port.unique_ids_f32(u.cpu())
            assert uu.numel() > 1
            cases.update({"layer_cl off by one": dict(layer_cl=eng.layer_cl + 1),
                          "one CL user dropped": dict(drop_user=int(uu[uu.numel() // 2])),
                          "Gcl not scaled by L": dict(gcl_scale=1.0 / L),
                          "tau x 1.05 in the backward": dict(tau_bwd_factor=1.05)})
        for name, kw in cases.items():
            r = check(**kw)
            caught["%s: %s" % (kind, name)] = sorted(k for k, x in r.items() if x > 1.0)
            assert caught["%s: %s" % (kind, name)], (kind, name, r)
    print("\nperturbations rejected by: %s" % caught)
