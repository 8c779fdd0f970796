"""Tensor-level wrappers over the C-ABI (one python function per agcf_* entry point).

All tensors must live on one CUDA device, be contiguous, fp32 / int32.  Launches go
to torch's CURRENT stream, so they compose with torch ops and are capturable in
``torch.cuda.graph``.  No function here has a CPU implementation.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib
from .graph import DeviceGraph


def _f32(t, name):
    if t is None:
        return None
    if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
        raise TypeError("%s must be a contiguous fp32 CUDA tensor (got %s %s %s)" % (name, t.device, t.dtype, t.is_contiguous()))
    return t


def _i32(t, name):
    if t is None:
        return None
    if not (t.is_cuda and t.dtype == torch.int32 and t.is_contiguous()):
        raise TypeError("%s must be a contiguous int32 CUDA tensor" % name)
    return t


def _p(t):
    return None if t is None else t.data_ptr()


def spmm(g: DeviceGraph, X, Y=None, addend=None, acc_in=None, acc_out=None, acc_div=1.0, noise=None, eps=0.0,
         row_mask=None, col_mask=None, peer_Y=None, peer_acc=None, mc_Y=None, mc_acc=None,
         worklist=None, adam=None, zero_acc_in=False, persistent=None, philox=None, aux=None, acc_terms=None,
         addend_mask=None):
    """agcf_spmm_csr_f32_ex: t = A X (+addend) (+noise perturbation); Y = t;
    acc_out = (acc_in + t) / acc_div.

    worklist = (vrows [cap,4], vpart [cap], count [1], partial [cap,d], tickets [cap]): a per-batch plan
    (spmm_batch_worklists) instead of the graph's; adam = (p, m, v, coefs, beta1, beta2, eps): the optimizer
    fused into the epilogue; zero_acc_in: re-zero the non-zero rows of acc_in; persistent (default: the graph's
    setting): persistent CTAs with dynamic block scheduling instead of one CTA per block; philox = (seed, stream,
    step_dev or None): draw the perturbation noise in the epilogue instead of reading ``noise`` (stream None: no
    main perturbation, the seed / step only serve ``aux``); aux = up to two (Y_q, noise table or None, stream) extra
    outputs perturbed with their own noise; acc_terms = up to 8 tables that take the place of acc_in:
    acc_out = (((acc_terms[0] + acc_terms[1]) + ...) + t) / acc_div; addend_mask = a row bitmap outside which addend /
    acc_in are known to be zero (not loaded; with zero_acc_in the rows inside it are re-zeroed)."""
    lib = _lib.load()
    _f32(X, "X"); _f32(Y, "Y"); _f32(addend, "addend"); _f32(acc_in, "acc_in"); _f32(acc_out, "acc_out"); _f32(noise, "noise")
    if X.shape[0] != g.n_rows:
        raise ValueError("X has %d rows, graph has %d" % (X.shape[0], g.n_rows))
    if peer_Y and peer_acc and len(peer_Y) != len(peer_acc):
        raise ValueError("peer lists must have equal length")
    d = X.shape[1]
    for t in (Y, addend, acc_in, acc_out, noise):
        if t is not None and tuple(t.shape) != (g.n_rows, d):
            raise ValueError("operand shape mismatch")
    py, n1 = _lib.ptr_array(peer_Y)
    pa, n2 = _lib.ptr_array(peer_acc)
    a = _lib.SpmmArgs()
    if worklist is None:
        a.vrows, a.vpart, a.n_vrows = g.vrows.data_ptr(), g.vpart.data_ptr(), g.n_vrows
        a.partial, a.tickets = g.partial_scratch(d).data_ptr(), g.tickets.data_ptr()
    else:
        wv, wp, wc, wpart, wtick = worklist
        if wpart.shape[1] != d or wpart.shape[0] < wv.shape[0] or wtick.numel() < wv.shape[0]:
            raise ValueError("work-list scratch too small")
        a.vrows, a.vpart, a.n_vrows, a.n_vrows_dev = wv.data_ptr(), wp.data_ptr(), wv.shape[0], wc.data_ptr()
        a.partial, a.tickets = wpart.data_ptr(), wtick.data_ptr()
    a.col, a.val = g.col.data_ptr(), g.val.data_ptr()
    a.X, a.Y, a.addend = X.data_ptr(), _p(Y), _p(addend)
    a.acc_in, a.acc_out, a.acc_div = _p(acc_in), _p(acc_out), float(acc_div)
    a.noise, a.eps = _p(noise), float(eps)
    if philox is not None:
        if int(philox[0]) == 0 or (noise is not None and philox[1] is not None):
            raise ValueError("philox noise needs a non-zero seed and no noise table")
        a.noise_seed, a.noise_step = int(philox[0]) & (2 ** 64 - 1), _p(philox[2])
        if philox[1] is not None:
            a.noise_stream, a.noise_main = int(philox[1]), 1
    for q, (y_q, tab_q, stream_q) in enumerate(aux or ()):
        _f32(y_q, "aux Y"); _f32(tab_q, "aux noise")
        if tuple(y_q.shape) != (g.n_rows, d) or (tab_q is not None and tuple(tab_q.shape) != (g.n_rows, d)):
            raise ValueError("aux operand shape mismatch")
        a.aux_Y[q], a.aux_noise[q], a.aux_stream[q] = y_q.data_ptr(), _p(tab_q), int(stream_q or 0)
    a.row_mask, a.col_mask, a.addend_mask = _p(row_mask), _p(col_mask), _p(addend_mask)
    a.mask_bits = g.n_rows
    a.peer_Y_host = ctypes.cast(py, ctypes.c_void_p) if py is not None else None
    a.peer_acc_host = ctypes.cast(pa, ctypes.c_void_p) if pa is not None else None
    a.n_peers = max(n1, n2)
    a.mc_Y, a.mc_acc = mc_Y or None, mc_acc or None
    if adam is not None:
        p_, m_, v_, coefs, b1, b2, aeps = adam
        for t in (p_, m_, v_):
            _f32(t, "adam table")
            if tuple(t.shape) != (g.n_rows, d):
                raise ValueError("adam table shape mismatch")
        a.adam_p, a.adam_m, a.adam_v, a.adam_coefs = p_.data_ptr(), m_.data_ptr(), v_.data_ptr(), coefs.data_ptr()
        a.adam_beta1, a.adam_beta2, a.adam_eps = float(b1), float(b2), float(aeps)
    a.zero_acc_in = 1 if zero_acc_in else 0
    a.d = d
    if g.persistent if persistent is None else persistent:
        a.sched = g.sched.data_ptr()
    a.flags = 0
    if acc_terms:
        if len(acc_terms) > len(a.acc_terms):
            raise ValueError("at most %d acc_terms" % len(a.acc_terms))
        for q, t in enumerate(acc_terms):
            _f32(t, "acc_terms")
            if tuple(t.shape) != (g.n_rows, d):
                raise ValueError("operand shape mismatch")
            a.acc_terms[q] = t.data_ptr()
        a.n_acc_terms = len(acc_terms)
    _lib.check(lib.agcf_spmm_csr_f32_ex(ctypes.byref(a), _lib.stream_ptr()), "agcf_spmm_csr_f32_ex")


def spmm_batch_worklists(seg_node, n_seg, n_batches, seg_stride, rowptr, row0, row1, split_above, segment,
                         wl_vrows, wl_vpart, wl_count):
    """agcf_spmm_batch_worklists: wl_vrows [n_batches, cap, 4], wl_vpart [n_batches, cap], wl_count [n_batches]."""
    lib = _lib.load()
    for t, n in ((seg_node, "seg_node"), (n_seg, "n_seg"), (rowptr, "rowptr"), (wl_vrows, "wl_vrows"),
                 (wl_vpart, "wl_vpart"), (wl_count, "wl_count")):
        _i32(t, n)
    cap = wl_vrows.shape[-2]
    _lib.check(lib.agcf_spmm_batch_worklists(seg_node.data_ptr(), n_seg.data_ptr(), int(n_batches), int(seg_stride),
                                             rowptr.data_ptr(), int(row0), int(row1), int(split_above), int(segment),
                                             wl_vrows.data_ptr(), wl_vpart.data_ptr(), wl_count.data_ptr(), int(cap),
                                             _lib.stream_ptr()), "agcf_spmm_batch_worklists")


def adam_coefs(step_dev, coefs, lr, beta1=0.9, beta2=0.999, increment=False):
    """agcf_adam_coefs: (optionally) advance the device step counter and write {lr/(1-b1^t), sqrt(1-b2^t)}, t = step + 1."""
    _lib.check(_lib.load().agcf_adam_coefs(step_dev.data_ptr(), 1 if increment else 0, float(lr), float(beta1),
                                           float(beta2), coefs.data_ptr(), _lib.stream_ptr()), "agcf_adam_coefs")


def sddmm(g: DeviceGraph, H, E, gval, accumulate=False):
    """agcf_sddmm_csr_f32: gval[p] (+)= <H[i], E[col[p]]> over the stored pattern."""
    lib = _lib.load()
    _f32(H, "H"); _f32(E, "E"); _f32(gval, "gval")
    _lib.check(lib.agcf_sddmm_csr_f32(g.rowptr.data_ptr(), g.col.data_ptr(), H.data_ptr(), E.data_ptr(), gval.data_ptr(),
                                      1 if accumulate else 0, None, g.n_rows, H.shape[1],
                                      _lib.stream_ptr()), "agcf_sddmm_csr_f32")


def concat_rows(a, b, out=None):
    """agcf_concat_rows_f32: [a; b] into one table."""
    lib = _lib.load()
    _f32(a, "a"); _f32(b, "b")
    d = a.shape[1]
    if out is None:
        out = torch.empty((a.shape[0] + b.shape[0], d), dtype=torch.float32, device=a.device)
    _lib.check(lib.agcf_concat_rows_f32(a.data_ptr(), a.shape[0], b.data_ptr(), b.shape[0], out.data_ptr(), d,
                                        _lib.stream_ptr()), "agcf_concat_rows_f32")
    return out


def bpr_sample_epoch(e_user, e_item, rej_rowptr, rej_items, n_items, seed, epoch, out_u, out_i, out_j):
    lib = _lib.load()
    for t, n in ((e_user, "e_user"), (e_item, "e_item"), (rej_rowptr, "rej_rowptr"), (rej_items, "rej_items"),
                 (out_u, "out_u"), (out_i, "out_i"), (out_j, "out_j")):
        _i32(t, n)
    _lib.check(lib.agcf_bpr_sample_epoch(e_user.data_ptr(), e_item.data_ptr(), e_user.numel(), rej_rowptr.data_ptr(),
                                         rej_items.data_ptr(), int(n_items), int(seed) & (2 ** 64 - 1), int(epoch),
                                         out_u.data_ptr(), out_i.data_ptr(), out_j.data_ptr(), _lib.stream_ptr()),
               "agcf_bpr_sample_epoch")


def bpr_group_batches(u, i, j, n_triples, batch, n_users, occ, seg_off, seg_node, n_seg, n_nodes=0, node_mask=None):
    lib = _lib.load()
    _lib.check(lib.agcf_bpr_group_batches(u.data_ptr(), i.data_ptr(), j.data_ptr(), int(n_triples), int(batch),
                                          int(n_users), occ.data_ptr(), seg_off.data_ptr(), seg_node.data_ptr(),
                                          n_seg.data_ptr(), int(n_nodes), _p(node_mask), _lib.stream_ptr()),
               "agcf_bpr_group_batches")


def bpr_cl_ids(occ, seg_off, seg_node, n_seg, n_triples, batch, n_users, cl_users, cl_items, n_cl):
    """agcf_bpr_cl_ids: per batch, the sorted unique user rows and positive-item rows of the contrastive loss."""
    _lib.check(_lib.load().agcf_bpr_cl_ids(occ.data_ptr(), seg_off.data_ptr(), seg_node.data_ptr(), n_seg.data_ptr(),
                                           int(n_triples), int(batch), int(n_users), cl_users.data_ptr(),
                                           cl_items.data_ptr(), n_cl.data_ptr(), _lib.stream_ptr()), "agcf_bpr_cl_ids")


def bpr_ws_bytes(nb):
    return int(_lib.load().agcf_bpr_ws_bytes(int(nb)))


def bpr_forward(F, u, i, j, nb, n_users, reg, out4, coef, ws):
    lib = _lib.load()
    _lib.check(lib.agcf_bpr_forward(F.data_ptr(), u.data_ptr(), i.data_ptr(), j.data_ptr(), int(nb), int(n_users),
                                    F.shape[1], float(reg), out4.data_ptr(), coef.data_ptr(), ws.data_ptr(),
                                    _lib.stream_ptr()), "agcf_bpr_forward")


def bpr_xchg_bytes(cap):
    return int(_lib.load().agcf_bpr_xchg_bytes(int(cap)))


def bpr_partial(F, u, i, j, nb, n_users, rank, cap, step_dev, xchg_all):
    """agcf_bpr_partial: this rank's column-slice share of the scores, stored on every rank."""
    lib = _lib.load()
    arr, n = _lib.ptr_array(xchg_all)
    _lib.check(lib.agcf_bpr_partial(F.data_ptr(), u.data_ptr(), i.data_ptr(), j.data_ptr(), int(nb), int(n_users),
                                    F.shape[1], int(rank), int(cap), _p(step_dev), arr, n, _lib.stream_ptr()),
               "agcf_bpr_partial")


def bpr_finish(xchg, world, cap, nb, reg, step_dev, out4, coef, ws):
    lib = _lib.load()
    _lib.check(lib.agcf_bpr_finish(xchg.data_ptr(), int(world), int(cap), int(nb), float(reg), _p(step_dev),
                                   out4.data_ptr(), coef.data_ptr(), ws.data_ptr(), _lib.stream_ptr()), "agcf_bpr_finish")


def bpr_backward(F, u, i, j, nb, n_users, reg, scale, out4, coef, occ, seg_off, seg_node, n_seg, G):
    lib = _lib.load()
    _lib.check(lib.agcf_bpr_backward(F.data_ptr(), u.data_ptr(), i.data_ptr(), j.data_ptr(), int(nb), int(n_users),
                                     F.shape[1], float(reg), float(scale), out4.data_ptr(), coef.data_ptr(),
                                     occ.data_ptr(), seg_off.data_ptr(), seg_node.data_ptr(), n_seg.data_ptr(),
                                     G.data_ptr(), _lib.stream_ptr()), "agcf_bpr_backward")


def zero_rows(seg_node, n_seg, max_seg, G):
    lib = _lib.load()
    _lib.check(lib.agcf_zero_rows(seg_node.data_ptr(), n_seg.data_ptr(), int(max_seg), G.data_ptr(), G.shape[1],
                                  _lib.stream_ptr()), "agcf_zero_rows")


def infonce_ws(n, d, device):
    need = int(_lib.load().agcf_infonce_ws_bytes(int(n), int(d)))
    if need < 0:
        _lib.check(need, "agcf_infonce_ws_bytes")
    return torch.empty(need, dtype=torch.uint8, device=device)


def infonce_forward(view1, view2, temperature, rows=None, n=None, n_dev=None, loss=None, ws=None):
    """agcf_infonce_forward -> (loss [1] fp32, workspace); the workspace feeds infonce_backward.
    With ``rows`` the views are rows[r] of the TABLES view1 / view2; n = capacity, n_dev = device row count."""
    lib = _lib.load()
    _f32(view1, "view1"); _f32(view2, "view2"); _i32(rows, "rows"); _i32(n_dev, "n_dev")
    if view1.shape != view2.shape or view1.dim() != 2:
        raise ValueError("views must be two [n, d] tensors of equal shape")
    d = view1.shape[1]
    if n is None:
        n = rows.numel() if rows is not None else view1.shape[0]
    if ws is None:
        ws = infonce_ws(n, d, view1.device)
    if loss is None:
        loss = torch.empty(1, dtype=torch.float32, device=view1.device)
    _lib.check(lib.agcf_infonce_forward(view1.data_ptr(), view2.data_ptr(), _p(rows), int(n), _p(n_dev), d,
                                        float(temperature), loss.data_ptr(), ws.data_ptr(), ws.numel(),
                                        _lib.stream_ptr()), "agcf_infonce_forward")
    return loss, ws


def infonce_backward(n, d, temperature, ws, grad_loss=None, scale=1.0, n_dev=None, grad1=None, rows1=None, acc1=False,
                     grad2=None, rows2=None, acc2=False):
    """agcf_infonce_backward: scale * grad_loss * d loss / d view into grad1 / grad2 ([n, d], or tables with rowsK)."""
    lib = _lib.load()
    _f32(grad_loss, "grad_loss"); _f32(grad1, "grad1"); _f32(grad2, "grad2")
    _lib.check(lib.agcf_infonce_backward(int(n), _p(n_dev), int(d), float(temperature), _p(grad_loss), float(scale),
                                         ws.data_ptr(), ws.numel(), _p(grad1), _p(rows1), 1 if acc1 else 0,
                                         _p(grad2), _p(rows2), 1 if acc2 else 0, _lib.stream_ptr()),
               "agcf_infonce_backward")


def ngcf_dense_forward(P, E, W, Enext, acc_in=None, acc_out=None, acc_div=1.0, peer_Enext=None, peer_acc=None, mc_Enext=0,
                       mc_acc=0):
    """agcf_ngcf_dense_forward: Enext = leaky_relu([P + E | P * E] @ W, 0.01); acc_out = (acc_in + Enext) / acc_div.

    Row-partitioned (agcf_ngcf_dense_forward_peers): P, E, Enext, acc_* are a rank's rows of the tables; peer_Enext /
    peer_acc list the other ranks' copies of the same rows (device pointers), mc_Enext / mc_acc their multicast
    addresses (0: none)."""
    for t, n in ((P, "P"), (E, "E"), (W, "W"), (Enext, "Enext"), (acc_in, "acc_in"), (acc_out, "acc_out")):
        _f32(t, n)
    n, d = P.shape
    if tuple(W.shape) != (2 * d, d) or tuple(E.shape) != (n, d) or tuple(Enext.shape) != (n, d):
        raise ValueError("NGCF layer shapes: P, E, Enext [N, d]; W [2d, d]")
    lib = _lib.load()
    if not (peer_Enext or peer_acc or mc_Enext or mc_acc):
        _lib.check(lib.agcf_ngcf_dense_forward(P.data_ptr(), E.data_ptr(), W.data_ptr(), Enext.data_ptr(), _p(acc_in),
                                               _p(acc_out), float(acc_div), n, d, _lib.stream_ptr()),
                   "agcf_ngcf_dense_forward")
        return
    if peer_Enext and peer_acc and len(peer_Enext) != len(peer_acc):
        raise ValueError("peer lists must have equal length")
    pe, n1 = _lib.ptr_array(peer_Enext)
    pa, n2 = _lib.ptr_array(peer_acc)
    _lib.check(lib.agcf_ngcf_dense_forward_peers(P.data_ptr(), E.data_ptr(), W.data_ptr(), Enext.data_ptr(), _p(acc_in),
                                                 _p(acc_out), float(acc_div), n, d, pe, pa, max(n1, n2), mc_Enext or None,
                                                 mc_acc or None, _lib.stream_ptr()), "agcf_ngcf_dense_forward_peers")


def ngcf_dense_backward(dOut, Enext, P, E, WT, dP, dEdir, dW_partial, dW, peer_dP=None, mc_dP=0, peer_dW=None, mc_dW=0):
    """agcf_ngcf_dense_backward + agcf_ngcf_reduce_wgrad: dP, dEdir [N, d] and dW [2d, d] (dW_partial: [n_partials, 2d*d]).

    Row-partitioned (the _peers entry points): the row operands are a rank's rows; dP also goes to the other ranks'
    copies (peer_dP / mc_dP) and the reduced dW -- this rank's share -- to its slot in theirs (peer_dW / mc_dW)."""
    for t, n in ((dOut, "dOut"), (Enext, "Enext"), (P, "P"), (E, "E"), (WT, "WT"), (dP, "dP"), (dEdir, "dEdir"),
                 (dW_partial, "dW_partial"), (dW, "dW")):
        _f32(t, n)
    n, d = P.shape
    if tuple(WT.shape) != (d, 2 * d) or dW_partial.shape[1] != 2 * d * d or dW.numel() != 2 * d * d:
        raise ValueError("NGCF backward shapes: WT [d, 2d]; dW_partial [n_partials, 2d*d]; dW [2d, d]")
    lib = _lib.load()
    st = _lib.stream_ptr()
    if peer_dP or mc_dP:
        pp, npp = _lib.ptr_array(peer_dP)
        _lib.check(lib.agcf_ngcf_dense_backward_peers(dOut.data_ptr(), Enext.data_ptr(), P.data_ptr(), E.data_ptr(),
                                                      WT.data_ptr(), dP.data_ptr(), dEdir.data_ptr(), dW_partial.data_ptr(),
                                                      dW_partial.shape[0], n, d, pp, npp, mc_dP or None, st),
                   "agcf_ngcf_dense_backward_peers")
    else:
        _lib.check(lib.agcf_ngcf_dense_backward(dOut.data_ptr(), Enext.data_ptr(), P.data_ptr(), E.data_ptr(), WT.data_ptr(),
                                                dP.data_ptr(), dEdir.data_ptr(), dW_partial.data_ptr(), dW_partial.shape[0],
                                                n, d, st), "agcf_ngcf_dense_backward")
    if peer_dW or mc_dW:
        pw, npw = _lib.ptr_array(peer_dW)
        _lib.check(lib.agcf_ngcf_reduce_wgrad_peers(dW_partial.data_ptr(), dW_partial.shape[0], dW.data_ptr(), d, pw, npw,
                                                    mc_dW or None, st), "agcf_ngcf_reduce_wgrad_peers")
    else:
        _lib.check(lib.agcf_ngcf_reduce_wgrad(dW_partial.data_ptr(), dW_partial.shape[0], dW.data_ptr(), d, st),
                   "agcf_ngcf_reduce_wgrad")


def ngcf_reduce_wgrad(dW_partial, dW):
    """agcf_ngcf_reduce_wgrad: dW = sum of the rows of dW_partial [n, 2d*d] in row order (the row-partitioned step sums
    the ranks' slots with it, the same bits on every rank)."""
    _f32(dW_partial, "dW_partial"); _f32(dW, "dW")
    d = dW.shape[-1]
    if dW_partial.shape[-1] != 2 * d * d or dW.numel() != 2 * d * d:
        raise ValueError("NGCF weight-gradient shapes: dW_partial [n, 2d*d]; dW [2d, d]")
    _lib.check(_lib.load().agcf_ngcf_reduce_wgrad(dW_partial.data_ptr(), dW_partial.numel() // (2 * d * d), dW.data_ptr(),
                                                  d, _lib.stream_ptr()), "agcf_ngcf_reduce_wgrad")


def adam_step(p, g, m, v, lr, beta1=0.9, beta2=0.999, eps=1e-8, step=0, step_dev=None, peer_p=None, mc_p=None):
    lib = _lib.load()
    _f32(p, "p"); _f32(g, "g"); _f32(m, "m"); _f32(v, "v")
    pp, n = _lib.ptr_array(peer_p)
    _lib.check(lib.agcf_adam_step_f32(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), float(lr),
                                      float(beta1), float(beta2), float(eps), int(step), _p(step_dev), pp, n, mc_p or None,
                                      _lib.stream_ptr()), "agcf_adam_step_f32")


def increment(counter):
    _lib.check(_lib.load().agcf_increment_i32(counter.data_ptr(), _lib.stream_ptr()), "agcf_increment_i32")


def group_handoff(flags, peer_flags, my_slot, stamp_dev, err):
    """agcf_group_handoff: publish the next stamp into slot ``my_slot`` of every partner's flag words (``peer_flags``:
    device pointers) and wait until every partner's stamp is in ``flags``; *err becomes 1 if one never arrives."""
    _i32(flags, "flags"); _i32(stamp_dev, "stamp_dev"); _i32(err, "err")
    if flags.numel() < len(peer_flags) + 1:
        raise ValueError("flags needs one word per group member")
    arr, n = _lib.ptr_array(peer_flags)
    _lib.check(_lib.load().agcf_group_handoff(flags.data_ptr(), arr, n, int(my_slot), stamp_dev.data_ptr(), err.data_ptr(),
                                              _lib.stream_ptr()), "agcf_group_handoff")


def score_topk(user_emb, item_emb, K, user_rows=None, mask_rowptr=None, mask_items=None, item_offset=0, impl=0,
               n_u=None, ws=None, return_flags=False, out=None, keep_mask_bits=False):
    """agcf_score_topk over users ``user_rows`` (or the first n_u rows).  Returns
    (values [n_u,K] fp32, item ids [n_u,K] int32) sorted by (score desc, id asc); ``out`` = (values, ids) to write into
    (contiguous [n_u, K] blocks, e.g. row slices of the caller's result tensors: no copy afterwards).
    ``keep_mask_bits``: ``ws`` still holds the mask bits of the previous call on it with the same users / items / mask
    (AGCF_TOPK_KEEP_MASK_BITS, include/agcf.h): the memset + bit scatter of stage 0 are skipped."""
    lib = _lib.load()
    _f32(user_emb, "user_emb"); _f32(item_emb, "item_emb"); _i32(user_rows, "user_rows")
    _i32(mask_rowptr, "mask_rowptr"); _i32(mask_items, "mask_items")
    if n_u is None:
        n_u = user_rows.numel() if user_rows is not None else user_emb.shape[0]
    n_items, d = item_emb.shape
    need = int(lib.agcf_score_topk_ws_bytes(n_u, n_items, d, K))
    if need < 0:
        _lib.check(need, "agcf_score_topk_ws_bytes")
    if ws is None or ws.numel() < need:
        ws = torch.empty(need, dtype=torch.uint8, device=user_emb.device)
    if out is not None:
        out_val, out_idx = out
        _f32(out_val, "out values"); _i32(out_idx, "out ids")
        if tuple(out_val.shape) != (n_u, K) or tuple(out_idx.shape) != (n_u, K):
            raise ValueError("score_topk: out blocks must be [%d, %d]" % (n_u, K))
    else:
        out_val = torch.empty((n_u, K), dtype=torch.float32, device=user_emb.device)
        out_idx = torch.empty((n_u, K), dtype=torch.int32, device=user_emb.device)
    flags = torch.empty(n_u, dtype=torch.int32, device=user_emb.device) if return_flags else None
    _lib.check(lib.agcf_score_topk(user_emb.data_ptr(), _p(user_rows), n_u, item_emb.data_ptr(), n_items, d,
                                   _p(mask_rowptr), _p(mask_items), int(K), int(item_offset),
                                   int(impl) | (0x100 if keep_mask_bits else 0),
                                   out_val.data_ptr(), out_idx.data_ptr(), _p(flags), ws.data_ptr(), ws.numel(),
                                   _lib.stream_ptr()), "agcf_score_topk")
    if return_flags:
        return out_val, out_idx, flags
    return out_val, out_idx


def score_group_max(user_emb, item_emb, user_rows=None, mask_rowptr=None, mask_items=None, item_offset=0, impl=1, n_u=None,
                    ws=None, want_output=True):
    """agcf_score_group_max: stages 0 + 1 of the top-K alone -> [n_u, ceil(I / 32)] masked group maxima (or None)."""
    lib = _lib.load()
    _f32(user_emb, "user_emb"); _f32(item_emb, "item_emb"); _i32(user_rows, "user_rows")
    if n_u is None:
        n_u = user_rows.numel() if user_rows is not None else user_emb.shape[0]
    n_items, d = item_emb.shape
    need = int(lib.agcf_score_topk_ws_bytes(n_u, n_items, d, 1))
    if need < 0:
        _lib.check(need, "agcf_score_topk_ws_bytes")
    if ws is None or ws.numel() < need:
        ws = torch.empty(need, dtype=torch.uint8, device=user_emb.device)
    out = torch.empty((n_u, (n_items + 31) // 32), dtype=torch.float32, device=user_emb.device) if want_output else None
    _lib.check(lib.agcf_score_group_max(user_emb.data_ptr(), _p(user_rows), n_u, item_emb.data_ptr(), n_items, d,
                                        _p(mask_rowptr), _p(mask_items), int(item_offset), int(impl), _p(out), ws.data_ptr(),
                                        ws.numel(), _lib.stream_ptr()), "agcf_score_group_max")
    return out


def topk_merge(vals, idx):
    """agcf_topk_merge: vals/idx [P, n_u, K] -> [n_u, K]."""
    lib = _lib.load()
    P, n_u, K = vals.shape
    out_val = torch.empty((n_u, K), dtype=torch.float32, device=vals.device)
    out_idx = torch.empty((n_u, K), dtype=torch.int32, device=vals.device)
    _lib.check(lib.agcf_topk_merge(vals.data_ptr(), idx.data_ptr(), P, n_u, K, out_val.data_ptr(), out_idx.data_ptr(),
                                   _lib.stream_ptr()), "agcf_topk_merge")
    return out_val, out_idx


def score_rows(user_emb, user_rows, item_emb):
    """agcf_score_rows: un-masked scores of a few users against all items."""
    lib = _lib.load()
    n_u = user_rows.numel()
    out = torch.empty((n_u, item_emb.shape[0]), dtype=torch.float32, device=item_emb.device)
    _lib.check(lib.agcf_score_rows(user_emb.data_ptr(), user_rows.data_ptr(), n_u, item_emb.data_ptr(),
                                   item_emb.shape[0], item_emb.shape[1], out.data_ptr(), _lib.stream_ptr()),
               "agcf_score_rows")
    return out


def rank_metrics(topk_idx, t_rowptr, t_items, test_total, cutoffs, inv_log):
    """agcf_rank_metrics -> [n_u, nc, 3] float64 (hits, dcg, idcg)."""
    lib = _lib.load()
    n_u, K = topk_idx.shape
    nc = cutoffs.numel()
    out = torch.empty((n_u, nc, 3), dtype=torch.float64, device=topk_idx.device)
    _lib.check(lib.agcf_rank_metrics(topk_idx.data_ptr(), K, t_rowptr.data_ptr(), t_items.data_ptr(),
                                     test_total.data_ptr(), n_u, cutoffs.data_ptr(), nc, inv_log.data_ptr(),
                                     out.data_ptr(), _lib.stream_ptr()), "agcf_rank_metrics")
    return out
