"""The row-partitioned entry points of the NGCF dense layer (agcf_ngcf_dense_forward_peers, _backward_peers,
agcf_ngcf_reduce_wgrad_peers) on one GPU: the "peer" copies are other buffers on the same device, prefilled with a
sentinel.  On a row range that does not start at row 0 and has an odd row count, the local outputs are bit-equal to the
plain entry points', every peer copy holds exactly the range's rows, and the sentinel is intact everywhere else."""
import pytest
import torch

from arlib_b200 import ops
from arlib_b200.engine import NGCFEngine

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N, R0, R1 = 700, 37, 37 + 333
SENTINEL = -12345.5


def _tables(n_tables, d):
    return [torch.full((N, d), SENTINEL, device=DEV) for _ in range(n_tables)]


def _rows_only(copy, want, what):
    assert torch.equal(copy[R0:R1], want[R0:R1]), what + ": rows differ"
    assert bool((copy[:R0] == SENTINEL).all()) and bool((copy[R1:] == SENTINEL).all()), what + ": sentinel overwritten"


def _ptrs(tables):
    return [t[R0].data_ptr() for t in tables]


@pytest.mark.parametrize("d", [8, 16, 32, 64, 128, 256])
def test_peer_stores_match_plain_entry_points(d):
    gen = torch.Generator().manual_seed(d)
    P, E, acc_in, dOut = (torch.randn(N, d, generator=gen).mul_(0.3).to(DEV) for _ in range(4))
    W = (torch.randn(2 * d, d, generator=gen) / d ** 0.5).to(DEV)
    WT = W.t().contiguous()
    rows = lambda t: t[R0:R1]

    # forward: plain entry point on the rows, then the peer variant storing Enext (and, separately, the mean) to peers
    Y0, M0 = _tables(2, d)
    ops.ngcf_dense_forward(rows(P), rows(E), W, rows(Y0), acc_in=rows(acc_in), acc_out=rows(M0), acc_div=3.0)
    Y1, M1 = _tables(2, d)
    pY, pM = _tables(2, d), _tables(2, d)
    ops.ngcf_dense_forward(rows(P), rows(E), W, rows(Y1), acc_in=rows(acc_in), acc_out=rows(M1), acc_div=3.0,
                           peer_Enext=_ptrs(pY), peer_acc=_ptrs(pM))
    _rows_only(Y1, Y0, "local Enext")
    _rows_only(M1, M0, "local mean")
    for q in range(2):
        _rows_only(pY[q], Y0, "peer Enext %d" % q)
        _rows_only(pM[q], M0, "peer mean %d" % q)
    # only the mean goes to the peers (the last layer of the engine)
    Y2, M2 = _tables(2, d)
    qY, qM = _tables(1, d), _tables(1, d)
    ops.ngcf_dense_forward(rows(P), rows(E), W, rows(Y2), acc_in=rows(acc_in), acc_out=rows(M2), acc_div=3.0,
                           peer_acc=_ptrs(qM))
    _rows_only(qM[0], M0, "peer mean only")
    assert bool((qY[0] == SENTINEL).all())

    # backward: dP to the peers, and this rank's reduced dW into its slot of every peer's slot buffer
    n_part = NGCFEngine.N_PARTIALS[d]
    dP0, dE0 = _tables(2, d)
    part = torch.empty((n_part, 2 * d * d), device=DEV)
    dW0 = torch.empty((2 * d, d), device=DEV)
    ops.ngcf_dense_backward(rows(dOut), rows(Y0), rows(P), rows(E), WT, rows(dP0), rows(dE0), part, dW0)
    dP1, dE1 = _tables(2, d)
    pdP = _tables(3, d)
    slots = [torch.full((4, 2 * d * d), SENTINEL, device=DEV) for _ in range(4)]      # 4 ranks' slot buffers; rank 1
    ops.ngcf_dense_backward(rows(dOut), rows(Y0), rows(P), rows(E), WT, rows(dP1), rows(dE1), part, slots[1][1],
                            peer_dP=_ptrs(pdP), peer_dW=[slots[q][1].data_ptr() for q in (0, 2, 3)])
    _rows_only(dP1, dP0, "local dP")
    _rows_only(dE1, dE0, "local dE_direct")
    for q in range(3):
        _rows_only(pdP[q], dP0, "peer dP %d" % q)
    for q in range(4):
        assert torch.equal(slots[q][1], dW0.view(-1)), "slot of rank 1 on rank %d" % q
        assert bool((slots[q][[0, 2, 3]] == SENTINEL).all()), "other slots on rank %d overwritten" % q

    # the rank-order sum of the slots is one more call of the plain reduce
    full = torch.stack([dW0.view(-1) * (k + 1) for k in range(4)])
    dW = torch.empty((2 * d, d), device=DEV)
    ops.ngcf_reduce_wgrad(full, dW)
    want = ((full[0] + full[1]) + full[2]) + full[3]
    assert torch.equal(dW.view(-1), want)
