"""Worker for tests/test_gpu_grid_one_device.py: the grid layout of LightGCNEngine and its column-group hand-off on ONE
GPU.  The R x C ranks run as threads, each on its own stream; a stand-in for DistContext gives every rank its own
allocation of each symmetric table (the hand-off flag words included) and the other ranks' allocations as peer
pointers, so the SpMM epilogues, Adam and bpr_partial store into the partners' copies and the hand-off kernels spin on
each other's flags exactly as over NVLink.

Ranks on one device can wait for each other in ways ranks on separate GPUs never do, and a rank's hand-off would then
spin behind the partner it waits for until it gives up.  So this runs in its own process with
CUDA_DEVICE_MAX_CONNECTIONS=32 (ranks whose streams share a hardware queue serialise) and CUDA_MODULE_LOADING=EAGER
(loading a kernel on its first launch synchronises the context), every rank finishes its allocations -- the engine's
and the SpMM's lazily allocated partial-sum scratch; an allocation also synchronises the device -- before any rank's
first hand-off, and graphs are captured in thread-local mode, one rank at a time."""
import argparse
import os
import sys
import threading

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import scipy.sparse as sp
import torch

DEV = torch.device("cuda:0")


class _Ranks:
    def __init__(self, world):
        self.world = world
        self.sync = threading.Barrier(world, timeout=300)
        self.slots = [None] * world


class _ThreadComm:
    """DistContext's interface for one rank of a _Ranks group"""

    def __init__(self, ranks, rank):
        self.ranks, self.rank, self.world = ranks, rank, ranks.world
        self.group = None

    def allocate(self, specs):
        bufs = {k: torch.zeros(shape, dtype=dt, device=DEV) for k, (shape, dt) in specs.items()}
        self.ranks.slots[self.rank] = bufs
        self.barrier()
        self.all_bufs = list(self.ranks.slots)
        self.barrier()
        return bufs

    def peers(self, name, extra_bytes=0, ranks=None):
        ranks = range(self.world) if ranks is None else ranks
        return [self.all_bufs[q][name].data_ptr() + int(extra_bytes) for q in ranks if q != self.rank]

    def all_ptrs(self, name, extra_bytes=0, ranks=None):
        ranks = range(self.world) if ranks is None else ranks
        return [self.all_bufs[q][name].data_ptr() + int(extra_bytes) for q in ranks]

    def multicast_ptr(self, name, extra_bytes=0):
        return 0

    def subgroups(self, groups):
        return None

    def barrier(self):
        torch.cuda.current_stream().synchronize()
        self.ranks.sync.wait()


def _threads(world, body):
    """body(rank, wait) on one thread per rank, each inside its own stream; the first exception is re-raised"""
    ranks = _Ranks(world)
    errors = []

    def main(r):
        stream = torch.cuda.Stream(device=DEV)

        def wait():
            stream.synchronize()
            ranks.sync.wait()

        try:
            with torch.cuda.stream(stream):
                body(r, wait, ranks)
        except BaseException as e:          # noqa: BLE001 -- reported by the main thread
            errors.append((r, e))
            ranks.sync.abort()

    threads = [threading.Thread(target=main, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    torch.cuda.synchronize()
    if errors:
        raise errors[0][1]


def check_engine(R, C, d, L, n_eager=2, n_graph=3):
    """R x C grid vs the single-GPU engine after n_eager eager steps and n_graph steps replayed from a CUDA graph"""
    from arlib_b200.engine import DeviceTrainSet, LightGCNEngine, dshard_columns
    from arlib_b200.graph import DeviceGraph
    from arlib_b200.util.synth import synth_edges

    U, I, E, B = 3000, 4000, 90000, 2048
    tu, ti, _, _ = synth_edges(U, I, E, seed=11)
    N = U + I
    half = sp.csr_matrix((np.ones(E, dtype=np.float32), (tu, ti + U)), shape=(N, N), dtype=np.float32)
    g = DeviceGraph.from_dataloader_adj(half + half.T, DEV)
    torch.manual_seed(0)
    table0 = (torch.rand(N, d) - 0.5) * 0.2
    ts = DeviceTrainSet.from_arrays(tu, ti, U, I, DEV)
    steps = n_eager + n_graph

    single = LightGCNEngine(g, table0.clone().to(DEV), U, L, 0.005, 1e-4, B, E)
    single.sample_epoch(ts, 7, 0)
    single.run_steps(0, steps, use_graph=False)
    Fs = single.forward_table().clone()
    torch.cuda.synchronize()
    world = R * C
    out = [None] * world

    def body(r, wait, ranks):
        eng = LightGCNEngine(g, table0.clone().to(DEV), U, L, 0.005, 1e-4, B, E, comm=_ThreadComm(ranks, r),
                             mode="grid", grid=(R, C))
        c0, c1 = dshard_columns(d, C, r % C)
        assert (eng.col0, eng.col1) == (c0, c1) and eng.d == d // C and eng.launches_per_step == 4 * L + 6
        eng.sample_epoch(ts, 7, 0)
        eng.g.partial_scratch(eng.d)
        wait()
        eng.run_steps(0, n_eager, use_graph=False)
        eng.check_handoff()
        wait()
        # capture one rank at a time, then replay all ranks at once through run_steps
        key = (n_eager, n_graph, eng.T)
        for turn in range(world):
            if turn == r:
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                    for b in range(n_eager, steps):
                        eng._launch_step(b)
                eng._graphs[key] = graph
            wait()
        eng.run_steps(n_eager, n_graph)
        eng.check_handoff()
        F = eng.forward_table()
        eng.check_handoff()
        out[r] = (c0, c1, eng.E0.clone(), F.clone(), eng.out4[:steps].clone(), int(eng.handoff_ctr.item()))
        wait()

    _threads(world, body)
    # the tolerance of the column-sharded layout (tests/dist_check.py): the row blocks' own SpMM plans and the sliced loss
    # sum in another order, and Adam turns the rounding residue of a gradient that nearly cancels into up to lr*|g|/eps
    for r, (c0, c1, E0, F, loss, stamps) in enumerate(out):
        e_err = float((E0 - single.E0[:, c0:c1]).abs().max())
        f_err = float((F - Fs[:, c0:c1]).abs().max())
        assert e_err < 2e-6, "grid %dx%d d=%d L=%d rank %d: E0 differs by %g" % (R, C, d, L, r, e_err)
        assert f_err < 2e-6, "grid %dx%d d=%d L=%d rank %d: forward table differs by %g" % (R, C, d, L, r, f_err)
        assert torch.equal(loss, out[0][4]), "rank %d: loss rows differ from rank 0" % r
        # hand-offs per step: L forward + (L - 1) backward + 1 closing the step, and L for the final forward
        assert stamps == steps * 2 * L + L, stamps
    lerr = float((out[0][4] - single.out4[:steps]).abs().max() / single.out4[:steps].abs().max())
    assert lerr < 1e-5, "loss rows differ from the single-GPU engine by %g" % lerr
    for c in range(C):
        col = [out[q * C + c][2] for q in range(R)]
        assert all(torch.equal(col[0], t) for t in col), "E0 slice %d differs inside its column group" % c
    return lerr, max(o[2].sub(single.E0[:, o[0]:o[1]]).abs().max().item() for o in out)


def check_handoff(n, reps=1000):
    """n ranks on n streams: an eager round from threads, then `reps` hand-offs captured in one graph per rank and
    replayed twice on all streams at once.  The stamp after every hand-off is logged: it must count 1, 2, 3, ..."""
    from arlib_b200 import ops
    flags = [torch.zeros(8, dtype=torch.int32, device=DEV) for _ in range(n)]
    ctr = [torch.zeros(1, dtype=torch.int32, device=DEV) for _ in range(n)]
    err = [torch.zeros(1, dtype=torch.int32, device=DEV) for _ in range(n)]
    log = [torch.zeros(reps, dtype=torch.int32, device=DEV) for _ in range(n)]
    peers = [[flags[q].data_ptr() for q in range(n) if q != r] for r in range(n)]
    torch.cuda.synchronize()
    eager = 5

    def body(r, wait, ranks):
        for _ in range(eager):
            ops.group_handoff(flags[r], peers[r], r, ctr[r], err[r])
        wait()

    _threads(n, body)
    assert all(int(c.item()) == eager for c in ctr) and all(int(e.item()) == 0 for e in err)
    graphs = []
    for r in range(n):
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, capture_error_mode="thread_local"):
            for k in range(reps):
                ops.group_handoff(flags[r], peers[r], r, ctr[r], err[r])
                log[r][k:k + 1].copy_(ctr[r])
        graphs.append(gr)
    streams = [torch.cuda.Stream(device=DEV) for _ in range(n)]
    torch.cuda.synchronize()
    for rep in range(2):
        for r in range(n):
            with torch.cuda.stream(streams[r]):
                graphs[r].replay()
        torch.cuda.synchronize()
        first = eager + rep * reps + 1
        want = torch.arange(first, first + reps, dtype=torch.int32, device=DEV)
        for r in range(n):
            assert int(err[r].item()) == 0, "rank %d: hand-off timed out" % r
            assert torch.equal(log[r], want), "rank %d: stamps are not 1, 2, 3, ..." % r
            slots = flags[r][:n].cpu().tolist()
            assert all(slots[q] == first + reps - 1 for q in range(n) if q != r), slots


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("what", choices=["engine", "handoff"])
    ap.add_argument("--grid", default="2x2")
    ap.add_argument("--d", type=int, nargs="+", default=[64, 128])
    ap.add_argument("--layers", type=int, nargs="+", default=[1, 2, 3])
    ap.add_argument("--ranks", type=int, nargs="+", default=[2, 3, 4, 8])
    a = ap.parse_args()
    torch.cuda.set_device(DEV)
    if a.what == "engine":
        R, C = (int(x) for x in a.grid.split("x"))
        for d in a.d:
            for L in a.layers:
                lerr, eerr = check_engine(R, C, d, L)
                print("GRID_OK %dx%d d=%d L=%d loss_rel_err=%.2e table_err=%.2e" % (R, C, d, L, lerr, eerr), flush=True)
    else:
        for n in a.ranks:
            check_handoff(n)
            print("HANDOFF_OK ranks=%d" % n, flush=True)


if __name__ == "__main__":
    main()
