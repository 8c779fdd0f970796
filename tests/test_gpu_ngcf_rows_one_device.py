"""The row-partitioned NGCFEngine on ONE GPU: P ranks run as threads, each on its own stream, and a stand-in for
DistContext gives every rank its own allocation of each symmetric table, the other ranks' allocations as peer pointers,
no multicast, and a barrier that drains the rank's stream and waits for the other threads.  The kernels then store into
the peers' copies exactly as over NVLink, so the whole data flow of the layout -- row ranges, which tables are
exchanged, dP parity, the dW slots, the owner's Adam on E0 -- runs against the single-GPU engine with the checks of
tests/dist_check_ngcf.py (all but graph replay -- this barrier is a host wait -- and the user-sharded top-K, whose
all-gather needs a process group)."""
import threading

import pytest
import torch

import dist_check_ngcf

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


class _Ranks:
    def __init__(self, world):
        self.world = world
        self.sync = threading.Barrier(world, timeout=300)
        self.wait = self.sync.wait
        self.slots = [None] * world


class _ThreadComm:
    """DistContext's interface for one rank of a _Ranks group"""

    def __init__(self, ranks, rank):
        self.ranks, self.rank, self.world = ranks, rank, ranks.world
        self.bufs = None

    def allocate(self, specs):
        self.bufs = {k: torch.empty(shape, dtype=dt, device=DEV) for k, (shape, dt) in specs.items()}
        self.ranks.slots[self.rank] = self.bufs
        self.barrier()
        self.peer_bufs = [self.ranks.slots[r] for r in range(self.world) if r != self.rank]
        self.barrier()
        return self.bufs

    def peers(self, name, extra_bytes=0):
        return [b[name].data_ptr() + int(extra_bytes) for b in self.peer_bufs]

    def multicast_ptr(self, name, extra_bytes=0):
        return 0

    def barrier(self):
        torch.cuda.current_stream().synchronize()
        self.ranks.wait()


def _run(world, d, L):
    ranks = _Ranks(world)
    gathered = [None] * world
    errors = []

    def rank_main(r):
        comm_of = lambda: _ThreadComm(ranks, r)
        stream = torch.cuda.Stream(device=DEV)

        def barrier():
            stream.synchronize()
            ranks.wait()

        def gather(t):
            gathered[r] = t.clone()
            barrier()
            out = list(gathered)
            barrier()
            return out

        try:
            with torch.cuda.stream(stream):
                dist_check_ngcf.check_rows_engine(comm_of, barrier, gather, r, world, DEV, d, L, graphs=False,
                                                  sharded_topk=False)
        except BaseException as e:          # noqa: BLE001 -- reported by the main thread
            errors.append((r, e))
            ranks.sync.abort()

    threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    torch.cuda.synchronize()
    if errors:
        raise errors[0][1]


@pytest.mark.parametrize("d", [8, 32, 64, 128, 256])
def test_two_rank_rows_layout_matches_single_gpu(d):
    _run(2, d, 2)


def test_three_rank_rows_layout_three_layers():
    _run(3, 64, 3)
