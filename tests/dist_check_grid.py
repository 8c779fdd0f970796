"""Worker for tests/test_gpu_grid_dist.py (run under torchrun, one rank per GPU, 4 or 8 ranks): the grid layout of
LightGCNEngine (R row blocks x C column slices) must reproduce the single-GPU engine.  Runs every grid shape of the
world size: 2x2 on 4 GPUs, 2x4 and 4x2 on 8."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import scipy.sparse as sp
import torch
import torch.distributed as dist


def main():
    rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"]); local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from arlib_b200.dist import DistContext
    from arlib_b200.engine import DeviceTrainSet, LightGCNEngine
    from arlib_b200.evaluator import FullRankEvaluator
    from arlib_b200.graph import DeviceGraph
    from arlib_b200.util.synth import synth_edges

    U, I, E, d, L, B = 3000, 4000, 90000, 64, 3, 2048
    tu, ti, su, si = synth_edges(U, I, E, seed=11)
    N = U + I
    half = sp.csr_matrix((np.ones(E, dtype=np.float32), (tu, ti + U)), shape=(N, N), dtype=np.float32)
    g = DeviceGraph.from_dataloader_adj(half + half.T, dev)
    torch.manual_seed(0)
    table0 = (torch.rand(N, d) - 0.5) * 0.2
    ts = DeviceTrainSet.from_arrays(tu, ti, U, I, dev)

    single = LightGCNEngine(g, table0.clone().to(dev), U, L, 0.005, 1e-4, B, E)
    single.sample_epoch(ts, 7, 0)
    single.run_steps(0, 5, use_graph=False)
    Fs = single.forward_table().clone()
    ev = FullRankEvaluator.from_arrays(U, I, tu, ti, su, si, dev)
    shapes = [s for s in ((2, 2), (2, 4), (4, 2)) if s[0] * s[1] == world]
    assert shapes, "the grid test runs on 4 or 8 ranks"
    for R, C in shapes:
        eng = LightGCNEngine(g, table0.clone().to(dev), U, L, 0.005, 1e-4, B, E, comm=DistContext(dev), mode="grid",
                             grid=(R, C))
        assert eng.d == d // C and (eng.grid_r, eng.grid_c) == divmod(rank, C)
        eng.sample_epoch(ts, 7, 0)
        eng.run_steps(0, 2, use_graph=False)
        eng.run_steps(2, 3, use_graph=True)                  # captured: hand-offs and the stamped loss exchange
        eng.check_handoff()
        dist.barrier()
        full = eng.full_table(eng.E0)
        err = float((full - single.E0).abs().max())
        assert err < 2e-6, "grid %dx%d rank %d: table differs from single-GPU by %g" % (R, C, rank, err)
        loss = eng.out4[:5].contiguous()
        lerr = float(((loss - single.out4[:5]).abs().max() / single.out4[:5].abs().max()))
        assert lerr < 1e-5, lerr
        rows = [torch.empty_like(loss) for _ in range(world)]
        dist.all_gather(rows, loss)
        assert all(torch.equal(rows[0], r) for r in rows), "loss rows differ between ranks"
        Fg = eng.full_table(eng.forward_table())
        ferr = float((Fg - Fs).abs().max())
        assert ferr < 2e-6, "grid %dx%d rank %d: full_table(forward) differs by %g" % (R, C, rank, ferr)
        # user-sharded top-K of the grid's forward table == its unsharded top-K
        v2, i2 = ev.topk(Fg[:U], Fg[U:], 50)
        v3, i3 = ev.topk_user_sharded(Fg[:U], Fg[U:], 50, rank, world)
        assert torch.equal(i2, i3) and torch.equal(v2, v3), "grid %dx%d: user-sharded top-K differs" % (R, C)
        # 200 steps back to back from one captured graph: the hand-offs and the loss exchange stay in step
        eng.run_steps(0, 40)
        for _ in range(4):
            eng.run_steps(0, 40)
        eng.check_handoff()
        dist.barrier()
        rows = [torch.empty_like(eng.out4[:40]) for _ in range(world)]
        dist.all_gather(rows, eng.out4[:40].contiguous())
        assert all(torch.equal(rows[0], r) for r in rows) and bool(torch.isfinite(rows[0]).all())
        # 2L per step (2 eager, a warm-up + 3 replayed, a warm-up + 200 replayed) and L for the forward table
        assert int(eng.handoff_ctr.item()) == (2 + 1 + 3 + 1 + 200) * 2 * L + L, int(eng.handoff_ctr.item())
        if rank == 0:
            print("GRID_DIST_OK %dx%d table_err=%.2e forward_err=%.2e loss_err=%.2e" % (R, C, err, ferr, lerr),
                  flush=True)
        dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
