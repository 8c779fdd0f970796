"""Row-partitioned NGCF step time on P GPUs (NGCFEngine(comm=DistContext)), run under torchrun; P = 1 is the
single-GPU engine.  One JSON line per (workload, d) from rank 0, after a line with the card's name, power limit and
max SM clock read in the same job:

  * ms per step of graph-replayed steps (>= 200 after warm-up), CUDA events, the maximum over ranks, three repeats;
  * per rank: rows and non-zeros owned, and the per-launch times of the step's kernels measured alone in an eager pass
    on the rank's rows (SpMM forward / backward, dense forward / backward with their peer stores, the dW slot sum, one
    barrier), with the per-step totals they make (L of each, 2L + 1 barriers);
  * at P = 1, the row-range weights a (us per non-zero of a layer's two SpMMs) and b (us per row of its dense forward
    and backward) that NGCFEngine.ROW_COST takes.

    torchrun --nproc-per-node P tools/ngcf_dist_bench.py [--workload gowalla] [--d 64 128 256] [--steps 200]
                                                         [--out FILE.jsonl]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import scipy.sparse as sp
import torch
import torch.distributed as dist

from bench import make_data
from arlib_b200 import ops
from arlib_b200.engine import DeviceTrainSet, NGCFEngine
from arlib_b200.graph import DeviceGraph

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="gowalla")
ap.add_argument("--d", type=int, nargs="+", default=[64, 128, 256])
ap.add_argument("--steps", type=int, default=200)
ap.add_argument("--repeats", type=int, default=3)
ap.add_argument("--out", default=None, help="append the JSON lines to this file (rank 0)")
cli = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("needs a CUDA device")

rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
local = int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
comm = None
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
    from arlib_b200.dist import DistContext


def emit(rec):
    if rank == 0:
        line = json.dumps(rec)
        print(line, flush=True)
        if cli.out:
            with open(cli.out, "a") as f:
                f.write(line + "\n")


def gather_obj(x):
    if world == 1:
        return [x]
    out = [None] * world
    dist.all_gather_object(out, x)
    return out


if rank == 0:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(local)], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    emit({"card": q or torch.cuda.get_device_name(dev), "gpus": world})

D = make_data(cli.workload, 0.5)
U, I, E, L, B = D["U"], D["I"], D["E"], D["L"], D["B"]
N = U + I
half = sp.csr_matrix((np.ones(E, dtype=np.float32), (D["tu"], D["ti"] + U)), shape=(N, N), dtype=np.float32)
g = DeviceGraph.from_dataloader_adj(half + half.T, dev)
ts = DeviceTrainSet.from_arrays(D["tu"], D["ti"], U, I, dev)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def timed_us(fn, n=50):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


for d in cli.d:
    gen = torch.Generator().manual_seed(2018)
    a = (6.0 / (N + d)) ** 0.5
    table = ((torch.rand(N, d, generator=gen) * 2 - 1) * a).to(dev)
    W = ((torch.rand(L, 2 * d, d, generator=gen) * 2 - 1) * (6.0 / (2 * d)) ** 0.5).to(dev).contiguous()
    if world > 1:
        comm = DistContext(dev)
    eng = NGCFEngine(g, table, W, U, 0.005, 1e-4, B, E, comm=comm)
    eng.sample_epoch(ts, 2018, 0)
    K = cli.steps
    if K > eng.n_batches:
        raise SystemExit("only %d batches per epoch at this shape" % eng.n_batches)
    eng.run_steps(0, 3, use_graph=False)
    eng.run_steps(0, K)                                  # capture + one replay: warm-up
    torch.cuda.synchronize()
    reps = []
    for _ in range(cli.repeats):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        eng.run_steps(0, K)
        e1.record()
        torch.cuda.synchronize()
        reps.append(max(gather_obj(e0.elapsed_time(e1) / K)))

    # eager pass: every launch of the step alone, on this rank's rows
    r0, r1 = eng.r0, eng.r1
    rows = lambda t: t[r0:r1]
    X, P_, Y = eng.E0, eng.P[0], eng.Ek[-1]
    rows_mode = eng.mode == "rows"
    pk = dict(peer_Enext=eng._peer_rows["E1"], mc_Enext=eng._mc_rows["E1"]) if rows_mode and L > 1 else {}
    spmm_fwd = timed_us(lambda: ops.spmm(eng.g, X, Y=P_))
    spmm_bwd = timed_us(lambda: ops.spmm(eng.g, eng.dPs[0], addend=eng.dEdir, acc_in=eng.G, acc_out=eng.dOut[0]))
    fwd = timed_us(lambda: ops.ngcf_dense_forward(rows(P_), rows(X), W[0], rows(eng.Ek[0]), **pk))
    bk = {}
    slot = eng.dW[0]
    if rows_mode:
        bk = dict(peer_dP=eng._peer_rows["dP0"], mc_dP=eng._mc_rows["dP0"], peer_dW=eng._peer_slot[0],
                  mc_dW=eng._mc_slot[0])
        slot = eng.dW_slots[0, comm.rank]
    bwd = timed_us(lambda: ops.ngcf_dense_backward(rows(eng.G), rows(Y), rows(P_), rows(X), eng.WT[0], rows(eng.dPs[0]),
                                                   rows(eng.dEdir), eng.dW_partial, slot, **bk))
    slot_sum = timed_us(lambda: ops.ngcf_reduce_wgrad(eng.dW_slots[0], eng.dW[0])) if rows_mode else 0.0
    barrier = timed_us(comm.barrier) if rows_mode else 0.0
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
    mine = {"rank": rank, "rows": r1 - r0, "nnz": eng.g.local_nnz, "spmm_fwd_us": spmm_fwd, "spmm_bwd_us": spmm_bwd,
            "dense_fwd_us": fwd, "dense_bwd_us": bwd, "slot_sum_us": slot_sum, "barrier_us": barrier,
            "step_spmm_us": L * (spmm_fwd + spmm_bwd), "step_dense_us": L * (fwd + bwd + slot_sum),
            "step_barrier_us": (2 * L + 1) * barrier}
    per_rank = gather_obj(mine)
    rec = {"workload": cli.workload, "N": N, "nnz": g.nnz, "L": L, "d": d, "B": B, "gpus": world, "mode": eng.mode,
           "steps_timed": K, "ms_per_step_repeats": reps, "ms_per_step": float(np.median(reps)),
           "spread_ms": max(reps) - min(reps), "launches_per_step": eng.launches_per_step,
           "row_cost": NGCFEngine.ROW_COST.get(d), "per_rank": per_rank}
    if world == 1:
        rec["row_cost_measured"] = [(spmm_fwd + spmm_bwd) / g.nnz, (fwd + bwd) / N]
    emit(rec)
    del eng
    torch.cuda.synchronize()

if world > 1:
    dist.barrier()
    dist.destroy_process_group()
