"""Multi-GPU layouts of the LightGCN step side by side: "dshard", "rows" and "grid" (R row blocks x C column slices) on
the synthetic shapes of bench.py, one JSON line per layout on rank 0.

    torchrun --nproc-per-node 8 tools/grid_bench.py --workload gowalla --grids 2x4 4x2 [--steps 200 --warmup 20]

Per layout: ms/step (device events around CUDA-graph replays of ``--steps`` consecutive steps, the slowest rank),
triples/s, the mean device time of one SpMM launch and of one hand-off / barrier (events around every launch of an
eager pass of ``--probe`` steps; eager, so these include no graph-launch savings), and the bytes of the step's tables
per GPU.  The card name and power limit are read in the same run.  On one process it times the single-GPU engine."""
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

from bench import LR, REG, WORKLOADS, make_data, xavier_tables


def card():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        power = out.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def table_bytes(eng):
    """bytes of the [N, d_local] tables one GPU holds for the step (parameters, layers, gradient, Adam moments)"""
    seen, total = set(), 0
    for t in [eng.E0, eng.F, eng.G, eng.dE0, eng.m, eng.v] + list(eng.fw) + list(eng.bw):
        if t.data_ptr() not in seen:
            seen.add(t.data_ptr())
            total += t.numel() * t.element_size()
    return total


def probe(eng, first, n, comm):
    """mean device time of one SpMM launch and of one hand-off / barrier over an eager pass of n steps"""
    from arlib_b200 import ops
    import arlib_b200.engine as engmod
    rec = {"spmm": [], "sync": []}

    def wrap(key, fn):
        def f(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            rec[key].append((e0, e1))
            return r
        return f

    saved = (engmod.ops.spmm, engmod.ops.group_handoff, comm.barrier if comm is not None else None)
    engmod.ops.spmm = wrap("spmm", ops.spmm)
    engmod.ops.group_handoff = wrap("sync", ops.group_handoff)
    if comm is not None:
        comm.barrier = wrap("sync", comm.barrier)
    try:
        eng.run_steps(first, n, use_graph=False)
        torch.cuda.synchronize()
    finally:
        engmod.ops.spmm, engmod.ops.group_handoff = saved[0], saved[1]
        if comm is not None:
            comm.barrier = saved[2]
    us = lambda evs: float(np.mean([a.elapsed_time(b) * 1e3 for a, b in evs])) if evs else 0.0
    return us(rec["spmm"]), us(rec["sync"]), len(rec["sync"]) // n


def run(args, mode, grid, D, g, table, ts, world, dev):
    from arlib_b200.dist import DistContext
    from arlib_b200.engine import LightGCNEngine
    U, L, B, E = D["U"], D["L"], D["B"], D["E"]
    comm = DistContext(dev) if world > 1 else None
    eng = LightGCNEngine(g, table.clone(), U, L, LR, REG, B, E, comm=comm, mode=mode, grid=grid)
    eng.sample_epoch(ts, 2018, 0)
    n = min(args.steps, eng.n_batches - 1)
    w = min(args.warmup, n)
    eng.run_steps(0, w)                                          # capture + warm-up replays of the short graph
    eng.run_steps(0, n)                                          # capture of the timed graph (its first replay)
    torch.cuda.synchronize()
    if comm is not None:
        dist.barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    eng.run_steps(0, n)
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / n
    if hasattr(eng, "check_handoff"):
        eng.check_handoff()
    spmm_us, sync_us, syncs = probe(eng, 0, min(args.probe, n), comm)
    loss = float(eng.out4[:n, 0].mean())
    vals = torch.tensor([ms, spmm_us, sync_us], dtype=torch.float64, device=dev)
    if comm is not None:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    ms, spmm_us, sync_us = vals.tolist()
    return {"mode": eng.mode, "grid": list(eng.grid) if eng.mode == "grid" else None, "gpus": world,
            "d_local": eng.d, "ms_per_step": round(ms, 4), "triples_per_s": round(B / ms * 1e3),
            "spmm_launch_us": round(spmm_us, 2), "sync_us": round(sync_us, 2), "syncs_per_step": syncs,
            "table_bytes_per_gpu": table_bytes(eng), "steps": n, "mean_loss": loss}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="gowalla", choices=sorted(WORKLOADS))
    ap.add_argument("--alpha", type=float, default=0.5)
    ap.add_argument("--modes", nargs="+", default=["dshard", "rows", "grid"])
    ap.add_argument("--grids", nargs="+", default=[], help="RxC shapes for mode grid, e.g. 2x4 4x2")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--probe", type=int, default=20)
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from arlib_b200.engine import DeviceTrainSet
    from arlib_b200.graph import DeviceGraph
    D = make_data(args.workload, args.alpha)
    U, I, E = D["U"], D["I"], D["E"]
    N = U + I
    half = sp.csr_matrix((np.ones(E, dtype=np.float32), (D["tu"], D["ti"] + U)), shape=(N, N), dtype=np.float32)
    g = DeviceGraph.from_dataloader_adj(half + half.T, dev)
    ue, ie = xavier_tables(U, I, D["d"])
    table = torch.cat([ue, ie]).to(dev)
    ts = DeviceTrainSet.from_arrays(D["tu"], D["ti"], U, I, dev)
    name, power = card()
    configs = [("rows", None)] if world == 1 else []
    if world > 1:
        for mode in args.modes:
            if mode == "grid":
                configs += [("grid", tuple(int(x) for x in s.split("x"))) for s in args.grids]
            else:
                configs.append((mode, None))
    for mode, grid in configs:
        res = run(args, mode, grid, D, g, table, ts, world, dev)
        res.update(workload=args.workload, d=D["d"], layers=D["L"], batch=D["B"], card=name, power_limit=power)
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps(res), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
