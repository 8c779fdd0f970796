#!/usr/bin/env python
"""bench.py -- LightGCN train triples/s (+ full-rank eval users/s) on synthetic
Gowalla-shaped data, B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" is one BPR batch of 2048 triples through
the whole hot path: L=3 propagation forward, fused loss, backward, Adam
(recommender/LightGCN.py:47-64 of the reference).  See DESIGN.md "Measurement".

--dump-outputs DIR also writes the tables after the last timed step, that step's loss row and the last timed
evaluation's top-K and per-user metrics as DIR/<name>.npy: the inputs are seeded, so two builds run with the same
arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

WORKLOADS = {
    # name: (users, items, edges, layers, d, batch)          BASELINE.json configs[1] = gowalla
    "gowalla": (29858, 40981, 1027370, 3, 64, 2048),
    "ml-100k": (943, 1682, 100000, 2, 64, 2048),
    "yelp2018": (31668, 38048, 1561406, 2, 64, 2048),
    "ml-1m": (6040, 3706, 1000209, 2, 64, 2048),
    "amazon-book": (52643, 91599, 2984108, 3, 128, 2048),
}
LR, REG, TOPK = 0.005, 1e-4, 50
L2_GATHER_PEAK_GBS = 18400.0      # measured on B200 this round (profiles/r1_l2_gather_peak.txt)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------- data
def make_data(name, alpha, seed=0):
    # generated on every run (about a second at the Gowalla shape) rather than cached: a cached graph would outlive a
    # change of the generator and feed two builds different inputs
    from arlib_b200.util.synth import synth_edges
    U, I, E, L, d, B = WORKLOADS[name]
    tu, ti, su, si = synth_edges(U, I, E, alpha, alpha, seed)
    return dict(U=U, I=I, E=E, L=L, d=d, B=B, tu=tu, ti=ti, su=su, si=si)


DUMP_BUDGET_BYTES = 63_000_000       # under 64 MB with the .npy headers


def dump_outputs(out_dir, arrays, budget=DUMP_BUDGET_BYTES):
    """Write ``{name: array}`` as ``out_dir/<name>.npy`` (float32 stays float32, everything else becomes float64).
    When the arrays exceed ``budget`` bytes in all, every array of two or more dimensions keeps a fixed, seeded sample
    of its rows (the same rows for arrays of the same length) and ``<name>_rows.npy`` holds the row numbers kept."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in arrays.items()}
    sampled = lambda v: v.ndim >= 2
    total = sum(v.nbytes + (8 * v.shape[0] if sampled(v) else 0) for v in arrays.values())
    keep = budget / total if total > budget else 1.0
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        if keep < 1.0 and sampled(v):
            n = v.shape[0]
            rows = np.sort(np.random.default_rng(0).choice(n, max(1, int(n * keep)), replace=False))
            v = v[rows]
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(out_dir, name + ".npy"), v)


def xavier_tables(U, I, d, seed=2018):
    torch.manual_seed(seed)
    ue = torch.nn.init.xavier_uniform_(torch.empty(U, d))
    ie = torch.nn.init.xavier_uniform_(torch.empty(I, d))
    return ue, ie


def algorithmic_bytes(N, nnz, d, L, B):
    """SURVEY.md 8d: contract figures."""
    T = N * d * 4
    b_spmm = nnz * 8 + (N + 1) * 4 + 2 * T
    b_step = 2 * L * b_spmm + 7 * T + 3 * B * d * 4 * (L + 1) * 2 + 24 * B
    return b_spmm, b_step


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi-equivalent clock / throttle sampling through NVML during the timed region."""

    def __init__(self, index=0, period=0.02):
        self.samples, self.reasons, self.period, self.index = [], set(), period, index
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.nv, self.max_mhz = None, None
            log("NVML unavailable:", e)

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "hw_power_brake": 0x80, "sync_boost": 0x10, "display_clock": 0x100, "app_clocks": 0x2}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t is not None:
            self._t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------- baseline legs
def host_threads():
    """all host cores for the CPU legs: torchrun exports OMP_NUM_THREADS=1 to every rank, which would make the
    reference arm single-threaded at N > 1 (VERDICT r1) -- the arm runs on rank 0 alone and may use the whole host"""
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        pass
    torch.set_num_threads(n)
    return n


def write_reference_dataset(D, name, max_test_users):
    """the synthetic graph in the reference's text format ("<user> <item> 1" per line, util/FileIO.py:22-31) under
    /tmp/arlib_b200_ref/data/clean/<name>/; the test file keeps the pairs of the first ``max_test_users`` test users
    (the bounded evaluation sample)"""
    root = "/tmp/arlib_b200_ref"
    d = os.path.join(root, "data", "clean", name)
    os.makedirs(d, exist_ok=True)
    users = np.unique(D["su"])[:max_test_users]
    keep = np.isin(D["su"], users)

    def dump(path, u, i):
        with open(path, "w") as fh:
            fh.write("".join("%d %d 1\n" % (a, b) for a, b in zip(u.tolist(), i.tolist())))
    dump(os.path.join(d, "train.txt"), D["tu"], D["ti"])
    dump(os.path.join(d, "test.txt"), D["su"][keep], D["si"][keep])
    dump(os.path.join(d, "val.txt"), D["su"][keep][:1000], D["si"][keep][:1000])
    return root, int(users.shape[0])


def reference_leg(D, name, n_steps, n_warm, cuda, eval_users=2000):
    """The UNMODIFIED reference (oracle/_ref, staged by oracle/make_ref.py) through its own public API:
    ``DataLoader(args)``, ``LightGCN(args, data)``, ``train(Epoch=1)`` and ``test()`` (recommender/LightGCN.py:29-80,
    137-161).  The only interception is the sampler generator, wrapped to stop after n_warm + n_steps batches and to
    take the timestamps -- so a timed step is exactly the reference's: Python rejection sampler (util/sampler.py:4-30),
    model(), gathers, bpr_loss + l2_reg_loss, backward, Adam.  ``cuda=False``: the reference's CPU torch path (its
    ``.cuda()`` calls made identities); ``cuda=True``: its own eager PyTorch + cuSPARSE path on this GPU.
    -> dict(triples_per_s, s_per_step, users_per_s, n_eval_users)"""
    import contextlib
    import io
    from oracle import ref_loader
    root, n_eval = write_reference_dataset(D, name, eval_users)
    stamps = []
    old = os.getcwd()
    os.chdir(root)
    try:
        with ref_loader.reference_modules(cuda=cuda) as ref, contextlib.redirect_stdout(io.StringIO()):
            args = ref_loader.make_args(ref, dataset=name, data_path="data/clean/", model_name="LightGCN", maxEpoch=1,
                                        n_layers=D["L"], emb_size=D["d"], batch_size=D["B"], lRate=LR, reg=REG,
                                        topK=str(TOPK))
            ref.tool.seedSet(2018)
            data = ref.DataLoader(args)
            rec = ref.LightGCN.LightGCN(args, data)
            real = ref.LightGCN.next_batch_pairwise

            def sync():
                if cuda:
                    torch.cuda.synchronize()

            def truncated(d_, bs):
                for k, b in enumerate(real(d_, bs)):
                    if k >= n_warm + n_steps:
                        break
                    if k == n_warm:
                        sync(); stamps.append(time.perf_counter())
                    yield b
                sync(); stamps.append(time.perf_counter())
            ref.LightGCN.next_batch_pairwise = truncated
            ref.algorithm.find_k_largest(TOPK, np.random.rand(D["I"]).astype(np.float32))      # numba JIT warm-up
            try:
                rec.train(Epoch=1)               # the truncated epoch, then the reference's own evaluate() (untimed here)
            finally:
                ref.LightGCN.next_batch_pairwise = real
            sync(); t0 = time.perf_counter()
            rec.test()
            sync(); t_eval = time.perf_counter() - t0
    finally:
        os.chdir(old)
    dt = stamps[1] - stamps[0]
    return {"triples_per_s": n_steps * D["B"] / dt, "s_per_step": dt / n_steps, "users_per_s": n_eval / t_eval,
            "n_eval_users": n_eval}


def port_leg(D, n_steps, n_warm, eval_users=300):
    """fallback when no reference copy is staged: oracle/port.py's restatement of the same loop body (torch CPU),
    incl. the reference's Python rejection sampler on an array-backed data shim"""
    from oracle import port
    U, I, L, d, B = D["U"], D["I"], D["L"], D["d"], D["B"]
    adj = port.bipartite_adjacency(D["tu"], D["ti"], U, I)
    norm = port.normalize_graph_mat(adj)
    ue, ie = xavier_tables(U, I, d)
    tr = port.LightGCNTrainer(norm, ue, ie, L, LR, REG)
    rng = np.random.default_rng(1)
    train_of = {}
    for u, i in zip(D["tu"].tolist(), D["ti"].tolist()):
        train_of.setdefault(u, set()).add(i)

    def batch(k):
        lo = (k * B) % (D["E"] - B)
        u, i = D["tu"][lo:lo + B].tolist(), D["ti"][lo:lo + B].tolist()
        j = []
        for uu in u:                                   # util/sampler.py:23-29: rejection sampling per triple
            neg = int(rng.integers(0, I))
            while neg in train_of[uu]:
                neg = int(rng.integers(0, I))
            j.append(neg)
        return u, i, j

    for k in range(n_warm):
        tr.step(*batch(k))
    t0 = time.perf_counter()
    for k in range(n_steps):
        tr.step(*batch(n_warm + k))
    dt = time.perf_counter() - t0
    users = np.unique(D["su"])[:eval_users]
    data = port.ArrayEvalData(U, I, D["tu"], D["ti"], D["su"], D["si"], users)
    port.find_k_largest(TOPK, np.random.rand(I).astype(np.float32))       # numba JIT warm-up
    names = [str(int(u)) for u in users]
    t1 = time.perf_counter()
    port.full_rank_test(data, ue, ie, TOPK, [TOPK], users=names)
    return {"triples_per_s": n_steps * B / dt, "s_per_step": dt / n_steps,
            "users_per_s": len(names) / (time.perf_counter() - t1), "n_eval_users": len(names)}


def cpu_leg(D, name, n_steps, n_warm):
    """-> (result dict, kind, sample description)"""
    from oracle import ref_loader
    cores = host_threads()
    if ref_loader.available():
        r = reference_leg(D, name, n_steps, n_warm, cuda=False)
        kind = "reference"
        what = ("%d warm-up + %d timed steps of the UNMODIFIED reference's LightGCN.train() loop (oracle/_ref; Python "
                "rejection sampler + model() + loss + backward + Adam, %d triples per step, torch CPU, %d threads) and its "
                "test() over %d test users" % (n_warm, n_steps, D["B"], cores, r["n_eval_users"]))
    else:
        r = port_leg(D, n_steps, n_warm)
        kind = "port"
        what = ("%d warm-up + %d timed steps of oracle/port.py's restatement of LightGCN.train() (sampler included, torch "
                "CPU, %d threads) and a %d-user full-rank eval" % (n_warm, n_steps, cores, r["n_eval_users"]))
    return r, kind, what, cores


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores (rank 0 alone)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    D = make_data(args.workload, args.alpha)
    cap = max(1, min(args.steps, 40))
    warm = max(1, min(args.warmup, 2))
    r, kind, what, cores = cpu_leg(D, args.workload, cap, warm)
    tps = r["triples_per_s"]
    line = {
        "impl": "reference", "metric": "LightGCN train triples/s", "value": tps, "unit": "triples/s",
        "n_gpus": args.gpus, "steps": cap, "warmup": warm, "ms_per_step": r["s_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(args, D),
        "cpu_baseline": {"value": tps, "unit": "triples/s", "cores": cores, "kind": kind, "sample": what},
        "e2e": {"value": tps, "unit": "triples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "eval": {"users_per_s": r["users_per_s"], "unit": "users/s", "n_users": r["n_eval_users"]},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def config_of(args, D):
    return {"workload": "LightGCN %d-layer d=%d BPR batch %d, synthetic %s shape %dx%d, %d edges, power-law alpha=%s"
                        % (D["L"], D["d"], D["B"], args.workload, D["U"], D["I"], D["E"], args.alpha),
            "lr": LR, "reg": REG, "topK": TOPK, "sampler": "device-philox",
            "l2": "per-step working set (10 tables + CSR, ~%.0f MB) exceeds the 126 MB L2; steady-state loop, no flush"
                  % ((10 * (D["U"] + D["I"]) * D["d"] * 4 + 2 * D["E"] * 8) / 1e6)}


# --------------------------------------------------------------------------- ours
def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; arlib_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from arlib_b200 import ops
    from arlib_b200.engine import DeviceTrainSet, LightGCNEngine
    from arlib_b200.evaluator import FullRankEvaluator
    from arlib_b200.graph import DeviceGraph
    import scipy.sparse as sp

    D = make_data(args.workload, args.alpha)
    U, I, E, L, d, B = D["U"], D["I"], D["E"], D["L"], D["d"], D["B"]
    N = U + I
    half = sp.csr_matrix((np.ones(E, dtype=np.float32), (D["tu"], D["ti"] + U)), shape=(N, N), dtype=np.float32)
    adj = half + half.T
    g = DeviceGraph.from_dataloader_adj(adj, dev)
    ue, ie = xavier_tables(U, I, d)
    table = torch.cat([ue, ie]).to(dev)
    ts = DeviceTrainSet.from_arrays(D["tu"], D["ti"], U, I, dev)
    comm = None
    if world > 1:
        from arlib_b200.dist import DistContext
        comm = DistContext(dev)
    # multi-GPU layout: column-sharded tables (one 16 B/triple exchange per step) when d/P is a supported slice
    # width, else (or with ARLIB_B200_DIST=rows) row-partitioned tables with the per-layer all-gather fused
    # into the SpMM epilogue
    mode = os.environ.get("ARLIB_B200_DIST", "dshard")
    if world > 1 and (d % world or d // world not in (8, 16, 32, 64, 128, 256)):
        mode = "rows"
    eng = LightGCNEngine(g, table, U, L, LR, REG, B, E, comm=comm, mode=mode)
    K, W = args.steps, max(args.warmup, 3)
    nb_epoch = (E + B - 1) // B
    full_batches = E // B

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    use_graph = world == 1 or eng.dist_graphs
    # ---- device-resident throughput: K steps replayed from CUDA graphs of <= one epoch each
    eng.sample_epoch(ts, 2018, 0)
    chunks = []
    left, first = K, 0
    while left > 0:                                   # steps cycle through the epoch's full batches
        n = min(left, full_batches - first)
        chunks.append((first, n))
        left -= n
        first = (first + n) % full_batches
    for k in range(W):
        eng.run_steps(k % full_batches, 1, use_graph=False)
    for c in set(chunks):
        eng.run_steps(c[0], c[1] if use_graph else min(c[1], 5), use_graph=use_graph)     # capture + one replay (warm)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        barrier()
        e0.record()
        for c in chunks:
            eng.run_steps(c[0], c[1], use_graph=use_graph)
        e1.record()
        barrier()
        if args.dump_outputs:           # what the last timed step left, before the untimed steps below train on
            dump = {"table": eng.full_table(eng.E0).clone(), "loss": eng.out4[chunks[-1][0] + chunks[-1][1] - 1].clone()}
        # keep the GPU under the same load while NVML gets enough samples (not timed)
        for _ in range(3 if world > 1 else 8):
            eng.run_steps(chunks[0][0], min(chunks[0][1], 200), use_graph=use_graph)
            torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1))
    value = K * B / (ms * 1e-3)
    loss_last = float(eng.out4[chunks[-1][0] + chunks[-1][1] - 1, 0])

    # ---- per-kernel live timing of the dominant kernel (SpMM) inside eager steps
    spmm_ms = []
    orig = ops.spmm

    def timed_spmm(*a, **k):
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(); orig(*a, **k); a1.record()
        if k.get("row_mask") is not None or k.get("worklist") is not None:
            kind = "row_masked"                   # last forward layer: the batch's rows only
        elif k.get("col_mask") is not None:
            kind = "col_masked"                   # first backward layer: the batch's gradient rows only
        elif k.get("adam") is not None:
            kind = "full_with_adam"               # last backward layer: + 6 table passes of the fused optimizer
        else:
            kind = "full"
        spmm_ms.append((kind, a0, a1))

    import arlib_b200.engine as engmod
    engmod.ops.spmm = timed_spmm
    try:
        for k in range(min(K, 50)):
            eng.run_steps(k % full_batches, 1, use_graph=False)
    finally:
        engmod.ops.spmm = orig
    torch.cuda.synchronize()
    by_kind = {}
    for kind, a, b_ in spmm_ms:
        by_kind.setdefault(kind, []).append(a.elapsed_time(b_))
    # the roofline figure is for the FULL launches (the contract bytes B_spmm are those of a full propagation);
    # the two batch-sparse launches of a step move fewer bytes and are reported beside it.  An event pair around a
    # single eager launch also sees the launch gap (~5-8 us); the kernel's own duration inside the replayed graph is
    # measured with one event pair around 100 back-to-back launches of each full-launch configuration of the step
    # (forward layer 1, forward layer 2, a middle backward layer) on the engine's own tables.
    eager_full_ms = float(np.mean(by_kind["full"]))
    spmm_avg_ms = eager_full_ms
    if eng.mode != "rows" and L > 1:
        cfgs = [lambda: orig(eng.g, eng.E0, Y=eng.fw[0], acc_in=eng.E0, acc_out=eng.F),
                lambda: orig(eng.g, eng.fw[0], Y=eng.fw[1], acc_in=eng.F, acc_out=eng.F),
                lambda: orig(eng.g, eng.bw[0], Y=eng.bw[1], addend=eng.G)]
        per_cfg = []
        for fn in cfgs:
            for _ in range(10):
                fn()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            for _ in range(100):
                fn()
            b1.record()
            torch.cuda.synchronize()
            per_cfg.append(b0.elapsed_time(b1) / 100)
        spmm_avg_ms = float(np.mean(per_cfg))
    b_spmm, b_step = algorithmic_bytes(N, g.nnz, d, L, B)
    if eng.mode == "dshard":        # per-GPU launch: whole graph, a [N, d/P] slice of the tables
        b_spmm = g.nnz * 8 + (N + 1) * 4 + 2 * N * eng.d * 4
    elif eng.mode == "rows":        # per-GPU launch: this rank's rows of the graph, all of X read, its rows of Y written
        b_spmm = eng.g.local_nnz * 8 + (eng.g.n_local_rows + 1) * 4 + N * d * 4 + eng.g.n_local_rows * d * 4
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    achieved = b_spmm / (spmm_avg_ms * 1e-3) / 1e9
    traffic = None                       # dram bytes of one launch from the ncu --set full capture; only valid for the
    if world == 1:                       # single-GPU full-width kernel it was captured on (null otherwise)
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "spmm_traffic.json"))).get(args.workload)
        except Exception:
            pass
    roofline = {"kernel": "spmm_csr_kernel<%d>" % eng.d, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_kind": peak_kind,
                "algorithmic_bytes_per_launch": b_spmm, "avg_launch_ms": spmm_avg_ms,
                "avg_launch_ms_eager_single": eager_full_ms,
                "launches_per_step": 2 * L, "full_launches_per_step": len(by_kind["full"]) // max(1, min(K, 50)),
                "batch_sparse_launch_ms": {k: float(np.mean(v)) for k, v in by_kind.items() if k != "full"},
                "step_algorithmic_bytes": b_step,
                "step_frac_of_hbm_roofline": (b_step / (ms / K * 1e-3) / 1e9) / peak,
                "l2_gather": {"bytes_per_launch": int(eng.g.local_nnz * (8 + 4 * eng.d)),
                              "achieved": eng.g.local_nnz * (8 + 4 * eng.d) / (spmm_avg_ms * 1e-3) / 1e9,
                              "peak": L2_GATHER_PEAK_GBS, "unit": "GB/s",
                              "frac": eng.g.local_nnz * (8 + 4 * eng.d) / (spmm_avg_ms * 1e-3) / 1e9 / L2_GATHER_PEAK_GBS,
                              "peak_kind": "measured: tools/l2_gather_peak.cu, power-law 256-byte row gathers from an "
                                           "L2-resident table (profiles/r1_l2_gather_peak.txt, re-measured r2_l2_gather_peak.txt: 18 404)"},
                "note": "table (%.1f MB) is L2-resident and no on-chip store holds it: the launch moves nnz*(8+4d) = %.0f MB "
                        "from L2, not from DRAM; a launch whose gathers all hit one cached row takes as long "
                        "(profiles/r2_summary.md 9): the LSU data pipe and the per-item dependent chain at 32 warps / SM are "
                        "what the time is made of, the L2-gather figure is what the memory system could deliver; DESIGN.md 4.1"
                        % (N * d * 4 / 1e6, g.nnz * (8 + 4 * d) / 1e6)}

    # ---- end to end through the public step API with HOST triples (pinned), loss read back
    tu_h = [torch.empty((3, B), dtype=torch.int32).pin_memory() for _ in range(4)]
    rng = np.random.default_rng(5)
    for t in tu_h:
        sl = int(rng.integers(0, E - B))
        t[0].copy_(torch.from_numpy(D["tu"][sl:sl + B].astype(np.int32)))
        t[1].copy_(torch.from_numpy(D["ti"][sl:sl + B].astype(np.int32)))
        t[2].copy_(torch.from_numpy(rng.integers(0, I, B).astype(np.int32)))
    for k in range(W):
        eng.step_external(tu_h[k % 4], B)
    barrier()
    e0.record()
    for k in range(K):
        loss_row = eng.step_external(tu_h[k % 4], B)      # pinned host row the step's loss is copied into
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    e2e = {"value": K * B / (e2e_ms * 1e-3), "unit": "triples/s", "h2d_bytes_per_step": 3 * B * 4,
           "d2h_bytes_per_step": 16, "ms_per_step": e2e_ms / K, "last_loss": float(loss_row[0]),
           "api": "LightGCNEngine.step_external: triples in HOST memory -> pinned staging slot -> one CUDA-graph replay "
                  "per step (H2D memcpy nodes, grouping, step kernels, D2H of the loss row)"}

    # ---- full-rank evaluation (users/s)
    ev = FullRankEvaluator.from_arrays(U, I, D["tu"], D["ti"], D["su"], D["si"], dev)
    F = eng.full_table(eng.forward_table()).clone()
    n_test = ev.user_rows.numel()
    eval_shard = os.environ.get("ARLIB_B200_EVAL_SHARD", "users")
    if world > 1:
        # users: every per-user cost divides by P, one all-gather of the [n/P, K] result blocks; items: the layout for
        # item tables that do not fit one GPU (per-user work replicated, top-K merge)
        if eval_shard == "users":
            ev.topk = lambda ue_, ie_, k_, impl=None: ev.topk_user_sharded(ue_, ie_, k_, rank, world, impl)
        else:
            ev.topk = lambda ue_, ie_, k_, impl=None: ev.topk_sharded(ue_, ie_, k_, rank, world, impl)
    for _ in range(2):
        vals, idx = ev.topk(F[:U], F[U:], TOPK)
    barrier()
    reps = 10
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    evs[0].record()
    for k_ in range(reps):
        vals, idx = ev.topk(F[:U], F[U:], TOPK)
        per = ev.per_user_metrics(idx, [TOPK])
        evs[k_ + 1].record()
    barrier()
    torch.cuda.synchronize()
    # an evaluation is ~1 ms: one descheduled host thread shows up as a 10-40 ms outlier among the repetitions (seen on the
    # shared boxes), so the line carries the median next to the mean
    ev_each = sorted(evs[k_].elapsed_time(evs[k_ + 1]) for k_ in range(reps))
    ev_ms_mean = max_over_ranks(evs[0].elapsed_time(evs[-1])) / reps
    ev_ms = max_over_ranks(ev_each[reps // 2])
    if args.dump_outputs:
        dump.update(topk_scores=vals, topk_items=idx, eval_metrics=per)
    t0 = time.perf_counter()
    vals, idx = ev.topk(F[:U], F[U:], TOPK)
    measure = ev.measure(idx, [TOPK])
    idx_host = idx.cpu()
    torch.cuda.synchronize()
    ev_e2e_s = time.perf_counter() - t0
    _, _, cg = ops.score_topk(F[:U].contiguous(), F[U:].contiguous(), TOPK, user_rows=ev.user_rows[:4096].contiguous(),
                              mask_rowptr=ev.mask_rowptr, mask_items=ev.mask_items,
                              impl=int(os.environ.get("ARLIB_B200_SCORE_IMPL", "1")), return_flags=True)
    cand_groups = float(cg.float().mean().item())
    flops = 2.0 * n_test * I * d
    # the one dense contraction on its own (stage 0 + 1: mask bits, row gather, tcgen05 TF32 group-max GEMM) per user chunk
    from arlib_b200.evaluator import user_chunk
    USER_CHUNK = user_chunk(I, d, TOPK)
    s1_ms = None
    if int(os.environ.get("ARLIB_B200_SCORE_IMPL", "1")) == 1 and world == 1:
        Fu, Fi = F[:U].contiguous(), F[U:].contiguous()
        chunks_u = [ev.user_rows[lo:lo + USER_CHUNK].contiguous() for lo in range(0, n_test, USER_CHUNK)]
        # a workspace of its own: the evaluator's per-chunk workspaces keep their mask bits between evaluations
        ws_s1 = torch.empty(int(ops._lib.load().agcf_score_topk_ws_bytes(max(c.numel() for c in chunks_u), I, d, 1)),
                            dtype=torch.uint8, device=dev)

        def stage1():
            for rows_ in chunks_u:
                ops.score_group_max(Fu, Fi, user_rows=rows_, mask_rowptr=ev.mask_rowptr, mask_items=ev.mask_items, impl=1,
                                    ws=ws_s1, want_output=False)
        stage1(); stage1()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            stage1()
        e1.record()
        torch.cuda.synchronize()
        s1_ms = e0.elapsed_time(e1) / 5
    # dense TF32 peak: half the measured BF16 figure (kind::tf32 issues K = 8 per instruction where kind::f16 issues 16)
    bf16_peak = peaks.get("bf16_tflops", 1590.0)
    tf32_peak = bf16_peak / 2
    evald = {"users_per_s": n_test / (ev_ms * 1e-3), "unit": "users/s", "n_users": n_test, "ms": ev_ms,
             "ms_stat": "median of %d evaluations (top-K + metric kernel each)" % reps, "ms_mean": ev_ms_mean,
             "ms_min": ev_each[0], "ms_max": ev_each[-1],
             "e2e_users_per_s": n_test / ev_e2e_s,
             "impl": "tcgen05-tf32 + exact fp32 rescore" if int(os.environ.get("ARLIB_B200_SCORE_IMPL", "1")) == 1 else "fp32 cuda-core",
             "roofline": {"kernel": "group_max_tc_kernel<%d> (+ mask bits, row gather)" % d, "bound": "tensor",
                          "achieved": None if s1_ms is None else flops / (s1_ms * 1e-3) / 1e12, "peak": tf32_peak,
                          "unit": "TFLOP/s", "frac": None if s1_ms is None else flops / (s1_ms * 1e-3) / 1e12 / tf32_peak,
                          "traffic": None, "ms": s1_ms,
                          "peak_kind": "TF32 dense = measured BF16 peak / 2 (MEASURED_PEAKS.json bf16_tflops)",
                          "pipeline_tflops": flops / (ev_ms * 1e-3) / 1e12,
                          "note": "K = d = %d: one 128 x 256 accumulator tile is 8 MMAs (~1 024 clk) but 128 KB of TMEM to read "
                                  "back at 64 B/clk/SM (~2 048 clk): the epilogue's TMEM read path caps the tensor pipe at ~50 %% "
                                  "for this contraction (DESIGN.md 4.3); ncu sm__pipe_tensor_cycles_active in profiles/" % d},
             "candidate_groups_mean": cand_groups, "measure": [m.strip() for m in measure],
             "sharding": "single GPU" if world == 1 else ("user-sharded x%d, results all-gathered" % world
                                                          if eval_shard == "users" else "item-sharded x%d + top-K merge" % world)}

    line = {
        "metric": "LightGCN train triples/s", "value": value, "unit": "triples/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config_of(args, D),
        "roofline": roofline, "e2e": e2e, "eval": evald, "clocks": clk.summary(),
        "parallelism": {"single": "single GPU",
                        "rows": "row-partitioned x%d: per-layer all-gather fused into the SpMM epilogue (NVLink P2P "
                                "stores), item-sharded eval" % world,
                        "dshard": "column-sharded x%d: every table split [N, d/%d], graph replicated, propagation / "
                                  "backward / Adam communication-free, one P2P exchange of the partial scores (32 B per "
                                  "triple per peer): the consumer spins on step-stamped words, no barrier launch; user-sharded eval" % (world, world)}[eng.mode],
        "gpu_launches": K * eng.launches_per_step, "last_loss": loss_last,
    }
    # ---- the recommender-level number (north_star: "trains one epoch plus full-rank eval"): wall clock of the drop-in
    # class's own public calls, LightGCN(args, data).train() with maxEpoch = 1 (DeviceTrainSet, Philox sampling of the
    # epoch, all ceil(E/B) steps, end-of-epoch forward, evaluate() incl. best-epoch bookkeeping) and test()
    if rank == 0 and world == 1 and not args.no_epoch_e2e:
        import contextlib, io, types
        from arlib_b200.recommender.LightGCN import LightGCN
        from arlib_b200.util.DataLoader import DataLoader
        t0 = time.perf_counter()
        data = DataLoader.from_arrays(D["tu"], D["ti"], D["su"], D["si"])
        t_data = time.perf_counter() - t0
        rargs = types.SimpleNamespace(topK=str(TOPK), emb_size=d, n_layers=L, batch_size=B, lRate=LR, reg=REG, maxEpoch=1,
                                      seed=2018, model_name="LightGCN")
        runs = []
        with contextlib.redirect_stdout(io.StringIO()):
            torch.manual_seed(2018)
            rec = LightGCN(rargs, data)
            for _ in range(2):                         # first call builds the device mirrors, the second re-uses them
                torch.cuda.synchronize(); t0 = time.perf_counter()
                rec.train()
                torch.cuda.synchronize(); t1 = time.perf_counter()
                _, measure_e = rec.test()
                torch.cuda.synchronize(); t2 = time.perf_counter()
                runs.append((t1 - t0, t2 - t1))
        line["epoch_e2e"] = {"api": "LightGCN(args, data).train() [maxEpoch=1: %d steps + evaluate()] ; test()" % nb_epoch,
                             "train_epoch_s": [r[0] for r in runs], "test_s": [r[1] for r in runs],
                             "triples_per_s": E / runs[-1][0], "test_users_per_s": n_test / runs[-1][1],
                             "data_object_build_s": t_data, "recall_after_2_epochs": measure_e[3].strip()}
    if rank == 0 and not args.no_cpu_baseline:
        r, kind, what, cores = cpu_leg(D, args.workload, 8, 2)
        line["cpu_baseline"] = {"value": r["triples_per_s"], "unit": "triples/s", "cores": cores, "kind": kind,
                                "eval_users_per_s": r["users_per_s"], "sample": what}
        # the honest prior-art bar (SURVEY.md 8d, BASELINE.md 3.4): the reference's OWN GPU path -- eager PyTorch,
        # uncoalesced COO torch.sparse.mm (cuSPARSE), Python sampler, per-user GEMV + D2H -- on this same B200
        from oracle import ref_loader
        if ref_loader.available() and world == 1:
            try:
                g_ = reference_leg(D, args.workload, 20, 3, cuda=True)
                line["gpu_eager_baseline"] = {
                    "value": g_["triples_per_s"], "unit": "triples/s", "ms_per_step": g_["s_per_step"] * 1e3,
                    "eval_users_per_s": g_["users_per_s"], "n_eval_users": g_["n_eval_users"],
                    "what": "the UNMODIFIED reference (oracle/_ref) on this GPU: LightGCN.train() loop, 3 warm-up + 20 timed "
                            "steps incl. its Python sampler, and test() over %d users" % g_["n_eval_users"],
                    "speedup_e2e": e2e["value"] / g_["triples_per_s"],
                    "speedup_eval_e2e": evald["e2e_users_per_s"] / g_["users_per_s"]}
            except Exception as ex:          # the baseline must never take the bench line down with it
                line["gpu_eager_baseline"] = {"unavailable": repr(ex)[:300]}
    if rank == 0 and args.dump_outputs:
        table = dump.pop("table").cpu().numpy()
        dump = {k: v.cpu().numpy() for k, v in dump.items()}
        dump_outputs(args.dump_outputs, {"user_emb": table[:U], "item_emb": table[U:], **dump})
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


# ------------------------------------------------------------------ scale stress (configs[4], second half)
SCALE_SHAPES = {
    # BASELINE.json configs[4]: "a 10M-user x 1M-item power-law graph row-partitioned across 2/4/8 B200"; the edge count is
    # SURVEY.md 8's choice (average user degree 20).  c5b-small keeps the code path testable on a short GPU slot.
    "c5b": (10_000_000, 1_000_000, 200_000_000, 3, 128, 2048),
    "c5b-small": (1_000_000, 100_000, 20_000_000, 3, 128, 2048),
}


def run_scale_stress(args):
    """LightGCN d = 128 on a graph built ON THE DEVICE (generator -> canonical CSR -> normalization -> work plan -> train
    set; nothing of it exists on the host, the reference's dict-of-dicts loader cannot hold it: no CPU arm).  A full
    epoch would be E / B = 97 657 full-graph steps, so -- as SURVEY.md 8d prescribes -- the line reports per-step and
    per-SpMM numbers over K steps on a 64-batch sample of the epoch."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from arlib_b200 import ops
    from arlib_b200.engine import DeviceTrainSet, LightGCNEngine
    from arlib_b200.graph import DeviceGraph
    from arlib_b200.util.synth import synth_edges_device
    U, I, E, L, d, B = SCALE_SHAPES[args.workload]
    N = U + I
    t0 = time.perf_counter()
    eu, ei = synth_edges_device(U, I, E, args.alpha, args.alpha, seed=0, device=dev)
    E = int(eu.numel())
    g = DeviceGraph.from_device_edges(eu, ei, U, I)
    del eu, ei
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t0
    ts = DeviceTrainSet.from_graph(g, U, I, epoch_edges=64 * B, seed=1)
    gen = torch.Generator(device=dev).manual_seed(2018)
    table = torch.empty((N, d), dtype=torch.float32, device=dev)
    for lo, hi in ((0, U), (U, N)):                      # xavier_uniform per table: U(-a, a), a = sqrt(6 / (rows + d))
        a = (6.0 / ((hi - lo) + d)) ** 0.5
        table[lo:hi] = (torch.rand((hi - lo, d), generator=gen, device=dev) * 2 - 1) * a
    comm = None
    mode = os.environ.get("ARLIB_B200_DIST", "rows")      # north_star's layout is the default here
    if world > 1:
        from arlib_b200.dist import DistContext
        comm = DistContext(dev)
    eng = LightGCNEngine(g, table, U, L, LR, REG, B, ts.n_edges, comm=comm, mode=mode)
    if eng.mode != "single":
        del table
    torch.cuda.empty_cache()
    K, W = args.steps, max(args.warmup, 3)
    nb = ts.n_edges // B

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    eng.sample_epoch(ts, 2018, 0)
    for k in range(W):
        eng.run_steps(k % nb, 1, use_graph=False)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        barrier()
        e0.record()
        for k in range(K):
            eng.run_steps((W + k) % nb, 1, use_graph=False)
        e1.record()
        barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    # per-launch timing of the SpMMs of a step (event pairs; launch gaps are negligible next to ms-scale launches)
    spmm_ms = []
    orig = ops.spmm
    import arlib_b200.engine as engmod

    def timed_spmm(*a, **k):
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(); orig(*a, **k); a1.record()
        kind = ("row_masked" if (k.get("row_mask") is not None or k.get("worklist") is not None) else
                "col_masked" if k.get("col_mask") is not None else "full_with_adam" if k.get("adam") is not None else "full")
        spmm_ms.append((kind, a0, a1))
    engmod.ops.spmm = timed_spmm
    try:
        for k in range(min(K, 5)):
            eng.run_steps(k % nb, 1, use_graph=False)
    finally:
        engmod.ops.spmm = orig
    torch.cuda.synchronize()
    by_kind = {}
    for kind, a, b_ in spmm_ms:
        by_kind.setdefault(kind, []).append(a.elapsed_time(b_))
    full_ms = max_over_ranks(float(np.mean(by_kind["full"])))
    bar_us = None
    if comm is not None:
        for _ in range(5):
            comm.barrier()
        e0.record()
        for _ in range(50):
            comm.barrier()
        e1.record()
        torch.cuda.synchronize()
        bar_us = e0.elapsed_time(e1) / 50 * 1e3
    Tbytes = N * d * 4
    ln, lr_ = eng.g.local_nnz, eng.g.n_local_rows
    if eng.mode == "rows":
        b_spmm = ln * 8 + (lr_ + 1) * 4 + Tbytes + lr_ * d * 4
    elif eng.mode == "dshard":
        b_spmm = g.nnz * 8 + (N + 1) * 4 + 2 * N * eng.d * 4
    else:
        b_spmm = g.nnz * 8 + (N + 1) * 4 + 2 * Tbytes
    b_gather = ln * (8 + 4 * eng.d) + lr_ * eng.d * 4
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    line = {
        "metric": "LightGCN train triples/s", "value": K * B / (ms * 1e-3), "unit": "triples/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "scale stress: LightGCN %d-layer d=%d BPR batch %d, power-law graph %d users x %d items, %d edges "
                               "(alpha=%s), generated and indexed on the device" % (L, d, B, U, I, E, args.alpha),
                   "lr": LR, "reg": REG, "sampler": "device-philox over a 64-batch sample of the epoch",
                   "l2": "one table = %.1f GB >> the 126 MB L2: every launch streams from HBM" % (Tbytes / 1e9)},
        "roofline": {"kernel": "spmm_csr_kernel<%d>" % eng.d, "bound": "hbm", "achieved": b_spmm / (full_ms * 1e-3) / 1e9,
                     "peak": peak, "unit": "GB/s", "frac": b_spmm / (full_ms * 1e-3) / 1e9 / peak, "traffic": None,
                     "algorithmic_bytes_per_launch": b_spmm, "avg_launch_ms": full_ms,
                     "gather_model": {"bytes_per_launch": b_gather, "achieved": b_gather / (full_ms * 1e-3) / 1e9,
                                      "frac": b_gather / (full_ms * 1e-3) / 1e9 / peak,
                                      "note": "no-reuse model nnz*(8+4d)+T (SURVEY.md 8d): what HBM sees when the table does not "
                                              "fit L2 -- can exceed the contract figure's fraction by the L2 hit rate"},
                     "launch_ms": {k: float(np.mean(v)) for k, v in by_kind.items()}},
        "clocks": clk.summary(),
        "parallelism": eng.mode if world > 1 else "single GPU",
        "comm": None if world == 1 else {
            "layout": eng.mode,
            "all_gather_bytes_received_per_layer_per_rank": int((world - 1) / world * Tbytes) if eng.mode == "rows" else 0,
            "exchanges_per_step": 2 * L + 1 if eng.mode == "rows" else 1, "barrier_us": bar_us,
            "transport": "NVSwitch multimem.st from the SpMM epilogue" if eng.mode == "rows" and eng._mc.get("F") else
                         "NVLink P2P stores from the kernels"},
        "graph_build_s": t_build, "gpu_launches": K * eng.launches_per_step,
        "last_loss": float(eng.out4[(W + K - 1) % nb, 0]),
        "cpu_baseline": {"unavailable": "the reference's dict-of-dicts DataLoader (util/DataLoader.py:32-55) cannot hold "
                                        "%d edges; SURVEY.md 8d: reference not run at this shape" % E},
        "hbm_gb_allocated": torch.cuda.max_memory_allocated() / 1e9,
    }
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


def main():
    # everything (NCCL banners, library chatter) goes to stderr; the ONE JSON line goes to the real stdout
    global print
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    _print = print

    def print(*a, **k):          # noqa: A001 - rank-0 JSON line writer
        k.pop("flush", None)
        _print(*a, file=real_stdout, **k)
        real_stdout.flush()

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="gowalla", choices=sorted(WORKLOADS) + sorted(SCALE_SHAPES))
    ap.add_argument("--alpha", type=float, default=0.5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-epoch-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed training step and the last timed evaluation computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload in SCALE_SHAPES):
        ap.error("--dump-outputs needs --impl ours and a workload of %s" % ", ".join(sorted(WORKLOADS)))
    if args.workload in SCALE_SHAPES:
        if args.impl == "reference":
            if int(os.environ.get("RANK", "0")) == 0:
                print(json.dumps({"impl": "reference", "unavailable": "the reference cannot load this shape (SURVEY.md 8d)"}))
            return
        run_scale_stress(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
