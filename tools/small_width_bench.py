"""Times the LightGCN training step (CUDA graph replay) and the full-rank evaluation at the Gowalla shape for
d in {8, 16, 32, 64}, and the three stage-1 candidates of the top-K at d = 8 and 16:

  fp32    the CUDA-core group-max GEMM (impl 0)
  tc      tcgen05 at K = d: 32- / 64-byte-swizzled TMA tiles, one or two MMAs per tile (impl 1)
  pad32   both tables zero-padded to 32 columns and fed to the d = 32 tcgen05 kernel (the copy timed apart)

    python tools/small_width_bench.py [--steps 300] [--evals 20]

Prints one line per measurement and the card's name and power limit first."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import scipy.sparse as sp
import torch

from bench import LR, REG, make_data, xavier_tables
from arlib_b200 import ops
from arlib_b200.engine import DeviceTrainSet, LightGCNEngine
from arlib_b200.evaluator import FullRankEvaluator
from arlib_b200.graph import DeviceGraph


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def timed(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--evals", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    print("card: %s" % card(), flush=True)
    D = make_data("gowalla", 0.5)
    U, I, E, L, B = D["U"], D["I"], D["E"], D["L"], D["B"]
    N = U + I
    half = sp.csr_matrix((np.ones(E, dtype=np.float32), (D["tu"], D["ti"] + U)), shape=(N, N), dtype=np.float32)
    g = DeviceGraph.from_dataloader_adj(half + half.T, dev)
    ts = DeviceTrainSet.from_arrays(D["tu"], D["ti"], U, I, dev)
    ev = FullRankEvaluator.from_arrays(U, I, D["tu"], D["ti"], D["su"], D["si"], dev)
    n_eval = ev.user_rows.numel()
    steps = min(args.steps, E // B)
    for d in (8, 16, 32, 64):
        ue, ie = xavier_tables(U, I, d)
        eng = LightGCNEngine(g, torch.cat([ue, ie]).to(dev), U, L, LR, REG, B, E)
        eng.sample_epoch(ts, 2018, 0)
        for k in range(3):
            eng.run_steps(k, 1, use_graph=False)
        eng.run_steps(0, steps, use_graph=True)                     # capture + one replay
        ms = timed(lambda: eng.run_steps(0, steps, use_graph=True), 3, warm=1) / steps
        print("d=%-3d train step (graph replay, %d steps, L=%d, B=%d): %.4f ms/step, %.2f M triples/s"
              % (d, steps, L, B, ms, B / ms / 1e3), flush=True)
        F = eng.forward_table().clone()
        uf, itf = F[:U].contiguous(), F[U:].contiguous()
        ms = timed(lambda: ev.topk(uf, itf, 50), args.evals)
        print("d=%-3d evaluation (top-50, %d users x %d items, default stage 1): %.3f ms" % (d, n_eval, I, ms), flush=True)
        if d >= 32:
            continue
        rows = ev.user_rows
        mk = dict(user_rows=rows, mask_rowptr=ev.mask_rowptr, mask_items=ev.mask_items, want_output=False)
        ws = {}
        pad = lambda x: torch.nn.functional.pad(x, (0, 32 - d)).contiguous()
        up, ip = pad(uf), pad(itf)
        for name, impl, a, b in (("fp32", 0, uf, itf), ("tc", 1, uf, itf), ("pad32", 1, up, ip)):
            need = int(ops._lib.load().agcf_score_topk_ws_bytes(n_eval, I, a.shape[1], 50))
            ws[name] = torch.empty(need, dtype=torch.uint8, device=dev)
            s1 = timed(lambda: ops.score_group_max(a, b, impl=impl, ws=ws[name], **mk), args.evals)
            full = timed(lambda: ops.score_topk(a, b, 50, user_rows=rows, mask_rowptr=ev.mask_rowptr,
                                                mask_items=ev.mask_items, impl=impl, ws=ws[name]), args.evals)
            print("d=%-3d stage 1 %-5s: %.3f ms (stage 0 + 1); whole top-K %.3f ms" % (d, name, s1, full), flush=True)
        cp = timed(lambda: (pad(uf), pad(itf)), args.evals)
        print("d=%-3d pad32 copy of both tables: %.3f ms" % (d, cp), flush=True)
        # stage-1 error of the TF32 candidates against the exact fp32 group maxima, over the documented bound
        ex = ops.score_group_max(uf, itf, impl=0, **dict(mk, want_output=True))
        bound = 1.01 * 2.0 ** -9 * uf[rows.long()].norm(dim=1, keepdim=True) * itf.norm(dim=1).max()
        for name, a, b in (("tc", uf, itf), ("pad32", up, ip)):
            got = ops.score_group_max(a, b, impl=1, **dict(mk, want_output=True))
            fin = ex > -1e8
            r = ((got - ex).abs() / bound)[fin].max().item()
            print("d=%-3d stage 1 %-5s: max |error| / delta = %.3g" % (d, name, r), flush=True)


if __name__ == "__main__":
    main()
