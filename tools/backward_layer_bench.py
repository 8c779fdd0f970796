"""Time the middle backward layer of the LightGCN training step (Y = A H + G) the way the step runs it: on the engine's
own tables, G non-zero at one batch's rows only, and -- where the build has it -- G read only at the batch's rows
(addend_mask).  bench.py's avg_launch_ms times this layer without the batch bitmap, so it cannot show that change.
One JSON line: mean us per launch over 200 back-to-back launches, per batch, for a few batches.

    python tools/backward_layer_bench.py [workload]"""
import inspect, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, scipy.sparse as sp, torch

from bench import LR, REG, make_data, xavier_tables
from arlib_b200 import ops
from arlib_b200.engine import DeviceTrainSet, LightGCNEngine
from arlib_b200.graph import DeviceGraph

name = sys.argv[1] if len(sys.argv) > 1 else "gowalla"
dev = torch.device("cuda", 0)
D = make_data(name, 0.5)
U, I, E, L, d, B = D["U"], D["I"], D["E"], D["L"], D["d"], D["B"]
N = U + I
half = sp.csr_matrix((np.ones(E, dtype=np.float32), (D["tu"], D["ti"] + U)), shape=(N, N), dtype=np.float32)
g = DeviceGraph.from_dataloader_adj(half + half.T, dev)
ue, ie = xavier_tables(U, I, d)
eng = LightGCNEngine(g, torch.cat([ue, ie]).to(dev), U, L, LR, REG, B, E)
eng.sample_epoch(DeviceTrainSet.from_arrays(D["tu"], D["ti"], U, I, dev), 2018, 0)
if L < 2:
    raise SystemExit("no middle backward layer at L = %d" % L)
masked = "addend_mask" in inspect.signature(ops.spmm).parameters
H, Y = eng.bw[L % 2], eng.bw[(L - 1) % 2]
gen = torch.Generator(device=dev).manual_seed(1)
H.copy_(torch.randn(N, d, device=dev, generator=gen))
res = []
for b in (0, 1, 2, 3):
    rows = eng.seg_node[b * 3 * B:b * 3 * B + int(eng.n_seg[b])].long()
    eng.G.zero_()
    eng.G[rows] = torch.randn(rows.numel(), d, device=dev, generator=gen)
    kw = {"addend_mask": eng.node_mask[b * eng.mask_words:]} if masked else {}
    fn = lambda: ops.spmm(eng.g, H, Y=Y, addend=eng.G, **kw)
    for _ in range(20):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(200):
        fn()
    e1.record()
    torch.cuda.synchronize()
    res.append(e0.elapsed_time(e1) / 200 * 1e3)
eng.G.zero_()
print(json.dumps({"workload": name, "launch": "middle backward layer", "addend_mask": masked,
                  "batch_rows_frac": float(eng.n_seg[:4].float().mean()) / N, "us_per_launch": res,
                  "us_mean": float(np.mean(res)), "gpu": torch.cuda.get_device_name(0)}))
