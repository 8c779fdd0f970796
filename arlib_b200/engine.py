"""Fused LightGCN BPR training engine: the body of LightGCN.train()
(recommender/LightGCN.py:46-64) as a fixed sequence of agcf kernels per batch,
replayed from a CUDA graph.

per step (L layers): L x spmm (forward, layer-mean fused) -> bpr_forward ->
bpr_backward (atomic-free rows of G) -> L x spmm (backward, A^T = A) -> zero_rows ->
adam -> step counter            = 2L + 5 kernel launches, no host sync.

per epoch: one Philox sampling launch (all E triples) + one grouping launch (all
batches), then the step graph(s).
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import ops
from .graph import DeviceGraph


def dshard_columns(d, world, rank):
    """Column range [c0, c1) of rank ``rank`` when d columns are split over ``world`` ranks; the slice
    width must be one the row kernels are compiled for."""
    if d % world:
        raise ValueError("embedding size %d is not divisible by %d ranks" % (d, world))
    w = d // world
    if w not in (8, 16, 32, 64, 128, 256):
        raise ValueError("d/P = %d: the row kernels take slices of 8, 16, 32, 64, 128 or 256 columns" % w)
    return rank * w, (rank + 1) * w


def grid_shape(grid, world):
    """(R, C) of the grid layout on ``world`` ranks: R row blocks x C column slices, R >= 2, C >= 2, R * C = world
    ((P, 1) and (1, P) are the modes "rows" and "dshard")."""
    try:
        R, C = (int(x) for x in grid)
    except (TypeError, ValueError):
        raise ValueError("grid must be a pair (R, C) of row blocks and column slices, got %r" % (grid,)) from None
    if R < 2 or C < 2:
        raise ValueError("grid (%d, %d): R >= 2 row blocks and C >= 2 column slices (a single row block is mode "
                         "'dshard', a single column slice mode 'rows')" % (R, C))
    if R * C != world:
        raise ValueError("grid (%d, %d): R * C = %d ranks, the process group has %d" % (R, C, R * C, world))
    return R, C


def grid_groups(R, C, rank):
    """Rank r * C + c of the grid owns row block r and column slice c.  Returns (r, c, column group, row group): the
    column group is the R ranks with slice c (they exchange layer rows), the row group the C ranks with block r (they
    exchange the loss's partial scores)."""
    r, c = divmod(rank, C)
    return r, c, [q * C + c for q in range(R)], [r * C + q for q in range(C)]


class DeviceTrainSet:
    """Device mirror of what util/sampler.py:4-30 reads from ``data``: the edge list
    (data.training_data through data.user / data.item) and, per user, the sorted item
    ids of data.training_set_u[user] (the rejection set; users without an entry --
    injected fake users, SURVEY.md App. B -- reject nothing)."""

    def __init__(self, data, device):
        edges = getattr(data, 'pristine_edges', lambda: None)()
        if edges is not None:              # untouched since the vectorised load: the dicts ARE these edges
            other = DeviceTrainSet.from_arrays(edges[0], edges[1], data.user_num, data.item_num, device)
            self.__dict__.update(other.__dict__)
            return
        n = len(data.training_data)
        user, item = data.user, data.item
        eu = np.fromiter((user[r[0]] for r in data.training_data), dtype=np.int32, count=n)
        ei = np.fromiter((item[r[1]] for r in data.training_data), dtype=np.int32, count=n)
        n_users = max(data.user_num, int(eu.max()) + 1 if n else 0)
        counts = np.zeros(n_users, dtype=np.int64)
        chunks = []
        tsu = data.training_set_u
        for name, uid in user.items():
            if uid < n_users and name in tsu:
                ids = np.fromiter((item[i] for i in tsu[name] if i in item), dtype=np.int32)
                ids.sort()
                counts[uid] = ids.shape[0]
                chunks.append((uid, ids))
        rowptr = np.zeros(n_users + 1, dtype=np.int64)
        np.cumsum(counts, out=rowptr[1:])
        items = np.zeros(max(int(rowptr[-1]), 1), dtype=np.int32)
        for uid, ids in chunks:
            items[rowptr[uid]:rowptr[uid + 1]] = ids
        self.n_edges, self.n_users, self.n_items = n, n_users, data.item_num
        self.e_user = torch.from_numpy(eu).to(device)
        self.e_item = torch.from_numpy(ei).to(device)
        self.rej_rowptr = torch.from_numpy(rowptr.astype(np.int32)).to(device)
        self.rej_items = torch.from_numpy(items).to(device)

    @classmethod
    def from_arrays(cls, e_user, e_item, n_users, n_items, device):
        """Directly from integer edge arrays (benchmark / tests): rejection set = the
        user's own train items."""
        self = cls.__new__(cls)
        eu = np.asarray(e_user, dtype=np.int32)
        ei = np.asarray(e_item, dtype=np.int32)
        order = np.lexsort((ei, eu))
        su, si = eu[order], ei[order]
        keep = np.ones(su.shape[0], dtype=bool)
        keep[1:] = (su[1:] != su[:-1]) | (si[1:] != si[:-1])
        su, si = su[keep], si[keep]
        rowptr = np.zeros(n_users + 1, dtype=np.int64)
        np.cumsum(np.bincount(su, minlength=n_users), out=rowptr[1:])
        self.n_edges, self.n_users, self.n_items = eu.shape[0], n_users, n_items
        self.e_user = torch.from_numpy(eu).to(device)
        self.e_item = torch.from_numpy(ei).to(device)
        self.rej_rowptr = torch.from_numpy(rowptr.astype(np.int32)).to(device)
        self.rej_items = torch.from_numpy(si if si.size else np.zeros(1, np.int32)).to(device)
        return self


    @classmethod
    def from_graph(cls, graph, n_users, n_items, epoch_edges=None, seed=0):
        """From the device adjacency itself (no host pass over the edges; the 10 M x 1 M scale-stress shape): the
        rejection lists ARE the user rows of the canonical CSR (sorted item columns minus the user offset); the
        positives of an "epoch" are all user -> item non-zeros, or a uniform sample of ``epoch_edges`` of them (a full
        epoch of a 200 M-edge graph is 97 657 full-graph steps -- SURVEY.md 8d reports per-step numbers there)."""
        self = cls.__new__(cls)
        dev = graph.rowptr.device
        U = int(n_users)
        n_ui = int(graph.rowptr[U])                                  # non-zeros of the user rows = E
        rowptr_u = graph.rowptr[:U + 1].contiguous()
        items = (graph.col[:n_ui] - U).contiguous()
        if epoch_edges is None or epoch_edges >= n_ui:
            pos = torch.arange(n_ui, device=dev)
        else:
            g = torch.Generator(device=dev).manual_seed(seed)
            pos = torch.randint(0, n_ui, (int(epoch_edges),), generator=g, device=dev)
        e_user = (torch.searchsorted(rowptr_u.long(), pos, right=True) - 1).to(torch.int32)
        self.n_edges, self.n_users, self.n_items = int(pos.numel()), U, int(n_items)
        self.e_user = e_user.contiguous()
        self.e_item = items[pos].contiguous()
        self.rej_rowptr = rowptr_u
        self.rej_items = items if items.numel() else torch.zeros(1, dtype=torch.int32, device=dev)
        return self


class LightGCNEngine:
    """``mode`` (multi-GPU only, SURVEY.md 8e):
      "rows"   -- node rows and adjacency rows partitioned; every layer's rows are all-gathered by the SpMM
                  epilogue (P2P stores) and closed by a barrier: 2L + 1 exchanges per step;
      "dshard" -- the graph is replicated and every table is COLUMN-sharded (rank r owns columns
                  [r*d/P, (r+1)*d/P)): propagation, backward and Adam need no communication at all, the
                  only exchange of a step is 32 bytes per triple per peer (the partial scores, each value
                  stamped with the step so that the consumer needs no barrier).  Needs d/P in {8, 16, 32, ...}
                  and the graph to fit on one GPU;
      "grid"   -- ``grid=(R, C)``: rank r*C + c owns row block r and column slice c.  Inside each column group (the R
                  ranks of slice c) the step is the "rows" step on [N, d/C] tables, each layer closed by a hand-off
                  among those R ranks (agcf_group_handoff) instead of an all-rank barrier; inside each row group (the
                  C ranks of block r) the loss is the "dshard" exchange.  Tables are N x d/C per GPU."""

    def __init__(self, graph: DeviceGraph, table: torch.Tensor, n_users: int, n_layers: int,
                 lr: float, reg: float, batch_size: int, max_triples: int,
                 betas=(0.9, 0.999), adam_eps=1e-8, sparse_layers=True, comm=None, mode="rows", grid=None):
        if 3 * batch_size > 16384:
            raise ValueError("batch_size %d too large for the single-CTA batch grouping (max 5461)" % batch_size)
        if n_layers < 1:
            raise ValueError("n_layers must be >= 1")
        if mode not in ("rows", "dshard", "grid"):
            raise ValueError("mode must be 'rows', 'dshard' or 'grid'")
        if mode == "grid":
            grid_shape(grid, comm.world if comm is not None else 1)
        self.N, self.d_full = table.shape
        self.d = self.d_full
        self.U, self.L = int(n_users), int(n_layers)
        self.lr, self.reg, self.B = float(lr), float(reg), int(batch_size)
        self.betas, self.adam_eps = betas, adam_eps
        dev = table.device
        self.comm = comm
        self.mode = mode if (comm is not None and comm.world > 1) else "single"
        f = lambda: torch.empty_like(table)
        # forward layers 1 .. L-1 of a training step keep their tables E_1 .. E_{L-1} (fw[k - 1]) for the last layer,
        # which forms the layer sum at the batch's rows (_forward_batch).  Once it has, they are dead: the backward layers
        # run in them (bw), so that the step's full tables -- E0, two layer tables, m, v -- and the graph fit in L2
        n_fw = max(2, self.L - 1) if self.L > 1 else 0
        if self.mode == "single":
            self.comm = None
            self.g, self.E0 = graph.planned_for(self.d), table
            self.r0, self.r1 = 0, self.N
            self.F = f()
            self.fw = [f() for _ in range(n_fw)]
            self.bw = [self.fw[1], self.fw[0]] if self.L > 1 else []
        elif self.mode == "dshard":
            c0, c1 = dshard_columns(self.d_full, comm.world, comm.rank)
            self.d = c1 - c0
            self.col0, self.col1 = c0, c1
            self.g = graph.planned_for(self.d)                         # narrow slices want short segments (graph.py)
            self.r0, self.r1 = 0, self.N
            self.E0 = table[:, c0:c1].contiguous()
            table = self.E0                      # every per-step table below has the slice's shape
            f = lambda: torch.empty_like(self.E0)
            self.F = f()
            self.fw = [f() for _ in range(n_fw)]
            self.bw = [self.fw[1], self.fw[0]] if self.L > 1 else []
            # exchange buffer of the partial scores: one symmetric allocation, every rank writes its slot everywhere
            nbytes = ops.bpr_xchg_bytes(self.B)
            bufs = comm.allocate({"xchg": ((nbytes,), torch.uint8)})
            self.xchg = bufs["xchg"]
            self.xchg.zero_()
            # the exchange's own counter (stamps / parity of the words): advanced by bpr_finish, NEVER restored with the
            # optimizer state -- a stamp is used once
            self.xchg_ctr = torch.zeros(1, dtype=torch.int32, device=dev)
            self._xchg_all = comm.all_ptrs("xchg")
            self.xchg_rank = comm.rank
            torch.cuda.synchronize()
            comm.barrier()
        elif self.mode == "grid":
            R, C = grid_shape(grid, comm.world)
            self.grid = (R, C)
            self.grid_r, self.grid_c, self.col_group, self.row_group = grid_groups(R, C, comm.rank)
            c0, c1 = dshard_columns(self.d_full, C, self.grid_c)
            self.d = c1 - c0
            self.col0, self.col1 = c0, c1
            self.bounds = self._row_ranges(graph, R)
            self.r0, self.r1 = self.bounds[self.grid_r], self.bounds[self.grid_r + 1]
            self.g = graph.partition(self.r0, self.r1).planned_for(self.d)
            specs = self._symmetric_tables(R)
            tables = list(specs)
            specs["xchg"] = ((ops.bpr_xchg_bytes(self.B),), torch.uint8)
            specs["handoff"] = ((8,), torch.int32)
            bufs = comm.allocate(specs)
            self.sym = bufs
            self.E0 = bufs["E0"]
            self.E0.copy_(table[:, c0:c1])
            table = self.E0
            f = lambda: torch.empty_like(self.E0)
            self.F = bufs["F"]
            self.fw = [bufs[k] for k in ("fw0", "fw1") if k in bufs]
            self.bw = [bufs[k] for k in ("bw0", "bw1") if k in bufs]
            # layer rows go to the column group's partners (no multicast: a multicast object spans every rank)
            self._peer = {k: comm.peers(k, ranks=self.col_group) for k in tables}
            self._peer_E0_rows = comm.peers("E0", self.r0 * self.d * 4, ranks=self.col_group)
            self._mc = {k: 0 for k in tables}
            self._mc_E0_rows = 0
            # the loss's partial scores go to the row group (bpr_partial / bpr_finish with group rank and pointers)
            self.xchg = bufs["xchg"]
            self.xchg.zero_()
            self.xchg_ctr = torch.zeros(1, dtype=torch.int32, device=dev)
            self._xchg_all = comm.all_ptrs("xchg", ranks=self.row_group)
            self.xchg_rank = self.grid_c
            # column-group hand-off: flag words (slot = position in the group), its own stamp counter, never restored
            self.handoff_flags = bufs["handoff"]
            self.handoff_flags.zero_()
            self._handoff_peers = comm.peers("handoff", ranks=self.col_group)
            self.handoff_ctr = torch.zeros(1, dtype=torch.int32, device=dev)
            self.handoff_err = torch.zeros(1, dtype=torch.int32, device=dev)
            self.row_pg = comm.subgroups([grid_groups(R, C, q * C)[3] for q in range(R)])
            torch.cuda.synchronize()
            comm.barrier()
        else:
            # row partition: this rank computes rows [r0, r1); the tables peers write live in one symmetric arena
            bounds = self._row_ranges(graph, comm.world)
            self.bounds = bounds
            self.r0, self.r1 = bounds[comm.rank], bounds[comm.rank + 1]
            self.g = graph.partition(self.r0, self.r1)
            specs = self._symmetric_tables(comm.world)
            bufs = comm.allocate(specs)
            self.sym = bufs
            self.E0 = bufs["E0"]
            self.E0.copy_(table)
            self.F = bufs["F"]
            self.fw = [bufs[k] for k in ("fw0", "fw1") if k in bufs]
            self.bw = [bufs[k] for k in ("bw0", "bw1") if k in bufs]
            row_off = self.r0 * self.d * 4
            self._peer = {k: comm.peers(k) for k in specs}
            self._peer_E0_rows = comm.peers("E0", row_off)
            # NVSwitch multicast mappings of the same buffers (0 when unavailable): one store reaches all copies
            self._mc = {k: comm.multicast_ptr(k) for k in specs}
            self._mc_E0_rows = comm.multicast_ptr("E0", row_off)
            torch.cuda.synchronize()
            comm.barrier()
        self.G = torch.zeros_like(table)
        self.dE0 = f()
        self.m = torch.zeros_like(table)
        self.v = torch.zeros_like(table)
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        # side stream of the step-counter / Adam-coefficient kernel (_fork_coefs); ARLIB_B200_COEF_STREAM=0: in line
        self._coef_stream = torch.cuda.Stream(device=dev) if os.environ.get("ARLIB_B200_COEF_STREAM", "1") == "1" else None
        self._coefs_forked = False
        self.T = 0
        self.cap = int(max_triples)
        nbmax = (self.cap + self.B - 1) // self.B
        i32 = lambda n: torch.empty(max(n, 1), dtype=torch.int32, device=dev)
        self.tu, self.ti, self.tj = i32(self.cap), i32(self.cap), i32(self.cap)
        self.occ = i32(nbmax * 3 * self.B)
        self.seg_off = i32(nbmax * (3 * self.B + 1))
        self.seg_node = i32(nbmax * 3 * self.B)
        self.n_seg = i32(nbmax)
        # per-batch node bitmaps drive the batch-sparse layers (last forward layer only computes the batch's
        # rows, first backward layer only gathers the batch's gradient rows); skipped if they would be huge
        self.mask_words = (self.N + 31) // 32
        self.sparse_layers = bool(sparse_layers) and nbmax * self.mask_words * 4 <= (1 << 29)
        self.node_mask = i32(nbmax * self.mask_words) if self.sparse_layers else None
        import os as _os
        flag = lambda name, default="1": _os.environ.get(name, default) == "1"
        # per-batch work lists: the last forward layer runs the batch's own plan (its <= 3B rows cut into short
        # segments) instead of testing every item of the static plan against the bitmap
        self.wl = None
        # narrow slices: shorter items (graph.default_segment); ARLIB_B200_WL_SEGMENT overrides
        self.wl_segment = self.WL_SEGMENT if (_os.environ.get('ARLIB_B200_WL_SEGMENT') or self.d > 8) else 32
        if self.sparse_layers and flag("ARLIB_B200_WORKLISTS"):
            self._init_worklists(nbmax, dev)
        # Adam fused into the epilogue of the last backward SpMM (own rows == all rows: not in "rows" mode,
        # where the updated rows also go to the peers)
        self.fuse_adam = self.mode not in ("rows", "grid") and flag("ARLIB_B200_FUSE_ADAM")
        self.adam_coefs = torch.zeros(2, dtype=torch.float32, device=dev)
        self.out4 = torch.zeros((nbmax, 4), dtype=torch.float32, device=dev)
        self.coef = torch.empty(self.B, dtype=torch.float32, device=dev)
        self.ws = torch.zeros(ops.bpr_ws_bytes(self.B), dtype=torch.uint8, device=dev)
        self._graphs = {}
        self._ext = None
        self._loss_eager = None
        self.dist_graphs = _os.environ.get("ARLIB_B200_DIST_GRAPHS", "1") == "1"
        self.launches_per_step = {"single": 2 * self.L + 5, "rows": 4 * self.L + 5, "dshard": 2 * self.L + 6,
                                  "grid": 4 * self.L + 6}[self.mode]
        if self.fuse_adam:       # no adam kernel; no zero_rows kernel either when the last backward layer re-zeroes G
            self.launches_per_step -= 2 if self.L > 1 else 1
        self._refresh_adam_coefs()

    WL_SEGMENT = int(__import__('os').environ.get('ARLIB_B200_WL_SEGMENT', '64'))

    def _row_ranges(self, graph, world):
        """row boundaries of the row-partitioned layout: the step is a chain of SpMMs, whose time follows the nnz"""
        return graph.row_ranges(world)

    def _symmetric_tables(self, world):
        """{name: (shape, dtype)} of the row-partitioned layout's symmetric arena: the tables peers store into"""
        return {k: ((self.N, self.d), torch.float32) for k in ("E0", "F", "fw0", "fw1", "bw0", "bw1")}

    def _init_worklists(self, nbmax, dev):
        """Capacity of a batch's work list = the 3B rows with the most segments (an upper bound for any batch)."""
        g = self.g
        rp = g.rowptr.long()
        deg = rp[g.r0 + 1:g.r1 + 1] - rp[g.r0:g.r1]
        seg = self.wl_segment
        nseg = torch.where(deg > seg, (deg + seg - 1) // seg, torch.ones_like(deg))
        if nseg.numel() == 0 or int(nseg.max()) >= (1 << 15):
            return
        top = torch.topk(nseg, min(3 * self.B, nseg.numel())).values
        cap = (int(top.sum()) + 63) // 64 * 64
        if nbmax * cap * 20 > (1 << 30):
            return
        i32 = lambda *shape: torch.zeros(shape, dtype=torch.int32, device=dev)
        self.wl = {"vrows": i32(nbmax, cap, 4), "vpart": i32(nbmax, cap), "count": i32(nbmax), "cap": cap,
                   "partial": torch.empty((cap, self.d), dtype=torch.float32, device=dev), "tickets": i32(cap)}

    def _worklist(self, b):
        w = self.wl
        return None if w is None else (w["vrows"][b], w["vpart"][b], w["count"][b:b + 1], w["partial"], w["tickets"])

    def _fork_coefs(self):
        """Step counter + 1 and the NEXT step's Adam coefficients on a side stream (a parallel branch of a captured
        graph): the one-thread kernel only has to be done before the next step's LAST launch, so the next step's
        propagation does not queue behind it (3.7 us + a launch boundary per step on the main chain otherwise)."""
        if self._coef_stream is None:
            ops.adam_coefs(self.step_dev, self.adam_coefs, self.lr, self.betas[0], self.betas[1], increment=True)
            return
        cur = torch.cuda.current_stream()
        self._coef_stream.wait_stream(cur)          # after this step's Adam launch has read the coefficients
        with torch.cuda.stream(self._coef_stream):
            ops.adam_coefs(self.step_dev, self.adam_coefs, self.lr, self.betas[0], self.betas[1], increment=True)
        self._coefs_forked = True

    def _join_coefs(self):
        if self._coefs_forked:
            torch.cuda.current_stream().wait_stream(self._coef_stream)
            self._coefs_forked = False

    def _refresh_adam_coefs(self):
        """coefs of the NEXT step from the device step counter (after construction / a restore of step_dev)"""
        ops.adam_coefs(self.step_dev, self.adam_coefs, self.lr, self.betas[0], self.betas[1], increment=False)

    def _peers(self, name):
        return self._peer[name] if self.mode in ("rows", "grid") else None

    def _mcast(self, name):
        return self._mc[name] if self.mode == "rows" else 0

    def _barrier(self):
        if self.mode == "rows":
            self.comm.barrier()
        elif self.mode == "grid":
            ops.group_handoff(self.handoff_flags, self._handoff_peers, self.grid_r, self.handoff_ctr, self.handoff_err)

    def check_handoff(self):
        """Grid layout: wait for the device and raise if a column-group hand-off gave up on a partner (4 s without
        its stamp: a rank that crashed or issued another launch sequence); the tables are then not to be trusted."""
        if self.mode == "grid":
            torch.cuda.current_stream().synchronize()
            if int(self.handoff_err.item()):
                raise RuntimeError("grid layout: rank %d waited 4 s for a column-group partner in a hand-off; the "
                                   "training state is inconsistent" % self.comm.rank)

    def full_table(self, local: torch.Tensor) -> torch.Tensor:
        """[N, d] table from this rank's copy: identity except in "dshard" mode, where the P column
        slices are all-gathered (NCCL) and interleaved back, and in "grid" mode, where the C slices of the
        row group are -- used once per evaluation / export, never inside a training step."""
        if self.mode not in ("dshard", "grid"):
            return local
        import torch.distributed as dist
        if self.mode == "dshard":
            w, group = self.comm.world, self.comm.group
        else:
            self.check_handoff()
            w, group = self.grid[1], self.row_pg
        parts = torch.empty((w * local.shape[0], local.shape[1]), dtype=local.dtype, device=local.device)
        dist.all_gather_into_tensor(parts, local.contiguous(), group=group)
        return parts.view(w, self.N, -1).permute(1, 0, 2).reshape(self.N, self.d_full).contiguous()

    # ------------------------------------------------------------ epoch set-up
    @property
    def n_batches(self):
        return (self.T + self.B - 1) // self.B

    def sample_epoch(self, ts: DeviceTrainSet, seed: int, epoch: int):
        """Philox on-device sampling of one epoch (replaces util/sampler.py:4-30)."""
        if ts.n_edges > self.cap:
            raise ValueError("engine capacity %d < %d edges" % (self.cap, ts.n_edges))
        ops.bpr_sample_epoch(ts.e_user, ts.e_item, ts.rej_rowptr, ts.rej_items, ts.n_items, seed, epoch,
                             self.tu, self.ti, self.tj)
        self.T = ts.n_edges
        self._group(0, self.T)

    def set_triples(self, u, i, j):
        """External triples for the whole epoch (device int32 tensors or host arrays)."""
        n = len(u)
        if n > self.cap:
            raise ValueError("engine capacity %d < %d triples" % (self.cap, n))
        for dst, src in ((self.tu, u), (self.ti, i), (self.tj, j)):
            src = torch.as_tensor(src, dtype=torch.int32)
            dst[:n].copy_(src, non_blocking=True)
        self.T = n
        self._group(0, n)

    def _group(self, first_triple, n):
        b0 = first_triple // self.B
        ops.bpr_group_batches(self.tu[first_triple:], self.ti[first_triple:], self.tj[first_triple:], n, self.B, self.U,
                              self.occ[b0 * 3 * self.B:], self.seg_off[b0 * (3 * self.B + 1):],
                              self.seg_node[b0 * 3 * self.B:], self.n_seg[b0:], self.N,
                              None if self.node_mask is None else self.node_mask[b0 * self.mask_words:])
        if self.wl is not None and n > 0:
            nb = (n + self.B - 1) // self.B
            w = self.wl
            ops.spmm_batch_worklists(self.seg_node[b0 * 3 * self.B:], self.n_seg[b0:], nb, 3 * self.B, self.g.rowptr,
                                     self.g.r0, self.g.r1, self.wl_segment, self.wl_segment,
                                     w["vrows"][b0:], w["vpart"][b0:], w["count"][b0:])

    # --------------------------------------------------------------- one step
    def forward_table(self, out=None, row_mask=None, worklist=None):
        """F = mean_k A^k E0 into self.F (or ``out``): the encoder forward alone
        (recommender/LightGCN.py:230-240), e.g. for the end-of-epoch embeddings.  With
        ``row_mask`` the LAST layer only computes (and F is only valid on) the masked rows.
        Multi-GPU: every layer's rows are also stored into the peers' tables by the SpMM
        epilogue and a barrier closes the layer (``out`` must then be self.F)."""
        F = self.F if out is None else out
        if self.mode in ("rows", "grid") and out is not None:
            raise ValueError("row-partitioned forward writes the symmetric F table")
        x = self.E0
        for k in range(1, self.L + 1):
            last = k == self.L
            name = "fw%d" % ((k - 1) % 2)
            y = None if last else self.fw[(k - 1) % 2]
            wl = worklist if last else None
            ops.spmm(self.g, x, Y=y, acc_in=self.E0 if k == 1 else F, acc_out=F,
                     acc_div=float(self.L + 1) if last else 1.0, row_mask=row_mask if (last and wl is None) else None,
                     peer_Y=None if last else self._peers(name), peer_acc=self._peers("F") if last else None,
                     mc_Y=0 if last else self._mcast(name), mc_acc=self._mcast("F") if last else 0,
                     worklist=wl)
            self._barrier()
            x = y
        return F

    def _forward_batch(self, row_mask, worklist):
        """The training step's forward: F = mean_k A^k E0 at the batch's rows only (row_mask / worklist).  Layers
        1 .. L-1 write only E_k; the last layer's epilogue forms ((E0 + E1) + ... + E_{L-1} + t) / (L + 1), the same
        adds in the same order as the running sum of forward_table, so F is bit-identical on those rows.  The
        row-partitioned layout (whose layers also go to the peers) and more than 8 layers keep forward_table."""
        if self.mode in ("rows", "grid") or self.L > 8:
            return self.forward_table(row_mask=row_mask, worklist=worklist)
        x = self.E0
        for k in range(1, self.L):
            ops.spmm(self.g, x, Y=self.fw[k - 1])
            x = self.fw[k - 1]
        ops.spmm(self.g, x, acc_out=self.F, acc_div=float(self.L + 1), acc_terms=[self.E0] + self.fw[:self.L - 1],
                 row_mask=row_mask if worklist is None else None, worklist=worklist)
        return self.F

    def _launch_step(self, b):
        B, L = self.B, self.L
        t0 = b * B
        nb = min(B, self.T - t0)
        u, i, j = self.tu[t0:], self.ti[t0:], self.tj[t0:]
        occ = self.occ[b * 3 * B:]
        seg_off = self.seg_off[b * (3 * B + 1):]
        seg_node = self.seg_node[b * 3 * B:]
        n_seg = self.n_seg[b:]
        out4 = self.out4[b]
        mask = self.node_mask[b * self.mask_words:] if self.sparse_layers else None
        if mask is not None:
            F = self._forward_batch(mask, self._worklist(b))
        else:
            F = self.forward_table()
        if self.mode in ("dshard", "grid"):
            # the step's only exchange: 32 B per triple to every peer, stamped with the step -- bpr_finish spins on
            # the words it needs, no barrier launch (csrc/bpr.cu).  Grid: among the row group's C column slices
            ops.bpr_partial(F, u, i, j, nb, self.U, self.xchg_rank, self.B, self.xchg_ctr, self._xchg_all)
            ops.bpr_finish(self.xchg, len(self._xchg_all), self.B, nb, self.reg, self.xchg_ctr, out4, self.coef, self.ws)
        else:
            ops.bpr_forward(F, u, i, j, nb, self.U, self.reg, out4, self.coef, self.ws)
        ops.bpr_backward(F, u, i, j, nb, self.U, self.reg, 1.0, out4, self.coef, occ, seg_off, seg_node, n_seg, self.G)
        H = self.G
        # G is non-zero only at the batch's rows: the backward layers read it (addend / acc_in) only there, and the fused
        # optimizer puts exactly those rows back to zero.  That pays where the batch covers few rows (Gowalla, 8 %: the
        # middle layer 43.2 -> 42.2 us); where it covers many, the bitmap load per work item costs more than the loads it
        # saves (ml-1m, 42 %: 37.1 -> 39.0 us), so graphs with fewer than 4 x 3B rows read G everywhere.  The
        # row-partitioned layout keeps the full reads too.
        g_mask = mask if self.mode not in ("rows", "grid") and 12 * self.B <= self.N else None
        # first backward layer: only the batch's gradient rows of H are non-zero.  The column-masked kernel skips the others
        # (27 vs 44 us at d = 64); on 8-column slices its extra bitmap round trip per chunk costs more than the zero rows it
        # avoids (26.4 vs 23.4 us, profiles/r2_summary.md section 5), so there the plain kernel gathers the zeros
        if mask is not None and self.d <= 8:
            mask = None
        for k in range(L, 0, -1):
            if k > 1:
                nxt = self.bw[k % 2]
                ops.spmm(self.g, H, Y=nxt, addend=self.G, col_mask=mask if k == L else None, addend_mask=g_mask,
                         peer_Y=self._peers("bw%d" % (k % 2)), mc_Y=self._mcast("bw%d" % (k % 2)))
                self._barrier()
                H = nxt
            elif self.fuse_adam:
                # dE0 = (G + A H) / (L + 1) never reaches memory: the epilogue applies Adam to the row and puts the
                # batch's rows of G back to zero (not when L == 1: G is then also the gathered operand)
                self._join_coefs()                  # this step's Adam coefficients (side branch of the previous step)
                ops.spmm(self.g, H, acc_in=self.G, acc_div=float(L + 1), col_mask=mask if k == L else None,
                         adam=(self.E0, self.m, self.v, self.adam_coefs, self.betas[0], self.betas[1], self.adam_eps),
                         zero_acc_in=L > 1, addend_mask=g_mask)
            else:
                ops.spmm(self.g, H, acc_in=self.G, acc_out=self.dE0, acc_div=float(L + 1),
                         col_mask=mask if k == L else None)
        if self.fuse_adam:
            if L == 1:
                ops.zero_rows(seg_node, n_seg, 3 * nb, self.G)
            self._fork_coefs()
            return
        ops.zero_rows(seg_node, n_seg, 3 * nb, self.G)
        # owner-computes: Adam on this rank's rows; the updated rows are stored into every peer's E0
        r0, r1 = self.r0, self.r1
        ops.adam_step(self.E0[r0:r1], self.dE0[r0:r1], self.m[r0:r1], self.v[r0:r1], self.lr, self.betas[0],
                      self.betas[1], self.adam_eps, step_dev=self.step_dev,
                      peer_p=self._peer_E0_rows if self.mode in ("rows", "grid") else None,
                      mc_p=self._mc_E0_rows if self.mode == "rows" else 0)
        ops.increment(self.step_dev)
        self._barrier()

    # ------------------------------------------------------------------ running
    def _trained_state(self):
        """the tensors a training step modifies (what a warm-up step before a graph capture has to put back)"""
        return [self.E0, self.m, self.v, self.step_dev]

    def _snapshot(self):
        return [t.clone() for t in self._trained_state()]

    def _restore(self, snap):
        for t, c in zip(self._trained_state(), snap):
            t.copy_(c)
        self._refresh_adam_coefs()

    def run_steps(self, first_batch=0, n_steps=None, use_graph=True):
        """Run batches [first_batch, first_batch + n_steps) of the current epoch.
        With use_graph the launch sequence is captured once per (first, n, T) and
        replayed.  Returns the [n_steps, 4] loss rows (device view)."""
        if n_steps is None:
            n_steps = self.n_batches - first_batch
        if first_batch + n_steps > self.n_batches:
            raise ValueError("not enough batches")
        if n_steps <= 0:
            return self.out4[0:0]
        if not use_graph or (self.comm is not None and not self.dist_graphs):
            for b in range(first_batch, first_batch + n_steps):
                self._launch_step(b)
            self._join_coefs()
        else:
            key = (first_batch, n_steps, self.T)
            g = self._graphs.get(key)
            if g is None:
                # warm-up outside capture is NOT needed for correctness of our kernels (no lazy
                # allocation), but the one-time cudaFuncSetAttribute of the grouping kernel and
                # module loading must not happen inside a capture: callers run sample_epoch /
                # set_triples (eager) before the first run_steps, which covers both.
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                state = self._snapshot()
                self._launch_step(first_batch)        # eager warm-up of every kernel in the step
                self._join_coefs()
                self._restore(state)
                torch.cuda.synchronize()
                self.check_handoff()
                with torch.cuda.graph(g):
                    for b in range(first_batch, first_batch + n_steps):
                        self._launch_step(b)
                    self._join_coefs()               # every branch of the capture ends in the capturing stream
                self._graphs[key] = g
                # capture does not execute: fall through to the replay below
            g.replay()
        return self.out4[first_batch:first_batch + n_steps]

    def step_external(self, host_triples: torch.Tensor, nb: int, use_graph=True):
        """One step on triples supplied by the HOST (int32 [3, >=nb], ideally pinned): H2D copy of the
        triples, grouping, the step kernels and the D2H copy of the 4-float loss row.  Returns the
        pinned host tensor the loss row lands in (valid after a stream synchronize / until the slot is
        reused ``n_slots`` calls later).

        With ``use_graph`` every staging slot owns two captured graphs: PREP (H2D memcpy nodes + the
        batch grouping, which depend on the triples only) runs on a side stream, STEP (propagation, loss,
        backward, Adam, D2H of the loss row) on the caller's stream after PREP's event.  Calls are
        asynchronous, so PREP of step k+1 overlaps STEP of step k: the single-CTA sort of the grouping
        and the copies leave the critical path.  CPU cost per step: one 24 KB memcpy into the slot and two
        graph launches instead of ~20 python -> ctypes kernel launches."""
        if not use_graph or (self.comm is not None and not self.dist_graphs):
            self.tu[:nb].copy_(host_triples[0, :nb], non_blocking=True)
            self.ti[:nb].copy_(host_triples[1, :nb], non_blocking=True)
            self.tj[:nb].copy_(host_triples[2, :nb], non_blocking=True)
            self.T = nb
            self._group(0, nb)
            self._launch_step(0)
            self._join_coefs()
            if self._loss_eager is None:
                self._loss_eager = torch.empty(4, dtype=torch.float32).pin_memory()
            self._loss_eager.copy_(self.out4[0], non_blocking=True)
            return self._loss_eager
        if self._ext is None or self._ext["nb"] != nb:
            self._ext = self._capture_external(nb)
        ext = self._ext
        k = ext["next"]
        ext["next"] = (k + 1) % len(ext["slots"])
        slot = ext["slots"][k]
        main = torch.cuda.current_stream()
        side = ext["side"]
        slot["prep_done"].synchronize()            # the PREP that last read this slot's host buffer has finished
        slot["host"][:, :nb].copy_(host_triples[:, :nb])
        side.wait_event(slot["step_done"])         # the STEP that last used this slot's device buffers has finished
        with torch.cuda.stream(side):
            slot["prep"].replay()
            slot["prep_done"].record(side)
        main.wait_event(slot["prep_done"])
        self.T = slot["batch"] * self.B + nb
        slot["step"].replay()
        slot["step_done"].record(main)
        return slot["loss"]

    def _capture_external(self, nb, n_slots=4):
        """Graphs of one externally fed step per pinned staging slot (a memcpy node's addresses are baked
        into the graph).  Slot k uses batch position k of the per-epoch triple / grouping arrays, so the
        PREP of one slot never writes what the STEP of another is reading."""
        n_slots = max(1, min(n_slots, self.cap // self.B))
        torch.cuda.synchronize()
        main = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        state = self._snapshot()
        slots = []
        for k in range(n_slots):
            slots.append({"batch": k, "host": torch.zeros((3, self.B), dtype=torch.int32).pin_memory(),
                          "loss": torch.zeros(4, dtype=torch.float32).pin_memory(),
                          "prep_done": torch.cuda.Event(), "step_done": torch.cuda.Event()})

        def prep(slot):
            t0 = slot["batch"] * self.B
            self.tu[t0:t0 + nb].copy_(slot["host"][0, :nb], non_blocking=True)
            self.ti[t0:t0 + nb].copy_(slot["host"][1, :nb], non_blocking=True)
            self.tj[t0:t0 + nb].copy_(slot["host"][2, :nb], non_blocking=True)
            self._group(t0, nb)

        def step(slot):
            self.T = slot["batch"] * self.B + nb
            self._launch_step(slot["batch"])
            self._join_coefs()
            slot["loss"].copy_(self.out4[slot["batch"]], non_blocking=True)

        prep(slots[0]); step(slots[0])              # eager warm-up (module loading, func attributes) on zeros
        torch.cuda.synchronize()
        for slot in slots:
            gp, gs = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(gp):
                prep(slot)
            prep(slot)                               # the grouping arrays of this slot must be valid while STEP is captured
            torch.cuda.synchronize()
            with torch.cuda.graph(gs):
                step(slot)
            slot["prep"], slot["step"] = gp, gs
        self._restore(state)
        torch.cuda.synchronize()
        for slot in slots:
            slot["prep_done"].record(main)
            slot["step_done"].record(main)
        torch.cuda.synchronize()
        return {"nb": nb, "slots": slots, "next": 0, "side": side}


class ContrastiveEngine(LightGCNEngine):
    """Fused SimGCL / XSimGCL training step (single GPU): the body of recommender/SimGCL.py:46-64 and
    recommender/XSimGCL.py:56-75 as a fixed kernel sequence, capturable in a CUDA graph.

    * propagation without layer 0 in the mean, the perturbation ``E += sign(E) * normalize(noise) * eps`` fused into
      the SpMM epilogue, the noise drawn there by Philox (or read from injected tables: ``noise_tables[(pass, layer)]``,
      the parity-test hook); last layers only compute the batch's rows;
    * BPR + L2 on the rec view (agcf_bpr_forward / backward), InfoNCE on the batch's unique users and unique positive
      items (agcf_bpr_cl_ids -> agcf_infonce_forward / backward with device-side counts, the ``emb[idx]`` gathers and
      the gradient scatter fused);
    * backward: sign() has zero gradient, so every view backpropagates through the SAME linear operator
      ``(A + ... + A^L) / L``.  SimGCL's three passes therefore need ONE backward propagation of the summed gradient
      (autograd runs three); XSimGCL adds the layer_cl view's gradient where that layer enters.  Adam is fused into
      the last backward SpMM.

    kind "xsimgcl": one perturbed pass, rec view F' = mean(E'_1..E'_L), CL between F' and E'_{layer_cl} (layer_cl < L).
    kind "simgcl": clean pass for the rec view + two perturbed passes for the CL views."""

    def __init__(self, graph, table, n_users, kind, n_layers, eps, cl_rate, tau, lr, reg, batch_size, max_triples,
                 layer_cl=1, noise_seed=0x5eed5eed, noise_tables=None, betas=(0.9, 0.999), adam_eps=1e-8):
        if kind not in ("simgcl", "xsimgcl"):
            raise ValueError("kind must be 'simgcl' or 'xsimgcl'")
        if kind == "xsimgcl" and not (1 <= layer_cl < n_layers):
            raise ValueError("the fused XSimGCL step needs 1 <= layer_cl < n_layers")
        super().__init__(graph, table, n_users, n_layers, lr, reg, batch_size, max_triples, betas=betas, adam_eps=adam_eps)
        if not self.sparse_layers:
            raise ValueError("graph too large for the per-batch bitmaps of the fused contrastive step")
        dev = table.device
        self.kind, self.eps, self.cl_rate, self.tau, self.layer_cl = kind, float(eps), float(cl_rate), float(tau), int(layer_cl)
        self.noise_seed = int(noise_seed) or 1
        self.noise_tables = noise_tables
        self.fuse_adam = True
        f = lambda: torch.empty_like(table)
        if self.L > 1 and not self.fw:
            self.fw, self.bw = [f(), f()], [f(), f()]
        if kind == "xsimgcl":
            self.Ecl = f()
            self.Gcl = torch.zeros_like(table)
        else:
            self.Va, self.Vb = f(), f()
            if self.L > 1:               # layer-1 tables of the three passes (they share A E0: one launch writes them)
                self.E1, self.E1a, self.E1b = f(), f(), f()
        nbmax = (self.cap + self.B - 1) // self.B
        i32 = lambda *shape: torch.zeros(shape, dtype=torch.int32, device=dev)
        self.cl_users, self.cl_items, self.n_cl = i32(nbmax, self.B), i32(nbmax, self.B), i32(nbmax, 2)
        self.cl_out = torch.zeros((nbmax, 2), dtype=torch.float32, device=dev)
        self.nce_ws = [ops.infonce_ws(self.B, self.d, dev), ops.infonce_ws(self.B, self.d, dev)]
        self._side_stream = torch.cuda.Stream(device=dev)
        self._fork_ev, self._join_ev = torch.cuda.Event(), torch.cuda.Event()
        n_prop = 1 if kind == "xsimgcl" else 3
        shared = 2 if (kind == "simgcl" and self.L > 1) else 0       # launches saved by the shared first layer
        # SpMM (n_prop * L forward + L backward) + bpr fwd/bwd + 2 x (3 InfoNCE fwd + 2 x 2 bwd) + zero rows + coefs
        self.launches_per_step = (n_prop + 1) * self.L - shared + 2 + 2 * 8 + (2 if kind == "xsimgcl" else 1) + 1

    # ------------------------------------------------------------------ set-up
    def _group(self, first_triple, n):
        super()._group(first_triple, n)
        if n <= 0:
            return
        b0 = first_triple // self.B
        ops.bpr_cl_ids(self.occ[b0 * 3 * self.B:], self.seg_off[b0 * (3 * self.B + 1):], self.seg_node[b0 * 3 * self.B:],
                       self.n_seg[b0:], n, self.B, self.U, self.cl_users[b0:], self.cl_items[b0:], self.n_cl[b0:])

    # ------------------------------------------------------------- propagation
    def _noise_kw(self, pass_id, k):
        if pass_id is None:
            return {}
        if self.noise_tables is not None:
            return {"noise": self.noise_tables[(pass_id, k)], "eps": self.eps}
        return {"philox": (self.noise_seed, pass_id * 64 + k, self.step_dev), "eps": self.eps}

    def _propagate(self, F, pass_id=None, mask=None, worklist=None, keep_layer=0, keep_into=None):
        """E_k = A E_{k-1} (perturbed if pass_id is not None); F = mean(E_1 .. E_L) (layer 0 excluded,
        recommender/SimGCL.py:198-210); layer ``keep_layer`` is kept in ``keep_into``.  With a mask / work list the
        LAST layer (and so F) is only computed on the batch's rows."""
        x = self.E0
        for k in range(1, self.L + 1):
            last = k == self.L
            if k == keep_layer:
                y = keep_into
            else:
                y = None if last else self.fw[(k - 1) % 2]
            wl = worklist if last else None
            ops.spmm(self.g, x, Y=y, acc_in=None if k == 1 else F, acc_out=F, acc_div=float(self.L) if last else 1.0,
                     row_mask=mask if (last and wl is None) else None, worklist=wl, **self._noise_kw(pass_id, k))
            x = y
        return F

    def _propagate_simgcl(self, mask, worklist):
        """The clean pass and the two perturbed passes of a SimGCL step (L >= 2).  Layer 1 of all three is A E0 -- the
        perturbation is added AFTER the product -- so ONE launch writes E1 (clean) and the two perturbed copies;
        layers 2..L run per pass, the last one on the batch's rows only.  4 + 3 (L - 2) full launches instead of 3 L."""
        tabs = self.noise_tables
        aux = [(self.E1a, None if tabs is None else tabs[(1, 1)], 64 + 1),
               (self.E1b, None if tabs is None else tabs[(2, 1)], 128 + 1)]
        ops.spmm(self.g, self.E0, Y=self.E1, aux=aux, eps=self.eps, philox=(self.noise_seed, None, self.step_dev))
        outs = []
        for pass_id, x, F in ((None, self.E1, self.F), (1, self.E1a, self.Va), (2, self.E1b, self.Vb)):
            first = x
            for k in range(2, self.L + 1):
                last = k == self.L
                y = None if last else self.fw[k % 2]
                wl = worklist if last else None
                ops.spmm(self.g, x, Y=y, acc_in=first if k == 2 else F, acc_out=F, acc_div=float(self.L) if last else 1.0,
                         row_mask=mask if (last and wl is None) else None, worklist=wl, **self._noise_kw(pass_id, k))
                x = y
            outs.append(F)
        return outs

    def forward_table(self, out=None, row_mask=None, worklist=None):
        """the unperturbed encoder forward (model() of the reference): what predict / test read"""
        return self._propagate(self.F if out is None else out, None, row_mask, worklist)

    # ---------------------------------------------------------------- one step
    def _launch_step(self, b):
        B, L = self.B, self.L
        t0 = b * B
        nb = min(B, self.T - t0)
        u, i, j = self.tu[t0:], self.ti[t0:], self.tj[t0:]
        occ = self.occ[b * 3 * B:]
        seg_off = self.seg_off[b * (3 * B + 1):]
        seg_node = self.seg_node[b * 3 * B:]
        n_seg = self.n_seg[b:]
        out4 = self.out4[b]
        mask = self.node_mask[b * self.mask_words:]
        wl = self._worklist(b)
        if self.kind == "xsimgcl":
            F = self._propagate(self.F, 0, mask, wl, keep_layer=self.layer_cl, keep_into=self.Ecl)
            v1, v2 = F, self.Ecl
        elif L == 1:
            F = self._propagate(self.F, None, mask, wl)
            v1 = self._propagate(self.Va, 1, mask, wl)
            v2 = self._propagate(self.Vb, 2, mask, wl)
        else:
            F, v1, v2 = self._propagate_simgcl(mask, wl)
        ops.bpr_forward(F, u, i, j, nb, self.U, self.reg, out4, self.coef, self.ws)
        ops.bpr_backward(F, u, i, j, nb, self.U, self.reg, 1.0, out4, self.coef, occ, seg_off, seg_node, n_seg, self.G)
        # contrastive terms: gradients land on the rows of G (rec / SimGCL views) and, pre-scaled by L, of Gcl
        g2_table = self.Gcl if self.kind == "xsimgcl" else self.G
        g2_scale = self.cl_rate * (L if self.kind == "xsimgcl" else 1)
        # the user-side and the item-side InfoNCE touch disjoint rows and own their workspaces: they run as two
        # parallel branches (a forked stream; inside a capture: two branches of the CUDA graph), each of them too
        # small (n <= B rows) to fill the GPU alone
        main = torch.cuda.current_stream()
        self._fork_ev.record(main)
        for side, rows in ((0, self.cl_users[b]), (1, self.cl_items[b])):
            stream = main if side == 0 else self._side_stream
            if side == 1:
                stream.wait_event(self._fork_ev)
            with torch.cuda.stream(stream):
                n_dev = self.n_cl[b, side:side + 1]
                ws = self.nce_ws[side]
                ops.infonce_forward(v1, v2, self.tau, rows=rows, n=B, n_dev=n_dev, loss=self.cl_out[b, side:side + 1], ws=ws)
                ops.infonce_backward(B, self.d, self.tau, ws, scale=self.cl_rate, n_dev=n_dev, grad1=self.G, rows1=rows,
                                     acc1=True)
                ops.infonce_backward(B, self.d, self.tau, ws, scale=g2_scale, n_dev=n_dev, grad2=g2_table, rows2=rows,
                                     acc2=self.kind != "xsimgcl")
                if side == 1:
                    self._join_ev.record(stream)
        main.wait_event(self._join_ev)
        # backward: D_L = G;  D_{k-1} = A D_k + G (+ Gcl where layer k-1 is the CL view);  dE0 = A D_1 / L
        adam = (self.E0, self.m, self.v, self.adam_coefs, self.betas[0], self.betas[1], self.adam_eps)
        H = self.G
        for k in range(L, 0, -1):
            cm = mask if k == L else None
            if k == 1:
                ops.spmm(self.g, H, acc_div=float(L), col_mask=cm, adam=adam)
                break
            nxt = self.bw[k % 2]
            if self.kind == "xsimgcl" and k - 1 == self.layer_cl:
                ops.spmm(self.g, H, addend=self.G, acc_in=self.Gcl, acc_out=nxt, col_mask=cm)
            else:
                ops.spmm(self.g, H, Y=nxt, addend=self.G, col_mask=cm)
            H = nxt
        ops.zero_rows(seg_node, n_seg, 3 * nb, self.G)
        if self.kind == "xsimgcl":
            ops.zero_rows(seg_node, n_seg, 3 * nb, self.Gcl)
        ops.adam_coefs(self.step_dev, self.adam_coefs, self.lr, self.betas[0], self.betas[1], increment=True)

    def losses(self, first_batch=0, n=None):
        """(rec_loss, cl_loss) per batch like the reference prints them (recommender/SimGCL.py:52-55)"""
        n = self.n_batches - first_batch if n is None else n
        rec = self.out4[first_batch:first_batch + n, 1]
        cl = self.cl_rate * self.cl_out[first_batch:first_batch + n].sum(1)
        return rec, cl


class NGCFEngine(LightGCNEngine):
    """Fused NGCF training step: the body of recommender/NGCF.py:48-66 with the encoder of :197-212 as a fixed kernel
    sequence, capturable in a CUDA graph.

    Per layer ONE propagation P = A E (agcf_spmm_csr_f32; the reference runs two -- A (E W1) = (A E) W1) and one fused
    dense kernel  E' = leaky_relu([P + E | P * E] [W1 ; W2])  that also keeps the running layer mean
    (agcf_ngcf_dense_forward); backward mirrors it (agcf_ngcf_dense_backward: dP, the direct gradient of E and the
    weight gradient in one pass over the rows; then A dP through the same SpMM with the direct term and the mean's share
    as addends).  Adam on the embedding table is fused into the last backward SpMM, Adam on the 2L weight matrices is
    one agcf_adam_step_f32 over their packed buffer ``W`` ([L, 2d, d], row block k = [W1_k ; W2_k]).

    launches per step: L x (SpMM + dense) + loss fwd/bwd + L x (dense + reduce + SpMM) + W transpose + 2 optimizer.

    ``comm`` (a DistContext, more than one rank): rows and adjacency rows split over the ranks (mode "rows"; the
    column-sharded "dshard" layout cannot hold NGCF, whose [2d, d] weights mix every column of a row).  Rank r owns rows
    [r0, r1) and runs every kernel of the step on them alone: the dense product is row-local, so it divides by the rank
    count.  The dense kernels' epilogues store E_1 .. E_{L-1}, the finished layer mean F and dP into every rank's copy
    (the next SpMM gathers them there), each rank's share of dW goes to its slot of every rank's [L, P, 2d*d] buffer, and
    every rank sums the P slots in rank order: dW, the W step and so W are bit-identical everywhere.  Adam updates the
    own rows of E0 in every copy.  One barrier per forward layer, one per backward layer, one closing the step."""

    # rows of the dW partial buffer.  d <= 64: the persistent CTAs of the backward dense kernel (two per SM).  d = 128 and
    # 256: the row slices of the split-K weight-gradient kernel, whose 2 / 8 output tiles times the slices fill the 148 SMs
    # once or twice; a partial is a whole 2d x d matrix (512 KB at d = 256), so 296 of them would be 150 MB
    N_PARTIALS = {8: 296, 16: 296, 32: 296, 64: 296, 128: 74, 256: 37}
    # row-partitioned layout: the ranks' row ranges balance a * nnz + b * rows (graph.balanced_row_ranges), with a and b
    # the single-GPU time in us per non-zero of a layer's two SpMMs and per row of its dense forward + backward, measured
    # at the Gowalla shape on a B200 at 1000 W (profiles/r5_ngcf_rows_p1.jsonl, tools/ngcf_dist_bench.py); other widths
    # balance the non-zeros
    ROW_COST = {64: (4.42e-5, 2.29e-3), 128: (7.04e-5, 7.39e-3), 256: (1.84e-4, 2.40e-2)}

    def __init__(self, graph, table, W, n_users, lr, reg, batch_size, max_triples, betas=(0.9, 0.999), adam_eps=1e-8,
                 comm=None, mode="rows"):
        n_layers = int(W.shape[0])
        d = table.shape[1]
        if d not in self.N_PARTIALS or tuple(W.shape) != (n_layers, 2 * d, d) or not W.is_contiguous():
            raise ValueError("NGCFEngine: d in {8, 16, 32, 64, 128, 256} and W packed as [L, 2d, d]")
        if mode in ("dshard", "grid"):
            raise ValueError("NGCFEngine cannot shard columns: its [2d, d] weight matrices mix every column of a row, so "
                             "a column slice of a layer needs all columns of the previous one; use mode='rows'")
        super().__init__(graph, table, n_users, n_layers, lr, reg, batch_size, max_triples, betas=betas, adam_eps=adam_eps,
                         sparse_layers=False, comm=comm, mode=mode)
        f = lambda: torch.empty_like(table)
        self.W = W
        self.Wm, self.Wv, self.dW = torch.zeros_like(W), torch.zeros_like(W), torch.zeros_like(W)
        self.WT = torch.empty((n_layers, d, 2 * d), dtype=torch.float32, device=table.device)
        self.dW_partial = torch.empty((self.N_PARTIALS[d], 2 * d * d), dtype=torch.float32, device=table.device)
        self.P = [f() for _ in range(self.L)]            # A E_{k-1}
        self.dEdir = f()
        self.dOut = [f(), f()]
        if self.mode == "rows":
            # E_1 .. E_{L-1} and dP (by layer parity: a fast rank writing layer k-1's dP must not overwrite the rows a slow
            # one still gathers for layer k) are gathered by the next SpMM: symmetric; E_L is only read row-locally
            self.Ek = [self.sym["E%d" % k] for k in range(1, self.L)] + [f()]
            self.dPs = [self.sym["dP0"], self.sym["dP1"]]
            self.dW_slots = self.sym["dW_slots"]             # [L, P, 2d*d]: slot r = rank r's share of dW
            row_off = self.r0 * self.d * 4
            tables = [k for k in self.sym if k != "dW_slots"]
            self._peer_rows = {k: self.comm.peers(k, row_off) for k in tables}
            self._mc_rows = {k: self.comm.multicast_ptr(k, row_off) for k in tables}
            P_, r = self.comm.world, self.comm.rank
            slot = lambda k: (k * P_ + r) * 2 * d * d * 4
            self._peer_slot = [self.comm.peers("dW_slots", slot(k)) for k in range(self.L)]
            self._mc_slot = [self.comm.multicast_ptr("dW_slots", slot(k)) for k in range(self.L)]
            self.fuse_adam = False
            # single-GPU count + the 2L + 1 barriers + L slot sums + zero_rows and the E0 Adam (not fused here)
            self.launches_per_step = 5 * self.L + 6 + (2 * self.L + 1) + self.L + 2
        else:
            self.Ek = [f() for _ in range(self.L)]       # layer outputs E_1 .. E_L
            self.dPs = [f()]
            self.fuse_adam = True
            self.launches_per_step = 5 * self.L + 6

    def _row_ranges(self, graph, world):
        return graph.row_ranges(world, cost=self.ROW_COST.get(self.d))

    def _symmetric_tables(self, world):
        t = ((self.N, self.d), torch.float32)
        specs = {"E0": t, "F": t, "dP0": t, "dP1": t}
        specs.update({"E%d" % k: t for k in range(1, self.L)})
        specs["dW_slots"] = ((self.L, world, 2 * self.d * self.d), torch.float32)
        return specs

    def _trained_state(self):
        return super()._trained_state() + [self.W, self.Wm, self.Wv]

    def _rows(self, t):
        return t[self.r0:self.r1]

    def forward_table(self, out=None, row_mask=None, worklist=None):
        F = self.F if out is None else out
        rows = self.mode == "rows"
        if rows and out is not None:
            raise ValueError("row-partitioned forward writes the symmetric F table")
        x = self.E0
        for k in range(1, self.L + 1):
            last = k == self.L
            ops.spmm(self.g, x, Y=self.P[k - 1])
            if rows:
                # own rows; E_k (k < L) and, at the last layer, F go to every rank's copy
                peer = "F" if last else "E%d" % k
                ops.ngcf_dense_forward(self._rows(self.P[k - 1]), self._rows(x), self.W[k - 1], self._rows(self.Ek[k - 1]),
                                       acc_in=self._rows(self.E0 if k == 1 else F), acc_out=self._rows(F),
                                       acc_div=float(self.L + 1) if last else 1.0,
                                       peer_Enext=None if last else self._peer_rows[peer],
                                       peer_acc=self._peer_rows[peer] if last else None,
                                       mc_Enext=0 if last else self._mc_rows[peer], mc_acc=self._mc_rows[peer] if last else 0)
                self._barrier()
            else:
                ops.ngcf_dense_forward(self.P[k - 1], x, self.W[k - 1], self.Ek[k - 1], acc_in=self.E0 if k == 1 else F,
                                       acc_out=F, acc_div=float(self.L + 1) if last else 1.0)
            x = self.Ek[k - 1]
        return F

    def _launch_step(self, b):
        B, L = self.B, self.L
        t0 = b * B
        nb = min(B, self.T - t0)
        u, i, j = self.tu[t0:], self.ti[t0:], self.tj[t0:]
        occ = self.occ[b * 3 * B:]
        seg_off = self.seg_off[b * (3 * B + 1):]
        seg_node = self.seg_node[b * 3 * B:]
        n_seg = self.n_seg[b:]
        out4 = self.out4[b]
        self.WT.copy_(self.W.transpose(1, 2))
        F = self.forward_table()
        ops.bpr_forward(F, u, i, j, nb, self.U, self.reg, out4, self.coef, self.ws)
        # G = dLoss/dF / (L + 1): the share every layer output (and E0) receives through the mean
        ops.bpr_backward(F, u, i, j, nb, self.U, self.reg, 1.0 / (L + 1), out4, self.coef, occ, seg_off, seg_node, n_seg, self.G)
        if self.mode == "rows":
            self._backward_rows(seg_node, n_seg, nb)
        else:
            d_out = self.G
            dP = self.dPs[0]
            adam = (self.E0, self.m, self.v, self.adam_coefs, self.betas[0], self.betas[1], self.adam_eps)
            for k in range(L, 0, -1):
                x_prev = self.E0 if k == 1 else self.Ek[k - 2]
                ops.ngcf_dense_backward(d_out, self.Ek[k - 1], self.P[k - 1], x_prev, self.WT[k - 1], dP, self.dEdir,
                                        self.dW_partial, self.dW[k - 1])
                if k > 1:                                    # dE_{k-1} = A dP + dE_direct + G
                    nxt = self.dOut[k % 2]
                    ops.spmm(self.g, dP, addend=self.dEdir, acc_in=self.G, acc_out=nxt)
                    d_out = nxt
                else:                                        # dE_0 goes straight into Adam; the batch's rows of G are re-zeroed
                    ops.spmm(self.g, dP, addend=self.dEdir, acc_in=self.G, adam=adam, zero_acc_in=True)
        ops.adam_step(self.W.view(-1), self.dW.view(-1), self.Wm.view(-1), self.Wv.view(-1), self.lr, self.betas[0],
                      self.betas[1], self.adam_eps, step_dev=self.step_dev)
        ops.adam_coefs(self.step_dev, self.adam_coefs, self.lr, self.betas[0], self.betas[1], increment=True)
        self._barrier()

    def _backward_rows(self, seg_node, n_seg, nb):
        """the row-partitioned backward: own rows throughout, dP and the dW slots exchanged before each layer's barrier"""
        R = self._rows
        d_out = self.G
        for k in range(self.L, 0, -1):
            x_prev = self.E0 if k == 1 else self.Ek[k - 2]
            dP, name = self.dPs[k % 2], "dP%d" % (k % 2)
            ops.ngcf_dense_backward(R(d_out), R(self.Ek[k - 1]), R(self.P[k - 1]), R(x_prev), self.WT[k - 1], R(dP),
                                    R(self.dEdir), self.dW_partial, self.dW_slots[k - 1, self.comm.rank],
                                    peer_dP=self._peer_rows[name], mc_dP=self._mc_rows[name],
                                    peer_dW=self._peer_slot[k - 1], mc_dW=self._mc_slot[k - 1])
            self._barrier()
            ops.ngcf_reduce_wgrad(self.dW_slots[k - 1], self.dW[k - 1])      # rank order: the same dW on every rank
            # dE_{k-1} = A dP + dE_direct + G on own rows (k = 1: the gradient of E0)
            nxt = self.dOut[k % 2] if k > 1 else self.dE0
            ops.spmm(self.g, dP, addend=self.dEdir, acc_in=self.G, acc_out=nxt)
            d_out = nxt
        ops.zero_rows(seg_node, n_seg, 3 * nb, self.G)
        # owner-computes: Adam on this rank's rows of E0, stored into every rank's copy
        r0, r1 = self.r0, self.r1
        ops.adam_step(self.E0[r0:r1], self.dE0[r0:r1], self.m[r0:r1], self.v[r0:r1], self.lr, self.betas[0],
                      self.betas[1], self.adam_eps, step_dev=self.step_dev, peer_p=self._peer_E0_rows,
                      mc_p=self._mc_E0_rows)
