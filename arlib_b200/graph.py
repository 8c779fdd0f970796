"""Device mirror of the normalized adjacency: int32 CSR + fp32 values + the row
processing plan of the SpMM kernel.

Reference objects this mirrors: ``data.norm_adj`` (scipy, util/DataLoader.py:73-87),
``LGCN_Encoder.sparse_norm_adj`` (torch sparse COO, recommender/LightGCN.py:210,
212-215, 247-252).  Bit-exactness contract (SURVEY.md 8a-1): the degree vectors are
computed on the host with the reference's own numpy expression; the O(nnz) products
``fl(fl(d_i*w)*d_j)`` run on device (agcf_norm_adj_csr) and reproduce scipy's
``(D.A).D`` association bit for bit.
"""
from __future__ import annotations

import os

import numpy as np
import scipy.sparse as sp
import torch

from . import _lib

# Rows with more than `split_above` non-zeros are processed as segments of at most `segment` non-zeros (the unit
# of work of the SpMM kernel), so that no row is a long pole: a hub with thousands of non-zeros becomes dozens
# of independent work items.  A lane group needs ~1.5 us per 16 non-zeros, a short launch cannot hide a long
# work item, and every segment costs a partial-sum round trip: measured on B200 (profiles/r1_summary.md), when a
# launch covers >= 1.5 M non-zeros segments of 256 are best (Gowalla shape: 43 us at alpha = 0.5 AND at alpha = 0.8,
# where an uncut 13 689-nnz row took 91 us); when a rank owns a fraction of the graph, or the rows are narrow column
# slices, 64 is (quarter partition: 16.5 us vs 24.7 us; d = 8 slices: 27 us vs 55 us).
SEGMENT_ENV = os.environ.get("ARLIB_B200_SEGMENT")
SPLIT_ENV = os.environ.get("ARLIB_B200_SPLIT_ABOVE")
# persistent CTAs + dynamic block scheduling in the SpMM launches (default 0: one CTA per block of 8 warps' work
# items -- measured on B200 at the Gowalla shape: 0.2538 ms / step vs 0.2613 ms with persistent CTAs; the hardware
# CTA scheduler already refills SM slots without a visible gap, profiles/r1_summary.md)
PERSISTENT_ENV = os.environ.get("ARLIB_B200_PERSISTENT", "0")


def default_segment(local_nnz, d=64):
    """(split_above, segment): rows with more than split_above non-zeros are cut into segments of `segment`."""
    if d <= 8:
        seg = 32          # d = 8 column slices (8 GPUs): 23.6 us per full launch vs 26.7 us with 64 (profiles/r2_summary.md)
    elif d <= 32:
        seg = 64
    elif local_nnz >= 1_500_000:
        seg = 256
    elif local_nnz >= 600_000:
        seg = 128
    else:
        seg = 64
    if SEGMENT_ENV:
        seg = int(SEGMENT_ENV)
    return (int(SPLIT_ENV) if SPLIT_ENV else seg), seg


def balanced_row_ranges(indptr, world, cost=None):
    """Boundaries b[0..world] with b[0]=0, b[world]=n_rows and ~nnz/world non-zeros per range.

    cost = (a, b): balance a * nnz + b * rows per range instead -- for a step whose propagation time follows the
    non-zeros and whose dense layer time follows the rows (NGCF), where nnz-balanced ranges give the ranks that hold
    the many low-degree rows far more dense work."""
    indptr = np.asarray(indptr, dtype=np.int64)
    n = indptr.shape[0] - 1
    if cost is None:
        prefix, total = indptr, int(indptr[-1])
        target_of = lambda p: total * p // world
    else:
        a, b = float(cost[0]), float(cost[1])
        if a < 0 or b < 0 or a + b <= 0:
            raise ValueError("row-range cost weights must be >= 0 and not both 0")
        prefix = a * indptr.astype(np.float64) + b * np.arange(n + 1, dtype=np.float64)
        total = float(prefix[-1])
        target_of = lambda p: total * p / world
    bounds = [0]
    for p in range(1, world):
        b_ = int(np.searchsorted(prefix, target_of(p), side="left"))
        bounds.append(min(max(b_, bounds[-1]), n))
    bounds.append(n)
    return bounds


class DeviceGraph:
    """CSR (rowptr, col, val) on the device + the work plan of the SpMM kernel.  Immutable after build.

    Plan ("virtual rows"): row r with deg(r) non-zeros is cut into nseg = max(1, ceil(deg / segment))
    segments; every segment is one work item ``vrows[v] = (start, len, row, k | nseg << 16)`` (start indexes
    col / val), items are sorted by length descending so that the lane groups of a warp walk equally long
    segments.  Rows with several segments own ``nseg`` consecutive slots of the partial-sum scratch starting
    at ``vpart[v]``; the segment that finishes last (a ticket per row) adds the partials in segment order and
    runs the epilogue -- deterministic, no floating-point atomics."""

    def __init__(self, rowptr, col, val, n_rows, r0=0, r1=None, segment=None):
        self.rowptr, self.col, self.val = rowptr, col, val
        self._segment_arg = segment
        self.n_rows = int(n_rows)                    # global row count (= rows of X / Y)
        self.nnz = int(col.numel())
        self.r0 = int(r0)
        self.r1 = self.n_rows if r1 is None else int(r1)
        self.n_local_rows = self.r1 - self.r0        # rows this graph computes (all, or one rank's partition)
        self._coo_idx = None
        self._scratch = {}
        self._host_pattern = None                    # (indptr, indices) host copies, kept by the _init_uiAdj builder
        self._build_plan()

    def _build_plan(self):
        dev = self.device
        rp = self.rowptr.long()
        rows = torch.arange(self.r0, self.r1, device=dev)
        deg = rp[rows + 1] - rp[rows]
        split, SEGMENT = self._segment_arg if self._segment_arg else default_segment(int(deg.sum()))
        self.split_above, self.segment = int(split), int(SEGMENT)
        if SEGMENT < 16 or SEGMENT > 4096 or split < SEGMENT:
            raise ValueError("segment length must be in [16, 4096] and split_above >= segment")
        nseg = torch.where(deg > split, (deg + SEGMENT - 1) // SEGMENT, torch.ones_like(deg))
        if int(nseg.max()) >= 1 << 15 if nseg.numel() else False:
            raise ValueError("a row has more than %d non-zeros" % (SEGMENT << 15))
        n_v = int(nseg.sum())
        v_row = torch.repeat_interleave(rows, nseg)                       # real row of every work item
        first = torch.cumsum(nseg, 0) - nseg                              # first item of each row
        v_k = torch.arange(n_v, device=dev) - torch.repeat_interleave(first, nseg)
        v_nseg = torch.repeat_interleave(nseg, nseg)
        v_deg = torch.repeat_interleave(deg, nseg)
        v_start = rp[v_row] + v_k * SEGMENT
        v_len = torch.where(v_nseg > 1, torch.clamp(v_deg - v_k * SEGMENT, max=SEGMENT), v_deg)
        # partial-sum slots: rows with nseg > 1 get nseg consecutive slots
        multi = nseg > 1
        pbase_row = torch.cumsum(torch.where(multi, nseg, torch.zeros_like(nseg)), 0) - torch.where(multi, nseg, torch.zeros_like(nseg))
        v_part = torch.repeat_interleave(pbase_row, nseg)
        self.n_partial = int(nseg[multi].sum()) if bool(multi.any()) else 0
        order = torch.argsort(v_len, descending=True, stable=True)
        vr = torch.stack([v_start, v_len, v_row, v_k | (v_nseg << 16)], 1)[order]
        self.vrows = vr.to(torch.int32).contiguous()                      # [n_v, 4]
        self.vpart = v_part[order].to(torch.int32).contiguous()
        self.n_vrows = n_v
        self.local_nnz = int(deg.sum())
        self.max_segments = int(nseg.max()) if nseg.numel() else 0
        self.tickets = torch.zeros(max(self.n_partial, 1), dtype=torch.int32, device=dev)
        # dynamic block scheduler of the persistent launch mode: {next block, CTAs done}, self-resetting
        self.sched = torch.zeros(2, dtype=torch.int32, device=dev)
        self.persistent = PERSISTENT_ENV == "1"

    def partial_scratch(self, d):
        """[n_partial, d] fp32 scratch for the partial sums of multi-segment rows (one per width, reused by
        every launch on this graph: launches on one graph must be stream-ordered)."""
        t = self._scratch.get(d)
        if t is None:
            t = torch.empty((max(self.n_partial, 1), d), dtype=torch.float32, device=self.device)
            self._scratch[d] = t
        return t

    def refresh_plan_values(self):
        """the plan indexes ``val`` in place: nothing to refresh after ``val`` was modified"""

    @property
    def device(self):
        return self.val.device

    # -------------------------------------------------------------- partitioning
    def row_ranges(self, world, cost=None):
        """world+1 boundaries of contiguous row ranges with ~equal nnz (power-law rows:
        balance by non-zeros, not by rows); cost = (a, b): ~equal a * nnz + b * rows."""
        return balanced_row_ranges(self.rowptr.cpu().numpy(), world, cost)

    def partition(self, r0, r1, segment=None):
        """Graph that COMPUTES only rows [r0, r1) (one rank of the row-partitioned
        multi-GPU path); X / Y keep global row ids, col ids are global."""
        return DeviceGraph(self.rowptr, self.col, self.val, self.n_rows, r0, r1, segment)

    def replan(self, split_above, segment):
        """The same graph (shared CSR arrays) with another split threshold / segment length."""
        if (split_above, segment) == (self.split_above, self.segment):
            return self
        return DeviceGraph(self.rowptr, self.col, self.val, self.n_rows, self.r0, self.r1, (split_above, segment))

    def planned_for(self, d):
        """The plan that suits tables of width d (narrow column slices want every row in short segments)."""
        return self.replan(*default_segment(self.local_nnz, d))

    # ---------------------------------------------------------------- builders
    @classmethod
    def _from_csr_host(cls, csr: sp.csr_matrix, device, values=None):
        if csr.shape[0] != csr.shape[1]:
            raise ValueError("adjacency must be square")
        if csr.nnz >= 2 ** 31 or csr.shape[0] >= 2 ** 31:
            raise ValueError("graph exceeds int32 indexing")
        dev = torch.device(device)
        rowptr = torch.from_numpy(csr.indptr.astype(np.int32)).to(dev)
        col = torch.from_numpy(csr.indices.astype(np.int32)).to(dev)
        if values is None:
            val = torch.from_numpy(np.ascontiguousarray(csr.data, dtype=np.float32)).to(dev)
        else:
            val = values
        return cls(rowptr, col, val, csr.shape[0])

    @classmethod
    def from_scipy(cls, mat, device="cuda"):
        """Upload an already-normalized scipy matrix as is (values untouched)."""
        csr = sp.csr_matrix(mat)
        csr.sum_duplicates()
        csr.sort_indices()
        return cls._from_csr_host(csr, device)

    @classmethod
    def normalized(cls, adj, d_row, d_col, device="cuda", reuse=None):
        """values = fl(fl(d_row[i]*w)*d_col[j]) computed ON DEVICE from the raw
        weights of ``adj`` (scipy, canonical CSR) and host-computed degree vectors.

        ``reuse``: a graph built by an earlier call.  If the sparsity PATTERN is the same (row pointers and column
        indices equal -- checked against host copies kept for this purpose) the new graph shares the device index
        arrays, the SpMM work plan and the COO index view of the old one; only the weights are uploaded and
        re-normalized.  That is the repeated ``_init_uiAdj`` of the white-box attack loops (attack/White/PGA.py:93-97:
        once per 128-item batch, fake rows with the same dense pattern and new fractional values).  Same bits as a
        full rebuild (the values come from the same kernel on the same inputs)."""
        csr = sp.csr_matrix(adj)
        csr.sum_duplicates()
        csr.sort_indices()
        dev = torch.device(device)
        w = torch.from_numpy(np.ascontiguousarray(csr.data, dtype=np.float32)).to(dev)
        dr = torch.from_numpy(np.ascontiguousarray(d_row, dtype=np.float32)).to(dev)
        dc = torch.from_numpy(np.ascontiguousarray(d_col, dtype=np.float32)).to(dev)
        val = torch.empty_like(w)
        g = None
        if reuse is not None and reuse._host_pattern is not None and reuse.device == dev and reuse.n_rows == csr.shape[0] \
                and reuse.nnz == csr.nnz and reuse.r0 == 0 and reuse.r1 == reuse.n_rows:
            hp, hi = reuse._host_pattern
            if np.array_equal(hp, csr.indptr) and np.array_equal(hi, csr.indices):
                g = reuse.with_values(val)
        if g is None:
            g = cls._from_csr_host(csr, device, values=val)
            g._host_pattern = (csr.indptr.copy(), csr.indices.copy())
        lib = _lib.load()
        _lib.check(lib.agcf_norm_adj_csr(g.rowptr.data_ptr(), g.col.data_ptr(), w.data_ptr(), dr.data_ptr(),
                                         dc.data_ptr(), val.data_ptr(), g.n_rows, g.nnz, _lib.stream_ptr()),
                   "agcf_norm_adj_csr")
        g.refresh_plan_values()
        return g

    def with_values(self, val):
        """A graph with the same pattern and plan (all index arrays shared) and another value array."""
        import copy
        g = copy.copy(self)
        g.val = val
        return g

    @classmethod
    def from_ui_adj(cls, ui_adj, device="cuda", reuse=None):
        """``_init_uiAdj`` (recommender/LightGCN.py:212-215): 1/np.sqrt of row AND
        column sums, no inf guard, fractional weights allowed."""
        d_row = np.array((1 / np.sqrt(ui_adj.sum(1)))).flatten()
        d_col = np.array((1 / np.sqrt(ui_adj.sum(0)))).flatten()
        return cls.normalized(ui_adj, d_row, d_col, device, reuse=reuse)

    @classmethod
    def from_dataloader_adj(cls, adj, device="cuda"):
        """``DataLoader.normalize_graph_mat`` (util/DataLoader.py:73-81): np.power(rowsum,
        -0.5) with inf -> 0, the same vector on both sides."""
        rowsum = np.array(adj.sum(1))
        d = np.power(rowsum, -0.5).flatten()
        d[np.isinf(d)] = 0.
        return cls.normalized(adj, d, d, device)

    @classmethod
    def from_device_edges(cls, e_user, e_item, n_users, n_items, segment=None):
        """Normalized bipartite adjacency straight from UNIQUE (user, item) edge tensors on the device -- the builder for
        graphs scipy cannot hold in reasonable time (400 M non-zeros at the 10 M x 1 M scale-stress shape).  Same result
        as ``from_dataloader_adj(bipartite adjacency of the edges)``, bit for bit: A = R_ext + R_ext^T with unit weights
        (util/DataLoader.py:57-71), canonical CSR (one device sort of the 2E keys), d = np.power(rowsum, -0.5) with
        inf -> 0 evaluated by numpy on the HOST over the N degree counts (:77-80 -- a libm pow no device routine is
        bit-compatible with), values fl(fl(d_i * 1) * d_j) as two separate fp32 multiplications (no FMA contraction)."""
        dev = e_user.device
        n = int(n_users) + int(n_items)
        if n >= 2 ** 31 or 2 * e_user.numel() >= 2 ** 31:
            raise ValueError("graph exceeds int32 indexing")
        u = e_user.to(torch.int64)
        it = e_item.to(torch.int64) + int(n_users)
        keys = torch.cat([u * n + it, it * n + u])
        del u, it
        keys = torch.sort(keys).values
        rows = keys // n
        col = (keys - rows * n).to(torch.int32)
        del keys
        counts = torch.bincount(rows, minlength=n)
        rowptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        torch.cumsum(counts, 0, out=rowptr[1:])
        rowsum = counts.to(torch.float32).cpu().numpy().reshape(-1, 1)      # sum of unit weights == the degree, exact in fp32
        d = np.power(rowsum, -0.5).flatten()
        d[np.isinf(d)] = 0.
        dd = torch.from_numpy(np.ascontiguousarray(d, dtype=np.float32)).to(dev)
        val = dd[rows] * 1.0
        val = val * dd[col.long()]
        del rows
        return cls(rowptr.to(torch.int32), col, val, n, segment=segment)

    @classmethod
    def from_coo_tensor(cls, t: torch.Tensor):
        """From a torch sparse COO tensor (someone assigned model.sparse_norm_adj)."""
        t = t.detach().coalesce()
        idx = t.indices()
        n = t.shape[0]
        counts = torch.bincount(idx[0], minlength=n)
        rowptr = torch.zeros(n + 1, dtype=torch.int64, device=t.device)
        rowptr[1:] = torch.cumsum(counts, 0)
        return cls(rowptr.to(torch.int32), idx[1].to(torch.int32).contiguous(), t.values().float().contiguous(), n)

    # ------------------------------------------------------------------ views
    def coo_indices(self):
        """int64 [2, nnz] COO indices (row-major order) -- built once on demand."""
        if self._coo_idx is None:
            lib = _lib.load()
            row = torch.empty(self.nnz, dtype=torch.int32, device=self.device)
            _lib.check(lib.agcf_csr_expand_rows(self.rowptr.data_ptr(), row.data_ptr(), self.n_rows, self.nnz,
                                                _lib.stream_ptr()), "agcf_csr_expand_rows")
            self._coo_idx = torch.stack([row.long(), self.col.long()])
        return self._coo_idx

    def to_coo_tensor(self):
        """torch sparse COO tensor sharing ``val`` -- the ``sparse_norm_adj`` attribute
        attacks touch (attack/White/PGA.py:98,117).  Unlike the reference's it IS
        coalesced (it is built from canonical CSR)."""
        return torch.sparse_coo_tensor(self.coo_indices(), self.val, (self.n_rows, self.n_rows),
                                       is_coalesced=True)

    def to_scipy(self):
        return sp.csr_matrix((self.val.cpu().numpy(), self.col.cpu().numpy(), self.rowptr.cpu().numpy()),
                             shape=(self.n_rows, self.n_rows))
