"""Multi-GPU plumbing for the row-partitioned path (one process per GPU).

Layout (SURVEY.md 8e): the N = U + I node rows are split into P contiguous ranges
of ~equal nnz; rank p owns those rows of the adjacency (global column ids), of every
layer table and of the Adam state.  Every layer table is REPLICATED in a symmetric
(peer-mapped) allocation: the owner computes its rows and the SpMM epilogue stores
them straight into all peers' copies over NVLink (agcf_spmm_csr_f32 peer_Y /
peer_acc) -- the per-layer all-gather is fused into the kernel.  A device-side
barrier on the symmetric memory's signal pads closes each layer.

torch.distributed (NCCL) and torch's symmetric memory are used for rendezvous,
peer mapping and the barrier only.
"""
from __future__ import annotations

import torch
import torch.distributed as dist


class DistContext:
    """Symmetric arena + peer pointers + barrier for one process group."""

    def __init__(self, device, group=None):
        if not dist.is_initialized():
            raise RuntimeError("torch.distributed must be initialized (backend nccl)")
        self.group = group if group is not None else dist.group.WORLD
        self.rank = dist.get_rank(self.group)
        self.world = dist.get_world_size(self.group)
        if self.world > 8:
            raise ValueError("one NVSwitch box: at most 8 ranks")
        self.device = torch.device(device)
        self.arena = None
        self.hdl = None
        self._off = {}
        self._chan = 0
        import os
        self.use_multicast = os.environ.get("ARLIB_B200_MULTICAST", "1") == "1"    # tuning switch

    def allocate(self, specs):
        """specs: {name: (shape, dtype)} -> {name: local tensor}; all in ONE symmetric
        arena so every rank has the same offsets."""
        import torch.distributed._symmetric_memory as symm_mem
        total, layout = 0, {}
        for name, (shape, dtype) in specs.items():
            nbytes = int(torch.tensor([], dtype=dtype).element_size())
            for s in shape:
                nbytes *= int(s)
            layout[name] = (total, nbytes, tuple(shape), dtype)
            total += (nbytes + 255) // 256 * 256
        self.arena = symm_mem.empty(max(total, 256), dtype=torch.uint8, device=self.device)
        self.hdl = symm_mem.rendezvous(self.arena, self.group)
        out = {}
        for name, (off, nbytes, shape, dtype) in layout.items():
            out[name] = self.arena[off:off + nbytes].view(dtype).view(shape)
            self._off[name] = off
        return out

    def peers(self, name, extra_bytes=0, ranks=None):
        """device pointers of buffer ``name`` on all OTHER ranks (+ byte offset); ``ranks``: only those of this
        subset, in its order"""
        base = self._off[name] + int(extra_bytes)
        ranks = range(self.world) if ranks is None else ranks
        return [int(self.hdl.buffer_ptrs[r]) + base for r in ranks if r != self.rank]

    def all_ptrs(self, name, extra_bytes=0, ranks=None):
        """device pointers of buffer ``name`` on ALL ranks in rank order (own copy included); ``ranks``: on the ranks
        of this subset, in its order"""
        base = self._off[name] + int(extra_bytes)
        ranks = range(self.world) if ranks is None else ranks
        return [int(self.hdl.buffer_ptrs[r]) + base for r in ranks]

    def subgroups(self, groups):
        """NCCL process groups of the disjoint rank lists ``groups`` (ranks of this context's group); returns the one
        that holds this rank.  Every rank must call this with the same lists in the same order."""
        mine = None
        for ranks in groups:
            pg = dist.new_group([dist.get_global_rank(self.group, r) for r in ranks])
            if self.rank in ranks:
                mine = pg
        return mine

    def multicast_ptr(self, name, extra_bytes=0):
        """NVSwitch multicast address of buffer ``name`` (a store to it lands in every rank's copy), or 0
        when the platform has no multicast mapping (then the per-peer pointers are used)."""
        base = int(getattr(self.hdl, "multicast_ptr", 0) or 0)
        if base == 0 or not self.use_multicast:
            return 0
        return base + self._off[name] + int(extra_bytes)

    def barrier(self):
        """device-side barrier across ranks on the current stream"""
        self.hdl.barrier(channel=0)
