// handoff.cu -- the column-group hand-off of the grid layout (R row blocks x C column slices).
//
// In the grid layout the ranks that share a column slice (a "column group") each compute a row block of every layer and
// store it into the partners' copies of the layer table (the SpMM epilogue's per-peer stores, agcf_spmm_csr_f32
// peer_Y / peer_acc; Adam's peer_p).  Before the next kernel gathers from a table, every partner's rows of it must have
// landed.  The row-partitioned layout closes each layer with an all-rank barrier launch; the grid closes it with this
// kernel, which involves only the R - 1 partners of the column group.
//
// Protocol.  Each rank has one flag word per group member (`flags`, in peer-mapped memory); partner q writes only
// flags[slot of q].  A hand-off takes stamp = *stamp_dev + 1, stores it with st.release.sys into its own slot of every
// partner's flag words, spins with ld.acquire.sys until every partner's slot in its own flag words carries that stamp
// (or a later one: a partner can be at most one hand-off ahead, it cannot pass the next one without this rank's
// stamp), and writes the stamp back to *stamp_dev.  stamp_dev is private to the group and never restored by the
// caller, so stamps only grow: a CUDA graph replayed after an eager warm-up of the same launches never sees a flag
// left by an earlier hand-off as the current one.  Comparisons are on the signed difference (wrap after 2^32
// hand-offs is harmless).
//
// Why the previous kernel's peer stores are visible to a partner once it sees the stamp.  The hand-off runs in stream
// order after the kernel whose stores it publishes, so those stores are complete before any of its threads runs.  The
// publishing thread then issues fence.acq_rel.sys and its st.release.sys: a release at system scope is cumulative, it
// orders every write this GPU has made visible to the thread -- the previous kernel's NVLink stores included -- before
// the flag.  The partner's ld.acquire.sys that reads the stamp synchronises with that release, the partner's spinning
// threads then meet at __syncwarp, and its next kernel starts only after this one completes, so every kernel it
// launches after the hand-off reads the stored rows.  This is the argument of the all-rank barrier the row-partitioned
// layout uses (release store into each peer's signal pad, acquire wait on its own), restricted to a group.
//
// Why the parity-double-buffered layer tables are not overwritten while a partner still gathers from them.  Forward
// layer k reads table fw[k % 2] (the output of layer k - 1) and stores into fw[(k - 1) % 2] of every partner; layer
// k + 1 stores into fw[k % 2].  A rank reaches layer k + 1 only after the hand-off that closes layer k, which needs
// every partner's stamp for that hand-off, which the partner publishes only after its layer-k SpMM -- the last reader
// of fw[k % 2] -- has completed.  The backward tables bw[0] / bw[1] alternate the same way, and E0 (stored into by
// Adam) is read only by the next step's first forward layer, which follows the hand-off that closes the step.
//
// The spin is bounded: a partner that never arrives (a crashed or mismatched rank) makes the wait give up after 4 s
// and set *err to 1; the stamp still advances, and the caller turns the error word into an exception at its next
// host synchronisation.  Nothing traps.
#include "common.cuh"

namespace {

struct HandoffPeers {
  int32_t* p[AGCF_MAX_PEERS];
};

constexpr unsigned long long kHandoffTimeoutNs = 4000000000ull;

__device__ __forceinline__ void st_release_sys_s32(int32_t* p, int32_t v) {
  asm volatile("fence.acq_rel.sys;\n\tst.release.sys.global.s32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int32_t ld_acquire_sys_s32(const int32_t* p) {
  int32_t v;
  asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long handoff_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

}  // namespace

// one warp: lane q < n_peers publishes to partner q, lane s <= n_peers (s != my_slot) waits for slot s
__global__ void __launch_bounds__(32) group_handoff_kernel(int32_t* flags, HandoffPeers peers, int n_peers, int my_slot,
                                                           int32_t* stamp_dev, int32_t* err) {
  const int lane = threadIdx.x;
  const uint32_t stamp = (uint32_t)*reinterpret_cast<volatile int32_t*>(stamp_dev) + 1u;
  int32_t* dst = nullptr;
#pragma unroll
  for (int q = 0; q < AGCF_MAX_PEERS; ++q)           // no dynamic index into the parameter struct (no stack frame)
    if (q == lane) dst = peers.p[q];
  if (lane < n_peers) st_release_sys_s32(dst + my_slot, (int32_t)stamp);
  if (lane <= n_peers && lane != my_slot) {
    const unsigned long long t_start = handoff_ns();
    while ((int32_t)((uint32_t)ld_acquire_sys_s32(flags + lane) - stamp) < 0) {
      if (handoff_ns() - t_start > kHandoffTimeoutNs) {
        atomicExch(err, 1);
        break;
      }
      __nanosleep(32);
    }
  }
  __syncwarp();
  if (lane == 0) *stamp_dev = (int32_t)stamp;
}

extern "C" int agcf_group_handoff(int32_t* flags, void* const* peer_flags_host, int32_t n_peers, int32_t my_slot,
                                  int32_t* stamp_dev, int32_t* err, agcf_stream_t stream) {
  if (!flags || !stamp_dev || !err || n_peers < 0 || n_peers >= AGCF_MAX_PEERS) return AGCF_EINVAL;
  if (my_slot < 0 || my_slot > n_peers || (n_peers > 0 && !peer_flags_host)) return AGCF_EINVAL;
  HandoffPeers peers;
  for (int q = 0; q < AGCF_MAX_PEERS; ++q) {
    peers.p[q] = q < n_peers ? reinterpret_cast<int32_t*>(peer_flags_host[q]) : nullptr;
    if (q < n_peers && peers.p[q] == nullptr) return AGCF_EINVAL;
  }
  group_handoff_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(flags, peers, n_peers, my_slot, stamp_dev, err);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}
