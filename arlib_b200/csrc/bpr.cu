// bpr.cu -- BPR triple sampling, fused gather-score-loss, atomic-free gradient
// scatter and the Adam step of the LightGCN training loop on B200.
//
// Reference: util/sampler.py:4-30 (next_batch_pairwise), util/loss.py:5-9
// (bpr_loss), :25-29 (l2_reg_loss), recommender/LightGCN.py:51-56,64 (gathers,
// backward, optimizer.step()).  All kernels here are HBM/L2-bound integer / fp32
// row work: coalesced 16-byte lanes, one lane group per embedding row, fixed-order
// reductions (results are run-to-run deterministic).
#include "common.cuh"

namespace agcf {

template <int D>
struct RowCfg2 {
  static constexpr int V4 = D / 4;
  static constexpr int LPR = V4 < 32 ? V4 : 32;
  static constexpr int VPL = V4 / LPR;
  static constexpr int RPW = 32 / LPR;
  static constexpr int THREADS = 256;
  static constexpr int RPB = (THREADS / 32) * RPW;
};

// =============================================================== sampler (Philox)
__device__ __forceinline__ uint32_t fmix32(uint32_t h) {
  h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
  return h;
}

// keyed bijection of [0, 2^(2*half_bits)) : 6-round balanced Feistel network whose
// round keys come from Philox(seed, epoch); cycle-walking restricts it to [0, n).
__device__ __forceinline__ uint32_t feistel_perm(uint32_t x, int half_bits, const uint32_t (&rk)[8]) {
  const uint32_t mask = (1u << half_bits) - 1u;
  uint32_t l = x >> half_bits, r = x & mask;
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const uint32_t f = fmix32(r ^ rk[k]) & mask;
    const uint32_t nl = r;
    r = l ^ f;
    l = nl;
  }
  return (l << half_bits) | r;
}

__global__ void __launch_bounds__(256) bpr_sample_kernel(const int32_t* __restrict__ e_user, const int32_t* __restrict__ e_item,
                                                         int n_edges, const int32_t* __restrict__ rej_rowptr,
                                                         const int32_t* __restrict__ rej_items, int n_items,
                                                         uint64_t seed, uint64_t epoch, int half_bits,
                                                         int32_t* __restrict__ out_u, int32_t* __restrict__ out_i,
                                                         int32_t* __restrict__ out_j) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_edges) return;
  // round keys: Philox stream (seed, epoch), counters reserved at the top of the space
  uint32_t rk[8], tmp[4];
  Philox::gen(seed, epoch, 0xFFFFFFFFFFFFFFFFull, tmp);
  rk[0] = tmp[0]; rk[1] = tmp[1]; rk[2] = tmp[2]; rk[3] = tmp[3];
  Philox::gen(seed, epoch, 0xFFFFFFFFFFFFFFFEull, tmp);
  rk[4] = tmp[0]; rk[5] = tmp[1]; rk[6] = tmp[2]; rk[7] = tmp[3];
  uint32_t x = (uint32_t)t;
  do { x = feistel_perm(x, half_bits, rk); } while (x >= (uint32_t)n_edges);   // cycle walk
  const int u = e_user[x];
  const int i = e_item[x];
  const int rs = rej_rowptr[u], re = rej_rowptr[u + 1];
  int j = 0;
  bool done = false;
  for (uint32_t blk = 0; blk < 64 && !done; ++blk) {     // <= 256 draws, then accept (degenerate user)
    uint32_t r4[4];
    Philox::gen(seed, ((uint64_t)blk << 32) | (uint32_t)t, epoch, r4);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (done) break;
      j = (int)__umulhi(r4[k], (uint32_t)n_items);       // uniform in [0, n_items), bias < n_items / 2^32
      int lo = rs, hi = re;                                // binary search in the sorted rejection list
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(rej_items + mid) < j) lo = mid + 1; else hi = mid;
      }
      done = !(lo < re && __ldg(rej_items + lo) == j);
    }
  }
  out_u[t] = u;
  out_i[t] = i;
  out_j[t] = j;
}

// ========================================================= batch grouping (sort)
// One CTA per batch: bitonic sort of (node << 32 | occurrence id) in shared memory,
// then segment heads by block scan.  Makes the gradient scatter atomic-free.
__global__ void __launch_bounds__(1024) bpr_group_kernel(const int32_t* __restrict__ u, const int32_t* __restrict__ i,
                                                         const int32_t* __restrict__ j, int n_triples, int batch,
                                                         int n_users, int pow2, int32_t* __restrict__ occ,
                                                         int32_t* __restrict__ seg_off, int32_t* __restrict__ seg_node,
                                                         int32_t* __restrict__ n_seg, int mask_words,
                                                         uint32_t* __restrict__ node_mask) {
  extern __shared__ unsigned long long keys[];
  __shared__ int warp_tot[32];
  __shared__ int block_total;
  const int b = blockIdx.x;
  const int t0 = b * batch;
  const int nb = min(batch, n_triples - t0);
  const int n_occ = 3 * nb;
  const int tid = threadIdx.x, nthr = blockDim.x;
  uint32_t* mask_b = node_mask != nullptr ? node_mask + (size_t)b * mask_words : nullptr;
  if (mask_b != nullptr)
    for (int k = tid; k < mask_words; k += nthr) mask_b[k] = 0u;      // visible block-wide after the sort's barriers
  for (int k = tid; k < pow2; k += nthr) {
    unsigned long long key = ~0ull;
    if (k < n_occ) {
      const int role = k / nb, t = k - role * nb;
      int node;
      if (role == 0) node = u[t0 + t];
      else if (role == 1) node = n_users + i[t0 + t];
      else node = n_users + j[t0 + t];
      key = ((unsigned long long)(uint32_t)node << 32) | (uint32_t)k;
    }
    keys[k] = key;
  }
  __syncthreads();
  for (int kk = 2; kk <= pow2; kk <<= 1) {
    for (int jj = kk >> 1; jj > 0; jj >>= 1) {
      for (int idx = tid; idx < (pow2 >> 1); idx += nthr) {
        const int a = ((idx & ~(jj - 1)) << 1) | (idx & (jj - 1));
        const int c = a | jj;
        const bool up = (a & kk) == 0;
        const unsigned long long ka = keys[a], kc = keys[c];
        if ((ka > kc) == up) { keys[a] = kc; keys[c] = ka; }
      }
      __syncthreads();
    }
  }
  // segment heads: contiguous chunk per thread, block-wide exclusive scan of head counts
  const int per = pow2 / nthr > 0 ? pow2 / nthr : 1;
  const int lo = tid * per, hi = min(lo + per, n_occ);
  int heads = 0;
  for (int k = lo; k < hi; ++k) {
    const uint32_t node = (uint32_t)(keys[k] >> 32);
    heads += (k == 0 || node != (uint32_t)(keys[k - 1] >> 32)) ? 1 : 0;
  }
  int incl = heads;
  const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = lane < (nthr >> 5) ? warp_tot[lane] : 0;
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += y;
    }
    warp_tot[lane] = winc - w;                    // exclusive warp offsets
    if (lane == 31) block_total = winc;
  }
  __syncthreads();
  int seg = warp_tot[warp] + incl - heads;         // exclusive prefix for this thread
  int32_t* occ_b = occ + (size_t)b * 3 * batch;
  int32_t* off_b = seg_off + (size_t)b * (3 * batch + 1);
  int32_t* node_b = seg_node + (size_t)b * 3 * batch;
  for (int k = lo; k < hi; ++k) {
    const unsigned long long key = keys[k];
    const uint32_t node = (uint32_t)(key >> 32);
    occ_b[k] = (int32_t)(uint32_t)key;
    if (k == 0 || node != (uint32_t)(keys[k - 1] >> 32)) {
      off_b[seg] = k;
      node_b[seg] = (int32_t)node;
      if (mask_b != nullptr) atomicOr(mask_b + (node >> 5), 1u << (node & 31));
      ++seg;
    }
  }
  if (tid == 0) {
    off_b[block_total] = n_occ;
    n_seg[b] = block_total;
  }
}

// ================================================================== BPR forward
struct BprWs {                 // layout of the workspace
  unsigned int ticket;         // must be 0 on entry; the kernel leaves it 0
  unsigned int pad[3];
  float partial[1];            // [3 * n_blocks]: loss, sum u^2, sum i^2
};

// Block partials -> workspace; the last block to arrive (ticket) reduces all partials in a fixed order with
// double accumulators and writes out4 = {loss, bpr term, ||F[u_.]||_F, ||F[i_.]||_F}.  Deterministic.
template <int NRED>
__device__ __forceinline__ void bpr_finalize(float (&red)[3][NRED], int nb, float reg, float* __restrict__ out4,
                                             BprWs* __restrict__ ws, int32_t* __restrict__ bump = nullptr) {
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < 3) {
    float acc = 0.f;
    for (int k = 0; k < NRED; ++k) acc += red[threadIdx.x][k];      // fixed order
    ws->partial[3 * blockIdx.x + threadIdx.x] = acc;
    __threadfence();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int tk = atomicAdd(&ws->ticket, 1u);
    is_last = (tk == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last || warp != 0) return;
  __threadfence();
  double a0 = 0.0, a1 = 0.0, a2 = 0.0;
  const volatile float* part = ws->partial;
  for (int k = lane; k < (int)gridDim.x; k += 32) {
    a0 += (double)part[3 * k + 0];
    a1 += (double)part[3 * k + 1];
    a2 += (double)part[3 * k + 2];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a0 += __shfl_xor_sync(0xffffffffu, a0, o);
    a1 += __shfl_xor_sync(0xffffffffu, a1, o);
    a2 += __shfl_xor_sync(0xffffffffu, a2, o);
  }
  if (lane == 0) {
    const float bpr = (float)(a0 / (double)nb);
    const float nu = (float)sqrt(a1), ni = (float)sqrt(a2);
    out4[0] = bpr + (nu + ni) * reg;                          // emb_loss * reg, util/loss.py:29
    out4[1] = bpr;
    out4[2] = nu;
    out4[3] = ni;
    ws->ticket = 0u;
    if (bump != nullptr) *bump += 1;       // every block of this launch read the counter before it took its ticket
  }
}

template <int D>
__global__ void __launch_bounds__(256) bpr_forward_kernel(const float4* __restrict__ F, const int32_t* __restrict__ u,
                                                          const int32_t* __restrict__ i, const int32_t* __restrict__ j,
                                                          int nb, int n_users, float reg, float* __restrict__ out4,
                                                          float* __restrict__ coef, BprWs* __restrict__ ws) {
  using C = RowCfg2<D>;
  __shared__ float red[3][C::RPB];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gl = lane & (C::LPR - 1), grp = lane / C::LPR;
  const int slot = warp * C::RPW + grp;
  const int t = blockIdx.x * C::RPB + slot;
  const bool valid = t < nb;
  float dpos = 0.f, dneg = 0.f, su = 0.f, si = 0.f;
  if (valid) {
    const float4* fu = F + (size_t)u[t] * C::V4 + gl;
    const float4* fi = F + ((size_t)n_users + i[t]) * C::V4 + gl;
    const float4* fj = F + ((size_t)n_users + j[t]) * C::V4 + gl;
#pragma unroll
    for (int v = 0; v < C::VPL; ++v) {
      const float4 a = __ldg(fu + v * C::LPR), p = __ldg(fi + v * C::LPR), n = __ldg(fj + v * C::LPR);
      dpos += dot4(a, p);
      dneg += dot4(a, n);
      su += dot4(a, a);
      si += dot4(p, p);
    }
  }
  dpos = group_sum<C::LPR>(dpos);
  dneg = group_sum<C::LPR>(dneg);
  su = group_sum<C::LPR>(su);
  si = group_sum<C::LPR>(si);
  float l = 0.f;
  if (valid) {
    const float x = dpos - dneg;
    const float s = 1.f / (1.f + expf(-x));
    l = -logf(1e-7f + s);                                   // util/loss.py:8  (10e-8 == 1e-7)
    if (gl == 0) coef[t] = -(s * (1.f - s)) / ((1e-7f + s) * (float)nb);
  } else {
    su = 0.f; si = 0.f;
  }
  if (gl == 0) { red[0][slot] = l; red[1][slot] = su; red[2][slot] = si; }
  __syncthreads();
  bpr_finalize<C::RPB>(red, nb, reg, out4, ws);
}

// ===================================================== d-sharded forward (multi-GPU)
// Every rank holds a column slice [N, d/P] of the tables.  bpr_partial computes, per triple, the slice's
// share of the two dot products and of the two squared norms and stores it into slot `rank` of the exchange
// buffer on EVERY rank (NVLink P2P stores); bpr_finish sums the P shares in rank order -- identical bits on all
// ranks -- and does what bpr_forward does from there on.
//
// The exchange carries its own synchronisation (the "LL" idea of collective libraries): every value travels as ONE
// naturally aligned 64-bit word {stamp : 32 | float bits : 32}, stamp = step + 1.  A 64-bit scalar store is
// single-copy atomic, so a reader that sees the stamp of the current step has the value that was written with it:
// no fence, no flag, NO BARRIER LAUNCH (the torch symmetric-memory barrier this replaces cost 41.5 us per step and
// was the largest single item of the 8-GPU step, profiles/r1_summary.md section 4).  bpr_finish spins on the words
// it needs (ld.relaxed.sys, L1 bypassed) -- it waits exactly as long as the slowest rank is behind, per triple.
// The buffer is double-buffered on the parity of the step: a writer can reach step s + 2 (the next use of the same
// half) only after its own finish(s + 1), which needed every reader's partial(s + 1), which that reader launched
// after its finish(s) had read the half.  "Step" here is the EXCHANGE COUNTER (a device int32 both kernels read; the
// last block of bpr_finish advances it), not the optimizer's step: a stamp must never be used twice -- an engine that
// restores its optimizer step after a warm-up launch (CUDA-graph capture) would otherwise let a fast rank read the
// warm-up's words of a slow peer as if they were the step's.
struct XchgPeers {
  int n;
  unsigned long long* p[AGCF_MAX_PEERS];
};

__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ unsigned long long ll_pack(float v, uint32_t stamp) {
  return ((unsigned long long)stamp << 32) | (unsigned long long)__float_as_uint(v);
}
// a rank that never shows up must not hang the GPU: after this long the reader gives up and poisons the loss
constexpr unsigned long long kXchgTimeoutNs = 4000000000ull;

template <int D>
__global__ void __launch_bounds__(256) bpr_partial_kernel(const float4* __restrict__ F, const int32_t* __restrict__ u,
                                                          const int32_t* __restrict__ i, const int32_t* __restrict__ j,
                                                          int nb, int n_users, int rank, int cap,
                                                          const int32_t* __restrict__ xchg_ctr, XchgPeers x) {
  using C = RowCfg2<D>;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gl = lane & (C::LPR - 1), grp = lane / C::LPR;
  const int t = blockIdx.x * C::RPB + warp * C::RPW + grp;
  const bool valid = t < nb;
  float dpos = 0.f, dneg = 0.f, su = 0.f, si = 0.f;
  if (valid) {
    const float4* fu = F + (size_t)u[t] * C::V4 + gl;
    const float4* fi = F + ((size_t)n_users + i[t]) * C::V4 + gl;
    const float4* fj = F + ((size_t)n_users + j[t]) * C::V4 + gl;
#pragma unroll
    for (int v = 0; v < C::VPL; ++v) {
      const float4 a = __ldg(fu + v * C::LPR), p = __ldg(fi + v * C::LPR), n = __ldg(fj + v * C::LPR);
      dpos += dot4(a, p);
      dneg += dot4(a, n);
      su += dot4(a, a);
      si += dot4(p, p);
    }
  }
  dpos = group_sum<C::LPR>(dpos);
  dneg = group_sum<C::LPR>(dneg);
  su = group_sum<C::LPR>(su);
  si = group_sum<C::LPR>(si);
  if (valid && gl < 4) {                                     // LPR >= 2 everywhere: 2 or 4 lanes share the stores
    const uint32_t step = xchg_ctr != nullptr ? (uint32_t)*reinterpret_cast<const volatile int32_t*>(xchg_ctr) : 0u;
    const size_t off = ((((size_t)(step & 1u) * AGCF_MAX_PEERS + rank) * cap + t) << 2);
    constexpr int STRIDE = C::LPR < 4 ? C::LPR : 4;
#pragma unroll
    for (int k = 0; k < 4 / STRIDE; ++k) {
      const int c = gl + k * STRIDE;
      const unsigned long long w = ll_pack(c == 0 ? dpos : (c == 1 ? dneg : (c == 2 ? su : si)), step + 1u);
#pragma unroll
      for (int q = 0; q < AGCF_MAX_PEERS; ++q)
        if (q < x.n) st_relaxed_sys_u64(x.p[q] + off + c, w);
    }
  }
}

__global__ void __launch_bounds__(256) bpr_finish_kernel(const unsigned long long* __restrict__ xchg, int world, int cap, int nb,
                                                         float reg, int32_t* __restrict__ xchg_ctr,
                                                         float* __restrict__ out4, float* __restrict__ coef,
                                                         BprWs* __restrict__ ws) {
  __shared__ float red[3][256];
  const int t = blockIdx.x * 256 + threadIdx.x;
  const uint32_t step = xchg_ctr != nullptr ? (uint32_t)*reinterpret_cast<const volatile int32_t*>(xchg_ctr) : 0u;
  float l = 0.f, su = 0.f, si = 0.f;
  if (t < nb) {
    float dpos = 0.f, dneg = 0.f;
    const unsigned long long t_start = global_ns();
    for (int r = 0; r < world; ++r) {                       // rank order: the same bits on every rank
      const unsigned long long* src = xchg + ((((size_t)(step & 1u) * AGCF_MAX_PEERS + r) * cap + t) << 2);
      float v[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        unsigned long long w = ld_relaxed_sys_u64(src + c);
        while ((uint32_t)(w >> 32) != step + 1u) {          // rank r's share of this triple has not landed yet
          if (global_ns() - t_start > kXchgTimeoutNs) { w = 0x7fc00000ull; break; }      // give up: NaN
          __nanosleep(40);
          w = ld_relaxed_sys_u64(src + c);
        }
        v[c] = __uint_as_float((uint32_t)w);
      }
      dpos += v[0]; dneg += v[1]; su += v[2]; si += v[3];
    }
    const float x = dpos - dneg;
    const float s = 1.f / (1.f + expf(-x));
    l = -logf(1e-7f + s);
    coef[t] = -(s * (1.f - s)) / ((1e-7f + s) * (float)nb);
  }
  red[0][threadIdx.x] = l; red[1][threadIdx.x] = su; red[2][threadIdx.x] = si;
  __syncthreads();
  bpr_finalize<256>(red, nb, reg, out4, ws, xchg_ctr);
}

// ================================================================= BPR backward
template <int D>
__global__ void __launch_bounds__(256) bpr_backward_kernel(const float4* __restrict__ F, const int32_t* __restrict__ u,
                                                           const int32_t* __restrict__ i, const int32_t* __restrict__ j,
                                                           int nb, int n_users, float reg, float scale,
                                                           const float* __restrict__ out4, const float* __restrict__ coef,
                                                           const int32_t* __restrict__ occ, const int32_t* __restrict__ seg_off,
                                                           const int32_t* __restrict__ seg_node,
                                                           const int32_t* __restrict__ n_seg, float4* __restrict__ G) {
  using C = RowCfg2<D>;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gl = lane & (C::LPR - 1), grp = lane / C::LPR;
  const int s = blockIdx.x * C::RPB + warp * C::RPW + grp;
  if (s >= __ldg(n_seg)) return;
  const int node = seg_node[s];
  const int o0 = seg_off[s], o1 = seg_off[s + 1];
  const float nu = out4[2], ni = out4[3];
  const float ru = nu > 0.f ? reg / nu : 0.f;
  const float ri = ni > 0.f ? reg / ni : 0.f;
  float4 self[C::VPL], acc[C::VPL];
#pragma unroll
  for (int v = 0; v < C::VPL; ++v) {
    self[v] = __ldg(F + (size_t)node * C::V4 + v * C::LPR + gl);
    acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (int o = o0; o < o1; ++o) {
    const int id = occ[o];
    const int role = id / nb, t = id - role * nb;
    const float c = coef[t];
    if (role == 0) {
      const float4* fi = F + ((size_t)n_users + i[t]) * C::V4 + gl;
      const float4* fj = F + ((size_t)n_users + j[t]) * C::V4 + gl;
#pragma unroll
      for (int v = 0; v < C::VPL; ++v) {
        const float4 p = __ldg(fi + v * C::LPR), n = __ldg(fj + v * C::LPR);
        acc[v].x += fmaf(c, p.x - n.x, ru * self[v].x);
        acc[v].y += fmaf(c, p.y - n.y, ru * self[v].y);
        acc[v].z += fmaf(c, p.z - n.z, ru * self[v].z);
        acc[v].w += fmaf(c, p.w - n.w, ru * self[v].w);
      }
    } else {
      const float4* fu = F + (size_t)u[t] * C::V4 + gl;
      const float cc = role == 1 ? c : -c;
      const float rr = role == 1 ? ri : 0.f;
#pragma unroll
      for (int v = 0; v < C::VPL; ++v) {
        const float4 a = __ldg(fu + v * C::LPR);
        acc[v].x += fmaf(cc, a.x, rr * self[v].x);
        acc[v].y += fmaf(cc, a.y, rr * self[v].y);
        acc[v].z += fmaf(cc, a.z, rr * self[v].z);
        acc[v].w += fmaf(cc, a.w, rr * self[v].w);
      }
    }
  }
#pragma unroll
  for (int v = 0; v < C::VPL; ++v)
    G[(size_t)node * C::V4 + v * C::LPR + gl] =
        make_float4(acc[v].x * scale, acc[v].y * scale, acc[v].z * scale, acc[v].w * scale);
}

template <int D>
__global__ void __launch_bounds__(256) zero_rows_kernel(const int32_t* __restrict__ seg_node, const int32_t* __restrict__ n_seg,
                                                        float4* __restrict__ G) {
  using C = RowCfg2<D>;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gl = lane & (C::LPR - 1), grp = lane / C::LPR;
  const int s = blockIdx.x * C::RPB + warp * C::RPW + grp;
  if (s >= __ldg(n_seg)) return;
  const int node = seg_node[s];
#pragma unroll
  for (int v = 0; v < C::VPL; ++v) G[(size_t)node * C::V4 + v * C::LPR + gl] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// ========================================================================= Adam
struct AdamPeers {
  int n;
  float* p[AGCF_MAX_PEERS];
  float* mc;        // multicast address of the same range (nullable): one store reaches every copy
};

__global__ void __launch_bounds__(256) adam_kernel(float4* __restrict__ p, const float4* __restrict__ g,
                                                   float4* __restrict__ m, float4* __restrict__ v, long long n4,
                                                   float* __restrict__ p_tail, const float* __restrict__ g_tail,
                                                   float* __restrict__ m_tail, float* __restrict__ v_tail, int n_tail,
                                                   float lr, float beta1, float beta2, float eps, int step,
                                                   const int32_t* __restrict__ step_dev, AdamPeers peers) {
  __shared__ float sh_step_size, sh_bc2_sqrt;
  if (threadIdx.x == 0) {
    const int t = step_dev != nullptr ? (*step_dev + 1) : step;
    const double bc1 = 1.0 - pow((double)beta1, (double)t);
    const double bc2 = 1.0 - pow((double)beta2, (double)t);
    sh_step_size = (float)((double)lr / bc1);
    sh_bc2_sqrt = (float)sqrt(bc2);
  }
  __syncthreads();
  const float step_size = sh_step_size, bc2_sqrt = sh_bc2_sqrt;
  const float w1 = 1.f - beta1, w2 = 1.f - beta2;
  auto upd = [&](float& pp, float gg, float& mm, float& vv) {
    mm = mm + w1 * (gg - mm);                                   // exp_avg.lerp_(grad, 1-beta1)
    vv = fmaf(w2 * gg, gg, vv * beta2);                        // mul_(beta2).addcmul_(g, g, 1-beta2)
    const float denom = __fdiv_rn(sqrtf(vv), bc2_sqrt) + eps;
    pp = pp - step_size * __fdiv_rn(mm, denom);                 // addcdiv_(m, denom, -step_size)
  };
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n4; k += stride) {
    float4 pp = p[k], mm = m[k], vv = v[k];
    const float4 gg = ld_stream_f4(g + k);
    upd(pp.x, gg.x, mm.x, vv.x);
    upd(pp.y, gg.y, mm.y, vv.y);
    upd(pp.z, gg.z, mm.z, vv.z);
    upd(pp.w, gg.w, mm.w, vv.w);
    p[k] = pp; m[k] = mm; v[k] = vv;
    if (peers.mc != nullptr) st_multicast_f4(reinterpret_cast<float4*>(peers.mc) + k, pp);
    else for (int q = 0; q < peers.n; ++q) reinterpret_cast<float4*>(peers.p[q])[k] = pp;
  }
  if (blockIdx.x == 0 && (int)threadIdx.x < n_tail) {
    float pp = p_tail[threadIdx.x], mm = m_tail[threadIdx.x], vv = v_tail[threadIdx.x];
    upd(pp, g_tail[threadIdx.x], mm, vv);
    p_tail[threadIdx.x] = pp; m_tail[threadIdx.x] = mm; v_tail[threadIdx.x] = vv;
    if (peers.mc != nullptr) asm volatile("multimem.st.weak.global.f32 [%0], %1;" :: "l"(peers.mc + n4 * 4 + threadIdx.x), "f"(pp) : "memory");
    else for (int q = 0; q < peers.n; ++q) peers.p[q][n4 * 4 + threadIdx.x] = pp;
  }
}

__global__ void increment_kernel(int32_t* c) { *c += 1; }

// same double-precision expressions as adam_kernel's thread 0
__global__ void adam_coefs_kernel(int32_t* step_dev, int increment, float lr, float beta1, float beta2, float* coefs) {
  int t = *step_dev;
  if (increment) { t += 1; *step_dev = t; }
  t += 1;
  const double bc1 = 1.0 - pow((double)beta1, (double)t);
  const double bc2 = 1.0 - pow((double)beta2, (double)t);
  coefs[0] = (float)((double)lr / bc1);
  coefs[1] = (float)sqrt(bc2);
}

// ==================================================== contrastive-loss id lists (SimGCL / XSimGCL)
// torch.unique of the batch's users and of its POSITIVE items (recommender/SimGCL.py:213-214, XSimGCL.py:40-41) from
// the grouping of agcf_bpr_group_batches: the distinct nodes are already sorted; a user node is any node < n_users, an
// item node counts if its first occurrence id (occurrences are sorted inside a segment) is a positive one
// (nb <= k < 2 nb).  One CTA per batch, ordered compaction by block scan; ids are TABLE rows (items: n_users + item).
__global__ void __launch_bounds__(1024) bpr_cl_ids_kernel(const int32_t* __restrict__ occ, const int32_t* __restrict__ seg_off,
                                                          const int32_t* __restrict__ seg_node, const int32_t* __restrict__ n_seg,
                                                          int n_triples, int batch, int n_users,
                                                          int32_t* __restrict__ cl_users, int32_t* __restrict__ cl_items,
                                                          int32_t* __restrict__ n_cl) {
  __shared__ int warp_u[32], warp_i[32];
  const int b = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int nb = min(batch, n_triples - b * batch);
  const int32_t* occ_b = occ + (size_t)b * 3 * batch;
  const int32_t* off_b = seg_off + (size_t)b * (3 * batch + 1);
  const int32_t* node_b = seg_node + (size_t)b * 3 * batch;
  const int n = n_seg[b];
  const int per = (n + nthr - 1) / nthr;
  const int lo = min(tid * per, n), hi = min(lo + per, n);
  auto kind = [&](int s) {                                    // 0 user, 1 positive item, 2 neither
    if (node_b[s] < n_users) return 0;
    return occ_b[off_b[s]] < 2 * nb ? 1 : 2;
  };
  int cu = 0, ci = 0;
  for (int s = lo; s < hi; ++s) {
    const int k = kind(s);
    cu += k == 0;
    ci += k == 1;
  }
  int iu = cu, ii = ci;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int yu = __shfl_up_sync(0xffffffffu, iu, o);
    const int yi = __shfl_up_sync(0xffffffffu, ii, o);
    if (lane >= o) { iu += yu; ii += yi; }
  }
  if (lane == 31) { warp_u[warp] = iu; warp_i[warp] = ii; }
  __syncthreads();
  if (warp == 0) {
    const int wu = lane < (nthr >> 5) ? warp_u[lane] : 0;
    const int wi = lane < (nthr >> 5) ? warp_i[lane] : 0;
    int su = wu, si = wi;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int yu = __shfl_up_sync(0xffffffffu, su, o);
      const int yi = __shfl_up_sync(0xffffffffu, si, o);
      if (lane >= o) { su += yu; si += yi; }
    }
    warp_u[lane] = su - wu;
    warp_i[lane] = si - wi;
    if (lane == 31) { n_cl[2 * b] = su; n_cl[2 * b + 1] = si; }
  }
  __syncthreads();
  int pu = warp_u[warp] + iu - cu, pi = warp_i[warp] + ii - ci;
  int32_t* out_u = cl_users + (size_t)b * batch;
  int32_t* out_i = cl_items + (size_t)b * batch;
  for (int s = lo; s < hi; ++s) {
    const int k = kind(s);
    if (k == 0) out_u[pu++] = node_b[s];
    else if (k == 1) out_i[pi++] = node_b[s];
  }
}

}  // namespace agcf

using namespace agcf;

extern "C" int agcf_bpr_sample_epoch(const int32_t* e_user, const int32_t* e_item, int32_t n_edges,
                                     const int32_t* rej_rowptr, const int32_t* rej_items, int32_t n_items,
                                     uint64_t seed, uint64_t epoch,
                                     int32_t* out_u, int32_t* out_i, int32_t* out_j, agcf_stream_t stream) {
  if (!e_user || !e_item || !rej_rowptr || !out_u || !out_i || !out_j || n_edges < 0 || n_items <= 0) return AGCF_EINVAL;
  if (n_edges == 0) return AGCF_OK;
  int bits = 2;
  while ((1ll << bits) < (long long)n_edges) ++bits;
  if (bits & 1) ++bits;                                      // balanced Feistel needs an even width
  if (bits > 32) return AGCF_EUNSUPPORTED;
  const unsigned blocks = (unsigned)((n_edges + 255) / 256);
  bpr_sample_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(e_user, e_item, n_edges, rej_rowptr, rej_items, n_items,
                                                              seed, epoch, bits / 2, out_u, out_i, out_j);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int agcf_bpr_group_batches(const int32_t* u, const int32_t* i, const int32_t* j,
                                      int32_t n_triples, int32_t batch, int32_t n_users,
                                      int32_t* occ, int32_t* seg_off, int32_t* seg_node, int32_t* n_seg,
                                      int32_t n_nodes, uint32_t* node_mask, agcf_stream_t stream) {
  if (!u || !i || !j || !occ || !seg_off || !seg_node || !n_seg || n_triples < 0 || batch <= 0 || n_users < 0) return AGCF_EINVAL;
  if (node_mask != nullptr && n_nodes <= 0) return AGCF_EINVAL;
  if (n_triples == 0) return AGCF_OK;
  if (3 * (long long)batch > 16384) return AGCF_EUNSUPPORTED;
  int pow2 = 1024;
  while (pow2 < 3 * batch) pow2 <<= 1;
  const size_t smem = (size_t)pow2 * sizeof(unsigned long long);
  static thread_local bool attr_set = false;                  // opt in to > 48 KB dynamic smem once
  if (!attr_set) {
    AGCF_CUDA_OK(cudaFuncSetAttribute(bpr_group_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 * 8));
    attr_set = true;
  }
  const unsigned blocks = (unsigned)((n_triples + batch - 1) / batch);
  bpr_group_kernel<<<blocks, 1024, smem, (cudaStream_t)stream>>>(u, i, j, n_triples, batch, n_users, pow2,
                                                                 occ, seg_off, seg_node, n_seg, (n_nodes + 31) / 32, node_mask);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int agcf_bpr_cl_ids(const int32_t* occ, const int32_t* seg_off, const int32_t* seg_node, const int32_t* n_seg,
                               int32_t n_triples, int32_t batch, int32_t n_users,
                               int32_t* cl_users, int32_t* cl_items, int32_t* n_cl, agcf_stream_t stream) {
  if (!occ || !seg_off || !seg_node || !n_seg || !cl_users || !cl_items || !n_cl) return AGCF_EINVAL;
  if (n_triples < 0 || batch <= 0 || n_users < 0 || 3 * (long long)batch > 16384) return AGCF_EINVAL;
  if (n_triples == 0) return AGCF_OK;
  const unsigned blocks = (unsigned)((n_triples + batch - 1) / batch);
  bpr_cl_ids_kernel<<<blocks, 1024, 0, (cudaStream_t)stream>>>(occ, seg_off, seg_node, n_seg, n_triples, batch, n_users,
                                                               cl_users, cl_items, n_cl);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int64_t agcf_bpr_ws_bytes(int32_t nb) {
  if (nb < 0) return AGCF_EINVAL;
  return 64 + 12ll * ((long long)nb / 8 + 2);
}

extern "C" int agcf_bpr_forward(const float* F, const int32_t* u, const int32_t* i, const int32_t* j,
                                int32_t nb, int32_t n_users, int32_t d, float reg,
                                float* out4, float* coef, void* ws, agcf_stream_t stream) {
  if (!F || !u || !i || !j || !out4 || !coef || !ws || nb <= 0 || n_users < 0) return AGCF_EINVAL;
  if (!supported_d(d)) return AGCF_EUNSUPPORTED;
  if (!aligned16(F) || !aligned16(ws)) return AGCF_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  const float4* F4 = reinterpret_cast<const float4*>(F);
  BprWs* w = reinterpret_cast<BprWs*>(ws);
#define AGCF_BPRF(DD)                                                                         \
  {                                                                                           \
    const unsigned blocks = (unsigned)((nb + RowCfg2<DD>::RPB - 1) / RowCfg2<DD>::RPB);        \
    bpr_forward_kernel<DD><<<blocks, 256, 0, st>>>(F4, u, i, j, nb, n_users, reg, out4, coef, w); \
  }
  switch (d) {
    case 8: AGCF_BPRF(8) break;
    case 16: AGCF_BPRF(16) break;
    case 32: AGCF_BPRF(32) break;
    case 64: AGCF_BPRF(64) break;
    case 128: AGCF_BPRF(128) break;
    case 256: AGCF_BPRF(256) break;
  }
#undef AGCF_BPRF
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int64_t agcf_bpr_xchg_bytes(int32_t cap) {
  if (cap < 0) return AGCF_EINVAL;
  return 2ll * AGCF_MAX_PEERS * (long long)cap * 32;       // 2 halves x ranks x cap x 4 words {stamp | value}
}

extern "C" int agcf_bpr_partial(const float* F, const int32_t* u, const int32_t* i, const int32_t* j,
                                int32_t nb, int32_t n_users, int32_t d, int32_t rank, int32_t cap,
                                const int32_t* xchg_ctr, void* const* xchg_all_host, int32_t world,
                                agcf_stream_t stream) {
  if (!F || !u || !i || !j || nb <= 0 || n_users < 0 || !xchg_all_host) return AGCF_EINVAL;
  if (world < 1 || world > AGCF_MAX_PEERS || rank < 0 || rank >= world || nb > cap) return AGCF_EINVAL;
  if (!supported_d(d)) return AGCF_EUNSUPPORTED;
  if (!aligned16(F)) return AGCF_EINVAL;
  XchgPeers x;
  x.n = world;
  for (int q = 0; q < AGCF_MAX_PEERS; ++q) {
    x.p[q] = q < world ? reinterpret_cast<unsigned long long*>(xchg_all_host[q]) : nullptr;
    if (q < world && (x.p[q] == nullptr || !aligned16(x.p[q]))) return AGCF_EINVAL;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const float4* F4 = reinterpret_cast<const float4*>(F);
#define AGCF_BPRP(DD)                                                                              \
  {                                                                                                \
    const unsigned blocks = (unsigned)((nb + RowCfg2<DD>::RPB - 1) / RowCfg2<DD>::RPB);             \
    bpr_partial_kernel<DD><<<blocks, 256, 0, st>>>(F4, u, i, j, nb, n_users, rank, cap, xchg_ctr, x); \
  }
  switch (d) {
    case 8: AGCF_BPRP(8) break;
    case 16: AGCF_BPRP(16) break;
    case 32: AGCF_BPRP(32) break;
    case 64: AGCF_BPRP(64) break;
    case 128: AGCF_BPRP(128) break;
    case 256: AGCF_BPRP(256) break;
  }
#undef AGCF_BPRP
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int agcf_bpr_finish(const void* xchg, int32_t world, int32_t cap, int32_t nb, float reg,
                               int32_t* xchg_ctr, float* out4, float* coef, void* ws, agcf_stream_t stream) {
  if (!xchg || !out4 || !coef || !ws || nb <= 0 || nb > cap || world < 1 || world > AGCF_MAX_PEERS) return AGCF_EINVAL;
  if (!aligned16(xchg) || !aligned16(ws)) return AGCF_EINVAL;
  const unsigned blocks = (unsigned)((nb + 255) / 256);
  bpr_finish_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const unsigned long long*>(xchg), world, cap, nb, reg,
                                                              xchg_ctr, out4, coef, reinterpret_cast<BprWs*>(ws));
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int agcf_bpr_backward(const float* F, const int32_t* u, const int32_t* i, const int32_t* j,
                                 int32_t nb, int32_t n_users, int32_t d, float reg, float scale,
                                 const float* out4, const float* coef,
                                 const int32_t* occ, const int32_t* seg_off, const int32_t* seg_node,
                                 const int32_t* n_seg, float* G, agcf_stream_t stream) {
  if (!F || !u || !i || !j || !out4 || !coef || !occ || !seg_off || !seg_node || !n_seg || !G || nb <= 0) return AGCF_EINVAL;
  if (!supported_d(d)) return AGCF_EUNSUPPORTED;
  if (!aligned16(F) || !aligned16(G) || F == G) return AGCF_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  const float4* F4 = reinterpret_cast<const float4*>(F);
  float4* G4 = reinterpret_cast<float4*>(G);
#define AGCF_BPRB(DD)                                                                              \
  {                                                                                                \
    const unsigned blocks = (unsigned)((3 * nb + RowCfg2<DD>::RPB - 1) / RowCfg2<DD>::RPB);        \
    bpr_backward_kernel<DD><<<blocks, 256, 0, st>>>(F4, u, i, j, nb, n_users, reg, scale, out4, coef, \
                                                    occ, seg_off, seg_node, n_seg, G4);            \
  }
  switch (d) {
    case 8: AGCF_BPRB(8) break;
    case 16: AGCF_BPRB(16) break;
    case 32: AGCF_BPRB(32) break;
    case 64: AGCF_BPRB(64) break;
    case 128: AGCF_BPRB(128) break;
    case 256: AGCF_BPRB(256) break;
  }
#undef AGCF_BPRB
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int agcf_zero_rows(const int32_t* seg_node, const int32_t* n_seg, int32_t max_seg,
                              float* G, int32_t d, agcf_stream_t stream) {
  if (!seg_node || !n_seg || !G || max_seg < 0) return AGCF_EINVAL;
  if (!supported_d(d)) return AGCF_EUNSUPPORTED;
  if (!aligned16(G)) return AGCF_EINVAL;
  if (max_seg == 0) return AGCF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  float4* G4 = reinterpret_cast<float4*>(G);
#define AGCF_ZR(DD)                                                                          \
  {                                                                                          \
    const unsigned blocks = (unsigned)((max_seg + RowCfg2<DD>::RPB - 1) / RowCfg2<DD>::RPB);  \
    zero_rows_kernel<DD><<<blocks, 256, 0, st>>>(seg_node, n_seg, G4);                       \
  }
  switch (d) {
    case 8: AGCF_ZR(8) break;
    case 16: AGCF_ZR(16) break;
    case 32: AGCF_ZR(32) break;
    case 64: AGCF_ZR(64) break;
    case 128: AGCF_ZR(128) break;
    case 256: AGCF_ZR(256) break;
  }
#undef AGCF_ZR
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int agcf_adam_step_f32(float* p, const float* g, float* m, float* v, int64_t n,
                                  float lr, float beta1, float beta2, float eps,
                                  int32_t step, const int32_t* step_dev,
                                  void* const* peer_p_host, int32_t n_peers, void* mc_p, agcf_stream_t stream) {
  if (!p || !g || !m || !v || n < 0) return AGCF_EINVAL;
  if (!aligned16(mc_p)) return AGCF_EINVAL;
  if (n_peers < 0 || n_peers > AGCF_MAX_PEERS || (n_peers > 0 && !peer_p_host)) return AGCF_EINVAL;
  AdamPeers peers;
  peers.n = n_peers;
  peers.mc = reinterpret_cast<float*>(mc_p);
  for (int q = 0; q < AGCF_MAX_PEERS; ++q) peers.p[q] = q < n_peers ? reinterpret_cast<float*>(peer_p_host[q]) : nullptr;
  if (step_dev == nullptr && step < 1) return AGCF_EINVAL;
  if (!aligned16(p) || !aligned16(g) || !aligned16(m) || !aligned16(v)) return AGCF_EINVAL;
  if (n == 0) return AGCF_OK;
  const long long n4 = n / 4;
  const int n_tail = (int)(n - n4 * 4);
  long long blocks = (n4 + 255) / 256;
  if (blocks > kSMs * 8) blocks = kSMs * 8;
  if (blocks < 1) blocks = 1;
  adam_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<float4*>(p), reinterpret_cast<const float4*>(g), reinterpret_cast<float4*>(m),
      reinterpret_cast<float4*>(v), n4, p + n4 * 4, g + n4 * 4, m + n4 * 4, v + n4 * 4, n_tail,
      lr, beta1, beta2, eps, step, step_dev, peers);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int agcf_adam_coefs(int32_t* step_dev, int32_t increment, float lr, float beta1, float beta2, float* coefs,
                               agcf_stream_t stream) {
  if (!step_dev || !coefs) return AGCF_EINVAL;
  adam_coefs_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(step_dev, increment, lr, beta1, beta2, coefs);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int agcf_increment_i32(int32_t* counter, agcf_stream_t stream) {
  if (!counter) return AGCF_EINVAL;
  increment_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(counter);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}
