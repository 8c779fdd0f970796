// propagate.cu -- normalized-adjacency propagation for graph-CF encoders on B200.
//
//   agcf_norm_adj_csr      values of D^-1/2 A D^-1/2 (bit-exact association)
//   agcf_spmm_csr_f32      Y = A X with fused layer-sum / addend / noise epilogue
//   agcf_sddmm_csr_f32     pattern-masked dL/dA
//   agcf_concat_rows_f32   [user_emb; item_emb] packing
//
// Reference call sites: recommender/LightGCN.py:230-240 (forward), its autograd
// (backward), recommender/SimGCL.py:198-210, XSimGCL.py:205-223 (noise),
// attack/White/PGA.py:97-117 (adjacency gradient), util/DataLoader.py:73-87 and
// recommender/LightGCN.py:212-215 (normalization).
//
// SpMM design (L2-gather bound, no tensor cores -- see DESIGN.md):
//   * a row of X is d fp32 = d/4 float4; LPR = min(d/4, 32) lanes own one row and
//     each lane loads 16 B, so one warp-level LDG.128 fetches whole 128 B lines of
//     32/LPR different neighbour rows (fully coalesced sectors);
//   * the unit of work is a SEGMENT of a row (at most 64 non-zeros, host plan `vrows`):
//     one lane group per segment, segments sorted by length so the groups of a warp
//     walk equally long ones.  A hub row is dozens of independent work items instead
//     of one long pole (that pole set a ~21 us floor under every launch, however few
//     rows a rank owned);
//   * col/val of a segment are read 16 at a time, coalesced, and broadcast by shuffle;
//     the 16 slots of a chunk are unrolled and predicated;
//   * rows with several segments: every segment stores its partial sum, the one that
//     arrives last (a ticket per row) adds the partials in segment order and runs the
//     epilogue -- no floating-point atomics, run-to-run deterministic;
//   * epilogue fuses: + addend (backward's G/(L+1)), SimGCL noise, Y store, the
//     running layer sum / mean (acc_out = (acc_in + t) / acc_div) and the stores to
//     the other GPUs (P2P or one NVSwitch multicast store).
#include "common.cuh"
#include <stdlib.h>

namespace agcf {

struct SpmmParams {
  const int4* vrows;          // work items {start, len, row, k | nseg << 16}
  const int32_t* vpart;       // first partial slot of the item's row (rows with nseg > 1)
  int32_t n_v;
  const int32_t* n_v_dev;     // nullable: device-side item count (per-batch work lists), clamps n_v
  int32_t* sched;             // nullable: {next block, CTAs done}, zero between launches -> persistent CTAs that take
                              // blocks of RPB items dynamically (no CTA turnover gaps, no tail of idle SMs)
  float4* partial;            // [n_partial][d/4] partial sums of multi-segment rows
  int32_t* tickets;           // [n_partial], zero between launches
  const int32_t* col;
  const float* val;
  const float4* X;
  float4* Y;
  const float4* addend;
  const float4* acc_in;
  float4* acc_out;
  float acc_div;
  const float4* noise;
  float eps;
  // in-kernel noise (noise == nullptr, noise_seed != 0): U[0,1) from Philox4x32-10, key = seed, counter =
  // (float4 slot of the element, step << 32 | stream) -- nothing is read, a replayed graph draws fresh noise every step
  unsigned long long noise_seed;
  uint32_t noise_stream;
  const int32_t* noise_step;
  int noise_main;             // perturb the main outputs (Y / acc_out) with the Philox stream `noise_stream`
  // up to two extra outputs aux_Y[q] = t perturbed with their OWN noise (table aux_noise[q], else Philox stream
  // aux_stream[q]): SimGCL's clean pass and its two perturbed passes share A E0, one launch writes all three
  float4* aux_Y[2];
  const float4* aux_noise[2];
  uint32_t aux_stream[2];
  const uint32_t* row_mask;   // nullable bitmap over rows: only rows with their bit set are computed / written
  const uint32_t* col_mask;   // nullable bitmap over columns: rows of X outside it are known to be zero (skipped)
  int mask_bits;              // bits in the bitmaps (0 = unknown)
  // fused all-gather: the same rows are also stored into the peer GPUs' copies of Y / acc_out
  // (NVLink P2P stores straight from the epilogue; peers see them after the next barrier)
  int n_peers;
  float4* peer_Y[AGCF_MAX_PEERS];
  float4* peer_acc[AGCF_MAX_PEERS];
  // NVSwitch multicast addresses of Y / acc_out (nullable): ONE multimem.st reaches every GPU's copy, so a
  // rank's egress per layer is its own rows once instead of once per peer
  float4* mc_Y;
  float4* mc_acc;
  // fused optimizer (last backward layer): the row's gradient o = (acc_in + t) / acc_div goes straight into
  // torch.optim.Adam's update of p / m / v; coefs = {lr / (1 - b1^t), sqrt(1 - b2^t)} (agcf_adam_coefs)
  float4* adam_p;
  float4* adam_m;
  float4* adam_v;
  const float* adam_coefs;
  float beta1, beta2, adam_eps;
  float4* zero_rows;          // nullable (== acc_in): rows of acc_in that were non-zero (AMASK: in addend_mask) are zeroed
  // nullable bitmap over rows (AMASK launches): rows of addend / acc_in outside it are exactly zero -- not loaded, +0.0f is
  // added instead.  The backward gradient G is non-zero only at the batch's <= 3B rows (~8 % at the Gowalla shape)
  const uint32_t* addend_mask;
  // layer sum formed in the epilogue (TERMS launches only, acc_in == nullptr): acc_in's row is replaced by
  // ((acc_terms[0] + acc_terms[1]) + ...) -- the running sum the earlier layers would have written, same adds in the
  // same order -- so those layers write only their Y and the sum is formed only at the rows this launch computes
  const float4* acc_terms[AGCF_MAX_ACC_TERMS];
  int n_acc_terms;
};

__device__ __forceinline__ bool bit_set(const uint32_t* __restrict__ m, int k) {
  return (__ldg(m + (k >> 5)) >> (k & 31)) & 1u;
}

// lanes per row: one float4 per lane up to d = 64.  d = 128 rows are held by 16 lanes x 2 float4 (AGCF_SPMM_LPR128, tuning
// builds override it): a warp per row meant 2.5x the work items per non-zero of the d = 64 mapping and their fixed costs --
// measured on B200, Amazon-book shape: 315 us (32 lanes, 3 CTAs / SM) -> 249 us (16 lanes, 3 CTAs) -> 215 us (16 lanes, 4 CTAs)
#ifndef AGCF_SPMM_LPR128
#define AGCF_SPMM_LPR128 16
#endif
#ifndef AGCF_SPMM_LPR64
#define AGCF_SPMM_LPR64 16
#endif
#define AGCF_SPMM_CM_THREADS_MAX 256               // largest CTA any SpMM kernel is launched with
constexpr int default_lpr(int d) { return d == 128 ? AGCF_SPMM_LPR128 : (d == 64 ? AGCF_SPMM_LPR64 : (d / 4 < 32 ? d / 4 : 32)); }

template <int D, int LPR_ = default_lpr(D)>
struct RowCfg {
  static constexpr int V4 = D / 4;                    // float4 per row
  static constexpr int LPR = LPR_;                    // lanes per row
  static constexpr int VPL = V4 / LPR;                // float4 per lane
  static constexpr int RPW = 32 / LPR;                // rows per warp
  static constexpr int EPL = LPR >= 16 ? 1 : 16 / LPR;  // col/val entries per lane and chunk
  static constexpr int CH = LPR * EPL;                // entries per chunk: >= 16 gathers in flight per lane group
  static constexpr int THREADS = 256;
  static constexpr int RPB = (THREADS / 32) * RPW;    // rows per block (short path)
  static constexpr int GROUPS = THREADS / LPR;        // lane groups per block (long path)
  static_assert(V4 % LPR == 0 && LPR <= 32 && VPL >= 1, "bad lane mapping");
};

__device__ __forceinline__ float sgnf(float x) { return (float)((x > 0.f) - (x < 0.f)); }

// one Adam update (torch.optim.Adam defaults), same operation order as adam_kernel in bpr.cu
__device__ __forceinline__ void adam_update(float& pp, float gg, float& mm, float& vv, float w1, float w2, float beta2,
                                            float step_size, float bc2_sqrt, float eps) {
  mm = mm + w1 * (gg - mm);
  vv = fmaf(w2 * gg, gg, vv * beta2);
  const float denom = __fdiv_rn(sqrtf(vv), bc2_sqrt) + eps;
  pp = pp - step_size * __fdiv_rn(mm, denom);
}

// t += sign(t) * normalize(noise) * eps for one row held by a lane group (recommender/SimGCL.py:204-205); the U[0,1)
// noise row comes from a table or from Philox (key = seed, counter = (float4 slot, step << 32 | stream)).  Every lane
// of the warp must call it (the row norm is a lane-group reduction); invalid rows see zero noise.
template <typename C>
__device__ __forceinline__ void spmm_perturb(const SpmmParams& p, size_t rbase, bool valid, int gl,
                                             const float4* __restrict__ noise_tab, uint32_t stream, float4 (&t)[C::VPL]) {
  float4 nz[C::VPL];
  float ss = 0.f;
  unsigned long long ctr_hi = 0ull;
  if (noise_tab == nullptr)
    ctr_hi = ((unsigned long long)(uint32_t)(p.noise_step != nullptr ? __ldg(p.noise_step) : 0) << 32) | stream;
#pragma unroll
  for (int v = 0; v < C::VPL; ++v) {
    nz[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) {
      if (noise_tab != nullptr) {
        nz[v] = ld_stream_f4(noise_tab + rbase + v * C::LPR + gl);
      } else {
        uint32_t r4[4];
        Philox::gen(p.noise_seed, (unsigned long long)(rbase + v * C::LPR + gl), ctr_hi, r4);
        nz[v] = make_float4((float)(r4[0] >> 8) * 5.9604644775390625e-8f, (float)(r4[1] >> 8) * 5.9604644775390625e-8f,
                            (float)(r4[2] >> 8) * 5.9604644775390625e-8f, (float)(r4[3] >> 8) * 5.9604644775390625e-8f);
      }
    }
    ss += dot4(nz[v], nz[v]);
  }
  ss = group_sum<C::LPR>(ss);
  const float nrm = fmaxf(sqrtf(ss), 1e-12f);   // F.normalize(dim=-1, eps=1e-12)
#pragma unroll
  for (int v = 0; v < C::VPL; ++v) {
    t[v].x = t[v].x + __fmul_rn(__fmul_rn(sgnf(t[v].x), __fdiv_rn(nz[v].x, nrm)), p.eps);
    t[v].y = t[v].y + __fmul_rn(__fmul_rn(sgnf(t[v].y), __fdiv_rn(nz[v].y, nrm)), p.eps);
    t[v].z = t[v].z + __fmul_rn(__fmul_rn(sgnf(t[v].z), __fdiv_rn(nz[v].z, nrm)), p.eps);
    t[v].w = t[v].w + __fmul_rn(__fmul_rn(sgnf(t[v].w), __fdiv_rn(nz[v].w, nrm)), p.eps);
  }
}

// live: the row's bit of addend_mask (AMASK launches; always true otherwise)
template <typename C, bool NOISE, bool TERMS = false, bool AMASK = false>
__device__ __forceinline__ void spmm_epilogue(const SpmmParams& p, int row, bool valid, bool live,
                                              float4 (&t)[C::VPL], int gl, const float4* pre_add = nullptr) {
  const size_t rbase = (size_t)row * C::V4;
  if (p.addend != nullptr && valid) {
    // a row outside addend_mask adds +0.0f: -0.0f + +0.0f is +0.0f, the bits of adding the zero row
#pragma unroll
    for (int v = 0; v < C::VPL; ++v)
      t[v] = add4(t[v], pre_add != nullptr ? pre_add[v]
                        : (live ? ld_stream_f4(p.addend + rbase + v * C::LPR + gl) : make_float4(0.f, 0.f, 0.f, 0.f)));
  }
  if (NOISE) {
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      if (p.aux_Y[q] == nullptr) continue;
      float4 tq[C::VPL];
#pragma unroll
      for (int v = 0; v < C::VPL; ++v) tq[v] = t[v];
      spmm_perturb<C>(p, rbase, valid, gl, p.aux_noise[q], p.aux_stream[q], tq);
      if (valid) {
#pragma unroll
        for (int v = 0; v < C::VPL; ++v) p.aux_Y[q][rbase + v * C::LPR + gl] = tq[v];
      }
    }
    if (p.noise != nullptr || p.noise_main) spmm_perturb<C>(p, rbase, valid, gl, p.noise, p.noise_stream, t);
  }
  if (!valid) return;
  if (p.Y != nullptr) {
#pragma unroll
    for (int v = 0; v < C::VPL; ++v) p.Y[rbase + v * C::LPR + gl] = t[v];
    if (p.mc_Y != nullptr) {
#pragma unroll
      for (int v = 0; v < C::VPL; ++v) st_multicast_f4(p.mc_Y + rbase + v * C::LPR + gl, t[v]);
    } else {
      for (int q = 0; q < p.n_peers; ++q) {
        if (p.peer_Y[q] == nullptr) continue;
#pragma unroll
        for (int v = 0; v < C::VPL; ++v) p.peer_Y[q][rbase + v * C::LPR + gl] = t[v];
      }
    }
  }
  if (p.acc_out != nullptr || p.adam_p != nullptr) {
    float step_size = 0.f, bc2_sqrt = 1.f;
    if (p.adam_p != nullptr) { step_size = __ldg(p.adam_coefs); bc2_sqrt = __ldg(p.adam_coefs + 1); }
#pragma unroll
    for (int v = 0; v < C::VPL; ++v) {
      const size_t at = rbase + v * C::LPR + gl;
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
      if constexpr (TERMS) {
        // four rows requested together per round trip (L <= 4: one), added in table order
        for (int q0 = 0; q0 < p.n_acc_terms; q0 += 4) {
          float4 term[4];
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (q0 + q < p.n_acc_terms) term[q] = ld_stream_f4(p.acc_terms[q0 + q] + at);
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (q0 + q < p.n_acc_terms) a = q0 + q == 0 ? term[0] : add4(a, term[q]);
        }
      } else if (p.acc_in != nullptr && live) {
        // (a table this kernel also writes must not go through the non-coherent path)
        a = p.zero_rows != nullptr ? __ldcg(p.acc_in + at) : ld_stream_f4(p.acc_in + at);
        // the batch's gradient rows are the only non-zero rows of G: put them back to zero for the next step
        if (!AMASK && p.zero_rows != nullptr && (a.x != 0.f || a.y != 0.f || a.z != 0.f || a.w != 0.f))
          p.zero_rows[at] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      float4 o = add4(a, t[v]);
      if (p.acc_div != 1.0f) {
        o.x = __fdiv_rn(o.x, p.acc_div); o.y = __fdiv_rn(o.y, p.acc_div);
        o.z = __fdiv_rn(o.z, p.acc_div); o.w = __fdiv_rn(o.w, p.acc_div);
      }
      if (p.acc_out != nullptr) {
        p.acc_out[at] = o;
        if (p.mc_acc != nullptr) {
          st_multicast_f4(p.mc_acc + at, o);
        } else {
          for (int q = 0; q < p.n_peers; ++q)
            if (p.peer_acc[q] != nullptr) p.peer_acc[q][at] = o;
        }
      }
      if (p.adam_p != nullptr) {
        // the moments are touched once per step: evict-first loads / stores, so that 36 MB of them do not push the layer
        // tables out of L2 (0.2499 -> 0.2480 ms per step at C2, two runs each); the parameters are read again right away
        float4 pp = p.adam_p[at], mm = __ldcs(p.adam_m + at), vv = __ldcs(p.adam_v + at);
        const float w1 = 1.f - p.beta1, w2 = 1.f - p.beta2;
        adam_update(pp.x, o.x, mm.x, vv.x, w1, w2, p.beta2, step_size, bc2_sqrt, p.adam_eps);
        adam_update(pp.y, o.y, mm.y, vv.y, w1, w2, p.beta2, step_size, bc2_sqrt, p.adam_eps);
        adam_update(pp.z, o.z, mm.z, vv.z, w1, w2, p.beta2, step_size, bc2_sqrt, p.adam_eps);
        adam_update(pp.w, o.w, mm.w, vv.w, w1, w2, p.beta2, step_size, bc2_sqrt, p.adam_eps);
        p.adam_p[at] = pp; __stcs(p.adam_m + at, mm); __stcs(p.adam_v + at, vv);
      }
      // AMASK: every row of the bitmap is put back to zero, whatever it held (a -0.0f gradient does not outlive its step
      // either).  Last, after the optimizer's stores: with no store ahead of them, the loads of p / m / v need not wait
      // for it, and at the ~92 % of rows that read no gradient they are the epilogue's only round trip.  Requesting them
      // together with the gradient row instead (ahead of the acc_out store too) measured slower: 65.1 vs 60.7 us per
      // fused launch at the Gowalla shape (profiles/r4_summary.md)
      if (AMASK && p.zero_rows != nullptr && live) p.zero_rows[at] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
}

// accumulate nnz [s + first, s + first + stride*k ...) chunk-wise; `len` = row length,
// `first`/`stride` = this lane group's starting offset and per-iteration advance,
// `iters` is WARP-UNIFORM (shuffles use the full mask).  A lane group walks its row in chunks of CH = LPR * EPL entries: lane gl holds
// entries k * LPR + gl (k < EPL) of the chunk -- consecutive lanes read consecutive col/val words --
// and every entry is broadcast by shuffle; the CH slots are fully unrolled and predicated, so up to CH
// independent row gathers are in flight per lane while the next chunk's indices are already loading.
// For narrow rows (d/4 < 16 lanes, the d-sharded multi-GPU tables) EPL > 1 keeps CH at 16.
// one chunk held in registers (lane gl owns entries k * LPR + gl): broadcast every entry to the lane group and
// gather-accumulate its row of X; slots with col < 0 (row end, masked column) are predicated off
// Rows of two float4 per lane (d = 128 / 256): the (col, val) pairs of a lane group's chunk reach its lanes through shared
// memory instead of 2 shuffles per entry -- every lane stores its pair (one STS.64 per warp), one LDS.128 then hands TWO
// entries to the whole group (the address is uniform per group: a broadcast).  Shuffles and shared loads are both
// wavefronts of the LSU data pipe, which the profile shows ~70 % busy with the gathers' data returns; per 32 entries of a
// warp this is 9 wavefronts instead of 32 and the chunk loop 125 instead of 205 instructions.  Same values, same order:
// bit-identical.  Measured on B200 (profiles/r2_summary.md section 9): Amazon-book shape d = 128 233 -> 209 us per full
// launch, 61 -> 51 us row-masked, 1.10 -> 1.053 ms per training step; at d = 64 (one float4 per lane) it is slower than
// the shuffles (46.8 vs 43.6 us), so those rows keep them.  A double-buffered form that stores chunk k + 1's pairs at the
// end of chunk k's iteration (the STS -> LDS hop off the gather path) measured WORSE at both widths (d = 128: 214 us and
// 1.097 ms per step; d = 64: 45.2 us): the next chunk's index registers stay live across the gathers and spill.  Columns
// and values in separate shared arrays (four entries per LDS.128, the column quad dead once its gathers are issued)
// measured equal stand-alone and slower in the step at both widths (profiles/r2_spmm_smem_split.txt).
#ifndef AGCF_SPMM_SMEM_BCAST_MIN_VPL
#define AGCF_SPMM_SMEM_BCAST_MIN_VPL 2
#endif
template <typename C>
constexpr bool spmm_smem_bcast() { return C::EPL == 1 && C::VPL >= AGCF_SPMM_SMEM_BCAST_MIN_VPL && C::LPR >= 16; }

template <typename C, bool PACKED>
__device__ __forceinline__ void spmm_consume_chunk(const SpmmParams& p, const int (&c)[C::EPL], const float (&v)[C::EPL],
                                                   int gl, float4 (&acc)[C::VPL]) {
  if constexpr (spmm_smem_bcast<C>()) {
    __shared__ __align__(16) int2 s_bcast[(AGCF_SPMM_CM_THREADS_MAX / 32) * 32];
    int2* mine = s_bcast + (threadIdx.x & ~31);
    const int lane = threadIdx.x & 31;
    __syncwarp();                                          // the previous chunk's pairs are no longer read
    mine[lane] = make_int2(c[0], __float_as_int(v[0]));
    __syncwarp();
    const int4* row = reinterpret_cast<const int4*>(mine + (lane & ~(C::LPR - 1)));
#pragma unroll
    for (int t2 = 0; t2 < C::CH / 2; ++t2) {
      const int4 two = row[t2];                            // entries 2 t2 and 2 t2 + 1 of this group's chunk
      if (two.x >= 0) {
        const float4* xr = p.X + (size_t)two.x * C::V4 + gl;
#pragma unroll
        for (int vv = 0; vv < C::VPL; ++vv) fma4_packed(acc[vv], __int_as_float(two.y), ld_gather_f4(xr + vv * C::LPR));
      }
      if (two.z >= 0) {
        const float4* xr = p.X + (size_t)two.z * C::V4 + gl;
#pragma unroll
        for (int vv = 0; vv < C::VPL; ++vv) fma4_packed(acc[vv], __int_as_float(two.w), ld_gather_f4(xr + vv * C::LPR));
      }
    }
  } else {
#pragma unroll
    for (int k = 0; k < C::EPL; ++k) {
#pragma unroll
      for (int t = 0; t < C::LPR; ++t) {
        const int ct = __shfl_sync(0xffffffffu, c[k], t, C::LPR);
        const float vt = __shfl_sync(0xffffffffu, v[k], t, C::LPR);
        if (ct >= 0) {
          const float4* xr = p.X + (size_t)ct * C::V4 + gl;
#pragma unroll
          for (int vv = 0; vv < C::VPL; ++vv) {
            if (PACKED) fma4_packed(acc[vv], vt, ld_gather_f4(xr + vv * C::LPR));
            else fma4(acc[vv], vt, ld_gather_f4(xr + vv * C::LPR));
          }
        }
      }
    }
  }
}

template <typename C, bool PACKED>
__device__ __forceinline__ void spmm_accumulate_chunks(const SpmmParams& p, int s, int len, int first, int stride,
                                                       int iters, int gl, float4 (&acc)[C::VPL]) {
  int c_next[C::EPL];
  float v_next[C::EPL];
  auto load_chunk = [&](int off) {
#pragma unroll
    for (int k = 0; k < C::EPL; ++k) {
      c_next[k] = -1;
      v_next[k] = 0.f;
      const int e = off + k * C::LPR + gl;
      if (e < len) {
        // narrow rows (EPL > 1): a lane group covers only LPR * 4 bytes per load, so the EPL loads of a chunk
        // touch the same 32-byte sectors again and again -- let L1 keep them; wide rows stream past L1
        c_next[k] = C::EPL > 1 ? __ldg(p.col + s + e) : ld_stream_i32(p.col + s + e);
        v_next[k] = C::EPL > 1 ? __ldg(p.val + s + e) : ld_stream_f32(p.val + s + e);
        if (p.col_mask != nullptr && !bit_set(p.col_mask, c_next[k])) c_next[k] = -1;
      }
    }
  };
  load_chunk(first);
  int off = first;
  for (int it = 0; it < iters; ++it, off += stride) {
    int c[C::EPL];
    float v[C::EPL];
#pragma unroll
    for (int k = 0; k < C::EPL; ++k) { c[k] = c_next[k]; v[k] = v_next[k]; }
    load_chunk(off + stride);                              // prefetch the next chunk's indices
    spmm_consume_chunk<C, PACKED>(p, c, v, gl, acc);
  }
}

#ifdef AGCF_SPMM_TRACE
// tuning aid (never in the shipped build): per-CTA timeline of the last launch -- start, metadata arrived,
// gathers accumulated, end (globaltimer ns, warp 0) and the SM id
__device__ unsigned long long g_spmm_trace[6 * 16384];
__device__ __forceinline__ unsigned long long trace_now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void trace_put(int blk, int k, unsigned long long v) {
  if (threadIdx.x == 0 && blk < 16384) g_spmm_trace[6 * blk + k] = v;
}
struct TraceScope {
  int blk;
  __device__ explicit TraceScope(int b) : blk(b) { trace_put(blk, 0, trace_now()); }
  __device__ ~TraceScope() {
    unsigned int sm;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
    trace_put(blk, 3, trace_now());
    trace_put(blk, 4, sm);
  }
};
extern "C" int agcf_debug_spmm_trace(unsigned long long* host_out) {
  return cudaMemcpyFromSymbol(host_out, g_spmm_trace, sizeof(g_spmm_trace)) == cudaSuccess ? 0 : -3;
}
#define AGCF_TRACE_AFTER(k, dep) trace_put(blk, k, trace_now() + ((dep) == 0x7fffff01 ? 1ull : 0ull))
#else
#define AGCF_TRACE_AFTER(k, dep)
#endif

// Column-masked accumulation (first backward layer: only the <= 3B gradient rows of the batch are non-zero, ~13 % of
// the non-zeros at the benchmark shape).  A chunk is LPR entries, one per lane; the lanes whose column is in the
// mask are found with a ballot and ONLY those are broadcast, gathered and accumulated, in entry order -- the same
// order as the dense loop, hence the same bits.  Few registers: the launch holds 2x the warps of the dense kernel,
// which is what a latency-bound chain (descriptor -> indices -> bitmap -> row) needs.
template <typename C>
__device__ __forceinline__ void spmm_accumulate_masked(const SpmmParams& p, int s, int len, int iters, int gl, int grp,
                                                       float4 (&acc)[C::VPL]) {
  // chunk layout as in the dense loop: lane gl holds entries k * LPR + gl (k < EPL) of a CH-entry chunk
  int c_next[C::EPL];
  float v_next[C::EPL];
  auto load_chunk = [&](int off) {
#pragma unroll
    for (int k = 0; k < C::EPL; ++k) {
      c_next[k] = -1;
      v_next[k] = 0.f;
      const int e = off + k * C::LPR + gl;
      if (e < len) {
        c_next[k] = C::EPL > 1 ? __ldg(p.col + s + e) : ld_stream_i32(p.col + s + e);
        v_next[k] = C::EPL > 1 ? __ldg(p.val + s + e) : ld_stream_f32(p.val + s + e);
      }
    }
  };
  load_chunk(0);
  for (int it = 0, off = 0; it < iters; ++it, off += C::CH) {
    int c[C::EPL];
    float v[C::EPL];
#pragma unroll
    for (int k = 0; k < C::EPL; ++k) { c[k] = c_next[k]; v[k] = v_next[k]; }
    load_chunk(off + C::CH);
#pragma unroll
    for (int k = 0; k < C::EPL; ++k) {
      const bool live = c[k] >= 0 && bit_set(p.col_mask, c[k]);
      unsigned bits = __ballot_sync(0xffffffffu, live);
      if constexpr (C::LPR < 32) bits = (bits >> (grp * C::LPR)) & ((1u << C::LPR) - 1u);
      while (__any_sync(0xffffffffu, bits != 0u)) {
        // two live entries per trip: both gathers are in flight together
        const bool on0 = bits != 0u;
        const int t0 = on0 ? __ffs(bits) - 1 : 0;
        bits &= bits - 1u;
        const bool on1 = bits != 0u;
        const int t1 = on1 ? __ffs(bits) - 1 : 0;
        bits &= bits - 1u;
        const int c0 = __shfl_sync(0xffffffffu, c[k], t0, C::LPR);
        const float v0 = __shfl_sync(0xffffffffu, v[k], t0, C::LPR);
        const int c1 = __shfl_sync(0xffffffffu, c[k], t1, C::LPR);
        const float v1 = __shfl_sync(0xffffffffu, v[k], t1, C::LPR);
        float4 x0[C::VPL], x1[C::VPL];
#pragma unroll
        for (int vv = 0; vv < C::VPL; ++vv) {
          x0[vv] = on0 ? ld_gather_f4(p.X + (size_t)c0 * C::V4 + vv * C::LPR + gl) : make_float4(0.f, 0.f, 0.f, 0.f);
          x1[vv] = on1 ? ld_gather_f4(p.X + (size_t)c1 * C::V4 + vv * C::LPR + gl) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (on0) {
#pragma unroll
          for (int vv = 0; vv < C::VPL; ++vv) fma4_packed(acc[vv], v0, x0[vv]);
        }
        if (on1) {
#pragma unroll
          for (int vv = 0; vv < C::VPL; ++vv) fma4_packed(acc[vv], v1, x1[vv]);
        }
      }
    }
  }
}

// the end of a work item, shared by the two accumulation schemes below: rows cut into several segments combine
// through the partial-sum scratch (every segment stores its partial sum, the one that arrives last -- a ticket per
// row -- adds them in segment order: deterministic, no floating-point atomics), then the fused epilogue
template <typename C, bool NOISE, bool TERMS = false, bool AMASK = false>
__device__ __forceinline__ void spmm_finish_item(const SpmmParams& p, bool valid, bool live, int row, int k, int nseg,
                                                 long long slot, float4 (&acc)[C::VPL], int gl, const float4* pre) {
  const bool multi = valid && nseg > 1;
  bool do_epilogue = valid;
  if (__any_sync(0xffffffffu, multi)) {
    int pb = 0;
    if (multi) {
      pb = __ldg(p.vpart + slot);
      float4* mine = p.partial + ((size_t)pb + k) * C::V4;
#pragma unroll
      for (int v = 0; v < C::VPL; ++v) mine[v * C::LPR + gl] = acc[v];
      __threadfence();                                     // partial visible before the ticket is taken
    }
    __syncwarp();
    int old = 0;
    if (multi && gl == 0) old = atomicAdd(p.tickets + pb, 1);
    old = __shfl_sync(0xffffffffu, old, 0, C::LPR);
    if (multi) {
      do_epilogue = old == nseg - 1;                       // the last segment to arrive finishes the row
      if (do_epilogue) {
        __threadfence();
#pragma unroll
        for (int v = 0; v < C::VPL; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
        if constexpr (C::LPR <= 8) {
          // narrow column slices: the launch is ONE wave of CTAs, so a hub row's combine is not hidden behind other CTAs:
          // eight partials are loaded together (one L2 round trip per batch instead of one per segment) and added in
          // segment order.  Measured neutral (24.1 vs 23.6 us at d = 8).  What the per-CTA timelines
          // (profiles/r2_spmm_cta_timeline_d8_seg{32,64}.txt) show instead: a warp needs ~4.5 us per 16-entry chunk
          // whatever else is resident -- the ~8 000 row sectors the SM's lane groups keep in flight queue at ~1 sector
          // per clock -- so an item's duration is its length x the groups resident, and the launch lasts as long as the
          // longest items' chains.  Tried against that and all SLOWER than one bundle per warp on hardware-scheduled
          // CTAs (profiles/r2_spmm_{interleave,warp_sched,vecidx}_experiment.txt, r2_spmm_narrow_matrix.txt): bundles
          // dealt round-robin to the CTAs (d = 8: 29.4 vs 26.4 us), warps that take bundles from a device counter
          // (28.9 vs 23.9), 5 / 6 CTAs per SM at 48 / 40 registers (26.8 / 30.9 vs 24.0), 16-entry segments (30.6);
          // 16-byte index loads on 4-entry-aligned item starts gain 4-14 % (22.6 vs 26.2 at 64-entry segments).
          constexpr int NB = 8;
          for (int kk = 0; kk < nseg; kk += NB) {
            float4 part[NB];
#pragma unroll
            for (int q = 0; q < NB; ++q) {
              const int ks = kk + q < nseg ? kk + q : nseg - 1;          // clamp: the surplus loads are discarded below
              part[q] = __ldcg(p.partial + ((size_t)pb + ks) * C::V4 + gl);
            }
#pragma unroll
            for (int q = 0; q < NB; ++q)
              if (kk + q < nseg) acc[0] = add4(acc[0], part[q]);
          }
        } else {
          for (int kk = 0; kk < nseg; ++kk) {                // segment order: deterministic
            const float4* part = p.partial + ((size_t)pb + kk) * C::V4;
#pragma unroll
            for (int v = 0; v < C::VPL; ++v) acc[v] = add4(acc[v], __ldcg(part + v * C::LPR + gl));
          }
        }
        if (gl == 0) p.tickets[pb] = 0;                    // ready for the next launch
      }
    }
  }
  spmm_epilogue<C, NOISE, TERMS, AMASK>(p, row, do_epilogue, live, acc, gl, pre);
}

// one block of RPB work items (one lane group each); TERMS: the layer sum is formed in the epilogue (acc_terms);
// AMASK: addend / acc_in are read only at the rows of addend_mask
template <int D, int LPR, bool NOISE, bool CMASK, bool TERMS = false, bool AMASK = false>
__device__ __forceinline__ void spmm_block(const SpmmParams& p, const int n_v, const int blk) {
#ifdef AGCF_SPMM_TRACE
  TraceScope trace_scope(blk);
#endif
  using C = RowCfg<D, LPR>;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int gl = lane & (C::LPR - 1);
  const int grp = lane / C::LPR;
  float4 acc[C::VPL];
#pragma unroll
  for (int v = 0; v < C::VPL; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  const long long slot = ((long long)blk * (blockDim.x >> 5) + warp) * C::RPW + grp;   // block size is a launch parameter
  bool valid = slot < n_v;
  int4 vr = make_int4(0, 0, 0, 1 << 16);
  if (valid) vr = __ldg(p.vrows + slot);                  // one 16-byte load: start, len, row, segment id
  const int s = vr.x, row = vr.z, k = vr.w & 0xffff, nseg = vr.w >> 16;
  int len = vr.y;
  if (valid && p.row_mask != nullptr && !bit_set(p.row_mask, row)) { valid = false; len = 0; }
  // the addend row's bit: requested with the item's first indices, needed only by the epilogue
  const bool live = !AMASK || (valid && bit_set(p.addend_mask, row));
  int maxlen = len;
#pragma unroll
  for (int o = C::LPR; o < 32; o <<= 1) {
    const int other = __shfl_xor_sync(0xffffffffu, maxlen, o);
    maxlen = other > maxlen ? other : maxlen;
  }
  AGCF_TRACE_AFTER(1, maxlen + row);
  float4 pre[C::VPL];                                      // CMASK: the epilogue's addend row, fetched before the gathers
  if constexpr (CMASK) {
    const int iters = (maxlen + C::CH - 1) / C::CH;        // warp-uniform
    const bool has_add = p.addend != nullptr && valid && live;
#pragma unroll
    for (int v = 0; v < C::VPL; ++v)
      pre[v] = has_add ? ld_stream_f4(p.addend + (size_t)row * C::V4 + v * C::LPR + gl) : make_float4(0.f, 0.f, 0.f, 0.f);
    spmm_accumulate_masked<C>(p, s, len, iters, gl, grp, acc);
  } else {
    const int iters = (maxlen + C::CH - 1) / C::CH;        // warp-uniform
    spmm_accumulate_chunks<C, true>(p, s, len, 0, C::CH, iters, gl, acc);
  }
  AGCF_TRACE_AFTER(2, __float_as_int(acc[0].x));
  spmm_finish_item<C, NOISE, TERMS, AMASK>(p, valid, live, row, k, nseg, slot, acc, gl,
                                          (CMASK && p.addend != nullptr) ? pre : nullptr);
}

// ------------------------------------------------------------------ narrow rows (column-sharded tables)
// d = 8 / 16 column slices (the d-sharded multi-GPU layout): a row is 32 / 64 bytes, LPR = 2 / 4 lanes.  With one work
// item per lane group (spmm_block) the 16 / 8 groups of a warp walk 16 / 8 DIFFERENT items, so every index load of a warp
// touches 16 different cache lines and is replayed as 16 L1 wavefronts, and every (col, val) pair is broadcast by two
// shuffles inside a 2-lane group -- the LSU data pipe, which has to serve one wavefront per gathered row anyway (a 32-byte
// row is one sector of its own line), carried ~4 wavefronts per non-zero; that, not bytes, bounded the kernel
// (26.5 us per launch at d = 8 for 82 MB of L2 traffic, profiles/r1_summary.md section 3).
// Here the WARP walks its G = 32 / LPR items one after the other: the item's indices are read with coalesced loads (lane l
// holds entries l and l + 32 of a 64-entry block), every gather instruction fetches G different entries of the SAME item
// (one per lane group, two shuffles for all of them), and the G partial sums are combined by a halving butterfly that ends
// with one value per lane, transposed so that lane group i receives item i's row -- from there on the groups own one item
// each, exactly like spmm_block (segment combine, epilogue).  Per non-zero: 1 gather wavefront + ~0.4 others.
// Summation order: entries j * G + grp of a block are summed per group in j order, groups by the fixed butterfly:
// deterministic, run-to-run identical, not the entry order of spmm_block (parity bars are tolerances, DESIGN.md).
template <typename C>
__device__ __forceinline__ float4 coop_reduce_transpose(float4 acc, int lane, int gl) {
  constexpr unsigned FULL = 0xffffffffu;
  // halving over lane bit 4 (keep x,y or z,w) and bit 3 (keep one of the two): 3 shuffles, 4 -> 1 value per lane
  const bool up = (lane & 16) != 0;
  const float r0 = __shfl_xor_sync(FULL, up ? acc.x : acc.z, 16);
  const float r1 = __shfl_xor_sync(FULL, up ? acc.y : acc.w, 16);
  const float a = (up ? acc.z : acc.x) + r0;
  const float b = (up ? acc.w : acc.y) + r1;
  const bool up2 = (lane & 8) != 0;
  const float r2 = __shfl_xor_sync(FULL, up2 ? a : b, 8);
  float t = (up2 ? b : a) + r2;                      // column gl * 4 + (bit4 ? 2 : 0) + (bit3 ? 1 : 0)
#pragma unroll
  for (int m = 4; m >= C::LPR; m >>= 1) t += __shfl_xor_sync(FULL, t, m);      // the remaining group bits
  // every lane fetches the float4 of ITS gl (lanes gl | 8 c0 | 16 c1 hold column 4 gl + c0 + 2 c1)
  float4 o;
  o.x = __shfl_sync(FULL, t, gl);
  o.y = __shfl_sync(FULL, t, gl | 8);
  o.z = __shfl_sync(FULL, t, gl | 16);
  o.w = __shfl_sync(FULL, t, gl | 24);
  return o;
}

template <int D, int LPR, bool NOISE, bool CMASK>
__device__ __forceinline__ void spmm_block_coop(const SpmmParams& p, const int n_v, const int blk,
                                                const uint32_t* __restrict__ cmask, int2* __restrict__ stage) {
  using C = RowCfg<D, LPR>;
  static_assert(C::VPL == 1 && LPR <= 4, "cooperative scheme: rows of at most 4 lanes");
  constexpr int G = C::RPW;                                // lane groups per warp = items per warp = entries per gather
  constexpr unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int gl = lane & (C::LPR - 1);
  const int grp = lane / C::LPR;
  const long long slot = ((long long)blk * (blockDim.x >> 5) + warp) * G + grp;
  bool valid = slot < n_v;
  int4 vr = make_int4(0, 0, 0, 1 << 16);
  if (valid) vr = __ldg(p.vrows + slot);
  const int s_mine = vr.x, row = vr.z, k = vr.w & 0xffff, nseg = vr.w >> 16;
  int len_mine = vr.y;
  if (valid && p.row_mask != nullptr && !bit_set(p.row_mask, row)) { valid = false; len_mine = 0; }
  if (!valid) len_mine = 0;
  float4 pre[1];
  if constexpr (CMASK) {
    const bool has_add = p.addend != nullptr && valid;
    pre[0] = has_add ? ld_stream_f4(p.addend + (size_t)row * C::V4 + gl) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float4 res = make_float4(0.f, 0.f, 0.f, 0.f);
  // entries [base, base + 64) of an item: lane l holds entries base + l and base + l + 32 (coalesced, streamed)
  auto load_block = [&](int s, int len, int base, int& c0, float& v0, int& c1, float& v1) {
    c0 = -1; c1 = -1; v0 = 0.f; v1 = 0.f;
    const int e0 = base + lane, e1 = base + lane + 32;
    if (e0 < len) { c0 = ld_stream_i32(p.col + s + e0); v0 = ld_stream_f32(p.val + s + e0); }
    if (e1 < len) { c1 = ld_stream_i32(p.col + s + e1); v1 = ld_stream_f32(p.val + s + e1); }
  };
  int s_i = __shfl_sync(FULL, s_mine, 0), len_i = __shfl_sync(FULL, len_mine, 0);
  int c0, c1; float v0, v1;
  load_block(s_i, len_i, 0, c0, v0, c1, v1);
  for (int i = 0; i < G; ++i) {
    int s_n = 0, len_n = 0, nc0 = -1, nc1 = -1; float nv0 = 0.f, nv1 = 0.f;
    if (i + 1 < G) {                                       // next item's first block: in flight during these gathers
      s_n = __shfl_sync(FULL, s_mine, (i + 1) * C::LPR);
      len_n = __shfl_sync(FULL, len_mine, (i + 1) * C::LPR);
      load_block(s_n, len_n, 0, nc0, nv0, nc1, nv1);
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int base = 0; base < len_i; base += 64) {         // warp-uniform
      if (base > 0) load_block(s_i, len_i, base, c0, v0, c1, v1);
      int n_here = len_i - base < 64 ? len_i - base : 64;
      if constexpr (CMASK) {
        // only entries whose column carries a non-zero row of X are gathered (~13 % at the benchmark shape): compact
        // them through a 64-slot staging row of this warp, in entry order
        const bool l0 = c0 >= 0 && ((cmask[c0 >> 5] >> (c0 & 31)) & 1u);
        const bool l1 = c1 >= 0 && ((cmask[c1 >> 5] >> (c1 & 31)) & 1u);
        const unsigned b0 = __ballot_sync(FULL, l0), b1 = __ballot_sync(FULL, l1);
        const unsigned lt = (1u << lane) - 1u;
        __syncwarp();
        if (l0) stage[__popc(b0 & lt)] = make_int2(c0, __float_as_int(v0));
        if (l1) stage[__popc(b0) + __popc(b1 & lt)] = make_int2(c1, __float_as_int(v1));
        __syncwarp();
        n_here = __popc(b0) + __popc(b1);
#pragma unroll
        for (int j = 0; j < 64 / G; ++j) {
          if (j * G >= n_here) break;
          const int e = j * G + grp;
          if (e < n_here) {
            const int2 cv = stage[e];
            fma4_packed(acc, __int_as_float(cv.y), ld_gather_f4(p.X + (size_t)cv.x * C::V4 + gl));
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < 64 / G; ++j) {
          if (j * G >= n_here) break;                      // warp-uniform
          const int e = j * G + grp;                       // this group's entry of the step
          const int cc = __shfl_sync(FULL, (j * G) < 32 ? c0 : c1, e & 31);
          const float vv = __shfl_sync(FULL, (j * G) < 32 ? v0 : v1, e & 31);
          if (cc >= 0) fma4_packed(acc, vv, ld_gather_f4(p.X + (size_t)cc * C::V4 + gl));
        }
      }
    }
    if (len_i > 0) {                                       // warp-uniform
      const float4 o = coop_reduce_transpose<C>(acc, lane, gl);
      if (grp == i) res = o;
    }
    s_i = s_n; len_i = len_n; c0 = nc0; c1 = nc1; v0 = nv0; v1 = nv1;
  }
  float4 accv[1] = {res};
  spmm_finish_item<C, NOISE>(p, valid, true, row, k, nseg, slot, accv, gl, (CMASK && p.addend != nullptr) ? pre : nullptr);
}

// the column bitmap of the first backward layer lives in shared memory while it fits (N <= 32 * kCoopMaskWords nodes)
constexpr int kCoopMaskWords = 8192;

template <int D, int LPR, int MINB, bool NOISE, bool CMASK>
__global__ void __launch_bounds__(256, MINB) spmm_coop_kernel(const SpmmParams p, int mask_words) {
  extern __shared__ __align__(16) unsigned char coop_smem[];
  int n_v = p.n_v;
  if (p.n_v_dev != nullptr) {
    const int n_dev = __ldg(p.n_v_dev);
    n_v = n_dev < n_v ? n_dev : n_v;
  }
  const uint32_t* cmask = p.col_mask;
  int2* stage = nullptr;
  if constexpr (CMASK) {
    stage = reinterpret_cast<int2*>(coop_smem) + (threadIdx.x >> 5) * 64;
    if (mask_words > 0) {                                  // bitmap copy: one coalesced pass per CTA, then LDS lookups
      uint32_t* sm = reinterpret_cast<uint32_t*>(coop_smem + 8 * 64 * sizeof(int2));
      for (int w = threadIdx.x; w < mask_words; w += 256) sm[w] = __ldg(p.col_mask + w);
      __syncthreads();
      cmask = sm;
    }
  }
  spmm_block_coop<D, LPR, NOISE, CMASK>(p, n_v, (int)blockIdx.x, cmask, stage);
}

// Grid: one CTA per block of RPB items (sched == nullptr), or PERSISTENT CTAs (148 x MINB of them) that take their
// first block by CTA id and every further one from a device counter, in plan order (long items first).  The ticket for
// the next block is taken before the current block is processed, so its latency is hidden; the last CTA to finish
// puts both counters back to zero for the next launch.
template <int D, int LPR, bool NOISE, bool CMASK, bool TERMS = false, bool AMASK = false>
__device__ __forceinline__ void spmm_grid(const SpmmParams& p) {
  using C = RowCfg<D, LPR>;
  int n_v = p.n_v;
  if (p.n_v_dev != nullptr) {
    const int n_dev = __ldg(p.n_v_dev);
    n_v = n_dev < n_v ? n_dev : n_v;
  }
  if (p.sched == nullptr) {
    spmm_block<D, LPR, NOISE, CMASK, TERMS, AMASK>(p, n_v, (int)blockIdx.x);
    return;
  }
  __shared__ int s_next[2];
  const int rpb = (int)(blockDim.x >> 5) * C::RPW;
  const int n_blocks = (n_v + rpb - 1) / rpb;
  int blk = (int)blockIdx.x;
  for (int it = 0; blk < n_blocks; ++it) {
    int nxt = 0;
    if (threadIdx.x == 0) nxt = atomicAdd(p.sched, 1) + (int)gridDim.x;
    spmm_block<D, LPR, NOISE, CMASK, TERMS, AMASK>(p, n_v, blk);
    if (threadIdx.x == 0) s_next[it & 1] = nxt;
    __syncthreads();
    blk = s_next[it & 1];
  }
  if (threadIdx.x == 0) {
    const int done = atomicAdd(p.sched + 1, 1);
    if (done == (int)gridDim.x - 1) { p.sched[0] = 0; p.sched[1] = 0; }
  }
}

template <int D, int LPR, int MINB, bool NOISE, bool TERMS = false, bool AMASK = false>
__global__ void __launch_bounds__(256, MINB) spmm_csr_kernel(const SpmmParams p) {
  spmm_grid<D, LPR, NOISE, false, TERMS, AMASK>(p);
}

// first backward layer: gathers only the rows in col_mask (spmm_accumulate_masked)
#ifndef AGCF_SPMM_CM_THREADS
#define AGCF_SPMM_CM_THREADS 128                   // 4-warp CTAs like the plain launches (d = 16: 19.6 -> 18.5 us, d = 128: 77.5 -> 74.3)
#endif
template <int D, int LPR, int MINB, bool AMASK>
__global__ void __launch_bounds__(AGCF_SPMM_CM_THREADS, MINB) spmm_colmask_kernel(const SpmmParams p) {
  spmm_grid<D, LPR, false, true, false, AMASK>(p);
}

// resident CTAs per SM the register allocation is held to: 4 (<= 64 registers) measured best at d <= 64
#ifndef AGCF_SPMM_MINB
#define AGCF_SPMM_MINB(D) ((D) <= 128 ? 4 : 2)
#endif
#ifndef AGCF_SPMM_CM_MINB
#define AGCF_SPMM_CM_MINB(D) ((D) < 64 ? 8 : ((D) == 64 ? 10 : ((D) == 128 ? 8 : 6)))   // CTAs of AGCF_SPMM_CM_THREADS = 128
#endif

template <int D>
static int launch_spmm(const SpmmParams& p, cudaStream_t st) {
  // lane mapping measured best on B200 (profiles/): one float4 per lane, d/4 lanes per row (16 at d = 64),
  // fully unrolled 16-entry chunks, packed FFMA2 accumulation
  constexpr int LPR = default_lpr(D);
  using C = RowCfg<D, LPR>;
  long long blocks = ((long long)p.n_v + C::RPB - 1) / C::RPB;
  if (blocks <= 0) return AGCF_OK;
  if (blocks > 0x7fffffffLL) return AGCF_EUNSUPPORTED;
  const bool cmask = p.col_mask != nullptr && p.noise == nullptr && !p.noise_main && p.aux_Y[0] == nullptr && p.aux_Y[1] == nullptr;
  if constexpr (D <= 16) {
    // narrow column slices: the warp-cooperative scheme, OFF by default (AGCF_SPMM_COOP=1 selects it).  Measured on B200
    // at the Gowalla shape (profiles/r2_summary.md): 31.0 vs 26.7 us at d = 8, 35.0 vs 24.8 us at d = 16 -- it does cut
    // the L1 wavefronts per non-zero, but a warp now walks its 16 items one after the other, and with ~1 wave of CTAs per
    // launch the launch lasts as long as that serial chain of 16 dependent index -> gather -> reduce round trips.
    static const bool coop = [] { const char* e = getenv("AGCF_SPMM_COOP"); return e != nullptr && atoi(e) != 0; }();
    if (coop && p.sched == nullptr && p.n_acc_terms == 0 && p.addend_mask == nullptr && (p.col_mask == nullptr || cmask)) {
      const bool noise = p.noise != nullptr || p.noise_main || p.aux_Y[0] != nullptr || p.aux_Y[1] != nullptr;
      if (cmask) {
        const int words = (p.mask_bits + 31) / 32;
        const int mw = (p.mask_bits > 0 && words <= kCoopMaskWords) ? words : 0;
        const size_t smem = 8 * 64 * sizeof(int2) + (size_t)mw * 4;
        auto kern = spmm_coop_kernel<D, LPR, AGCF_SPMM_MINB(D), false, true>;
        if (smem > 48 * 1024) AGCF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<(unsigned)blocks, C::THREADS, smem, st>>>(p, mw);
      } else if (noise) {
        spmm_coop_kernel<D, LPR, AGCF_SPMM_MINB(D), true, false><<<(unsigned)blocks, C::THREADS, 0, st>>>(p, 0);
      } else {
        spmm_coop_kernel<D, LPR, AGCF_SPMM_MINB(D), false, false><<<(unsigned)blocks, C::THREADS, 0, st>>>(p, 0);
      }
      AGCF_LAUNCH_OK();
      return AGCF_OK;
    }
  }
  if (p.sched != nullptr) {                                  // persistent: every CTA resident at once
    const long long resident = (long long)kSMs * (cmask ? AGCF_SPMM_CM_MINB(D) : AGCF_SPMM_MINB(D));
    blocks = blocks < resident ? blocks : resident;
  }
  if (cmask) {
    const long long rpb = (AGCF_SPMM_CM_THREADS / 32) * C::RPW;
    long long cb = ((long long)p.n_v + rpb - 1) / rpb;
    if (p.sched != nullptr) cb = cb < blocks ? cb : blocks;
    if (p.addend_mask != nullptr)
      spmm_colmask_kernel<D, LPR, AGCF_SPMM_CM_MINB(D), true><<<(unsigned)cb, AGCF_SPMM_CM_THREADS, 0, st>>>(p);
    else
      spmm_colmask_kernel<D, LPR, AGCF_SPMM_CM_MINB(D), false><<<(unsigned)cb, AGCF_SPMM_CM_THREADS, 0, st>>>(p);
    AGCF_LAUNCH_OK();
    return AGCF_OK;
  }
  // CTA size of the plain launches: 4 warps (the kernel derives its slots from blockDim; AGCF_SPMM_THREADS = 64 / 128 /
  // 256 for tuning).  Same warps per SM as 8-warp CTAs, but a CTA's slot is handed on as soon as ITS four warps are done:
  // measured on B200 (profiles/r2_summary.md section 9) 44.0 -> 43.2 us at d = 64, 30.8 -> 28.9 at d = 32, 24.7 -> 23.1 at
  // d = 16, 234.9 -> 231.6 at d = 128 (Amazon-book shape); 64 threads measured the same as 128
  static const int csr_threads = [] {
    const char* e = getenv("AGCF_SPMM_THREADS");
    const int t = e != nullptr ? atoi(e) : 128;
    return (t == 64 || t == 128 || t == 256) ? t : 128;
  }();
  if (p.sched == nullptr && csr_threads != C::THREADS) {
    const long long rpb = (long long)(csr_threads / 32) * C::RPW;
    blocks = ((long long)p.n_v + rpb - 1) / rpb;
  }
  const int threads = p.sched == nullptr ? csr_threads : C::THREADS;
  if (p.noise != nullptr || p.noise_main || p.aux_Y[0] != nullptr || p.aux_Y[1] != nullptr)
    spmm_csr_kernel<D, LPR, AGCF_SPMM_MINB(D), true><<<(unsigned)blocks, threads, 0, st>>>(p);
  else if (p.n_acc_terms > 0)
    spmm_csr_kernel<D, LPR, AGCF_SPMM_MINB(D), false, true><<<(unsigned)blocks, threads, 0, st>>>(p);
  else if (p.addend_mask != nullptr)
    spmm_csr_kernel<D, LPR, AGCF_SPMM_MINB(D), false, false, true><<<(unsigned)blocks, threads, 0, st>>>(p);
  else
    spmm_csr_kernel<D, LPR, AGCF_SPMM_MINB(D), false><<<(unsigned)blocks, threads, 0, st>>>(p);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

// ------------------------------------------------------------------------ SDDMM
template <int D>
__global__ void __launch_bounds__(256) sddmm_csr_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                        const float4* __restrict__ H, const float4* __restrict__ E,
                                                        float* __restrict__ gval, int accumulate,
                                                        const int32_t* __restrict__ row_order, int n_rows) {
  using C = RowCfg<D>;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int gl = lane & (C::LPR - 1);
  const int grp = lane / C::LPR;
  const long long slot = ((long long)blockIdx.x * (C::THREADS / 32) + warp) * C::RPW + grp;
  const bool valid = slot < n_rows;
  int row = 0, s = 0, len = 0;
  if (valid) {
    row = row_order != nullptr ? row_order[slot] : (int)slot;
    s = rowptr[row];
    len = rowptr[row + 1] - s;
  }
  int maxlen = len;
#pragma unroll
  for (int o = C::LPR; o < 32; o <<= 1) {
    const int other = __shfl_xor_sync(0xffffffffu, maxlen, o);
    maxlen = other > maxlen ? other : maxlen;
  }
  float4 h[C::VPL];
#pragma unroll
  for (int v = 0; v < C::VPL; ++v)
    h[v] = valid ? __ldg(H + (size_t)row * C::V4 + v * C::LPR + gl) : make_float4(0.f, 0.f, 0.f, 0.f);
  for (int off = 0; off < maxlen; off += C::LPR) {
    int c = 0;
    if (off + gl < len) c = ld_stream_i32(col + s + off + gl);
    int n = len - off;
    n = n < 0 ? 0 : (n > C::LPR ? C::LPR : n);
    float mine = 0.f;
#pragma unroll
    for (int t = 0; t < C::LPR; ++t) {
      const int ct = __shfl_sync(0xffffffffu, c, t, C::LPR);
      float partial = 0.f;
      if (t < n) {
#pragma unroll
        for (int vv = 0; vv < C::VPL; ++vv)
          partial += dot4(h[vv], ld_gather_f4(E + (size_t)ct * C::V4 + vv * C::LPR + gl));
      }
      partial = group_sum<C::LPR>(partial);
      if (gl == t) mine = partial;
    }
    if (off + gl < len) {
      float* dst = gval + s + off + gl;
      *dst = accumulate ? (*dst + mine) : mine;
    }
  }
}

// ------------------------------------------------------------------ normalization
__global__ void __launch_bounds__(256) norm_adj_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                       const float* __restrict__ w, const float* __restrict__ d_row,
                                                       const float* __restrict__ d_col, float* __restrict__ val,
                                                       int32_t* __restrict__ row_of, int n_rows, long long nnz) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nnz) return;
  // row of nnz p: largest i with rowptr[i] <= p (empty rows are skipped by the search)
  int lo = 0, hi = n_rows;           // invariant: rowptr[lo] <= p < rowptr[hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if ((long long)__ldg(rowptr + mid) <= p) lo = mid; else hi = mid;
  }
  if (row_of != nullptr) row_of[p] = lo;
  if (val != nullptr) val[p] = __fmul_rn(__fmul_rn(d_row[lo], w[p]), d_col[col[p]]);
}

__global__ void __launch_bounds__(256) concat_rows_kernel(const float4* __restrict__ a, long long na4,
                                                          const float4* __restrict__ b, long long nb4,
                                                          float4* __restrict__ out) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < na4 + nb4; k += stride)
    out[k] = k < na4 ? ld_stream_f4(a + k) : ld_stream_f4(b + (k - na4));
}

// ------------------------------------------------- per-batch work lists (last forward layer)
// The loss reads F only at the <= 3B nodes of a batch, so the last forward layer is computed for those rows only.
// Instead of testing every work item of the static plan against the batch bitmap (4 448 CTAs that mostly exit),
// the PREP phase writes the batch's OWN plan: one CTA per batch walks the batch's sorted distinct nodes
// (agcf_bpr_group_batches), cuts each row into segments of `segment` entries and emits the same
// {start, len, row, k | nseg << 16} descriptors the SpMM kernel consumes, with partial-sum slots numbered per batch.
__global__ void __launch_bounds__(1024) batch_worklist_kernel(const int32_t* __restrict__ seg_node,
                                                              const int32_t* __restrict__ n_seg, int seg_stride,
                                                              const int32_t* __restrict__ rowptr, int row0, int row1,
                                                              int split_above, int segment, int4* __restrict__ wl_vrows,
                                                              int32_t* __restrict__ wl_vpart, int32_t* __restrict__ wl_count,
                                                              int cap) {
  __shared__ int warp_items[32], warp_slots[32];
  __shared__ int total_items;
  const int b = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int32_t* nodes = seg_node + (size_t)b * seg_stride;
  const int n = n_seg[b];
  const int per = (n + nthr - 1) / nthr;
  const int lo = min(tid * per, n), hi = min(lo + per, n);
  auto segments_of = [&](int node, int& start, int& deg) {
    if (node < row0 || node >= row1) { start = 0; deg = 0; return 0; }   // another rank's row
    start = __ldg(rowptr + node);
    deg = __ldg(rowptr + node + 1) - start;
    return deg > split_above ? (deg + segment - 1) / segment : 1;
  };
  int items = 0, slots = 0;
  for (int q = lo; q < hi; ++q) {
    int start, deg;
    const int ns = segments_of(nodes[q], start, deg);
    items += ns;
    slots += ns > 1 ? ns : 0;
  }
  int inc_i = items, inc_s = slots;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int yi = __shfl_up_sync(0xffffffffu, inc_i, o);
    const int ys = __shfl_up_sync(0xffffffffu, inc_s, o);
    if (lane >= o) { inc_i += yi; inc_s += ys; }
  }
  if (lane == 31) { warp_items[warp] = inc_i; warp_slots[warp] = inc_s; }
  __syncthreads();
  if (warp == 0) {
    const int wi = lane < (nthr >> 5) ? warp_items[lane] : 0;
    const int ws = lane < (nthr >> 5) ? warp_slots[lane] : 0;
    int ci = wi, cs = ws;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int yi = __shfl_up_sync(0xffffffffu, ci, o);
      const int ys = __shfl_up_sync(0xffffffffu, cs, o);
      if (lane >= o) { ci += yi; cs += ys; }
    }
    warp_items[lane] = ci - wi;
    warp_slots[lane] = cs - ws;
    if (lane == 31) total_items = ci;
  }
  __syncthreads();
  int w = warp_items[warp] + inc_i - items;          // first item of this thread
  int ps = warp_slots[warp] + inc_s - slots;         // first partial slot of this thread
  int4* out_v = wl_vrows + (size_t)b * cap;
  int32_t* out_p = wl_vpart + (size_t)b * cap;
  for (int q = lo; q < hi; ++q) {
    int start, deg;
    const int node = nodes[q];
    const int ns = segments_of(node, start, deg);
    for (int k = 0; k < ns; ++k, ++w) {
      if (w >= cap) break;
      int len = deg;
      if (ns > 1) { len = deg - k * segment; len = len > segment ? segment : len; }
      out_v[w] = make_int4(start + k * segment, len, node, k | (ns << 16));
      out_p[w] = ps;
    }
    if (ns > 1) ps += ns;
  }
  if (tid == 0) wl_count[b] = total_items < cap ? total_items : cap;
}

}  // namespace agcf

using namespace agcf;

static_assert(sizeof(((agcf_spmm_args*)nullptr)->acc_terms) == AGCF_MAX_ACC_TERMS * sizeof(const float*),
              "acc_terms holds AGCF_MAX_ACC_TERMS tables");

extern "C" int agcf_spmm_csr_f32_ex(const agcf_spmm_args* a, agcf_stream_t stream) {
  if (a == nullptr) return AGCF_EINVAL;
  if (a->n_peers < 0 || a->n_peers > AGCF_MAX_PEERS) return AGCF_EINVAL;
  if (!a->vrows || !a->vpart || !a->col || !a->val || !a->partial || !a->tickets || !a->X || a->n_vrows < 0) return AGCF_EINVAL;
  if (a->Y == nullptr && a->acc_out == nullptr && a->adam_p == nullptr) return AGCF_EINVAL;
  if (!supported_d(a->d)) return AGCF_EUNSUPPORTED;
  if (!aligned16(a->vrows) || !aligned16(a->partial)) return AGCF_EINVAL;
  if (!aligned16(a->X) || !aligned16(a->Y) || !aligned16(a->addend) || !aligned16(a->acc_in) || !aligned16(a->acc_out) ||
      !aligned16(a->noise) || !aligned16(a->mc_Y) || !aligned16(a->mc_acc))
    return AGCF_EINVAL;
  if (a->X == a->Y || a->X == a->acc_out) return AGCF_EINVAL;   // rows of X are read by other CTAs
  if (a->acc_div == 0.f) return AGCF_EINVAL;
  if (a->adam_p != nullptr) {
    if (!a->adam_m || !a->adam_v || !a->adam_coefs) return AGCF_EINVAL;
    if (!aligned16(a->adam_p) || !aligned16(a->adam_m) || !aligned16(a->adam_v)) return AGCF_EINVAL;
    if (a->adam_p == a->X) return AGCF_EINVAL;
  }
  if (a->zero_acc_in && (a->acc_in == nullptr || a->acc_in == a->X)) return AGCF_EINVAL;
  SpmmParams p;
  p.vrows = reinterpret_cast<const int4*>(a->vrows); p.vpart = a->vpart; p.n_v = a->n_vrows; p.n_v_dev = a->n_vrows_dev;
  p.partial = reinterpret_cast<float4*>(a->partial); p.tickets = a->tickets;
  p.col = a->col; p.val = a->val;
  p.X = reinterpret_cast<const float4*>(a->X);
  p.Y = reinterpret_cast<float4*>(a->Y);
  p.addend = reinterpret_cast<const float4*>(a->addend);
  p.acc_in = reinterpret_cast<const float4*>(a->acc_in);
  p.acc_out = reinterpret_cast<float4*>(a->acc_out);
  p.acc_div = a->acc_div;
  p.noise = reinterpret_cast<const float4*>(a->noise);
  p.eps = a->eps;
  p.noise_seed = a->noise_seed; p.noise_stream = a->noise_stream; p.noise_step = a->noise_step;
  p.noise_main = (a->noise_main != 0 && a->noise == nullptr) ? 1 : 0;
  if (p.noise_main && a->noise_seed == 0ull) return AGCF_EINVAL;
  for (int q = 0; q < 2; ++q) {
    p.aux_Y[q] = reinterpret_cast<float4*>(a->aux_Y[q]);
    p.aux_noise[q] = reinterpret_cast<const float4*>(a->aux_noise[q]);
    p.aux_stream[q] = a->aux_stream[q];
    if (!aligned16(a->aux_Y[q]) || !aligned16(a->aux_noise[q]) || (a->aux_Y[q] != nullptr && a->aux_Y[q] == a->X)) return AGCF_EINVAL;
    if (a->aux_Y[q] != nullptr && a->aux_noise[q] == nullptr && a->noise_seed == 0ull) return AGCF_EINVAL;
  }
  p.row_mask = a->row_mask; p.col_mask = a->col_mask; p.mask_bits = a->mask_bits > 0 ? a->mask_bits : 0;
  p.mc_Y = a->Y != nullptr ? reinterpret_cast<float4*>(a->mc_Y) : nullptr;
  p.mc_acc = a->acc_out != nullptr ? reinterpret_cast<float4*>(a->mc_acc) : nullptr;
  p.n_peers = a->n_peers;
  for (int q = 0; q < AGCF_MAX_PEERS; ++q) {
    p.peer_Y[q] = (q < a->n_peers && a->peer_Y_host) ? reinterpret_cast<float4*>(a->peer_Y_host[q]) : nullptr;
    p.peer_acc[q] = (q < a->n_peers && a->peer_acc_host) ? reinterpret_cast<float4*>(a->peer_acc_host[q]) : nullptr;
  }
  p.adam_p = reinterpret_cast<float4*>(a->adam_p);
  p.adam_m = reinterpret_cast<float4*>(a->adam_m);
  p.adam_v = reinterpret_cast<float4*>(a->adam_v);
  p.adam_coefs = a->adam_coefs;
  p.beta1 = a->adam_beta1; p.beta2 = a->adam_beta2; p.adam_eps = a->adam_eps;
  p.zero_rows = a->zero_acc_in ? reinterpret_cast<float4*>(const_cast<float*>(a->acc_in)) : nullptr;
  p.addend_mask = a->addend_mask;
  if (a->flags != 0) return AGCF_EINVAL;
  if (a->n_acc_terms < 0 || a->n_acc_terms > AGCF_MAX_ACC_TERMS) return AGCF_EINVAL;
  p.n_acc_terms = a->n_acc_terms;
  for (int q = 0; q < AGCF_MAX_ACC_TERMS; ++q) {
    p.acc_terms[q] = q < a->n_acc_terms ? reinterpret_cast<const float4*>(a->acc_terms[q]) : nullptr;
    if (q < a->n_acc_terms && (a->acc_terms[q] == nullptr || !aligned16(a->acc_terms[q]) || a->acc_terms[q] == a->acc_out))
      return AGCF_EINVAL;
  }
  if (p.n_acc_terms > 0) {
    const bool noisy = p.noise != nullptr || p.noise_main || p.aux_Y[0] != nullptr || p.aux_Y[1] != nullptr;
    if (a->acc_in != nullptr || a->acc_out == nullptr || a->col_mask != nullptr || a->adam_p != nullptr || noisy ||
        a->addend_mask != nullptr)
      return AGCF_EINVAL;
  }
  if (a->addend_mask != nullptr && (p.noise != nullptr || p.noise_main || p.aux_Y[0] != nullptr || p.aux_Y[1] != nullptr))
    return AGCF_EINVAL;
  p.sched = a->sched;
  cudaStream_t st = (cudaStream_t)stream;
  switch (a->d) {
    case 8: return launch_spmm<8>(p, st);
    case 16: return launch_spmm<16>(p, st);
    case 32: return launch_spmm<32>(p, st);
    case 64: return launch_spmm<64>(p, st);
    case 128: return launch_spmm<128>(p, st);
    case 256: return launch_spmm<256>(p, st);
  }
  return AGCF_EUNSUPPORTED;
}

extern "C" int agcf_spmm_csr_f32(const int32_t* vrows, const int32_t* vpart, int32_t n_vrows,
                                 const int32_t* col, const float* val, float* partial, int32_t* tickets,
                                 const float* X, float* Y, const float* addend,
                                 const float* acc_in, float* acc_out, float acc_div,
                                 const float* noise, float eps,
                                 const uint32_t* row_mask, const uint32_t* col_mask,
                                 void* const* peer_Y_host, void* const* peer_acc_host, int32_t n_peers,
                                 void* mc_Y, void* mc_acc,
                                 int32_t d, agcf_stream_t stream) {
  agcf_spmm_args a = {};
  a.vrows = vrows; a.vpart = vpart; a.n_vrows = n_vrows;
  a.col = col; a.val = val; a.partial = partial; a.tickets = tickets;
  a.X = X; a.Y = Y; a.addend = addend; a.acc_in = acc_in; a.acc_out = acc_out; a.acc_div = acc_div;
  a.noise = noise; a.eps = eps; a.row_mask = row_mask; a.col_mask = col_mask;
  a.peer_Y_host = peer_Y_host; a.peer_acc_host = peer_acc_host; a.n_peers = n_peers;
  a.mc_Y = mc_Y; a.mc_acc = mc_acc; a.d = d;
  return agcf_spmm_csr_f32_ex(&a, stream);
}

extern "C" int agcf_spmm_batch_worklists(const int32_t* seg_node, const int32_t* n_seg, int32_t n_batches,
                                         int32_t seg_stride, const int32_t* rowptr, int32_t row0, int32_t row1,
                                         int32_t split_above, int32_t segment, int32_t* wl_vrows, int32_t* wl_vpart,
                                         int32_t* wl_count, int32_t cap, agcf_stream_t stream) {
  if (!seg_node || !n_seg || !rowptr || !wl_vrows || !wl_vpart || !wl_count) return AGCF_EINVAL;
  if (n_batches < 0 || seg_stride <= 0 || seg_stride > 16384 || cap <= 0 || row0 < 0 || row1 < row0) return AGCF_EINVAL;
  if (segment < 16 || segment > 4096 || split_above < segment || !aligned16(wl_vrows)) return AGCF_EINVAL;
  if (n_batches == 0) return AGCF_OK;
  batch_worklist_kernel<<<(unsigned)n_batches, 1024, 0, (cudaStream_t)stream>>>(
      seg_node, n_seg, seg_stride, rowptr, row0, row1, split_above, segment, reinterpret_cast<int4*>(wl_vrows), wl_vpart,
      wl_count, cap);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int agcf_sddmm_csr_f32(const int32_t* rowptr, const int32_t* col, const float* H, const float* E,
                                  float* gval, int32_t accumulate, const int32_t* row_order,
                                  int32_t n_rows, int32_t d, agcf_stream_t stream) {
  if (!rowptr || !col || !H || !E || !gval || n_rows < 0) return AGCF_EINVAL;
  if (!supported_d(d)) return AGCF_EUNSUPPORTED;
  if (!aligned16(H) || !aligned16(E)) return AGCF_EINVAL;
  if (n_rows == 0) return AGCF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const float4* H4 = reinterpret_cast<const float4*>(H);
  const float4* E4 = reinterpret_cast<const float4*>(E);
#define AGCF_SDDMM(DD)                                                                          \
  {                                                                                             \
    const unsigned blocks = (unsigned)((n_rows + RowCfg<DD>::RPB - 1) / RowCfg<DD>::RPB);        \
    sddmm_csr_kernel<DD><<<blocks, 256, 0, st>>>(rowptr, col, H4, E4, gval, accumulate, row_order, n_rows); \
  }
  switch (d) {
    case 8: AGCF_SDDMM(8) break;
    case 16: AGCF_SDDMM(16) break;
    case 32: AGCF_SDDMM(32) break;
    case 64: AGCF_SDDMM(64) break;
    case 128: AGCF_SDDMM(128) break;
    case 256: AGCF_SDDMM(256) break;
  }
#undef AGCF_SDDMM
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

static int norm_or_expand(const int32_t* rowptr, const int32_t* col, const float* w, const float* d_row,
                          const float* d_col, float* val, int32_t* row_of, int32_t n_rows, int64_t nnz,
                          cudaStream_t st) {
  if (n_rows == 0 || nnz == 0) return AGCF_OK;
  if (nnz < 0 || nnz > 0x7fffffffLL) return AGCF_EINVAL;
  const unsigned blocks = (unsigned)(((long long)nnz + 255) / 256);
  norm_adj_kernel<<<blocks, 256, 0, st>>>(rowptr, col, w, d_row, d_col, val, row_of, n_rows, nnz);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int agcf_norm_adj_csr(const int32_t* rowptr, const int32_t* col, const float* w,
                                 const float* d_row, const float* d_col, float* val,
                                 int32_t n_rows, int64_t nnz, agcf_stream_t stream) {
  if (!rowptr || !col || !w || !d_row || !d_col || !val || n_rows < 0) return AGCF_EINVAL;
  return norm_or_expand(rowptr, col, w, d_row, d_col, val, nullptr, n_rows, nnz, (cudaStream_t)stream);
}

extern "C" int agcf_csr_expand_rows(const int32_t* rowptr, int32_t* row_of, int32_t n_rows, int64_t nnz,
                                    agcf_stream_t stream) {
  if (!rowptr || !row_of || n_rows < 0) return AGCF_EINVAL;
  return norm_or_expand(rowptr, nullptr, nullptr, nullptr, nullptr, nullptr, row_of, n_rows, nnz, (cudaStream_t)stream);
}

extern "C" int agcf_concat_rows_f32(const float* a, int64_t n_a, const float* b, int64_t n_b,
                                    float* out, int32_t d, agcf_stream_t stream) {
  if (!out || n_a < 0 || n_b < 0 || (n_a > 0 && !a) || (n_b > 0 && !b) || d <= 0 || (d & 3)) return AGCF_EINVAL;
  if (!aligned16(a) || !aligned16(b) || !aligned16(out)) return AGCF_EINVAL;
  const long long na4 = n_a * (d / 4), nb4 = n_b * (d / 4);
  if (na4 + nb4 == 0) return AGCF_OK;
  long long blocks = (na4 + nb4 + 255) / 256;
  if (blocks > kSMs * 16) blocks = kSMs * 16;
  concat_rows_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(a), na4, reinterpret_cast<const float4*>(b), nb4, reinterpret_cast<float4*>(out));
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}
