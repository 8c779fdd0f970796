// score.cu -- full-rank evaluation: user x item scoring fused with masked top-K.
//
// Reference: recommender/LightGCN.py:86-90 (predict: one GEMV per user + D2H),
// :148-156 (test loop: mask train items with -10e8, find_k_largest),
// util/algorithm.py:155-167 (heap top-K), util/metrics.py:9-85 (hits / NDCG).
//
// Pipeline (scores are never written to HBM):
//   stage 0  mask bits    : [n_u, ceil(I/32)] words from the train-item CSR
//   stage 1  group maxima : S = U_tile . I^T ; per (user, 32-item group) the max of
//                           the masked scores.  impl 0: fp32 CUDA-core GEMM whose
//                           per-score FMA chain is bit-identical to stage 2's;
//                           impl 1: TF32 tcgen05 GEMM (score_tc.cu), approximate.
//   stage 2  per user     : R = K-th largest group max  ->  candidate groups are
//                           those with max >= R - margin (margin = 2*delta bounds the
//                           stage-1 error, 0 for impl 0) -- every true top-K item is in
//                           one of them (DESIGN.md "top-K exactness");  candidates are
//                           re-scored in exact fp32 (k ascending, fmaf), the K-th
//                           largest exact score s* is radix-selected, ties at s* are
//                           resolved with the reference heap's rule, and the K
//                           survivors are sorted by (score desc, item asc).
//
// Why the result is exact although stage 1 may be approximate (impl 1, TF32):
//   let e_i be the exact (fp32, fixed-order) masked score of item i, a_i the stage-1 value,
//   |a_i - e_i| <= delta for all i (TF32 truncates each operand by < 2^-10 relative, so
//   |a_i - e_i| <= 2^-9 * sum_k |u_k v_ik| (1 + o(1)) <= 1.01 * 2^-9 * |u| * max_i |v_i| =: delta).
//   tau := K-th largest GROUP maximum of a.  The K groups attaining it contain K distinct items
//   with a >= tau, hence e >= tau - delta, hence the K-th largest exact score s* >= tau - delta.
//   Any item of the exact top-K (incl. every item tied at s*) has e_i >= s* >= tau - delta, so
//   a_i >= tau - 2*delta, so its group's maximum is >= tau - 2*delta: it is in a candidate group.
//   Candidates are re-scored exactly and the selection / tie rule only look at items with
//   e >= s*, all of which are candidates.  For impl 0, a == e bit for bit and delta = 0.
//   delta holds at every d, d = 8 and 16 included: the truncation term and Cauchy-Schwarz do not depend on d, and the
//   fp32 accumulation inside the tensor core adds at most ~d 2^-24 sum_k |u_k v_ik|, which the factor 1.01 covers for
//   d <= 256 (smaller d only shrinks it).  Zero columns (padded operands) add exact zeros and change neither a nor e.
#include "common.cuh"
#include <float.h>
#include <stdlib.h>

namespace agcf {

constexpr float kMasked = -1.0e9f;         // -10e8, recommender/LightGCN.py:153
constexpr int kGroup = 32;                 // items per group

__device__ __forceinline__ uint32_t f2key(float f) {          // order-preserving float -> uint
  const uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// exact reference score: fp32, k ascending, fused multiply-add, start from 0
template <int D>
__device__ __forceinline__ float exact_dot(const float* __restrict__ urow_smem, const float4* __restrict__ irow) {
  float acc = 0.f;
#pragma unroll 4
  for (int k4 = 0; k4 < D / 4; ++k4) {
    const float4 v = __ldg(irow + k4);
    acc = fmaf(urow_smem[4 * k4 + 0], v.x, acc);
    acc = fmaf(urow_smem[4 * k4 + 1], v.y, acc);
    acc = fmaf(urow_smem[4 * k4 + 2], v.z, acc);
    acc = fmaf(urow_smem[4 * k4 + 3], v.w, acc);
  }
  return acc;
}

// ------------------------------------------------------------------ stage 0: mask
__global__ void __launch_bounds__(256) mask_bits_kernel(const int32_t* __restrict__ user_rows, int n_u,
                                                        const int32_t* __restrict__ mask_rowptr,
                                                        const int32_t* __restrict__ mask_items, int n_items,
                                                        int item_offset, int pitch, uint32_t* __restrict__ bits) {
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n_u) return;
  const int uid = user_rows != nullptr ? user_rows[r] : r;
  const int s = mask_rowptr[uid], e = mask_rowptr[uid + 1];
  for (int k = s + lane; k < e; k += 32) {
    const int it = mask_items[k] - item_offset;         // item shards: mask ids are global
    if (it >= 0 && it < n_items) atomicOr(bits + (size_t)r * pitch + (it >> 5), 1u << (it & 31));
  }
}

// max L2 norm over item rows (for the TF32 error margin)
template <int D>
__global__ void __launch_bounds__(256) max_row_norm_kernel(const float4* __restrict__ T, int n_rows, float* __restrict__ out) {
  // out must be zeroed; norms are >= 0 so uint ordering of the bit pattern is monotone
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  float ss = 0.f;
  if (r < n_rows) {
    for (int k = 0; k < D / 4; ++k) { const float4 v = __ldg(T + (size_t)r * (D / 4) + k); ss += dot4(v, v); }
  }
  float m = sqrtf(ss);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int*>(out), __float_as_uint(m));
}

// ------------------------------------------------- stage 1 (impl 0): fp32 GEMM
// CTA = 64 users x (loop over 128-item tiles of its item split); 256 threads, each
// owns 4 users x 8 items (items tx + 16*ii, so that the 16 tx-lanes read 16
// consecutive item rows with LDS.128 at a 68-float stride: conflict-free).
constexpr int S1_TU = 64, S1_TI = 128, S1_LD = 68;
template <int D>
struct S1Smem { static constexpr int LD = D + 4; static constexpr size_t bytes = (size_t)(S1_TU + S1_TI) * LD * sizeof(float); };

template <int D>
__global__ void __launch_bounds__(256) group_max_fp32_kernel(const float4* __restrict__ Uemb, const int32_t* __restrict__ user_rows,
                                                             int n_u, const float4* __restrict__ Iemb, int n_items,
                                                             const uint32_t* __restrict__ bits, int n_groups, int pitch,
                                                             int tiles_per_split, float* __restrict__ gmax) {
  constexpr int LD = D + 4;                 // padded row stride in floats (multiple of 4)
  constexpr int V4 = D / 4;
  extern __shared__ __align__(16) float smem[];
  float* Us = smem;                         // [64][LD]
  float* Is = smem + S1_TU * LD;            // [128][LD]
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;   // ty: 0..15 -> users ty*4..ty*4+3
  const int u0 = blockIdx.x * S1_TU;
  // load the user tile once
  for (int k = tid; k < S1_TU * V4; k += 256) {
    const int r = k / V4, c = k - r * V4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (u0 + r < n_u) {
      const int uid = user_rows != nullptr ? user_rows[u0 + r] : (u0 + r);
      v = __ldg(Uemb + (size_t)uid * V4 + c);
    }
    *reinterpret_cast<float4*>(Us + r * LD + 4 * c) = v;
  }
  const int n_tiles = (n_items + S1_TI - 1) / S1_TI;
  const int t_begin = blockIdx.y * tiles_per_split;
  const int t_end = min(n_tiles, t_begin + tiles_per_split);
  for (int tile = t_begin; tile < t_end; ++tile) {
    const int i0 = tile * S1_TI;
    __syncthreads();                        // previous tile fully consumed (and Us visible)
    for (int k = tid; k < S1_TI * V4; k += 256) {
      const int r = k / V4, c = k - r * V4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i0 + r < n_items) v = __ldg(Iemb + (size_t)(i0 + r) * V4 + c);
      *reinterpret_cast<float4*>(Is + r * LD + 4 * c) = v;
    }
    __syncthreads();
    float acc[4][8];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;
#pragma unroll 2
    for (int k4 = 0; k4 < V4; ++k4) {
      float4 uu[4], vv[8];
#pragma unroll
      for (int a = 0; a < 4; ++a) uu[a] = *reinterpret_cast<const float4*>(Us + (ty * 4 + a) * LD + 4 * k4);
#pragma unroll
      for (int b = 0; b < 8; ++b) vv[b] = *reinterpret_cast<const float4*>(Is + (tx + 16 * b) * LD + 4 * k4);
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) {       // k ascending: x, y, z, w
          acc[a][b] = fmaf(uu[a].x, vv[b].x, acc[a][b]);
          acc[a][b] = fmaf(uu[a].y, vv[b].y, acc[a][b]);
          acc[a][b] = fmaf(uu[a].z, vv[b].z, acc[a][b]);
          acc[a][b] = fmaf(uu[a].w, vv[b].w, acc[a][b]);
        }
    }
    // masked group maxima: group gq (q=0..3) of this tile = items i0 + 32q .. +31 = {tx + 16*(2q), tx + 16*(2q+1)}
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int ur = u0 + ty * 4 + a;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int g = (i0 >> 5) + q;
        uint32_t w = 0u;
        if (ur < n_u && g < n_groups) w = __ldg(bits + (size_t)ur * pitch + g);
        float m = -FLT_MAX;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int b = 2 * q + h;
          const int item = i0 + tx + 16 * b;
          float sc = acc[a][b];
          if ((w >> ((tx + 16 * h) & 31)) & 1u) sc = kMasked;
          if (item >= n_items) sc = -FLT_MAX;
          m = fmaxf(m, sc);
        }
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (tx == 0 && ur < n_u && g < n_groups) gmax[(size_t)ur * pitch + g] = m;
      }
    }
  }
}

// --------------------------------------------------------------- stage 2 helpers
// block-wide radix select of the R-th largest (R >= 1) among n keys produced by
// keyfn(k); returns the key (uniform).  4 passes of 8 bits, smem histogram.
struct SelectSmem {
  unsigned int hist[256];
  unsigned int prefix;
  unsigned int remaining;
};

template <typename KeyFn>
__device__ uint32_t block_radix_select(SelectSmem& sm, int n, unsigned int R, KeyFn keyfn) {
  const int tid = threadIdx.x, nthr = blockDim.x;
  if (tid == 0) { sm.prefix = 0u; sm.remaining = R; }
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    for (int k = tid; k < 256; k += nthr) sm.hist[k] = 0u;
    __syncthreads();
    const uint32_t prefix = sm.prefix;
    const uint32_t pmask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
    for (int k = tid; k < n; k += nthr) {
      const uint32_t key = keyfn(k);
      if ((key & pmask) == prefix) atomicAdd(&sm.hist[(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (tid < 32) {
      // lane l owns bins [8l, 8l+8); find the digit where the count from the top reaches `remaining`
      unsigned int mine = 0u;
#pragma unroll
      for (int b = 0; b < 8; ++b) mine += sm.hist[tid * 8 + b];
      unsigned int above = 0u;           // sum over lanes > tid
      unsigned int run = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned int y = __shfl_down_sync(0xffffffffu, run, o);
        if (tid + o < 32) run += y;
      }
      above = run - mine;                // inclusive suffix minus own
      const unsigned int rem = sm.remaining;
      const bool here = above < rem && rem <= above + mine;
      if (here) {
        unsigned int acc = above;
        int digit = tid * 8;
        for (int b = 7; b >= 0; --b) {
          const unsigned int c = sm.hist[tid * 8 + b];
          if (acc + c >= rem) { digit = tid * 8 + b; break; }
          acc += c;
        }
        sm.prefix = prefix | ((uint32_t)digit << shift);
        sm.remaining = rem - acc;
      }
    }
    __syncthreads();
  }
  return sm.prefix;
}

// block-wide exclusive scan of one int per thread (256 threads): warp shuffles + one
// barrier; the 8 warp totals go through a double-buffered smem row (``flip`` alternates)
__device__ __forceinline__ int block_excl_scan_256(int v, int (*warp_buf)[8], int& flip, int& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  int* buf = warp_buf[flip];
  flip ^= 1;
  if (lane == 31) buf[warp] = incl;
  __syncthreads();
  int before = 0, all = 0;
#pragma unroll
  for (int w = 0; w < 8; ++w) {
    const int t = buf[w];
    all += t;
    if (w < warp) before += t;
  }
  total = all;
  return before + incl - v;
}

struct Stage2Params {
  const float4* Uemb;
  const int32_t* user_rows;
  int n_u;
  const float4* Iemb;
  int n_items;
  const uint32_t* bits;
  const float* gmax;
  int n_groups;
  int pitch;                   // row stride (words) of bits / gmax
  int K;
  int item_offset;
  float margin_scale;          // 0 for impl 0; 2 * 1.01 * 2^-9 for TF32
  const float* max_item_norm;  // scalar (device) or null
  float* out_val;
  int32_t* out_idx;
  int32_t* out_flags;
  // per-CTA scratch of the block kernel (global, L2-resident)
  int32_t* cand_groups;        // [grid][n_groups]
  float* cand_val;             // [grid][n_groups*32]
  // block kernel as the overflow path of the warp kernel: users list[0 .. *list_count) instead of 0 .. n_u-1
  const int32_t* list;
  const int32_t* list_count;
  // warp kernel: per-warp scratch for at most cmax candidate groups; users with more go to the overflow list
  int cmax;
  int32_t* w_groups;           // [warps][cmax]
  float* w_val;                // [warps][cmax*32]
  int32_t* overflow_list;      // [n_u]
  int32_t* overflow_count;     // zeroed by the caller
  // group-major re-scoring (stage 2 split into candidates -> per-group pair lists -> re-score -> select)
  int32_t* u_groups;           // [n_u][cmax] candidate groups of every user
  int32_t* u_ncg;              // [n_u] their count, -1 = overflow (block kernel)
  float* u_val;                // [n_u][cmax*32] exact scores of the candidates
  int32_t* g_count;            // [n_groups] users that have the group as a candidate (zeroed by the caller)
  int32_t* pairs;              // [n_groups][n_u] (user << 8 | candidate slot) of the users that have the group
  // item-compacting variant of the group-major stage 2: the re-scoring keeps only the exact scores that can still matter
  float* u_thr;                // [n_u] T_u <= s*_u (K-th largest exact score): nothing below it can be selected or tie
  int32_t* u_cnt;              // [n_u] kept (item, score) entries (zeroed by the caller); > cap_items = overflow
  int2* u_items;               // [n_u][cap_items] {item, score bits}, unordered
  int cap_items;
  const float4* Udense;        // nullable: the user rows gathered for the tcgen05 stage 1 ([n_u][D], row r = user r of the
                               // call) -- the same bits as Uemb[user_rows[r]] without the index hop
  int cand_stage;              // s2_candidates: > 0 = every warp keeps its user's row of group maxima in shared memory
                               // (cand_stage floats per warp, dynamic) for the five passes over it
};

template <int D>
__global__ void __launch_bounds__(256) topk_select_kernel(const Stage2Params p) {
  __shared__ SelectSmem sel;
  __shared__ int warp_buf[3][8];      // rotating rows: a row is rewritten only two scans (two barriers) later
  int flip = 0;
  __shared__ __align__(16) float urow[D];
  __shared__ int sh_p_pos, sh_gp;
  extern __shared__ __align__(16) unsigned char dyn[];   // K-sized sort buffers
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int kpow2 = 1;
  while (kpow2 < p.K) kpow2 <<= 1;
  unsigned long long* sort_keys = reinterpret_cast<unsigned long long*>(dyn);   // [kpow2]
  int32_t* my_groups = p.cand_groups + (size_t)blockIdx.x * p.n_groups;
  float* my_val = p.cand_val + (size_t)blockIdx.x * p.n_groups * kGroup;

  const int n_list = p.list_count != nullptr ? *p.list_count : p.n_u;
  for (int q = blockIdx.x; q < n_list; q += gridDim.x) {
    const int r = p.list != nullptr ? p.list[q] : q;
    const int uid = p.user_rows != nullptr ? p.user_rows[r] : r;
    const float* grow = p.gmax + (size_t)r * p.pitch;
    const uint32_t* brow = p.bits + (size_t)r * p.pitch;
    __syncthreads();
    if (tid < D / 4) reinterpret_cast<float4*>(urow)[tid] = __ldg(p.Uemb + (size_t)uid * (D / 4) + tid);
    __syncthreads();
    // ---- 1. threshold on the group maxima
    const unsigned int R = (unsigned int)min(p.K, p.n_groups);
    const uint32_t tkey = block_radix_select(sel, p.n_groups, R, [&](int k) { return f2key(grow[k]); });
    float thr = key2f(tkey);
    if (p.margin_scale > 0.f) {
      float ss = 0.f;
      for (int k = 0; k < D; ++k) ss = fmaf(urow[k], urow[k], ss);
      thr -= p.margin_scale * sqrtf(ss) * __ldg(p.max_item_norm);
    }
    // ---- 2. ordered compaction of candidate groups
    int n_cg = 0;
    for (int base = 0; base < p.n_groups; base += 256) {
      const int g = base + tid;
      const int flag = (g < p.n_groups && grow[g] >= thr) ? 1 : 0;
      int total;
      const int pos = block_excl_scan_256(flag, warp_buf, flip, total);
      if (flag) my_groups[n_cg + pos] = g;
      n_cg += total;
    }
    __syncthreads();
    // ---- 3. exact re-scoring of the candidates (warp per group, lane per item)
    for (int c = warp; c < n_cg; c += 8) {
      const int g = my_groups[c];
      const int item = g * kGroup + lane;
      float sc = -FLT_MAX;
      if (item < p.n_items) {
        sc = exact_dot<D>(urow, p.Iemb + (size_t)item * (D / 4));
        if ((__ldg(brow + g) >> lane) & 1u) sc = kMasked;
      }
      my_val[c * kGroup + lane] = sc;
    }
    __syncthreads();
    const int nc = n_cg * kGroup;
    // number of real items among the candidates (only the last group can be partial)
    int n_valid = nc;
    if (n_cg > 0 && my_groups[n_cg - 1] == p.n_groups - 1) n_valid = nc - (p.n_groups * kGroup - p.n_items);
    const int Keff = min(p.K, n_valid);
    // ---- 4. K-th largest exact score, then the reference heap's tie rule
    //   s* = K-th largest; m = #(> s*); walking items in index order, pos_p = first
    //   position where #(>= s*) reaches K, g_p = #(> s*) at positions <= pos_p; the ties
    //   kept are those with tie-rank in [m - g_p, K - g_p)   (SURVEY.md 8a-11).
    int n_sel = 0;
    if (Keff > 0) {
      const uint32_t skey = block_radix_select(sel, nc, (unsigned int)Keff, [&](int k) { return f2key(my_val[k]); });
      const float sstar = key2f(skey);
      // pass A: m, pos_p, g_p  (one packed scan per chunk: #(>= s*) in the low half, #(> s*) in the high half)
      if (tid == 0) { sh_p_pos = -1; sh_gp = 0; }
      int run_ge = 0, run_gt = 0;
      for (int base = 0; base < nc; base += 256) {
        const int k = base + tid;
        const float v = k < nc ? my_val[k] : -FLT_MAX;
        const bool real = k < n_valid;
        const int gt = (real && v > sstar) ? 1 : 0;
        const int ge = (real && v >= sstar) ? 1 : 0;
        int tot;
        const int ex = block_excl_scan_256(ge | (gt << 16), warp_buf, flip, tot);
        const int ex_ge = ex & 0xffff, ex_gt = ex >> 16;
        if (ge && run_ge + ex_ge + 1 == Keff) { sh_p_pos = k; sh_gp = run_gt + ex_gt + gt; }
        run_ge += tot & 0xffff;
        run_gt += tot >> 16;
      }
      const int m = run_gt;
      // pass B: select (ordered), pack (score key desc, idx asc) into 64-bit sort keys
      for (int k = tid; k < kpow2; k += 256) sort_keys[k] = ~0ull;
      __syncthreads();
      const int gp = sh_gp;
      const int tie_lo = m - gp, tie_n = Keff - m;                  // kept ties: tie-rank in [tie_lo, tie_lo + tie_n)
      int run_eq = 0;
      run_gt = 0;
      for (int base = 0; base < nc; base += 256) {
        const int k = base + tid;
        const float v = k < nc ? my_val[k] : -FLT_MAX;
        const bool real = k < n_valid;
        const int gt = (real && v > sstar) ? 1 : 0;
        const int eq = (real && v == sstar) ? 1 : 0;
        int tot;
        const int ex = block_excl_scan_256(eq | (gt << 16), warp_buf, flip, tot);
        const int trank = run_eq + (ex & 0xffff);                    // ties before this one
        const int gt_before = run_gt + (ex >> 16);
        const bool take = gt || (eq && trank >= tie_lo && trank < tie_lo + tie_n);
        if (take) {
          // output slot = selected items before this one = (> s*) before + kept ties before
          int ties_before = trank - tie_lo;
          ties_before = ties_before < 0 ? 0 : (ties_before > tie_n ? tie_n : ties_before);
          const int item = my_groups[k >> 5] * kGroup + (k & 31);
          // ascending sort of (~scorekey, item) == score desc, item asc
          sort_keys[gt_before + ties_before] = ((unsigned long long)(~f2key(v)) << 32) | (uint32_t)item;
        }
        run_eq += tot & 0xffff;
        run_gt += tot >> 16;
      }
      const int run_sel = Keff;
      n_sel = run_sel;
      __syncthreads();
      for (int kk = 2; kk <= kpow2; kk <<= 1)
        for (int jj = kk >> 1; jj > 0; jj >>= 1) {
          for (int idx = tid; idx < (kpow2 >> 1); idx += 256) {
            const int a = ((idx & ~(jj - 1)) << 1) | (idx & (jj - 1));
            const int c = a | jj;
            const bool up = (a & kk) == 0;
            const unsigned long long ka = sort_keys[a], kc = sort_keys[c];
            if ((ka > kc) == up) { sort_keys[a] = kc; sort_keys[c] = ka; }
          }
          __syncthreads();
        }
    }
    for (int k = tid; k < p.K; k += 256) {
      float v = -INFINITY;
      int idx = -1;
      if (k < n_sel) {
        const unsigned long long key = sort_keys[k];
        v = key2f(~(uint32_t)(key >> 32));
        idx = (int)(uint32_t)key + p.item_offset;
      }
      p.out_val[(size_t)r * p.K + k] = v;
      p.out_idx[(size_t)r * p.K + k] = idx;
    }
    if (tid == 0 && p.out_flags != nullptr) p.out_flags[r] = n_cg;   // diagnostics: candidate groups examined
  }
}

// ------------------------------------------------------- stage 2, one WARP per user
// Same algorithm as topk_select_kernel, but a warp owns a user: every block barrier becomes a __syncwarp,
// block scans become ballots, and 8x as many users are in flight per SM -- the block version spends its
// ~65 barriers per user waiting.  Shared memory per warp: a 256-bin histogram, the user row, K sort keys.
// Candidate groups beyond p.cmax (never seen at the benchmark shapes) send the user to the overflow list,
// which the block kernel then processes.
__device__ __forceinline__ uint32_t warp_radix_select(unsigned int* hist, int n, unsigned int R, int lane,
                                                      const float* __restrict__ vals) {
  uint32_t prefix = 0u;
  unsigned int remaining = R;
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
#pragma unroll
    for (int b = 0; b < 8; ++b) hist[lane * 8 + b] = 0u;
    __syncwarp();
    const uint32_t pmask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
    // (lanes of equal bin combined through match.any before the atomic was measured 4.5x SLOWER for the whole kernel --
    // 392 vs 87 us per chunk, profiles/r2_launches_eval.csv: MATCH.ANY serialises over the distinct values of a warp)
    for (int k = lane; k < n; k += 32) {
      const uint32_t key = f2key(vals[k]);
      if ((key & pmask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
    }
    __syncwarp();
    unsigned int mine = 0u;
#pragma unroll
    for (int b = 0; b < 8; ++b) mine += hist[lane * 8 + b];
    unsigned int run = mine;                     // inclusive suffix sum over lanes >= lane
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int y = __shfl_down_sync(0xffffffffu, run, o);
      if (lane + o < 32) run += y;
    }
    const unsigned int above = run - mine;
    const bool here = above < remaining && remaining <= above + mine;
    uint32_t new_prefix = prefix;
    unsigned int new_remaining = remaining;
    if (here) {
      unsigned int acc = above;
      int digit = lane * 8;
      for (int b = 7; b >= 0; --b) {
        const unsigned int c = hist[lane * 8 + b];
        if (acc + c >= remaining) { digit = lane * 8 + b; break; }
        acc += c;
      }
      new_prefix = prefix | ((uint32_t)digit << shift);
      new_remaining = remaining - acc;
    }
    const unsigned int who = __ballot_sync(0xffffffffu, here);
    const int src = who != 0u ? (__ffs(who) - 1) : 0;
    prefix = __shfl_sync(0xffffffffu, new_prefix, src);
    remaining = __shfl_sync(0xffffffffu, new_remaining, src);
    __syncwarp();
  }
  return prefix;
}

// warps per CTA of the warp kernel: the per-warp item tile ([32][D+4] floats) bounds how many fit
template <int D>
struct S2W {
  static constexpr int WPC = D <= 64 ? 4 : (D == 128 ? 2 : 1);
  static constexpr int LD = D + 4;                                   // padded tile row (floats): conflict-free LDS.128
  static constexpr size_t tile_bytes = (size_t)kGroup * LD * 4;
  __host__ __device__ static size_t per_warp(int kpow2) { return 1024 + (size_t)D * 4 + (size_t)kpow2 * 8 + tile_bytes; }
};

template <int D>
__global__ void __launch_bounds__(32 * S2W<D>::WPC) topk_select_warp_kernel(const Stage2Params p) {
  extern __shared__ __align__(16) unsigned char dyn[];
  constexpr int WPC = S2W<D>::WPC, LD = S2W<D>::LD, V4 = D / 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int kpow2 = 1;
  while (kpow2 < p.K) kpow2 <<= 1;
  const size_t per_warp = S2W<D>::per_warp(kpow2);
  unsigned char* mine = dyn + (size_t)warp * per_warp;
  unsigned int* hist = reinterpret_cast<unsigned int*>(mine);
  float* urow = reinterpret_cast<float*>(mine + 1024);
  unsigned long long* sort_keys = reinterpret_cast<unsigned long long*>(mine + 1024 + (size_t)D * 4);
  float* tile = reinterpret_cast<float*>(mine + 1024 + (size_t)D * 4 + (size_t)kpow2 * 8);
  const uint32_t tile_s = (uint32_t)__cvta_generic_to_shared(tile);
  const int gw = blockIdx.x * WPC + warp, n_warps = gridDim.x * WPC;
  int32_t* my_groups = p.w_groups + (size_t)gw * p.cmax;
  float* my_val = p.w_val + (size_t)gw * p.cmax * kGroup;
  const unsigned int lt_mask = (1u << lane) - 1u;

  for (int r = gw; r < p.n_u; r += n_warps) {
    const int uid = p.user_rows != nullptr ? p.user_rows[r] : r;
    const float* grow = p.gmax + (size_t)r * p.pitch;
    const uint32_t* brow = p.bits + (size_t)r * p.pitch;
    __syncwarp();
    for (int k = lane; k < D / 4; k += 32) reinterpret_cast<float4*>(urow)[k] = __ldg(p.Uemb + (size_t)uid * (D / 4) + k);
    __syncwarp();
    // ---- 1. threshold on the group maxima
    const unsigned int R = (unsigned int)min(p.K, p.n_groups);
    float thr = key2f(warp_radix_select(hist, p.n_groups, R, lane, grow));
    if (p.margin_scale > 0.f) {
      float ss = 0.f;
      for (int k = 0; k < D; ++k) ss = fmaf(urow[k], urow[k], ss);
      thr -= p.margin_scale * sqrtf(ss) * __ldg(p.max_item_norm);
    }
    // ---- 2. ordered compaction of candidate groups
    int n_cg = 0;
    bool overflow = false;
    for (int base = 0; base < p.n_groups; base += 32) {
      const int g = base + lane;
      const bool flag = g < p.n_groups && grow[g] >= thr;
      const unsigned int b = __ballot_sync(0xffffffffu, flag);
      const int pos = n_cg + __popc(b & lt_mask);
      if (n_cg + __popc(b) > p.cmax) { overflow = true; break; }       // warp-uniform
      if (flag) my_groups[pos] = g;
      n_cg += __popc(b);
    }
    if (overflow) {
      if (lane == 0) p.overflow_list[atomicAdd(p.overflow_count, 1)] = r;
      continue;
    }
    __syncwarp();
    // ---- 3. exact re-scoring of the candidates.  A group's 32 item rows are one contiguous block: it is
    // copied global -> shared with coalesced cp.async (a lane-per-item read would fetch 16 B out of every
    // 128 B line per instruction), then lane l walks ITS item's row in shared memory in the reference
    // order (k ascending, fmaf) -- the same bits as exact_dot.
    for (int c = 0; c < n_cg; ++c) {
      const int g = my_groups[c];
      const int rows_here = min(kGroup, p.n_items - g * kGroup);
      const float4* src = p.Iemb + (size_t)g * kGroup * V4;
#pragma unroll
      for (int i = 0; i < V4; ++i) {
        const int f = i * 32 + lane, row = f / V4, c4 = f % V4;
        const bool in = row < rows_here;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(tile_s + (uint32_t)(row * LD + 4 * c4) * 4u),
                     "l"(in ? src + f : p.Iemb), "r"(in ? 16 : 0) : "memory");
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      __syncwarp();
      float sc = 0.f;
      const float* mine_row = tile + lane * LD;
#pragma unroll 4
      for (int k4 = 0; k4 < V4; ++k4) {
        const float4 v = *reinterpret_cast<const float4*>(mine_row + 4 * k4);
        const float4 u = *reinterpret_cast<const float4*>(urow + 4 * k4);
        sc = fmaf(u.x, v.x, sc);
        sc = fmaf(u.y, v.y, sc);
        sc = fmaf(u.z, v.z, sc);
        sc = fmaf(u.w, v.w, sc);
      }
      if (lane >= rows_here) sc = -FLT_MAX;
      else if ((__ldg(brow + g) >> lane) & 1u) sc = kMasked;
      my_val[c * kGroup + lane] = sc;
      __syncwarp();                                        // the tile is refilled by the next group
    }
    __syncwarp();
    const int nc = n_cg * kGroup;
    int n_valid = nc;
    if (n_cg > 0 && my_groups[n_cg - 1] == p.n_groups - 1) n_valid = nc - (p.n_groups * kGroup - p.n_items);
    const int Keff = min(p.K, n_valid);
    // ---- 4. K-th largest exact score s*, then the reference heap's tie rule (see topk_select_kernel)
    int n_sel = 0;
    if (Keff > 0) {
      const float sstar = key2f(warp_radix_select(hist, nc, (unsigned int)Keff, lane, my_val));
      int run_ge = 0, run_gt = 0, gp_local = 0;
      bool found = false;
      for (int base = 0; base < nc; base += 32) {
        const int k = base + lane;
        const float v = my_val[k];
        const bool real = k < n_valid;
        const bool gt = real && v > sstar, ge = real && v >= sstar;
        const unsigned int bge = __ballot_sync(0xffffffffu, ge), bgt = __ballot_sync(0xffffffffu, gt);
        if (ge && run_ge + __popc(bge & lt_mask) + 1 == Keff) { found = true; gp_local = run_gt + __popc(bgt & lt_mask) + (gt ? 1 : 0); }
        run_ge += __popc(bge);
        run_gt += __popc(bgt);
      }
      const int m = run_gt;
      const unsigned int fb = __ballot_sync(0xffffffffu, found);
      const int gp = __shfl_sync(0xffffffffu, gp_local, fb != 0u ? (__ffs(fb) - 1) : 0);
      for (int k = lane; k < kpow2; k += 32) sort_keys[k] = ~0ull;
      __syncwarp();
      const int tie_lo = m - gp, tie_n = Keff - m;
      int run_eq = 0;
      run_gt = 0;
      for (int base = 0; base < nc; base += 32) {
        const int k = base + lane;
        const float v = my_val[k];
        const bool real = k < n_valid;
        const bool gt = real && v > sstar, eq = real && v == sstar;
        const unsigned int beq = __ballot_sync(0xffffffffu, eq), bgt = __ballot_sync(0xffffffffu, gt);
        const int trank = run_eq + __popc(beq & lt_mask);
        const int gt_before = run_gt + __popc(bgt & lt_mask);
        if (gt || (eq && trank >= tie_lo && trank < tie_lo + tie_n)) {
          int ties_before = trank - tie_lo;
          ties_before = ties_before < 0 ? 0 : (ties_before > tie_n ? tie_n : ties_before);
          const int item = my_groups[k >> 5] * kGroup + (k & 31);
          sort_keys[gt_before + ties_before] = ((unsigned long long)(~f2key(v)) << 32) | (uint32_t)item;
        }
        run_eq += __popc(beq);
        run_gt += __popc(bgt);
      }
      n_sel = Keff;
      __syncwarp();
      for (int kk = 2; kk <= kpow2; kk <<= 1)
        for (int jj = kk >> 1; jj > 0; jj >>= 1) {
          for (int idx = lane; idx < (kpow2 >> 1); idx += 32) {
            const int a = ((idx & ~(jj - 1)) << 1) | (idx & (jj - 1));
            const int c = a | jj;
            const bool up = (a & kk) == 0;
            const unsigned long long ka = sort_keys[a], kc = sort_keys[c];
            if ((ka > kc) == up) { sort_keys[a] = kc; sort_keys[c] = ka; }
          }
          __syncwarp();
        }
    }
    for (int k = lane; k < p.K; k += 32) {
      float v = -INFINITY;
      int idx = -1;
      if (k < n_sel) {
        const unsigned long long key = sort_keys[k];
        v = key2f(~(uint32_t)(key >> 32));
        idx = (int)(uint32_t)key + p.item_offset;
      }
      p.out_val[(size_t)r * p.K + k] = v;
      p.out_idx[(size_t)r * p.K + k] = idx;
    }
    if (lane == 0 && p.out_flags != nullptr) p.out_flags[r] = n_cg;
  }
}

// ------------------------------------------------ stage 2, GROUP-MAJOR re-scoring
// The warp-per-user kernel above copies every candidate group (32 item rows, 8 KB at d = 64) once per user that
// has it: 57 groups x 8 KB = 467 KB of L2 -> SM traffic per user, 12 GB per Gowalla evaluation -- the whole cost of
// stage 2.  A group is a candidate of ~1 200 users; here it is loaded ONCE per CTA and the users stream past it
// (256 B each): ~0.65 GB per evaluation.  Three kernels:
//   s2_candidates : per user (warp) the threshold and the ordered candidate groups; the (user, slot) pairs are
//                   bucketed by group on the spot (every group owns n_u slots)
//   s2_rescore    : CTA per (group, slice): tile in shared memory, one warp per pair, lane l walks ITS item's row in
//                   the reference order (k ascending, fmaf) -- the same bits as exact_dot / the warp kernel
//   s2_select     : per user (warp) step 4 of the warp kernel on the stored scores
// Results are bit-identical to the warp kernel (tests run both).
template <int D>
__global__ void __launch_bounds__(256) s2_candidates_kernel(const Stage2Params p) {
  extern __shared__ __align__(16) float s2c_rows[];                  // [8][cand_stage] when cand_stage > 0
  __shared__ unsigned int hist_all[8][256];
  __shared__ float urow_all[8][D];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned int* hist = hist_all[warp];
  float* urow = urow_all[warp];
  const int gw = blockIdx.x * 8 + warp, n_warps = gridDim.x * 8;
  const unsigned int lt_mask = (1u << lane) - 1u;
  for (int r = gw; r < p.n_u; r += n_warps) {
    const int uid = p.user_rows != nullptr ? p.user_rows[r] : r;
    const float* grow = p.gmax + (size_t)r * p.pitch;
    __syncwarp();
    for (int k = lane; k < D / 4; k += 32) reinterpret_cast<float4*>(urow)[k] = __ldg(p.Uemb + (size_t)uid * (D / 4) + k);
    __syncwarp();
    if (p.cand_stage > 0) {
      // the radix select sweeps the row four times and the compaction once more: 5 x n_u x n_groups x 4 B from L2
      // (420 MB per 16 384-user chunk at 1 281 groups) -- one sweep into shared memory, the rest from there
      float* srow = s2c_rows + (size_t)warp * p.cand_stage;
      const float4* g4 = reinterpret_cast<const float4*>(grow);      // pitch is a multiple of 8 words: rows are 32-byte aligned
      for (int k = lane; k < (p.n_groups + 3) / 4; k += 32) reinterpret_cast<float4*>(srow)[k] = __ldcs(g4 + k);
      __syncwarp();
      grow = srow;
    }
    const unsigned int R = (unsigned int)min(p.K, p.n_groups);
    float thr = key2f(warp_radix_select(hist, p.n_groups, R, lane, grow));
    float keep_from = thr;                                           // tau itself when stage 1 is exact
    if (p.margin_scale > 0.f) {
      float ss = 0.f;
      for (int k = 0; k < D; ++k) ss = fmaf(urow[k], urow[k], ss);
      const float margin = p.margin_scale * sqrtf(ss) * __ldg(p.max_item_norm);      // 2 delta
      keep_from = thr - 0.75f * margin;                              // tau - 1.5 delta  <=  tau - delta  <=  s*
      thr -= margin;
    }
    if (p.u_thr != nullptr && lane == 0) p.u_thr[r] = keep_from;
    int32_t* my_groups = p.u_groups + (size_t)r * p.cmax;
    int n_cg = 0;
    bool overflow = false;
    for (int base = 0; base < p.n_groups; base += 32) {
      const int g = base + lane;
      const bool flag = g < p.n_groups && grow[g] >= thr;
      const unsigned int b = __ballot_sync(0xffffffffu, flag);
      if (n_cg + __popc(b) > p.cmax) { overflow = true; break; }       // warp-uniform
      if (flag) my_groups[n_cg + __popc(b & lt_mask)] = g;
      n_cg += __popc(b);
    }
    if (overflow) {
      if (lane == 0) { p.overflow_list[atomicAdd(p.overflow_count, 1)] = r; p.u_ncg[r] = -1; }
      continue;
    }
    __syncwarp();
    // bucket the (user, slot) pairs by group: every group owns n_u slots (a group is a candidate of every user at
    // most once), so a pair takes the next free one -- no scan, no second pass; the order inside a bucket is
    // irrelevant (each pair's scores land at a fixed place)
    for (int c = lane; c < n_cg; c += 32) {
      const int g = my_groups[c];
      const int pos = atomicAdd(p.g_count + g, 1);
      p.pairs[(size_t)g * p.n_u + pos] = (r << 8) | c;
    }
    if (lane == 0) p.u_ncg[r] = n_cg;
  }
}

#ifndef AGCF_S2_PB
#define AGCF_S2_PB 4            // pairs a warp scores per trip (4: 219 us per chunk)
#endif
constexpr int kS2Slices = 8;               // CTAs per group in s2_rescore (popular groups have >10 000 users)

template <int D>
__global__ void __launch_bounds__(256) s2_rescore_kernel(const Stage2Params p) {
  constexpr int LD = D + 4, V4 = D / 4;
  extern __shared__ __align__(16) unsigned char dyn[];
  float* tile = reinterpret_cast<float*>(dyn);                       // [32][LD]
  float* urow_all = tile + kGroup * LD;                              // [8 warps][PB][D]
  const int g = blockIdx.x, slice = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int cnt = p.g_count[g];
  if (slice * 8 >= cnt) return;                                      // nothing for this slice (uniform per CTA)
  const int32_t* my_pairs = p.pairs + (size_t)g * p.n_u;
  const int rows_here = min(kGroup, p.n_items - g * kGroup);
  const float4* src = p.Iemb + (size_t)g * kGroup * V4;
  // (lane l keeping ITS item's row in registers instead -- no tile reads, only the broadcast user row -- was measured
  //  slower: 494 vs 308 us per chunk; 94 registers halve the resident warps and the per-lane row load is uncoalesced)
  for (int f = threadIdx.x; f < kGroup * V4; f += 256) {
    const int row = f / V4, c4 = f - row * V4;
    const float4 v = row < rows_here ? __ldg(src + f) : make_float4(0.f, 0.f, 0.f, 0.f);
    *reinterpret_cast<float4*>(tile + row * LD + 4 * c4) = v;
  }
  __syncthreads();
  // A warp scores PB pairs per trip: the 32 lanes read 32 different tile rows (4 wavefronts per float4 step), a user
  // row is a broadcast (1 wavefront) -- sharing every tile read between PB users cuts the shared-memory traffic per
  // pair from 5 to (4 + PB) / PB wavefronts per step; it bounded the kernel.
  constexpr int PB = AGCF_S2_PB;
  float* urows = urow_all + warp * PB * D;
  const float* mine_row = tile + lane * LD;
  const int stride = kS2Slices * 8;
  for (int q0 = slice * 8 + warp; q0 < cnt; q0 += PB * stride) {
    int pr[PB];
    uint32_t word[PB];
    __syncwarp();
#pragma unroll
    for (int j = 0; j < PB; ++j) {
      const int q = q0 + j * stride;
      pr[j] = q < cnt ? my_pairs[q] : -1;
      word[j] = 0u;
      if (pr[j] >= 0) {
        const int r = pr[j] >> 8;
        const int uid = p.user_rows != nullptr ? p.user_rows[r] : r;
        for (int k = lane; k < V4; k += 32) reinterpret_cast<float4*>(urows + j * D)[k] = __ldg(p.Uemb + (size_t)uid * V4 + k);
        word[j] = __ldg(p.bits + (size_t)r * p.pitch + g);
      }
    }
    __syncwarp();
    float sc[PB];
#pragma unroll
    for (int j = 0; j < PB; ++j) sc[j] = 0.f;
#pragma unroll 4
    for (int k4 = 0; k4 < V4; ++k4) {
      const float4 v = *reinterpret_cast<const float4*>(mine_row + 4 * k4);
#pragma unroll
      for (int j = 0; j < PB; ++j) {
        const float4 w = *reinterpret_cast<const float4*>(urows + j * D + 4 * k4);
        sc[j] = fmaf(w.x, v.x, sc[j]);
        sc[j] = fmaf(w.y, v.y, sc[j]);
        sc[j] = fmaf(w.z, v.z, sc[j]);
        sc[j] = fmaf(w.w, v.w, sc[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < PB; ++j) {
      if (pr[j] < 0) continue;
      float v = sc[j];
      if (lane >= rows_here) v = -FLT_MAX;
      else if ((word[j] >> lane) & 1u) v = kMasked;
      p.u_val[((size_t)(pr[j] >> 8) * p.cmax + (pr[j] & 255)) * kGroup + lane] = v;
    }
  }
}

template <int D>
__global__ void __launch_bounds__(256) s2_select_kernel(const Stage2Params p) {
  extern __shared__ __align__(16) unsigned char dyn[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int kpow2 = 1;
  while (kpow2 < p.K) kpow2 <<= 1;
  const size_t per_warp = 1024 + (size_t)kpow2 * 8;
  unsigned int* hist = reinterpret_cast<unsigned int*>(dyn + (size_t)warp * per_warp);
  unsigned long long* sort_keys = reinterpret_cast<unsigned long long*>(dyn + (size_t)warp * per_warp + 1024);
  const int gw = blockIdx.x * 8 + warp, n_warps = gridDim.x * 8;
  const unsigned int lt_mask = (1u << lane) - 1u;
  for (int r = gw; r < p.n_u; r += n_warps) {
    const int n_cg = p.u_ncg[r];
    if (n_cg < 0) continue;                                          // overflow user: the block kernel writes its row
    const int32_t* my_groups = p.u_groups + (size_t)r * p.cmax;
    const float* my_val = p.u_val + (size_t)r * p.cmax * kGroup;
    __syncwarp();
    const int nc = n_cg * kGroup;
    int n_valid = nc;
    if (n_cg > 0 && my_groups[n_cg - 1] == p.n_groups - 1) n_valid = nc - (p.n_groups * kGroup - p.n_items);
    const int Keff = min(p.K, n_valid);
    // K-th largest exact score s*, then the reference heap's tie rule (see topk_select_kernel)
    int n_sel = 0;
    if (Keff > 0) {
      const float sstar = key2f(warp_radix_select(hist, nc, (unsigned int)Keff, lane, my_val));
      int run_ge = 0, run_gt = 0, gp_local = 0;
      bool found = false;
      for (int base = 0; base < nc; base += 32) {
        const int k = base + lane;
        const float v = my_val[k];
        const bool real = k < n_valid;
        const bool gt = real && v > sstar, ge = real && v >= sstar;
        const unsigned int bge = __ballot_sync(0xffffffffu, ge), bgt = __ballot_sync(0xffffffffu, gt);
        if (ge && run_ge + __popc(bge & lt_mask) + 1 == Keff) { found = true; gp_local = run_gt + __popc(bgt & lt_mask) + (gt ? 1 : 0); }
        run_ge += __popc(bge);
        run_gt += __popc(bgt);
      }
      const int m = run_gt;
      const unsigned int fb = __ballot_sync(0xffffffffu, found);
      const int gp = __shfl_sync(0xffffffffu, gp_local, fb != 0u ? (__ffs(fb) - 1) : 0);
      for (int k = lane; k < kpow2; k += 32) sort_keys[k] = ~0ull;
      __syncwarp();
      const int tie_lo = m - gp, tie_n = Keff - m;
      int run_eq = 0;
      run_gt = 0;
      for (int base = 0; base < nc; base += 32) {
        const int k = base + lane;
        const float v = my_val[k];
        const bool real = k < n_valid;
        const bool gt = real && v > sstar, eq = real && v == sstar;
        const unsigned int beq = __ballot_sync(0xffffffffu, eq), bgt = __ballot_sync(0xffffffffu, gt);
        const int trank = run_eq + __popc(beq & lt_mask);
        const int gt_before = run_gt + __popc(bgt & lt_mask);
        if (gt || (eq && trank >= tie_lo && trank < tie_lo + tie_n)) {
          int ties_before = trank - tie_lo;
          ties_before = ties_before < 0 ? 0 : (ties_before > tie_n ? tie_n : ties_before);
          const int item = my_groups[k >> 5] * kGroup + (k & 31);
          sort_keys[gt_before + ties_before] = ((unsigned long long)(~f2key(v)) << 32) | (uint32_t)item;
        }
        run_eq += __popc(beq);
        run_gt += __popc(bgt);
      }
      n_sel = Keff;
      __syncwarp();
      for (int kk = 2; kk <= kpow2; kk <<= 1)
        for (int jj = kk >> 1; jj > 0; jj >>= 1) {
          for (int idx = lane; idx < (kpow2 >> 1); idx += 32) {
            const int a = ((idx & ~(jj - 1)) << 1) | (idx & (jj - 1));
            const int c = a | jj;
            const bool up = (a & kk) == 0;
            const unsigned long long ka = sort_keys[a], kc = sort_keys[c];
            if ((ka > kc) == up) { sort_keys[a] = kc; sort_keys[c] = ka; }
          }
          __syncwarp();
        }
    }
    for (int k = lane; k < p.K; k += 32) {
      float v = -INFINITY;
      int idx = -1;
      if (k < n_sel) {
        const unsigned long long key = sort_keys[k];
        v = key2f(~(uint32_t)(key >> 32));
        idx = (int)(uint32_t)key + p.item_offset;
      }
      p.out_val[(size_t)r * p.K + k] = v;
      p.out_idx[(size_t)r * p.K + k] = idx;
    }
    if (lane == 0 && p.out_flags != nullptr) p.out_flags[r] = n_cg;
  }
}

// ------------------------------------- stage 2, group-major, ITEM-compacting variant
// s2_rescore above stores all 32 exact scores of every candidate group (57 x 32 = 1 824 per user at the Gowalla shape)
// and s2_select radix-selects the K-th largest of them in four passes -- yet only ~60 of them can matter: with tau the
// K-th largest stage-1 group maximum and delta the stage-1 error bound, the K-th largest EXACT score s* is >= tau - delta
// (file header), and neither the selection nor the reference's tie rule looks at a score below s*.  s2_candidates
// publishes T_u = tau - 1.5 delta (<= s*), the re-scoring keeps only entries with score >= T_u (a ballot + one atomic per
// pair, {item, score} compacted per user in arrival order), and the per-user selection first orders its <= 128 entries
// by item id (the tie rule is defined on item order) and then runs the SAME selection / tie / sort code on ~60 values
// instead of 1 824.  Users with more than cap_items entries (heavy ties, fewer than K unmasked items) go to the block
// kernel like the candidate-group overflows.  Bit-identical results (tests run all stage-2 variants).
constexpr int kS2ItemCap = 128;

// Re-scoring as a register-tiled product: a CTA owns (group, slice) and walks the group's users in tiles of 128.  The
// group's 32 item rows and the tile's 128 user rows are staged in shared memory; thread (tu, ti) computes a 4 x 4 block
// of (user, item) scores: per float4 step of k it reads 4 + 4 vectors and issues 64 FMAs (the warp-per-pair
// kernel above reads 5 vectors per 16 FMAs and sits on the shared-memory bandwidth).  Every score is still ONE chain
// acc = fmaf(u[k], v[k], acc), k ascending from 0 -- the bits of exact_dot.
// (A software-pipelined form -- a CTA owns several tiles of a group, the next tile's user rows travel global -> shared with
// cp.async while the current one is computed, pair ids / mask words / T_u loaded one tile further ahead -- was built, passed
// the bit-identity tests and measured SLOWER: 1.14-1.18 vs 1.05 ms per evaluation at the Gowalla shape, 5.52 vs 5.18 ms at the
// Amazon-book shape (profiles/r2_eval_rescore_pipelined_experiment.txt): its two 35 KB buffers leave 2 CTAs per SM where this
// kernel runs 4, and 32 resident warps hide the load -> barrier -> compute chain better than the pipeline does.)
constexpr int kS2TU = 128;                 // users per tile

#ifndef AGCF_S2RI_MINB
#define AGCF_S2RI_MINB 4          // 64 registers, no spills: 4 CTAs / SM measured faster than 3 at 80 (profiles/r2_summary.md)
#endif
template <int D>
__global__ void __launch_bounds__(256, AGCF_S2RI_MINB) s2_rescore_items_kernel(const Stage2Params p) {
  constexpr int LD = D + 4, V4 = D / 4;
  extern __shared__ __align__(16) unsigned char dyn[];
  float* tile = reinterpret_cast<float*>(dyn);                       // [32][LD] item rows of the group
  float* urows = tile + kGroup * LD;                                 // [kS2TU][LD] user rows of the tile
  int* u_r = reinterpret_cast<int*>(urows + kS2TU * LD);             // [kS2TU] user position r (-1: none)
  uint32_t* u_word = reinterpret_cast<uint32_t*>(u_r + kS2TU);       // [kS2TU] train-item mask word of (user, group)
  float* u_keep = reinterpret_cast<float*>(u_word + kS2TU);          // [kS2TU] T_u
  const int g = blockIdx.x, slice = blockIdx.y;
  const int tid = threadIdx.x;
  const int cnt = p.g_count[g];
  if (slice * kS2TU >= cnt) return;                                  // nothing for this slice (uniform per CTA)
  const int32_t* my_pairs = p.pairs + (size_t)g * p.n_u;
  const int rows_here = min(kGroup, p.n_items - g * kGroup);
  const float4* src = p.Iemb + (size_t)g * kGroup * V4;
  for (int f = tid; f < kGroup * V4; f += 256) {
    const int row = f / V4, c4 = f - row * V4;
    const float4 v = row < rows_here ? __ldg(src + f) : make_float4(0.f, 0.f, 0.f, 0.f);
    *reinterpret_cast<float4*>(tile + row * LD + 4 * c4) = v;
  }
  // thread (tu, ti): users tu + 32 a, items ti + 8 b (a, b < 4) -- the threads of a warp read CONSECUTIVE tile rows, whose
  // stride of LD = D + 4 floats puts them 4 banks apart: conflict-free LDS.128
  const int tu = tid >> 3, ti = tid & 7;
  for (int t0 = slice * kS2TU; t0 < cnt; t0 += kS2Slices * kS2TU) {
    __syncthreads();                                                 // the previous tile's rows are no longer read
    if (tid < kS2TU) {
      const int q = t0 + tid;
      int r = -1;
      uint32_t word = 0u;
      float keep_from = 0.f;
      if (q < cnt) {
        r = my_pairs[q] >> 8;
        word = __ldg(p.bits + (size_t)r * p.pitch + g);
        keep_from = __ldg(p.u_thr + r);
      }
      u_r[tid] = r; u_word[tid] = word; u_keep[tid] = keep_from;
    }
    for (int f = tid; f < kS2TU * V4; f += 256) {
      const int row = f / V4, c4 = f - row * V4;
      const int q = t0 + row;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (q < cnt) {
        const int r = my_pairs[q] >> 8;
        if (p.Udense != nullptr) {
          v = __ldg(p.Udense + (size_t)r * V4 + c4);
        } else {
          const int uid = p.user_rows != nullptr ? p.user_rows[r] : r;
          v = __ldg(p.Uemb + (size_t)uid * V4 + c4);
        }
      }
      *reinterpret_cast<float4*>(urows + row * LD + 4 * c4) = v;
    }
    __syncthreads();
    float acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
#pragma unroll 4
    for (int k4 = 0; k4 < V4; ++k4) {
      float4 uv[4], iv[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) uv[a] = *reinterpret_cast<const float4*>(urows + (tu + 32 * a) * LD + 4 * k4);
#pragma unroll
      for (int b = 0; b < 4; ++b) iv[b] = *reinterpret_cast<const float4*>(tile + (ti + 8 * b) * LD + 4 * k4);
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          float s_ = acc[a][b];
          s_ = fmaf(uv[a].x, iv[b].x, s_);
          s_ = fmaf(uv[a].y, iv[b].y, s_);
          s_ = fmaf(uv[a].z, iv[b].z, s_);
          s_ = fmaf(uv[a].w, iv[b].w, s_);
          acc[a][b] = s_;
        }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int lu = tu + 32 * a;
      const int r = u_r[lu];
      if (r < 0) continue;
      const uint32_t word = u_word[lu];
      const float keep_from = u_keep[lu];
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int it = ti + 8 * b;
        if (it >= rows_here) continue;
        float v = acc[a][b];
        if ((word >> it) & 1u) v = kMasked;
        if (v >= keep_from) {                                        // ~3 % of the scores survive
          const int pos = atomicAdd(p.u_cnt + r, 1);
          if (pos < p.cap_items) p.u_items[(size_t)r * p.cap_items + pos] = make_int2(g * kGroup + it, __float_as_int(v));
        }
      }
    }
  }
}

template <int D>
__global__ void __launch_bounds__(256) s2_select_items_kernel(const Stage2Params p) {
  extern __shared__ __align__(16) unsigned char dyn[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int kpow2 = 1;
  while (kpow2 < p.K) kpow2 <<= 1;
  // per warp: histogram (1 KB), K sort keys, the entries as 64-bit keys / as (score, item) arrays
  const size_t per_warp = 1024 + (size_t)kpow2 * 8 + (size_t)kS2ItemCap * 16;
  unsigned char* mine = dyn + (size_t)warp * per_warp;
  unsigned int* hist = reinterpret_cast<unsigned int*>(mine);
  unsigned long long* sort_keys = reinterpret_cast<unsigned long long*>(mine + 1024);
  unsigned long long* ekeys = reinterpret_cast<unsigned long long*>(mine + 1024 + (size_t)kpow2 * 8);
  float* my_val = reinterpret_cast<float*>(ekeys + kS2ItemCap);
  int* my_item = reinterpret_cast<int*>(my_val + kS2ItemCap);
  const int gw = blockIdx.x * 8 + warp, n_warps = gridDim.x * 8;
  const unsigned int lt_mask = (1u << lane) - 1u;
  for (int r = gw; r < p.n_u; r += n_warps) {
    const int n_cg = p.u_ncg[r];
    if (n_cg < 0) continue;                                          // candidate-group overflow: already on the list
    const int n = p.u_cnt[r];
    const int Keff = min(p.K, p.n_items);
    if (n > p.cap_items || n < Keff) {                               // too many survivors (ties / few unmasked items)
      if (lane == 0) p.overflow_list[atomicAdd(p.overflow_count, 1)] = r;
      continue;
    }
    __syncwarp();
    // order the entries by item id: the tie rule of the reference's heap is defined on item order
    for (int k = lane; k < kS2ItemCap; k += 32) {
      unsigned long long key = ~0ull;
      if (k < n) {
        const int2 e = p.u_items[(size_t)r * p.cap_items + k];
        key = ((unsigned long long)(uint32_t)e.x << 32) | (uint32_t)e.y;
      }
      ekeys[k] = key;
    }
    __syncwarp();
    for (int kk = 2; kk <= kS2ItemCap; kk <<= 1)
      for (int jj = kk >> 1; jj > 0; jj >>= 1) {
        for (int idx = lane; idx < (kS2ItemCap >> 1); idx += 32) {
          const int a = ((idx & ~(jj - 1)) << 1) | (idx & (jj - 1));
          const int c = a | jj;
          const bool up = (a & kk) == 0;
          const unsigned long long ka = ekeys[a], kc = ekeys[c];
          if ((ka > kc) == up) { ekeys[a] = kc; ekeys[c] = ka; }
        }
        __syncwarp();
      }
    for (int k = lane; k < n; k += 32) {
      const unsigned long long key = ekeys[k];
      my_item[k] = (int)(uint32_t)(key >> 32);
      my_val[k] = __uint_as_float((uint32_t)key);
    }
    __syncwarp();
    // K-th largest exact score s*, then the reference heap's tie rule (see topk_select_kernel) -- on n entries
    const float sstar = key2f(warp_radix_select(hist, n, (unsigned int)Keff, lane, my_val));
    int run_ge = 0, run_gt = 0, gp_local = 0;
    bool found = false;
    for (int base = 0; base < n; base += 32) {
      const int k = base + lane;
      const bool real = k < n;
      const float v = real ? my_val[k] : 0.f;
      const bool gt = real && v > sstar, ge = real && v >= sstar;
      const unsigned int bge = __ballot_sync(0xffffffffu, ge), bgt = __ballot_sync(0xffffffffu, gt);
      if (ge && run_ge + __popc(bge & lt_mask) + 1 == Keff) { found = true; gp_local = run_gt + __popc(bgt & lt_mask) + (gt ? 1 : 0); }
      run_ge += __popc(bge);
      run_gt += __popc(bgt);
    }
    const int m = run_gt;
    const unsigned int fb = __ballot_sync(0xffffffffu, found);
    const int gp = __shfl_sync(0xffffffffu, gp_local, fb != 0u ? (__ffs(fb) - 1) : 0);
    for (int k = lane; k < kpow2; k += 32) sort_keys[k] = ~0ull;
    __syncwarp();
    const int tie_lo = m - gp, tie_n = Keff - m;
    int run_eq = 0;
    run_gt = 0;
    for (int base = 0; base < n; base += 32) {
      const int k = base + lane;
      const bool real = k < n;
      const float v = real ? my_val[k] : 0.f;
      const bool gt = real && v > sstar, eq = real && v == sstar;
      const unsigned int beq = __ballot_sync(0xffffffffu, eq), bgt = __ballot_sync(0xffffffffu, gt);
      const int trank = run_eq + __popc(beq & lt_mask);
      const int gt_before = run_gt + __popc(bgt & lt_mask);
      if (gt || (eq && trank >= tie_lo && trank < tie_lo + tie_n)) {
        int ties_before = trank - tie_lo;
        ties_before = ties_before < 0 ? 0 : (ties_before > tie_n ? tie_n : ties_before);
        sort_keys[gt_before + ties_before] = ((unsigned long long)(~f2key(v)) << 32) | (uint32_t)my_item[k];
      }
      run_eq += __popc(beq);
      run_gt += __popc(bgt);
    }
    __syncwarp();
    for (int kk = 2; kk <= kpow2; kk <<= 1)
      for (int jj = kk >> 1; jj > 0; jj >>= 1) {
        for (int idx = lane; idx < (kpow2 >> 1); idx += 32) {
          const int a = ((idx & ~(jj - 1)) << 1) | (idx & (jj - 1));
          const int c = a | jj;
          const bool up = (a & kk) == 0;
          const unsigned long long ka = sort_keys[a], kc = sort_keys[c];
          if ((ka > kc) == up) { sort_keys[a] = kc; sort_keys[c] = ka; }
        }
        __syncwarp();
      }
    for (int k = lane; k < p.K; k += 32) {
      float v = -INFINITY;
      int idx = -1;
      if (k < Keff) {
        const unsigned long long key = sort_keys[k];
        v = key2f(~(uint32_t)(key >> 32));
        idx = (int)(uint32_t)key + p.item_offset;
      }
      p.out_val[(size_t)r * p.K + k] = v;
      p.out_idx[(size_t)r * p.K + k] = idx;
    }
    if (lane == 0 && p.out_flags != nullptr) p.out_flags[r] = n_cg;
  }
}

// --------------------------------------------------------------------- predict
template <int D>
__global__ void __launch_bounds__(256) score_rows_kernel(const float4* __restrict__ Uemb, const int32_t* __restrict__ user_rows,
                                                         const float4* __restrict__ Iemb, int n_items, float* __restrict__ out) {
  __shared__ __align__(16) float urow[D];
  const int r = blockIdx.y;
  const int uid = user_rows != nullptr ? user_rows[r] : r;
  if (threadIdx.x < D / 4) reinterpret_cast<float4*>(urow)[threadIdx.x] = __ldg(Uemb + (size_t)uid * (D / 4) + threadIdx.x);
  __syncthreads();
  const int item = blockIdx.x * blockDim.x + threadIdx.x;
  if (item < n_items) out[(size_t)r * n_items + item] = exact_dot<D>(urow, Iemb + (size_t)item * (D / 4));
}

// ------------------------------------------------------------------ top-K merge
__global__ void __launch_bounds__(128) topk_merge_kernel(const float* __restrict__ vals, const int32_t* __restrict__ idx,
                                                         int P, int n_u, int K, int pow2,
                                                         float* __restrict__ out_val, int32_t* __restrict__ out_idx) {
  extern __shared__ unsigned long long mk[];
  const int r = blockIdx.x, tid = threadIdx.x;
  for (int k = tid; k < pow2; k += blockDim.x) {
    unsigned long long key = ~0ull;
    if (k < P * K) {
      const int pp = k / K, kk = k - pp * K;
      const size_t src = ((size_t)pp * n_u + r) * K + kk;
      const int id = idx[src];
      if (id >= 0) key = ((unsigned long long)(~f2key(vals[src])) << 32) | (uint32_t)id;
    }
    mk[k] = key;
  }
  __syncthreads();
  for (int kk = 2; kk <= pow2; kk <<= 1)
    for (int jj = kk >> 1; jj > 0; jj >>= 1) {
      for (int i2 = tid; i2 < (pow2 >> 1); i2 += blockDim.x) {
        const int a = ((i2 & ~(jj - 1)) << 1) | (i2 & (jj - 1));
        const int c = a | jj;
        const bool up = (a & kk) == 0;
        const unsigned long long ka = mk[a], kc = mk[c];
        if ((ka > kc) == up) { mk[a] = kc; mk[c] = ka; }
      }
      __syncthreads();
    }
  for (int k = tid; k < K; k += blockDim.x) {
    const unsigned long long key = mk[k];
    const bool ok = key != ~0ull;
    out_val[(size_t)r * K + k] = ok ? key2f(~(uint32_t)(key >> 32)) : -INFINITY;
    out_idx[(size_t)r * K + k] = ok ? (int)(uint32_t)key : -1;
  }
}

// ---------------------------------------------------------------------- metrics
// One WARP per user: the K ids of a user are read coalesced, every lane runs the binary search of its id, and the hits are
// collected with a ballot; lane 0 then adds inv_log[k] over the set bits in ASCENDING k -- the same fp64 summation order as a
// sequential loop over k (the metric strings are compared character by character with the reference's).  A thread per user
// walked its 50 ids one dependent search after the other behind strided loads: ~0.15 ms of the 1.2 ms evaluation.
__global__ void __launch_bounds__(256) rank_metrics_kernel(const int32_t* __restrict__ topk_idx, int K,
                                                           const int32_t* __restrict__ t_rowptr, const int32_t* __restrict__ t_items,
                                                           const int32_t* __restrict__ test_total, int n_u,
                                                           const int32_t* __restrict__ cutoffs, int nc,
                                                           const double* __restrict__ inv_log, double* __restrict__ out) {
  const int r = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (r >= n_u) return;                                              // warp-uniform
  const int s = t_rowptr[r], e = t_rowptr[r + 1];
  for (int c = 0; c < nc; ++c) {
    const int n = min(cutoffs[c], K);
    double hits = 0.0, dcg = 0.0, idcg = 0.0;
    for (int base = 0; base < n; base += 32) {
      const int k = base + lane;
      bool hit = false;
      if (k < n) {
        const int it = topk_idx[(size_t)r * K + k];
        if (it >= 0) {
          int lo = s, hi = e;
          while (lo < hi) { const int mid = (lo + hi) >> 1; if (t_items[mid] < it) lo = mid + 1; else hi = mid; }
          hit = lo < e && t_items[lo] == it;
        }
      }
      unsigned int m = __ballot_sync(0xffffffffu, hit);
      if (lane == 0) {
        while (m != 0u) {
          const int b = __ffs(m) - 1;
          hits += 1.0;
          dcg += inv_log[base + b];
          m &= m - 1u;
        }
      }
    }
    if (lane == 0) {
      const int ni = min(test_total[r], cutoffs[c]);
      for (int k = 0; k < ni; ++k) idcg += inv_log[k];
      double* o = out + ((size_t)r * nc + c) * 3;
      o[0] = hits; o[1] = dcg; o[2] = idcg;
    }
  }
}

// provided by score_tc.cu (tcgen05 TF32 group-max GEMM)
int launch_group_max_tc(const float* Uemb, const int32_t* user_rows, int n_u, const float* Iemb, int n_items, int d,
                        const uint32_t* bits, int n_groups, int pitch, float* gmax, float* u_dense, cudaStream_t st);

struct WsLayout {
  size_t bits_off, gmax_off, norm_off, groups_off, cval_off, udense_off, wgroups_off, wval_off, ovf_off, total;
  size_t ugroups_off, uncg_off, uval_off, gcount_off, pairs_off;   // group-major stage 2
  size_t uthr_off, ucnt_off, uitems_off;                            // its item-compacting variant
  int n_groups, pitch, grid2, grid_w, cmax, wpc;
};

constexpr int kStage2OverflowCtas = 32;      // block-kernel CTAs that mop up users with > cmax candidate groups
constexpr int kStage2CandMax = 160;          // candidate groups a warp can hold (mean 55, max 72 seen at K = 50)

// stage 2 implementation: 2 = group-major re-scoring that keeps only the entries >= T_u (default), 1 = group-major, all 32
// scores of every candidate group stored and selected from, 0 = the warp-per-user kernel (re-loads every candidate group
// per user); identical results
static int stage2_impl() {
  const char* e = getenv("AGCF_STAGE2_IMPL");
  return e ? atoi(e) : 2;
}

static int stage2_ctas_per_sm() {
  static int v = 0;
  if (v == 0) {
    const char* e = getenv("AGCF_STAGE2_CTAS_PER_SM");      // tuning hook
    v = e ? atoi(e) : 5;
    if (v < 1) v = 1;
    if (v > 16) v = 16;
  }
  return v;
}

static WsLayout ws_layout(int n_u, int n_items, int d) {
  WsLayout L;
  L.n_groups = (n_items + kGroup - 1) / kGroup;
  L.pitch = (L.n_groups + 7) & ~7;                               // 32-byte rows: vector loads / stores in the tcgen05 epilogue
  L.grid2 = kStage2OverflowCtas;
  int cmax = kStage2CandMax;
  if (const char* e = getenv("AGCF_STAGE2_CMAX")) {                // test hook: force the overflow path
    const int v = atoi(e);
    if (v >= 1 && v < cmax) cmax = v;
  }
  L.cmax = L.n_groups < cmax ? L.n_groups : cmax;
  const int wpc = d <= 64 ? 4 : (d == 128 ? 2 : 1);                // S2W<D>::WPC
  const int want = (n_u + wpc - 1) / wpc;                          // one warp per user
  const int resident = stage2_ctas_per_sm() * kSMs;
  L.grid_w = want < resident ? (want > 0 ? want : 1) : resident;
  L.wpc = wpc;
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  size_t off = 0;
  L.bits_off = off; off = up(off + (size_t)n_u * L.pitch * 4);
  L.gmax_off = off; off = up(off + (size_t)n_u * L.pitch * 4);
  L.norm_off = off; off = up(off + 256);
  L.groups_off = off; off = up(off + (size_t)L.grid2 * L.n_groups * 4);
  L.cval_off = off; off = up(off + (size_t)L.grid2 * L.n_groups * kGroup * 4);
  L.udense_off = off; off = up(off + (size_t)n_u * d * 4);          // gathered user rows for the TMA path
  L.wgroups_off = off; off = up(off + (size_t)L.grid_w * L.wpc * L.cmax * 4);
  L.wval_off = off; off = up(off + (size_t)L.grid_w * L.wpc * L.cmax * kGroup * 4);
  L.ovf_off = off; off = up(off + ((size_t)n_u + 64) * 4);          // [0] = count, [64 ..] = list
  L.ugroups_off = off; off = up(off + (size_t)n_u * L.cmax * 4);
  L.uncg_off = off; off = up(off + (size_t)n_u * 4);
  L.uval_off = off; off = up(off + (size_t)n_u * L.cmax * kGroup * 4);
  L.gcount_off = off; off = up(off + ((size_t)L.n_groups + 1) * 4);
  L.pairs_off = off; off = up(off + (size_t)L.n_groups * n_u * 4);
  L.uthr_off = off; off = up(off + (size_t)n_u * 4);
  L.ucnt_off = off; off = up(off + (size_t)n_u * 4);
  L.uitems_off = off; off = up(off + (size_t)n_u * kS2ItemCap * 8);
  L.total = off;
  return L;
}

}  // namespace agcf

using namespace agcf;

// stages 0 and 1 of agcf_score_topk: mask bits, then the masked group maxima (impl 1: tcgen05 TF32 GEMM, impl 0: fp32)
static int run_stage01(const float* Uemb, const int32_t* user_rows, int n_u, const float* Iemb, int n_items, int d,
                       const int32_t* mask_rowptr, const int32_t* mask_items, int item_offset, int impl, const WsLayout& L,
                       unsigned char* base, cudaStream_t st, float* margin_out, bool keep_mask_bits = false) {
  uint32_t* bits = reinterpret_cast<uint32_t*>(base + L.bits_off);
  float* gmax = reinterpret_cast<float*>(base + L.gmax_off);
  float* norm = reinterpret_cast<float*>(base + L.norm_off);
  const float4* U4 = reinterpret_cast<const float4*>(Uemb);
  const float4* I4 = reinterpret_cast<const float4*>(Iemb);
  *margin_out = 0.f;
  // stage 0 (skipped when the caller vouches for the bits of the previous call: AGCF_TOPK_KEEP_MASK_BITS)
  if (!keep_mask_bits) AGCF_CUDA_OK(cudaMemsetAsync(bits, 0, (size_t)n_u * L.pitch * 4, st));
  if (mask_rowptr != nullptr && !keep_mask_bits) {
    mask_bits_kernel<<<(unsigned)((n_u + 7) / 8), 256, 0, st>>>(user_rows, n_u, mask_rowptr, mask_items, n_items, item_offset, L.pitch, bits);
    AGCF_LAUNCH_OK();
  }
  // stage 1
  if (impl == 1) {
    AGCF_CUDA_OK(cudaMemsetAsync(norm, 0, 4, st));
#define AGCF_NORM(DD) max_row_norm_kernel<DD><<<(unsigned)((n_items + 255) / 256), 256, 0, st>>>(I4, n_items, norm);
    switch (d) { case 8: AGCF_NORM(8) break; case 16: AGCF_NORM(16) break; case 32: AGCF_NORM(32) break; case 64: AGCF_NORM(64) break; case 128: AGCF_NORM(128) break; case 256: AGCF_NORM(256) break; }
#undef AGCF_NORM
    AGCF_LAUNCH_OK();
    const int rc = launch_group_max_tc(Uemb, user_rows, n_u, Iemb, n_items, d, bits, L.n_groups, L.pitch, gmax,
                                       reinterpret_cast<float*>(base + L.udense_off), st);
    if (rc != AGCF_OK) return rc;
    *margin_out = 2.0f * 1.01f * 0.001953125f;      // 2 * delta, delta = 1.01 * 2^-9 * |u| * max|v|
  } else {
    const int n_tiles = (n_items + S1_TI - 1) / S1_TI;
    const int u_tiles = (n_u + S1_TU - 1) / S1_TU;
    int splits = (4 * kSMs * 3 + u_tiles - 1) / u_tiles;          // aim at >= 3 waves of 4 CTAs/SM
    if (splits < 1) splits = 1;
    if (splits > n_tiles) splits = n_tiles;
    if (splits > 65535) splits = 65535;
    const int tps = (n_tiles + splits - 1) / splits;
    splits = (n_tiles + tps - 1) / tps;
    dim3 grid((unsigned)u_tiles, (unsigned)splits);
#define AGCF_S1(DD)                                                                                           \
  {                                                                                                           \
    AGCF_CUDA_OK(cudaFuncSetAttribute(group_max_fp32_kernel<DD>, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                                      (int)S1Smem<DD>::bytes));                                               \
    group_max_fp32_kernel<DD><<<grid, 256, S1Smem<DD>::bytes, st>>>(U4, user_rows, n_u, I4, n_items, bits,    \
                                                                    L.n_groups, L.pitch, tps, gmax);          \
  }
    switch (d) { case 8: AGCF_S1(8) break; case 16: AGCF_S1(16) break; case 32: AGCF_S1(32) break; case 64: AGCF_S1(64) break; case 128: AGCF_S1(128) break; case 256: AGCF_S1(256) break; }
#undef AGCF_S1
    AGCF_LAUNCH_OK();
  }
  return AGCF_OK;
}

extern "C" int64_t agcf_score_topk_ws_bytes(int32_t n_u, int32_t n_items, int32_t d, int32_t K) {
  if (n_u < 0 || n_items <= 0 || K <= 0) return AGCF_EINVAL;
  if (!supported_d(d) || K > 1024) return AGCF_EUNSUPPORTED;
  return (int64_t)ws_layout(n_u, n_items, d).total;
}

extern "C" int agcf_score_group_max(const float* Uemb, const int32_t* user_rows, int32_t n_u,
                                    const float* Iemb, int32_t n_items, int32_t d,
                                    const int32_t* mask_rowptr, const int32_t* mask_items, int32_t item_offset, int32_t impl,
                                    float* gmax_out, void* ws, int64_t ws_bytes, agcf_stream_t stream) {
  if (!Uemb || !Iemb || !ws || n_u < 0 || n_items <= 0) return AGCF_EINVAL;
  if ((mask_rowptr == nullptr) != (mask_items == nullptr)) return AGCF_EINVAL;
  if (!supported_d(d) || (impl != 0 && impl != 1)) return AGCF_EUNSUPPORTED;
  if (!aligned16(Uemb) || !aligned16(Iemb) || (reinterpret_cast<uintptr_t>(ws) & 255u)) return AGCF_EINVAL;
  if (n_u == 0) return AGCF_OK;
  const WsLayout L = ws_layout(n_u, n_items, d);
  if ((int64_t)L.total > ws_bytes) return AGCF_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* base = reinterpret_cast<unsigned char*>(ws);
  float margin = 0.f;
  const int rc = run_stage01(Uemb, user_rows, n_u, Iemb, n_items, d, mask_rowptr, mask_items, item_offset, impl, L, base, st, &margin);
  if (rc != AGCF_OK) return rc;
  if (gmax_out != nullptr)                                            // [n_u][n_groups] dense copy of the pitched rows
    AGCF_CUDA_OK(cudaMemcpy2DAsync(gmax_out, (size_t)L.n_groups * 4, base + L.gmax_off, (size_t)L.pitch * 4,
                                   (size_t)L.n_groups * 4, (size_t)n_u, cudaMemcpyDeviceToDevice, st));
  return AGCF_OK;
}

extern "C" int agcf_score_topk(const float* Uemb, const int32_t* user_rows, int32_t n_u,
                               const float* Iemb, int32_t n_items, int32_t d,
                               const int32_t* mask_rowptr, const int32_t* mask_items,
                               int32_t K, int32_t item_offset, int32_t impl,
                               float* out_val, int32_t* out_idx, int32_t* out_flags,
                               void* ws, int64_t ws_bytes, agcf_stream_t stream) {
  if (!Uemb || !Iemb || !out_val || !out_idx || !ws || n_u < 0 || n_items <= 0 || K <= 0) return AGCF_EINVAL;
  if ((mask_rowptr == nullptr) != (mask_items == nullptr)) return AGCF_EINVAL;
  const bool keep_mask_bits = (impl & AGCF_TOPK_KEEP_MASK_BITS) != 0;
  impl &= ~AGCF_TOPK_KEEP_MASK_BITS;
  if (!supported_d(d) || K > 1024 || (impl != 0 && impl != 1)) return AGCF_EUNSUPPORTED;
  if (!aligned16(Uemb) || !aligned16(Iemb) || (reinterpret_cast<uintptr_t>(ws) & 255u)) return AGCF_EINVAL;
  if (n_u == 0) return AGCF_OK;
  const WsLayout L = ws_layout(n_u, n_items, d);
  if ((int64_t)L.total > ws_bytes) return AGCF_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* base = reinterpret_cast<unsigned char*>(ws);
  uint32_t* bits = reinterpret_cast<uint32_t*>(base + L.bits_off);
  float* gmax = reinterpret_cast<float*>(base + L.gmax_off);
  float* norm = reinterpret_cast<float*>(base + L.norm_off);
  const float4* U4 = reinterpret_cast<const float4*>(Uemb);
  const float4* I4 = reinterpret_cast<const float4*>(Iemb);

  float margin_scale = 0.f;
  {
    const int rc = run_stage01(Uemb, user_rows, n_u, Iemb, n_items, d, mask_rowptr, mask_items, item_offset, impl, L, base, st,
                               &margin_scale, keep_mask_bits);
    if (rc != AGCF_OK) return rc;
  }
  // stage 2
  Stage2Params p;
  p.Uemb = U4; p.user_rows = user_rows; p.n_u = n_u; p.Iemb = I4; p.n_items = n_items;
  p.bits = bits; p.gmax = gmax; p.n_groups = L.n_groups; p.pitch = L.pitch; p.K = K; p.item_offset = item_offset;
  p.margin_scale = margin_scale; p.max_item_norm = norm; p.cand_stage = 0;
  p.out_val = out_val; p.out_idx = out_idx; p.out_flags = out_flags;
  p.cand_groups = reinterpret_cast<int32_t*>(base + L.groups_off);
  p.cand_val = reinterpret_cast<float*>(base + L.cval_off);
  int32_t* ovf = reinterpret_cast<int32_t*>(base + L.ovf_off);
  p.list = ovf + 64; p.list_count = ovf;
  p.cmax = L.cmax;
  p.w_groups = reinterpret_cast<int32_t*>(base + L.wgroups_off);
  p.w_val = reinterpret_cast<float*>(base + L.wval_off);
  p.overflow_list = ovf + 64; p.overflow_count = ovf;
  AGCF_CUDA_OK(cudaMemsetAsync(ovf, 0, 4, st));
  p.u_groups = reinterpret_cast<int32_t*>(base + L.ugroups_off);
  p.u_ncg = reinterpret_cast<int32_t*>(base + L.uncg_off);
  p.u_val = reinterpret_cast<float*>(base + L.uval_off);
  p.g_count = reinterpret_cast<int32_t*>(base + L.gcount_off);
  p.pairs = reinterpret_cast<int32_t*>(base + L.pairs_off);
  p.u_thr = nullptr; p.u_cnt = nullptr; p.u_items = nullptr; p.cap_items = kS2ItemCap;
  p.Udense = (impl == 1 && user_rows != nullptr && d <= 128) ? reinterpret_cast<const float4*>(base + L.udense_off) : nullptr;
  int kpow2 = 1;
  while (kpow2 < K) kpow2 <<= 1;
  const size_t dyn = (size_t)kpow2 * 8;
  if (stage2_impl() >= 1 && n_u < (1 << 23) && L.cmax <= 256) {
    // the item-compacting variant needs T_u <= s*, which the file header proves for K <= n_groups; with few groups (tiny
    // item tables) nearly every item is wanted anyway and the plain group-major kernels run
    const bool items = stage2_impl() == 2 && L.n_groups >= 2 * K;
    if (items) {
      p.u_thr = reinterpret_cast<float*>(base + L.uthr_off);
      p.u_cnt = reinterpret_cast<int32_t*>(base + L.ucnt_off);
      p.u_items = reinterpret_cast<int2*>(base + L.uitems_off);
      AGCF_CUDA_OK(cudaMemsetAsync(p.u_cnt, 0, (size_t)n_u * 4, st));
    }
    // group-major: candidates -> per-group pair lists -> re-score each group's tile once per CTA -> select
    AGCF_CUDA_OK(cudaMemsetAsync(p.g_count, 0, ((size_t)L.n_groups + 1) * 4, st));
    const unsigned warp_grid = (unsigned)min((n_u + 7) / 8, 8 * kSMs);
    const size_t dyn_sel = 8 * (1024 + (size_t)kpow2 * 8);
    const size_t dyn_sel_items = 8 * (1024 + (size_t)kpow2 * 8 + (size_t)kS2ItemCap * 16);
    if (dyn_sel_items > 200 * 1024) return AGCF_EUNSUPPORTED;
    // the group-maxima row of a warp's user staged in shared memory while 8 rows fit next to the static 10 KB
    // (two CTAs per SM at least): up to ~2 800 groups = 90 k items; wider item tables read the row from L2 as before
    static const bool stage_env = [] { const char* e = getenv("AGCF_S2_CAND_STAGE"); return e == nullptr || atoi(e) != 0; }();
    const int stage_words = (L.n_groups + 3) / 4 * 4;
    p.cand_stage = (stage_env && (size_t)stage_words * 4 * 8 <= 96 * 1024) ? stage_words : 0;
    const size_t dyn_cand = (size_t)p.cand_stage * 4 * 8;
#define AGCF_S2G(DD)                                                                                             \
  {                                                                                                              \
    const size_t dyn_r = ((size_t)kGroup * (DD + 4) + 8 * AGCF_S2_PB * DD) * 4;   /* tile + 8 warps x PB user rows */ \
    if (dyn_r > 48 * 1024)                                                                                       \
      AGCF_CUDA_OK(cudaFuncSetAttribute(s2_rescore_kernel<DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_r)); \
    if (dyn_sel > 48 * 1024)                                                                                     \
      AGCF_CUDA_OK(cudaFuncSetAttribute(s2_select_kernel<DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_sel)); \
    if (dyn_cand + 12 * 1024 > 48 * 1024)   /* static 10 KB + dynamic beyond the 48 KB default */                \
      AGCF_CUDA_OK(cudaFuncSetAttribute(s2_candidates_kernel<DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_cand)); \
    s2_candidates_kernel<DD><<<warp_grid, 256, dyn_cand, st>>>(p);                                               \
    if (items) {                                                                                                 \
      const size_t dyn_ri = ((size_t)(kGroup + kS2TU) * (DD + 4) + 3 * kS2TU) * 4;   /* item tile + user tile + per-user words */ \
      if (dyn_ri > 48 * 1024)                                                                                    \
        AGCF_CUDA_OK(cudaFuncSetAttribute(s2_rescore_items_kernel<DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_ri)); \
      if (dyn_sel_items > 48 * 1024)                                                                             \
        AGCF_CUDA_OK(cudaFuncSetAttribute(s2_select_items_kernel<DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_sel_items)); \
      s2_rescore_items_kernel<DD><<<dim3((unsigned)L.n_groups, kS2Slices), 256, dyn_ri, st>>>(p);                \
      s2_select_items_kernel<DD><<<warp_grid, 256, dyn_sel_items, st>>>(p);                                      \
    } else {                                                                                                     \
      s2_rescore_kernel<DD><<<dim3((unsigned)L.n_groups, kS2Slices), 256, dyn_r, st>>>(p);                       \
      s2_select_kernel<DD><<<warp_grid, 256, dyn_sel, st>>>(p);                                                  \
    }                                                                                                            \
    topk_select_kernel<DD><<<(unsigned)L.grid2, 256, dyn, st>>>(p);                                              \
  }
    switch (d) { case 8: AGCF_S2G(8) break; case 16: AGCF_S2G(16) break; case 32: AGCF_S2G(32) break; case 64: AGCF_S2G(64) break; case 128: AGCF_S2G(128) break; case 256: AGCF_S2G(256) break; }
#undef AGCF_S2G
    AGCF_LAUNCH_OK();
    return AGCF_OK;
  }
  // warp per user, then the block kernel on the users the warp kernel could not hold (normally none)
#define AGCF_S2(DD)                                                                                              \
  {                                                                                                              \
    const size_t dyn_w = S2W<DD>::WPC * S2W<DD>::per_warp(kpow2);                                                \
    if (dyn_w > 200 * 1024) return AGCF_EUNSUPPORTED;                                                            \
    if (dyn_w > 48 * 1024)                                                                                       \
      AGCF_CUDA_OK(cudaFuncSetAttribute(topk_select_warp_kernel<DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_w)); \
    topk_select_warp_kernel<DD><<<(unsigned)L.grid_w, 32 * S2W<DD>::WPC, dyn_w, st>>>(p);                        \
    topk_select_kernel<DD><<<(unsigned)L.grid2, 256, dyn, st>>>(p);                                              \
  }
  switch (d) { case 8: AGCF_S2(8) break; case 16: AGCF_S2(16) break; case 32: AGCF_S2(32) break; case 64: AGCF_S2(64) break; case 128: AGCF_S2(128) break; case 256: AGCF_S2(256) break; }
#undef AGCF_S2
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int agcf_topk_merge(const float* vals, const int32_t* idx, int32_t P, int32_t n_u, int32_t K,
                               float* out_val, int32_t* out_idx, agcf_stream_t stream) {
  if (!vals || !idx || !out_val || !out_idx || P <= 0 || n_u < 0 || K <= 0) return AGCF_EINVAL;
  if ((long long)P * K > 8192) return AGCF_EUNSUPPORTED;
  if (n_u == 0) return AGCF_OK;
  int pow2 = 2;
  while (pow2 < P * K) pow2 <<= 1;
  if (pow2 * 8 > 48 * 1024) {
    AGCF_CUDA_OK(cudaFuncSetAttribute(topk_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, pow2 * 8));
  }
  topk_merge_kernel<<<(unsigned)n_u, 128, (size_t)pow2 * 8, (cudaStream_t)stream>>>(vals, idx, P, n_u, K, pow2, out_val, out_idx);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int agcf_score_rows(const float* Uemb, const int32_t* user_rows, int32_t n_u,
                               const float* Iemb, int32_t n_items, int32_t d, float* out, agcf_stream_t stream) {
  if (!Uemb || !Iemb || !out || n_u < 0 || n_items <= 0) return AGCF_EINVAL;
  if (!supported_d(d)) return AGCF_EUNSUPPORTED;
  if (!aligned16(Uemb) || !aligned16(Iemb)) return AGCF_EINVAL;
  if (n_u == 0) return AGCF_OK;
  if (n_u > 65535) return AGCF_EUNSUPPORTED;
  dim3 grid((unsigned)((n_items + 255) / 256), (unsigned)n_u);
  cudaStream_t st = (cudaStream_t)stream;
  const float4* U4 = reinterpret_cast<const float4*>(Uemb);
  const float4* I4 = reinterpret_cast<const float4*>(Iemb);
  switch (d) {
    case 8: score_rows_kernel<8><<<grid, 256, 0, st>>>(U4, user_rows, I4, n_items, out); break;
    case 16: score_rows_kernel<16><<<grid, 256, 0, st>>>(U4, user_rows, I4, n_items, out); break;
    case 32: score_rows_kernel<32><<<grid, 256, 0, st>>>(U4, user_rows, I4, n_items, out); break;
    case 64: score_rows_kernel<64><<<grid, 256, 0, st>>>(U4, user_rows, I4, n_items, out); break;
    case 128: score_rows_kernel<128><<<grid, 256, 0, st>>>(U4, user_rows, I4, n_items, out); break;
    case 256: score_rows_kernel<256><<<grid, 256, 0, st>>>(U4, user_rows, I4, n_items, out); break;
  }
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

extern "C" int agcf_rank_metrics(const int32_t* topk_idx, int32_t K, const int32_t* t_rowptr, const int32_t* t_items,
                                 const int32_t* test_total, int32_t n_u, const int32_t* cutoffs, int32_t nc,
                                 const double* inv_log, double* out, agcf_stream_t stream) {
  if (!topk_idx || !t_rowptr || !test_total || !cutoffs || !inv_log || !out || K <= 0 || n_u < 0 || nc <= 0) return AGCF_EINVAL;
  if (n_u == 0) return AGCF_OK;
  rank_metrics_kernel<<<(unsigned)((n_u + 7) / 8), 256, 0, (cudaStream_t)stream>>>(topk_idx, K, t_rowptr, t_items, test_total,
                                                                                    n_u, cutoffs, nc, inv_log, out);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}
