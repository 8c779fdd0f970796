// score_tc.cu -- stage 1 of agcf_score_topk on the 5th-generation tensor cores.
//
//   gmax[u, g] = max over the 32 items of group g of  masked( <U[u,:], I[i,:]> )
//
// The one dense contraction of the hot path (recommender/LightGCN.py:86-90,148-156:
// one GEMV per user in the reference) as a persistent, warp-specialised tcgen05 GEMM:
//   * operands are the fp32 embedding tables themselves, consumed as TF32
//     (kind::tf32 reads the upper 19 bits of each fp32 word): no conversion pass;
//   * TMA (cp.async.bulk.tensor.2d, 128-byte swizzle; 32- / 64-byte at d = 8 / 16, whose rows are
//     narrower than one 128-byte atom row) stages a 128-user A tile once per work unit and streams
//     256-item B tiles through a 2-stage ring;
//   * one elected thread issues d/8 x tcgen05.mma (M128 x N256 x K8) per tile into one of
//     two 256-column TMEM accumulators, tcgen05.commit signals the mbarriers;
//   * four epilogue warps read the accumulator with tcgen05.ld (32 lanes x 32 columns =
//     one user x one 32-item group per thread), apply the train-item mask bits, reduce
//     to the group maximum and store ONE float per (user, group): the 128 x 256 scores
//     never leave the SM.  MMA of tile t+1 overlaps the epilogue of tile t.
// The result is approximate (TF32); agcf_score_topk's stage 2 selects candidate groups
// with a rigorous margin and re-scores them in exact fp32, so the final top-K does not
// depend on this kernel's rounding (DESIGN.md "top-K exactness").
#include "common.cuh"
#include <cuda.h>
#include <float.h>

namespace agcf {
namespace tc {

constexpr int kTileM = 128;            // users per tile (UMMA M)
constexpr int kUmmaK = 8;              // K per tcgen05.mma for tf32 (32 bytes)
constexpr int kStages = 2;
#ifndef AGCF_TC_EPI_WG
#define AGCF_TC_EPI_WG 4
#endif
constexpr int kEpiWG = AGCF_TC_EPI_WG;  // epilogue warpgroups: each covers all 128 rows and 1/kEpiWG of a tile's columns
constexpr int kEpiWarps = 4 * kEpiWG;
constexpr int kThreads = 64 + 32 * kEpiWarps;   // warp 0: TMA, warp 1: MMA + TMEM alloc, then the epilogue warps
constexpr uint32_t kTmemCols = 512;    // two fp32 accumulators of kTileN columns (all of TMEM: 1 CTA / SM)
constexpr float kMaskedScore = -1.0e9f;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// bounded wait: a protocol bug traps (context error) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  for (uint32_t spins = 0;; ++spins) {
    uint32_t done;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) return;
    if (spins > (1u << 24)) __trap();
  }
}

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// K-major, swizzled shared-memory matrix descriptor (cute::UMMA::SmemDescriptor) for atom rows of
// ROW_BYTES = 128, 64 or 32: start address >> 4, LBO = 1 (ignored for swizzled K-major),
// SBO = 8 rows x ROW_BYTES, version 1 (Blackwell), layout type 2 / 4 / 6 = SWIZZLE_128B / 64B / 32B.
template <int ROW_BYTES>
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  static_assert(ROW_BYTES == 128 || ROW_BYTES == 64 || ROW_BYTES == 32, "swizzle width");
  constexpr uint64_t layout = ROW_BYTES == 128 ? 2 : (ROW_BYTES == 64 ? 4 : 6);
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)((8 * ROW_BYTES) >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= layout << 61;
  return d;
}

// cute::UMMA::InstrDescriptor for kind::tf32: D = F32, A = B = TF32, both K-major
constexpr uint32_t make_idesc(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}
// the loads of a tile are issued back to back and waited for ONCE: the TMEM read path (64 B/clk per SM) is what bounds
// this kernel, a wait after every load left it idle for a load latency per 32 columns
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

struct alignas(8) Barriers {
  uint64_t a_full, a_empty;
  uint64_t b_full[kStages], b_empty[kStages];
  uint64_t acc_full[2], acc_empty[2];
  uint32_t tmem_base;
};

template <int D>
struct Smem {
  static constexpr int kTileN = D <= 64 ? 256 : 128;   // items per tile (UMMA N); smaller for d = 128 (smem)
  static constexpr int kKBlock = D < 32 ? D : 32;       // fp32 elements per swizzle atom row (a row of 128, 64 or 32 B)
  static constexpr int kRowBytes = kKBlock * 4;
  static constexpr int kKBlocks = D / kKBlock;
  static constexpr int kABytes = kKBlocks * kTileM * kRowBytes;
  static constexpr int kBBytes = kKBlocks * kTileN * kRowBytes;
  static constexpr int kTotal = kABytes + kStages * kBBytes + 1024 /*alignment slack*/ + 256 /*barriers*/;
};

// work unit = (user tile, chunk of item tiles); units are dealt round-robin to the persistent CTAs
template <int D>
__global__ void __launch_bounds__(kThreads, 1)
group_max_tc_kernel(const __grid_constant__ CUtensorMap tmap_u, const __grid_constant__ CUtensorMap tmap_i,
                    int n_u, int n_items, int n_groups, int pitch, int n_item_tiles, int tiles_per_chunk, int n_chunks, int n_units,
                    const uint32_t* __restrict__ bits, float* __restrict__ gmax) {
  using S = Smem<D>;
  constexpr int kTileN = S::kTileN;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = smem + S::kABytes;
  Barriers* bars = reinterpret_cast<Barriers*>(smem + S::kABytes + kStages * S::kBBytes);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    mbar_init(&bars->a_full, 1);
    mbar_init(&bars->a_empty, 1);
    for (int s = 0; s < kStages; ++s) { mbar_init(&bars->b_full[s], 1); mbar_init(&bars->b_empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&bars->acc_full[a], 1); mbar_init(&bars->acc_empty[a], kEpiWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_u)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_i)) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)), "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (lane == 0) {
      uint32_t stage = 0, b_phase = 0, unit_iter = 0;
      for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++unit_iter) {
        const int ut = unit / n_chunks, ch = unit - ut * n_chunks;
        const int t0 = ch * tiles_per_chunk;
        const int t1 = min(n_item_tiles, t0 + tiles_per_chunk);
        mbar_wait(&bars->a_empty, (unit_iter & 1) ^ 1);            // MMA finished with the previous A tile
        mbar_arrive_expect_tx(&bars->a_full, S::kABytes);
        for (int kb = 0; kb < S::kKBlocks; ++kb)
          tma_load_2d(sA + kb * kTileM * S::kRowBytes, &tmap_u, &bars->a_full, kb * S::kKBlock, ut * kTileM);
        for (int t = t0; t < t1; ++t) {
          mbar_wait(&bars->b_empty[stage], b_phase ^ 1);
          mbar_arrive_expect_tx(&bars->b_full[stage], S::kBBytes);
          for (int kb = 0; kb < S::kKBlocks; ++kb)
            tma_load_2d(sB + stage * S::kBBytes + kb * kTileN * S::kRowBytes, &tmap_i, &bars->b_full[stage], kb * S::kKBlock,
                        t * kTileN);
          if (++stage == kStages) { stage = 0; b_phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ==================================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(kTileM, kTileN);
      uint32_t stage = 0, b_phase = 0, acc = 0, acc_phase = 0, unit_iter = 0;
      for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++unit_iter) {
        const int ut = unit / n_chunks, ch = unit - ut * n_chunks;
        const int t0 = ch * tiles_per_chunk;
        const int t1 = min(n_item_tiles, t0 + tiles_per_chunk);
        mbar_wait(&bars->a_full, unit_iter & 1);
        for (int t = t0; t < t1; ++t) {
          mbar_wait(&bars->acc_empty[acc], acc_phase ^ 1);         // epilogue drained this accumulator
          mbar_wait(&bars->b_full[stage], b_phase);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t d_tmem = tmem_base + acc * kTileN;
#pragma unroll
          for (int kb = 0; kb < S::kKBlocks; ++kb) {
            const uint64_t adesc = make_smem_desc<S::kRowBytes>(smem_u32(sA + kb * kTileM * S::kRowBytes));
            const uint64_t bdesc = make_smem_desc<S::kRowBytes>(smem_u32(sB + stage * S::kBBytes + kb * kTileN * S::kRowBytes));
#pragma unroll
            for (int k = 0; k < S::kKBlock / kUmmaK; ++k)         // +32 bytes along K inside the swizzle atom
              umma_tf32(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0);
          }
          umma_commit(&bars->b_empty[stage]);                      // smem stage reusable once these MMAs retire
          umma_commit(&bars->acc_full[acc]);                       // accumulator ready for the epilogue
          if (++stage == kStages) { stage = 0; b_phase ^= 1; }
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        umma_commit(&bars->a_empty);                               // A tile free after the unit's last MMA
      }
    }
  } else {
    // ================================ epilogue (kEpiWarps warps) ===================
    // The epilogue (TMEM -> registers, mask, max over 32 columns, one float per group) takes longer than the 8 MMAs of
    // a K = 64 tile: with 4 warps the tensor pipe idled 74 % of the time (ncu: 26 % active, 35 % with 8 warps).  kEpiWG
    // warpgroups split the tile's columns; a warp may only read the TMEM lanes 32 (id % 4) .. +32, so every group of
    // four consecutive warps covers all 128 rows.
    const int quarter = warp & 3;                                  // TMEM lanes [32q, 32q+32) belong to warp (id % 4) == q
    const int half = (warp - 2) >> 2;                              // which half of the tile's groups this warpgroup takes
    const int row_in_tile = quarter * 32 + lane;
    uint32_t acc = 0, acc_phase = 0;
    for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
      const int ut = unit / n_chunks, ch = unit - ut * n_chunks;
      const int t0 = ch * tiles_per_chunk;
      const int t1 = min(n_item_tiles, t0 + tiles_per_chunk);
      const int r = ut * kTileM + row_in_tile;
      const bool row_ok = r < n_u;
      // rows of bits / gmax are `pitch` words apart (multiple of 8 = 32 B), a tile covers GPT consecutive
      // groups, a thread GH of them: one aligned 8/16-byte vector per thread per tile for the mask words and the maxima
      constexpr int GPT = kTileN / 32;                               // groups per tile: 8 (or 4 for d = 128)
      constexpr int GH = GPT / kEpiWG;                               // groups per thread and tile
      static_assert(GH == 1 || GH == 2 || GH == 4, "epilogue split");
      const uint32_t* brow = bits + (size_t)(row_ok ? r : 0) * pitch + half * GH;
      float* grow = gmax + (size_t)(row_ok ? r : 0) * pitch + half * GH;
      uint32_t w[GH], wn[GH];
      auto load_words = [&](int t, uint32_t (&dst)[GH]) {
        if constexpr (GH == 4) {
          const uint4 x = row_ok ? __ldg(reinterpret_cast<const uint4*>(brow + t * GPT)) : make_uint4(0u, 0u, 0u, 0u);
          dst[0] = x.x; dst[1] = x.y; dst[2] = x.z; dst[3] = x.w;
        } else if constexpr (GH == 2) {
          const uint2 x = row_ok ? __ldg(reinterpret_cast<const uint2*>(brow + t * GPT)) : make_uint2(0u, 0u);
          dst[0] = x.x; dst[1] = x.y;
        } else {
          dst[0] = row_ok ? __ldg(brow + t * GPT) : 0u;
        }
      };
      load_words(t0, w);
      for (int t = t0; t < t1; ++t) {
        if (t + 1 < t1) load_words(t + 1, wn);                       // mask words of the next tile: in flight during this one
        mbar_wait(&bars->acc_full[acc], acc_phase);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * kTileN + half * GH * 32;
        float mx[GH];
        uint32_t v[GH][32];
#pragma unroll
        for (int q = 0; q < GH; ++q) tmem_ld32(taddr + q * 32, v[q]);
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < GH; ++q) {
          const int g = t * GPT + half * GH + q;
          const int valid = n_items - g * 32;                        // < 32 only in the table's last group; <= 0 past it
          float m = -FLT_MAX;
          if (w[q] == 0u && valid >= 32) {
#pragma unroll
            for (int c = 0; c < 32; ++c) m = fmaxf(m, __uint_as_float(v[q][c]));
          } else {
#pragma unroll
            for (int c = 0; c < 32; ++c) {
              float sc = __uint_as_float(v[q][c]);
              if ((w[q] >> c) & 1u) sc = kMaskedScore;
              if (c >= valid) sc = -FLT_MAX;
              m = fmaxf(m, sc);
            }
          }
          mx[q] = m;
        }
        if (row_ok) {
          if constexpr (GH == 4) *reinterpret_cast<float4*>(grow + t * GPT) = make_float4(mx[0], mx[1], mx[2], mx[3]);
          else if constexpr (GH == 2) *reinterpret_cast<float2*>(grow + t * GPT) = make_float2(mx[0], mx[1]);
          else grow[t * GPT] = mx[0];
        }
#pragma unroll
        for (int q = 0; q < GH; ++q) w[q] = wn[q];
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->acc_empty[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// rows user_rows[r] of Uemb -> contiguous [n_u, d] (TMA needs a dense 2-D tensor)
__global__ void __launch_bounds__(256) gather_rows_kernel(const float4* __restrict__ src, const int32_t* __restrict__ rows,
                                                          long long n4, int v4, float4* __restrict__ dst) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n4; k += stride) {
    const long long r = k / v4;
    const int c = (int)(k - r * v4);
    dst[k] = __ldg(src + (size_t)rows[r] * v4 + c);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// [rows, d] fp32 row-major; box = box_cols floats (one swizzle atom row of 4 box_cols bytes) x box_rows
static int make_tmap(CUtensorMap* m, const float* base, int rows, int d, int box_cols, int box_rows) {
  EncodeTiledFn enc = get_encode_fn();
  if (enc == nullptr) return AGCF_ECUDA;
  cuuint64_t dims[2] = {(cuuint64_t)d, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)d * sizeof(float)};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  const CUtensorMapSwizzle swz = box_cols == 32 ? CU_TENSOR_MAP_SWIZZLE_128B
                                                : (box_cols == 16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? AGCF_OK : AGCF_ECUDA;
}

template <int D>
static int launch(const float* U, int n_u, const float* I, int n_items, const uint32_t* bits, int n_groups, int pitch,
                  float* gmax, cudaStream_t st) {
  CUtensorMap tu, ti;
  int rc = make_tmap(&tu, U, n_u, D, Smem<D>::kKBlock, kTileM);
  if (rc != AGCF_OK) return rc;
  constexpr int kTileN = Smem<D>::kTileN;
  rc = make_tmap(&ti, I, n_items, D, Smem<D>::kKBlock, kTileN);
  if (rc != AGCF_OK) return rc;
  const int n_user_tiles = (n_u + kTileM - 1) / kTileM;
  const int n_item_tiles = (n_items + kTileN - 1) / kTileN;
  // enough units for ~10 rounds over the SMs so the tail wave stays short
  int n_chunks = (10 * kSMs + n_user_tiles - 1) / n_user_tiles;
  if (n_chunks > n_item_tiles) n_chunks = n_item_tiles;
  if (n_chunks < 1) n_chunks = 1;
  const int tiles_per_chunk = (n_item_tiles + n_chunks - 1) / n_chunks;
  n_chunks = (n_item_tiles + tiles_per_chunk - 1) / tiles_per_chunk;
  const int n_units = n_user_tiles * n_chunks;
  const int grid = n_units < kSMs ? n_units : kSMs;
  AGCF_CUDA_OK(cudaFuncSetAttribute(group_max_tc_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, Smem<D>::kTotal));
  group_max_tc_kernel<D><<<grid, kThreads, Smem<D>::kTotal, st>>>(tu, ti, n_u, n_items, n_groups, pitch, n_item_tiles, tiles_per_chunk,
                                                                  n_chunks, n_units, bits, gmax);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

}  // namespace tc

// entry point used by agcf_score_topk (score.cu); `u_dense` is workspace for the gathered user rows
int launch_group_max_tc(const float* Uemb, const int32_t* user_rows, int n_u, const float* Iemb, int n_items, int d,
                        const uint32_t* bits, int n_groups, int pitch, float* gmax, float* u_dense, cudaStream_t st) {
  const float* U = Uemb;
  if (user_rows != nullptr) {
    const long long n4 = (long long)n_u * (d / 4);
    long long blocks = (n4 + 255) / 256;
    if (blocks > kSMs * 8) blocks = kSMs * 8;
    tc::gather_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(Uemb), user_rows, n4, d / 4,
                                                             reinterpret_cast<float4*>(u_dense));
    AGCF_LAUNCH_OK();
    U = u_dense;
  }
  switch (d) {
    case 8: return tc::launch<8>(U, n_u, Iemb, n_items, bits, n_groups, pitch, gmax, st);
    case 16: return tc::launch<16>(U, n_u, Iemb, n_items, bits, n_groups, pitch, gmax, st);
    case 32: return tc::launch<32>(U, n_u, Iemb, n_items, bits, n_groups, pitch, gmax, st);
    case 64: return tc::launch<64>(U, n_u, Iemb, n_items, bits, n_groups, pitch, gmax, st);
    case 128: return tc::launch<128>(U, n_u, Iemb, n_items, bits, n_groups, pitch, gmax, st);
  }
  return AGCF_EUNSUPPORTED;
}

}  // namespace agcf
