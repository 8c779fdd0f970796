// contrast.cu -- InfoNCE contrastive loss of SimGCL / XSimGCL, forward and backward, on B200.
//
// Reference: util/loss.py:42-49
//     view1, view2 = F.normalize(view1, dim=1), F.normalize(view2, dim=1)
//     pos = exp(<v1_r, v2_r> / t);  ttl = sum_c exp(<v1_r, v2_c> / t);  loss = mean_r -log(pos_r / ttl_r)
// called on the <= B unique users and <= B unique positive items of a batch
// (recommender/SimGCL.py:212-219, XSimGCL.py:39-44).
//
// The n x n logit matrix is never written to memory: tiles of it are produced in registers, exponentiated and
// reduced on the spot (forward: row sums; backward: P = exp(S)/ttl goes through shared memory straight into the
// second product P.V).  fp32 CUDA cores on purpose: the logits are multiplied by 1/t = 5..10 and exponentiated, a
// TF32 product (10-bit mantissa) would put ~1e-2 relative error on exp(S) -- outside the 1e-4 parity bar -- and the
// whole problem is 2 x 2048^2 x 64 MACs (~10 us), nowhere near a tensor-pipe bound.
// Work is split over (row tile) x (SPLIT slices of the reduced dimension); partial sums are combined in slice order
// by a finishing kernel: deterministic, no floating-point atomics.
#include "common.cuh"

namespace agcf {

constexpr int kNceThreads = 256;           // 16 x 16 thread grid per CTA

template <int D>
struct NceCfg {
  static constexpr int TM = D <= 64 ? 64 : 32;      // vectors per tile (own side and reduced side)
  static constexpr int RS = TM / 16;                // tile rows / cols per thread in the logit product
  // second product P.V: thread (ty, tx) owns KS consecutive columns, KS (tx % CT) ..., and PA of the RS own rows,
  // ty + 16 (PA (tx / CT) + a).  D >= 16: CT = 16 threads cover the D columns, every thread takes all RS rows;
  // D = 8: the 8 columns need only 8 threads, so the two halves of tx split the rows instead
  static constexpr int KS = D >= 16 ? D / 16 : 1;   // embedding columns per thread
  static constexpr int CT = D / KS;                 // threads across the columns (16, or 8 at D = 8)
  static constexpr int PA = RS * CT / 16;           // own rows per thread
  static constexpr int LD = D + 4;                  // padded row stride (floats): 16-byte aligned rows whose float4
  static constexpr int PLD = TM + 4;                // reads by 16 different rows need the minimal 2 wavefronts
  static constexpr size_t smem_fwd = (size_t)(2 * TM * LD) * sizeof(float);
  static constexpr size_t smem_bwd = (size_t)(2 * TM * LD + TM * PLD + 2 * TM) * sizeof(float);
};

// rows [row0, row0 + TM) of a [n, D] table into a padded shared tile (rows >= n are zero); 16 bytes per thread
template <int D>
__device__ __forceinline__ void nce_load_tile(float* __restrict__ sm, const float* __restrict__ g, int row0, int n) {
  using C = NceCfg<D>;
  for (int idx = threadIdx.x; idx < C::TM * (D / 4); idx += kNceThreads) {
    const int r = idx / (D / 4), k4 = idx - r * (D / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row0 + r < n) v = __ldg(reinterpret_cast<const float4*>(g + (size_t)(row0 + r) * D) + k4);
    *reinterpret_cast<float4*>(sm + r * C::LD + 4 * k4) = v;
  }
}

// s[a][b] = <own[ty + 16a], other[tx + 16b]>, k ascending; operands read 4 columns at a time (LDS.128)
template <int D>
__device__ __forceinline__ void nce_logits(const float* __restrict__ own, const float* __restrict__ other, int ty, int tx,
                                           float (&s)[NceCfg<D>::RS][NceCfg<D>::RS]) {
  using C = NceCfg<D>;
#pragma unroll
  for (int a = 0; a < C::RS; ++a)
#pragma unroll
    for (int b = 0; b < C::RS; ++b) s[a][b] = 0.f;
#pragma unroll 4
  for (int k4 = 0; k4 < D / 4; ++k4) {
    float4 av[C::RS], bv[C::RS];
#pragma unroll
    for (int a = 0; a < C::RS; ++a) av[a] = *reinterpret_cast<const float4*>(own + (ty + 16 * a) * C::LD + 4 * k4);
#pragma unroll
    for (int b = 0; b < C::RS; ++b) bv[b] = *reinterpret_cast<const float4*>(other + (tx + 16 * b) * C::LD + 4 * k4);
#pragma unroll
    for (int a = 0; a < C::RS; ++a)
#pragma unroll
      for (int b = 0; b < C::RS; ++b) {
        float t = s[a][b];
        t = fmaf(av[a].x, bv[b].x, t);
        t = fmaf(av[a].y, bv[b].y, t);
        t = fmaf(av[a].z, bv[b].z, t);
        t = fmaf(av[a].w, bv[b].w, t);
        s[a][b] = t;
      }
  }
}

// ---------------------------------------------------------------- normalize
// F.normalize(v, dim=1): v / max(||v||, 1e-12); one warp per row, both views in one launch
// rows: nullable gather list (row r of the view is row rows[r] of the table); n_dev: nullable device row count
__device__ __forceinline__ int nce_rows(int n_max, const int32_t* __restrict__ n_dev) {
  if (n_dev == nullptr) return n_max;
  const int n = __ldg(n_dev);
  return n < n_max ? n : n_max;
}

__global__ void __launch_bounds__(256) nce_normalize_kernel(const float* __restrict__ v1, const float* __restrict__ v2,
                                                            const int32_t* __restrict__ rows, int n_max,
                                                            const int32_t* __restrict__ n_dev, int d,
                                                            float* __restrict__ h1, float* __restrict__ h2,
                                                            float* __restrict__ inv1, float* __restrict__ inv2) {
  const int n = nce_rows(n_max, n_dev);
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= 2 * n) return;
  const bool second = w >= n;
  const int r = second ? w - n : w;
  const size_t src = rows != nullptr ? (size_t)__ldg(rows + r) : (size_t)r;
  const float* v = (second ? v2 : v1) + src * d;
  float* h = (second ? h2 : h1) + (size_t)r * d;
  float ss = 0.f;
  for (int k = lane; k < d; k += 32) { const float x = __ldg(v + k); ss = fmaf(x, x, ss); }
  ss = group_sum<32>(ss);
  const float nrm = fmaxf(sqrtf(ss), 1e-12f);
  for (int k = lane; k < d; k += 32) h[k] = __fdiv_rn(__ldg(v + k), nrm);
  if (lane == 0) (second ? inv2 : inv1)[r] = __fdiv_rn(1.f, nrm);
}

// ------------------------------------------------------------------ forward
// partial[sp][r] = sum over the column tiles of slice sp of exp(<h1_r, h2_c> / t)
template <int D>
__global__ void __launch_bounds__(kNceThreads) nce_rowsum_kernel(const float* __restrict__ h1, const float* __restrict__ h2,
                                                                 int n_max, const int32_t* __restrict__ n_dev, float inv_t,
                                                                 int split, float* __restrict__ partial) {
  using C = NceCfg<D>;
  extern __shared__ __align__(16) float sm[];
  float* own = sm;
  float* other = sm + C::TM * C::LD;
  const int n = nce_rows(n_max, n_dev);
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
  const int row0 = blockIdx.x * C::TM, sp = blockIdx.y;
  if (row0 >= n) return;
  const int n_tiles = (n + C::TM - 1) / C::TM;
  nce_load_tile<D>(own, h1, row0, n);
  float rs[C::RS];
#pragma unroll
  for (int a = 0; a < C::RS; ++a) rs[a] = 0.f;
  for (int ct = sp; ct < n_tiles; ct += split) {
    __syncthreads();                                        // previous tile fully consumed (and `own` visible)
    nce_load_tile<D>(other, h2, ct * C::TM, n);
    __syncthreads();
    float s[C::RS][C::RS];
    nce_logits<D>(own, other, ty, tx, s);
#pragma unroll
    for (int a = 0; a < C::RS; ++a)
#pragma unroll
      for (int b = 0; b < C::RS; ++b)
        if (ct * C::TM + tx + 16 * b < n) rs[a] += expf(s[a][b] * inv_t);
  }
#pragma unroll
  for (int a = 0; a < C::RS; ++a) {
    const float tot = group_sum<16>(rs[a]);                 // the 16 threads that share row ty + 16a
    const int r = row0 + ty + 16 * a;
    if (tx == 0 && r < n) partial[(size_t)sp * n_max + r] = tot;
  }
}

// ttl_r = sum_sp partial (slice order); rowloss_r = -log(exp(<h1_r, h2_r>/t) / ttl_r); one warp per row
__global__ void __launch_bounds__(256) nce_rowloss_kernel(const float* __restrict__ h1, const float* __restrict__ h2, int n_max,
                                                          const int32_t* __restrict__ n_dev, int d, float inv_t, int split,
                                                          const float* __restrict__ partial, float* __restrict__ ttl,
                                                          float* __restrict__ rowloss) {
  const int n = nce_rows(n_max, n_dev);
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= n) return;
  float dot = 0.f;
  for (int k = lane; k < d; k += 32) dot = fmaf(h1[(size_t)r * d + k], h2[(size_t)r * d + k], dot);
  dot = group_sum<32>(dot);
  if (lane == 0) {
    float t = 0.f;
    for (int sp = 0; sp < split; ++sp) t += partial[(size_t)sp * n_max + r];
    ttl[r] = t;
    rowloss[r] = -logf(__fdiv_rn(expf(dot * inv_t), t));
  }
}

// loss = mean_r rowloss_r: one CTA, double accumulation in a fixed order
__global__ void __launch_bounds__(1024) nce_loss_kernel(const float* __restrict__ rowloss, int n_max,
                                                        const int32_t* __restrict__ n_dev, float* __restrict__ loss) {
  __shared__ double red[1024];
  const int n = nce_rows(n_max, n_dev);
  double mine = 0.0;
  for (int r = threadIdx.x; r < n; r += blockDim.x) mine += (double)rowloss[r];
  red[threadIdx.x] = mine;
  __syncthreads();
  for (int o = blockDim.x >> 1; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *loss = n > 0 ? (float)(red[0] / (double)n) : 0.f;
}

// ----------------------------------------------------------------- backward
// SIDE 0: own = h1 rows r, reduced = h2 rows c:  acc_r = sum_c P_rc h2_c,  P_rc = exp(S_rc) / ttl_r
// SIDE 1: own = h2 rows c, reduced = h1 rows r:  acc_c = sum_r P_rc h1_r  (ttl of the REDUCED index)
// partial_acc[sp][own row][:] for the tiles of slice sp.
template <int D, int SIDE>
__global__ void __launch_bounds__(kNceThreads) nce_bwd_kernel(const float* __restrict__ h_own, const float* __restrict__ h_red,
                                                              const float* __restrict__ ttl, int n_max,
                                                              const int32_t* __restrict__ n_dev, float inv_t, int split,
                                                              float* __restrict__ partial_acc) {
  using C = NceCfg<D>;
  extern __shared__ __align__(16) float sm[];
  float* own = sm;
  float* other = own + C::TM * C::LD;
  float* Ps = other + C::TM * C::LD;
  float* ttl_own = Ps + C::TM * C::PLD;
  float* ttl_red = ttl_own + C::TM;
  const int n = nce_rows(n_max, n_dev);
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
  const int row0 = blockIdx.x * C::TM, sp = blockIdx.y;
  if (row0 >= n) return;
  const int n_tiles = (n + C::TM - 1) / C::TM;
  nce_load_tile<D>(own, h_own, row0, n);
  if (threadIdx.x < C::TM) ttl_own[threadIdx.x] = (row0 + (int)threadIdx.x < n) ? ttl[row0 + threadIdx.x] : 1.f;
  const int cx = tx % C::CT, a0 = C::PA * (tx / C::CT);  // columns KS cx .. KS cx + KS - 1, own rows ty + 16 (a0 + a)
  float acc[C::PA][C::KS];
#pragma unroll
  for (int a = 0; a < C::PA; ++a)
#pragma unroll
    for (int b = 0; b < C::KS; ++b) acc[a][b] = 0.f;
  for (int ct = sp; ct < n_tiles; ct += split) {
    __syncthreads();                                        // previous tile (other, Ps) fully consumed
    nce_load_tile<D>(other, h_red, ct * C::TM, n);
    if (threadIdx.x < C::TM) ttl_red[threadIdx.x] = (ct * C::TM + (int)threadIdx.x < n) ? ttl[ct * C::TM + threadIdx.x] : 1.f;
    __syncthreads();
    float s[C::RS][C::RS];
    nce_logits<D>(own, other, ty, tx, s);
#pragma unroll
    for (int a = 0; a < C::RS; ++a)
#pragma unroll
      for (int b = 0; b < C::RS; ++b) {
        const int o = ty + 16 * a, x = tx + 16 * b;
        const float den = SIDE == 0 ? ttl_own[o] : ttl_red[x];
        Ps[o * C::PLD + x] = (ct * C::TM + x < n) ? __fdiv_rn(expf(s[a][b] * inv_t), den) : 0.f;
      }
    __syncthreads();
    // acc[o][k] += sum_x P[o][x] * other[x][k];  thread (ty, tx) owns o = ty + 16 (a0 + a) and the KS consecutive
    // columns k = KS cx + b; P is read 4 x at a time, the operand row KS floats at a time (x ascending in every accumulator)
    for (int x4 = 0; x4 < C::TM; x4 += 4) {
      float4 pv[C::PA];
#pragma unroll
      for (int a = 0; a < C::PA; ++a) pv[a] = *reinterpret_cast<const float4*>(Ps + (ty + 16 * (a0 + a)) * C::PLD + x4);
#pragma unroll
      for (int xx = 0; xx < 4; ++xx) {
        float ov[C::KS];
        const float* orow = other + (x4 + xx) * C::LD + C::KS * cx;
        if constexpr (C::KS % 4 == 0) {
#pragma unroll
          for (int q = 0; q < C::KS / 4; ++q) {
            const float4 t4 = *reinterpret_cast<const float4*>(orow + 4 * q);
            ov[4 * q] = t4.x; ov[4 * q + 1] = t4.y; ov[4 * q + 2] = t4.z; ov[4 * q + 3] = t4.w;
          }
        } else if constexpr (C::KS == 2) {
          const float2 t2 = *reinterpret_cast<const float2*>(orow);
          ov[0] = t2.x; ov[1] = t2.y;
        } else {
          ov[0] = orow[0];
        }
#pragma unroll
        for (int a = 0; a < C::PA; ++a) {
          const float pa = xx == 0 ? pv[a].x : (xx == 1 ? pv[a].y : (xx == 2 ? pv[a].z : pv[a].w));
#pragma unroll
          for (int b = 0; b < C::KS; ++b) acc[a][b] = fmaf(pa, ov[b], acc[a][b]);
        }
      }
    }
  }
#pragma unroll
  for (int a = 0; a < C::PA; ++a) {
    const int r = row0 + ty + 16 * (a0 + a);
    if (r >= n) continue;
    float* dst = partial_acc + ((size_t)sp * n_max + r) * D + C::KS * cx;
#pragma unroll
    for (int b = 0; b < C::KS; ++b) dst[b] = acc[a][b];
  }
}

// d_hat = coef * (sum_sp partial_acc - partner_hat), coef = g * scale / (n t);  through F.normalize:
// d_v = (d_hat - h <h, d_hat>) / max(||v||, eps).  One warp per row.  Output: grad[r] (dense [n, d]) or, with a
// gather list, row rows[r] of a TABLE (the ids are unique, so rows never collide); accumulate != 0 adds.
__global__ void __launch_bounds__(256) nce_bwd_finish_kernel(const float* __restrict__ partial_acc, int split,
                                                             const float* __restrict__ h, const float* __restrict__ partner,
                                                             const float* __restrict__ inv_norm, const float* __restrict__ g_loss,
                                                             float scale, int n_max, const int32_t* __restrict__ n_dev, int d,
                                                             const int32_t* __restrict__ rows, int accumulate,
                                                             float* __restrict__ grad) {
  const int n = nce_rows(n_max, n_dev);
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= n) return;
  const float coef = (g_loss != nullptr ? __ldg(g_loss) : 1.f) * scale / (float)n;
  float dh[8];                                               // d <= 256: up to 8 columns per lane
  float dot = 0.f;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const int k = lane + 32 * q;
    dh[q] = 0.f;
    if (k < d) {
      float a = 0.f;
      for (int sp = 0; sp < split; ++sp) a += partial_acc[((size_t)sp * n_max + r) * d + k];
      dh[q] = coef * (a - partner[(size_t)r * d + k]);
      dot = fmaf(h[(size_t)r * d + k], dh[q], dot);
    }
  }
  dot = group_sum<32>(dot);
  const float inv = inv_norm[r];
  float* out = grad + (rows != nullptr ? (size_t)__ldg(rows + r) : (size_t)r) * d;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const int k = lane + 32 * q;
    if (k < d) {
      const float gv = (dh[q] - h[(size_t)r * d + k] * dot) * inv;
      out[k] = accumulate ? out[k] + gv : gv;
    }
  }
}

// workspace layout (floats): h1 [n,d] | h2 [n,d] | inv1 [n] | inv2 [n] | ttl [n] | rowloss [n] | partial [split,n] | acc [split,n,d]
struct NceWs {
  float *h1, *h2, *inv1, *inv2, *ttl, *rowloss, *partial, *acc;
  int split;
};

static int nce_tile(int d) { return d <= 64 ? 64 : 32; }

static int nce_split(int n, int d) {
  const int nt = (n + nce_tile(d) - 1) / nce_tile(d);
  int s = (2 * kSMs + nt - 1) / nt;                          // ~2 CTAs per SM per launch; the user and item sides run concurrently
  s = s < 1 ? 1 : s;
  s = s > nt ? nt : s;
  return s > 16 ? 16 : s;
}

static int64_t nce_ws_floats(int n, int d) {
  const int64_t s = nce_split(n, d);
  return 2ll * n * d + 4ll * (n + 4) + s * n + s * (int64_t)n * d + 16;
}

static NceWs nce_carve(void* ws, int n, int d) {
  NceWs w;
  float* p = reinterpret_cast<float*>(ws);
  w.split = nce_split(n, d);
  w.h1 = p; p += (size_t)n * d;
  w.h2 = p; p += (size_t)n * d;
  const size_t n4 = ((size_t)n + 3) & ~(size_t)3;               // keeps every table 16-byte aligned
  w.inv1 = p; p += n4;
  w.inv2 = p; p += n4;
  w.ttl = p; p += n4;
  w.rowloss = p; p += n4;
  w.partial = p; p += ((size_t)w.split * n + 3) & ~(size_t)3;
  w.acc = p;
  return w;
}

struct NceGrad {             // where one view's gradient goes
  float* out;                // dense [n, d], or a table when rows != nullptr; nullptr = not wanted
  const int32_t* rows;
  int accumulate;
};

template <int D>
static int nce_forward_d(const float* v1, const float* v2, const int32_t* rows, int n, const int32_t* n_dev, float inv_t,
                         float* loss, const NceWs& w, cudaStream_t st) {
  using C = NceCfg<D>;
  static thread_local bool attr = false;
  if (!attr) {
    AGCF_CUDA_OK(cudaFuncSetAttribute(nce_rowsum_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::smem_fwd));
    attr = true;
  }
  nce_normalize_kernel<<<(unsigned)((2ll * n * 32 + 255) / 256), 256, 0, st>>>(v1, v2, rows, n, n_dev, D, w.h1, w.h2, w.inv1,
                                                                              w.inv2);
  AGCF_LAUNCH_OK();
  const dim3 grid((n + C::TM - 1) / C::TM, w.split);
  nce_rowsum_kernel<D><<<grid, kNceThreads, C::smem_fwd, st>>>(w.h1, w.h2, n, n_dev, inv_t, w.split, w.partial);
  AGCF_LAUNCH_OK();
  nce_rowloss_kernel<<<(unsigned)(((long long)n * 32 + 255) / 256), 256, 0, st>>>(w.h1, w.h2, n, n_dev, D, inv_t, w.split,
                                                                                 w.partial, w.ttl, w.rowloss);
  AGCF_LAUNCH_OK();
  nce_loss_kernel<<<1, 1024, 0, st>>>(w.rowloss, n, n_dev, loss);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

template <int D>
static int nce_backward_d(int n, const int32_t* n_dev, float inv_t, const float* g_loss, float scale, const NceWs& w,
                          const NceGrad& g1, const NceGrad& g2, cudaStream_t st) {
  using C = NceCfg<D>;
  static thread_local bool attr = false;
  if (!attr) {
    AGCF_CUDA_OK(cudaFuncSetAttribute(nce_bwd_kernel<D, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::smem_bwd));
    AGCF_CUDA_OK(cudaFuncSetAttribute(nce_bwd_kernel<D, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::smem_bwd));
    attr = true;
  }
  const dim3 grid((n + C::TM - 1) / C::TM, w.split);
  const float s = scale * inv_t;                              // the finishing kernel divides by the (device) n
  const unsigned fin_blocks = (unsigned)(((long long)n * 32 + 255) / 256);
  if (g1.out != nullptr) {
    nce_bwd_kernel<D, 0><<<grid, kNceThreads, C::smem_bwd, st>>>(w.h1, w.h2, w.ttl, n, n_dev, inv_t, w.split, w.acc);
    AGCF_LAUNCH_OK();
    nce_bwd_finish_kernel<<<fin_blocks, 256, 0, st>>>(w.acc, w.split, w.h1, w.h2, w.inv1, g_loss, s, n, n_dev, D, g1.rows,
                                                      g1.accumulate, g1.out);
    AGCF_LAUNCH_OK();
  }
  if (g2.out != nullptr) {
    nce_bwd_kernel<D, 1><<<grid, kNceThreads, C::smem_bwd, st>>>(w.h2, w.h1, w.ttl, n, n_dev, inv_t, w.split, w.acc);
    AGCF_LAUNCH_OK();
    nce_bwd_finish_kernel<<<fin_blocks, 256, 0, st>>>(w.acc, w.split, w.h2, w.h1, w.inv2, g_loss, s, n, n_dev, D, g2.rows,
                                                      g2.accumulate, g2.out);
    AGCF_LAUNCH_OK();
  }
  return AGCF_OK;
}

}  // namespace agcf

using namespace agcf;

extern "C" int64_t agcf_infonce_ws_bytes(int32_t n, int32_t d) {
  if (n <= 0 || !supported_d(d)) return n == 0 ? 64 : AGCF_EUNSUPPORTED;
  return nce_ws_floats(n, d) * (int64_t)sizeof(float);
}

extern "C" int agcf_infonce_forward(const float* view1, const float* view2, const int32_t* rows, int32_t n,
                                    const int32_t* n_dev, int32_t d, float temperature, float* loss, void* ws,
                                    int64_t ws_bytes, agcf_stream_t stream) {
  if (!view1 || !view2 || !loss || !ws || n <= 0 || !(temperature > 0.f)) return AGCF_EINVAL;
  if (!supported_d(d)) return AGCF_EUNSUPPORTED;
  if (ws_bytes < agcf_infonce_ws_bytes(n, d)) return AGCF_EWORKSPACE;
  const NceWs w = nce_carve(ws, n, d);
  const float inv_t = 1.f / temperature;
  cudaStream_t st = (cudaStream_t)stream;
  switch (d) {
    case 8: return nce_forward_d<8>(view1, view2, rows, n, n_dev, inv_t, loss, w, st);
    case 16: return nce_forward_d<16>(view1, view2, rows, n, n_dev, inv_t, loss, w, st);
    case 32: return nce_forward_d<32>(view1, view2, rows, n, n_dev, inv_t, loss, w, st);
    case 64: return nce_forward_d<64>(view1, view2, rows, n, n_dev, inv_t, loss, w, st);
    case 128: return nce_forward_d<128>(view1, view2, rows, n, n_dev, inv_t, loss, w, st);
    case 256: return nce_forward_d<256>(view1, view2, rows, n, n_dev, inv_t, loss, w, st);
  }
  return AGCF_EUNSUPPORTED;
}

extern "C" int agcf_infonce_backward(int32_t n, const int32_t* n_dev, int32_t d, float temperature,
                                     const float* grad_loss, float scale, void* ws, int64_t ws_bytes,
                                     float* grad_view1, const int32_t* rows1, int32_t accumulate1,
                                     float* grad_view2, const int32_t* rows2, int32_t accumulate2,
                                     agcf_stream_t stream) {
  if (!ws || n <= 0 || !(temperature > 0.f) || (!grad_view1 && !grad_view2)) return AGCF_EINVAL;
  if (!supported_d(d)) return AGCF_EUNSUPPORTED;
  if (ws_bytes < agcf_infonce_ws_bytes(n, d)) return AGCF_EWORKSPACE;
  const NceWs w = nce_carve(ws, n, d);
  const float inv_t = 1.f / temperature;
  const NceGrad g1 = {grad_view1, rows1, accumulate1}, g2 = {grad_view2, rows2, accumulate2};
  cudaStream_t st = (cudaStream_t)stream;
  switch (d) {
    case 8: return nce_backward_d<8>(n, n_dev, inv_t, grad_loss, scale, w, g1, g2, st);
    case 16: return nce_backward_d<16>(n, n_dev, inv_t, grad_loss, scale, w, g1, g2, st);
    case 32: return nce_backward_d<32>(n, n_dev, inv_t, grad_loss, scale, w, g1, g2, st);
    case 64: return nce_backward_d<64>(n, n_dev, inv_t, grad_loss, scale, w, g1, g2, st);
    case 128: return nce_backward_d<128>(n, n_dev, inv_t, grad_loss, scale, w, g1, g2, st);
    case 256: return nce_backward_d<256>(n, n_dev, inv_t, grad_loss, scale, w, g1, g2, st);
  }
  return AGCF_EUNSUPPORTED;
}
