// ngcf.cu -- the dense half of an NGCF layer, forward and backward, fused around the SpMM.
//
// Reference: recommender/NGCF.py:197-212 -- per layer
//     T = E W1 ;  E' = leaky_relu( A T + T + ((A E) * E) W2 , 0.01 )
// (torch.mm x 2, torch.sparse.mm x 2, four element-wise kernels, and autograd's mirror of all of it).
// A is linear, so A (E W1) = (A E) W1: with P = A E the layer is
//     Z = (P + E) W1 + (P * E) W2 = [P + E | P * E] [W1 ; W2] ,   E' = leaky_relu(Z)
// -- ONE propagation per layer instead of two (agcf_spmm_csr_f32 computes P), and one [N, 2d] x [2d, d] product whose
// left operand is formed on the fly from the rows of P and E while they are staged in shared memory.  The product is
// N x 2d x d (1.16 GFLOP per layer at the Gowalla shape, d = 64) next to a 44 us SpMM: fp32 FMA on CUDA cores with a
// register-blocked 64-row tile, exact fp32 like the reference's torch.mm (a TF32 tensor-core product would put 1e-3 on
// every activation; a 3 x TF32 split is not worth a kernel this small).
//
//   agcf_ngcf_dense_forward    E' (and the running layer mean)               from P, E, W = [W1 ; W2]
//   agcf_ngcf_dense_backward   dP, dE_direct and per-CTA partials of dW       from dE', E' (sign of Z), P, E, W^T
//   agcf_ngcf_reduce_wgrad     dW = sum of the partials in CTA order (deterministic)
// d in {8, 16, 32, 64, 128, 256}: a 64-row tile on a 16 x 16 thread grid at 32 and 64, a row per thread at 8 and 16, and
// at 128 and 256 a 128 x 128 tile per product, with dW split over row slices (one partial per slice).
//
// Backward:  dZ = dE' * (E' > 0 ? 1 : 0.01)      (leaky_relu keeps the sign, so E' tells which branch Z took)
//            [dA | dB] = dZ [W1 ; W2]^T ;  dP = dA + dB * E ;  dE_direct = dA + dB * P ;  dW = [P + E | P * E]^T dZ
//            dE = A dP + dE_direct (the caller's next agcf_spmm_csr_f32, A = A^T)
#include "common.cuh"

namespace agcf {
namespace ngcf {

constexpr int kTM = 64;        // rows per tile
constexpr int kKC = 64;        // k chunk staged in shared memory
constexpr float kSlope = 0.01f;

// Where a row-partitioned launch (one rank's rows of the multi-GPU layout) also stores an output: the other ranks'
// copies (n device pointers over NVLink) or, when mc is set, one NVSwitch multicast address that reaches every copy.
// Both are offset to the launch's first row like the local pointer, so a row has the same index in all of them.
// Kernels take it under the compile-time flag PEERS: with PEERS false the argument is never read.
struct RowPeers {
  int n;
  float* p[AGCF_MAX_PEERS];
  float* mc;
};

// v[0 .. N) -> element `at` of every peer copy (at is a multiple of min(N, 4)); visible there after a barrier
template <int N>
__device__ __forceinline__ void store_peers(const RowPeers& pr, size_t at, const float (&v)[N]) {
  if (pr.mc != nullptr) {
    if constexpr (N % 4 == 0) {
#pragma unroll
      for (int i = 0; i < N; i += 4)
        st_multicast_f4(reinterpret_cast<float4*>(pr.mc + at + i), make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]));
    } else if constexpr (N == 2) {
      asm volatile("multimem.st.weak.global.v2.f32 [%0], {%1,%2};" :: "l"(pr.mc + at), "f"(v[0]), "f"(v[1]) : "memory");
    } else {
#pragma unroll
      for (int i = 0; i < N; ++i)
        asm volatile("multimem.st.weak.global.f32 [%0], %1;" :: "l"(pr.mc + at + i), "f"(v[i]) : "memory");
    }
    return;
  }
#pragma unroll
  for (int q = 0; q < AGCF_MAX_PEERS; ++q) {        // static indices: the pointer array stays in the parameter bank
    if (q >= pr.n) break;
    if constexpr (N % 4 == 0) {
#pragma unroll
      for (int i = 0; i < N; i += 4)
        *reinterpret_cast<float4*>(pr.p[q] + at + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
    } else if constexpr (N == 2) {
      *reinterpret_cast<float2*>(pr.p[q] + at) = make_float2(v[0], v[1]);
    } else {
#pragma unroll
      for (int i = 0; i < N; ++i) pr.p[q][at + i] = v[i];
    }
  }
}

template <int CN>
__device__ __forceinline__ void load_cols(const float* __restrict__ src, float (&w)[CN]) {
  if constexpr (CN == 2) {
    const float2 v = *reinterpret_cast<const float2*>(src);
    w[0] = v.x; w[1] = v.y;
  } else {
#pragma unroll
    for (int q = 0; q < CN / 4; ++q) {
      const float4 v = *reinterpret_cast<const float4*>(src + 4 * q);
      w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w;
    }
  }
}

// acc[RM][CN] += As[ty*RM + r][0 .. KC) . Bs[0 .. KC)[tx*CN + c]      (As rows padded to KC + 4 floats)
template <int RM, int CN>
__device__ __forceinline__ void tile_mac(const float (*As)[kKC + 4], const float* __restrict__ Bs, int ldb, int ty, int tx,
                                         float (&acc)[RM][CN]) {
#pragma unroll 4
  for (int k = 0; k < kKC; k += 4) {
    float4 a[RM];
#pragma unroll
    for (int r = 0; r < RM; ++r) a[r] = *reinterpret_cast<const float4*>(&As[ty * RM + r][k]);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      float w[CN];
      load_cols<CN>(Bs + (size_t)(k + kk) * ldb + tx * CN, w);
#pragma unroll
      for (int r = 0; r < RM; ++r) {
        const float av = kk == 0 ? a[r].x : (kk == 1 ? a[r].y : (kk == 2 ? a[r].z : a[r].w));
#pragma unroll
        for (int c = 0; c < CN; ++c) acc[r][c] = fmaf(av, w[c], acc[r][c]);
      }
    }
  }
}

// ---------------------------------------------------------------------------- forward
template <int D, bool PEERS>
__global__ void __launch_bounds__(256) dense_fwd_kernel(const float* __restrict__ P, const float* __restrict__ E,
                                                        const float* __restrict__ W, float* __restrict__ Enext,
                                                        const float* __restrict__ acc_in, float* __restrict__ acc_out,
                                                        float acc_div, int N, RowPeers peer_next, RowPeers peer_acc) {
  constexpr int CN = D / 16;                       // output columns per thread
  __shared__ __align__(16) float As[kTM][kKC + 4];
  __shared__ __align__(16) float Ws[kKC * D];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int row0 = blockIdx.x * kTM;
  float acc[4][CN];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < CN; ++c) acc[r][c] = 0.f;
  for (int kc = 0; kc < 2 * D; kc += kKC) {
    for (int f = tid; f < kTM * (kKC / 4); f += 256) {
      const int r = f / (kKC / 4), k4 = f - r * (kKC / 4);
      const int kk = kc + 4 * k4;
      const int part = kk / D, col = kk - part * D;                  // 4 consecutive k stay inside one part (D % 4 == 0)
      const int row = row0 + r;
      float4 p = make_float4(0.f, 0.f, 0.f, 0.f), e = p;
      if (row < N) {
        p = __ldg(reinterpret_cast<const float4*>(P + (size_t)row * D + col));
        e = __ldg(reinterpret_cast<const float4*>(E + (size_t)row * D + col));
      }
      const float4 v = part == 0 ? make_float4(p.x + e.x, p.y + e.y, p.z + e.z, p.w + e.w)
                                 : make_float4(p.x * e.x, p.y * e.y, p.z * e.z, p.w * e.w);
      *reinterpret_cast<float4*>(&As[r][4 * k4]) = v;
    }
    for (int f = tid; f < kKC * D / 4; f += 256)
      reinterpret_cast<float4*>(Ws)[f] = __ldg(reinterpret_cast<const float4*>(W + (size_t)kc * D) + f);
    __syncthreads();
    tile_mac<4, CN>(As, Ws, D, ty, tx, acc);
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int row = row0 + ty * 4 + r;
    if (row >= N) continue;
    const size_t at = (size_t)row * D + tx * CN;
    float ov[CN], mv[CN];                                            // the stored values, for the peer stores
#pragma unroll
    for (int c = 0; c < CN; ++c) {
      const float z = acc[r][c];
      const float o = z > 0.f ? z : kSlope * z;                      // F.leaky_relu(z, 0.01)
      Enext[at + c] = o;
      ov[c] = o;
      if (acc_out != nullptr) {
        float m = (acc_in != nullptr ? acc_in[at + c] : 0.f) + o;
        if (acc_div != 1.0f) m = __fdiv_rn(m, acc_div);
        acc_out[at + c] = m;
        mv[c] = m;
      }
    }
    if constexpr (PEERS) {
      store_peers<CN>(peer_next, at, ov);
      if (acc_out != nullptr) store_peers<CN>(peer_acc, at, mv);
    }
  }
}

// --------------------------------------------------------------------------- backward
template <int D>
struct BwdSmem {
  static constexpr int LD = D + 4;
  static constexpr size_t bytes = (size_t)(3 * kTM * LD + kKC * D) * 4 + (size_t)kTM * (kKC + 4) * 4;
};

template <int D, bool PEERS>
__global__ void __launch_bounds__(256, 2) dense_bwd_kernel(const float* __restrict__ dOut, const float* __restrict__ Enext,
                                                           const float* __restrict__ P, const float* __restrict__ E,
                                                           const float* __restrict__ WT, float* __restrict__ dP,
                                                           float* __restrict__ dEdir, float* __restrict__ dWpart, int N,
                                                           RowPeers peer_dP) {
  constexpr int CN = D / 16, LD = D + 4;
  constexpr int JW = 2 * D / 16, CW = D / 16;       // weight-gradient block of a thread: JW rows of dW x CW columns
  extern __shared__ __align__(16) unsigned char bwd_smem[];
  float* Ps = reinterpret_cast<float*>(bwd_smem);                    // [TM][LD]
  float* Es = Ps + kTM * LD;
  float* Zs = Es + kTM * LD;
  float* Bs = Zs + kTM * LD;                                         // [KC][D] chunk of W^T columns
  float (*As)[kKC + 4] = reinterpret_cast<float (*)[kKC + 4]>(Bs + kKC * D);   // [TM][KC + 4]: dZ chunk for the products
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int jy = tid >> 4, cx = tid & 15;
  float wacc[JW][CW];
#pragma unroll
  for (int a = 0; a < JW; ++a)
#pragma unroll
    for (int c = 0; c < CW; ++c) wacc[a][c] = 0.f;
  const int n_tiles = (N + kTM - 1) / kTM;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row0 = tile * kTM;
    for (int f = tid; f < kTM * (D / 4); f += 256) {
      const int r = f / (D / 4), c4 = f - r * (D / 4);
      const int row = row0 + r;
      float4 p = make_float4(0.f, 0.f, 0.f, 0.f), e = p, z = p;
      if (row < N) {
        const size_t at = (size_t)row * D + 4 * c4;
        p = __ldg(reinterpret_cast<const float4*>(P + at));
        e = __ldg(reinterpret_cast<const float4*>(E + at));
        const float4 g = __ldg(reinterpret_cast<const float4*>(dOut + at));
        const float4 y = __ldg(reinterpret_cast<const float4*>(Enext + at));
        z = make_float4(y.x > 0.f ? g.x : kSlope * g.x, y.y > 0.f ? g.y : kSlope * g.y,
                        y.z > 0.f ? g.z : kSlope * g.z, y.w > 0.f ? g.w : kSlope * g.w);
      }
      *reinterpret_cast<float4*>(Ps + r * LD + 4 * c4) = p;
      *reinterpret_cast<float4*>(Es + r * LD + 4 * c4) = e;
      *reinterpret_cast<float4*>(Zs + r * LD + 4 * c4) = z;
    }
    __syncthreads();
    // [dA | dB] = dZ W^T: two products with the same left operand; K = D in chunks of KC
    float accA[4][CN], accB[4][CN];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < CN; ++c) { accA[r][c] = 0.f; accB[r][c] = 0.f; }
    for (int half = 0; half < 2; ++half) {
      for (int kc = 0; kc < D; kc += kKC) {
        const int kn = D - kc < kKC ? D - kc : kKC;                  // D = 32: one chunk of 32
        for (int f = tid; f < kTM * (kKC / 4); f += 256) {
          const int r = f / (kKC / 4), k4 = f - r * (kKC / 4);
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (4 * k4 < kn) v = *reinterpret_cast<const float4*>(Zs + r * LD + kc + 4 * k4);
          *reinterpret_cast<float4*>(&As[r][4 * k4]) = v;
        }
        for (int f = tid; f < kKC * D / 4; f += 256) {
          const int k = f / (D / 4), j4 = f - k * (D / 4);
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (k < kn) v = __ldg(reinterpret_cast<const float4*>(WT + (size_t)(kc + k) * 2 * D + half * D + 4 * j4));
          reinterpret_cast<float4*>(Bs)[f] = v;
        }
        __syncthreads();
        if (half == 0) tile_mac<4, CN>(As, Bs, D, ty, tx, accA);
        else tile_mac<4, CN>(As, Bs, D, ty, tx, accB);
        __syncthreads();
      }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int lr = ty * 4 + r, row = row0 + lr;
      if (row >= N) continue;
      float pv[CN];
#pragma unroll
      for (int c = 0; c < CN; ++c) {
        const int col = tx * CN + c;
        const float e = Es[lr * LD + col], p = Ps[lr * LD + col];
        pv[c] = fmaf(accB[r][c], e, accA[r][c]);
        dP[(size_t)row * D + col] = pv[c];
        dEdir[(size_t)row * D + col] = fmaf(accB[r][c], p, accA[r][c]);
      }
      if constexpr (PEERS) store_peers<CN>(peer_dP, (size_t)row * D + tx * CN, pv);
    }
    // dW[j'][c] += sum_n A'[n][j'] dZ[n][c]   with A' = [P + E | P * E] formed from the staged rows
    const int j0 = jy * JW, part = j0 / D, col0 = j0 - part * D;     // JW consecutive rows of dW stay inside one part
#pragma unroll 2
    for (int n = 0; n < kTM; ++n) {
      float a[JW], z[CW];
      load_cols<JW>(Ps + n * LD + col0, a);
      {
        float e[JW];
        load_cols<JW>(Es + n * LD + col0, e);
#pragma unroll
        for (int q = 0; q < JW; ++q) a[q] = part == 0 ? a[q] + e[q] : a[q] * e[q];
      }
      load_cols<CW>(Zs + n * LD + cx * CW, z);
#pragma unroll
      for (int q = 0; q < JW; ++q)
#pragma unroll
        for (int c = 0; c < CW; ++c) wacc[q][c] = fmaf(a[q], z[c], wacc[q][c]);
    }
    __syncthreads();                                                 // the next tile overwrites the staged rows
  }
  float* out = dWpart + (size_t)blockIdx.x * 2 * D * D;
#pragma unroll
  for (int q = 0; q < JW; ++q)
#pragma unroll
    for (int c = 0; c < CW; ++c) out[(size_t)(jy * JW + q) * D + cx * CW + c] = wacc[q][c];
}

// ------------------------------------------------------------------- d = 8 and 16
// The 16 x 16 thread grid above gives each thread D / 16 output columns: none at D = 8, and the k chunk of 64 is wider
// than 2D.  At these widths a row is 2D inputs and D outputs, so a thread owns a whole row: it reads its row of P and E
// (two or four float4 each), keeps [P + E | P * E] and the D accumulators in registers, and walks W (512 or 2 048 B, in
// shared memory, the same word for every lane: a broadcast).  Every output is the same chain as the tiled kernels'
// (fmaf, k ascending from 0).  The weight gradient is reduced per CTA through shared memory in row order, then across
// CTAs by reduce_wgrad_kernel in CTA order: deterministic.
constexpr int kSmallTM = 128;    // rows per CTA (one per thread)

template <int D>
__device__ __forceinline__ void load_row(const float* __restrict__ src, size_t row, float (&x)[D]) {
#pragma unroll
  for (int q = 0; q < D / 4; ++q) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(src + row * D) + q);
    x[4 * q] = v.x; x[4 * q + 1] = v.y; x[4 * q + 2] = v.z; x[4 * q + 3] = v.w;
  }
}

template <int D, bool PEERS>
__global__ void __launch_bounds__(kSmallTM) dense_fwd_small_kernel(const float* __restrict__ P, const float* __restrict__ E,
                                                                   const float* __restrict__ W, float* __restrict__ Enext,
                                                                   const float* __restrict__ acc_in, float* __restrict__ acc_out,
                                                                   float acc_div, int N, RowPeers peer_next,
                                                                   RowPeers peer_acc) {
  __shared__ __align__(16) float Ws[2 * D * D];
  for (int f = threadIdx.x; f < 2 * D * D; f += kSmallTM) Ws[f] = __ldg(W + f);
  __syncthreads();
  const int row = blockIdx.x * kSmallTM + threadIdx.x;
  if (row >= N) return;
  float p[D], e[D], acc[D];
  load_row<D>(P, (size_t)row, p);
  load_row<D>(E, (size_t)row, e);
#pragma unroll
  for (int c = 0; c < D; ++c) acc[c] = 0.f;
#pragma unroll
  for (int k = 0; k < 2 * D; ++k) {
    const float a = k < D ? p[k] + e[k] : p[k - D] * e[k - D];
#pragma unroll
    for (int c = 0; c < D; ++c) acc[c] = fmaf(a, Ws[k * D + c], acc[c]);
  }
  const size_t at = (size_t)row * D;
  float ov[D], mv[D];                                                // the stored values, for the peer stores
#pragma unroll
  for (int c = 0; c < D; ++c) {
    const float z = acc[c];
    const float o = z > 0.f ? z : kSlope * z;                        // F.leaky_relu(z, 0.01)
    Enext[at + c] = o;
    ov[c] = o;
    if (acc_out != nullptr) {
      float m = (acc_in != nullptr ? acc_in[at + c] : 0.f) + o;
      if (acc_div != 1.0f) m = __fdiv_rn(m, acc_div);
      acc_out[at + c] = m;
      mv[c] = m;
    }
  }
  if constexpr (PEERS) {
    store_peers<D>(peer_next, at, ov);
    if (acc_out != nullptr) store_peers<D>(peer_acc, at, mv);
  }
}

template <int D, bool PEERS>
__global__ void __launch_bounds__(kSmallTM) dense_bwd_small_kernel(const float* __restrict__ dOut, const float* __restrict__ Enext,
                                                                   const float* __restrict__ P, const float* __restrict__ E,
                                                                   const float* __restrict__ WT, float* __restrict__ dP,
                                                                   float* __restrict__ dEdir, float* __restrict__ dWpart, int N,
                                                                   RowPeers peer_dP) {
  constexpr int NW = 2 * D * D, WPT = NW / kSmallTM;                // dW entries, and per thread in the reduction (1 or 4)
  __shared__ __align__(16) float WTs[NW];                            // W^T: [D][2D]
  __shared__ float As[kSmallTM][2 * D + 1];                          // [P + E | P * E] of the tile's rows (+1: odd stride)
  __shared__ float Zs[kSmallTM][D + 1];                              // dZ of the tile's rows
  for (int f = threadIdx.x; f < NW; f += kSmallTM) WTs[f] = __ldg(WT + f);
  float wacc[WPT];
#pragma unroll
  for (int q = 0; q < WPT; ++q) wacc[q] = 0.f;
  const int n_tiles = (N + kSmallTM - 1) / kSmallTM;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int lr = threadIdx.x, row = tile * kSmallTM + lr;
    __syncthreads();                                                 // WTs staged / the previous tile's rows consumed
    if (row < N) {
      float p[D], e[D], z[D];
      load_row<D>(P, (size_t)row, p);
      load_row<D>(E, (size_t)row, e);
      {
        float g[D], y[D];
        load_row<D>(dOut, (size_t)row, g);
        load_row<D>(Enext, (size_t)row, y);
#pragma unroll
        for (int c = 0; c < D; ++c) z[c] = y[c] > 0.f ? g[c] : kSlope * g[c];
      }
      // [dA | dB] = dZ W^T, k ascending from 0
      float dA[D], dB[D];
#pragma unroll
      for (int j = 0; j < D; ++j) { dA[j] = 0.f; dB[j] = 0.f; }
#pragma unroll
      for (int k = 0; k < D; ++k)
#pragma unroll
        for (int j = 0; j < D; ++j) {
          dA[j] = fmaf(z[k], WTs[k * 2 * D + j], dA[j]);
          dB[j] = fmaf(z[k], WTs[k * 2 * D + D + j], dB[j]);
        }
      const size_t at = (size_t)row * D;
      float pv[D];
#pragma unroll
      for (int j = 0; j < D; ++j) {
        pv[j] = fmaf(dB[j], e[j], dA[j]);
        dP[at + j] = pv[j];
        dEdir[at + j] = fmaf(dB[j], p[j], dA[j]);
        As[lr][j] = p[j] + e[j];
        As[lr][D + j] = p[j] * e[j];
        Zs[lr][j] = z[j];
      }
      if constexpr (PEERS) store_peers<D>(peer_dP, at, pv);
    } else {
#pragma unroll
      for (int j = 0; j < D; ++j) { As[lr][j] = 0.f; As[lr][D + j] = 0.f; Zs[lr][j] = 0.f; }
    }
    __syncthreads();
    // dW[j'][c] += sum_n A'[n][j'] dZ[n][c], n ascending; thread t owns the entries t, t + 128, ...
#pragma unroll
    for (int q = 0; q < WPT; ++q) {
      const int w = threadIdx.x + q * kSmallTM, jr = w / D, c = w - jr * D;
      float s_ = wacc[q];
      for (int n = 0; n < kSmallTM; ++n) s_ = fmaf(As[n][jr], Zs[n][c], s_);
      wacc[q] = s_;
    }
  }
  float* out = dWpart + (size_t)blockIdx.x * NW;
#pragma unroll
  for (int q = 0; q < WPT; ++q) out[threadIdx.x + q * kSmallTM] = wacc[q];
}

// ------------------------------------------------------------------ d = 128 and 256
// The 64-row tiles above do not fit these widths: the forward's weight chunk takes its static shared memory past 48 KB,
// the backward would stage 150 / 281 KB and hold 128 / 512 dW accumulators per thread.  So each of the three products
// is a kernel of its own on one tile shape -- 128 rows x 128 columns on the 16 x 16 thread grid, 8 x 8 outputs per
// thread, K in chunks of 64 staged in 66 KB of dynamic shared memory -- over column blocks of its output:
//   dense_fwd_wide_kernel    Z = A' W                  grid (row tiles, D / 128)
//   dense_dzwt_wide_kernel   [dA | dB] = dZ W^T        grid (row tiles, D / 64); the tile's columns interleave dA_j and
//                            dB_j, so the thread that holds both forms dP and dE_direct
//   dense_wgrad_wide_kernel  dW = A'^T dZ, split over K: grid (dW tiles, n_partials row slices), one partial per slice,
//                            which reduce_wgrad_kernel adds in slice order
// dZ and A' are recomputed from dOut, Enext, P and E wherever a kernel stages them.  Every output is one fmaf chain, k
// ascending (dW: within its slice): exact fp32 and deterministic, like the narrower kernels.
constexpr int kWM = 128;          // rows and columns of a wide tile
constexpr int kWR = kWM / 16;     // rows and columns per thread
constexpr size_t kWideSmemBytes = (size_t)(kWM * (kKC + 4) + kKC * kWM) * 4;

__device__ __forceinline__ float4 dz_of(float4 g, float4 y) {        // dZ = dE' * (E' > 0 ? 1 : 0.01)
  return make_float4(y.x > 0.f ? g.x : kSlope * g.x, y.y > 0.f ? g.y : kSlope * g.y,
                     y.z > 0.f ? g.z : kSlope * g.z, y.w > 0.f ? g.w : kSlope * g.w);
}

template <int D, bool PEERS>
__global__ void __launch_bounds__(256) dense_fwd_wide_kernel(const float* __restrict__ P, const float* __restrict__ E,
                                                             const float* __restrict__ W, float* __restrict__ Enext,
                                                             const float* __restrict__ acc_in, float* __restrict__ acc_out,
                                                             float acc_div, int N, RowPeers peer_next, RowPeers peer_acc) {
  extern __shared__ __align__(16) unsigned char wide_smem[];
  float (*As)[kKC + 4] = reinterpret_cast<float (*)[kKC + 4]>(wide_smem);   // [WM][KC + 4]: A' chunk
  float* Ws = reinterpret_cast<float*>(wide_smem) + kWM * (kKC + 4);         // [KC][WM]: W chunk of the column block
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int row0 = blockIdx.x * kWM, c0 = blockIdx.y * kWM;
  float acc[kWR][kWR];
#pragma unroll
  for (int r = 0; r < kWR; ++r)
#pragma unroll
    for (int c = 0; c < kWR; ++c) acc[r][c] = 0.f;
  for (int kc = 0; kc < 2 * D; kc += kKC) {
    const int part = kc / D, col = kc - part * D;                   // a chunk stays inside one part (D % KC == 0)
    for (int f = tid; f < kWM * (kKC / 4); f += 256) {
      const int r = f / (kKC / 4), k4 = f - r * (kKC / 4);
      const int row = row0 + r;
      float4 p = make_float4(0.f, 0.f, 0.f, 0.f), e = p;
      if (row < N) {
        p = __ldg(reinterpret_cast<const float4*>(P + (size_t)row * D + col) + k4);
        e = __ldg(reinterpret_cast<const float4*>(E + (size_t)row * D + col) + k4);
      }
      *reinterpret_cast<float4*>(&As[r][4 * k4]) = part == 0 ? make_float4(p.x + e.x, p.y + e.y, p.z + e.z, p.w + e.w)
                                                             : make_float4(p.x * e.x, p.y * e.y, p.z * e.z, p.w * e.w);
    }
    for (int f = tid; f < kKC * (kWM / 4); f += 256) {
      const int k = f / (kWM / 4), c4 = f - k * (kWM / 4);
      reinterpret_cast<float4*>(Ws)[f] = __ldg(reinterpret_cast<const float4*>(W + (size_t)(kc + k) * D + c0) + c4);
    }
    __syncthreads();
    tile_mac<kWR, kWR>(As, Ws, kWM, ty, tx, acc);
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < kWR; ++r) {
    const int row = row0 + ty * kWR + r;
    if (row >= N) continue;
    const size_t at = (size_t)row * D + c0 + tx * kWR;
    float ov[kWR], mv[kWR];                                          // the stored values, for the peer stores
#pragma unroll
    for (int c = 0; c < kWR; ++c) {
      const float z = acc[r][c];
      const float o = z > 0.f ? z : kSlope * z;                      // F.leaky_relu(z, 0.01)
      Enext[at + c] = o;
      ov[c] = o;
      if (acc_out != nullptr) {
        float m = (acc_in != nullptr ? acc_in[at + c] : 0.f) + o;
        if (acc_div != 1.0f) m = __fdiv_rn(m, acc_div);
        acc_out[at + c] = m;
        mv[c] = m;
      }
    }
    if constexpr (PEERS) {
      store_peers<kWR>(peer_next, at, ov);
      if (acc_out != nullptr) store_peers<kWR>(peer_acc, at, mv);
    }
  }
}

template <int D, bool PEERS>
__global__ void __launch_bounds__(256) dense_dzwt_wide_kernel(const float* __restrict__ dOut, const float* __restrict__ Enext,
                                                              const float* __restrict__ P, const float* __restrict__ E,
                                                              const float* __restrict__ WT, float* __restrict__ dP,
                                                              float* __restrict__ dEdir, int N, RowPeers peer_dP) {
  extern __shared__ __align__(16) unsigned char wide_smem[];
  float (*As)[kKC + 4] = reinterpret_cast<float (*)[kKC + 4]>(wide_smem);   // [WM][KC + 4]: dZ chunk
  float* Bs = reinterpret_cast<float*>(wide_smem) + kWM * (kKC + 4);         // [KC][WM]: Bs[k][2j + h] = W^T[k][h D + j0 + j]
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int row0 = blockIdx.x * kWM, j0 = blockIdx.y * (kWM / 2);
  float acc[kWR][kWR];                                                // acc[r][2q] = dA, acc[r][2q + 1] = dB of column j0 + 4 tx + q
#pragma unroll
  for (int r = 0; r < kWR; ++r)
#pragma unroll
    for (int c = 0; c < kWR; ++c) acc[r][c] = 0.f;
  for (int kc = 0; kc < D; kc += kKC) {
    for (int f = tid; f < kWM * (kKC / 4); f += 256) {
      const int r = f / (kKC / 4), k4 = f - r * (kKC / 4);
      const int row = row0 + r;
      float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row < N) {
        const size_t at = (size_t)row * D + kc + 4 * k4;
        z = dz_of(__ldg(reinterpret_cast<const float4*>(dOut + at)), __ldg(reinterpret_cast<const float4*>(Enext + at)));
      }
      *reinterpret_cast<float4*>(&As[r][4 * k4]) = z;
    }
    for (int f = tid; f < kKC * (kWM / 8); f += 256) {
      const int k = f / (kWM / 8), j4 = f - k * (kWM / 8);
      const float* src = WT + (size_t)(kc + k) * 2 * D + j0 + 4 * j4;
      const float4 a = __ldg(reinterpret_cast<const float4*>(src)), b = __ldg(reinterpret_cast<const float4*>(src + D));
      float4* dst = reinterpret_cast<float4*>(Bs + k * kWM + 8 * j4);
      dst[0] = make_float4(a.x, b.x, a.y, b.y);
      dst[1] = make_float4(a.z, b.z, a.w, b.w);
    }
    __syncthreads();
    tile_mac<kWR, kWR>(As, Bs, kWM, ty, tx, acc);
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < kWR; ++r) {
    const int row = row0 + ty * kWR + r;
    if (row >= N) continue;
    const size_t at = (size_t)row * D + j0 + 4 * tx;
    const float4 e = __ldg(reinterpret_cast<const float4*>(E + at)), p = __ldg(reinterpret_cast<const float4*>(P + at));
    const float4 g = make_float4(fmaf(acc[r][1], e.x, acc[r][0]), fmaf(acc[r][3], e.y, acc[r][2]),
                                 fmaf(acc[r][5], e.z, acc[r][4]), fmaf(acc[r][7], e.w, acc[r][6]));
    *reinterpret_cast<float4*>(dP + at) = g;
    if constexpr (PEERS) {
      const float pv[4] = {g.x, g.y, g.z, g.w};
      store_peers<4>(peer_dP, at, pv);
    }
    *reinterpret_cast<float4*>(dEdir + at) = make_float4(fmaf(acc[r][1], p.x, acc[r][0]), fmaf(acc[r][3], p.y, acc[r][2]),
                                                         fmaf(acc[r][5], p.z, acc[r][4]), fmaf(acc[r][7], p.w, acc[r][6]));
  }
}

template <int D>
__global__ void __launch_bounds__(256) dense_wgrad_wide_kernel(const float* __restrict__ dOut, const float* __restrict__ Enext,
                                                               const float* __restrict__ P, const float* __restrict__ E,
                                                               float* __restrict__ dWpart, int N) {
  extern __shared__ __align__(16) unsigned char wide_smem[];
  float (*As)[kKC + 4] = reinterpret_cast<float (*)[kKC + 4]>(wide_smem);   // [WM][KC + 4]: As[j][n] = A'[n0 + n][j0 + j]
  float* Zs = reinterpret_cast<float*>(wide_smem) + kWM * (kKC + 4);         // [KC][WM]:     Zs[n][c] = dZ[n0 + n][c0 + c]
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  constexpr int kColTiles = D / kWM;
  const int j0 = (blockIdx.x / kColTiles) * kWM, c0 = (blockIdx.x % kColTiles) * kWM;
  const int part = j0 / D, col0 = j0 - part * D;                   // a 128-row block of dW stays inside one part
  const int n_chunks = (N + kKC - 1) / kKC, per = (n_chunks + gridDim.y - 1) / gridDim.y;
  const int ch0 = blockIdx.y * per, ch1 = min(n_chunks, ch0 + per);
  float acc[kWR][kWR];
#pragma unroll
  for (int r = 0; r < kWR; ++r)
#pragma unroll
    for (int c = 0; c < kWR; ++c) acc[r][c] = 0.f;
  for (int ch = ch0; ch < ch1; ++ch) {
    const int n0 = ch * kKC;
    for (int f = tid; f < kKC * (kWM / 4); f += 256) {              // n fastest across a warp: conflict-free stores
      const int n = f % kKC, j4 = f / kKC;
      const int row = n0 + n;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row < N) {
        const float4 p = __ldg(reinterpret_cast<const float4*>(P + (size_t)row * D + col0) + j4);
        const float4 e = __ldg(reinterpret_cast<const float4*>(E + (size_t)row * D + col0) + j4);
        v = part == 0 ? make_float4(p.x + e.x, p.y + e.y, p.z + e.z, p.w + e.w)
                      : make_float4(p.x * e.x, p.y * e.y, p.z * e.z, p.w * e.w);
      }
      As[4 * j4][n] = v.x; As[4 * j4 + 1][n] = v.y; As[4 * j4 + 2][n] = v.z; As[4 * j4 + 3][n] = v.w;
    }
    for (int f = tid; f < kKC * (kWM / 4); f += 256) {
      const int n = f / (kWM / 4), c4 = f - n * (kWM / 4);
      const int row = n0 + n;
      float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row < N) {
        const size_t at = (size_t)row * D + c0 + 4 * c4;
        z = dz_of(__ldg(reinterpret_cast<const float4*>(dOut + at)), __ldg(reinterpret_cast<const float4*>(Enext + at)));
      }
      reinterpret_cast<float4*>(Zs)[f] = z;
    }
    __syncthreads();
    tile_mac<kWR, kWR>(As, Zs, kWM, ty, tx, acc);
    __syncthreads();
  }
  float* out = dWpart + (size_t)blockIdx.y * 2 * D * D;
#pragma unroll
  for (int r = 0; r < kWR; ++r) {
    float4* dst = reinterpret_cast<float4*>(out + (size_t)(j0 + ty * kWR + r) * D + c0 + tx * kWR);
    dst[0] = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
    dst[1] = make_float4(acc[r][4], acc[r][5], acc[r][6], acc[r][7]);
  }
}

template <bool PEERS>
__global__ void __launch_bounds__(256) reduce_wgrad_kernel(const float* __restrict__ part, int n_part, int n, float* __restrict__ dW,
                                                           RowPeers peer_dW) {
  const int k = blockIdx.x * 256 + threadIdx.x;
  if (k >= n) return;
  float s = 0.f;
  for (int b = 0; b < n_part; ++b) s += part[(size_t)b * n + k];      // CTA (d >= 128: slice) order: deterministic
  dW[k] = s;
  if constexpr (PEERS) {
    const float sv[1] = {s};
    store_peers<1>(peer_dW, (size_t)k, sv);
  }
}

}  // namespace ngcf
}  // namespace agcf

using namespace agcf;

namespace {

// host arrays of peer pointers (+ multicast address) -> the kernel argument; false on a malformed list
bool make_peers(void* const* host, int32_t n_peers, void* mc, ngcf::RowPeers& out) {
  out = ngcf::RowPeers{};
  out.mc = reinterpret_cast<float*>(mc);
  if (mc != nullptr) return aligned16(mc);
  if (host == nullptr) return true;
  for (int q = 0; q < n_peers; ++q) {
    if (host[q] == nullptr || !aligned16(host[q])) return false;
    out.p[q] = reinterpret_cast<float*>(host[q]);
  }
  out.n = n_peers;
  return true;
}

template <bool PEERS>
int dense_forward(const float* P, const float* E, const float* W, float* Enext, const float* acc_in, float* acc_out,
                  float acc_div, int32_t n_rows, int32_t d, ngcf::RowPeers pn, ngcf::RowPeers pa, cudaStream_t st) {
  if (!P || !E || !W || !Enext || n_rows < 0 || acc_div == 0.f) return AGCF_EINVAL;
  if (d != 8 && d != 16 && d != 32 && d != 64 && d != 128 && d != 256) return AGCF_EUNSUPPORTED;
  if (!aligned16(P) || !aligned16(E) || !aligned16(W) || !aligned16(Enext) || !aligned16(acc_in) || !aligned16(acc_out)) return AGCF_EINVAL;
  if (Enext == P || Enext == E) return AGCF_EINVAL;
  if (n_rows == 0) return AGCF_OK;
  if (d >= 128) {
    const dim3 grid((unsigned)((n_rows + ngcf::kWM - 1) / ngcf::kWM), (unsigned)(d / ngcf::kWM));
#define AGCF_NGCF_FWD_WIDE(DD)                                                                                      \
  {                                                                                                                 \
    AGCF_CUDA_OK(cudaFuncSetAttribute(ngcf::dense_fwd_wide_kernel<DD, PEERS>,                                       \
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ngcf::kWideSmemBytes));     \
    ngcf::dense_fwd_wide_kernel<DD, PEERS><<<grid, 256, ngcf::kWideSmemBytes, st>>>(P, E, W, Enext, acc_in, acc_out, \
                                                                                    acc_div, n_rows, pn, pa);       \
  }
    if (d == 256) AGCF_NGCF_FWD_WIDE(256) else AGCF_NGCF_FWD_WIDE(128)
#undef AGCF_NGCF_FWD_WIDE
    AGCF_LAUNCH_OK();
    return AGCF_OK;
  }
  if (d <= 16) {
    const unsigned small_blocks = (unsigned)((n_rows + ngcf::kSmallTM - 1) / ngcf::kSmallTM);
    if (d == 16) ngcf::dense_fwd_small_kernel<16, PEERS><<<small_blocks, ngcf::kSmallTM, 0, st>>>(P, E, W, Enext, acc_in, acc_out, acc_div, n_rows, pn, pa);
    else ngcf::dense_fwd_small_kernel<8, PEERS><<<small_blocks, ngcf::kSmallTM, 0, st>>>(P, E, W, Enext, acc_in, acc_out, acc_div, n_rows, pn, pa);
    AGCF_LAUNCH_OK();
    return AGCF_OK;
  }
  const unsigned blocks = (unsigned)((n_rows + ngcf::kTM - 1) / ngcf::kTM);
  if (d == 64) ngcf::dense_fwd_kernel<64, PEERS><<<blocks, 256, 0, st>>>(P, E, W, Enext, acc_in, acc_out, acc_div, n_rows, pn, pa);
  else ngcf::dense_fwd_kernel<32, PEERS><<<blocks, 256, 0, st>>>(P, E, W, Enext, acc_in, acc_out, acc_div, n_rows, pn, pa);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

template <bool PEERS>
int dense_backward(const float* dOut, const float* Enext, const float* P, const float* E, const float* WT, float* dP,
                   float* dEdir, float* dW_partial, int32_t n_partials, int32_t n_rows, int32_t d, ngcf::RowPeers pp,
                   cudaStream_t st) {
  if (!dOut || !Enext || !P || !E || !WT || !dP || !dEdir || !dW_partial || n_rows < 0 || n_partials < 1) return AGCF_EINVAL;
  if (d != 8 && d != 16 && d != 32 && d != 64 && d != 128 && d != 256) return AGCF_EUNSUPPORTED;
  if (!aligned16(dOut) || !aligned16(Enext) || !aligned16(P) || !aligned16(E) || !aligned16(WT) || !aligned16(dP) ||
      !aligned16(dEdir) || !aligned16(dW_partial))
    return AGCF_EINVAL;
  if (dP == dOut || dEdir == dOut || dP == dEdir) return AGCF_EINVAL;
  if (d >= 128) {                       // [dA | dB] over row tiles, then dW split over n_partials row slices
    const dim3 grid_dz((unsigned)((n_rows + ngcf::kWM - 1) / ngcf::kWM), (unsigned)(d / (ngcf::kWM / 2)));
    const dim3 grid_w((unsigned)((2 * d / ngcf::kWM) * (d / ngcf::kWM)), (unsigned)n_partials);
#define AGCF_NGCF_BWD_WIDE(DD)                                                                                       \
  {                                                                                                                  \
    AGCF_CUDA_OK(cudaFuncSetAttribute(ngcf::dense_dzwt_wide_kernel<DD, PEERS>,                                       \
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ngcf::kWideSmemBytes));      \
    AGCF_CUDA_OK(cudaFuncSetAttribute(ngcf::dense_wgrad_wide_kernel<DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                      (int)ngcf::kWideSmemBytes));                                                   \
    if (n_rows > 0)                                                                                                  \
      ngcf::dense_dzwt_wide_kernel<DD, PEERS><<<grid_dz, 256, ngcf::kWideSmemBytes, st>>>(dOut, Enext, P, E, WT, dP,  \
                                                                                          dEdir, n_rows, pp);        \
    ngcf::dense_wgrad_wide_kernel<DD><<<grid_w, 256, ngcf::kWideSmemBytes, st>>>(dOut, Enext, P, E, dW_partial,       \
                                                                                 n_rows);                            \
  }
    if (d == 256) AGCF_NGCF_BWD_WIDE(256) else AGCF_NGCF_BWD_WIDE(128)
#undef AGCF_NGCF_BWD_WIDE
    AGCF_LAUNCH_OK();
    return AGCF_OK;
  }
  if (d <= 16) {
    if (d == 16) ngcf::dense_bwd_small_kernel<16, PEERS><<<(unsigned)n_partials, ngcf::kSmallTM, 0, st>>>(dOut, Enext, P, E, WT, dP, dEdir, dW_partial, n_rows, pp);
    else ngcf::dense_bwd_small_kernel<8, PEERS><<<(unsigned)n_partials, ngcf::kSmallTM, 0, st>>>(dOut, Enext, P, E, WT, dP, dEdir, dW_partial, n_rows, pp);
    AGCF_LAUNCH_OK();
    return AGCF_OK;
  }
#define AGCF_NGCF_BWD(DD)                                                                                      \
  {                                                                                                            \
    AGCF_CUDA_OK(cudaFuncSetAttribute(ngcf::dense_bwd_kernel<DD, PEERS>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                      (int)ngcf::BwdSmem<DD>::bytes));                                         \
    ngcf::dense_bwd_kernel<DD, PEERS><<<(unsigned)n_partials, 256, ngcf::BwdSmem<DD>::bytes, st>>>(            \
        dOut, Enext, P, E, WT, dP, dEdir, dW_partial, n_rows, pp);                                             \
  }
  if (d == 64) AGCF_NGCF_BWD(64) else AGCF_NGCF_BWD(32)
#undef AGCF_NGCF_BWD
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

template <bool PEERS>
int reduce_wgrad(const float* dW_partial, int32_t n_partials, float* dW, int32_t d, ngcf::RowPeers pw, cudaStream_t st) {
  if (!dW_partial || !dW || n_partials < 1) return AGCF_EINVAL;
  if (d != 8 && d != 16 && d != 32 && d != 64 && d != 128 && d != 256) return AGCF_EUNSUPPORTED;
  const int n = 2 * d * d;
  ngcf::reduce_wgrad_kernel<PEERS><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dW_partial, n_partials, n, dW, pw);
  AGCF_LAUNCH_OK();
  return AGCF_OK;
}

}  // namespace

extern "C" int agcf_ngcf_dense_forward(const float* P, const float* E, const float* W, float* Enext,
                                       const float* acc_in, float* acc_out, float acc_div,
                                       int32_t n_rows, int32_t d, agcf_stream_t stream) {
  return dense_forward<false>(P, E, W, Enext, acc_in, acc_out, acc_div, n_rows, d, ngcf::RowPeers{}, ngcf::RowPeers{},
                              (cudaStream_t)stream);
}

extern "C" int agcf_ngcf_dense_backward(const float* dOut, const float* Enext, const float* P, const float* E,
                                        const float* WT, float* dP, float* dEdir, float* dW_partial,
                                        int32_t n_partials, int32_t n_rows, int32_t d, agcf_stream_t stream) {
  return dense_backward<false>(dOut, Enext, P, E, WT, dP, dEdir, dW_partial, n_partials, n_rows, d, ngcf::RowPeers{},
                               (cudaStream_t)stream);
}

extern "C" int agcf_ngcf_reduce_wgrad(const float* dW_partial, int32_t n_partials, float* dW, int32_t d,
                                      agcf_stream_t stream) {
  return reduce_wgrad<false>(dW_partial, n_partials, dW, d, ngcf::RowPeers{}, (cudaStream_t)stream);
}

extern "C" int agcf_ngcf_dense_forward_peers(const float* P, const float* E, const float* W, float* Enext,
                                             const float* acc_in, float* acc_out, float acc_div,
                                             int32_t n_rows, int32_t d,
                                             void* const* peer_Enext_host, void* const* peer_acc_host, int32_t n_peers,
                                             void* mc_Enext, void* mc_acc, agcf_stream_t stream) {
  if (n_peers < 0 || n_peers > AGCF_MAX_PEERS || (mc_acc != nullptr && acc_out == nullptr) ||
      ((peer_acc_host != nullptr || mc_acc != nullptr) && acc_out == nullptr))
    return AGCF_EINVAL;
  ngcf::RowPeers pn, pa;
  if (!make_peers(peer_Enext_host, n_peers, mc_Enext, pn) || !make_peers(peer_acc_host, n_peers, mc_acc, pa)) return AGCF_EINVAL;
  return dense_forward<true>(P, E, W, Enext, acc_in, acc_out, acc_div, n_rows, d, pn, pa, (cudaStream_t)stream);
}

extern "C" int agcf_ngcf_dense_backward_peers(const float* dOut, const float* Enext, const float* P, const float* E,
                                              const float* WT, float* dP, float* dEdir, float* dW_partial,
                                              int32_t n_partials, int32_t n_rows, int32_t d,
                                              void* const* peer_dP_host, int32_t n_peers, void* mc_dP,
                                              agcf_stream_t stream) {
  if (n_peers < 0 || n_peers > AGCF_MAX_PEERS) return AGCF_EINVAL;
  ngcf::RowPeers pp;
  if (!make_peers(peer_dP_host, n_peers, mc_dP, pp)) return AGCF_EINVAL;
  return dense_backward<true>(dOut, Enext, P, E, WT, dP, dEdir, dW_partial, n_partials, n_rows, d, pp, (cudaStream_t)stream);
}

extern "C" int agcf_ngcf_reduce_wgrad_peers(const float* dW_partial, int32_t n_partials, float* dW, int32_t d,
                                            void* const* peer_dW_host, int32_t n_peers, void* mc_dW,
                                            agcf_stream_t stream) {
  if (n_peers < 0 || n_peers > AGCF_MAX_PEERS) return AGCF_EINVAL;
  ngcf::RowPeers pw;
  if (!make_peers(peer_dW_host, n_peers, mc_dW, pw)) return AGCF_EINVAL;
  return reduce_wgrad<true>(dW_partial, n_partials, dW, d, pw, (cudaStream_t)stream);
}
