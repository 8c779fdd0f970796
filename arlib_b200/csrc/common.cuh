// common.cuh -- shared helpers for libagcf (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/agcf.h"

namespace agcf {

extern thread_local int g_last_cuda_error;
extern thread_local const char* g_last_cuda_file;
extern thread_local int g_last_cuda_line;

inline int cuda_fail(cudaError_t e, const char* file = "", int line = 0) {
  g_last_cuda_error = (int)e;
  g_last_cuda_file = file;
  g_last_cuda_line = line;
  return AGCF_ECUDA;
}

#define AGCF_CUDA_OK(expr)                                                       \
  do {                                                                           \
    cudaError_t _e = (expr);                                                     \
    if (_e != cudaSuccess) return ::agcf::cuda_fail(_e, __FILE__, __LINE__);     \
  } while (0)

#define AGCF_LAUNCH_OK()                                                         \
  do {                                                                           \
    cudaError_t _e = cudaGetLastError();                                         \
    if (_e != cudaSuccess) return ::agcf::cuda_fail(_e, __FILE__, __LINE__);     \
  } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
// embedding widths every kernel family is compiled for (the NGCF dense layer and the tcgen05 scoring stage take subsets)
inline bool supported_d(int d) { return d == 8 || d == 16 || d == 32 || d == 64 || d == 128 || d == 256; }

constexpr int kSMs = 148;  // B200

// streaming (read-once) loads: keep L1 for the gathered embedding rows
__device__ __forceinline__ int ld_stream_i32(const int* p) {
  int v;
  asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_stream_f32(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
// cached read-only gather (rows are re-used across a CTA's neighbours)
__device__ __forceinline__ float4 ld_gather_f4(const float4* p) { return __ldg(p); }

__device__ __forceinline__ void st_stream_f4(float4* p, const float4& v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// store through an NVSwitch multicast mapping: the switch replicates the 16 bytes into every GPU's copy
__device__ __forceinline__ void st_multicast_f4(float4* mc, const float4& v) {
  asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1,%2,%3,%4};"
               :: "l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ void fma4(float4& acc, float a, const float4& x) {
  acc.x = fmaf(a, x.x, acc.x);
  acc.y = fmaf(a, x.y, acc.y);
  acc.z = fmaf(a, x.z, acc.z);
  acc.w = fmaf(a, x.w, acc.w);
}
// packed fp32x2 FMA (sm_100 FFMA2): two IEEE fused multiply-adds per instruction --
// bit-identical to two fmaf() calls, half the issue slots
__device__ __forceinline__ void fma4_packed(float4& acc, float a, const float4& x) {
  unsigned long long lo, hi, xl, xh, aa;
  asm("mov.b64 %0, {%1, %2};" : "=l"(lo) : "f"(acc.x), "f"(acc.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(hi) : "f"(acc.z), "f"(acc.w));
  asm("mov.b64 %0, {%1, %2};" : "=l"(xl) : "f"(x.x), "f"(x.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(xh) : "f"(x.z), "f"(x.w));
  asm("mov.b64 %0, {%1, %1};" : "=l"(aa) : "f"(a));
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(lo) : "l"(aa), "l"(xl));
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(hi) : "l"(aa), "l"(xh));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(acc.x), "=f"(acc.y) : "l"(lo));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(acc.z), "=f"(acc.w) : "l"(hi));
}
__device__ __forceinline__ float4 add4(const float4& a, const float4& b) {
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
__device__ __forceinline__ float dot4(const float4& a, const float4& b) {
  return fmaf(a.w, b.w, fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x)));
}

// reduce over a group of LPR consecutive lanes (LPR power of two <= 32); all
// lanes of the group get the sum; fixed butterfly order => deterministic
template <int LPR>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- Philox4x32-10 (Salmon et al. 2011), counter-based -----------------------
struct Philox {
  static constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  static constexpr uint32_t W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
  __host__ __device__ static inline void round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
    uint64_t p0 = (uint64_t)M0 * c[0];
    uint64_t p1 = (uint64_t)M1 * c[2];
    uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
    uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
    uint32_t n0 = hi1 ^ c[1] ^ k0;
    uint32_t n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
  }
  __host__ __device__ static inline void gen(uint64_t key, uint64_t ctr_lo, uint64_t ctr_hi, uint32_t (&out)[4]) {
    uint32_t c[4] = {(uint32_t)ctr_lo, (uint32_t)(ctr_lo >> 32), (uint32_t)ctr_hi, (uint32_t)(ctr_hi >> 32)};
    uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      round(c, k0, k1);
      k0 += W0; k1 += W1;
    }
    out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
  }
};

}  // namespace agcf
