// Shared device/host helpers for libcor_b200.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/cor_b200.h"

namespace cor {

// ---- host-side error plumbing ---------------------------------------------------------------
void set_error(const char* fmt, ...);
int check_launch(const char* what);   // cudaGetLastError -> COR_ECUDA
int sm_count();                       // cached multiprocessor count of the current device
// lse[q] from `nparts` (max,sum) partials laid out [qtile][nparts][qt][2] (sim_stream.cu)
int launch_lse_combine(const float* part, int Nq, int nparts, int qt, float* lse, cudaStream_t st);
// tcgen05 similarity producer (sim_umma.cu): S or lse, not both; nparts/qt non-NULL: leave the LSE partials in `work`,
// report their layout.  Every InfoNCE kernel takes (inv_tau, scale): a non-NULL scale is the device-resident logit scale
// that replaces inv_tau.
int sim_umma_launch(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, const float* scale, float* S,
                    float* lse, void* work, int* nparts, int* qt, cudaStream_t st);

// same, queries held in tensor memory (sim_umma_ts.cu); log-sum-exp partials only: [qtile][*nparts][256][2] in `work`
int sim_umma_ts_launch(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, const float* scale, void* work,
                       int* nparts, cudaStream_t st);

#define COR_REQUIRE(cond, ...)          \
  do {                                  \
    if (!(cond)) {                      \
      ::cor::set_error(__VA_ARGS__);    \
      return COR_EINVAL;                \
    }                                   \
  } while (0)

#define COR_CUDA(expr)                                                          \
  do {                                                                          \
    cudaError_t _e = (expr);                                                    \
    if (_e != cudaSuccess) {                                                    \
      ::cor::set_error("%s: %s", #expr, cudaGetErrorString(_e));                \
      return COR_ECUDA;                                                         \
    }                                                                           \
  } while (0)

static inline cudaStream_t as_stream(cor_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// ---- device helpers -------------------------------------------------------------------------
typedef __nv_bfloat16 bf16;

template <typename T>
__device__ __forceinline__ float to_f(T v);
template <>
__device__ __forceinline__ float to_f<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f<bf16>(bf16 v) { return __bfloat162float(v); }
template <>
__device__ __forceinline__ float to_f<uint8_t>(uint8_t v) { return (float)v; }

template <typename T>
__device__ __forceinline__ T from_f(float v);
template <>
__device__ __forceinline__ float from_f<float>(float v) { return v; }
template <>
__device__ __forceinline__ bf16 from_f<bf16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

constexpr int kQT = 16;          // queries per tile of the streaming similarity kernels (one lane per query after the transposed reduce)

// ---- warp-per-region-row similarity: transposed butterfly -------------------------------------------
// After the per-lane partial dot products a transposed butterfly leaves S[q0+lane, r] in lane `lane`
// (lanes >= kQT idle): 16+8+4+2+1 = 31 shuffles instead of 16*5.
__device__ __forceinline__ float transpose_reduce16(float (&a)[kQT], int lane) {
  // step 1: fold the two half-warps; every lane keeps all 16 partials
#pragma unroll
  for (int q = 0; q < kQT; ++q) a[q] += __shfl_xor_sync(0xffffffffu, a[q], 16);
  // steps 2..5: keep the half that belongs to this lane's bit
#pragma unroll
  for (int s = 8, n = kQT; s >= 1; s >>= 1, n >>= 1) {
    const bool up = lane & s;
#pragma unroll
    for (int q = 0; q < n / 2; ++q) {
      const float mine = up ? a[q + n / 2] : a[q];
      const float theirs = up ? a[q] : a[q + n / 2];
      a[q] = mine + __shfl_xor_sync(0xffffffffu, theirs, s);
    }
  }
  return a[0];   // lane l (l < 16, counting bits 8,4,2,1) holds query index l
}

// ---- GELU (erf form, torch nn.GELU() default) on the SFU, branch-free --------------------------------------------------
// 1 - Phi(|x|) = 0.5 erfc(|x| / sqrt 2) through Abramowitz-Stegun 7.1.26: erfc(z) = (a1 t + .. + a5 t^5) exp(-z^2),
// t = 1 / (1 + p z), |error| <= 1.5e-7 absolute.  MUFU.RCP + MUFU.EX2 + 9 FMA-pipe instructions; the 0.5 is folded into
// the coefficients and exp(-z^2) = 2^(-x^2 * log2(e) / 2).  `e` returns that exponential (the Gaussian of gelu').
// Used where the result is rounded to bf16 anyway (GEMM epilogue with bf16 output, activation backward): libdevice's
// erff + expf + IEEE reciprocal cost 45 instructions and a branch per element and made the epilogue the bottleneck.
__device__ __forceinline__ float gelu_tail(float x, float& e) {
  const float z = fabsf(x) * 0.70710678118654752f;
  float t, ee;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.f)));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ee) : "f"(x * x * -0.72134752044448170f));
  float p = fmaf(0.5307027145f, t, -0.7265760135f);
  p = fmaf(p, t, 0.7107068705f);
  p = fmaf(p, t, -0.142248368f);
  p = fmaf(p, t, 0.127414796f);
  e = ee;
  return p * t * ee;                                          // 1 - Phi(|x|)
}
__device__ __forceinline__ float gelu_cdf_fast(float x, float& e) {
  const float q = gelu_tail(x, e);
  return 0.5f + copysignf(0.5f - q, x);                      // Phi(x) = 1 - q (x >= 0), q (x < 0)
}
__device__ __forceinline__ float gelu_fast(float x) {
  float e;
  return x * gelu_cdf_fast(x, e);
}
// d gelu / dx = Phi(x) + x phi(x), phi(x) = exp(-x^2 / 2) / sqrt(2 pi): one exponential for both terms
__device__ __forceinline__ float gelu_grad_fast(float x) {
  float e;
  const float cdf = gelu_cdf_fast(x, e);
  return fmaf(x * 0.3989422804014327f, e, cdf);
}

// Sum over `nparts` partial rows of column c (part[k * ld + c]) by a (32, kFoldTy = 32) thread block: thread row ty takes
// k = ty, ty + kFoldTy, ... with eight independent accumulators (loads pipeline; a single serial chain over ~2000 partials
// cost 100 us), then the kFoldTy row sums are added in fixed order.  Deterministic; the total is returned to ty == 0.
constexpr int kFoldTy = 32;
__device__ __forceinline__ float fold_parts(const float* __restrict__ part, int nparts, long long ld, long long c, bool ok,
                                            float (*sm)[32]) {
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (ok) {
    int k = threadIdx.y;
    for (; k + 7 * kFoldTy < nparts; k += 8 * kFoldTy) {
#pragma unroll
      for (int u = 0; u < 8; ++u) s[u] += part[(long long)(k + u * kFoldTy) * ld + c];
    }
    for (; k < nparts; k += kFoldTy) s[0] += part[(long long)k * ld + c];
  }
  sm[threadIdx.y][threadIdx.x] = ((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7]));
  __syncthreads();
  float t = 0.f;
  if (threadIdx.y == 0) {
#pragma unroll
    for (int j = 0; j < kFoldTy; ++j) t += sm[j][threadIdx.x];
  }
  return t;
}

// Block-wide sum of NV values per thread; result valid in every thread.  `scratch` needs
// NV * 32 floats.  Deterministic (fixed tree).
template <int NV, typename T>
__device__ __forceinline__ void block_sum(T (&v)[NV], T* scratch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) scratch[i * 32 + warp] = v[i];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    T x = (lane < nwarp) ? scratch[i * 32 + lane] : T(0);
    v[i] = warp_sum(x);
  }
}

// 16-byte streaming load that does not pollute L1 (read-once data).
__device__ __forceinline__ uint4 ld_stream16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ float bf16lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }
__device__ __forceinline__ float sigmoid_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

// ATen area_pixel_compute_source_index (align_corners=False, non-cubic), UpSample.cuh.
__device__ __forceinline__ void src_index(float scale, int dst, int in_size, int& i0, int& i1, float& l0, float& l1) {
  float src = scale * ((float)dst + 0.5f) - 0.5f;
  src = src < 0.f ? 0.f : src;
  i0 = min((int)src, in_size - 1);
  i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
  l1 = src - (float)i0;
  l0 = 1.0f - l1;
}

}  // namespace cor
