// General bf16 GEMM on tcgen05 tensor cores with a fused epilogue: the building block of the learned modules either side
// of the region path (SURVEY.md 8f): the 1x1 convolutions and the 4x point-wise MLP of the ConvNeXt blocks in
// GenerateMaskAdapterMap (lib/support_model/mask_adapter.py:97-223), and the linear layers of the composed-query head
// (lib/support_model/cir_feature_fuse.py:20-43, lib/support_branch.py:47-54), forward AND backward:
//
//   C[b][m][n] = epilogue( sum_k A[b](m, k) * B[b](n, k) )        fp32 accumulate in TMEM
//
// Each operand is read as it lies in memory, in either orientation, so no transpose is ever materialised:
//   K-major  : stored [rows][K]  (K contiguous)      e.g. activations [pixels][C], weights [out][in]
//   MN-major : stored [K][rows]  (rows contiguous)   e.g. an NCHW feature map as A (K = channels, M = pixels), a
//              weight [out][in] as the B of dX = dY W (K = out), dY / X as both operands of dW = dY^T X (K = rows)
// (TMA SW128 tiles either way; MN-major tiles are 64-row x 64-k boxes whose UMMA descriptor has LBO = one box, SBO = 1024 B.)
//
// Persistent CTAs walk 128 x 128 output tiles (x batch x split-K); 6-stage TMA ring; TMEM accumulator double-buffered
// so the MMAs of tile i+1 run under the epilogue of tile i; the whole MMA warp walks the issue loop and one elected
// lane issues (descriptors stay in uniform registers).  Epilogue per element, in this order:
//   v = acc * alpha; v += bias[n]; pre[m][n] = v (optional, bf16); v = act(v); v *= emul[m][n] (dropout mask, optional);
//   v *= colscale[n]; v += residual[m][n]; C = v
// Split-K (gridDim.y > 1, for the weight-gradient GEMMs whose K is the row count) writes raw fp32 partials and a fold
// kernel applies the epilogue in fixed order (deterministic).
// Warp roles (576 threads): 0..15 epilogue (TMEM lane quarter w % 4, 32-column chunk w / 4 of the 128-column tile -- four
// epilogue warps per scheduler: with two the short-K GEMMs, which are epilogue-bound, filled 40 % of the issue slots),
// 16 TMA producer, 17 MMA issuer.
#include "umma.cuh"

namespace cor {

using namespace umma;

constexpr int kGmBM = 128, kGmBN = 128, kGmBK = 64;
constexpr int kGmTile = 128 * 64 * 2;            // 16 KB: one operand stage
constexpr int kGmStages = 5;
constexpr int kGmStgPitch = 80, kGmStgBytes = 32 * kGmStgPitch;      // per-warp transpose block: 32 rows x (64 B + 16 B pad)
constexpr int kGmEpiWarps = 16, kGmTmaWarp = 16, kGmMmaWarp = 17, kGmThreads = 32 * (kGmEpiWarps + 2);

struct GemmSmemTail {
  uint64_t full[kGmStages], empty[kGmStages], acc_full[2], acc_empty[2];
  uint32_t tmem_base;
};

struct GemmArgs {
  int M, N, K, batch;
  int a_mn, b_mn;                       // operand orientation: 0 = K-major ([rows][K]), 1 = MN-major ([K][rows])
  long long a_batch_rows, b_batch_rows; // rows of the 2-D tensor map one batch entry spans (0 = operand shared by all)
  int ksplit;                           // == gridDim.y
  float alpha;
  const float* bias;                    // [N] or null
  const float* colscale;                // [N] or null
  const float* emul;                    // [batch][M][N] element-wise multiplier after the activation (dropout mask) or null
  const void* residual;                 // [batch][M][ldr] or null
  int res_bf16;
  long long ldr;
  int act;                              // COR_ACT_*
  void* C;                              // [batch][M][ldc]  (ksplit == 1)
  int c_bf16;
  long long ldc;
  bf16* pre;                            // [batch][M][ldc] pre-activation copy or null
  float* part;                          // [ksplit][batch][M][N] raw partials (ksplit > 1)
};

__device__ __forceinline__ float gemm_act(float v, int act) {
  if (act == COR_ACT_RELU) return fmaxf(v, 0.f);
  if (act == COR_ACT_GELU) return 0.5f * v * (1.f + erff(v * 0.70710678118654752f));     // torch nn.GELU() default (erf form)
  if (act == COR_ACT_SIGMOID) return 1.f / (1.f + __expf(-v));
  return v;
}

// The activation over a 32-column chunk with the switch OUTSIDE the unrolled loop: one branch per chunk, 32 independent
// evaluations in flight (a per-element switch compiled to an indirect branch per element and serialised the epilogue).
// ``fast_gelu`` (bf16 outputs only): gelu_fast of common.cuh (SFU form, |error| <= 1.5e-7 absolute on Phi, far below the
// bf16 rounding of the stored value).
__device__ __forceinline__ void gemm_act32(float (&o)[32], int act, bool fast_gelu) {
  switch (act) {
    case COR_ACT_RELU:
#pragma unroll
      for (int j = 0; j < 32; ++j) o[j] = fmaxf(o[j], 0.f);
      break;
    case COR_ACT_GELU:
      if (fast_gelu) {
#pragma unroll
        for (int j = 0; j < 32; ++j) o[j] = gelu_fast(o[j]);
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) o[j] = 0.5f * o[j] * (1.f + erff(o[j] * 0.70710678118654752f));
      }
      break;
    case COR_ACT_SIGMOID:
#pragma unroll
      for (int j = 0; j < 32; ++j) o[j] = 1.f / (1.f + __expf(-o[j]));
      break;
    default: break;
  }
}

__device__ __forceinline__ uint64_t make_desc_sw128_mnmajor(uint32_t smem_addr) {       // LBO = one 64 x 64 box (8 KB), SBO = 1024 B
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(8192 >> 4) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// The epilogue thread owns one ROW of the tile (TMEM lane), so a direct 16-byte store per lane touches 32 different rows:
// 32 half-written sectors per instruction.  These two primitives transpose 32 rows x 64 bytes through a per-warp shared
// block so that every global access instruction covers 8 rows x 64 contiguous bytes (16 whole sectors): lane r writes its
// row (pitch 80 B: the eight lanes of a phase hit eight different 16-byte bank groups), then lane l moves chunk l / 8 of row
// 8 it + l % 8.  Rows >= rows_valid are skipped (ragged M).  All 32 lanes must call.
// (explicit shared-space accesses: through a pointer derived from the dynamic-smem base the compiler emitted generic
// LD / ST, which wait on the long scoreboard)
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void warp_rows_store64(uint32_t stg, int lane, const uint4 (&c)[4], uint8_t* gbase, long long pitch, int rows_valid) {
#pragma unroll
  for (int j = 0; j < 4; ++j) sts128(stg + lane * kGmStgPitch + j * 16, c[j]);
  __syncwarp();
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int r = it * 8 + (lane & 7), ch = lane >> 3;
    const uint4 v = lds128(stg + r * kGmStgPitch + ch * 16);
    if (r < rows_valid) *reinterpret_cast<uint4*>(gbase + r * pitch + ch * 16) = v;
  }
  __syncwarp();
}
__device__ __forceinline__ void warp_rows_load64(uint32_t stg, int lane, uint4 (&c)[4], const uint8_t* gbase, long long pitch, int rows_valid) {
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int r = it * 8 + (lane & 7), ch = lane >> 3;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (r < rows_valid) v = *reinterpret_cast<const uint4*>(gbase + r * pitch + ch * 16);
    sts128(stg + r * kGmStgPitch + ch * 16, v);
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 4; ++j) c[j] = lds128(stg + lane * kGmStgPitch + j * 16);
  __syncwarp();
}
__device__ __forceinline__ void pack_bf16_16(const float* o, uint4 (&c)[4]) {      // 32 floats -> 64 bytes
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint32_t w[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      __nv_bfloat162 pk = __floats2bfloat162_rn(o[8 * j + 2 * q], o[8 * j + 2 * q + 1]);
      w[q] = *reinterpret_cast<uint32_t*>(&pk);
    }
    c[j] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

__global__ void __launch_bounds__(kGmThreads, 1) gemm_umma_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                                                           GemmArgs g) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* base = reinterpret_cast<uint8_t*>(((uintptr_t)smem + 1023) & ~(uintptr_t)1023);
  GemmSmemTail* tail = reinterpret_cast<GemmSmemTail*>(base + (size_t)kGmStages * 2 * kGmTile);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t stg = smem_u32(reinterpret_cast<uint8_t*>(tail) + ((sizeof(GemmSmemTail) + 15) & ~(size_t)15)) + (uint32_t)((warp < kGmEpiWarps ? warp : 0) * kGmStgBytes);
  const int mt = (g.M + kGmBM - 1) / kGmBM, nt = (g.N + kGmBN - 1) / kGmBN;
  const int ntiles = mt * nt * g.batch;
  const int nkb_all = (g.K + kGmBK - 1) / kGmBK;
  const int ks = blockIdx.y;
  const int kb0 = (int)((long long)ks * nkb_all / g.ksplit), kb1 = (int)((long long)(ks + 1) * nkb_all / g.ksplit);
  const int nkb = kb1 - kb0;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int i = 0; i < kGmStages; ++i) { mbar_init(&tail->full[i], 1); mbar_init(&tail->empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tail->acc_full[i], 1); mbar_init(&tail->acc_empty[i], kGmEpiWarps); }
    fence_barrier_init();
  }
  if (warp == kGmMmaWarp) tmem_alloc(&tail->tmem_base, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tail->tmem_base;

  if (warp == kGmTmaWarp) {
    if (lane == 0) {
      int st = 0;
      uint32_t ph = 1;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int b = t / (mt * nt), r = t % (mt * nt);
        const int m0 = (r / nt) * kGmBM, n0 = (r % nt) * kGmBN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&tail->empty[st], ph);
          uint8_t* sa = base + (size_t)st * 2 * kGmTile;
          uint8_t* sb = sa + kGmTile;
          mbar_expect_tx(&tail->full[st], 2 * kGmTile);
          const int k0 = kb * kGmBK;
          if (g.a_mn) {   // stored [K][M]: two 64-row boxes side by side
            tma_load_2d(sa, &tmA, &tail->full[st], m0, (int)(b * g.a_batch_rows) + k0, kEvictNormal);
            tma_load_2d(sa + 8192, &tmA, &tail->full[st], m0 + 64, (int)(b * g.a_batch_rows) + k0, kEvictNormal);
          } else {
            tma_load_2d(sa, &tmA, &tail->full[st], k0, (int)(b * g.a_batch_rows) + m0, kEvictNormal);
          }
          if (g.b_mn) {
            tma_load_2d(sb, &tmB, &tail->full[st], n0, (int)(b * g.b_batch_rows) + k0, kEvictLast);
            tma_load_2d(sb + 8192, &tmB, &tail->full[st], n0 + 64, (int)(b * g.b_batch_rows) + k0, kEvictLast);
          } else {
            tma_load_2d(sb, &tmB, &tail->full[st], k0, (int)(b * g.b_batch_rows) + n0, kEvictLast);
          }
          if (++st == kGmStages) { st = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == kGmMmaWarp) {
    const bool leader = elect_one();
    const uint32_t idesc = make_idesc_bf16(kGmBM, kGmBN) | (g.a_mn ? (1u << 15) : 0u) | (g.b_mn ? (1u << 16) : 0u);
    const uint32_t s_base = smem_u32(base);
    int st = 0, i = 0;
    uint32_t ph = 0;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++i) {
      const int buf = i & 1;
      mbar_wait(&tail->acc_empty[buf], ((i >> 1) & 1) ^ 1);
      tc_fence_after();
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(&tail->full[st], ph);
        tc_fence_after();
        if (leader) {
          const uint32_t sa = s_base + (uint32_t)(st * 2 * kGmTile), sb = sa + kGmTile;
          const uint64_t da = g.a_mn ? make_desc_sw128_mnmajor(sa) : make_desc_sw128(sa);
          const uint64_t db = g.b_mn ? make_desc_sw128_mnmajor(sb) : make_desc_sw128(sb);
          const uint32_t sta = g.a_mn ? 128u : 2u, stb = g.b_mn ? 128u : 2u;      // one UMMA_K: 2048 B of k-rows / 32 B inside the atom
          mma_bf16_ss(tmem + (uint32_t)(buf * kGmBN), da, db, idesc, kb != 0);
#pragma unroll
          for (int k = 1; k < kGmBK / 16; ++k) mma_bf16_ss_acc(tmem + (uint32_t)(buf * kGmBN), da + (uint64_t)(k * sta), db + (uint64_t)(k * stb), idesc);
          mma_commit(&tail->empty[st]);
        }
        __syncwarp();
        if (++st == kGmStages) { st = 0; ph ^= 1u; }
      }
      if (leader) mma_commit(&tail->acc_full[buf]);
      __syncwarp();
    }
  } else {
    const int qd = warp & 3, colq = warp >> 2;
    int i = 0;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++i) {
      const int buf = i & 1;
      const int b = t / (mt * nt), r = t % (mt * nt);
      const int m = (r / nt) * kGmBM + qd * 32 + lane;
      const int n0 = (r % nt) * kGmBN + colq * 32;
      const bool mok = m < g.M;
      if (nkb > 0) {
        mbar_wait(&tail->acc_full[buf], (i >> 1) & 1);
        tc_fence_after();
      }
      uint32_t va[32];
      if (nkb > 0) {
        tmem_ld_32(tmem + ((uint32_t)(qd * 32) << 16) + (uint32_t)(buf * kGmBN + colq * 32), va);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) va[j] = 0u;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0 && nkb > 0) mbar_arrive(&tail->acc_empty[buf]);
      const long long row = (long long)b * g.M + m;
      const int mw0 = (r / nt) * kGmBM + qd * 32;                  // first row of this warp's 32
      const int rows_valid = g.M - mw0;                            // <= 0: nothing of this warp's rows exists
      const long long roww0 = (long long)b * g.M + mw0;
      auto emit = [&](uint32_t (&v)[32], int nb) {
        if (nb >= g.N) return;
        // bias and colscale are read as float4 on the fast path: an offset view of either must take the per-element path
        const bool al16 = ((reinterpret_cast<uintptr_t>(g.C) | reinterpret_cast<uintptr_t>(g.pre) | reinterpret_cast<uintptr_t>(g.residual) |
                            reinterpret_cast<uintptr_t>(g.emul) | reinterpret_cast<uintptr_t>(g.part) | reinterpret_cast<uintptr_t>(g.bias) |
                            reinterpret_cast<uintptr_t>(g.colscale)) & 15) == 0;
        if (g.ksplit > 1) {
          float* dst = g.part + (((long long)ks * g.batch + b) * g.M + m) * g.N + nb;
          if ((g.N % 4 == 0) && nb + 32 <= g.N && al16) {         // warp-uniform: all lanes take the transposing store
            uint8_t* gb = reinterpret_cast<uint8_t*>(g.part + (((long long)ks * g.batch + b) * g.M + mw0) * g.N + nb);
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              uint4 c[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) c[j] = make_uint4(v[16 * hh + 4 * j], v[16 * hh + 4 * j + 1], v[16 * hh + 4 * j + 2], v[16 * hh + 4 * j + 3]);
              warp_rows_store64(stg, lane, c, gb + hh * 64, (long long)g.N * 4, rows_valid);
            }
          } else if (mok) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (nb + j < g.N) dst[j] = __uint_as_float(v[j]);
          }
          return;
        }
        float o[32];
        const bool fast = nb + 32 <= g.N && g.N % 8 == 0 && g.ldc % 8 == 0 && (!g.residual || g.ldr % 8 == 0) && al16;
        if (fast) {
          // whole 32-column chunk, 16-byte aligned rows (warp-uniform): per-column operands as 128-bit vectors, per-element
          // operands and results through the transposing 64-byte row moves
#pragma unroll
          for (int j = 0; j < 32; ++j) o[j] = __uint_as_float(v[j]) * g.alpha;
          if (g.bias) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 t = __ldg(reinterpret_cast<const float4*>(g.bias + nb) + j);
              o[4 * j] += t.x; o[4 * j + 1] += t.y; o[4 * j + 2] += t.z; o[4 * j + 3] += t.w;
            }
          }
          if (g.pre) {
            uint4 c[4];
            pack_bf16_16(o, c);
            warp_rows_store64(stg, lane, c, reinterpret_cast<uint8_t*>(g.pre + roww0 * g.ldc + nb), g.ldc * 2, rows_valid);
          }
          gemm_act32(o, g.act, g.c_bf16 != 0);
          if (g.emul) {
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              uint4 c[4];
              warp_rows_load64(stg, lane, c, reinterpret_cast<const uint8_t*>(g.emul + roww0 * g.N + nb) + hh * 64, (long long)g.N * 4, rows_valid);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                o[16 * hh + 4 * j] *= __uint_as_float(c[j].x); o[16 * hh + 4 * j + 1] *= __uint_as_float(c[j].y);
                o[16 * hh + 4 * j + 2] *= __uint_as_float(c[j].z); o[16 * hh + 4 * j + 3] *= __uint_as_float(c[j].w);
              }
            }
          }
          if (g.colscale) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 t = __ldg(reinterpret_cast<const float4*>(g.colscale + nb) + j);
              o[4 * j] *= t.x; o[4 * j + 1] *= t.y; o[4 * j + 2] *= t.z; o[4 * j + 3] *= t.w;
            }
          }
          if (g.residual) {
            if (g.res_bf16) {
              uint4 c[4];
              warp_rows_load64(stg, lane, c, reinterpret_cast<const uint8_t*>(reinterpret_cast<const bf16*>(g.residual) + roww0 * g.ldr + nb),
                               g.ldr * 2, rows_valid);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint4 t = c[j];
                o[8 * j] += bf16lo(t.x); o[8 * j + 1] += bf16hi(t.x); o[8 * j + 2] += bf16lo(t.y); o[8 * j + 3] += bf16hi(t.y);
                o[8 * j + 4] += bf16lo(t.z); o[8 * j + 5] += bf16hi(t.z); o[8 * j + 6] += bf16lo(t.w); o[8 * j + 7] += bf16hi(t.w);
              }
            } else {
#pragma unroll
              for (int hh = 0; hh < 2; ++hh) {
                uint4 c[4];
                warp_rows_load64(stg, lane, c, reinterpret_cast<const uint8_t*>(reinterpret_cast<const float*>(g.residual) + roww0 * g.ldr + nb) + hh * 64,
                                 g.ldr * 4, rows_valid);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  o[16 * hh + 4 * j] += __uint_as_float(c[j].x); o[16 * hh + 4 * j + 1] += __uint_as_float(c[j].y);
                  o[16 * hh + 4 * j + 2] += __uint_as_float(c[j].z); o[16 * hh + 4 * j + 3] += __uint_as_float(c[j].w);
                }
              }
            }
          }
          if (g.c_bf16) {
            uint4 c[4];
            pack_bf16_16(o, c);
            warp_rows_store64(stg, lane, c, reinterpret_cast<uint8_t*>(reinterpret_cast<bf16*>(g.C) + roww0 * g.ldc + nb), g.ldc * 2, rows_valid);
          } else {
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              uint4 c[4];
#pragma unroll
              for (int j = 0; j < 4; ++j)
                c[j] = make_uint4(__float_as_uint(o[16 * hh + 4 * j]), __float_as_uint(o[16 * hh + 4 * j + 1]), __float_as_uint(o[16 * hh + 4 * j + 2]),
                                  __float_as_uint(o[16 * hh + 4 * j + 3]));
              warp_rows_store64(stg, lane, c, reinterpret_cast<uint8_t*>(reinterpret_cast<float*>(g.C) + roww0 * g.ldc + nb) + hh * 64, g.ldc * 4,
                                rows_valid);
            }
          }
          return;
        }
        if (!mok) return;
        {                                                           // ragged / unaligned chunk: per-thread, per-element
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int n = nb + j;
            float x = __uint_as_float(v[j]) * g.alpha;
            if (n < g.N) {
              if (g.bias) x += __ldg(g.bias + n);
              if (g.pre) g.pre[row * g.ldc + n] = __float2bfloat16_rn(x);
            }
            o[j] = x;
          }
          gemm_act32(o, g.act, g.c_bf16 != 0);
          if (g.emul || g.colscale || g.residual) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int n = nb + j;
              if (n < g.N) {
                float x = o[j];
                if (g.emul) x *= g.emul[row * g.N + n];
                if (g.colscale) x *= __ldg(g.colscale + n);
                if (g.residual)
                  x += g.res_bf16 ? __bfloat162float(reinterpret_cast<const bf16*>(g.residual)[row * g.ldr + n])
                                  : reinterpret_cast<const float*>(g.residual)[row * g.ldr + n];
                o[j] = x;
              }
            }
          }
        }
        const bool full = nb + 32 <= g.N;
        if (g.c_bf16) {
          bf16* dst = reinterpret_cast<bf16*>(g.C) + row * g.ldc + nb;
          if (full && (g.ldc % 8 == 0) && ((reinterpret_cast<uintptr_t>(g.C) & 15) == 0)) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint32_t w[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                __nv_bfloat162 pk = __floats2bfloat162_rn(o[8 * j + 2 * q], o[8 * j + 2 * q + 1]);
                w[q] = *reinterpret_cast<uint32_t*>(&pk);
              }
              reinterpret_cast<uint4*>(dst)[j] = make_uint4(w[0], w[1], w[2], w[3]);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (nb + j < g.N) dst[j] = __float2bfloat16_rn(o[j]);
          }
        } else {
          float* dst = reinterpret_cast<float*>(g.C) + row * g.ldc + nb;
          if (full && (g.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.C) & 15) == 0)) {
#pragma unroll
            for (int j = 0; j < 8; ++j) reinterpret_cast<float4*>(dst)[j] = make_float4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (nb + j < g.N) dst[j] = o[j];
          }
        }
      };
      emit(va, n0);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kGmMmaWarp) tmem_dealloc(tmem, 256);
}

// split-K fold + epilogue: C = epi(sum_s part[s]) in ascending s
__global__ void __launch_bounds__(256) gemm_fold_kernel(GemmArgs g) {
  const long long total = (long long)g.batch * g.M * g.N;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i % g.N);
    const long long row = i / g.N;
    float x = 0.f;
    for (int s = 0; s < g.ksplit; ++s) x += g.part[(long long)s * total + i];
    x *= g.alpha;
    if (g.bias) x += g.bias[n];
    if (g.pre) g.pre[row * g.ldc + n] = __float2bfloat16_rn(x);
    x = gemm_act(x, g.act);
    if (g.emul) x *= g.emul[i];
    if (g.colscale) x *= g.colscale[n];
    if (g.residual)
      x += g.res_bf16 ? __bfloat162float(reinterpret_cast<const bf16*>(g.residual)[row * g.ldr + n])
                      : reinterpret_cast<const float*>(g.residual)[row * g.ldr + n];
    if (g.c_bf16) reinterpret_cast<bf16*>(g.C)[row * g.ldc + n] = __float2bfloat16_rn(x);
    else reinterpret_cast<float*>(g.C)[row * g.ldc + n] = x;
  }
}

static int gemm_ksplit(int M, int N, int K, int batch, int want) {
  const int tiles = ceil_div(M, kGmBM) * ceil_div(N, kGmBN) * batch, nkb = ceil_div(K, kGmBK);
  if (want > 0) return want > nkb ? nkb : want;
  if (tiles * 2 >= sm_count() || nkb < 8) return 1;           // enough tiles, or nothing to split
  int ks = sm_count() / tiles;
  if (ks > nkb / 4) ks = nkb / 4;
  if (ks > 32) ks = 32;
  return ks < 1 ? 1 : ks;
}

}  // namespace cor

using namespace cor;

extern "C" size_t cor_gemm_bf16_work_bytes(int M, int N, int K, int batch, int ksplit) {
  const int ks = gemm_ksplit(M, N, K, batch, ksplit);
  return ks > 1 ? (size_t)ks * batch * M * N * sizeof(float) + 16 : 16;
}

extern "C" int cor_gemm_bf16(const void* A, int a_mn, long long a_rows_total, long long a_batch_rows, const void* B, int b_mn,
                             long long b_rows_total, long long b_batch_rows, int M, int N, int K, int batch, float alpha, const float* bias,
                             int act, const float* emul, const float* colscale, const void* residual, int res_dtype, long long ldr, void* C, int c_dtype,
                             long long ldc, void* pre_bf16, int ksplit, void* work, cor_stream_t stream) {
  COR_REQUIRE(A && B && C, "cor_gemm_bf16: null pointer");
  COR_REQUIRE(M > 0 && N > 0 && K > 0 && batch > 0, "cor_gemm_bf16: bad shape M=%d N=%d K=%d batch=%d", M, N, K, batch);
  COR_REQUIRE(c_dtype == COR_F32 || c_dtype == COR_BF16, "cor_gemm_bf16: output dtype %d", c_dtype);
  COR_REQUIRE(!residual || res_dtype == COR_F32 || res_dtype == COR_BF16, "cor_gemm_bf16: residual dtype %d", res_dtype);
  COR_REQUIRE(act >= COR_ACT_NONE && act <= COR_ACT_SIGMOID, "cor_gemm_bf16: act %d", act);
  // tensor maps: K-major [rows_total][K] with a 64(k) x 128(rows) box; MN-major [rows_total = batch*K][rows] with a 64(rows) x 64(k) box
  CUtensorMap tmA, tmB;
  int rc = a_mn ? umma::encode_tmap_bf16_2d(&tmA, A, (uint64_t)a_rows_total, (uint64_t)M, 64, 64)
                : umma::encode_tmap_bf16_2d(&tmA, A, (uint64_t)a_rows_total, (uint64_t)K, kGmBM, kGmBK);
  if (rc) return rc;
  rc = b_mn ? umma::encode_tmap_bf16_2d(&tmB, B, (uint64_t)b_rows_total, (uint64_t)N, 64, 64)
            : umma::encode_tmap_bf16_2d(&tmB, B, (uint64_t)b_rows_total, (uint64_t)K, kGmBN, kGmBK);
  if (rc) return rc;
  // a batched MN-major operand must not let a k-block run into the next batch entry's rows
  COR_REQUIRE(batch == 1 || ((!a_mn || a_batch_rows == 0 || K % kGmBK == 0) && (!b_mn || b_batch_rows == 0 || K % kGmBK == 0)),
              "cor_gemm_bf16: batched MN-major operands need K %% 64 == 0 (K=%d)", K);
  GemmArgs g;
  g.M = M; g.N = N; g.K = K; g.batch = batch; g.a_mn = a_mn; g.b_mn = b_mn;
  g.a_batch_rows = a_batch_rows; g.b_batch_rows = b_batch_rows;
  g.ksplit = gemm_ksplit(M, N, K, batch, ksplit);
  g.alpha = alpha; g.bias = bias; g.emul = emul; g.colscale = colscale; g.residual = residual; g.res_bf16 = res_dtype == COR_BF16; g.ldr = ldr;
  g.act = act; g.C = C; g.c_bf16 = c_dtype == COR_BF16; g.ldc = ldc; g.pre = reinterpret_cast<bf16*>(pre_bf16);
  g.part = reinterpret_cast<float*>(work);
  COR_REQUIRE(g.ksplit == 1 || work, "cor_gemm_bf16: split-K needs a work buffer");
  const int tiles = ceil_div(M, kGmBM) * ceil_div(N, kGmBN) * batch;
  int gx = sm_count() / g.ksplit;
  if (gx < 1) gx = 1;
  if (gx > tiles) gx = tiles;
  const size_t smem = (size_t)kGmStages * 2 * kGmTile + sizeof(GemmSmemTail) + 16 + (size_t)kGmEpiWarps * kGmStgBytes + 1024;
  COR_CUDA(cudaFuncSetAttribute(gemm_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaStream_t st = as_stream(stream);
  gemm_umma_kernel<<<dim3(gx, g.ksplit), kGmThreads, smem, st>>>(tmA, tmB, g);
  rc = check_launch("gemm_umma_kernel");
  if (rc || g.ksplit == 1) return rc;
  const long long total = (long long)batch * M * N;
  const int blocks = (int)((total + 255) / 256 < (long long)sm_count() * 8 ? (total + 255) / 256 : (long long)sm_count() * 8);
  gemm_fold_kernel<<<blocks, 256, 0, st>>>(g);
  return check_launch("gemm_fold_kernel");
}
