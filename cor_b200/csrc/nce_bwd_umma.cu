// InfoNCE backward for MANY queries, entirely on tcgen05 tensor cores (Class N; no reference implementation):
//
//   P[q, r]  = (exp(S[q,r]/tau - lse[q]) - [r == target(q)]) * g / (tau * Nq),    S = Q R^T
//   dQ = P R            dR = P^T Q
//
// Neither S nor P ever exists in global memory.  ONE kernel serves both products, with the roles of the operands
// swapped (mode 0: X = queries, Y = regions, G = dQ;  mode 1: X = regions, Y = queries, G = dR):
//
//   a CTA keeps 128 X rows resident in tensor memory and walks Y tiles of 64 rows through shared memory:
//     GEMM 1   S^(X)[128 x 64] = X Y^T             A = X (TMEM: row x in lane x, two bf16 per column, stored once by
//              the epilogue threads)                B = Y tile (K-major, TMA, SW128)
//     epilogue the thread that owns TMEM lane x turns its S row into bf16 coefficients and stores them into
//              shared memory in the canonical K-major SW128 layout (manual swizzle) -> A operand of GEMM 2
//     GEMM 2   G[128 x D] += P[128 x 64] Y          A = P (K-major, K = Y rows)      B = THE SAME Y TILE, read
//              as an MN-major operand (its [y][d] rows are K = y, N = d with d contiguous; SW128 atoms are the
//              8-row x 128-byte groups TMA wrote; LBO = distance between 64-wide d blocks, SBO = 1024 B)
//   so every Y byte fetched from L2 feeds both GEMMs.  A Y tile stays in shared memory from its load to the end of its
//   GEMM 2, i.e. through a whole TMA -> GEMM 1 -> epilogue -> GEMM 2 round trip: the tiles are kept SMALL (64 rows, 32 KB
//   at D = 256) and up to four of them are in flight -- with two 128-row slots the next load could only start when a GEMM 2
//   finished and the tensor pipe idled through every load latency (measured 5 700 cycles per 128 rows against 2 048 of
//   tensor work).  TMEM: S double-buffered (2 x 64 columns), X in D/2 columns from 128, G in 256 columns; P double-buffered
//   in shared memory.
//
// Warp roles (320 threads): 0..7 = epilogue (warp w owns TMEM lane quarter w % 4 and column half w / 4, i.e. exactly one
// 128-byte row of one P k-block per thread), 8 = TMA producer, 9 = TMEM owner + MMA issuer (highest warp ids: the
// issue arbiter favours them, see sim_umma.cu).  The producer prefetches Y tiles into L2 ahead of the stage loads.
// Split over Y (gridDim.x) leaves fp32 partials [split][Nx][D] that a fixed-order fold sums (deterministic).
// Logit-scale gradient (mode 0 only): the epilogue thread of query row x also keeps sum_y (P/gscale)[x][y] S[x][y] in a
// register across its Y tiles and leaves one partial per (split, column half, query); nce_scale_fold_kernel sums them.
// Region memory (mode 0, cor_memory_dq): Y = the memory's bank, its row count read on the device (count), no targets (a
// memory row is never a positive); both folds ADD into the gradients the current rows' backward already wrote.
#include <stdlib.h>

#include "umma.cuh"

namespace cor {

using namespace umma;

constexpr int kNbM = 128;                  // X rows per CTA (UMMA M)
constexpr int kNbN = 64;                   // Y rows per tile (GEMM 1 N, GEMM 2 K)
constexpr int kNbBK = 64;
constexpr int kNbBlk = kNbM * kNbBK * 2;   // 16 KB: one P buffer [128 x 64]
constexpr int kNbYBlk = kNbN * kNbBK * 2;  // 8 KB: one 64-wide k-block of a Y tile
constexpr int kNbMaxSlots = 4;
constexpr int kNbTmaWarp = 8, kNbMmaWarp = 9;
constexpr int kNbPrefetch = 3;

struct NceSmemTail {
  uint64_t xfull, yfull[kNbMaxSlots], yempty[kNbMaxSlots], s_full[2], s_empty[2], p_full[2], p_empty[2], g_full;
  uint32_t tmem_base;
};

struct NceArgs {
  int Nx, Ny, Nq, nkb, nslots, mode;       // mode 0: X = queries (G = dQ), 1: X = regions (G = dR)
  float c2;                                // log2(e) / tau
  float gmul;                              // g_mul / (tau * Nq); multiplied by g_loss[0] on the device
  float g_mul;
  const float* scale;                      // device logit scale replacing 1/tau in c2 and gmul, or NULL
  float* lspart;                           // mode 0: [gridDim.x][2][Nq] logit-scale gradient partials, or NULL
  const float* lse;                        // [Nq]
  const long long* targets;                // [Nq] region index of each query's positive, or NULL (no positives)
  const int* count;                        // device row count: Y rows past min(Ny, *count) are not scored; or NULL
  const float* g_loss;                     // [1]
  float* out;                              // [gridDim.x][Nx][D] partials (or the result itself when gridDim.x == 1); NULL = not written
  const bf16* X;                           // [Nx][D]: the epilogue threads store the CTA's rows into TMEM
};

// instruction descriptor with an MN-major B operand (bit 16)
__host__ __device__ constexpr uint32_t make_idesc_bf16_bmn(int M, int N) { return make_idesc_bf16(M, N) | (1u << 16); }

// MN-major SW128 operand: 64 MN-elements (128 B) x 8 K-rows per swizzle atom; LBO = byte distance between consecutive
// 64-element blocks along MN, SBO = byte distance between consecutive 8-row groups along K (cute::UMMA::make_umma_desc<MN>:
// ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units).
__device__ __forceinline__ uint64_t make_desc_sw128_mn(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

__device__ __forceinline__ uint32_t pack_bf16x2_rn(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

__global__ void __launch_bounds__(320, 1) nce_bwd_umma_kernel(const __grid_constant__ CUtensorMap tmY, NceArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* base = reinterpret_cast<uint8_t*>(((uintptr_t)smem + 1023) & ~(uintptr_t)1023);
  uint8_t* y_smem = base;                                                    // nslots x nkb x 8 KB
  uint8_t* p_smem = y_smem + (size_t)a.nslots * a.nkb * kNbYBlk;             // 2 buffers x 16 KB
  NceSmemTail* tail = reinterpret_cast<NceSmemTail*>(p_smem + 2 * kNbBlk);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int x0 = blockIdx.y * kNbM;
  const int Ny = a.count ? min(a.Ny, max(*a.count, 0)) : a.Ny;
  const int ntiles = (Ny + kNbN - 1) / kNbN;
  const int D = a.nkb * kNbBK;
  const int n_my = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;      // tiles blockIdx.x, +gridDim.x, ...

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmY);
    mbar_init(&tail->xfull, 4);
    for (int i = 0; i < a.nslots; ++i) { mbar_init(&tail->yfull[i], 1); mbar_init(&tail->yempty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tail->s_full[i], 1); mbar_init(&tail->s_empty[i], 8); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tail->p_full[i], 8); mbar_init(&tail->p_empty[i], 1); }
    mbar_init(&tail->g_full, 1);
    fence_barrier_init();
  }
  if (warp == kNbMmaWarp) tmem_alloc(&tail->tmem_base, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tail->tmem_base;
  const uint32_t tmem_g = tmem + 256u;
  const uint32_t tmem_x = tmem + 128u;             // X rows in lanes, D/2 packed-bf16 columns [128, 128 + D/2)

  if (warp == kNbTmaWarp) {
    if (lane == 0) {
      for (int i = 0; i < n_my && i < kNbPrefetch; ++i)
        for (int kb = 0; kb < a.nkb; ++kb) tma_prefetch_2d(&tmY, kb * kNbBK, ((int)blockIdx.x + i * (int)gridDim.x) * kNbN);
      for (int i = 0; i < n_my; ++i) {
        const int t = blockIdx.x + i * gridDim.x;
        if (i + kNbPrefetch < n_my)
          for (int kb = 0; kb < a.nkb; ++kb) tma_prefetch_2d(&tmY, kb * kNbBK, (t + kNbPrefetch * (int)gridDim.x) * kNbN);
        const int slot = i % a.nslots;
        mbar_wait(&tail->yempty[slot], ((i / a.nslots) & 1) ^ 1);
        mbar_expect_tx(&tail->yfull[slot], (uint32_t)(a.nkb * kNbYBlk));
        for (int kb = 0; kb < a.nkb; ++kb)
          tma_load_2d(y_smem + (size_t)(slot * a.nkb + kb) * kNbYBlk, &tmY, &tail->yfull[slot], kb * kNbBK, t * kNbN, kEvictLast);
      }
    }
  } else if (warp == kNbMmaWarp) {
    // the whole warp walks the loop, one elected lane issues (descriptors stay in uniform registers; see sim_umma.cu)
    if (n_my > 0) {
      const bool leader = elect_one();
      const uint32_t idesc1 = make_idesc_bf16(kNbM, kNbN);
      const uint32_t idesc2 = make_idesc_bf16_bmn(kNbM, D);
      const uint32_t y_base = smem_u32(y_smem), p_base = smem_u32(p_smem);
      mbar_wait(&tail->xfull, 0);
      tc_fence_after();
      auto gemm1 = [&](int i) {
        const int slot = i % a.nslots, buf = i & 1;
        mbar_wait(&tail->yfull[slot], (i / a.nslots) & 1);
        mbar_wait(&tail->s_empty[buf], ((i >> 1) & 1) ^ 1);
        tc_fence_after();
        if (leader) {
          for (int kb = 0; kb < a.nkb; ++kb) {
            const uint64_t db = make_desc_sw128(y_base + (uint32_t)((slot * a.nkb + kb) * kNbYBlk));
            // A from TMEM: 16 k-elements = 8 packed columns per MMA; only the Y tile is fetched from shared memory (with both
            // operands there the 64 KB X tile was re-read for every 64-row Y tile: 144 KB of operand fetch per tile against
            // ~1 000 tensor cycles, i.e. shared-memory bandwidth, not the tensor pipe, paced the loop)
#pragma unroll
            for (int k = 0; k < kNbBK / 16; ++k)
              mma_bf16_ts(tmem + (uint32_t)(buf * kNbN), tmem_x + (uint32_t)(kb * (kNbBK / 2) + k * 8), db + 2 * k, idesc1, (kb | k) != 0);
          }
          mma_commit(&tail->s_full[buf]);
        }
        __syncwarp();
      };
      gemm1(0);
      if (n_my > 1) gemm1(1);
      for (int i = 0; i < n_my; ++i) {
        if (i + 2 < n_my) gemm1(i + 2);            // needs only the S buffer of tile i, which the epilogue frees early
        const int slot = i % a.nslots, pb = i & 1;
        mbar_wait(&tail->p_full[pb], (i >> 1) & 1);
        tc_fence_after();
        if (leader) {
          // B = the Y tile as an MN-major operand: N = d (nkb blocks of 64, kNbYBlk apart), K = y rows (8-row groups 1024 B apart)
          const uint64_t db0 = make_desc_sw128_mn(y_base + (uint32_t)(slot * a.nkb * kNbYBlk), kNbYBlk, 1024);
          const uint64_t dp0 = make_desc_sw128(p_base + (uint32_t)(pb * kNbBlk));
          mma_bf16_ss(tmem_g, dp0, db0, idesc2, i != 0);
#pragma unroll
          for (int j = 1; j < kNbN / 16; ++j)       // 16 y rows = 2048 B = 128 x 16 B
            mma_bf16_ss_acc(tmem_g, dp0 + 2 * j, db0 + (uint64_t)(j * 128), idesc2);
          mma_commit(&tail->p_empty[pb]);
          mma_commit(&tail->yempty[slot]);
        }
        __syncwarp();
      }
      if (leader) mma_commit(&tail->g_full);
      __syncwarp();
    }
  } else {
    const int e = warp;
    const int qd = warp & 3;                       // TMEM lane quarter this warp may read
    const int half = e >> 2;                       // which 64 columns of the S tile / which half of G's columns
    const int row = qd * 32 + lane;
    const int xg = x0 + row;
    const bool xok = xg < a.Nx;
    // ---- this thread's X row -> TMEM (its own lane), two bf16 per 32-bit column; the four warps of column half 0 cover the
    // 128 lanes ----
    if (half == 0) {
      const uint32_t* src = reinterpret_cast<const uint32_t*>(a.X + (long long)xg * D);
      for (int c = 0; c < D / 2; c += 32) {
        uint32_t v[32];
        if (xok) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint4 u = __ldg(reinterpret_cast<const uint4*>(src + c) + j);
            v[4 * j] = u.x; v[4 * j + 1] = u.y; v[4 * j + 2] = u.z; v[4 * j + 3] = u.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;
        }
        tmem_st_32(tmem_x + ((uint32_t)(qd * 32) << 16) + (uint32_t)c, v);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tail->xfull);
    }
    const float log2e = 1.4426950408889634f;
    float c2 = a.c2, gmul = a.gmul;
    if (a.scale) {
      const float s = __ldg(a.scale);
      c2 = s * log2e;
      gmul = a.g_mul * s / (float)a.Nq;
    }
    const float gscale = a.g_loss[0] * gmul;
    float ls = 0.f;                                 // mode 0 with lspart: sum over this thread's S columns of coef * S
    float my_nl = 0.f;                              // mode 0: -lse[q] log2e of this thread's query
    int my_tg = -1;
    if (a.mode == 0 && xok) {
      my_nl = -a.lse[xg] * log2e;
      my_tg = a.targets ? (int)a.targets[xg] : -1;
    }
    for (int i = 0; i < n_my; ++i) {
      const int t = blockIdx.x + i * gridDim.x;
      const int buf = i & 1;
      const int y0 = t * kNbN + half * 32;          // first Y row (S column) this thread handles
      // mode 1: the columns are queries -- lane l fetches the constants of column y0 + l, shuffled out below
      float nl_a = 0.f;
      int tg_a = -1;
      if (a.mode == 1) {
        const int qa = y0 + lane;
        nl_a = qa < a.Nq ? -__ldg(a.lse + qa) * log2e : -INFINITY;      // exp2(-inf) = 0: columns past Nq contribute nothing
        tg_a = qa < a.Nq ? (int)__ldg(a.targets + qa) : -1;
      }
      mbar_wait(&tail->s_full[buf], (i >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem + ((uint32_t)(qd * 32) << 16) + (uint32_t)(buf * kNbN + half * 32);
      uint32_t va[32];
      tmem_ld_32(taddr, va);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tail->s_empty[buf]);          // S is in registers: GEMM 1 of tile i+2 may overwrite the buffer
      uint32_t w[16];                                            // 32 bf16 coefficients = this thread's half of a 128-byte P row
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        float n0, n1;
        int hit0, hit1;
        if (a.mode == 0) {
          // columns past Ny get no coefficient (exp2(-inf) = 0): a memory's stale rows in its last tile add nothing
          n0 = y0 + 2 * j < Ny ? my_nl : -INFINITY;
          n1 = y0 + 2 * j + 1 < Ny ? my_nl : -INFINITY;
          hit0 = (y0 + 2 * j == my_tg);
          hit1 = (y0 + 2 * j + 1 == my_tg);
        } else {
          n0 = __shfl_sync(0xffffffffu, nl_a, 2 * j);
          n1 = __shfl_sync(0xffffffffu, nl_a, 2 * j + 1);
          hit0 = (__shfl_sync(0xffffffffu, tg_a, 2 * j) == xg);
          hit1 = (__shfl_sync(0xffffffffu, tg_a, 2 * j + 1) == xg);
        }
        float c0 = ex2_approx(fmaf(__uint_as_float(va[2 * j]), c2, n0));
        float c1 = ex2_approx(fmaf(__uint_as_float(va[2 * j + 1]), c2, n1));
        if (hit0) c0 -= 1.f;
        if (hit1) c1 -= 1.f;
        if (a.lspart) {                             // columns past Ny have a zero coefficient: they add nothing
          ls = fmaf(c0, __uint_as_float(va[2 * j]), ls);
          ls = fmaf(c1, __uint_as_float(va[2 * j + 1]), ls);
        }
        w[j] = pack_bf16x2_rn(c0 * gscale, c1 * gscale);
      }
      // P row -> shared memory, K-major SW128: 16-byte chunk c of row r at c ^ (r & 7); this thread owns chunks half*4 .. +3
      const int pb = i & 1;
      mbar_wait(&tail->p_empty[pb], ((i >> 1) & 1) ^ 1);        // GEMM 2 of tile i-2 has consumed this buffer
      uint8_t* prow = p_smem + pb * kNbBlk + row * 128;
#pragma unroll
      for (int c = 0; c < 4; ++c)
        *reinterpret_cast<uint4*>(prow + (((half * 4 + c) ^ (row & 7)) << 4)) = make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
      fence_proxy_async();                                        // generic-proxy stores -> visible to the tensor core's async proxy
      __syncwarp();
      if (lane == 0) mbar_arrive(&tail->p_full[pb]);
    }
    if (a.lspart && a.mode == 0 && xok) a.lspart[((long long)blockIdx.x * 2 + half) * a.Nq + xg] = ls;
    // ---- drain G: this thread's X row, columns [half * D/2, +D/2) ----
    if (n_my > 0) {
      mbar_wait(&tail->g_full, 0);
      tc_fence_after();
      const int ncol = D / 2;
      float* dst = a.out + ((long long)blockIdx.x * a.Nx + xg) * D + half * ncol;
      for (int c = 0; c < ncol; c += 32) {
        uint32_t v[32];
        tmem_ld_32(tmem_g + ((uint32_t)(qd * 32) << 16) + (uint32_t)(half * ncol + c), v);
        tmem_ld_wait();
        if (xok && a.out) {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            reinterpret_cast<float4*>(dst + c)[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                                                __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        }
      }
    } else if (xok && a.out) {                    // a split with no Y tile (a memory filled below the grid): zero partials
      float* dst = a.out + ((long long)blockIdx.x * a.Nx + xg) * D + half * (D / 2);
      for (int c = 0; c < D / 2; c += 4) *reinterpret_cast<float4*>(dst + c) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kNbMmaWarp) tmem_dealloc(tmem, 512);
}

// out[x][d] = sum over splits (ascending) of part[s][x][d]; accumulate: out[x][d] += that sum
__global__ void __launch_bounds__(256) nce_fold_kernel(const float4* __restrict__ part, float4* __restrict__ out, long long vecs, int nsplit,
                                                       int accumulate) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < vecs; i += (long long)gridDim.x * blockDim.x) {
    float4 acc = part[i];
    for (int s = 1; s < nsplit; ++s) {
      const float4 v = part[(long long)s * vecs + i];
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    if (accumulate) {
      const float4 o = out[i];
      acc.x = o.x + acc.x; acc.y = o.y + acc.y; acc.z = o.z + acc.z; acc.w = o.w + acc.w;
    }
    out[i] = acc;
  }
}

// *g_scale = g_loss[0] * g_mul / Nq * sum_q sum_p lspart[p][q]: one CTA, partials in order per query, queries in a fixed tree.
// accumulate: *g_scale += that value
__global__ void __launch_bounds__(256) nce_scale_fold_kernel(const float* __restrict__ lspart, int nparts, int Nq, const float* __restrict__ g_loss,
                                                             float g_mul, float* __restrict__ g_scale, int accumulate) {
  __shared__ float red[256];
  float v = 0.f;
  for (int q = threadIdx.x; q < Nq; q += 256) {
    float s = 0.f;
    for (int p = 0; p < nparts; ++p) s += lspart[(long long)p * Nq + q];
    v += s;
  }
  red[threadIdx.x] = v;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const float v = red[0] * (g_loss[0] * g_mul / (float)Nq);
    g_scale[0] = accumulate ? g_scale[0] + v : v;
  }
}

static int nce_splits(int xtiles, int ytiles) {
  int s = sm_count() / xtiles;
  if (s < 1) s = 1;
  if (s > ytiles) s = ytiles;
  return s;
}

// out == NULL (mode 0): only the logit-scale partials are wanted -- the dQ GEMM still runs, its result is not stored.
// count: device row count of Y (see NceArgs); accumulate: the fold adds into `out` (then the partials always go to `part`)
static int nce_launch(const void* X, const void* Y, int Nx, int Ny, int Nq, int D, int mode, float inv_tau, const float* scale,
                      const float* lse, const long long* targets, const float* g_loss, float g_mul, float* out, float* part,
                      float* lspart, cudaStream_t st, const int* count = nullptr, int accumulate = 0) {
  const int nkb = D / kNbBK;
  const int xtiles = ceil_div(Nx, kNbM), ytiles = ceil_div(Ny, kNbN);
  const int nsplit = nce_splits(xtiles, ytiles);
  COR_REQUIRE(((uintptr_t)X & 15) == 0, "cor_infonce_bwd_umma: X rows are read as 16-byte vectors: X must be 16-byte aligned");
  CUtensorMap tmY;
  int rc = encode_tmap_bf16_2d(&tmY, Y, (uint64_t)Ny, (uint64_t)D, kNbN, kNbBK);
  if (rc) return rc;
  // shared memory: 2 P buffers + as many whole-Y-tile slots as fit, at most kNbMaxSlots
  const size_t fixed = (size_t)2 * kNbBlk + sizeof(NceSmemTail) + 1024;
  int nslots = (int)((227 * 1024 - fixed) / ((size_t)nkb * kNbYBlk));
  if (nslots > kNbMaxSlots) nslots = kNbMaxSlots;
  COR_REQUIRE(nslots >= 2, "cor_infonce_bwd_umma: shared memory budget (D=%d)", D);
  const size_t smem = fixed + (size_t)nslots * nkb * kNbYBlk;
  COR_CUDA(cudaFuncSetAttribute(nce_bwd_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  NceArgs a;
  a.Nx = Nx; a.Ny = Ny; a.Nq = Nq; a.nkb = nkb; a.nslots = nslots; a.mode = mode;
  a.c2 = inv_tau * 1.4426950408889634f;
  a.gmul = g_mul * inv_tau / (float)Nq;
  a.g_mul = g_mul; a.scale = scale; a.lspart = lspart;
  a.lse = lse; a.targets = targets; a.count = count; a.g_loss = g_loss;
  a.X = reinterpret_cast<const bf16*>(X);
  const bool direct = nsplit == 1 && !accumulate;
  a.out = !out ? nullptr : (direct ? out : part);
  nce_bwd_umma_kernel<<<dim3(nsplit, xtiles), 320, smem, st>>>(tmY, a);
  rc = check_launch("nce_bwd_umma_kernel");
  if (rc || direct || !out) return rc;
  const long long vecs = (long long)Nx * D / 4;
  const int blocks = (int)((vecs + 255) / 256 < (long long)sm_count() * 4 ? (vecs + 255) / 256 : (long long)sm_count() * 4);
  nce_fold_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(part), reinterpret_cast<float4*>(out), vecs, nsplit, accumulate);
  return check_launch("nce_fold_kernel");
}

}  // namespace cor

using namespace cor;

// the two launches' partials (nce_launch: X tiles of kNbM rows, Y tiles of kNbN rows), one after the other in the same buffer,
// then the logit-scale partials of the dQ launch [splits][2][Nq]
static size_t nce_part_bytes(int Nq, int Nr, int D) {
  const size_t sq = (size_t)nce_splits(ceil_div(Nq, kNbM), ceil_div(Nr, kNbN)) * Nq * D * sizeof(float);      // mode 0: X = queries
  const size_t sr = (size_t)nce_splits(ceil_div(Nr, kNbM), ceil_div(Nq, kNbN)) * Nr * D * sizeof(float);      // mode 1: X = regions
  return ((sq > sr ? sq : sr) + 255) / 256 * 256;
}

extern "C" size_t cor_infonce_bwd_umma_work_bytes(int Nq, int Nr, int D) {
  const size_t ls = (size_t)nce_splits(ceil_div(Nq, kNbM), ceil_div(Nr, kNbN)) * 2 * Nq * sizeof(float);
  return nce_part_bytes(Nq, Nr, D) + ls + 256;
}

static int infonce_bwd_umma(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, const float* scale,
                            const float* lse, const long long* targets, const float* g_loss, float g_mul, float* g_regions,
                            float* g_queries, float* g_scale, void* work, cor_stream_t stream) {
  COR_REQUIRE(regions && queries && lse && targets && g_loss && work, "cor_infonce_bwd_umma: null pointer");
  COR_REQUIRE(Nr > 0 && Nq > 0 && D % kNbBK == 0 && D >= kNbBK && D <= 256, "cor_infonce_bwd_umma: need D in {64,128,192,256} (D=%d)", D);
  COR_REQUIRE(g_regions || g_queries || g_scale, "cor_infonce_bwd_umma: nothing to compute");
  cudaStream_t st = as_stream(stream);
  float* part = reinterpret_cast<float*>(work);
  float* lspart = g_scale ? reinterpret_cast<float*>(reinterpret_cast<char*>(work) + nce_part_bytes(Nq, Nr, D)) : nullptr;
  int rc = COR_OK;
  if (g_queries || g_scale)
    rc = nce_launch(queries, regions, Nq, Nr, Nq, D, 0, inv_tau, scale, lse, targets, g_loss, g_mul, g_queries, part, lspart, st);
  if (rc) return rc;
  if (g_scale) {
    const int nparts = 2 * nce_splits(ceil_div(Nq, kNbM), ceil_div(Nr, kNbN));
    nce_scale_fold_kernel<<<1, 256, 0, st>>>(lspart, nparts, Nq, g_loss, g_mul, g_scale, 0);
    rc = check_launch("nce_scale_fold_kernel");
    if (rc) return rc;
  }
  if (g_regions)
    rc = nce_launch(regions, queries, Nr, Nq, Nq, D, 1, inv_tau, scale, lse, targets, g_loss, g_mul, g_regions, part, nullptr, st);
  return rc;
}

extern "C" int cor_infonce_bwd_umma(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, const float* lse,
                                    const long long* targets, const float* g_loss, float g_mul, float* g_regions, float* g_queries,
                                    void* work, cor_stream_t stream) {
  return infonce_bwd_umma(regions, queries, Nr, Nq, D, inv_tau, nullptr, lse, targets, g_loss, g_mul, g_regions, g_queries, nullptr, work,
                          stream);
}

extern "C" int cor_infonce_bwd_umma_ls(const void* regions, const void* queries, int Nr, int Nq, int D, const float* logit_scale,
                                       const float* lse, const long long* targets, const float* g_loss, float g_mul, float* g_regions,
                                       float* g_queries, float* g_logit_scale, void* work, cor_stream_t stream) {
  COR_REQUIRE(logit_scale, "cor_infonce_bwd_umma_ls: null logit_scale");
  return infonce_bwd_umma(regions, queries, Nr, Nq, D, 0.f, logit_scale, lse, targets, g_loss, g_mul, g_regions, g_queries, g_logit_scale,
                          work, stream);
}

// ---- region memory: the queries' gradient through the memory rows (Y = the bank, no positives), added in ----
static int mem_dq_splits(int Nq, int K) { return nce_splits(ceil_div(Nq, kNbM), ceil_div(K, kNbN)); }

static size_t mem_dq_part_bytes(int Nq, int K, int D) {
  return ((size_t)mem_dq_splits(Nq, K) * Nq * D * sizeof(float) + 255) / 256 * 256;
}

extern "C" size_t cor_memory_dq_work_bytes(int Nq, int K, int D) {
  if (Nq <= 0 || K <= 0 || D <= 0) return 0;
  return mem_dq_part_bytes(Nq, K, D) + (size_t)mem_dq_splits(Nq, K) * 2 * Nq * sizeof(float) + 256;
}

extern "C" int cor_memory_dq(const void* bank, int K, const int* state, const void* queries, int Nq, int D, float inv_tau,
                             const float* logit_scale, const float* lse, const float* g_loss, float g_mul, float* g_queries,
                             float* g_logit_scale, void* work, cor_stream_t stream) {
  COR_REQUIRE(bank && state && queries && lse && g_loss && work, "cor_memory_dq: null pointer");
  COR_REQUIRE(K >= 1 && Nq >= 1, "cor_memory_dq: need K >= 1 and Nq >= 1 (K=%d Nq=%d)", K, Nq);
  COR_REQUIRE(D % kNbBK == 0 && D >= kNbBK && D <= 256, "cor_memory_dq: need D in {64,128,192,256} (D=%d)", D);
  COR_REQUIRE(g_queries || g_logit_scale, "cor_memory_dq: nothing to compute");
  COR_REQUIRE(!g_logit_scale || logit_scale, "cor_memory_dq: g_logit_scale needs logit_scale");
  cudaStream_t st = as_stream(stream);
  float* part = reinterpret_cast<float*>(work);
  float* lspart = g_logit_scale ? reinterpret_cast<float*>(reinterpret_cast<char*>(work) + mem_dq_part_bytes(Nq, K, D)) : nullptr;
  int rc = nce_launch(queries, bank, Nq, K, Nq, D, 0, inv_tau, logit_scale, lse, nullptr, g_loss, g_mul, g_queries, part, lspart, st,
                      state + 1, 1);
  if (rc || !g_logit_scale) return rc;
  nce_scale_fold_kernel<<<1, 256, 0, st>>>(lspart, 2 * mem_dq_splits(Nq, K), Nq, g_loss, g_mul, g_logit_scale, 1);
  return check_launch("nce_scale_fold_kernel");
}
