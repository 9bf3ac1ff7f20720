// Region x query similarity + online log-sum-exp (InfoNCE forward), "TS" form: the QUERY operand lives in TENSOR
// MEMORY, only the region tiles stream through shared memory.
//
// Why: with both operands in shared memory (sim_umma.cu) a 128 x 128 x 16 tcgen05.mma reads 8 KB of shared memory per
// 64 tensor-pipe cycles -- 128 B/clk, the whole shared-memory bandwidth of an SM -- and the TMA fills of the region
// ring come on top, so the tensor pipe never gets past ~60 % (trace build: ~830 cycles per k-block of 8 MMAs that the
// pipe executes in 512).  Queries are constant for a CTA's lifetime: each epilogue thread writes ITS query row into TMEM
// once (tcgen05.st, packed bf16 pairs, 128 columns for D = 256) and every MMA then takes A from TMEM and only B from
// shared memory: 64 B/clk + the fills.  That also frees the 128 KB the resident queries occupied: the region ring
// grows to 14 stages (3.5 tiles of look-ahead).
//
// TMEM (512 columns): accumulators of the two 128-query halves [0,128) [128,256) -- single-buffered per half, the halves
// ping-pong (the epilogue of half 0 runs under the MMAs of half 1 and vice versa) -- and the queries [256, 256 + D).
// With <= 128 queries there is one half and its accumulator alternates between the two slots tile by tile.
// Warp roles (320 threads): 0..7 epilogue (lane quarter w % 4, half w / 4), 8 TMA producer, 9 TMEM owner + MMA issuer.
// LSE partials in the work buffer as [qtile][gridDim.x][256][2], the layout sim_lse_combine_kernel and cor_infonce_tail read.
#include <stdlib.h>

#include "umma.cuh"

namespace cor {

using namespace umma;

constexpr int kTsHalf = 128, kTsBM = 256, kTsBN = 128, kTsBK = 64;
constexpr int kTsBBytes = kTsBN * kTsBK * 2;     // 16 KB: one stage of regions
constexpr int kTsMaxStages = 14;
constexpr int kTsTmaWarp = 8, kTsMmaWarp = 9;
#ifndef COR_SIM_TS_POLY_OF4
#define COR_SIM_TS_POLY_OF4 0          // of every 4 element pairs, how many take the FMA-pipe exp2 instead of MUFU (A/B knob)
#endif

struct TsSmemTail {
  uint64_t afull, full[kTsMaxStages], empty[kTsMaxStages], acc_full[2], acc_empty[2];
  uint32_t tmem_base;
};

__global__ void __launch_bounds__(320, 1) sim_umma_ts_kernel(const __grid_constant__ CUtensorMap tmR, const bf16* __restrict__ queries, int Nr,
                                                             int Nq, int nkb, int nstages, float inv_tau, const float* __restrict__ scale,
                                                             float* __restrict__ part, const int* __restrict__ count) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* base = reinterpret_cast<uint8_t*>(((uintptr_t)smem + 1023) & ~(uintptr_t)1023);
  uint8_t* r_smem = base;
  TsSmemTail* tail = reinterpret_cast<TsSmemTail*>(r_smem + (size_t)nstages * kTsBBytes);

  if (count) Nr = min(Nr, max(*count, 0));       // a region memory: only its filled rows; no tiles at all when it is empty
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.y * kTsBM;
  const int nhalf = (Nq - q0 > kTsHalf) ? 2 : 1;
  const int ntiles = (Nr + kTsBN - 1) / kTsBN;
  const int D = nkb * kTsBK;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmR);
    mbar_init(&tail->afull, 8);
    for (int i = 0; i < nstages; ++i) { mbar_init(&tail->full[i], 1); mbar_init(&tail->empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tail->acc_full[i], 1); mbar_init(&tail->acc_empty[i], 4); }
    fence_barrier_init();
  }
  if (warp == kTsMmaWarp) tmem_alloc(&tail->tmem_base, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tail->tmem_base;
  const uint32_t tmem_a = tmem + 256u;             // queries: half hf at columns [256 + hf * D/2, +D/2)

  if (warp == kTsTmaWarp) {
    if (lane == 0) {
      int st = 0;
      uint32_t ph = 1;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&tail->empty[st], ph);
          mbar_expect_tx(&tail->full[st], kTsBBytes);
          tma_load_2d(r_smem + (size_t)st * kTsBBytes, &tmR, &tail->full[st], kb * kTsBK, t * kTsBN, gridDim.y > 1 ? kEvictLast : kEvictFirst);
          if (++st == nstages) { st = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == kTsMmaWarp) {
    const bool leader = elect_one();
    const uint32_t idesc = make_idesc_bf16(kTsHalf, kTsBN);
    const uint32_t r_base = smem_u32(r_smem);
    mbar_wait(&tail->afull, 0);                    // every epilogue warp has stored its query rows into TMEM
    tc_fence_after();
    int st0 = 0, i = 0;                            // st0 / ph0: ring position of the tile's first k-block
    uint32_t ph0 = 0;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++i) {
      for (int hf = 0; hf < nhalf; ++hf) {
        const int seq = i * nhalf + hf, slot = seq & 1, use = seq >> 1;
        mbar_wait(&tail->acc_empty[slot], (uint32_t)((use & 1) ^ 1));
        tc_fence_after();
        int st = st0;
        uint32_t ph = ph0;
        for (int kb = 0; kb < nkb; ++kb) {
          if (hf == 0) {                           // the second half walks stages the first one already waited for
            mbar_wait(&tail->full[st], ph);
            tc_fence_after();
          }
          if (leader) {
            const uint64_t db = make_desc_sw128(r_base + (uint32_t)(st * kTsBBytes));
            const uint32_t d_addr = tmem + (uint32_t)(slot * kTsBN);
            const uint32_t a_addr = tmem_a + (uint32_t)(hf * (D / 2) + kb * (kTsBK / 2));
#pragma unroll
            for (int k = 0; k < kTsBK / 16; ++k) mma_bf16_ts(d_addr, a_addr + (uint32_t)(k * 8), db + 2 * k, idesc, (kb | k) != 0);
            if (hf == nhalf - 1) mma_commit(&tail->empty[st]);      // last reader of the stage
          }
          __syncwarp();
          if (++st == nstages) { st = 0; ph ^= 1u; }
        }
        if (leader) mma_commit(&tail->acc_full[slot]);
        __syncwarp();
        if (hf == nhalf - 1) { st0 = st; ph0 = ph; }
      }
    }
  } else {
    const int qd = warp & 3, hf = warp >> 2;
    const int q = q0 + hf * kTsHalf + qd * 32 + lane;
    const bool active = hf < nhalf;
    // ---- this thread's query row -> TMEM (its own lane), two bf16 per 32-bit column ----
    if (active) {
      const uint32_t* src = reinterpret_cast<const uint32_t*>(queries + (long long)q * D);
      for (int c = 0; c < D / 2; c += 32) {
        uint32_t v[32];
        if (q < Nq) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint4 u = __ldg(reinterpret_cast<const uint4*>(src + c) + j);
            v[4 * j] = u.x; v[4 * j + 1] = u.y; v[4 * j + 2] = u.z; v[4 * j + 3] = u.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;
        }
        tmem_st_32(tmem_a + ((uint32_t)(qd * 32) << 16) + (uint32_t)(hf * (D / 2) + c), v);
      }
      tmem_st_wait();
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&tail->afull);

    if (scale) inv_tau = __ldg(scale);
    const float c2 = inv_tau * 1.4426950408889634f;
    float m = -INFINITY, ssum = 0.f;
    auto proc = [&](uint32_t (&v)[32], int r0, int col) {
      const int nval = min(32, Nr - (r0 + col));
      if (nval == 32) {
        float t10[10];
#pragma unroll
        for (int j = 0; j < 10; ++j) t10[j] = max3(__uint_as_float(v[3 * j]), __uint_as_float(v[3 * j + 1]), __uint_as_float(v[3 * j + 2]));
        const float u0 = max3(t10[0], t10[1], t10[2]), u1 = max3(t10[3], t10[4], t10[5]), u2 = max3(t10[6], t10[7], t10[8]);
        const float u3 = max3(t10[9], __uint_as_float(v[30]), __uint_as_float(v[31]));
        const float cm = fmaxf(max3(u0, u1, u2), u3);
        if (cm > m) { ssum *= ex2_approx((m - cm) * c2); m = cm; }
        const float mc = m * c2;
        const uint64_t C2 = pack2(c2, c2), NM = pack2(-mc, -mc);
        uint64_t a0 = 0ull, a1 = 0ull;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const uint64_t x2 = fma2(pack2u(v[2 * j], v[2 * j + 1]), C2, NM);
          uint64_t e2;
          if ((j % 4) < COR_SIM_TS_POLY_OF4) {
            e2 = exp2_poly2(x2);
          } else {
            float x0, x1;
            unpack2(x2, x0, x1);
            e2 = pack2(ex2_approx(x0), ex2_approx(x1));
          }
          if (j & 1) a1 = add2(a1, e2);
          else a0 = add2(a0, e2);
        }
        float s0, s1;
        unpack2(add2(a0, a1), s0, s1);
        ssum += s0 + s1;
      } else {
        float cm = -INFINITY;
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j < nval) cm = fmaxf(cm, __uint_as_float(v[j]));
        if (cm > m) { ssum *= ex2_approx((m - cm) * c2); m = cm; }
        const float mc = m * c2;
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j < nval) ssum += ex2_approx(fmaf(__uint_as_float(v[j]), c2, -mc));
      }
    };
    if (active) {
      int i = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++i) {
        const int seq = i * nhalf + hf, slot = seq & 1, use = seq >> 1;
        mbar_wait(&tail->acc_full[slot], (uint32_t)(use & 1));
        tc_fence_after();
        const int r0 = t * kTsBN;
        const uint32_t taddr = tmem + ((uint32_t)(qd * 32) << 16) + (uint32_t)(slot * kTsBN);
        const int nch = min(kTsBN / 32, (Nr - r0 + 31) / 32);
        uint32_t va[32], vb[32];
        tmem_ld_32(taddr, va);
        tmem_ld_wait();
        if (nch > 1) tmem_ld_32(taddr + 32u, vb);
        proc(va, r0, 0);
        tmem_ld_wait();
        if (nch > 2) tmem_ld_32(taddr + 64u, va);
        if (nch > 1) proc(vb, r0, 32);
        tmem_ld_wait();
        if (nch > 3) tmem_ld_32(taddr + 96u, vb);
        if (nch > 2) proc(va, r0, 64);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tail->acc_empty[slot]);     // accumulator in registers: the MMAs of the next use may start
        if (nch > 3) proc(vb, r0, 96);
      }
      float* o = part + (((long long)blockIdx.y * gridDim.x + blockIdx.x) * kTsBM + hf * kTsHalf + qd * 32 + lane) * 2;
      o[0] = m * inv_tau;
      o[1] = ssum;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kTsMmaWarp) tmem_dealloc(tmem, 512);
}

// LSE-only launcher (sim_umma.cu stores S with the kernel that keeps both operands in shared memory).  Returns the
// number of partial records per query tile in *nparts.
static_assert(kTsBM == kMemQT, "a region memory's scan partials are laid out per kTsBM-query tile");

int sim_umma_ts_launch(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, const float* scale, void* work,
                       int* nparts, cudaStream_t st, const int* count) {
  const int qtiles = ceil_div(Nq, kTsBM), ntiles = ceil_div(Nr, kTsBN);
  CUtensorMap tmR;
  int rc = umma::encode_tmap_bf16_2d(&tmR, regions, (uint64_t)Nr, (uint64_t)D, kTsBN, kTsBK);
  if (rc) return rc;
  int gx = sm_count() / qtiles;
  if (gx < 1) gx = 1;
  if (gx > ntiles) gx = ntiles;
  const int nkb = D / kTsBK;
  int nstages = (int)((227 * 1024 - sizeof(TsSmemTail) - 1024) / kTsBBytes);
  if (nstages > kTsMaxStages) nstages = kTsMaxStages;
  const size_t smem = (size_t)nstages * kTsBBytes + sizeof(TsSmemTail) + 1024;
  COR_CUDA(cudaFuncSetAttribute(sim_umma_ts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  sim_umma_ts_kernel<<<dim3(gx, qtiles), 320, smem, st>>>(tmR, reinterpret_cast<const bf16*>(queries), Nr, Nq, nkb, nstages, inv_tau,
                                                         scale, reinterpret_cast<float*>(work), count);
  *nparts = gx;
  return check_launch("sim_umma_ts_kernel");
}

}  // namespace cor
