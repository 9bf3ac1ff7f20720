// Region x query similarity on tcgen05 tensor cores with the InfoNCE log-sum-exp fused into the
// epilogue (Class N; no reference implementation -- the reference's F.cosine_similarity at
// utils/loss_func.py:84,123 is the diagonal of this matrix).
//
//   S[q, r] = sum_d Q[q,d] * R[r,d]          Q: queries, A operand, up to 256 rows resident in shared memory
//                                            R: regions, B operand, 128 rows x 64 d per TMA stage
//   lse[q]  = log sum_r exp(S[q,r] / tau)    accumulated on line by the thread that owns TMEM lane q
//
// Orientation: queries on the MMA M axis (TMEM lanes), regions on N (TMEM columns).  An epilogue thread
// therefore owns one query row: its running (max, sum) is two registers, and the optional S store is
// 64 contiguous bytes per thread per 16-column chunk.
//
// A CTA holds TWO 128-query halves and issues two M128 x N128 x K16 MMAs per region k-slice, so every
// region byte fetched from L2 feeds 256 query rows (the region stream, not the tensor pipe, is what
// saturates first at M = 128).  Persistent CTAs walk region tiles with a 5-stage TMA ring and a
// double-buffered TMEM accumulator (2 buffers x 2 halves x 128 columns = all 512), so the MMAs of tile
// i+1 overlap the epilogue of tile i.  With few queries the kernel is HBM-bound on the region stream;
// with hundreds of queries it is tensor-pipe-bound (SURVEY.md 8d).
//
// Warp roles (320 threads): 0..7 = epilogue (warp w reads TMEM lane quarter w % 4 of half w / 4), 8 = TMA producer,
// 9 = TMEM owner + MMA issuer.  The two single-thread roles sit at the HIGHEST warp ids on purpose: the SM's issue
// arbiter favours high warp ids, and a producer / MMA thread that has to queue behind two busy epilogue warps of its
// sub-partition starves the tensor pipe.  (An optional L2 prefetch of region tiles ahead of the stage loads,
// COR_SIM_PREFETCH, measured slower and is off.)
#include <stdlib.h>

#include "umma.cuh"

namespace cor {

using namespace umma;

constexpr int kSimMaxStages = 6;                 // ring depth (A/B on B200: 4, 6 and 10 stages time the same; 6 leaves margin)
constexpr int kSimHalf = 128;                    // queries per MMA (UMMA M)
constexpr int kSimBM = 2 * kSimHalf;             // queries per CTA
constexpr int kSimBN = 128;                      // regions per tile (UMMA N)
constexpr int kSimBK = 64;
constexpr int kSimABytes = kSimHalf * kSimBK * 2;  // 16 KB: one k-block of one query half
constexpr int kSimBBytes = kSimBN * kSimBK * 2;    // 16 KB: one stage of regions
constexpr int kSimMaxKB = 4;                       // D <= 256
#ifndef COR_SIM_POLY_OF4
#define COR_SIM_POLY_OF4 0                         // of every 4 element pairs, how many take the FMA-pipe exp2 (0 = all MUFU)
#endif
constexpr int kSimPolyOf4 = COR_SIM_POLY_OF4;
constexpr int kSimTmaWarp = 8, kSimMmaWarp = 9;    // epilogue = warps 0..7
#ifndef COR_SIM_PREFETCH
#define COR_SIM_PREFETCH 0
#endif
constexpr int kSimPrefetch = COR_SIM_PREFETCH;     // region tiles prefetched into L2 ahead of the stage loads (0 = off: measured 55.3 vs 57.3 us at 1024 x 102 400, 20.5 vs 26.6 us at 16 x 102 400)
static_assert(kSimBN == 128, "the epilogue is unrolled for four 32-column chunks");

#ifdef COR_SIM_TRACE
// Debug build only (benchmarks/build_variants.sh ... "-DCOR_SIM_TRACE"): CTA (0,0) stamps clock64() at the hand-offs of
// its first 32 tiles: [tile][0] MMA thread starts issuing, [1] all MMAs of the tile issued, [2] epilogue warp 0 sees
// acc_full, [3] its last TMEM load has landed (buffer released), [4] tile done, [5] producer issued the tile's last stage.
__device__ long long g_sim_trace[32][8];
#define SIM_TRACE(tile, ev) do { if (blockIdx.x == 0 && blockIdx.y == 0 && (tile) < 32) g_sim_trace[(tile)][(ev)] = clock64(); } while (0)
#else
#define SIM_TRACE(tile, ev) do { } while (0)
#endif

struct SimSmemTail {
  uint64_t qfull, full[kSimMaxStages], empty[kSimMaxStages], acc_full[2], acc_empty[2];
  uint32_t tmem_base;
};

// Third epilogue mode (InfoNCE backward, many queries): the S tile leaves TMEM as the bf16 coefficient matrix
//   P[q,r] = (exp(S[q,r]/tau - lse[q]) - [r == target(q)]) * g_loss[0] * g_mul / (tau * Nq)
// so neither S nor an fp32 P is ever written; dQ = P R and dR = P^T Q follow as plain GEMMs.
struct SimCoef {
  const float* lse;
  const long long* targets;
  const float* g_loss;
  float g_mul;
  bf16* P;
};

// part layout (shared with the streaming producer's combine kernel): [qtile][gridDim.x][kSimBM][2]
__global__ void __launch_bounds__(320, 1) sim_umma_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmR,
                                                          int Nr, int Nq, int nkb, int nstages, int q_slots, int cl, float inv_tau,
                                                          const float* __restrict__ scale, float* __restrict__ S, float* __restrict__ part, SimCoef coef) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* base = reinterpret_cast<uint8_t*>(((uintptr_t)smem + 1023) & ~(uintptr_t)1023);
  uint8_t* q_smem = base;                                                   // [half][kb] x 16 KB
  uint8_t* r_smem = base + (size_t)q_slots * kSimABytes;                    // nstages x 16 KB
  SimSmemTail* tail = reinterpret_cast<SimSmemTail*>(r_smem + (size_t)nstages * kSimBBytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.y * kSimBM;
  const int nhalf = (Nq - q0 > kSimHalf) ? 2 : 1;
  const int ntiles = (Nr + kSimBN - 1) / kSimBN;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmQ);
    prefetch_tmap(&tmR);
    mbar_init(&tail->qfull, 1);
    // a stage is released once the MMAs of ALL cl CTAs of the cluster have read it (every CTA's TMA slice lands in all of them)
    for (int i = 0; i < nstages; ++i) { mbar_init(&tail->full[i], 1); mbar_init(&tail->empty[i], (uint32_t)cl); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tail->acc_full[i], 1); mbar_init(&tail->acc_empty[i], 8); }
    fence_barrier_init();
  }
  if (warp == kSimMmaWarp) tmem_alloc(&tail->tmem_base, 512);
  tc_fence_before();
  __syncthreads();
  if (cl > 1) cluster_sync();       // every CTA's barriers are initialised before any peer multicasts into them
  tc_fence_after();
  const uint32_t tmem = tail->tmem_base;
  const uint32_t crank = cl > 1 ? cluster_ctarank() : 0;
  const uint16_t cmask = (uint16_t)((1u << cl) - 1u);
  const int slice_rows = kSimBN / cl;

  if (warp == kSimTmaWarp) {
    if (lane == 0) {
      mbar_expect_tx(&tail->qfull, (uint32_t)(nhalf * nkb * kSimABytes));
      for (int hf = 0; hf < nhalf; ++hf)
        for (int kb = 0; kb < nkb; ++kb)
          tma_load_2d(q_smem + (hf * nkb + kb) * kSimABytes, &tmQ, &tail->qfull, kb * kSimBK, q0 + hf * kSimHalf, kEvictLast);
      int it = 0;
      for (int t = blockIdx.x; t < ntiles && t < (int)blockIdx.x + kSimPrefetch * (int)gridDim.x; t += gridDim.x)
        if (crank == 0)
          for (int kb = 0; kb < nkb; ++kb) tma_prefetch_2d(&tmR, kb * kSimBK, t * kSimBN);
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int tp = t + kSimPrefetch * (int)gridDim.x;          // keep kSimPrefetch tiles of this CTA on their way into L2
        if (kSimPrefetch > 0 && tp < ntiles && crank == 0)
          for (int kb = 0; kb < nkb; ++kb) tma_prefetch_2d(&tmR, kb * kSimBK, tp * kSimBN);
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int st = it % nstages;
          mbar_wait(&tail->empty[st], ((it / nstages) & 1) ^ 1);
          mbar_expect_tx(&tail->full[st], kSimBBytes);
          if (cl > 1)   // this CTA fetches rows [crank*slice, +slice) of the stage and multicasts them to the whole cluster
            tma_load_2d_mc(r_smem + st * kSimBBytes + crank * slice_rows * (kSimBK * 2), &tmR, &tail->full[st], kb * kSimBK,
                           t * kSimBN + (int)crank * slice_rows, cmask, gridDim.y > (unsigned)cl ? kEvictLast : kEvictFirst);
          else
            tma_load_2d(r_smem + st * kSimBBytes, &tmR, &tail->full[st], kb * kSimBK, t * kSimBN, gridDim.y > 1 ? kEvictLast : kEvictFirst);
        }
        SIM_TRACE((t - (int)blockIdx.x) / (int)gridDim.x, 5);
      }
    }
  } else if (warp == kSimMmaWarp) {
    // The WHOLE warp walks this loop (barrier waits, descriptor arithmetic) and one elected lane issues: with the role
    // wrapped in `if (lane == 0)` the compiler must treat every descriptor as divergent (R2UR + ELECT + BRA.U.ANY around
    // each UTCHMMA, ~140 cycles per MMA on a lone warp's dependent-issue chain -- measured with the trace build: 4 450
    // cycles to issue the 32 MMAs of a tile that the tensor pipe executes in 2 048).
    const bool leader = elect_one();
    const uint32_t idesc = make_idesc_bf16(kSimHalf, kSimBN);
    const uint32_t q_base = smem_u32(q_smem), r_base = smem_u32(r_smem);
    mbar_wait(&tail->qfull, 0);
    int st = 0, i = 0;
    uint32_t ph = 0;
    bool ready = false;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++i) {
      const int buf = i & 1;
      mbar_wait(&tail->acc_empty[buf], ((i >> 1) & 1) ^ 1);
      tc_fence_after();
      if (leader) SIM_TRACE(i, 0);
      for (int kb = 0; kb < nkb; ++kb) {
        if (!ready) mbar_wait(&tail->full[st], ph);
        tc_fence_after();
        const uint64_t db = make_desc_sw128(r_base + (uint32_t)(st * kSimBBytes));
        {   // poll the NEXT stage now: the try_wait's latency passes under this stage's MMA issue
          const int nst = st + 1 == nstages ? 0 : st + 1;
          ready = mbar_try_wait(&tail->full[nst], nst == 0 ? ph ^ 1u : ph);
        }
        if (leader) {
          for (int hf = 0; hf < nhalf; ++hf) {
            const uint64_t da = make_desc_sw128(q_base + (uint32_t)((hf * nkb + kb) * kSimABytes));
            const uint32_t d_addr = tmem + (uint32_t)((buf * 2 + hf) * kSimBN);
            mma_bf16_ss(d_addr, da, db, idesc, kb != 0);
#pragma unroll
            for (int k = 1; k < kSimBK / 16; ++k) mma_bf16_ss_acc(d_addr, da + 2 * k, db + 2 * k, idesc);
          }
          if (cl > 1) mma_commit_mc(&tail->empty[st], cmask);
          else mma_commit(&tail->empty[st]);
        }
        __syncwarp();
        if (++st == nstages) { st = 0; ph ^= 1u; }
      }
      if (leader) {
        mma_commit(&tail->acc_full[buf]);
        SIM_TRACE(i, 1);
      }
      __syncwarp();
    }
  } else {
    const int e = warp;
    const int qd = warp & 3;                       // TMEM lane quarter this warp may read
    const int hf = e >> 2;                         // query half (accumulator) this warp drains
    const int q = q0 + hf * kSimHalf + qd * 32 + lane;
    const bool active = hf < nhalf;
    const bool qok = active && q < Nq;
    if (scale) inv_tau = __ldg(scale);
    const float c2 = inv_tau * 1.4426950408889634f;   // exp(x/tau) = exp2(x * c2)
    float m = -INFINITY, ssum = 0.f;               // running max of raw S and sum exp2((S - m) c2)
    const bool vec_ok = (Nr % 4 == 0) && ((((uintptr_t)S) & 15) == 0);
    const bool want_coef = coef.P != nullptr;
    const bool pvec_ok = (Nr % 8 == 0) && ((((uintptr_t)coef.P) & 15) == 0);
    float neg_lse2 = 0.f, gscale = 0.f;
    long long tq = -1;
    if (want_coef && qok) {
      neg_lse2 = -coef.lse[q] * 1.4426950408889634f;
      gscale = coef.g_loss[0] * coef.g_mul * inv_tau / (float)Nq;
      tq = coef.targets[q];
    }
    // One 32-column chunk of this thread's query row (registers v[0..31] = S[q, r0+col .. +31]).
    auto proc = [&](uint32_t (&v)[32], int r0, int col) {
      const int nval = min(32, Nr - (r0 + col));
      if (S && qok) {
        float* dst = S + (long long)q * Nr + r0 + col;
        if (vec_ok && nval == 32) {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            reinterpret_cast<float4*>(dst)[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                                            __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (j < nval) dst[j] = __uint_as_float(v[j]);
        }
      }
      if (want_coef && qok) {
        bf16* dst = coef.P + (long long)q * Nr + r0 + col;
        const long long hit = tq - (long long)(r0 + col);        // position of the target inside this chunk, if any
        uint32_t w[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          float c0 = ex2_approx(fmaf(__uint_as_float(v[2 * j]), c2, neg_lse2));
          float c1 = ex2_approx(fmaf(__uint_as_float(v[2 * j + 1]), c2, neg_lse2));
          if (hit == 2 * j) c0 -= 1.f;
          if (hit == 2 * j + 1) c1 -= 1.f;
          __nv_bfloat162 pk = __floats2bfloat162_rn(c0 * gscale, c1 * gscale);
          w[j] = *reinterpret_cast<uint32_t*>(&pk);
        }
        if (pvec_ok && nval == 32) {
#pragma unroll
          for (int j = 0; j < 4; ++j) reinterpret_cast<uint4*>(dst)[j] = make_uint4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (j < nval) {
              const uint32_t u = w[j >> 1];
              reinterpret_cast<uint16_t*>(dst)[j] = (uint16_t)((j & 1) ? (u >> 16) : (u & 0xffffu));
            }
        }
      }
      if (part) {
        if (nval == 32) {
          // Full chunk.  The MMA of a 128 x 128 x 256 tile and 16 384 MUFU.EX2 both take ~1024 SM cycles, so an
          // all-MUFU epilogue paces the tensor pipe.  Here: max by 3-input FMNMX (16 ops), the exponent arguments by
          // packed FFMA2, kSimPolyPairs of the 16 pairs through the FMA-pipe polynomial exp2 and the rest through
          // MUFU, packed FADD2 accumulation in independent chains.
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
            if ((j % 4) < kSimPolyOf4) {        // spread the polynomial pairs evenly through the chunk
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
      }
    };
    int i = 0;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++i) {
      const int buf = i & 1;
      mbar_wait(&tail->acc_full[buf], (i >> 1) & 1);
      tc_fence_after();
      if (warp == 0 && lane == 0) SIM_TRACE(i, 2);
      if (active) {
        const int r0 = t * kSimBN;
        const uint32_t taddr = tmem + ((uint32_t)(qd * 32) << 16) + (uint32_t)((buf * 2 + hf) * kSimBN);
        // chunk c+1 is in flight (tcgen05.ld) while chunk c is processed; columns beyond Nr hold zeros (TMA fills
        // out-of-range region rows), loading them is harmless and proc() masks them
        const int nch = min(kSimBN / 32, (Nr - r0 + 31) / 32);       // warp-uniform
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
        // the accumulator is in registers: hand the TMEM buffer back BEFORE the last chunk is processed
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tail->acc_empty[buf]);
        if (warp == 0 && lane == 0) SIM_TRACE(i, 3);
        if (nch > 3) proc(vb, r0, 96);
        if (warp == 0 && lane == 0) SIM_TRACE(i, 4);
      } else {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tail->acc_empty[buf]);
      }
    }
    if (part && active) {
      float* o = part + (((long long)blockIdx.y * gridDim.x + blockIdx.x) * kSimBM + hf * kSimHalf + qd * 32 + lane) * 2;
      o[0] = m * inv_tau;     // partial max in units of S / tau, as the combine kernel expects
      o[1] = ssum;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (cl > 1) cluster_sync();       // no CTA leaves while a peer may still multicast into it or arrive on its barriers
  if (warp == kSimMmaWarp) tmem_dealloc(tmem, 512);
}

}  // namespace cor

using namespace cor;

namespace cor {
static int sim_umma_launch_impl(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, const float* scale, float* S, float* lse,
                                void* work, int* nparts, int* qt, SimCoef coef, cudaStream_t st) {
  const bool want_lse = lse || nparts;
  COR_REQUIRE(regions && queries && (S || want_lse || coef.P), "cor_sim_umma_fwd: null pointer");
  COR_REQUIRE(Nr > 0 && Nq > 0 && D % kSimBK == 0 && D >= kSimBK && D <= kSimMaxKB * kSimBK, "cor_sim_umma_fwd: need D in {64,128,192,256} (D=%d)", D);
  COR_REQUIRE(!want_lse || work, "cor_sim_umma_fwd: lse needs a work buffer");
  const int qtiles = ceil_div(Nq, kSimBM), ntiles = ceil_div(Nr, kSimBN);
  // CTAs that walk the same region tiles for different query tiles can form a cluster (along grid.y) and share every
  // region stage through TMA multicast (L2 -> SM traffic of the region stream / cluster size).  Measured on B200
  // (profiles/README.md): no gain at cluster 2, -12 % at cluster 4 (only 132 of 148 SMs host whole clusters) -- the
  // kernel is paced by the TMEM read-out of the S tile, not by L2 -- so the default stays 1; COR_SIM_CLUSTER=2|4 enables it.
  int cl = 1;
  if (const char* e = getenv("COR_SIM_CLUSTER")) { const int v = atoi(e); if ((v == 1 || v == 2 || v == 4) && qtiles % v == 0) cl = v; }
  // log-sum-exp only (the InfoNCE forward): the kernel that keeps the queries in tensor memory (sim_umma_ts.cu) -- the
  // tensor pipe is no longer throttled by shared-memory bandwidth.  COR_SIM_TS=0 keeps this file's kernel (A/B).
  {
    const char* e = getenv("COR_SIM_TS");
    if (want_lse && !S && !coef.P && cl == 1 && !(e && atoi(e) == 0)) {
      int gx_ts = 0;
      int rc_ts = sim_umma_ts_launch(regions, queries, Nr, Nq, D, inv_tau, scale, work, &gx_ts, st);
      if (rc_ts) return rc_ts;
      if (nparts) {
        *nparts = gx_ts;
        *qt = kSimBM;
        return COR_OK;
      }
      return launch_lse_combine((const float*)work, Nq, gx_ts, kSimBM, lse, st);
    }
  }
  CUtensorMap tmQ, tmR;
  int rc = umma::encode_tmap_bf16_2d(&tmQ, queries, (uint64_t)Nq, (uint64_t)D, kSimHalf, kSimBK);
  if (rc) return rc;
  rc = umma::encode_tmap_bf16_2d(&tmR, regions, (uint64_t)Nr, (uint64_t)D, kSimBN / cl, kSimBK);
  if (rc) return rc;
  int gx = sm_count() / qtiles;
  if (gx < 1) gx = 1;
  if (gx > ntiles) gx = ntiles;
  // queries take nhalf * nkb 16-KB slots; the ring gets up to kSimMaxStages of the remaining 16-KB slots
  const int nkb = D / kSimBK;
  const int q_slots = (Nq > kSimHalf ? 2 : 1) * nkb;
  int nstages = (int)((227 * 1024 - sizeof(SimSmemTail) - 1024) / kSimBBytes) - q_slots;
  if (nstages > kSimMaxStages) nstages = kSimMaxStages;
  if (const char* e = getenv("COR_SIM_STAGES")) { const int v = atoi(e); if (v >= 2 && v <= nstages) nstages = v; }   // A/B knob
  const size_t smem = (size_t)q_slots * kSimABytes + (size_t)nstages * kSimBBytes + sizeof(SimSmemTail) + 1024;
  COR_CUDA(cudaFuncSetAttribute(sim_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  float* part = want_lse ? (float*)work : nullptr;
  const int nkb_arg = nkb;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(gx, qtiles);
  cfg.blockDim = dim3(320);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1;
  attr[0].val.clusterDim.y = (unsigned)cl;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (cl > 1) {
    // persistent CTAs: every cluster must be resident at once (a GPC may not fit a whole number of clusters)
    int max_clusters = 0;
    COR_CUDA(cudaOccupancyMaxActiveClusters(&max_clusters, sim_umma_kernel, &cfg));
    const int per_x = qtiles / cl;
    if (max_clusters >= per_x && gx > max_clusters / per_x) {
      gx = max_clusters / per_x;
      cfg.gridDim = dim3(gx, qtiles);
    }
  }
  COR_CUDA(cudaLaunchKernelEx(&cfg, sim_umma_kernel, tmQ, tmR, Nr, Nq, nkb_arg, nstages, q_slots, cl, inv_tau, scale, S, part, coef));
  rc = check_launch("sim_umma_kernel");
  if (rc || !want_lse) return rc;
  if (nparts) {                       // deferred: the caller merges the partials (cor_infonce_tail)
    *nparts = gx;
    *qt = kSimBM;
    return COR_OK;
  }
  // inactive query rows of a half-empty last tile publish nothing; the combine only reads rows < Nq
  return launch_lse_combine(part, Nq, gx, kSimBM, lse, st);
}

int sim_umma_launch(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, const float* scale, float* S, float* lse,
                    void* work, int* nparts, int* qt, cudaStream_t st) {
  return sim_umma_launch_impl(regions, queries, Nr, Nq, D, inv_tau, scale, S, lse, work, nparts, qt, SimCoef{nullptr, nullptr, nullptr, 0.f, nullptr}, st);
}
}  // namespace cor

extern "C" int cor_sim_umma_coef(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, const float* lse,
                                 const long long* targets, const float* g_loss, float g_mul, void* P_bf16, cor_stream_t stream) {
  COR_REQUIRE(lse && targets && g_loss && P_bf16, "cor_sim_umma_coef: null pointer");
  return cor::sim_umma_launch_impl(regions, queries, Nr, Nq, D, inv_tau, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                                   cor::SimCoef{lse, targets, g_loss, g_mul, (cor::bf16*)P_bf16}, cor::as_stream(stream));
}

extern "C" int cor_sim_umma_fwd(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, float* S, float* lse,
                                void* work, cor_stream_t stream) {
  return cor::sim_umma_launch(regions, queries, Nr, Nq, D, inv_tau, nullptr, S, lse, work, nullptr, nullptr, as_stream(stream));
}

// cor_sim_umma_fwd with the logit scale read from device memory
extern "C" int cor_sim_umma_fwd_ls(const void* regions, const void* queries, int Nr, int Nq, int D, const float* logit_scale, float* S,
                                   float* lse, void* work, cor_stream_t stream) {
  COR_REQUIRE(logit_scale, "cor_sim_umma_fwd_ls: null logit_scale");
  return cor::sim_umma_launch(regions, queries, Nr, Nq, D, 0.f, logit_scale, S, lse, work, nullptr, nullptr, as_stream(stream));
}

#ifdef COR_SIM_TRACE
extern "C" int cor_debug_sim_trace(long long* host_out) {
  COR_CUDA(cudaDeviceSynchronize());
  COR_CUDA(cudaMemcpyFromSymbol(host_out, cor::g_sim_trace, sizeof(long long) * 32 * 8));
  return COR_OK;
}
#endif
