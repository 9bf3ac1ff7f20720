// Region x query similarity matrix on tcgen05 tensor cores, both operands in shared memory (Class N; no reference
// implementation -- the reference's F.cosine_similarity at utils/loss_func.py:84,123 is the diagonal of this matrix).
//
//   S[q, r] = sum_d Q[q,d] * R[r,d]          Q: queries, A operand, up to 256 rows resident in shared memory
//                                            R: regions, B operand, 128 rows x 64 d per TMA stage
//
// This kernel stores S (the top-k prefilter and ops.similarity).  The log-sum-exp of the InfoNCE forward never needs S
// and runs on the kernel that keeps the queries in tensor memory (sim_umma_ts.cu): the launcher below sends every lse
// request there.
//
// Orientation: queries on the MMA M axis (TMEM lanes), regions on N (TMEM columns).  An epilogue thread therefore owns
// one query row, and its S store is 128 contiguous bytes per thread per 32-column chunk.
//
// A CTA holds TWO 128-query halves and issues two M128 x N128 x K16 MMAs per region k-slice, so every region byte
// fetched from L2 feeds 256 query rows (the region stream, not the tensor pipe, is what saturates first at M = 128).
// Persistent CTAs walk region tiles with a TMA ring of up to kSimMaxStages stages and a double-buffered TMEM
// accumulator (2 buffers x 2 halves x 128 columns = all 512), so the MMAs of tile i+1 overlap the epilogue of tile i.
//
// Warp roles (320 threads): 0..7 = epilogue (warp w reads TMEM lane quarter w % 4 of half w / 4), 8 = TMA producer,
// 9 = TMEM owner + MMA issuer.  The two single-thread roles sit at the HIGHEST warp ids on purpose: the SM's issue
// arbiter favours high warp ids, and a producer / MMA thread that has to queue behind two busy epilogue warps of its
// sub-partition starves the tensor pipe.
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
constexpr int kSimTmaWarp = 8, kSimMmaWarp = 9;    // epilogue = warps 0..7
static_assert(kSimBN == 128, "the epilogue is unrolled for four 32-column chunks");

struct SimSmemTail {
  uint64_t qfull, full[kSimMaxStages], empty[kSimMaxStages], acc_full[2], acc_empty[2];
  uint32_t tmem_base;
};

__global__ void __launch_bounds__(320, 1) sim_umma_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmR,
                                                          int Nr, int Nq, int nkb, int nstages, int q_slots, float* __restrict__ S) {
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
    for (int i = 0; i < nstages; ++i) { mbar_init(&tail->full[i], 1); mbar_init(&tail->empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tail->acc_full[i], 1); mbar_init(&tail->acc_empty[i], 8); }
    fence_barrier_init();
  }
  if (warp == kSimMmaWarp) tmem_alloc(&tail->tmem_base, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tail->tmem_base;

  if (warp == kSimTmaWarp) {
    if (lane == 0) {
      mbar_expect_tx(&tail->qfull, (uint32_t)(nhalf * nkb * kSimABytes));
      for (int hf = 0; hf < nhalf; ++hf)
        for (int kb = 0; kb < nkb; ++kb)
          tma_load_2d(q_smem + (hf * nkb + kb) * kSimABytes, &tmQ, &tail->qfull, kb * kSimBK, q0 + hf * kSimHalf, kEvictLast);
      int it = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int st = it % nstages;
          mbar_wait(&tail->empty[st], ((it / nstages) & 1) ^ 1);
          mbar_expect_tx(&tail->full[st], kSimBBytes);
          tma_load_2d(r_smem + st * kSimBBytes, &tmR, &tail->full[st], kb * kSimBK, t * kSimBN, gridDim.y > 1 ? kEvictLast : kEvictFirst);
        }
      }
    }
  } else if (warp == kSimMmaWarp) {
    // The WHOLE warp walks this loop (barrier waits, descriptor arithmetic) and one elected lane issues: with the role
    // wrapped in `if (lane == 0)` the compiler must treat every descriptor as divergent (R2UR + ELECT + BRA.U.ANY around
    // each UTCHMMA, ~140 cycles per MMA on a lone warp's dependent-issue chain -- measured with clock64() stamps: 4 450
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
          mma_commit(&tail->empty[st]);
        }
        __syncwarp();
        if (++st == nstages) { st = 0; ph ^= 1u; }
      }
      if (leader) {
        mma_commit(&tail->acc_full[buf]);
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
    const bool vec_ok = (Nr % 4 == 0) && ((((uintptr_t)S) & 15) == 0);
    // One 32-column chunk of this thread's query row (registers v[0..31] = S[q, r0+col .. +31]).
    auto proc = [&](uint32_t (&v)[32], int r0, int col) {
      const int nval = min(32, Nr - (r0 + col));
      if (!qok) return;
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
    };
    int i = 0;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++i) {
      const int buf = i & 1;
      mbar_wait(&tail->acc_full[buf], (i >> 1) & 1);
      tc_fence_after();
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
        if (nch > 3) proc(vb, r0, 96);
      } else {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tail->acc_empty[buf]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kSimMmaWarp) tmem_dealloc(tmem, 512);
}

// S or the log-sum-exp, never both in one call: lse (or its partials, when nparts is given) comes from
// sim_umma_ts_kernel, S from sim_umma_kernel.
int sim_umma_launch(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, const float* scale, float* S, float* lse,
                    void* work, int* nparts, int* qt, cudaStream_t st) {
  const bool want_lse = lse || nparts;
  COR_REQUIRE(regions && queries && (S || want_lse), "cor_sim_umma_fwd: null pointer");
  COR_REQUIRE(!(S && want_lse), "cor_sim_umma_fwd: ask for S and lse in separate calls");
  COR_REQUIRE(Nr > 0 && Nq > 0 && D % kSimBK == 0 && D >= kSimBK && D <= kSimMaxKB * kSimBK, "cor_sim_umma_fwd: need D in {64,128,192,256} (D=%d)", D);
  COR_REQUIRE(!want_lse || work, "cor_sim_umma_fwd: lse needs a work buffer");
  if (want_lse) {
    int gx = 0;
    const int rc = sim_umma_ts_launch(regions, queries, Nr, Nq, D, inv_tau, scale, work, &gx, st);
    if (rc) return rc;
    if (nparts) {                     // deferred: the caller merges the partials (cor_infonce_tail)
      *nparts = gx;
      *qt = kSimBM;
      return COR_OK;
    }
    return launch_lse_combine((const float*)work, Nq, gx, kSimBM, lse, st);
  }
  const int qtiles = ceil_div(Nq, kSimBM), ntiles = ceil_div(Nr, kSimBN);
  CUtensorMap tmQ, tmR;
  int rc = umma::encode_tmap_bf16_2d(&tmQ, queries, (uint64_t)Nq, (uint64_t)D, kSimHalf, kSimBK);
  if (rc) return rc;
  rc = umma::encode_tmap_bf16_2d(&tmR, regions, (uint64_t)Nr, (uint64_t)D, kSimBN, kSimBK);
  if (rc) return rc;
  int gx = sm_count() / qtiles;
  if (gx < 1) gx = 1;
  if (gx > ntiles) gx = ntiles;
  // queries take nhalf * nkb 16-KB slots; the ring gets up to kSimMaxStages of the remaining 16-KB slots
  const int nkb = D / kSimBK;
  const int q_slots = (Nq > kSimHalf ? 2 : 1) * nkb;
  int nstages = (int)((227 * 1024 - sizeof(SimSmemTail) - 1024) / kSimBBytes) - q_slots;
  if (nstages > kSimMaxStages) nstages = kSimMaxStages;
  const size_t smem = (size_t)q_slots * kSimABytes + (size_t)nstages * kSimBBytes + sizeof(SimSmemTail) + 1024;
  COR_CUDA(cudaFuncSetAttribute(sim_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  sim_umma_kernel<<<dim3(gx, qtiles), 320, smem, st>>>(tmQ, tmR, Nr, Nq, nkb, nstages, q_slots, S);
  return check_launch("sim_umma_kernel");
}

}  // namespace cor

using namespace cor;

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
