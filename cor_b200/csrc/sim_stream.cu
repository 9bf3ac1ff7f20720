// Region x query similarity, InfoNCE and top-k -- CUDA-core streaming kernels.
//
// Class N (no reference implementation, SURVEY.md 0.2): the reference only ever computes the
// diagonal, F.cosine_similarity at utils/loss_func.py:84,123.  These kernels cover the HBM-bound
// regime (a handful of queries against many regions, AI ~ Nq flop/B) and the small utility steps
// (row L2-normalise of lib/support_branch.py:85, target logits, exact top-k re-rank); the
// tensor-core variants for many queries live in sim_umma.cu (S) and sim_umma_ts.cu (lse, same work-buffer layout).
#include "common.cuh"

namespace cor {

// ---- row L2 normalise ------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128) l2_normalize_kernel(const T* __restrict__ x, int D, float* __restrict__ y32,
                                                           bf16* __restrict__ y16, float* __restrict__ inv_norm) {
  __shared__ float scratch[32];
  const long long row = blockIdx.x;
  float ss[1] = {0.f};
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const float v = to_f<T>(x[row * D + d]);
    ss[0] = fmaf(v, v, ss[0]);
  }
  block_sum<1>(ss, scratch);
  const float inv = 1.f / fmaxf(sqrtf(ss[0]), 1e-12f);
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const float v = to_f<T>(x[row * D + d]) * inv;
    if (y32) y32[row * D + d] = v;
    if (y16) y16[row * D + d] = __float2bfloat16_rn(v);
  }
  if (threadIdx.x == 0 && inv_norm) inv_norm[row] = inv;
}

// ---- S = Q R^T, warp per region row (transpose_reduce16: common.cuh) -----------------------------------
// grid = (region CTAs, query tiles); block = 256.  dynamic smem = kQT * D floats.
// work layout: part [qtiles][gridDim.x][kQT][2] (running max, sum) -> lse by sim_lse_combine_kernel.
__global__ void __launch_bounds__(256) sim_stream_kernel(const bf16* __restrict__ regions, const bf16* __restrict__ queries, int Nr,
                                                         int Nq, int D, float inv_tau, const float* __restrict__ scale,
                                                         float* __restrict__ S, float* __restrict__ part) {
  extern __shared__ float qs[];   // [kQT][D]
  __shared__ float cm[8][kQT], cs[8][kQT];
  if (scale) inv_tau = __ldg(scale);
  const int q0 = blockIdx.y * kQT;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < kQT * D; i += blockDim.x) {
    const int q = i / D, d = i % D;
    qs[i] = (q0 + q < Nq) ? __bfloat162float(queries[(long long)(q0 + q) * D + d]) : 0.f;
  }
  __syncthreads();
  float m = -INFINITY, s = 0.f;   // online log-sum-exp of S/tau for query q0+lane over this warp's rows
  const int nvec = D / 8;
  for (long long r = (long long)blockIdx.x * 8 + warp; r < Nr; r += (long long)gridDim.x * 8) {
    float a[kQT];
#pragma unroll
    for (int q = 0; q < kQT; ++q) a[q] = 0.f;
    const uint4* row = reinterpret_cast<const uint4*>(regions + r * D);
    for (int v = lane; v < nvec; v += 32) {
      const uint4 raw = ld_stream16(row + v);
      float f[8];
      f[0] = bf16lo(raw.x); f[1] = bf16hi(raw.x); f[2] = bf16lo(raw.y); f[3] = bf16hi(raw.y);
      f[4] = bf16lo(raw.z); f[5] = bf16hi(raw.z); f[6] = bf16lo(raw.w); f[7] = bf16hi(raw.w);
#pragma unroll
      for (int q = 0; q < kQT; ++q) {
        const float4 x = *reinterpret_cast<const float4*>(&qs[q * D + v * 8]);
        const float4 y = *reinterpret_cast<const float4*>(&qs[q * D + v * 8 + 4]);
        a[q] = fmaf(f[0], x.x, a[q]); a[q] = fmaf(f[1], x.y, a[q]); a[q] = fmaf(f[2], x.z, a[q]); a[q] = fmaf(f[3], x.w, a[q]);
        a[q] = fmaf(f[4], y.x, a[q]); a[q] = fmaf(f[5], y.y, a[q]); a[q] = fmaf(f[6], y.z, a[q]); a[q] = fmaf(f[7], y.w, a[q]);
      }
    }
    const float sv = transpose_reduce16(a, lane);
    const int ql = ((lane >> 3) & 1) * 8 + ((lane >> 2) & 1) * 4 + ((lane >> 1) & 1) * 2 + (lane & 1);
    if (lane < 16 && q0 + ql < Nq) {
      if (S) S[(long long)(q0 + ql) * Nr + r] = sv;
      const float x = sv * inv_tau;
      if (x > m) { s = s * __expf(m - x) + 1.f; m = x; } else { s += __expf(x - m); }
    }
  }
  if (!part) return;
  // lane -> query map is the identity for lanes < 16 (bits 3..0); combine the 8 warps, then publish
  if (lane < kQT) { cm[warp][lane] = m; cs[warp][lane] = s; }
  __syncthreads();
  if (threadIdx.x < kQT) {
    float M = -INFINITY;
    for (int w = 0; w < 8; ++w) M = fmaxf(M, cm[w][threadIdx.x]);
    float Ssum = 0.f;
    for (int w = 0; w < 8; ++w) Ssum += (cm[w][threadIdx.x] == -INFINITY) ? 0.f : cs[w][threadIdx.x] * __expf(cm[w][threadIdx.x] - M);
    float* o = part + (((long long)blockIdx.y * gridDim.x + blockIdx.x) * kQT + threadIdx.x) * 2;
    o[0] = M; o[1] = Ssum;
  }
}

// lse[q] = log sum_r exp(S[q,r]/tau): merge of `nparts` (max,sum) partials per query, one warp per query
// (lanes stride over the partials, butterfly max / sum: fixed order, deterministic).
// part layout [qtiles][nparts][qt][2]; works for both the streaming and the UMMA producer.
__global__ void __launch_bounds__(256) sim_lse_combine_kernel(const float* __restrict__ part, int Nq, int nparts, int qt, float* __restrict__ lse) {
  const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (q >= Nq) return;
  const int tile = q / qt, ql = q % qt;
  const float* base = part + ((long long)tile * nparts * qt + ql) * 2;
  float M = -INFINITY;
  for (int p = lane; p < nparts; p += 32) M = fmaxf(M, base[(long long)p * qt * 2]);
  M = warp_max(M);
  double acc = 0.0;
  for (int p = lane; p < nparts; p += 32) {
    const float pm = base[(long long)p * qt * 2], ps = base[(long long)p * qt * 2 + 1];
    if (pm != -INFINITY) acc += (double)ps * exp((double)pm - (double)M);
  }
  acc = warp_sum(acc);
  if (lane == 0) lse[q] = M + (float)log(acc);
}

// ---- InfoNCE forward: target logits and the mean loss ------------------------------------------------
__global__ void __launch_bounds__(1024) infonce_fwd_kernel(const bf16* __restrict__ regions, const bf16* __restrict__ queries,
                                                           const long long* __restrict__ targets, const float* __restrict__ lse, int Nr,
                                                           int Nq, int D, float inv_tau, const float* __restrict__ scale,
                                                           float* __restrict__ loss, float* __restrict__ tgt_logit) {
  __shared__ double scratch[32];
  if (scale) inv_tau = __ldg(scale);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  double acc[1] = {0.0};
  for (int q = warp; q < Nq; q += nwarp) {
    long long t = targets[q];
    t = t < 0 ? 0 : (t >= Nr ? Nr - 1 : t);
    float d = 0.f;
    for (int k = lane; k < D; k += 32) d = fmaf(__bfloat162float(queries[(long long)q * D + k]), __bfloat162float(regions[t * D + k]), d);
    d = warp_sum(d);
    if (lane == 0) {
      tgt_logit[q] = d;
      acc[0] += (double)lse[q] - (double)d * (double)inv_tau;
    }
  }
  block_sum<1>(acc, scratch);
  if (threadIdx.x == 0) loss[0] = (float)(acc[0] / (double)Nq);
}

// ---- the fused step's tail in ONE launch: merge of the log-sum-exp partials (as sim_lse_combine_kernel), target
//      logits, mean InfoNCE loss and the step's total loss (seg + w_fg fg + w_bg bg + w_nce nce).  One CTA, one warp per query.
__global__ void __launch_bounds__(1024) infonce_tail_kernel(const float* __restrict__ part, int nparts, int qt,
                                                            const bf16* __restrict__ regions, const bf16* __restrict__ queries,
                                                            const long long* __restrict__ targets, int Nr, int Nq, int D, float inv_tau,
                                                            const float* __restrict__ scale, float* __restrict__ lse, float* __restrict__ nce,
                                                            float* __restrict__ tgt_logit, const float* __restrict__ seg,
                                                            const float* __restrict__ fgbg, float w_fg, float w_bg, float w_nce,
                                                            float* __restrict__ total) {
  __shared__ double scratch[32];
  if (scale) inv_tau = __ldg(scale);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  double acc[1] = {0.0};
  for (int q = warp; q < Nq; q += nwarp) {
    const int tile = q / qt, ql = q % qt;
    const float* base = part + ((long long)tile * nparts * qt + ql) * 2;
    float M = -INFINITY;
    for (int p = lane; p < nparts; p += 32) M = fmaxf(M, base[(long long)p * qt * 2]);
    M = warp_max(M);
    // fp32 rescale (expf of a non-positive argument, relative error ~1e-7) and fp64 only for the sum: the fp64 exp
    // of sim_lse_combine_kernel costs microseconds on this single-CTA critical path
    double a = 0.0;
    for (int p = lane; p < nparts; p += 32) {
      const float pm = base[(long long)p * qt * 2], ps = base[(long long)p * qt * 2 + 1];
      if (pm != -INFINITY) a += (double)(ps * expf(pm - M));
    }
    a = warp_sum(a);
    long long t = targets[q];
    t = t < 0 ? 0 : (t >= Nr ? Nr - 1 : t);
    float d = 0.f;
    for (int k = lane; k < D; k += 32) d = fmaf(__bfloat162float(queries[(long long)q * D + k]), __bfloat162float(regions[t * D + k]), d);
    d = warp_sum(d);
    if (lane == 0) {
      const float l = M + logf((float)a);
      lse[q] = l;
      tgt_logit[q] = d;
      acc[0] += (double)l - (double)d * (double)inv_tau;
    }
  }
  block_sum<1>(acc, scratch);
  if (threadIdx.x == 0) {
    const float v = (float)(acc[0] / (double)Nq);
    nce[0] = v;
    if (total) total[0] = seg[0] + w_fg * fgbg[0] + w_bg * fgbg[1] + w_nce * v;
  }
}

// ---- InfoNCE backward (streaming; D <= 256) ------------------------------------------------------------
//   coef[q,r] = (exp(S[q,r]/tau - lse[q]) - [r == t(q)]) * g / (tau * Nq)
//   g_regions[r,:] = sum_q coef[q,r] Q[q,:]      g_queries[q,:] = sum_r coef[q,r] R[r,:]
// grid = region CTAs (persistent), block = 256; loops over query tiles of 16 so that every region row
// is owned by exactly one warp (deterministic, no atomics).  qpart [gridDim.x][Nq][D] per-CTA partials
// of g_queries are reduced in fixed order by infonce_bwd_q_kernel.  With lspart (the logit-scale gradient wanted) every
// CTA also leaves sum_r (exp(s S - lse) - [r == t(q)]) S[q,r] over its rows per query, lspart [gridDim.x][Nq], for the same
// fold kernel.
template <bool WANT_R>
__global__ void __launch_bounds__(256, 1) infonce_bwd_kernel(const bf16* __restrict__ regions, const bf16* __restrict__ queries,
                                                             const long long* __restrict__ targets, const float* __restrict__ lse,
                                                             int Nr, int Nq, int D, float inv_tau, const float* __restrict__ scale,
                                                             const float* __restrict__ g_loss, float g_mul, float* __restrict__ g_regions,
                                                             float* __restrict__ qpart, float* __restrict__ lspart) {
  extern __shared__ float smem[];
  float* qs = smem;                    // [kQT][D]
  float* red = smem + kQT * D;         // [8 warps][kQT][D] reduction scratch (reuses after the row loop)
  __shared__ float lse_s[kQT];
  __shared__ long long tgt_s[kQT];
  __shared__ float ls_s[8][kQT];
  if (scale) inv_tau = __ldg(scale);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nvec = D / 8;              // <= 32: one 16-byte vector per lane
  const bool has = lane < nvec;
  const float gscale = g_loss[0] * g_mul * inv_tau / (float)Nq;
  for (int q0 = 0; q0 < Nq; q0 += kQT) {
    __syncthreads();
    for (int i = threadIdx.x; i < kQT * D; i += blockDim.x) {
      const int q = i / D, d = i % D;
      qs[i] = (q0 + q < Nq) ? __bfloat162float(queries[(long long)(q0 + q) * D + d]) : 0.f;
    }
    if (threadIdx.x < kQT) {
      lse_s[threadIdx.x] = (q0 + threadIdx.x < Nq) ? lse[q0 + threadIdx.x] : 0.f;
      tgt_s[threadIdx.x] = (q0 + threadIdx.x < Nq) ? targets[q0 + threadIdx.x] : -1;
    }
    __syncthreads();
    float dq[kQT][8];
#pragma unroll
    for (int q = 0; q < kQT; ++q)
#pragma unroll
      for (int e = 0; e < 8; ++e) dq[q][e] = 0.f;
    // the row of the NEXT iteration is loaded before this one is processed: a warp owns ~7 rows at 8 GPUs and the load was a
    // third of each row's dependent chain
    const long long rstep = (long long)gridDim.x * 8;
    long long r = (long long)blockIdx.x * 8 + warp;
    uint4 raw_next = make_uint4(0u, 0u, 0u, 0u);
    if (has && r < Nr) raw_next = ld_stream16(reinterpret_cast<const uint4*>(regions + r * D) + lane);
    float ls = 0.f;                    // lane q: this warp's share of the logit-scale gradient sum of query q0 + q
    for (; r < Nr; r += rstep) {
      float f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      const uint4 raw = raw_next;
      if (has && r + rstep < Nr) raw_next = ld_stream16(reinterpret_cast<const uint4*>(regions + (r + rstep) * D) + lane);
      if (has) {
        f[0] = bf16lo(raw.x); f[1] = bf16hi(raw.x); f[2] = bf16lo(raw.y); f[3] = bf16hi(raw.y);
        f[4] = bf16lo(raw.z); f[5] = bf16hi(raw.z); f[6] = bf16lo(raw.w); f[7] = bf16hi(raw.w);
      }
      float a[kQT];
#pragma unroll
      for (int q = 0; q < kQT; ++q) {
        float t = 0.f;
        if (has) {
          const float4 x = *reinterpret_cast<const float4*>(&qs[q * D + lane * 8]);
          const float4 y = *reinterpret_cast<const float4*>(&qs[q * D + lane * 8 + 4]);
          t = f[0] * x.x + f[1] * x.y + f[2] * x.z + f[3] * x.w + f[4] * y.x + f[5] * y.y + f[6] * y.z + f[7] * y.w;
        }
        a[q] = t;
      }
      const float sv = transpose_reduce16(a, lane);
      float coef = 0.f;
      if (lane < kQT && q0 + lane < Nq) {
        coef = __expf(sv * inv_tau - lse_s[lane]);
        if (tgt_s[lane] == r) coef -= 1.f;
        if (lspart) ls = fmaf(coef, sv, ls);
        coef *= gscale;
      }
      float gr[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int q = 0; q < kQT; ++q) {
        const float c = __shfl_sync(0xffffffffu, coef, q);
        if (has) {
          const float4 x = *reinterpret_cast<const float4*>(&qs[q * D + lane * 8]);
          const float4 y = *reinterpret_cast<const float4*>(&qs[q * D + lane * 8 + 4]);
          if (WANT_R) {
            gr[0] = fmaf(c, x.x, gr[0]); gr[1] = fmaf(c, x.y, gr[1]); gr[2] = fmaf(c, x.z, gr[2]); gr[3] = fmaf(c, x.w, gr[3]);
            gr[4] = fmaf(c, y.x, gr[4]); gr[5] = fmaf(c, y.y, gr[5]); gr[6] = fmaf(c, y.z, gr[6]); gr[7] = fmaf(c, y.w, gr[7]);
          }
#pragma unroll
          for (int e = 0; e < 8; ++e) dq[q][e] = fmaf(c, f[e], dq[q][e]);
        }
      }
      if (WANT_R && has) {
        float4* o = reinterpret_cast<float4*>(g_regions + r * D + lane * 8);
        if (q0 == 0) {
          o[0] = make_float4(gr[0], gr[1], gr[2], gr[3]);
          o[1] = make_float4(gr[4], gr[5], gr[6], gr[7]);
        } else {
          float4 p0 = o[0], p1 = o[1];
          o[0] = make_float4(p0.x + gr[0], p0.y + gr[1], p0.z + gr[2], p0.w + gr[3]);
          o[1] = make_float4(p1.x + gr[4], p1.y + gr[5], p1.z + gr[6], p1.w + gr[7]);
        }
      }
    }
    // reduce dq over the 8 warps (fixed order) and publish this CTA's partial for the query tile
    if (has) {
#pragma unroll
      for (int q = 0; q < kQT; ++q)
#pragma unroll
        for (int e = 0; e < 8; ++e) red[(warp * kQT + q) * D + lane * 8 + e] = dq[q][e];
    }
    if (lspart && lane < kQT) ls_s[warp][lane] = ls;
    __syncthreads();
    for (int i = threadIdx.x; i < kQT * D; i += blockDim.x) {
      const int q = i / D;
      if (q0 + q >= Nq) continue;
      float t = 0.f;
      for (int w = 0; w < 8; ++w) t += red[w * kQT * D + i];
      qpart[((long long)blockIdx.x * Nq + q0 + q) * D + (i % D)] = t;
    }
    if (lspart && threadIdx.x < kQT && q0 + threadIdx.x < Nq) {
      float t = 0.f;
      for (int w = 0; w < 8; ++w) t += ls_s[w][threadIdx.x];
      lspart[(long long)blockIdx.x * Nq + q0 + threadIdx.x] = t;
    }
  }
}

// g_regions only (no dQ): all queries (chunks of kRQ) stay in shared memory, every region row is read once
// and its gradient accumulates in registers across ALL query tiles -- one write per row, no block syncs
// inside the row loop.  cor_infonce_bwd takes it when neither g_queries nor the logit-scale gradient is wanted.
constexpr int kRQ = 128;
__global__ void __launch_bounds__(256, 1) infonce_bwd_regions_kernel(const bf16* __restrict__ regions, const bf16* __restrict__ queries,
                                                                     const long long* __restrict__ targets, const float* __restrict__ lse,
                                                                     int Nr, int Nq, int D, float inv_tau, const float* __restrict__ scale,
                                                                     const float* __restrict__ g_loss, float g_mul,
                                                                     float* __restrict__ g_regions) {
  extern __shared__ float qs[];        // [kRQ][D]
  __shared__ float lse_s[kRQ];
  __shared__ long long tgt_s[kRQ];
  if (scale) inv_tau = __ldg(scale);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nvec = D / 8;
  const bool has = lane < nvec;
  const float gscale = g_loss[0] * g_mul * inv_tau / (float)Nq;
  for (int qc0 = 0; qc0 < Nq; qc0 += kRQ) {
    const int qn = min(kRQ, Nq - qc0);
    const int qn16 = (qn + kQT - 1) / kQT * kQT;
    __syncthreads();
    for (int i = threadIdx.x; i < qn16 * D; i += blockDim.x) {
      const int q = i / D, d = i % D;
      qs[i] = q < qn ? __bfloat162float(queries[(long long)(qc0 + q) * D + d]) : 0.f;
    }
    for (int i = threadIdx.x; i < qn16; i += blockDim.x) {
      lse_s[i] = i < qn ? lse[qc0 + i] : 0.f;
      tgt_s[i] = i < qn ? targets[qc0 + i] : -1;
    }
    __syncthreads();
    // the row of the NEXT iteration is loaded before this one is processed: a warp owns ~7 rows at 8 GPUs and the load was a
    // third of each row's dependent chain
    const long long rstep = (long long)gridDim.x * 8;
    long long r = (long long)blockIdx.x * 8 + warp;
    uint4 raw_next = make_uint4(0u, 0u, 0u, 0u);
    if (has && r < Nr) raw_next = ld_stream16(reinterpret_cast<const uint4*>(regions + r * D) + lane);
    for (; r < Nr; r += rstep) {
      float f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      const uint4 raw = raw_next;
      if (has && r + rstep < Nr) raw_next = ld_stream16(reinterpret_cast<const uint4*>(regions + (r + rstep) * D) + lane);
      if (has) {
        f[0] = bf16lo(raw.x); f[1] = bf16hi(raw.x); f[2] = bf16lo(raw.y); f[3] = bf16hi(raw.y);
        f[4] = bf16lo(raw.z); f[5] = bf16hi(raw.z); f[6] = bf16lo(raw.w); f[7] = bf16hi(raw.w);
      }
      float gr[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int qt = 0; qt < qn16; qt += kQT) {
        const float* qb = qs + (size_t)qt * D + lane * 8;
        float a[kQT];
#pragma unroll
        for (int q = 0; q < kQT; ++q) {
          float t = 0.f;
          if (has) {
            const float4 x = *reinterpret_cast<const float4*>(qb + q * D);
            const float4 y = *reinterpret_cast<const float4*>(qb + q * D + 4);
            t = f[0] * x.x + f[1] * x.y + f[2] * x.z + f[3] * x.w + f[4] * y.x + f[5] * y.y + f[6] * y.z + f[7] * y.w;
          }
          a[q] = t;
        }
        const float sv = transpose_reduce16(a, lane);
        float coef = 0.f;
        if (lane < kQT && qt + lane < qn) {
          coef = __expf(sv * inv_tau - lse_s[qt + lane]);
          if (tgt_s[qt + lane] == r) coef -= 1.f;
          coef *= gscale;
        }
#pragma unroll
        for (int q = 0; q < kQT; ++q) {
          const float c = __shfl_sync(0xffffffffu, coef, q);
          if (has) {
            const float4 x = *reinterpret_cast<const float4*>(qb + q * D);
            const float4 y = *reinterpret_cast<const float4*>(qb + q * D + 4);
            gr[0] = fmaf(c, x.x, gr[0]); gr[1] = fmaf(c, x.y, gr[1]); gr[2] = fmaf(c, x.z, gr[2]); gr[3] = fmaf(c, x.w, gr[3]);
            gr[4] = fmaf(c, y.x, gr[4]); gr[5] = fmaf(c, y.y, gr[5]); gr[6] = fmaf(c, y.z, gr[6]); gr[7] = fmaf(c, y.w, gr[7]);
          }
        }
      }
      if (has) {
        float4* o = reinterpret_cast<float4*>(g_regions + r * D + lane * 8);
        if (qc0 == 0) {
          o[0] = make_float4(gr[0], gr[1], gr[2], gr[3]);
          o[1] = make_float4(gr[4], gr[5], gr[6], gr[7]);
        } else {
          float4 p0 = o[0], p1 = o[1];
          o[0] = make_float4(p0.x + gr[0], p0.y + gr[1], p0.z + gr[2], p0.w + gr[3]);
          o[1] = make_float4(p1.x + gr[4], p1.y + gr[5], p1.z + gr[6], p1.w + gr[7]);
        }
      }
    }
  }
}

// g_queries[i] = sum_p qpart[p][i]: block (32, 8) -- 8 thread rows split the partials, fixed-order smem fold.
// With g_scale, block 0 also folds lspart [nparts][Nq] (partials in CTA order per query, then the queries in a fixed
// tree) into the logit-scale gradient *g_scale = g_loss[0] * g_mul / Nq * sum.
__global__ void __launch_bounds__(256) infonce_bwd_q_kernel(const float* __restrict__ qpart, int nparts, long long n, float* __restrict__ g_queries,
                                                            const float* __restrict__ lspart, int Nq, const float* __restrict__ g_loss,
                                                            float g_mul, float* __restrict__ g_scale) {
  __shared__ float red[8][33];
  const long long i = (long long)blockIdx.x * 32 + threadIdx.x;
  float t = 0.f;
  if (g_queries) {
    if (i < n)
      for (int p = threadIdx.y; p < nparts; p += 8) t += qpart[(long long)p * n + i];
    red[threadIdx.y][threadIdx.x] = t;
    __syncthreads();
    if (threadIdx.y == 0 && i < n) {
      float a = 0.f;
#pragma unroll
      for (int y = 0; y < 8; ++y) a += red[y][threadIdx.x];
      g_queries[i] = a;
    }
  }
  if (g_scale && blockIdx.x == 0) {
    __shared__ float ls_red[256];
    const int tid = threadIdx.y * 32 + threadIdx.x;
    float v = 0.f;
    for (int q = tid; q < Nq; q += 256) {
      float s = 0.f;
      for (int p = 0; p < nparts; ++p) s += lspart[(long long)p * Nq + q];
      v += s;
    }
    ls_red[tid] = v;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
      if (tid < o) ls_red[tid] += ls_red[tid + o];
      __syncthreads();
    }
    if (tid == 0) g_scale[0] = ls_red[0] * (g_loss[0] * g_mul / (float)Nq);
  }
}

// ---- top-k: radix select on the prefilter scores, exact fp64 re-score, bitonic sort -----------------------
constexpr int kTopkMaxCand = 512;

__device__ __forceinline__ uint32_t fkey(float x) {
  const uint32_t u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__global__ void __launch_bounds__(256) topk_kernel(const float* __restrict__ S, const bf16* __restrict__ regions, const bf16* __restrict__ queries,
                                                   int Nr, int D, int k, int ncand, long long* __restrict__ idx_out,
                                                   float* __restrict__ score_out) {
  __shared__ unsigned hist[256];
  __shared__ unsigned sel_prefix, sel_remaining, n_gt, n_eq, warp_off[9];
  __shared__ unsigned long long cand[kTopkMaxCand];
  __shared__ int cand_idx[kTopkMaxCand];
  const int q = blockIdx.x;
  const float* row = S + (long long)q * Nr;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  // 1. radix select: key of the ncand-th largest prefilter score
  if (threadIdx.x == 0) { sel_prefix = 0; sel_remaining = (unsigned)ncand; }
  __syncthreads();
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    hist[threadIdx.x] = 0;
    __syncthreads();
    const unsigned prefix = sel_prefix;
    const unsigned mask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
    for (int r = threadIdx.x; r < Nr; r += blockDim.x) {
      const unsigned key = fkey(row[r]);
      if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (warp == 0) {
      // digit = largest d with (count of keys whose digit > d) < remaining: warp-parallel suffix scan over
      // the 256 bins (lane l owns bins 8l..8l+7, higher lanes = higher digits)
      const unsigned rem = sel_remaining;
      unsigned c[8], own = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) { c[j] = hist[lane * 8 + j]; own += c[j]; }
      // inclusive suffix sum of `own` over lanes
      unsigned suf = own;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned v = __shfl_down_sync(0xffffffffu, suf, o);
        if (lane + o < 32) suf += v;
      }
      const unsigned above = suf - own;                     // keys in bins of higher lanes
      // the selected digit lies in the unique lane with above < rem <= above + own
      const bool mine = above < rem && rem <= above + own;
      if (mine) {
        unsigned acc = above;
        int d = 7;
        for (; d > 0; --d) {
          if (acc + c[d] >= rem) break;
          acc += c[d];
        }
        sel_prefix = prefix | ((unsigned)(lane * 8 + d) << shift);
        sel_remaining = rem - acc;   // how many of the threshold-digit keys are still needed
      }
    }
    __syncthreads();
  }
  const unsigned T = sel_prefix;
  const unsigned need_eq = sel_remaining;   // number of keys == T to take (smallest indices first)

  // 2. collect: all keys > T (any order), then the first `need_eq` keys == T in index order
  if (threadIdx.x == 0) { n_gt = 0; n_eq = 0; }
  __syncthreads();
  for (int r0 = 0; r0 < Nr; r0 += blockDim.x) {
    const int r = r0 + threadIdx.x;
    const unsigned key = r < Nr ? fkey(row[r]) : 0u;
    const bool gt = r < Nr && key > T, eq = r < Nr && key == T;
    if (gt) {
      const unsigned slot = atomicAdd(&n_gt, 1u);
      if (slot < (unsigned)kTopkMaxCand) cand_idx[slot] = r;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, eq);
    if (lane == 0) warp_off[warp] = __popc(bal);
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned run = n_eq;
      for (int w = 0; w < 8; ++w) { const unsigned c = warp_off[w]; warp_off[w] = run; run += c; }
      warp_off[8] = run;
    }
    __syncthreads();
    if (eq) {
      const unsigned pos = warp_off[warp] + __popc(bal & ((1u << lane) - 1u));
      if (pos < need_eq) cand_idx[ncand - need_eq + pos] = r;
    }
    __syncthreads();
    if (threadIdx.x == 0) n_eq = warp_off[8];
    __syncthreads();
  }

  // 3. exact re-score (fp64 accumulation of exact bf16 products, rounded once to fp32) and sort key
  int npow = 1;
  while (npow < ncand) npow <<= 1;
  for (int c = threadIdx.x; c < npow; c += blockDim.x) cand[c] = 0ull;   // padding sorts last
  __syncthreads();
  // one warp per candidate: lanes take 8-element slices of the row pair, fp64 FMA, fixed-order butterfly
  for (int c = warp; c < ncand; c += 8) {
    const int r = cand_idx[c];
    double acc = 0.0;
    for (int d0 = lane * 8; d0 < D; d0 += 256) {
      const uint4 qa = *reinterpret_cast<const uint4*>(queries + (long long)q * D + d0);
      const uint4 ra = *reinterpret_cast<const uint4*>(regions + (long long)r * D + d0);
      const uint32_t qw[4] = {qa.x, qa.y, qa.z, qa.w}, rw[4] = {ra.x, ra.y, ra.z, ra.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        acc += (double)bf16lo(qw[j]) * (double)bf16lo(rw[j]);
        acc += (double)bf16hi(qw[j]) * (double)bf16hi(rw[j]);
      }
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      const float sc = (float)acc;
      cand[c] = ((unsigned long long)fkey(sc) << 32) | (unsigned long long)(0xffffffffu - (unsigned)r);
    }
  }
  __syncthreads();
  // bitonic sort, descending on (score, -index)
  for (int size = 2; size <= npow; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = threadIdx.x; i < npow; i += blockDim.x) {
        const int j = i ^ stride;
        if (j > i) {
          const bool desc = (i & size) == 0;
          const unsigned long long a = cand[i], b = cand[j];
          if ((a < b) == desc) { cand[i] = b; cand[j] = a; }
        }
      }
      __syncthreads();
    }
  }
  for (int c = threadIdx.x; c < k; c += blockDim.x) {
    const unsigned long long key = cand[c];
    const unsigned fk = (unsigned)(key >> 32);
    const unsigned u = (fk & 0x80000000u) ? (fk & 0x7fffffffu) : ~fk;
    idx_out[(long long)q * k + c] = (long long)(0xffffffffu - (unsigned)(key & 0xffffffffu));
    score_out[(long long)q * k + c] = __uint_as_float(u);
  }
}

}  // namespace cor

namespace cor {
int launch_lse_combine(const float* part, int Nq, int nparts, int qt, float* lse, cudaStream_t st) {
  sim_lse_combine_kernel<<<ceil_div(Nq, 8), 256, 0, st>>>(part, Nq, nparts, qt, lse);
  return check_launch("sim_lse_combine_kernel");
}
}  // namespace cor

using namespace cor;

static int stream_region_ctas(int Nr) {
  int c = sm_count() * 2;
  const int need = ceil_div(Nr, 8);
  return c < need ? c : need;
}

extern "C" size_t cor_sim_work_bytes(int Nq, int Nr, int D) {
  // LSE partials (either producer) and the g_queries partials of the streaming backward
  const size_t ctas = (size_t)sm_count() * 2 + 1024;
  const size_t lse_part = (size_t)ceil_div(Nq, kQT) * ctas * 256 * 2 * sizeof(float);
  const size_t qpart = ctas * (size_t)Nq * (D + 1) * sizeof(float);     // + the logit-scale partials [ctas][Nq]
  (void)Nr;
  return (lse_part > qpart ? lse_part : qpart) + 256;
}

extern "C" int cor_l2_normalize(const void* x, int x_dtype, int n, int D, float* y_f32, void* y_bf16, float* inv_norm,
                                cor_stream_t stream) {
  COR_REQUIRE(x && (y_f32 || y_bf16) && n > 0 && D > 0, "cor_l2_normalize: bad arguments");
  if (x_dtype == COR_F32) l2_normalize_kernel<float><<<n, 128, 0, as_stream(stream)>>>((const float*)x, D, y_f32, (bf16*)y_bf16, inv_norm);
  else if (x_dtype == COR_BF16) l2_normalize_kernel<bf16><<<n, 128, 0, as_stream(stream)>>>((const bf16*)x, D, y_f32, (bf16*)y_bf16, inv_norm);
  else COR_REQUIRE(false, "cor_l2_normalize: unsupported dtype %d", x_dtype);
  return check_launch("l2_normalize_kernel");
}

static int sim_stream_launch(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, const float* scale, float* S,
                             float* lse, void* work, int* nparts, int* qt, cudaStream_t st) {
  const bool want_lse = lse || nparts;
  COR_REQUIRE(regions && queries && (S || want_lse), "cor_sim_stream: null pointer");
  COR_REQUIRE(Nr > 0 && Nq > 0 && D > 0 && D % 8 == 0, "cor_sim_stream: need D %% 8 == 0 (D=%d)", D);
  COR_REQUIRE(!want_lse || work, "cor_sim_stream: lse needs a work buffer");
  COR_REQUIRE((((uintptr_t)regions) & 15) == 0, "cor_sim_stream: regions must be 16-byte aligned");
  const size_t smem = (size_t)kQT * D * sizeof(float);
  COR_REQUIRE(smem <= 96 * 1024, "cor_sim_stream: D=%d too large", D);
  COR_CUDA(cudaFuncSetAttribute(sim_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int ctas = stream_region_ctas(Nr), qtiles = ceil_div(Nq, kQT);
  float* part = want_lse ? (float*)work : nullptr;
  sim_stream_kernel<<<dim3(ctas, qtiles), 256, smem, st>>>((const bf16*)regions, (const bf16*)queries, Nr, Nq, D, inv_tau, scale, S, part);
  int rc = check_launch("sim_stream_kernel");
  if (rc || !want_lse) return rc;
  if (nparts) {                       // deferred: the caller merges the partials (cor_infonce_tail)
    *nparts = ctas;
    *qt = kQT;
    return COR_OK;
  }
  return launch_lse_combine(part, Nq, ctas, kQT, lse, st);
}

extern "C" int cor_sim_stream_fwd(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, float* S,
                                  float* lse, void* work, cor_stream_t stream) {
  return sim_stream_launch(regions, queries, Nr, Nq, D, inv_tau, nullptr, S, lse, work, nullptr, nullptr, as_stream(stream));
}

extern "C" int cor_sim_stream_fwd_ls(const void* regions, const void* queries, int Nr, int Nq, int D, const float* logit_scale, float* S,
                                     float* lse, void* work, cor_stream_t stream) {
  COR_REQUIRE(logit_scale, "cor_sim_stream_fwd_ls: null logit_scale");
  return sim_stream_launch(regions, queries, Nr, Nq, D, 0.f, logit_scale, S, lse, work, nullptr, nullptr, as_stream(stream));
}

static int sim_lse_parts(int engine, const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, const float* scale,
                         void* work, int* nparts, int* qt, cor_stream_t stream) {
  COR_REQUIRE(nparts && qt, "cor_sim_lse_parts: null pointer");
  if (engine == 1)
    return cor::sim_umma_launch(regions, queries, Nr, Nq, D, inv_tau, scale, nullptr, nullptr, work, nparts, qt, as_stream(stream));
  COR_REQUIRE(engine == 0, "cor_sim_lse_parts: engine %d (0 = stream, 1 = umma)", engine);
  return sim_stream_launch(regions, queries, Nr, Nq, D, inv_tau, scale, nullptr, nullptr, work, nparts, qt, as_stream(stream));
}

extern "C" int cor_sim_lse_parts(int engine, const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, void* work,
                                 int* nparts, int* qt, cor_stream_t stream) {
  return sim_lse_parts(engine, regions, queries, Nr, Nq, D, inv_tau, nullptr, work, nparts, qt, stream);
}

extern "C" int cor_sim_lse_parts_ls(int engine, const void* regions, const void* queries, int Nr, int Nq, int D, const float* logit_scale,
                                    void* work, int* nparts, int* qt, cor_stream_t stream) {
  COR_REQUIRE(logit_scale, "cor_sim_lse_parts_ls: null logit_scale");
  return sim_lse_parts(engine, regions, queries, Nr, Nq, D, 0.f, logit_scale, work, nparts, qt, stream);
}

static int infonce_tail(const float* lse_part, int nparts, int qt, const void* regions, const void* queries, const long long* targets, int Nr,
                        int Nq, int D, float inv_tau, const float* scale, float* lse, float* nce, float* tgt_logit, const float* seg,
                        const float* fgbg, float w_fg, float w_bg, float w_nce, float* total, cor_stream_t stream) {
  COR_REQUIRE(lse_part && regions && queries && targets && lse && nce && tgt_logit, "cor_infonce_tail: null pointer");
  COR_REQUIRE(nparts > 0 && qt > 0 && Nr > 0 && Nq > 0 && D > 0, "cor_infonce_tail: bad sizes");
  COR_REQUIRE(!total || (seg && fgbg), "cor_infonce_tail: total needs seg and fgbg");
  infonce_tail_kernel<<<1, 1024, 0, as_stream(stream)>>>(lse_part, nparts, qt, (const bf16*)regions, (const bf16*)queries, targets, Nr, Nq, D,
                                                        inv_tau, scale, lse, nce, tgt_logit, seg, fgbg, w_fg, w_bg, w_nce, total);
  return check_launch("infonce_tail_kernel");
}

extern "C" int cor_infonce_tail(const float* lse_part, int nparts, int qt, const void* regions, const void* queries,
                                const long long* targets, int Nr, int Nq, int D, float inv_tau, float* lse, float* nce, float* tgt_logit,
                                const float* seg, const float* fgbg, float w_fg, float w_bg, float w_nce, float* total,
                                cor_stream_t stream) {
  return infonce_tail(lse_part, nparts, qt, regions, queries, targets, Nr, Nq, D, inv_tau, nullptr, lse, nce, tgt_logit, seg, fgbg, w_fg,
                      w_bg, w_nce, total, stream);
}

extern "C" int cor_infonce_tail_ls(const float* lse_part, int nparts, int qt, const void* regions, const void* queries,
                                   const long long* targets, int Nr, int Nq, int D, const float* logit_scale, float* lse, float* nce,
                                   float* tgt_logit, const float* seg, const float* fgbg, float w_fg, float w_bg, float w_nce, float* total,
                                   cor_stream_t stream) {
  COR_REQUIRE(logit_scale, "cor_infonce_tail_ls: null logit_scale");
  return infonce_tail(lse_part, nparts, qt, regions, queries, targets, Nr, Nq, D, 0.f, logit_scale, lse, nce, tgt_logit, seg, fgbg, w_fg,
                      w_bg, w_nce, total, stream);
}

static int infonce_fwd(const void* regions, const void* queries, const long long* targets, const float* lse, int Nr, int Nq, int D,
                       float inv_tau, const float* scale, float* loss, float* tgt_logit, cor_stream_t stream) {
  COR_REQUIRE(regions && queries && targets && lse && loss && tgt_logit, "cor_infonce_fwd: null pointer");
  infonce_fwd_kernel<<<1, 1024, 0, as_stream(stream)>>>((const bf16*)regions, (const bf16*)queries, targets, lse, Nr, Nq, D, inv_tau,
                                                       scale, loss, tgt_logit);
  return check_launch("infonce_fwd_kernel");
}

extern "C" int cor_infonce_fwd(const void* regions, const void* queries, const long long* targets, const float* lse, int Nr,
                               int Nq, int D, float inv_tau, float* loss, float* tgt_logit, cor_stream_t stream) {
  return infonce_fwd(regions, queries, targets, lse, Nr, Nq, D, inv_tau, nullptr, loss, tgt_logit, stream);
}

extern "C" int cor_infonce_fwd_ls(const void* regions, const void* queries, const long long* targets, const float* lse, int Nr,
                                  int Nq, int D, const float* logit_scale, float* loss, float* tgt_logit, cor_stream_t stream) {
  COR_REQUIRE(logit_scale, "cor_infonce_fwd_ls: null logit_scale");
  return infonce_fwd(regions, queries, targets, lse, Nr, Nq, D, 0.f, logit_scale, loss, tgt_logit, stream);
}

static int infonce_bwd(const void* regions, const void* queries, const long long* targets, const float* lse, int Nr, int Nq, int D,
                       float inv_tau, const float* scale, const float* g_loss, float g_mul, float* g_regions, float* g_queries,
                       float* g_scale, void* work, cor_stream_t stream) {
  COR_REQUIRE(regions && queries && targets && lse && g_loss && (g_regions || g_queries || g_scale), "cor_infonce_bwd: null pointer");
  COR_REQUIRE(!(g_queries || g_scale) || work, "cor_infonce_bwd: g_queries / g_logit_scale need a work buffer");
  COR_REQUIRE(D % 8 == 0 && D <= 256, "cor_infonce_bwd: streaming backward supports D %% 8 == 0 and D <= 256 (D=%d)", D);
  COR_REQUIRE((((uintptr_t)regions) & 15) == 0 && (((uintptr_t)g_regions) & 15) == 0, "cor_infonce_bwd: 16-byte alignment required");
  cudaStream_t st = as_stream(stream);
  int ctas = sm_count();
  const int need = ceil_div(Nr, 8);
  if (ctas > need) ctas = need;
  if (!g_queries && !g_scale) {
    const size_t smem_r = (size_t)kRQ * D * sizeof(float);
    COR_CUDA(cudaFuncSetAttribute(infonce_bwd_regions_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_r));
    infonce_bwd_regions_kernel<<<ctas, 256, smem_r, st>>>((const bf16*)regions, (const bf16*)queries, targets, lse, Nr, Nq, D, inv_tau,
                                                         scale, g_loss, g_mul, g_regions);
    return check_launch("infonce_bwd_regions_kernel");
  }
  const size_t smem = (size_t)(kQT * D + 8 * kQT * D) * sizeof(float);
  // work: qpart [ctas][Nq][D], then (logit-scale gradient wanted) lspart [ctas][Nq]
  float* lspart = g_scale ? (float*)work + (size_t)ctas * Nq * D : nullptr;
  if (g_regions) {
    COR_CUDA(cudaFuncSetAttribute(infonce_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    infonce_bwd_kernel<true><<<ctas, 256, smem, st>>>((const bf16*)regions, (const bf16*)queries, targets, lse, Nr, Nq, D, inv_tau, scale,
                                                     g_loss, g_mul, g_regions, (float*)work, lspart);
  } else {
    COR_CUDA(cudaFuncSetAttribute(infonce_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    infonce_bwd_kernel<false><<<ctas, 256, smem, st>>>((const bf16*)regions, (const bf16*)queries, targets, lse, Nr, Nq, D, inv_tau, scale,
                                                      g_loss, g_mul, nullptr, (float*)work, lspart);
  }
  int rc = check_launch("infonce_bwd_kernel");
  if (rc) return rc;
  const long long n = (long long)Nq * D;
  infonce_bwd_q_kernel<<<ceil_div(n, 32), dim3(32, 8), 0, st>>>((const float*)work, ctas, n, g_queries, lspart, Nq, g_loss, g_mul, g_scale);
  return check_launch("infonce_bwd_q_kernel");
}

extern "C" int cor_infonce_bwd(const void* regions, const void* queries, const long long* targets, const float* lse, int Nr,
                               int Nq, int D, float inv_tau, const float* g_loss, float g_mul, float* g_regions, float* g_queries,
                               void* work, cor_stream_t stream) {
  return infonce_bwd(regions, queries, targets, lse, Nr, Nq, D, inv_tau, nullptr, g_loss, g_mul, g_regions, g_queries, nullptr, work, stream);
}

extern "C" int cor_infonce_bwd_ls(const void* regions, const void* queries, const long long* targets, const float* lse, int Nr,
                                  int Nq, int D, const float* logit_scale, const float* g_loss, float g_mul, float* g_regions,
                                  float* g_queries, float* g_logit_scale, void* work, cor_stream_t stream) {
  COR_REQUIRE(logit_scale, "cor_infonce_bwd_ls: null logit_scale");
  return infonce_bwd(regions, queries, targets, lse, Nr, Nq, D, 0.f, logit_scale, g_loss, g_mul, g_regions, g_queries, g_logit_scale, work,
                     stream);
}

extern "C" int cor_topk(const float* S, const void* regions, const void* queries, int Nr, int Nq, int D, int k, long long* idx,
                        float* score, cor_stream_t stream) {
  COR_REQUIRE(S && regions && queries && idx && score, "cor_topk: null pointer");
  COR_REQUIRE(k > 0 && k <= Nr && k <= 256, "cor_topk: need 0 < k <= min(Nr, 256) (k=%d, Nr=%d)", k, Nr);
  int slack = k / 2 < 16 ? 16 : k / 2;
  int ncand = k + slack;
  if (ncand > Nr) ncand = Nr;
  if (ncand > kTopkMaxCand) ncand = kTopkMaxCand;
  topk_kernel<<<Nq, 256, 0, as_stream(stream)>>>(S, (const bf16*)regions, (const bf16*)queries, Nr, D, k, ncand, idx, score);
  return check_launch("topk_kernel");
}
