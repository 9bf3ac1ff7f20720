// The fused step's chain after the pooling GEMM and before the pooling-backward GEMM, one launch each way
// (cor_b200/region.py, single-rank path, bg_mode 0).
//
// At the benched shape (16 queries x 1024 region rows x 256 channels) the kernels this replaces -- row epilogue,
// similarity, log-sum-exp merge, fg/bg losses forward; InfoNCE backward, fg/bg backward, epilogue backward, operand cast
// -- each touch a few MB resident in L2 and are latency-bound: the step paid a launch-and-drain per kernel.  Here every
// region row is owned by one warp (8 channels per lane, C <= 256) from the split-K partials to the unit row, its bf16
// copy and its 16 scores; everything that needs all rows (log-sum-exp merge, fg/bg column statistics, losses) is done
// by the last CTA to finish.  Arithmetic is that of rows_finalize_kernel, sim_stream_kernel, infonce_tail_kernel,
// fgbg_rows/reduce/bwd_kernel, infonce_bwd_kernel and rows_finalize_bwd_kernel; only the order of some fp32 sums
// differs.  Deterministic: no float atomics, every fold in a fixed order.
#include "common.cuh"

namespace cor {

namespace {

constexpr float kDenEps = 1e-8f;    // eps added to the pooling denominator (cor_rows_finalize's eps in region.py)
constexpr float kCosEps = 1e-8f;    // F.cosine_similarity default eps (fgbg_loss.cu)
constexpr int kTailRowsQ = 64;      // region rows per dQ CTA of the backward: 8 per warp, held in registers
constexpr int kCounterWords = 32;   // [0]: forward; [1 + q]: backward query q; [1 + kQT]: backward, all queries (logit scale)

__device__ __forceinline__ void load8(const float* p, float (&v)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void store8(float* p, const float (&v)[8]) {
  reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void unpack8(uint4 raw, float (&f)[8]) {
  f[0] = bf16lo(raw.x); f[1] = bf16hi(raw.x); f[2] = bf16lo(raw.y); f[3] = bf16hi(raw.y);
  f[4] = bf16lo(raw.z); f[5] = bf16hi(raw.z); f[6] = bf16lo(raw.w); f[7] = bf16hi(raw.w);
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
  return make_uint4(pack2(v[0], v[1]), pack2(v[2], v[3]), pack2(v[4], v[5]), pack2(v[6], v[7]));
}

// qs[q][c] = queries[q][c] as f32 for q < nq, 0 up to kQT rows: 16-byte loads, all in flight at once
__device__ __forceinline__ void fill_queries(float* qs, const bf16* q16, int nq, int C) {
  const int nvec = kQT * C / 8;
  for (int i = threadIdx.x; i < nvec; i += blockDim.x) {
    float f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (i * 8 / C < nq) unpack8(*reinterpret_cast<const uint4*>(q16 + (long long)i * 8), f);
    reinterpret_cast<float4*>(qs)[2 * i] = make_float4(f[0], f[1], f[2], f[3]);
    reinterpret_cast<float4*>(qs)[2 * i + 1] = make_float4(f[4], f[5], f[6], f[7]);
  }
}

// sum[e] = p[0][e] + p[1][e] + ... + p[n-1][e] (copies `stride` floats apart) in that order; four copies in flight per step
__device__ __forceinline__ void sum_splits(const float* p, int n, long long stride, float (&sum)[8]) {
#pragma unroll
  for (int e = 0; e < 8; ++e) sum[e] = 0.f;
  for (int k0 = 0; k0 < n; k0 += 4) {
    float t[4][8];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (k0 + u < n) load8(p + (k0 + u) * stride, t[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (k0 + u < n)
#pragma unroll
        for (int e = 0; e < 8; ++e) sum[e] += t[u][e];
  }
}

}  // namespace

struct StepTailFwd {
  const float* part; int nsplit; long long split_stride; long long img_stride; int B, M, C; float p_total;
  const float* stats; const bf16* q16; const float* comb; const long long* targets; float inv_tau; const float* scale;
  const float* seg; float w_fg, w_bg, w_nce;
  float* fg; bf16* fg16; float* inv_fg; float* bg; float* inv_bg; float* out4; float* aux;
  float* lse; float* nce; float* tgt; float* total; float* lse_part; unsigned* counter;
  const float* mem_part; int mem_nparts; const int* mem_state;     // region memory's scan partials (cor_memory_scan) or NULL
};

// grid = ceil(B*M / 8), block = 256 (warp per region row), dynamic smem = kQT * C floats.
__global__ void __launch_bounds__(256, 1) step_tail_fwd_kernel(const StepTailFwd a) {
  extern __shared__ float qs[];   // [kQT][C] queries, bf16 values as f32
  __shared__ float cm[8][kQT], cs[8][kQT];
  __shared__ double dscratch[32];
  __shared__ float lse_s[kQT];
  __shared__ bool last;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int C = a.C, M = a.M, Nq = a.B, Nr = a.B * a.M;
  const float inv_tau = a.scale ? __ldg(a.scale) : a.inv_tau;
  fill_queries(qs, a.q16, Nq, C);
  const bool has = lane * 8 < C;
  const int c0 = lane * 8;
  float m_run = -INFINITY, s_run = 0.f;
  const int r = blockIdx.x * 8 + warp;
  const int b = r / M, mi = r - b * M;
  // 1. split-K sum (fixed order) / denominator, L2-normalise: rows_finalize_kernel
  float sum[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, v[8], y[8];
  const float d = r < Nr ? a.stats[(long long)r * 4 + 3] : 0.f;
  if (has && r < Nr) sum_splits(a.part + b * a.img_stride + (long long)mi * C + c0, a.nsplit, a.split_stride, sum);
  __syncthreads();   // queries in shared memory
  if (r < Nr) {
    float ss = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) { v[e] = sum[e] / (d + kDenEps); ss += v[e] * v[e]; }
    const float inv = 1.f / fmaxf(sqrtf(warp_sum(ss)), 1e-12f);
    float fb[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { y[e] = v[e] * inv; fb[e] = __bfloat162float(__float2bfloat16_rn(y[e])); }
    if (has) {
      store8(a.fg + (long long)r * C + c0, y);
      *reinterpret_cast<uint4*>(a.fg16 + (long long)r * C + c0) = pack8(y);
    }
    if (lane == 0) a.inv_fg[r] = inv;
    // 2. the row's 16 scores from its bf16 copy (sim_stream_kernel's per-lane order and transposed reduce)
    float s[kQT];
#pragma unroll
    for (int q = 0; q < kQT; ++q) {
      s[q] = 0.f;
      if (has) {
        const float4 x = *reinterpret_cast<const float4*>(&qs[q * C + c0]);
        const float4 z = *reinterpret_cast<const float4*>(&qs[q * C + c0 + 4]);
        s[q] = fmaf(fb[0], x.x, s[q]); s[q] = fmaf(fb[1], x.y, s[q]); s[q] = fmaf(fb[2], x.z, s[q]); s[q] = fmaf(fb[3], x.w, s[q]);
        s[q] = fmaf(fb[4], z.x, s[q]); s[q] = fmaf(fb[5], z.y, s[q]); s[q] = fmaf(fb[6], z.z, s[q]); s[q] = fmaf(fb[7], z.w, s[q]);
      }
    }
    const float sv = transpose_reduce16(s, lane);
    if (lane < Nq) {           // lane < kQT: lane l holds query l
      m_run = sv * inv_tau;
      s_run = 1.f;
      if (a.targets[lane] == r) a.tgt[lane] = sv;
    }
    // 3. the ground-truth row of triplet b: its background row and the fg / bg cosine statistics (fgbg_rows_kernel)
    if (mi == 0) {
      float g[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, x[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      const float db = a.p_total - d;
      float ssb = 0.f;
      if (has) {
        float all[8];   // the all-ones weight row: sum_p F
        sum_splits(a.part + b * a.img_stride + (long long)M * C + c0, a.nsplit, a.split_stride, all);
#pragma unroll
        for (int e = 0; e < 8; ++e) { g[e] = (all[e] - sum[e]) / (db + kDenEps); ssb += g[e] * g[e]; }
        load8(a.comb + (long long)b * C + c0, x);
      }
      const float invb = 1.f / fmaxf(sqrtf(warp_sum(ssb)), 1e-12f);
      float st[5] = {0.f, 0.f, 0.f, 0.f, 0.f};   // f.q, g.q, f.f, g.g, q.q
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        g[e] *= invb;
        st[0] = fmaf(y[e], x[e], st[0]); st[1] = fmaf(g[e], x[e], st[1]); st[2] = fmaf(y[e], y[e], st[2]);
        st[3] = fmaf(g[e], g[e], st[3]); st[4] = fmaf(x[e], x[e], st[4]);
      }
#pragma unroll
      for (int k = 0; k < 5; ++k) st[k] = warp_sum(st[k]);
      if (has) store8(a.bg + (long long)b * C + c0, g);
      if (lane == 0) {
        a.inv_bg[b] = invb;
        const float nf = fmaxf(sqrtf(st[2]), kCosEps), nb = fmaxf(sqrtf(st[3]), kCosEps), nq = fmaxf(sqrtf(st[4]), kCosEps);
        float* o = a.aux + (long long)b * 8;
        o[0] = st[0] / (nf * nq);
        o[1] = st[1] / (nb * nq);
        o[2] = nf; o[3] = nb; o[4] = nq;
        o[5] = a.stats[(long long)r * 4 + 0] > 0.f ? 1.f : 0.f;
        o[6] = a.stats[(long long)r * 4 + 1] > 0.f ? 1.f : 0.f;
        o[7] = 0.f;
      }
    }
  }
  // this CTA's log-sum-exp partial per query (sim_stream_kernel's layout with qt = kQT)
  if (lane < kQT) { cm[warp][lane] = m_run; cs[warp][lane] = s_run; }
  __syncthreads();
  if (threadIdx.x < kQT) {
    float Mx = -INFINITY;
    for (int w = 0; w < 8; ++w) Mx = fmaxf(Mx, cm[w][threadIdx.x]);
    float S = 0.f;
    for (int w = 0; w < 8; ++w) S += (cm[w][threadIdx.x] == -INFINITY) ? 0.f : cs[w][threadIdx.x] * __expf(cm[w][threadIdx.x] - Mx);
    float* o = a.lse_part + ((long long)blockIdx.x * kQT + threadIdx.x) * 2;
    o[0] = Mx; o[1] = S;
  }
  if (!arrive_last(a.counter, gridDim.x, &last)) return;

  // ---- last CTA: log-sum-exp merge and InfoNCE (infonce_tail_kernel), fg / bg losses (fgbg_reduce_kernel), total ----
  // 16 threads per query merge the CTAs' partials (thread j takes parts j, j + 16, ...; 8 in flight), fixed-order folds
  __shared__ float rs_s[kQT][8], tgt_s[kQT];
  if (threadIdx.x < kQT * 8) rs_s[threadIdx.x >> 3][threadIdx.x & 7] = (threadIdx.x >> 3) < Nq ? __ldcg(a.aux + threadIdx.x) : 0.f;
  if (threadIdx.x < kQT) tgt_s[threadIdx.x] = threadIdx.x < Nq ? __ldcg(a.tgt + threadIdx.x) : 0.f;
  {
    const int nparts = gridDim.x, q = threadIdx.x >> 4, j = threadIdx.x & 15;
    const float2* lp = reinterpret_cast<const float2*>(a.lse_part);
    float2 pv[8];
    float Mx = -INFINITY;
    for (int p0 = 0; p0 < nparts; p0 += 128) {
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int p = p0 + j + 16 * u;
        pv[u] = p < nparts ? __ldcg(lp + (long long)p * kQT + q) : make_float2(-INFINITY, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) Mx = fmaxf(Mx, pv[u].x);
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) Mx = fmaxf(Mx, __shfl_xor_sync(0xffffffffu, Mx, o));
    double acc = 0.0;
    for (int p0 = 0; p0 < nparts; p0 += 128) {
      if (nparts > 128) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int p = p0 + j + 16 * u;
          pv[u] = p < nparts ? __ldcg(lp + (long long)p * kQT + q) : make_float2(-INFINITY, 0.f);
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (pv[u].x != -INFINITY) acc += (double)(pv[u].y * expf(pv[u].x - Mx));
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    float l = Mx + logf((float)acc);
    // a region memory: its partials merged in after this batch's, only when it holds rows (an empty one changes no bit)
    if (a.mem_part && __ldcg(a.mem_state + 1) > 0) l = logaddexpf_(l, mem_lse<16>(a.mem_part, a.mem_nparts, q, j));
    if (j == 0 && q < Nq) {
      a.lse[q] = l;
      lse_s[q] = l;
    }
  }
  __syncthreads();
  // fg / bg counts and paired sums over the B ground-truth rows: every thread the same fixed-order loop
  double v0 = 0.0, nfg = 0.0, nbg = 0.0;
  for (int i = 0; i < Nq; ++i) {
    if (rs_s[i][5] > 0.f) { v0 += rs_s[i][0]; nfg += 1.0; }
    if (rs_s[i][6] > 0.f) nbg += 1.0;
  }
  // column statistics of the reference's broadcast bg cosine (bg_mode 0), one thread per channel
  double quirk[1] = {0.0};
  if (nbg > 0) {
    const float sq = sqrtf((float)nbg);
    float* colstat = a.aux + (long long)Nq * 8;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      float xs[kQT], qv[kQT];
#pragma unroll
      for (int i = 0; i < kQT; ++i) {
        xs[i] = i < Nq ? __ldcg(a.bg + (long long)i * C + c) : 0.f;
        qv[i] = i < Nq ? a.comb[(long long)i * C + c] : 0.f;
      }
      float A = 0.f, S1 = 0.f, ss = 0.f;
#pragma unroll
      for (int i = 0; i < kQT; ++i) {
        if (i < Nq && rs_s[i][6] > 0.f) {
          A += xs[i] / fmaxf(sq * fabsf(xs[i]), kCosEps);
          S1 += qv[i];
          ss = fmaf(qv[i], qv[i], ss);
        }
      }
      const float s2 = fmaxf(sqrtf(ss), kCosEps);
      colstat[c] = A; colstat[C + c] = S1; colstat[2 * C + c] = s2;
      quirk[0] += (double)(A * S1 / s2);
    }
  }
  block_sum<1>(quirk, dscratch);
  if (threadIdx.x == 0) {
    double acc = 0.0;
    for (int q = 0; q < Nq; ++q) acc += (double)lse_s[q] - (double)tgt_s[q] * (double)inv_tau;
    const float nce = (float)(acc / (double)Nq);
    const float fl = nfg > 0 ? (float)(1.0 - v0 / nfg) : 0.f;
    const float bl = nbg > 0 ? (float)(1.0 + quirk[0] / (nbg * (double)C)) : 0.f;
    a.out4[0] = fl; a.out4[1] = bl; a.out4[2] = (float)nfg; a.out4[3] = (float)nbg;
    a.nce[0] = nce;
    a.total[0] = a.seg[0] + a.w_fg * fl + a.w_bg * bl + a.w_nce * nce;
  }
}

struct StepTailBwd {
  const bf16* r16; const bf16* q16; const long long* targets; const float* lse; int B, M, C; float inv_tau; const float* scale;
  const float* g_loss; float w_nce; const float* fg; const float* inv_fg; const float* stats; const float* comb;
  const float* out4; const float* aux; float w_fg, w_bg;
  bf16* a16; int Kp; float* g_q; float* g_scale; float* qpart; float* lspart; float* lsq; unsigned* counter; int nreg, nsplit_q;
};

// grid = nreg region CTAs (warp per row: InfoNCE + fg-loss gradient of the row, epilogue backward, bf16 GEMM operand) +
// B * nsplit_q dQ CTAs (query q, kTailRowsQ rows each; the last of a query's CTAs folds the partials in split order).
// The logit-scale gradient sum_r (p_qr - [r == t(q)]) S_qr rides on the dQ CTAs: one partial per (query, split), folded in
// split order by the query's last CTA, and the last of those folds the queries in order into *g_scale.
// block = 256; dynamic smem = kQT * C floats.
__global__ void __launch_bounds__(256, 1) step_tail_bwd_kernel(const StepTailBwd a) {
  extern __shared__ float sm[];
  __shared__ bool last;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int C = a.C, M = a.M, Nq = a.B, Nr = a.B * a.M;
  const bool has = lane * 8 < C;
  const int c0 = lane * 8;
  const float g = a.g_loss[0];
  const float inv_tau = a.scale ? __ldg(a.scale) : a.inv_tau;
  const float gscale = g * a.w_nce * inv_tau / (float)Nq;
  const float nfg = a.out4[2], nbg = a.out4[3];
  if ((int)blockIdx.x < a.nreg) {
    float* qs = sm;   // [kQT][C]
    fill_queries(qs, a.q16, Nq, C);
    const int r = blockIdx.x * 8 + warp;
    uint4 raw = make_uint4(0u, 0u, 0u, 0u);
    if (has && r < Nr) raw = *reinterpret_cast<const uint4*>(a.r16 + (long long)r * C + c0);
    __syncthreads();
    if (r < Nr) {
      const int b = r / M, mi = r - b * M;
      float f[8];
      unpack8(raw, f);
      float s[kQT];
#pragma unroll
      for (int q = 0; q < kQT; ++q) {
        float t = 0.f;
        if (has) {
          const float4 x = *reinterpret_cast<const float4*>(&qs[q * C + c0]);
          const float4 y = *reinterpret_cast<const float4*>(&qs[q * C + c0 + 4]);
          t = f[0] * x.x + f[1] * x.y + f[2] * x.z + f[3] * x.w + f[4] * y.x + f[5] * y.y + f[6] * y.z + f[7] * y.w;
        }
        s[q] = t;
      }
      const float sv = transpose_reduce16(s, lane);
      float coef = 0.f;
      if (lane < Nq) {
        coef = __expf(sv * inv_tau - a.lse[lane]);
        if (a.targets[lane] == r) coef -= 1.f;
        coef *= gscale;
      }
      float gr[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int q = 0; q < kQT; ++q) {
        const float c = __shfl_sync(0xffffffffu, coef, q);
        if (has) {
          const float4 x = *reinterpret_cast<const float4*>(&qs[q * C + c0]);
          const float4 y = *reinterpret_cast<const float4*>(&qs[q * C + c0 + 4]);
          gr[0] = fmaf(c, x.x, gr[0]); gr[1] = fmaf(c, x.y, gr[1]); gr[2] = fmaf(c, x.z, gr[2]); gr[3] = fmaf(c, x.w, gr[3]);
          gr[4] = fmaf(c, y.x, gr[4]); gr[5] = fmaf(c, y.y, gr[5]); gr[6] = fmaf(c, y.z, gr[6]); gr[7] = fmaf(c, y.w, gr[7]);
        }
      }
      float y[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (has) load8(a.fg + (long long)r * C + c0, y);
      if (mi == 0) {            // fg-loss gradient of the ground-truth row (fgbg_bwd_kernel; bg_mode 0 puts none on bg rows)
        const float* rs = a.aux + (long long)b * 8;
        const float sf = (rs[5] > 0.f && nfg > 0.f) ? -(g * a.w_fg) / nfg : 0.f;
        const float cf = rs[0], nf = rs[2], nq = rs[4];
        float x[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (has) load8(a.comb + (long long)b * C + c0, x);
#pragma unroll
        for (int e = 0; e < 8; ++e) gr[e] = gr[e] + sf * (x[e] / (nf * nq) - cf * y[e] / (nf * nf));
      }
      // epilogue backward (rows_finalize_bwd_kernel): through the L2 normalisation and the denominator
      float dot = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) dot += gr[e] * y[e];
      dot = warp_sum(dot);
      const float inv = a.inv_fg[r], den = a.stats[(long long)r * 4 + 3] + kDenEps;
      float o[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = inv * (gr[e] - y[e] * dot) / den;
      if (has) *reinterpret_cast<uint4*>(a.a16 + ((long long)b * a.Kp + mi) * C + c0) = pack8(o);
    }
    // zero K-padding rows M..Kp-1 of every image
    const int pad = a.Kp - M;
    for (long long p = (long long)blockIdx.x * 8 + warp; p < (long long)Nq * pad; p += (long long)a.nreg * 8) {
      const long long b = p / pad, mi = M + p % pad;
      if (has) *reinterpret_cast<uint4*>(a.a16 + (b * a.Kp + mi) * C + c0) = make_uint4(0u, 0u, 0u, 0u);
    }
    return;
  }
  // ---- dQ: query q over rows [split * kTailRowsQ, +kTailRowsQ); warp w owns 8 of them, loaded once, kept in registers ----
  const int qb = blockIdx.x - a.nreg, q = qb / a.nsplit_q, split = qb - q * a.nsplit_q;
  float* red = sm;                  // [8][C]
  const int rw = split * kTailRowsQ + warp * 8;
  float qv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (has) unpack8(*reinterpret_cast<const uint4*>(a.q16 + (long long)q * C + c0), qv);
  uint4 raw[8];
#pragma unroll
  for (int u = 0; u < 8; ++u)
    raw[u] = (has && rw + u < Nr) ? *reinterpret_cast<const uint4*>(a.r16 + (long long)(rw + u) * C + c0) : make_uint4(0u, 0u, 0u, 0u);
  const float lq = a.lse[q];
  const long long tq = a.targets[q];
  // 1. this query's score against each of the warp's rows: eight independent butterflies; every lane ends with all eight
  float t[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    float f[8];
    unpack8(raw[u], f);
    t[u] = f[0] * qv[0] + f[1] * qv[1] + f[2] * qv[2] + f[3] * qv[3] + f[4] * qv[4] + f[5] * qv[5] + f[6] * qv[6] + f[7] * qv[7];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
#pragma unroll
    for (int u = 0; u < 8; ++u) t[u] += __shfl_xor_sync(0xffffffffu, t[u], o);
  // 2. sum_r coef[r] R[r] over the warp's rows in row order, then the 8 warp sums in warp order
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float ls = 0.f;                   // sum_r coef[r] S[r] / gscale over the warp's rows (the same in every lane)
  __shared__ float ls_w[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    if (rw + u < Nr) {
      float c = __expf(t[u] * inv_tau - lq);
      if (tq == rw + u) c -= 1.f;
      if (a.g_scale) ls = fmaf(c, t[u], ls);
      c *= gscale;
      float f[8];
      unpack8(raw[u], f);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] = fmaf(c, f[e], acc[e]);
    }
  }
  if (has) store8(red + warp * C + c0, acc);
  if (lane == 0) ls_w[warp] = ls;
  __syncthreads();
  if (a.g_q) {
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      float v = 0.f;
      for (int w = 0; w < 8; ++w) v += red[w * C + c];
      a.qpart[((long long)q * a.nsplit_q + split) * C + c] = v;
    }
  }
  if (a.g_scale && threadIdx.x == 0) {
    float v = 0.f;
    for (int w = 0; w < 8; ++w) v += ls_w[w];
    a.lspart[q * a.nsplit_q + split] = v;
  }
  if (!arrive_last(a.counter + q, a.nsplit_q, &last)) return;
  // last dQ CTA of query q: fold the splits in order, add the fg-loss and bg-quirk gradients (fgbg_bwd_kernel, bg_mode 0)
  const float* rs = a.aux + (long long)q * 8;
  const float sf = (rs[5] > 0.f && nfg > 0.f) ? -(g * a.w_fg) / nfg : 0.f;
  const float quirk = (rs[6] > 0.f && nbg > 0.f) ? (g * a.w_bg) / (nbg * (float)C) : 0.f;
  const float cf = rs[0], nf = rs[2], nq = rs[4];
  const float* colstat = a.aux + (long long)Nq * 8;
  for (int c = threadIdx.x; a.g_q && c < C; c += blockDim.x) {
    float t = 0.f;
    for (int k0 = 0; k0 < a.nsplit_q; k0 += 8) {      // eight partials in flight, added in split order
      float pk[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) pk[u] = k0 + u < a.nsplit_q ? __ldcg(a.qpart + ((long long)q * a.nsplit_q + k0 + u) * C + c) : 0.f;
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (k0 + u < a.nsplit_q) t += pk[u];
    }
    const float fv = a.fg[(long long)q * M * C + c], x = a.comb[(long long)q * C + c];
    float gq = sf * (fv / (nf * nq) - cf * x / (nq * nq));
    if (quirk != 0.f) {
      const float A = colstat[c], S1 = colstat[C + c], s2 = colstat[2 * C + c];
      gq += quirk * A * (1.f / s2 - S1 * x / (s2 * s2 * s2));
    }
    a.g_q[(long long)q * C + c] = t + gq;
  }
  if (!a.g_scale) return;
  if (threadIdx.x == 0) {
    float v = 0.f;
    for (int k = 0; k < a.nsplit_q; ++k) v += __ldcg(a.lspart + q * a.nsplit_q + k);
    a.lsq[q] = v;
  }
  if (!arrive_last(a.counter + 1 + kQT, Nq, &last)) return;
  // last query to finish: the queries in order, scaled like the InfoNCE term of the total loss
  if (threadIdx.x == 0) {
    float v = 0.f;
    for (int i = 0; i < Nq; ++i) v += __ldcg(a.lsq + i);
    a.g_scale[0] = v * (g * a.w_nce / (float)Nq);
  }
}

}  // namespace cor

using namespace cor;

static int tail_nsplit_q(int B, int M) { return ceil_div((long long)B * M, kTailRowsQ); }

extern "C" int cor_step_tail_counter_words(void) { return kCounterWords; }

extern "C" size_t cor_step_tail_work_bytes(int B, int M, int C) {
  if (B <= 0 || M <= 0 || C <= 0) return 0;
  const size_t fwd = (size_t)ceil_div((long long)B * M, 8) * kQT * 2 * sizeof(float);
  const size_t bwd = (size_t)B * tail_nsplit_q(B, M) * (C + 1) * sizeof(float) + kQT * sizeof(float);   // + logit-scale partials
  return fwd > bwd ? fwd : bwd;
}

static int tail_shape_ok(int B, int M, int C, const char* who) {
  COR_REQUIRE(B > 0 && B <= kQT && M > 0 && C > 0 && C % 8 == 0 && C <= 256,
              "%s: needs 1 <= B <= %d queries and C %% 8 == 0, C <= 256 (B=%d M=%d C=%d)", who, kQT, B, M, C);
  return COR_OK;
}

static int step_tail_fwd(const float* part, int nsplit, long long split_stride, int Rp, int B, int M, int C, float p_total,
                         const float* stats, const void* queries_bf16, const float* comb, const long long* targets, float inv_tau,
                         const float* scale, const float* seg, float w_fg, float w_bg, float w_nce, float* fg, void* fg_bf16, float* inv_fg,
                         float* bg, float* inv_bg, float* fgbg_out4, float* aux, float* lse, float* nce, float* tgt_logit, float* total,
                         void* work, unsigned* counter, cor_stream_t stream, const float* mem_part = nullptr, int mem_nparts = 0,
                         const int* mem_state = nullptr) {
  int rc = tail_shape_ok(B, M, C, "cor_step_tail_fwd");
  if (rc) return rc;
  COR_REQUIRE(!mem_part || (mem_state && mem_nparts > 0), "cor_step_tail_fwd_mem: memory partials need mem_state and mem_nparts > 0");
  COR_REQUIRE(part && stats && queries_bf16 && comb && targets && seg && fg && fg_bf16 && inv_fg && bg && inv_bg && fgbg_out4 && aux &&
                  lse && nce && tgt_logit && total && work && counter,
              "cor_step_tail_fwd: null pointer");
  COR_REQUIRE(nsplit >= 1 && Rp > M && split_stride % 4 == 0 && (((uintptr_t)part | (uintptr_t)fg | (uintptr_t)fg_bf16 | (uintptr_t)bg |
                                                                     (uintptr_t)comb) & 15) == 0,
              "cor_step_tail_fwd: bad partial layout or alignment (nsplit=%d Rp=%d M=%d)", nsplit, Rp, M);
  StepTailFwd a{part, nsplit, split_stride, (long long)Rp * C, B, M, C, p_total, stats, (const bf16*)queries_bf16, comb, targets, inv_tau,
                scale, seg, w_fg, w_bg, w_nce, fg, (bf16*)fg_bf16, inv_fg, bg, inv_bg, fgbg_out4, aux, lse, nce, tgt_logit, total,
                (float*)work, counter, mem_part, mem_nparts, mem_state};
  const int grid = ceil_div((long long)B * M, 8);
  step_tail_fwd_kernel<<<grid, 256, (size_t)kQT * C * sizeof(float), as_stream(stream)>>>(a);
  return check_launch("step_tail_fwd_kernel");
}

extern "C" int cor_step_tail_fwd(const float* part, int nsplit, long long split_stride, int Rp, int B, int M, int C, float p_total,
                                 const float* stats, const void* queries_bf16, const float* comb, const long long* targets, float inv_tau,
                                 const float* seg, float w_fg, float w_bg, float w_nce, float* fg, void* fg_bf16, float* inv_fg, float* bg,
                                 float* inv_bg, float* fgbg_out4, float* aux, float* lse, float* nce, float* tgt_logit, float* total,
                                 void* work, unsigned* counter, cor_stream_t stream) {
  return step_tail_fwd(part, nsplit, split_stride, Rp, B, M, C, p_total, stats, queries_bf16, comb, targets, inv_tau, nullptr, seg, w_fg, w_bg,
                       w_nce, fg, fg_bf16, inv_fg, bg, inv_bg, fgbg_out4, aux, lse, nce, tgt_logit, total, work, counter, stream);
}

extern "C" int cor_step_tail_fwd_ls(const float* part, int nsplit, long long split_stride, int Rp, int B, int M, int C, float p_total,
                                    const float* stats, const void* queries_bf16, const float* comb, const long long* targets,
                                    const float* logit_scale, const float* seg, float w_fg, float w_bg, float w_nce, float* fg, void* fg_bf16,
                                    float* inv_fg, float* bg, float* inv_bg, float* fgbg_out4, float* aux, float* lse, float* nce,
                                    float* tgt_logit, float* total, void* work, unsigned* counter, cor_stream_t stream) {
  COR_REQUIRE(logit_scale, "cor_step_tail_fwd_ls: null logit_scale");
  return step_tail_fwd(part, nsplit, split_stride, Rp, B, M, C, p_total, stats, queries_bf16, comb, targets, 0.f, logit_scale, seg, w_fg,
                       w_bg, w_nce, fg, fg_bf16, inv_fg, bg, inv_bg, fgbg_out4, aux, lse, nce, tgt_logit, total, work, counter, stream);
}

extern "C" int cor_step_tail_fwd_mem(const float* part, int nsplit, long long split_stride, int Rp, int B, int M, int C, float p_total,
                                     const float* stats, const void* queries_bf16, const float* comb, const long long* targets, float inv_tau,
                                     const float* logit_scale, const float* mem_part, int mem_nparts, const int* mem_state, const float* seg,
                                     float w_fg, float w_bg, float w_nce, float* fg, void* fg_bf16, float* inv_fg, float* bg, float* inv_bg,
                                     float* fgbg_out4, float* aux, float* lse, float* nce, float* tgt_logit, float* total, void* work,
                                     unsigned* counter, cor_stream_t stream) {
  return step_tail_fwd(part, nsplit, split_stride, Rp, B, M, C, p_total, stats, queries_bf16, comb, targets, inv_tau, logit_scale, seg, w_fg,
                       w_bg, w_nce, fg, fg_bf16, inv_fg, bg, inv_bg, fgbg_out4, aux, lse, nce, tgt_logit, total, work, counter, stream,
                       mem_part, mem_nparts, mem_state);
}

static int step_tail_bwd(const void* regions_bf16, const void* queries_bf16, const long long* targets, const float* lse, int B, int M,
                         int C, float inv_tau, const float* scale, const float* g_loss, float w_nce, const float* fg, const float* inv_fg,
                         const float* stats, const float* comb, const float* fgbg_out4, const float* aux, float w_fg, float w_bg,
                         void* a16, int Kp, float* g_queries, float* g_scale, void* work, unsigned* counter, cor_stream_t stream) {
  int rc = tail_shape_ok(B, M, C, "cor_step_tail_bwd");
  if (rc) return rc;
  COR_REQUIRE(regions_bf16 && queries_bf16 && targets && lse && g_loss && fg && inv_fg && stats && comb && fgbg_out4 && aux,
              "cor_step_tail_bwd: null pointer");
  COR_REQUIRE(!(g_queries || g_scale) || (work && counter), "cor_step_tail_bwd: g_queries / g_logit_scale need a work buffer and the counters");
  COR_REQUIRE(!a16 || Kp >= M, "cor_step_tail_bwd: Kp=%d < M=%d", Kp, M);
  COR_REQUIRE((((uintptr_t)regions_bf16 | (uintptr_t)queries_bf16 | (uintptr_t)fg | (uintptr_t)comb | (uintptr_t)a16) & 15) == 0,
              "cor_step_tail_bwd: 16-byte alignment required");
  if (!a16 && !g_queries && !g_scale) return COR_OK;
  const int nreg = a16 ? ceil_div((long long)B * M, 8) : 0;
  const int nsq = tail_nsplit_q(B, M);
  const int grid = nreg + (g_queries || g_scale ? B * nsq : 0);
  // work: qpart [B][nsq][C], then the logit-scale partials lspart [B][nsq] and per-query sums lsq [kQT]
  float* qpart = (float*)work;
  float* lspart = qpart ? qpart + (size_t)B * nsq * C : nullptr;
  float* lsq = lspart ? lspart + (size_t)B * nsq : nullptr;
  StepTailBwd a{(const bf16*)regions_bf16, (const bf16*)queries_bf16, targets, lse, B, M, C, inv_tau, scale, g_loss, w_nce, fg, inv_fg,
                stats, comb, fgbg_out4, aux, w_fg, w_bg, (bf16*)a16, Kp, g_queries, g_scale, qpart, lspart, lsq, counter, nreg, nsq};
  step_tail_bwd_kernel<<<grid, 256, (size_t)kQT * C * sizeof(float), as_stream(stream)>>>(a);
  return check_launch("step_tail_bwd_kernel");
}

extern "C" int cor_step_tail_bwd(const void* regions_bf16, const void* queries_bf16, const long long* targets, const float* lse, int B, int M,
                                 int C, float inv_tau, const float* g_loss, float w_nce, const float* fg, const float* inv_fg,
                                 const float* stats, const float* comb, const float* fgbg_out4, const float* aux, float w_fg, float w_bg,
                                 void* a16, int Kp, float* g_queries, void* work, unsigned* counter, cor_stream_t stream) {
  return step_tail_bwd(regions_bf16, queries_bf16, targets, lse, B, M, C, inv_tau, nullptr, g_loss, w_nce, fg, inv_fg, stats, comb, fgbg_out4,
                       aux, w_fg, w_bg, a16, Kp, g_queries, nullptr, work, counter, stream);
}

extern "C" int cor_step_tail_bwd_ls(const void* regions_bf16, const void* queries_bf16, const long long* targets, const float* lse, int B,
                                    int M, int C, const float* logit_scale, const float* g_loss, float w_nce, const float* fg,
                                    const float* inv_fg, const float* stats, const float* comb, const float* fgbg_out4, const float* aux,
                                    float w_fg, float w_bg, void* a16, int Kp, float* g_queries, float* g_logit_scale, void* work,
                                    unsigned* counter, cor_stream_t stream) {
  COR_REQUIRE(logit_scale, "cor_step_tail_bwd_ls: null logit_scale");
  return step_tail_bwd(regions_bf16, queries_bf16, targets, lse, B, M, C, 0.f, logit_scale, g_loss, w_nce, fg, inv_fg, stats, comb,
                       fgbg_out4, aux, w_fg, w_bg, a16, Kp, g_queries, g_logit_scale, work, counter, stream);
}
