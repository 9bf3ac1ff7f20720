// Foreground / background cosine losses on pooled unit rows (utils/loss_func.py:59-126).
//
//   fg = 1 - mean_{valid i} cos(fg_i, q_i)                                   loss_func.py:84
//   bg = mean(cos(...) + 1)                                                  loss_func.py:123-124
// where, in the reference, the bg cosine is taken between [V,1,C] and [V,C] along dim=1, i.e. over
// the broadcast ROW axis (loss_func.py:120-123).  bg_mode 0 reproduces that value exactly:
//   bg = 1 + 1/(V*C) * sum_c A[c] * S1[c] / max(s2[c], eps),
//   A[c]  = sum_{valid i} bg[i,c] / max(sqrt(V)*|bg[i,c]|, eps)
//   S1[c] = sum_{valid j} q[j,c],   s2[c] = sqrt(sum_{valid j} q[j,c]^2)
// (its derivative w.r.t. the bg rows is identically zero); bg_mode 1 is the paired per-sample cosine.
// Validity comes from the full-resolution sums of mask_prep (stats[i][0] > 0, stats[i][1] > 0) and is
// resolved on the device: no host sync, unlike `valid.any()` at loss_func.py:76,109.
#include "common.cuh"

namespace cor {

constexpr float kCosEps = 1e-8f;  // F.cosine_similarity default eps

// aux layout: rowstat [n][8] = {cos_fg, cos_bg, N_fg, N_bg, N_q, valid_fg, valid_bg, 0}; then colstat [3][C]
__global__ void __launch_bounds__(128) fgbg_rows_kernel(const float* __restrict__ fg, long long row_stride, const float* __restrict__ bg,
                                                        long long bg_stride, const float* __restrict__ comb, long long comb_stride,
                                                        const float* __restrict__ stats, long long stats_stride, int C,
                                                        float* __restrict__ rowstat) {
  __shared__ float scratch[5 * 32];
  const int i = blockIdx.x;
  const float* f = fg + i * row_stride;
  const float* g = bg ? bg + i * bg_stride : nullptr;
  const float* q = comb + i * comb_stride;
  float v[5] = {0.f, 0.f, 0.f, 0.f, 0.f};  // f.q, g.q, f.f, g.g, q.q
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float a = f[c], b = g ? g[c] : 0.f, x = q[c];
    v[0] = fmaf(a, x, v[0]); v[1] = fmaf(b, x, v[1]); v[2] = fmaf(a, a, v[2]); v[3] = fmaf(b, b, v[3]); v[4] = fmaf(x, x, v[4]);
  }
  block_sum<5>(v, scratch);
  if (threadIdx.x == 0) {
    const float nf = fmaxf(sqrtf(v[2]), kCosEps), nb = fmaxf(sqrtf(v[3]), kCosEps), nq = fmaxf(sqrtf(v[4]), kCosEps);
    float* o = rowstat + (long long)i * 8;
    o[0] = v[0] / (nf * nq);
    o[1] = v[1] / (nb * nq);
    o[2] = nf; o[3] = nb; o[4] = nq;
    o[5] = stats[i * stats_stride + 0] > 0.f ? 1.f : 0.f;
    o[6] = stats[i * stats_stride + 1] > 0.f ? 1.f : 0.f;
    o[7] = 0.f;
  }
}

__global__ void __launch_bounds__(1024) fgbg_reduce_kernel(const float* __restrict__ bg, long long bg_stride, const float* __restrict__ comb,
                                                           long long comb_stride, int n, int C, int bg_mode,
                                                           const float* __restrict__ rowstat, float* __restrict__ colstat,
                                                           float* __restrict__ out4) {
  __shared__ double scratch[5 * 32];
  double v[5] = {0, 0, 0, 0, 0};  // sum cos_fg (valid), n_fg, sum cos_bg paired (valid), n_bg, quirk sum
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float* r = rowstat + (long long)i * 8;
    if (r[5] > 0.f) { v[0] += r[0]; v[1] += 1.0; }
    if (r[6] > 0.f) { v[2] += r[1]; v[3] += 1.0; }
  }
  block_sum<5>(v, scratch);  // v[4] is still 0 here
  const double nfg = v[1], nbg = v[3];
  if (bg_mode == 0 && bg && nbg > 0) {
    // column statistics of the reference's broadcast: 256 columns x 4 row-parts per pass, the parts combined in a fixed order
    __shared__ float colpart[3][4][256];
    const float sq = sqrtf((float)nbg);
    const int cl = threadIdx.x & 255, part = threadIdx.x >> 8;
    for (int c0 = 0; c0 < C; c0 += 256) {
      const int c = c0 + cl;
      float A = 0.f, S1 = 0.f, ss = 0.f;
      if (c < C) {
#pragma unroll 4
        for (int i = part; i < n; i += 4) {
          if (rowstat[(long long)i * 8 + 6] > 0.f) {
            const float x = bg[i * bg_stride + c], q = comb[i * comb_stride + c];
            A += x / fmaxf(sq * fabsf(x), kCosEps);
            S1 += q;
            ss = fmaf(q, q, ss);
          }
        }
      }
      __syncthreads();
      colpart[0][part][cl] = A; colpart[1][part][cl] = S1; colpart[2][part][cl] = ss;
      __syncthreads();
      if (part == 0 && c < C) {
        A = (colpart[0][0][cl] + colpart[0][1][cl]) + (colpart[0][2][cl] + colpart[0][3][cl]);
        S1 = (colpart[1][0][cl] + colpart[1][1][cl]) + (colpart[1][2][cl] + colpart[1][3][cl]);
        ss = (colpart[2][0][cl] + colpart[2][1][cl]) + (colpart[2][2][cl] + colpart[2][3][cl]);
        const float s2 = fmaxf(sqrtf(ss), kCosEps);
        colstat[c] = A; colstat[C + c] = S1; colstat[2 * C + c] = s2;
        v[4] += (double)(A * S1 / s2);
      }
    }
  }
  __syncthreads();
  double q[1] = {v[4]};
  block_sum<1>(q, scratch);
  if (threadIdx.x == 0) {
    out4[0] = nfg > 0 ? (float)(1.0 - v[0] / nfg) : 0.f;
    float bgl = 0.f;
    if (bg && nbg > 0) bgl = bg_mode == 0 ? (float)(1.0 + q[0] / (nbg * (double)C)) : (float)(v[2] / nbg + 1.0);
    out4[1] = bgl;
    out4[2] = (float)nfg;
    out4[3] = (float)nbg;
  }
}

__global__ void __launch_bounds__(128) fgbg_bwd_kernel(const float* __restrict__ fg, long long row_stride, const float* __restrict__ bg,
                                                       long long bg_stride, const float* __restrict__ comb, long long comb_stride, int C,
                                                       int bg_mode, const float* __restrict__ rowstat, const float* __restrict__ colstat,
                                                       const float* __restrict__ out4, const float* __restrict__ g2, long long g2_stride,
                                                       float gw_fg, float gw_bg, float* __restrict__ g_fg, long long gfg_stride, int fg_acc,
                                                       float* __restrict__ g_bg, long long gbg_stride, float* __restrict__ g_comb,
                                                       long long gcomb_stride, int comb_acc) {
  const int i = blockIdx.x;
  const float* r = rowstat + (long long)i * 8;
  const float nfg = out4[2], nbg = out4[3];
  const float gf_up = g2[0] * gw_fg, gb_up = g2[g2_stride] * gw_bg;            // upstream scalars (x caller weights)
  const float sf = (r[5] > 0.f && nfg > 0.f) ? -gf_up / nfg : 0.f;            // d loss_fg / d cos_fg_i
  const float sb = (bg && bg_mode == 1 && r[6] > 0.f && nbg > 0.f) ? gb_up / nbg : 0.f;
  const float quirk = (bg && bg_mode == 0 && r[6] > 0.f && nbg > 0.f) ? gb_up / (nbg * (float)C) : 0.f;
  const float cf = r[0], cb = r[1], nf = r[2], nb = r[3], nq = r[4];
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float a = fg[i * row_stride + c], x = comb[i * comb_stride + c];
    const float b = bg ? bg[i * bg_stride + c] : 0.f;
    float gq = sf * (a / (nf * nq) - cf * x / (nq * nq));
    const float ga = sf * (x / (nf * nq) - cf * a / (nf * nf));
    float* pf = g_fg + i * gfg_stride + c;
    *pf = fg_acc ? *pf + ga : ga;
    float gb = 0.f;
    if (sb != 0.f) {
      gb = sb * (x / (nb * nq) - cb * b / (nb * nb));
      gq += sb * (b / (nb * nq) - cb * x / (nq * nq));
    }
    if (quirk != 0.f) {
      const float A = colstat[c], S1 = colstat[C + c], s2 = colstat[2 * C + c];
      gq += quirk * A * (1.f / s2 - S1 * x / (s2 * s2 * s2));
    }
    if (g_bg) g_bg[i * gbg_stride + c] = gb;
    float* pq = g_comb + i * gcomb_stride + c;
    *pq = comb_acc ? *pq + gq : gq;
  }
}

}  // namespace cor

using namespace cor;

extern "C" size_t cor_fgbg_aux_floats(int n, int C) { return (size_t)n * 8 + (size_t)3 * C; }

extern "C" int cor_fgbg_loss_fwd(const float* fg_rows, long long fg_stride, const float* bg_rows, long long bg_stride, const float* comb,
                                 long long comb_stride, const float* stats, long long stats_stride, int n, int C, int bg_mode,
                                 float* out4, float* aux, cor_stream_t stream) {
  COR_REQUIRE(fg_rows && comb && stats && out4 && aux, "cor_fgbg_loss_fwd: null pointer");
  COR_REQUIRE(n > 0 && C > 0 && (bg_mode == 0 || bg_mode == 1), "cor_fgbg_loss_fwd: bad arguments n=%d C=%d mode=%d", n, C, bg_mode);
  cudaStream_t st = as_stream(stream);
  fgbg_rows_kernel<<<n, 128, 0, st>>>(fg_rows, fg_stride, bg_rows, bg_stride, comb, comb_stride, stats, stats_stride, C, aux);
  int rc = check_launch("fgbg_rows_kernel");
  if (rc) return rc;
  fgbg_reduce_kernel<<<1, 1024, 0, st>>>(bg_rows, bg_stride, comb, comb_stride, n, C, bg_mode, aux, aux + (size_t)n * 8, out4);
  return check_launch("fgbg_reduce_kernel");
}

extern "C" int cor_fgbg_loss_bwd(const float* fg_rows, long long fg_stride, const float* bg_rows, long long bg_stride, const float* comb,
                                 long long comb_stride, int n, int C, int bg_mode, const float* out4, const float* aux, const float* g2,
                                 long long g2_stride, float gw_fg, float gw_bg, float* g_fg_rows, long long gfg_stride, int fg_accumulate, float* g_bg_rows, long long gbg_stride,
                                 float* g_comb, long long gcomb_stride, int comb_accumulate, cor_stream_t stream) {
  COR_REQUIRE(fg_rows && comb && out4 && aux && g2 && g_fg_rows && g_comb, "cor_fgbg_loss_bwd: null pointer");
  fgbg_bwd_kernel<<<n, 128, 0, as_stream(stream)>>>(fg_rows, fg_stride, bg_rows, bg_stride, comb, comb_stride, C, bg_mode, aux,
                                                    aux + (size_t)n * 8, out4, g2, g2_stride, gw_fg, gw_bg, g_fg_rows, gfg_stride, fg_accumulate, g_bg_rows,
                                                    gbg_stride, g_comb, gcomb_stride, comb_accumulate);
  return check_launch("fgbg_bwd_kernel");
}
