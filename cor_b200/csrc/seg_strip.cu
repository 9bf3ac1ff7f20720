// Segmentation loss forward, row-strip streaming version (utils/loss_func.py:5-32 + the target resample of
// utils/trainer_v3_g.py:67) for the two shapes the reference actually produces: the target already at the logit size
// (what `wbce_with_wiou_loss(pred, target)` receives, loss_func.py:5) and the full-resolution mask at exactly 4x the
// logit size (1024^2 -> 256^2, trainer_v3_g.py:67, whose 2x2 taps are columns 4x+1, 4x+2 of rows 4y+1, 4y+2).
//
// A CTA owns a strip of R logit rows of one sample, all W <= 256 columns wide, so the 31x31 box filter needs a halo in
// y only.  Input rows stream through a TMA ring, kSG logit rows per stage:
//   * exact-4x masks: a 4-D tensor map [x, r = row % 4, g = row / 4, n] with box {256, 2, kSG, 1} at r = 1 fetches ONLY
//     rows 4y+1 and 4y+2 -- whole 128-byte lines, every DRAM sector that holds a tap exactly once, nothing else;
//   * the logits ride in the same stage (3-D map, box {W, kSG, 1});
//   * out-of-image rows are zero-filled by TMA = the zero padding of avg_pool2d(31, 1, 15, count_include_pad=True).
// One thread per column.  The vertical 31-row sum is a sliding window in a REGISTER (+ new row - row 31 back); the
// 32-row ring of targets it needs lives in REGISTERS too (the row loop is unrolled 32 deep so every ring index is a
// compile-time constant), which leaves the shared memory to the TMA ring: three 4-row stages per CTA, two CTAs per SM.  The
// horizontal 31-column sum is a warp shuffle prefix scan plus two shared-memory reads for the neighbouring warps'
// prefixes -- one named barrier per kSG rows.  Per-pixel terms accumulate in registers; one fixed-order block
// reduction per CTA at the end (deterministic).
// Warp roles (288 threads): 0..7 consumers (column = threadIdx.x), 8 = TMA producer.
#include <stdlib.h>

#include "seg_common.cuh"
#include "umma.cuh"

namespace cor {

using namespace umma;

constexpr int kSW = 256;        // columns per CTA (= consumer threads)
constexpr int kSG = 4;          // logit rows per stage (A/B on B200: 2-row stages x 6 were 18 % slower -- the per-stage scan + barrier chain, not DRAM latency, paces a CTA)
constexpr int kSStages = 3;
constexpr int kSRing = 32;      // rows of targets kept per column (31-row window + the row being written), in registers
constexpr int kSUnroll = kSRing / kSG;   // chunks per unrolled group: one full turn of the ring
constexpr int kSThreads = kSW + 32;
constexpr int kSHalo = 15;
constexpr int kStripFill = 85;    // per cent of the 2 x SM CTA slots a strip height must fill (B = 128: 128-row strips = 256 CTAs in one wave 92 us, 64-row strips = 512 CTAs in 1.7 waves 113 us; B = 64: 64-row strips 63 us, 128-row 72 us)

struct StripSmemTail {
  uint64_t full[kSStages], empty[kSStages];
};

template <typename T>
__device__ __forceinline__ float2 mid_pair(const uint8_t* p);   // elements 1 and 2 of the 4-element group at p
template <>
__device__ __forceinline__ float2 mid_pair<float>(const uint8_t* p) {
  const float4 v = *reinterpret_cast<const float4*>(p);
  return make_float2(v.y, v.z);
}
template <>
__device__ __forceinline__ float2 mid_pair<bf16>(const uint8_t* p) {
  const uint2 v = *reinterpret_cast<const uint2*>(p);
  return make_float2(bf16hi(v.x), bf16lo(v.y));
}
template <>
__device__ __forceinline__ float2 mid_pair<uint8_t>(const uint8_t* p) {
  const uint32_t v = *reinterpret_cast<const uint32_t*>(p);
  return make_float2((float)((v >> 8) & 0xffu), (float)((v >> 16) & 0xffu));
}

template <typename T>
__device__ __forceinline__ float ld_smem_f(const uint8_t* p) { return to_f<T>(*reinterpret_cast<const T*>(p)); }

struct StripArgs {
  int H, W, R, nstrips, fast4, nbox, box_x;
  int mask_stage_bytes, stage_bytes, tx_bytes;    // stage layout: [mask boxes | pad to 128 | logit box | pad]; tx = bytes TMA delivers
  float mscale, focal_alpha, focal_gamma;
  float* t_save;
  float* w_save;
  double* part;
};

template <typename TP, typename TM>
__global__ void __launch_bounds__(kSThreads, 2) seg_loss_strip_kernel(const __grid_constant__ CUtensorMap tmM,
                                                                      const __grid_constant__ CUtensorMap tmP, StripArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* base = reinterpret_cast<uint8_t*>(((uintptr_t)smem + 127) & ~(uintptr_t)127);
  uint8_t* stages = base;
  float* pbuf = reinterpret_cast<float*>(base + (size_t)kSStages * a.stage_bytes);        // [2][kSG][kSW]
  StripSmemTail* tail = reinterpret_cast<StripSmemTail*>(pbuf + 2 * kSG * kSW);
  double* scratch = reinterpret_cast<double*>(stages);      // block reduction scratch: the ring is drained by then

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = blockIdx.x / a.nstrips, strip = blockIdx.x % a.nstrips;
  const int y0 = strip * a.R;
  const int rows = min(a.R, a.H - y0);
  const int jstart = y0 - kSHalo;                       // first input row of the strip (may be < 0: zero-filled)
  const int nchunks = (rows + 2 * kSHalo + kSG - 1) / kSG;

  if (threadIdx.x == 0) {
    prefetch_tmap(&tmM);
    prefetch_tmap(&tmP);
    for (int i = 0; i < kSStages; ++i) { mbar_init(&tail->full[i], 1); mbar_init(&tail->empty[i], kSW / 32); }
    fence_barrier_init();
  }
  __syncthreads();

  double acc[kNP];
#pragma unroll
  for (int k = 0; k < kNP; ++k) acc[k] = 0.0;

  if (warp == kSW / 32) {
    // ---- producer: one thread streams the strip's rows, kSG logit rows per stage ----
    if (lane == 0) {
      int st = 0, ph = 1;
      for (int c = 0; c < nchunks; ++c, st = (st + 1 == kSStages ? 0 : st + 1), ph ^= (st == 0)) {
        mbar_wait(&tail->empty[st], (uint32_t)ph);
        uint8_t* dst = stages + (size_t)st * a.stage_bytes;
        mbar_expect_tx(&tail->full[st], (uint32_t)a.tx_bytes);
        const int j0 = jstart + c * kSG;
        if (a.fast4) {
          const int box_bytes = kSG * 2 * a.box_x * (int)sizeof(TM);
          for (int b = 0; b < a.nbox; ++b) tma_load_4d(dst + (size_t)b * box_bytes, &tmM, &tail->full[st], b * a.box_x, 1, j0, n, kEvictFirst);
        } else {
          tma_load_3d(dst, &tmM, &tail->full[st], 0, j0, n, kEvictFirst);
        }
        tma_load_3d(dst + a.mask_stage_bytes, &tmP, &tail->full[st], 0, j0 - kSHalo, n, kEvictFirst);
      }
    }
  } else {
    // ---- consumers: thread = column ----
    const int x = threadIdx.x;
    const bool colok = x < a.W;
    float ring[kSRing];                                // this column's last 32 target rows; slot = (row - jstart) % 32
#pragma unroll
    for (int r = 0; r < kSRing; ++r) ring[r] = 0.f;
    float V = 0.f;                                     // sum of the last 31 target rows of this column
    float f[kNP];
#pragma unroll
    for (int k = 0; k < kNP; ++k) f[k] = 0.f;
    // where this column's taps live inside a stage
    int tap_off;
    if (a.fast4) {
      const int xb = (4 * x) / a.box_x, off = (4 * x) % a.box_x;
      tap_off = (xb * kSG * 2 * a.box_x + off) * (int)sizeof(TM);
    } else {
      tap_off = x * (int)sizeof(TM);
    }
    const int row_pitch = (a.fast4 ? 2 * a.box_x : a.W) * (int)sizeof(TM);     // bytes between consecutive g inside a stage
    const int r1_off = a.box_x * (int)sizeof(TM);
    int st = 0, ph = 0;
    for (int c0 = 0; c0 < nchunks; c0 += kSUnroll) {
#pragma unroll
      for (int cc = 0; cc < kSUnroll; ++cc) {
        const int c = c0 + cc;
        if (c < nchunks) {
          mbar_wait(&tail->full[st], (uint32_t)ph);
          const uint8_t* sm = stages + (size_t)st * a.stage_bytes;
          float tn[kSG], z[kSG];
#pragma unroll
          for (int g = 0; g < kSG; ++g) {
            tn[g] = 0.f;
            z[g] = 0.f;
            if (colok) {
              const uint8_t* p = sm + tap_off + g * row_pitch;
              if (a.fast4) {
                const float2 u = mid_pair<TM>(p), v = mid_pair<TM>(p + r1_off);
                // ATen upsample_bilinear2d at an exact 4x ratio: all four weights are 0.5
                tn[g] = (0.5f * (0.5f * u.x + 0.5f * u.y) + 0.5f * (0.5f * v.x + 0.5f * v.y)) * a.mscale;
              } else {
                tn[g] = ld_smem_f<TM>(p) * a.mscale;
              }
              z[g] = ld_smem_f<TP>(sm + a.mask_stage_bytes + (g * a.W + x) * (int)sizeof(TP));
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&tail->empty[st]);     // the stage is in registers: let the producer refill it
          if (++st == kSStages) { st = 0; ph ^= 1; }
          const int j0 = jstart + c * kSG;                  // input rows j0 .. j0+kSG-1; output rows (j - 15)
          float Vg[kSG];
#pragma unroll
          for (int g = 0; g < kSG; ++g) {
            constexpr int dummy = 0; (void)dummy;
            const int rr = cc * kSG + g;                     // compile-time ring slot of input row j0 + g
            V += tn[g] - ring[(rr + 1) & (kSRing - 1)];      // row j - 31 sits in the slot row j + 1 will take
            ring[rr] = tn[g];
            Vg[g] = V;
          }
          // any output row in this chunk?  (uniform over the CTA)
          const int jo_lo = j0 - kSHalo, jo_hi = jo_lo + kSG - 1;
          if (!(jo_hi < y0 || jo_lo >= y0 + rows)) {
            // horizontal 31-sums: inclusive prefix inside the warp ...
            float P[kSG];
#pragma unroll
            for (int g = 0; g < kSG; ++g) P[g] = Vg[g];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
              for (int g = 0; g < kSG; ++g) {
                const float up = __shfl_up_sync(0xffffffffu, P[g], o);
                if (lane >= o) P[g] += up;
              }
            }
            float* pb = pbuf + (c & 1) * kSG * kSW;
#pragma unroll
            for (int g = 0; g < kSG; ++g) pb[g * kSW + x] = P[g];
            asm volatile("bar.sync 1, %0;" ::"n"(kSW) : "memory");
            // ... combined across at most two warps: columns [x-15, x+15]
#pragma unroll
            for (int g = 0; g < kSG; ++g) {
              const float hi = __shfl_sync(0xffffffffu, P[g], min(lane + 15, 31));
              const float lo = __shfl_sync(0xffffffffu, P[g], max(lane - 16, 0));
              float box = hi - (lane >= 16 ? lo : 0.f);
              if (lane < 15 && warp > 0) box += pb[g * kSW + (warp - 1) * 32 + 31] - pb[g * kSW + (warp - 1) * 32 + lane + 16];
              if (lane > 16 && warp < kSW / 32 - 1) box += pb[g * kSW + (warp + 1) * 32 + lane - 17];
              const int jo = jo_lo + g;
              if (colok && jo >= y0 && jo < y0 + rows) {
                const float t = ring[(cc * kSG + g + kSRing - kSHalo) & (kSRing - 1)];     // row jo = j - 15
                float wgt;
                seg_pixel_terms(z[g], t, box, a.focal_alpha, a.focal_gamma, f, wgt);
                if (a.t_save) {
                  const long long o = ((long long)n * a.H + jo) * a.W + x;
                  a.t_save[o] = t;
                  a.w_save[o] = wgt;
                }
              }
            }
          }
        }
      }
    }
#pragma unroll
    for (int k = 0; k < kNP; ++k) acc[k] = (double)f[k];
  }
  __syncthreads();                                          // every stage consumed: its memory becomes the scratch
  block_sum<kNP>(acc, scratch);
  if (threadIdx.x == 0) {
    double* o = a.part + (long long)blockIdx.x * kNP;
#pragma unroll
    for (int k = 0; k < kNP; ++k) o[k] = acc[k];
  }
}

int seg_strip_max_strips(int H) { return ceil_div(H, 16); }

static int strip_rows(int N, int H) {
  // largest strip (least halo re-reads: (R+30)/R of the rows come through L2) that still fills most of the machine's
  // 2-CTAs-per-SM slots in ONE wave (a second, partly filled wave costs more than a few idle slots)
  const long long want = (long long)2 * sm_count() * kStripFill / 100;
  for (int R = 128; R >= 32; R >>= 1)
    if ((long long)N * ceil_div(H, R) >= want) return R;
  return 16;
}

template <typename TP, typename TM>
static int strip_launch(const void* pred, const void* mask, float mscale, int N, int H, int W, int Hm, int Wm, long long ns, float fa,
                        float fg_, float* t_save, float* w_save, double* part, int* strips, cudaStream_t st) {
  StripArgs a{};
  a.H = H; a.W = W; a.fast4 = (Hm != H) ? 1 : 0;
  a.R = strip_rows(N, H);
  a.nstrips = ceil_div(H, a.R);
  a.mscale = mscale; a.focal_alpha = fa; a.focal_gamma = fg_;
  a.t_save = t_save; a.w_save = w_save; a.part = part;
  CUtensorMap tmM, tmP;
  int rc;
  if (a.fast4) {
    a.box_x = Wm < 256 ? Wm : 256;
    a.nbox = ceil_div(Wm, a.box_x);
    a.mask_stage_bytes = a.nbox * kSG * 2 * a.box_x * (int)sizeof(TM);
    const uint64_t dims[4] = {(uint64_t)Wm, 4, (uint64_t)H, (uint64_t)N};
    const uint64_t strides[3] = {(uint64_t)Wm * sizeof(TM), (uint64_t)4 * Wm * sizeof(TM), (uint64_t)ns * sizeof(TM)};
    const uint32_t box[4] = {(uint32_t)a.box_x, 2, (uint32_t)kSG, 1};
    rc = encode_tmap_tiled(&tmM, mask, (int)sizeof(TM), 4, dims, strides, box);
  } else {
    a.box_x = W;
    a.nbox = 1;
    a.mask_stage_bytes = kSG * W * (int)sizeof(TM);
    const uint64_t dims[3] = {(uint64_t)W, (uint64_t)H, (uint64_t)N};
    const uint64_t strides[2] = {(uint64_t)W * sizeof(TM), (uint64_t)ns * sizeof(TM)};
    const uint32_t box[3] = {(uint32_t)W, (uint32_t)kSG, 1};
    rc = encode_tmap_tiled(&tmM, mask, (int)sizeof(TM), 3, dims, strides, box);
  }
  if (rc) return rc;
  a.mask_stage_bytes = (a.mask_stage_bytes + 127) & ~127;
  {
    const uint64_t dims[3] = {(uint64_t)W, (uint64_t)H, (uint64_t)N};
    const uint64_t strides[2] = {(uint64_t)W * sizeof(TP), (uint64_t)H * W * sizeof(TP)};
    const uint32_t box[3] = {(uint32_t)W, (uint32_t)kSG, 1};
    rc = encode_tmap_tiled(&tmP, pred, (int)sizeof(TP), 3, dims, strides, box);
    if (rc) return rc;
  }
  const int logit_bytes = (kSG * W * (int)sizeof(TP) + 127) & ~127;
  a.stage_bytes = a.mask_stage_bytes + logit_bytes;
  // the bytes TMA actually delivers per stage (boxes are dense; the 128-byte padding between the parts carries none)
  a.tx_bytes = (a.fast4 ? a.nbox * kSG * 2 * a.box_x : kSG * W) * (int)sizeof(TM) + kSG * W * (int)sizeof(TP);
  const size_t smem = (size_t)kSStages * a.stage_bytes + (size_t)(2 * kSG) * kSW * sizeof(float) + sizeof(StripSmemTail) + 128;
  auto k = seg_loss_strip_kernel<TP, TM>;
  COR_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<N * a.nstrips, kSThreads, smem, st>>>(tmM, tmP, a);
  *strips = a.nstrips;
  return check_launch("seg_loss_strip_kernel");
}

int seg_strip_try_launch(const void* pred, int pred_dtype, const void* mask, int mask_dtype, float mscale, int N, int H, int W, int Hm,
                         int Wm, long long ns, float fa, float fg_, float* t_save, float* w_save, double* part, int* strips,
                         cudaStream_t st) {
  const bool same = (Hm == H && Wm == W), four = (Hm == 4 * H && Wm == 4 * W);
  const int em = mask_dtype == COR_F32 ? 4 : mask_dtype == COR_BF16 ? 2 : 1;
  const int ep = pred_dtype == COR_F32 ? 4 : 2;
  // shapes the strip kernel serves; everything else (other ratios, wide or oddly pitched images) takes the tile kernel
  if (!(same || four) || W > kSW || W % 16 != 0) return COR_EINVAL;
  // a handful of samples with 2/4-byte 4x masks: too few strips to hide each CTA's serial row chain -- the 64x64 tile kernel
  // measures faster there (B=16, 1024^2 fp32 -> 256^2: 32.8 vs 38.9 us; B=128: 147 vs 111 us).  COR_SEG_STRIP=2 forces strips.
  {
    const char* knob = getenv("COR_SEG_STRIP");
    const bool force = knob && atoi(knob) == 2;
    if (!force && four && em >= 2 && (long long)N * H * W < (1ll << 21)) return COR_EINVAL;
  }
  if (((uintptr_t)mask & 15) || ((uintptr_t)pred & 15) || (ns * em) % 16 != 0 || ((long long)Wm * em) % 16 != 0 || ((long long)W * ep) % 16 != 0)
    return COR_EINVAL;
#define COR_STRIP(TP, TM) return strip_launch<TP, TM>(pred, mask, mscale, N, H, W, Hm, Wm, ns, fa, fg_, t_save, w_save, part, strips, st)
  if (pred_dtype == COR_F32 && mask_dtype == COR_F32) COR_STRIP(float, float);
  if (pred_dtype == COR_BF16 && mask_dtype == COR_F32) COR_STRIP(bf16, float);
  if (pred_dtype == COR_F32 && mask_dtype == COR_U8) COR_STRIP(float, uint8_t);
  if (pred_dtype == COR_BF16 && mask_dtype == COR_U8) COR_STRIP(bf16, uint8_t);
  if (pred_dtype == COR_F32 && mask_dtype == COR_BF16) COR_STRIP(float, bf16);
  if (pred_dtype == COR_BF16 && mask_dtype == COR_BF16) COR_STRIP(bf16, bf16);
#undef COR_STRIP
  return COR_EINVAL;
}

}  // namespace cor
