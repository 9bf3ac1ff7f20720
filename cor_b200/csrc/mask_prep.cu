// mask_prep: one pass over full-resolution masks producing
//   (1) the bilinear (align_corners=False) resample to the feature grid  -- replaces F.interpolate at
//       mask_adapter.py:19-20 / loss_func.py:46-47 (ATen upsample_bilinear2d),
//   (2) sum(mask) and sum(1-mask) over the FULL-resolution mask -- the validity tests of
//       loss_func.py:73-74 and :103-107,
//   (3) the pooling denominators sum_p w.
// HBM-bound streaming kernel: every mask byte is read exactly once with 128-bit no-allocate loads;
// the 4 taps per output pixel hit lines the same CTA streams.  Deterministic: per-CTA partials in
// double, reduced in fixed order by a second tiny kernel.

#include "common.cuh"

namespace cor {

template <typename T>
struct VecSum;  // sums a 16-byte vector of T into (sum m) and count

template <>
struct VecSum<float> {
  static constexpr int N = 4;
  __device__ static __forceinline__ void add(uint4 v, float& s) {
    s += (__uint_as_float(v.x) + __uint_as_float(v.y)) + (__uint_as_float(v.z) + __uint_as_float(v.w));
  }
};
template <>
struct VecSum<bf16> {
  static constexpr int N = 8;
  __device__ static __forceinline__ void add(uint4 v, float& s) {
    s += ((bf16lo(v.x) + bf16hi(v.x)) + (bf16lo(v.y) + bf16hi(v.y))) + ((bf16lo(v.z) + bf16hi(v.z)) + (bf16lo(v.w) + bf16hi(v.w)));
  }
};
template <>
struct VecSum<uint8_t> {
  static constexpr int N = 16;
  __device__ static __forceinline__ void add(uint4 v, float& s) {
    // exact integer byte sum (<= 16*255), added to an fp32 accumulator of integers < 2^24 per thread
    unsigned t = __dp4a(v.x, 0x01010101u, 0u);
    t = __dp4a(v.y, 0x01010101u, t);
    t = __dp4a(v.z, 0x01010101u, t);
    t = __dp4a(v.w, 0x01010101u, t);
    s += (float)t;
  }
};

__device__ __forceinline__ float apply_transform(float r, int transform) {
  if (transform == COR_W_CLAMP) return fminf(fmaxf(r, 0.f), 1.f);
  if (transform == COR_W_SIGMOID) return sigmoid_acc(r);
  return r;
}

template <typename T, bool kNeedOneMinus>
__device__ __forceinline__ void add_vec(uint4 a, float mscale, float& s, float& s1m) {
  VecSum<T>::add(a, s);
  if (kNeedOneMinus) {
    const float* f = reinterpret_cast<const float*>(&a);
    s1m += (1.f - f[0] * mscale) + (1.f - f[1] * mscale) + (1.f - f[2] * mscale) + (1.f - f[3] * mscale);
  }
}

// grid.x = n_masks * chunks.  CTA (n, chunk) owns output rows [r0, r1) and input rows [i0, i1).
template <typename T, bool kNeedOneMinus>
__global__ void __launch_bounds__(256) mask_prep_kernel(const T* __restrict__ masks, float mscale, int Hm, int Wm, int h,
                                                        int w, int chunks, int transform, float* __restrict__ w_f32,
                                                        bf16* __restrict__ w_bf16, long long ldw, int group,
                                                        long long group_stride, double* __restrict__ part) {
  const int n = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  const int r0 = (int)((long long)chunk * h / chunks), r1 = (int)((long long)(chunk + 1) * h / chunks);
  const long long i0 = (long long)r0 * Hm / h, i1 = (long long)r1 * Hm / h;
  const T* base = masks + (long long)n * Hm * Wm;

  // ---- part A: stream input rows [i0, i1) for the full-resolution sums -------------------------
  const T* p = base + i0 * Wm;
  const long long cnt = (i1 - i0) * Wm;
  constexpr int VE = VecSum<T>::N;
  float s[4] = {0.f, 0.f, 0.f, 0.f};   // 4 independent accumulators (ILP)
  float s1m = 0.f;                     // sum(1 - m) for float types when values may exceed [0,1]
  long long head = ((16 - ((uintptr_t)p & 15)) & 15) / sizeof(T);
  if (head > cnt) head = cnt;
  for (long long i = threadIdx.x; i < head; i += blockDim.x) {
    float v = to_f<T>(p[i]);
    s[0] += v;
    if (kNeedOneMinus) s1m += 1.f - v * mscale;
  }
  const long long nvec = (cnt - head) / VE;
  const uint4* pv = reinterpret_cast<const uint4*>(p + head);
  long long i = threadIdx.x;
  for (; i + 3 * (long long)blockDim.x < nvec; i += 4 * (long long)blockDim.x) {
    uint4 a = ld_stream16(pv + i), b = ld_stream16(pv + i + blockDim.x), c = ld_stream16(pv + i + 2 * blockDim.x),
          d = ld_stream16(pv + i + 3 * blockDim.x);
    VecSum<T>::add(a, s[0]);
    VecSum<T>::add(b, s[1]);
    VecSum<T>::add(c, s[2]);
    VecSum<T>::add(d, s[3]);
    if (kNeedOneMinus) {
      // float masks outside [0,1] (contract violation) still get the reference's exact predicate
      const float* f;
      f = reinterpret_cast<const float*>(&a); s1m += (1.f - f[0] * mscale) + (1.f - f[1] * mscale) + (1.f - f[2] * mscale) + (1.f - f[3] * mscale);
      f = reinterpret_cast<const float*>(&b); s1m += (1.f - f[0] * mscale) + (1.f - f[1] * mscale) + (1.f - f[2] * mscale) + (1.f - f[3] * mscale);
      f = reinterpret_cast<const float*>(&c); s1m += (1.f - f[0] * mscale) + (1.f - f[1] * mscale) + (1.f - f[2] * mscale) + (1.f - f[3] * mscale);
      f = reinterpret_cast<const float*>(&d); s1m += (1.f - f[0] * mscale) + (1.f - f[1] * mscale) + (1.f - f[2] * mscale) + (1.f - f[3] * mscale);
    }
  }
  for (; i < nvec; i += blockDim.x) {
    uint4 a = ld_stream16(pv + i);
    VecSum<T>::add(a, s[0]);
    if (kNeedOneMinus) {
      const float* f = reinterpret_cast<const float*>(&a);
      s1m += (1.f - f[0] * mscale) + (1.f - f[1] * mscale) + (1.f - f[2] * mscale) + (1.f - f[3] * mscale);
    }
  }
  for (long long j = head + nvec * VE + threadIdx.x; j < cnt; j += blockDim.x) {
    float v = to_f<T>(p[j]);
    s[0] += v;
    if (kNeedOneMinus) s1m += 1.f - v * mscale;
  }

  // ---- part B: resample output rows [r0, r1) --------------------------------------------------
  const float sh = (float)Hm / (float)h, sw = (float)Wm / (float)w;
  float den = 0.f, den16 = 0.f;
  const int nout = (r1 - r0) * w;
  for (int o = threadIdx.x; o < nout; o += blockDim.x) {
    const int r = r0 + o / w, x = o % w;
    int y0, y1, x0, x1;
    float ly0, ly1, lx0, lx1;
    src_index(sh, r, Hm, y0, y1, ly0, ly1);
    src_index(sw, x, Wm, x0, x1, lx0, lx1);
    const T* row0 = base + (long long)y0 * Wm;
    const T* row1 = base + (long long)y1 * Wm;
    const float v00 = to_f<T>(__ldg(row0 + x0)), v01 = to_f<T>(__ldg(row0 + x1));
    const float v10 = to_f<T>(__ldg(row1 + x0)), v11 = to_f<T>(__ldg(row1 + x1));
    const float rv = (ly0 * (lx0 * v00 + lx1 * v01) + ly1 * (lx0 * v10 + lx1 * v11)) * mscale;
    const long long pix = (long long)r * w + x;
    const long long off = (long long)(n / group) * group_stride + (long long)(n % group) * ldw + pix;
    if (w_f32) w_f32[(long long)n * ldw + pix] = rv;
    const float tv = apply_transform(rv, transform);
    den += tv;
    if (w_bf16) {
      const bf16 q = __float2bfloat16_rn(tv);
      w_bf16[off] = q;
      den16 += __bfloat162float(q);
    }
  }

  __shared__ double scratch[4 * 32];
  double v[4];
  v[0] = ((double)s[0] + (double)s[1]) + ((double)s[2] + (double)s[3]);
  v[1] = (double)s1m;
  v[2] = (double)den;
  v[3] = (double)den16;
  block_sum<4>(v, scratch);
  if (threadIdx.x == 0) {
    double* o = part + (long long)blockIdx.x * 4;
    o[0] = v[0];
    o[1] = kNeedOneMinus ? v[1] : (double)cnt;   // element count when sum(1-m) is derived exactly
    o[2] = v[2];
    o[3] = v[3];
  }
}

// ---- staged variant ---------------------------------------------------------------------------------
// Same contract, but the input rows that carry bilinear taps are parked in shared memory AS THEY STREAM
// BY, so DRAM and L2 see every mask byte exactly once (the two-phase kernel above re-reads the tap rows,
// +12.5 % traffic at 16x down-sampling).  A CTA owns <= kMaxRO output rows: one row-structured streaming
// loop over its band of input rows (no synchronisation inside), ONE __syncthreads, then all threads form
// the 4-tap samples from shared memory.  Needs rows that are whole, aligned 16-byte vectors.
constexpr int kMaxRO = 8;          // upper bound on output rows per CTA (2*max_ro tap rows in smem)
constexpr int kSU = 4;             // independent 16-byte loads in flight per thread
constexpr int kMaxBand = 4096;     // input rows per CTA the slot table can describe

template <typename T, bool kNeedOneMinus>
__global__ void __launch_bounds__(256, 5) mask_prep_staged_kernel(const T* __restrict__ masks, float mscale, int Hm, int Wm, int h, int w,
                                                               int chunks, int transform, int lanes_per_row, int max_ro, float* __restrict__ w_f32,
                                                               bf16* __restrict__ w_bf16, long long ldw, int group, long long group_stride,
                                                               double* __restrict__ part) {
  extern __shared__ uint4 tap_smem[];                 // [2*ro][vpr] vectors, then the slot table
  constexpr int VE = VecSum<T>::N;
  const int n = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  const int r0 = (int)((long long)chunk * h / chunks), r1 = (int)((long long)(chunk + 1) * h / chunks);
  const int ro = r1 - r0;
  const long long i_begin = (long long)r0 * Hm / h, i_end = (long long)r1 * Hm / h;
  const int band = (int)(i_end - i_begin);
  const int vpr = Wm / VE;
  const T* base = masks + (long long)n * Hm * Wm;
  const float sh = (float)Hm / (float)h, sw = (float)Wm / (float)w;
  short* first_slot = reinterpret_cast<short*>(tap_smem + (size_t)2 * max_ro * vpr);   // [band] first slot fed by that row, or -1
  __shared__ int tap_row[2 * kMaxRO];
  __shared__ float tap_l1[kMaxRO];

  for (int i = threadIdx.x; i < band; i += blockDim.x) first_slot[i] = -1;
  if (threadIdx.x < ro) {
    int y0, y1;
    float l0, l1;
    src_index(sh, r0 + threadIdx.x, Hm, y0, y1, l0, l1);
    tap_row[2 * threadIdx.x] = y0;
    tap_row[2 * threadIdx.x + 1] = y1;
    tap_l1[threadIdx.x] = l1;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    // tap rows are non-decreasing in slot order: record, per band row, the first slot it feeds
    for (int sidx = 2 * ro - 1; sidx >= 0; --sidx) {
      const long long rel = (long long)tap_row[sidx] - i_begin;
      if (rel >= 0 && rel < band) first_slot[rel] = (short)sidx;
    }
  }
  __syncthreads();

  float s[4] = {0.f, 0.f, 0.f, 0.f};
  float s1m = 0.f;
  const int L = lanes_per_row, rows_par = blockDim.x / L;
  const int rofs = threadIdx.x / L, v0 = threadIdx.x % L;
  for (long long row = i_begin + rofs; row < i_end; row += (long long)kSU * rows_par) {
    for (int v = v0; v < vpr; v += L) {
      uint4 a[kSU];
#pragma unroll
      for (int k = 0; k < kSU; ++k) {
        const long long rr = row + (long long)k * rows_par;
        if (rr < i_end) a[k] = ld_stream16(reinterpret_cast<const uint4*>(base + rr * Wm) + v);
      }
#pragma unroll
      for (int k = 0; k < kSU; ++k) {
        const long long rr = row + (long long)k * rows_par;
        if (rr < i_end) {
          add_vec<T, kNeedOneMinus>(a[k], mscale, s[k & 3], s1m);
          int sl = first_slot[rr - i_begin];
          if (sl >= 0) {
            do {
              tap_smem[(size_t)sl * vpr + v] = a[k];
              ++sl;
            } while (sl < 2 * ro && tap_row[sl] == (int)rr);
          }
        }
      }
    }
  }
  __syncthreads();

  // ---- 4-tap samples for the CTA's ro x w outputs; taps outside the band (edge clamps when up-sampling)
  //      come from global memory
  const long long obase = (long long)(n / group) * group_stride + (long long)(n % group) * ldw;
  float den = 0.f, den16 = 0.f;
  for (int o = threadIdx.x; o < ro * w; o += blockDim.x) {
    const int j = o / w, x = o % w, r = r0 + j;
    const int y0 = tap_row[2 * j], y1 = tap_row[2 * j + 1];
    const float ly1 = tap_l1[j], ly0 = 1.f - ly1;
    int x0, x1;
    float lx0, lx1;
    src_index(sw, x, Wm, x0, x1, lx0, lx1);
    const bool in0 = y0 >= i_begin && y0 < i_end, in1 = y1 >= i_begin && y1 < i_end;
    const T* row0 = in0 ? reinterpret_cast<const T*>(tap_smem + (size_t)(2 * j) * vpr) : base + (long long)y0 * Wm;
    const T* row1 = in1 ? reinterpret_cast<const T*>(tap_smem + (size_t)(2 * j + 1) * vpr) : base + (long long)y1 * Wm;
    const float v00 = to_f<T>(row0[x0]), v01 = to_f<T>(row0[x1]);
    const float v10 = to_f<T>(row1[x0]), v11 = to_f<T>(row1[x1]);
    const float rv = (ly0 * (lx0 * v00 + lx1 * v01) + ly1 * (lx0 * v10 + lx1 * v11)) * mscale;
    const long long pix = (long long)r * w + x;
    if (w_f32) w_f32[(long long)n * ldw + pix] = rv;
    const float tv = apply_transform(rv, transform);
    den += tv;
    if (w_bf16) {
      const bf16 q = __float2bfloat16_rn(tv);
      w_bf16[obase + pix] = q;
      den16 += __bfloat162float(q);
    }
  }

  __shared__ double scratch[4 * 32];
  double v[4];
  v[0] = ((double)s[0] + (double)s[1]) + ((double)s[2] + (double)s[3]);
  v[1] = (double)s1m;
  v[2] = (double)den;
  v[3] = (double)den16;
  block_sum<4>(v, scratch);
  if (threadIdx.x == 0) {
    double* o = part + (long long)blockIdx.x * 4;
    o[0] = v[0];
    o[1] = kNeedOneMinus ? v[1] : (double)((long long)band * Wm);
    o[2] = v[2];
    o[3] = v[3];
  }
}

// stats[n] = {sum m, sum (1-m), den, den_bf16}; fixed-order reduction of the chunk partials: one warp per mask, lane k
// sums chunks k, k+32, ... in order, then a fixed shuffle tree (deterministic; the loads of a mask are all in flight at once).
__global__ void __launch_bounds__(256) mask_prep_reduce_kernel(const double* __restrict__ part, int n_masks, int chunks, float mscale,
                                                               int one_minus_direct, float* __restrict__ stats) {
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (n >= n_masks) return;
  double a = 0, b = 0, c = 0, d = 0;
  for (int k = lane; k < chunks; k += 32) {
    const double2* o = reinterpret_cast<const double2*>(part + ((long long)n * chunks + k) * 4);
    const double2 v0 = o[0], v1 = o[1];
    a += v0.x; b += v0.y; c += v1.x; d += v1.y;
  }
  a = warp_sum(a); b = warp_sum(b); c = warp_sum(c); d = warp_sum(d);
  if (lane != 0) return;
  float* s = stats + (long long)n * 4;
  const double sm = a * (double)mscale;
  // one_minus_direct 1: b is sum(1-m) accumulated directly (f32 masks);
  //                  0: b is the element count, sum(1-m) = count - sum (bf16 masks);
  //                  2: u8 masks, exact integers: (count*vmax - sum_bytes) * scale with vmax = round(1/scale)
  double om;
  if (one_minus_direct == 1) om = b;
  else if (one_minus_direct == 2) om = (b * (double)lrintf(1.0f / mscale) - a) * (double)mscale;
  else om = b - sm;
  s[0] = (float)sm;
  s[1] = (float)fmax(om, 0.0);
  s[2] = (float)c;
  s[3] = (float)d;
}

static int pick_chunks(int n_masks, int Hm, int Wm, int h, size_t esize) {
  long long target = (long long)sm_count() * 8;
  long long chunks = (target + n_masks - 1) / n_masks;
  long long by_bytes = ((long long)Hm * Wm * (long long)esize) / 16384;
  if (by_bytes < 1) by_bytes = 1;
  if (chunks > by_bytes) chunks = by_bytes;
  if (chunks > h) chunks = h;
  if (chunks > Hm) chunks = Hm;
  if (chunks < 1) chunks = 1;
  return (int)chunks;
}

}  // namespace cor

using namespace cor;

extern "C" size_t cor_mask_prep_work_bytes(int n_masks, int Hm, int Wm, int h, int w) {
  (void)w;
  // upper bound independent of dtype: chunks <= h
  return (size_t)n_masks * (size_t)(h > 0 ? h : 1) * 4 * sizeof(double);
}

extern "C" int cor_mask_prep(const void* masks, int mask_dtype, float mask_scale, int n_masks, int Hm, int Wm, int h,
                             int w, int transform, float* w_f32, void* w_bf16, long long ldw, int group,
                             long long group_stride, float* stats, void* work, cor_stream_t stream) {
  COR_REQUIRE(masks && stats && work, "cor_mask_prep: null pointer");
  COR_REQUIRE(n_masks > 0 && Hm > 0 && Wm > 0 && h > 0 && w > 0, "cor_mask_prep: bad shape n=%d %dx%d -> %dx%d", n_masks,
              Hm, Wm, h, w);
  COR_REQUIRE(ldw >= (long long)h * w, "cor_mask_prep: ldw %lld < h*w", ldw);
  COR_REQUIRE(transform >= 0 && transform <= 2, "cor_mask_prep: bad transform %d", transform);
  if (group <= 0) { group = 1; group_stride = ldw; }
  COR_REQUIRE(group_stride >= (long long)group * ldw, "cor_mask_prep: group_stride %lld < group*ldw", group_stride);
  const size_t es = mask_dtype == COR_F32 ? 4 : mask_dtype == COR_BF16 ? 2 : 1;
  cudaStream_t st = as_stream(stream);
  double* part = reinterpret_cast<double*>(work);
  int direct = mask_dtype == COR_F32 ? 1 : mask_dtype == COR_BF16 ? 0 : 2;
  // staged kernel: rows are whole aligned 16-byte vectors, <= kMaxRO output rows (and a describable band) per CTA
  const size_t row_bytes = (size_t)Wm * es;
  // measured (profiles/): 4 output rows per CTA is best for fp32/bf16 masks (5 CTAs/SM), 8 for 1-byte masks
  const int max_ro = es == 1 ? 8 : 4;
  int chunks_s = ceil_div(h, max_ro);
  {
    const int want = pick_chunks(n_masks, Hm, Wm, h, es);
    if (want > chunks_s) chunks_s = want;
  }
  const long long band_max = ((long long)ceil_div(h, chunks_s) * Hm + h - 1) / h + 2;
  const size_t smem_s = (size_t)2 * max_ro * row_bytes + (size_t)band_max * sizeof(short) + 16;
  // measured on B200 (profiles/): staged beats the two-phase kernel for every mask dtype (f32 0.70 vs 0.73 ms, u8 0.24 vs
  // 0.49 ms at 1024 masks of 1024^2); the two-phase kernel takes what staged cannot: up-sampling (Hm < h), unaligned
  // rows and bands over budget.
  const bool staged = (row_bytes % 16 == 0) && (((uintptr_t)masks & 15) == 0) && smem_s <= 96 * 1024 && band_max <= kMaxBand &&
                      ceil_div(h, chunks_s) <= max_ro && chunks_s <= h && Hm >= h;
  int chunks = staged ? chunks_s : pick_chunks(n_masks, Hm, Wm, h, es);
  COR_REQUIRE((long long)n_masks * chunks < 2147483647LL, "cor_mask_prep: grid too large");
  dim3 grid((unsigned)(n_masks * chunks));
  if (staged) {
    const int vpr = (int)(row_bytes / 16);
    int L = 1;
    while (L < vpr && L < 256) L <<= 1;
#define COR_PREP_S(T_, OM_)                                                                                                   \
  do {                                                                                                                        \
    COR_CUDA(cudaFuncSetAttribute(mask_prep_staged_kernel<T_, OM_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_s)); \
    mask_prep_staged_kernel<T_, OM_><<<grid, 256, smem_s, st>>>((const T_*)masks, mask_scale, Hm, Wm, h, w, chunks, transform, L, max_ro, w_f32, \
                                                                (bf16*)w_bf16, ldw, group, group_stride, part);               \
  } while (0)
    if (mask_dtype == COR_F32) COR_PREP_S(float, true);
    else if (mask_dtype == COR_BF16) COR_PREP_S(bf16, false);
    else if (mask_dtype == COR_U8) COR_PREP_S(uint8_t, false);
    else COR_REQUIRE(false, "cor_mask_prep: unsupported mask dtype %d", mask_dtype);
#undef COR_PREP_S
  } else {
    switch (mask_dtype) {
      case COR_F32:
        mask_prep_kernel<float, true><<<grid, 256, 0, st>>>((const float*)masks, mask_scale, Hm, Wm, h, w, chunks, transform,
                                                            w_f32, (bf16*)w_bf16, ldw, group, group_stride, part);
        break;
      case COR_BF16:
        mask_prep_kernel<bf16, false><<<grid, 256, 0, st>>>((const bf16*)masks, mask_scale, Hm, Wm, h, w, chunks, transform,
                                                            w_f32, (bf16*)w_bf16, ldw, group, group_stride, part);
        break;
      case COR_U8:
        mask_prep_kernel<uint8_t, false><<<grid, 256, 0, st>>>((const uint8_t*)masks, mask_scale, Hm, Wm, h, w, chunks,
                                                               transform, w_f32, (bf16*)w_bf16, ldw, group, group_stride, part);
        break;
      default:
        COR_REQUIRE(false, "cor_mask_prep: unsupported mask dtype %d", mask_dtype);
    }
  }
  int rc = check_launch("mask_prep_kernel");
  if (rc) return rc;
  mask_prep_reduce_kernel<<<ceil_div(n_masks, 8), 256, 0, st>>>(part, n_masks, chunks, mask_scale, direct, stats);
  return check_launch("mask_prep_reduce_kernel");
}
