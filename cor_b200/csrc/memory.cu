// Cross-batch region memory (XBM-style; Class N, no reference implementation): a ring buffer of K bf16 unit rows whose
// rows serve the InfoNCE as extra negatives.  Its state lives in device memory, int32 {head, count, arrivals, 0}, so that
// a captured CUDA graph advances it at every replay:
//   cor_memory_enqueue  writes a batch at slots (head + i) mod K and advances {head, count}: one launch, no host sync;
//   cor_memory_scan     the tensor-core log-sum-exp kernel (sim_umma_ts.cu) over the first min(K, count) rows -- the
//                       valid ones: the ring is full before it wraps, and reset() empties it;
//   cor_memory_dq       (nce_bwd_umma.cu) the queries' gradient through the memory rows.
// The memory is scanned on tensor cores only: at 16 queries a streaming scan does 16 flop per byte of bf16 row, more than
// the CUDA cores sustain at HBM rate.
#include "common.cuh"

namespace cor {

namespace {

constexpr int kMemStateWords = 4;

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}

// grid-stride over 8-element vectors of the n x C batch (C % 8 == 0: a vector never spans two rows).  Every CTA reads
// head before it arrives, so the last CTA's update of the state follows every read of the old head.
template <typename T>
__global__ void __launch_bounds__(256) memory_enqueue_kernel(const T* __restrict__ rows, int n, int C, bf16* __restrict__ bank, int K,
                                                             int* __restrict__ state) {
  __shared__ bool last;
  const int head = state[0];
  const long long nvec = (long long)n * C / 8;
  for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += (long long)gridDim.x * blockDim.x) {
    const long long e = v * 8, i = e / C;
    const int c = (int)(e - i * C);
    const long long slot = ((long long)head + i) % K;
    uint4 out;
    if constexpr (sizeof(T) == 4) {
      const float4 a = *reinterpret_cast<const float4*>(rows + e), b = *reinterpret_cast<const float4*>(rows + e + 4);
      out = make_uint4(pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w), pack_bf16x2(b.x, b.y), pack_bf16x2(b.z, b.w));
    } else {
      out = *reinterpret_cast<const uint4*>(rows + e);
    }
    *reinterpret_cast<uint4*>(bank + slot * C + c) = out;
  }
  if (!arrive_last(reinterpret_cast<unsigned*>(state + 2), gridDim.x, &last)) return;
  if (threadIdx.x == 0) {
    state[0] = (int)(((long long)head + n) % K);
    state[1] = min(state[1] + n, K);
  }
}

int mem_width_ok(int D, const char* who) {
  COR_REQUIRE(D == 64 || D == 128 || D == 192 || D == 256, "%s: row width D=%d must be 64, 128, 192 or 256 (the tensor-core kernels' widths)",
              who, D);
  return COR_OK;
}

int mem_scan_ctas(int Nq, int K) {
  const int qtiles = ceil_div(Nq, kMemQT), ntiles = ceil_div(K, 128);
  int gx = sm_count() / qtiles;
  if (gx < 1) gx = 1;
  return gx > ntiles ? ntiles : gx;
}

}  // namespace

}  // namespace cor

using namespace cor;

extern "C" int cor_memory_state_words(void) { return kMemStateWords; }

extern "C" int cor_memory_reset(int* state, cor_stream_t stream) {
  COR_REQUIRE(state, "cor_memory_reset: null state");
  COR_CUDA(cudaMemsetAsync(state, 0, kMemStateWords * sizeof(int), as_stream(stream)));
  return COR_OK;
}

extern "C" int cor_memory_enqueue(const void* rows, int rows_dtype, int n, int C, void* bank, int K, int* state, cor_stream_t stream) {
  COR_REQUIRE(rows && bank && state, "cor_memory_enqueue: null pointer");
  COR_REQUIRE(K >= 1 && n >= 1 && n <= K, "cor_memory_enqueue: need 1 <= n <= K (n=%d K=%d)", n, K);
  int rc = mem_width_ok(C, "cor_memory_enqueue");
  if (rc) return rc;
  COR_REQUIRE(rows_dtype == COR_F32 || rows_dtype == COR_BF16, "cor_memory_enqueue: rows must be f32 or bf16 (dtype %d)", rows_dtype);
  COR_REQUIRE((((uintptr_t)rows | (uintptr_t)bank) & 15) == 0, "cor_memory_enqueue: rows and bank must be 16-byte aligned");
  const long long nvec = (long long)n * C / 8;
  long long grid = (nvec + 255) / 256;
  if (grid > (long long)sm_count() * 8) grid = (long long)sm_count() * 8;
  if (rows_dtype == COR_F32)
    memory_enqueue_kernel<float><<<(int)grid, 256, 0, as_stream(stream)>>>((const float*)rows, n, C, (bf16*)bank, K, state);
  else
    memory_enqueue_kernel<bf16><<<(int)grid, 256, 0, as_stream(stream)>>>((const bf16*)rows, n, C, (bf16*)bank, K, state);
  return check_launch("memory_enqueue_kernel");
}

extern "C" size_t cor_memory_scan_work_bytes(int Nq, int K, int D) {
  if (Nq <= 0 || K <= 0 || D <= 0) return 0;
  return (size_t)ceil_div(Nq, kMemQT) * mem_scan_ctas(Nq, K) * kMemQT * 2 * sizeof(float);
}

extern "C" int cor_memory_scan(const void* bank, int K, const int* state, const void* queries, int Nq, int D, float inv_tau,
                               const float* logit_scale, void* work, int* nparts, cor_stream_t stream) {
  COR_REQUIRE(bank && state && queries && work && nparts, "cor_memory_scan: null pointer");
  COR_REQUIRE(K >= 1 && Nq >= 1, "cor_memory_scan: need K >= 1 and Nq >= 1 (K=%d Nq=%d)", K, Nq);
  int rc = mem_width_ok(D, "cor_memory_scan");
  if (rc) return rc;
  return sim_umma_ts_launch(bank, queries, K, Nq, D, inv_tau, logit_scale, work, nparts, as_stream(stream), state + 1);
}
