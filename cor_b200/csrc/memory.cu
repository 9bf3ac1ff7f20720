// Cross-batch region memory (XBM-style; Class N, no reference implementation): a ring buffer of K bf16 unit rows whose
// rows serve the InfoNCE as extra negatives.  Its state lives in device memory, int32 {head, count, arrivals, 0}, so that
// a captured CUDA graph advances it at every replay:
//   cor_memory_enqueue  writes a batch at slots (head + i) mod K and advances {head, count}: one launch, no host sync;
//   cor_memory_scan     the tensor-core log-sum-exp kernel (sim_umma_ts.cu) over the first min(K, count) rows -- the
//                       valid ones: the ring is full before it wraps, and reset() empties it;
//   cor_memory_dq       (nce_bwd_umma.cu) the queries' gradient through the memory rows.
// Row ids (as XBM's labels): cor_memory_enqueue_ids also writes an int64 id ring [K] at the same slots, and
// cor_memory_exclude turns it and the queries' ids into a bit mask [Nq][ceil(K / 32)] over ring slots; the _x twins of the
// scan and the dQ leave every masked (query, row) pair out: slot r is masked for query q iff r < count, id[r] >= 0 and
// id[r] == query_id[q].
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
// head before it arrives, so the last CTA's update of the state follows every read of the old head.  kIds: the thread
// that writes a row's first vector also writes the row's id: ids[i / group] on the first row of each group, -1 on the
// others and everywhere when ids is NULL, so no id of an overwritten row survives a wrap.
template <typename T, bool kIds = false>
__global__ void __launch_bounds__(256) memory_enqueue_kernel(const T* __restrict__ rows, int n, int C, bf16* __restrict__ bank, int K,
                                                             int* __restrict__ state, long long* __restrict__ ring = nullptr,
                                                             const long long* __restrict__ ids = nullptr, int group = 1) {
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
    if constexpr (kIds) {
      if (c == 0) ring[slot] = (ids && i % group == 0) ? ids[i / group] : -1ll;
    }
  }
  if (!arrive_last(reinterpret_cast<unsigned*>(state + 2), gridDim.x, &last)) return;
  if (threadIdx.x == 0) {
    state[0] = (int)(((long long)head + n) % K);
    state[1] = min(state[1] + n, K);
  }
}

// One warp per 32-slot chunk w of the ring: lane j holds the id of slot 32 w + j (-1 past the fill), and one ballot per
// query gives the query's mask word.  8 warps per CTA.
__global__ void __launch_bounds__(256) memory_exclude_kernel(const long long* __restrict__ ring, int K, const int* __restrict__ state,
                                                             const long long* __restrict__ qids, int Nq, unsigned* __restrict__ mask) {
  const int nw = (K + 31) / 32;
  const int w = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= nw) return;
  const int fill = min(max(state[1], 0), K);
  const int slot = w * 32 + lane;
  const long long id = slot < fill ? ring[slot] : -1ll;
  for (int q = 0; q < Nq; ++q) {
    const long long qid = __ldg(qids + q);
    const unsigned bits = __ballot_sync(0xffffffffu, id >= 0 && id == qid);
    if (lane == 0) mask[(long long)q * nw + w] = bits;
  }
}

int mem_width_ok(int D, const char* who) {
  COR_REQUIRE(D == 64 || D == 128 || D == 192 || D == 256, "%s: row width D=%d must be 64, 128, 192 or 256 (the tensor-core kernels' widths)",
              who, D);
  return COR_OK;
}

int mem_enqueue_grid(int n, int C) {
  const long long nvec = (long long)n * C / 8;
  long long grid = (nvec + 255) / 256;
  if (grid > (long long)sm_count() * 8) grid = (long long)sm_count() * 8;
  return (int)grid;
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
  const int grid = mem_enqueue_grid(n, C);
  if (rows_dtype == COR_F32)
    memory_enqueue_kernel<float><<<grid, 256, 0, as_stream(stream)>>>((const float*)rows, n, C, (bf16*)bank, K, state);
  else
    memory_enqueue_kernel<bf16><<<grid, 256, 0, as_stream(stream)>>>((const bf16*)rows, n, C, (bf16*)bank, K, state);
  return check_launch("memory_enqueue_kernel");
}

extern "C" int cor_memory_enqueue_ids(const void* rows, int rows_dtype, int n, int C, void* bank, int K, int* state, long long* ids_ring,
                                      const long long* ids, int group, cor_stream_t stream) {
  COR_REQUIRE(rows && bank && state && ids_ring, "cor_memory_enqueue_ids: null pointer");
  COR_REQUIRE(K >= 1 && n >= 1 && n <= K, "cor_memory_enqueue_ids: need 1 <= n <= K (n=%d K=%d)", n, K);
  COR_REQUIRE(group >= 1 && n % group == 0, "cor_memory_enqueue_ids: group=%d must be >= 1 and divide n=%d", group, n);
  int rc = mem_width_ok(C, "cor_memory_enqueue_ids");
  if (rc) return rc;
  COR_REQUIRE(rows_dtype == COR_F32 || rows_dtype == COR_BF16, "cor_memory_enqueue_ids: rows must be f32 or bf16 (dtype %d)", rows_dtype);
  COR_REQUIRE((((uintptr_t)rows | (uintptr_t)bank) & 15) == 0, "cor_memory_enqueue_ids: rows and bank must be 16-byte aligned");
  const int grid = mem_enqueue_grid(n, C);
  if (rows_dtype == COR_F32)
    memory_enqueue_kernel<float, true><<<grid, 256, 0, as_stream(stream)>>>((const float*)rows, n, C, (bf16*)bank, K, state, ids_ring, ids,
                                                                            group);
  else
    memory_enqueue_kernel<bf16, true><<<grid, 256, 0, as_stream(stream)>>>((const bf16*)rows, n, C, (bf16*)bank, K, state, ids_ring, ids,
                                                                           group);
  return check_launch("memory_enqueue_kernel");
}

extern "C" size_t cor_memory_exclude_bytes(int Nq, int K) {
  if (Nq <= 0 || K <= 0) return 0;
  return (size_t)Nq * ceil_div(K, 32) * sizeof(unsigned);
}

extern "C" int cor_memory_exclude(const long long* ids_ring, int K, const int* state, const long long* query_ids, int Nq, unsigned* exclude,
                                  cor_stream_t stream) {
  COR_REQUIRE(ids_ring && state && query_ids && exclude, "cor_memory_exclude: null pointer");
  COR_REQUIRE(K >= 1 && Nq >= 1, "cor_memory_exclude: need K >= 1 and Nq >= 1 (K=%d Nq=%d)", K, Nq);
  memory_exclude_kernel<<<ceil_div(ceil_div(K, 32), 8), 256, 0, as_stream(stream)>>>(ids_ring, K, state, query_ids, Nq, exclude);
  return check_launch("memory_exclude_kernel");
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

extern "C" int cor_memory_scan_x(const void* bank, int K, const int* state, const void* queries, int Nq, int D, float inv_tau,
                                 const float* logit_scale, const unsigned* exclude, void* work, int* nparts, cor_stream_t stream) {
  COR_REQUIRE(bank && state && queries && exclude && work && nparts, "cor_memory_scan_x: null pointer");
  COR_REQUIRE(K >= 1 && Nq >= 1, "cor_memory_scan_x: need K >= 1 and Nq >= 1 (K=%d Nq=%d)", K, Nq);
  int rc = mem_width_ok(D, "cor_memory_scan_x");
  if (rc) return rc;
  return sim_umma_ts_launch(bank, queries, K, Nq, D, inv_tau, logit_scale, work, nparts, as_stream(stream), state + 1, exclude);
}
