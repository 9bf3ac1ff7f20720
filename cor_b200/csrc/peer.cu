// Region-row exchange between the GPUs of one node over NVLink peer memory (SURVEY.md §8e).
//
// One process per GPU.  Every rank owns a "symmetric" allocation (plain cudaMalloc, exported with CUDA IPC and mapped
// by its peers), holding
//     pub   [n_local, C] bf16   the rank's normalised region rows      (written by cor_rows_finalize)
//     gall  [world*n_local, C] f32   d loss / d (all gathered rows)    (written by cor_infonce_bwd)
//     flags [2 channels][2 phases][kPeerMaxWorld] u32                  (written by the PEERS, polled locally)
// and two kernels replace the NCCL pair of the step:
//     peer_gather_kernel   all[p*n : (p+1)*n] = pub of rank p                 (all-gather, pulled over NVLink)
//     peer_reduce_kernel   out = sum_p gall_p[rank*n : (rank+1)*n], p ascending  (reduce-scatter, fixed order -> the
//                          result is bit-identical on every run)
// Both are "enter barrier -> pull -> exit barrier" on monotonically increasing epochs kept in device memory, so the
// launches carry no per-step host state and replay inside a CUDA graph.  enter(e): "what I produced for step e is
// in my buffer" (stream order put the producer kernel before this one); exit(e): "I have finished reading yours" -
// a rank leaves the kernel only after every peer has signalled exit(e), hence the next step's producer kernel may
// overwrite the buffer.  Waits are bounded by COR_PEER_TIMEOUT_S of globaltimer (default 600 s, 0 = wait for ever):
// on expiry the kernel does NOT trap (that would take the whole CUDA context with it, where the NCCL pair this
// replaces would simply have blocked through a slow rank's checkpoint save) -- it records the epoch in the local
// error word (state[kErrWord]) and carries on; the host raises CorError from PeerExchange.check().
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace cor {

constexpr int kPeerMaxWorld = 16;
constexpr int kPeerThreads = 512;
constexpr int kPeerCtas = 64;
constexpr int kStateWords = 4;
constexpr int kErrWord = 2 * kStateWords;       // state[8]: 0, or 0x80000000 | epoch of the first wait that expired

// flags block of one rank: [channel][phase][source rank]
__device__ __forceinline__ unsigned* flag_slot(unsigned* flags, int channel, int phase, int src) {
  return flags + ((channel * 2 + phase) * kPeerMaxWorld + src);
}

__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint4 ld_peer16(const void* p) {
  uint4 r;
  asm volatile("ld.relaxed.sys.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
  return r;
}
__device__ __forceinline__ unsigned long long now_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

struct PeerCtl {
  unsigned* const* flags;   // device array [world]: every rank's flag block (entry `rank` is the local one)
  unsigned* state;          // local: [channel] {epoch done, CTA counter, epoch signalled, -}, then the error word
  int rank, world, channel;
  unsigned long long timeout_ns;   // 0 = no limit
};

__device__ __forceinline__ void wait_flag(const unsigned* p, unsigned epoch, const PeerCtl& c) {
  const unsigned long long t0 = now_ns();
  while ((int)(ld_acquire_sys(p) - epoch) < 0) {
    __nanosleep(64);
    if (c.timeout_ns && now_ns() - t0 > c.timeout_ns) {
      atomicCAS(&c.state[kErrWord], 0u, 0x80000000u | epoch);     // first failure wins; the host reports it
      return;
    }
  }
}

// "What I produced for my next epoch on this channel is in my buffer": one tiny CTA right after the producer kernel,
// so that whatever the stream runs between this and the exchange kernel hides the skew between the ranks.
__global__ void peer_signal_kernel(PeerCtl c) {
  unsigned* st = c.state + kStateWords * c.channel;
  const unsigned epoch = st[2] + 1u;
  if (threadIdx.x < c.world) {
    __threadfence_system();
    st_release_sys(flag_slot(c.flags[threadIdx.x], c.channel, 0, c.rank), epoch);
  }
  __syncthreads();
  if (threadIdx.x == 0) st[2] = epoch;
}

// Before the producer overwrites the buffer: every peer has finished reading what the last exchange published.
__global__ void peer_wait_exit_kernel(PeerCtl c) {
  const unsigned done = c.state[kStateWords * c.channel];
  if (threadIdx.x < c.world) wait_flag(flag_slot(c.flags[c.rank], c.channel, 1, threadIdx.x), done, c);
}

// Every CTA waits until all peers have signalled the epoch this launch serves.
__device__ __forceinline__ unsigned peer_enter(const PeerCtl& c) {
  const unsigned epoch = c.state[kStateWords * c.channel] + 1u;
  if (threadIdx.x < c.world) wait_flag(flag_slot(c.flags[c.rank], c.channel, 0, threadIdx.x), epoch, c);
  __syncthreads();
  return epoch;
}

// The last CTA to get here tells the peers "rank has finished reading" (nobody waits for it here: see
// peer_wait_exit_kernel) and publishes the new epoch for the next launch.
__device__ __forceinline__ void peer_exit(const PeerCtl& c, unsigned epoch) {
  __shared__ int last;
  unsigned* st = c.state + kStateWords * c.channel;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = (atomicAdd(&st[1], 1u) == gridDim.x - 1);
  __syncthreads();
  if (!last) return;
  if (threadIdx.x < c.world) {
    __threadfence_system();
    st_release_sys(flag_slot(c.flags[threadIdx.x], c.channel, 1, c.rank), epoch);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    st[1] = 0u;
    st[0] = epoch;
  }
}

// all[p] = src[p] for every rank p; `vecs` 16-byte vectors per rank.
__global__ void __launch_bounds__(kPeerThreads) peer_gather_kernel(const uint4* const* __restrict__ src, uint4* __restrict__ all,
                                                                   long long vecs, PeerCtl c) {
  const unsigned epoch = peer_enter(c);
  const long long total = vecs * c.world, stride = (long long)gridDim.x * blockDim.x;
  constexpr int U = 4;
  for (long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < total; i0 += stride * U) {
    uint4 v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = i0 + u * stride;
      if (i < total) {
        // start with the rank's own slice and walk the ring, so the ranks do not all pull from rank 0 first
        const int k = (int)(i / vecs);
        const int p = (c.rank + k) % c.world;
        v[u] = ld_peer16(src[p] + (i - (long long)k * vecs));
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = i0 + u * stride;
      if (i < total) {
        const int k = (int)(i / vecs);
        const int p = (c.rank + k) % c.world;
        all[(long long)p * vecs + (i - (long long)k * vecs)] = v[u];
      }
    }
  }
  peer_exit(c, epoch);
}

// ---- fused all-gather + similarity (few local queries) ----------------------------------------------------------------
// The forward exchange and its consumer in ONE kernel: every region row is pulled over NVLink exactly once, written into
// the local gathered buffer (the backward and the target-logit gather read it there) and, while it is in registers, dotted
// with this rank's <= 16 queries -- the online log-sum-exp partials of the InfoNCE forward.  Replaces peer_gather_kernel +
// the similarity kernel of the step (two launches, two passes over the gathered rows, one of them through HBM).
// Warp per row, one 16-byte vector per lane (D <= 256), two rows prefetched ahead of the row being processed so the
// ~2 us NVLink latency overlaps the arithmetic; rows are walked ring-wise starting with the rank's own slice.
// part layout = the streaming similarity kernel's: [gridDim.x][kQT][2] (running max, sum) for cor_infonce_tail.
constexpr int kPgsThreads = 256;
__global__ void __launch_bounds__(kPgsThreads) peer_gather_sim_kernel(const uint4* const* __restrict__ src, uint4* __restrict__ all,
                                                                      long long n_local, int D, const bf16* __restrict__ queries, int Nq,
                                                                      float inv_tau, const float* __restrict__ scale, float* __restrict__ part,
                                                                      PeerCtl c) {
  extern __shared__ float qs[];   // [kQT][D]
  __shared__ float cm[kPgsThreads / 32][kQT], cs[kPgsThreads / 32][kQT];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < kQT * D; i += blockDim.x) {
    const int q = i / D, d = i - q * D;
    qs[i] = q < Nq ? __bfloat162float(queries[(long long)q * D + d]) : 0.f;
  }
  const unsigned epoch = peer_enter(c);          // includes a __syncthreads: qs is complete, every peer's rows are published
  if (scale) inv_tau = __ldg(scale);
  const int nvec = D / 8;
  const bool has = lane < nvec;
  const long long total = n_local * c.world, step = (long long)gridDim.x * (kPgsThreads / 32);
  auto fetch = [&](long long g, uint4& v, long long& dst) {
    const int k = (int)(g / n_local);
    const int p = (c.rank + k) % c.world;
    const long long i = g - (long long)k * n_local;
    dst = ((long long)p * n_local + i) * nvec + lane;
    v = ld_peer16(src[p] + i * nvec + lane);
  };
  float m = -INFINITY, s = 0.f;
  long long g = (long long)blockIdx.x * (kPgsThreads / 32) + warp;
  uint4 v0 = make_uint4(0u, 0u, 0u, 0u), v1 = v0;
  long long d0 = 0, d1 = 0;
  if (has && g < total) fetch(g, v0, d0);
  if (has && g + step < total) fetch(g + step, v1, d1);
  for (; g < total; g += step) {
    const uint4 raw = v0;
    const long long dst = d0;
    v0 = v1;
    d0 = d1;
    if (has && g + 2 * step < total) fetch(g + 2 * step, v1, d1);
    float a[kQT];
#pragma unroll
    for (int q = 0; q < kQT; ++q) a[q] = 0.f;
    if (has) {
      all[dst] = raw;
      float f[8];
      f[0] = bf16lo(raw.x); f[1] = bf16hi(raw.x); f[2] = bf16lo(raw.y); f[3] = bf16hi(raw.y);
      f[4] = bf16lo(raw.z); f[5] = bf16hi(raw.z); f[6] = bf16lo(raw.w); f[7] = bf16hi(raw.w);
#pragma unroll
      for (int q = 0; q < kQT; ++q) {
        const float4 x = *reinterpret_cast<const float4*>(&qs[q * D + lane * 8]);
        const float4 y = *reinterpret_cast<const float4*>(&qs[q * D + lane * 8 + 4]);
        a[q] = fmaf(f[0], x.x, a[q]); a[q] = fmaf(f[1], x.y, a[q]); a[q] = fmaf(f[2], x.z, a[q]); a[q] = fmaf(f[3], x.w, a[q]);
        a[q] = fmaf(f[4], y.x, a[q]); a[q] = fmaf(f[5], y.y, a[q]); a[q] = fmaf(f[6], y.z, a[q]); a[q] = fmaf(f[7], y.w, a[q]);
      }
    }
    const float sv = transpose_reduce16(a, lane);
    if (lane < kQT && lane < Nq) {
      const float x = sv * inv_tau;
      if (x > m) { s = s * __expf(m - x) + 1.f; m = x; } else { s += __expf(x - m); }
    }
  }
  if (lane < kQT) { cm[warp][lane] = m; cs[warp][lane] = s; }
  __syncthreads();
  if (threadIdx.x < kQT) {
    float M = -INFINITY;
    for (int w = 0; w < kPgsThreads / 32; ++w) M = fmaxf(M, cm[w][threadIdx.x]);
    float Ssum = 0.f;
    for (int w = 0; w < kPgsThreads / 32; ++w) Ssum += (cm[w][threadIdx.x] == -INFINITY) ? 0.f : cs[w][threadIdx.x] * __expf(cm[w][threadIdx.x] - M);
    float* o = part + ((long long)blockIdx.x * kQT + threadIdx.x) * 2;
    o[0] = M; o[1] = Ssum;
  }
  peer_exit(c, epoch);
}

static int peer_gather_sim_grid(long long rows) {
  long long g = (rows + 2 * (kPgsThreads / 32) - 1) / (2 * (kPgsThreads / 32));      // >= 2 rows per warp
  const long long cap = sm_count();
  if (g > cap) g = cap;
  return (int)(g < 1 ? 1 : g);
}

// out[i] = sum over ranks p (ascending) of src[p][rank*vecs + i]; float4 vectors.
template <int W>
__device__ __forceinline__ void reduce_body(const uint4* const* __restrict__ src, float4* __restrict__ out, long long vecs, int rank,
                                            int world) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < vecs; i += stride) {
    uint4 v[W];
#pragma unroll
    for (int p = 0; p < W; ++p)
      if (p < world) v[p] = ld_peer16(src[p] + (long long)rank * vecs + i);
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int p = 0; p < W; ++p)
      if (p < world) {
        a.x += __uint_as_float(v[p].x);
        a.y += __uint_as_float(v[p].y);
        a.z += __uint_as_float(v[p].z);
        a.w += __uint_as_float(v[p].w);
      }
    out[i] = a;
  }
}

__global__ void __launch_bounds__(kPeerThreads) peer_reduce_kernel(const uint4* const* __restrict__ src, float4* __restrict__ out,
                                                                   long long vecs, PeerCtl c) {
  const unsigned epoch = peer_enter(c);
  if (c.world <= 2) reduce_body<2>(src, out, vecs, c.rank, c.world);
  else if (c.world <= 4) reduce_body<4>(src, out, vecs, c.rank, c.world);
  else if (c.world <= 8) reduce_body<8>(src, out, vecs, c.rank, c.world);
  else reduce_body<kPeerMaxWorld>(src, out, vecs, c.rank, c.world);
  peer_exit(c, epoch);
}

static int peer_grid(long long vecs) {
  long long g = (vecs + kPeerThreads - 1) / kPeerThreads;
  if (g < 1) g = 1;
  return (int)(g < kPeerCtas ? g : kPeerCtas);
}

}  // namespace cor

using namespace cor;

extern "C" {

int cor_peer_max_world(void) { return kPeerMaxWorld; }
size_t cor_peer_flag_bytes(void) { return sizeof(unsigned) * 2 * 2 * kPeerMaxWorld; }
size_t cor_peer_state_bytes(void) { return sizeof(unsigned) * (2 * kStateWords + 4); }
int cor_peer_error_word(void) { return kErrWord; }

int cor_peer_alloc(int device, size_t bytes, void** ptr) {
  COR_REQUIRE(ptr && bytes > 0, "cor_peer_alloc: bad arguments");
  int prev = 0;
  COR_CUDA(cudaGetDevice(&prev));
  COR_CUDA(cudaSetDevice(device));
  cudaError_t e = cudaMalloc(ptr, bytes);
  if (e == cudaSuccess) e = cudaMemset(*ptr, 0, bytes);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  cudaSetDevice(prev);
  if (e != cudaSuccess) {
    set_error("cor_peer_alloc(%zu bytes): %s", bytes, cudaGetErrorString(e));
    return COR_ECUDA;
  }
  return COR_OK;
}

int cor_peer_free(void* ptr) {
  if (ptr) COR_CUDA(cudaFree(ptr));
  return COR_OK;
}

int cor_peer_export(void* ptr, unsigned char* handle64) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  COR_REQUIRE(ptr && handle64, "cor_peer_export: bad arguments");
  cudaIpcMemHandle_t h;
  COR_CUDA(cudaIpcGetMemHandle(&h, ptr));
  memcpy(handle64, &h, 64);
  return COR_OK;
}

int cor_peer_open(int device, const unsigned char* handle64, void** ptr) {
  COR_REQUIRE(ptr && handle64, "cor_peer_open: bad arguments");
  int prev = 0;
  COR_CUDA(cudaGetDevice(&prev));
  COR_CUDA(cudaSetDevice(device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  cudaError_t e = cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
  cudaSetDevice(prev);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("cor_peer_open: %s", cudaGetErrorString(e));
    return COR_ECUDA;
  }
  return COR_OK;
}

int cor_peer_close(void* ptr) {
  if (ptr) COR_CUDA(cudaIpcCloseMemHandle(ptr));
  return COR_OK;
}

// COR_PEER_TIMEOUT_S: seconds a wait may last before the error word is set (default 600; 0 = unbounded)
static unsigned long long peer_timeout_ns() {
  double s = 600.0;                                   // read per launch: a getenv is nothing beside a kernel launch
  if (const char* e = getenv("COR_PEER_TIMEOUT_S")) s = atof(e);
  return s <= 0.0 ? 0ull : (unsigned long long)(s * 1e9);
}

static int peer_ctl(const char* what, void* const* peer_flags, void* state, int rank, int world, int channel, PeerCtl* c) {
  COR_REQUIRE(peer_flags && state, "%s: null pointer", what);
  COR_REQUIRE(world >= 1 && world <= kPeerMaxWorld && rank >= 0 && rank < world, "%s: rank %d / world %d (max %d)", what, rank, world,
              kPeerMaxWorld);
  COR_REQUIRE(channel == 0 || channel == 1, "%s: channel %d", what, channel);
  *c = PeerCtl{reinterpret_cast<unsigned* const*>(peer_flags), reinterpret_cast<unsigned*>(state), rank, world, channel, peer_timeout_ns()};
  return COR_OK;
}

int cor_peer_signal(void* const* peer_flags, void* state, int rank, int world, int channel, cor_stream_t stream) {
  PeerCtl c;
  int rc = peer_ctl("cor_peer_signal", peer_flags, state, rank, world, channel, &c);
  if (rc) return rc;
  peer_signal_kernel<<<1, 32, 0, as_stream(stream)>>>(c);
  return check_launch("peer_signal_kernel");
}

int cor_peer_wait_exit(void* const* peer_flags, void* state, int rank, int world, int channel, cor_stream_t stream) {
  PeerCtl c;
  int rc = peer_ctl("cor_peer_wait_exit", peer_flags, state, rank, world, channel, &c);
  if (rc) return rc;
  peer_wait_exit_kernel<<<1, 32, 0, as_stream(stream)>>>(c);
  return check_launch("peer_wait_exit_kernel");
}

int cor_peer_gather_rows(const void* const* peer_src, void* all, long long bytes_per_rank, void* const* peer_flags, void* state,
                         int rank, int world, int channel, cor_stream_t stream) {
  COR_REQUIRE(peer_src && all && peer_flags && state, "cor_peer_gather_rows: null pointer");
  COR_REQUIRE(world >= 1 && world <= kPeerMaxWorld && rank >= 0 && rank < world, "cor_peer_gather_rows: rank %d / world %d (max %d)", rank,
              world, kPeerMaxWorld);
  COR_REQUIRE(channel == 0 || channel == 1, "cor_peer_gather_rows: channel %d", channel);
  COR_REQUIRE(bytes_per_rank > 0 && bytes_per_rank % 16 == 0 && (uintptr_t)all % 16 == 0, "cor_peer_gather_rows: %lld bytes per rank must be a positive multiple of 16, 16-byte aligned", bytes_per_rank);
  PeerCtl c{reinterpret_cast<unsigned* const*>(peer_flags), reinterpret_cast<unsigned*>(state), rank, world, channel, peer_timeout_ns()};
  const long long vecs = bytes_per_rank / 16;
  peer_gather_kernel<<<peer_grid(vecs * world), kPeerThreads, 0, as_stream(stream)>>>(reinterpret_cast<const uint4* const*>(peer_src),
                                                                                     reinterpret_cast<uint4*>(all), vecs, c);
  return check_launch("peer_gather_kernel");
}

size_t cor_peer_gather_sim_work_bytes(void) { return (size_t)sm_count() * kQT * 2 * sizeof(float) + 16; }

static int peer_gather_sim_launch(const void* const* peer_src, void* all, long long n_local, int D, const void* queries, int Nq,
                                 float inv_tau, const float* scale, float* part, int* nparts, void* const* peer_flags, void* state, int rank,
                                 int world, int channel, cor_stream_t stream) {
  COR_REQUIRE(peer_src && all && queries && part && nparts && peer_flags && state, "cor_peer_gather_sim: null pointer");
  COR_REQUIRE(world >= 1 && world <= kPeerMaxWorld && rank >= 0 && rank < world, "cor_peer_gather_sim: rank %d / world %d (max %d)", rank,
              world, kPeerMaxWorld);
  COR_REQUIRE(channel == 0 || channel == 1, "cor_peer_gather_sim: channel %d", channel);
  COR_REQUIRE(n_local > 0 && D > 0 && D % 8 == 0 && D <= 256, "cor_peer_gather_sim: need D %% 8 == 0 and D <= 256 (D=%d)", D);
  COR_REQUIRE(Nq > 0 && Nq <= kQT, "cor_peer_gather_sim: at most %d local queries (Nq=%d)", kQT, Nq);
  COR_REQUIRE((uintptr_t)all % 16 == 0, "cor_peer_gather_sim: gathered buffer must be 16-byte aligned");
  PeerCtl c{reinterpret_cast<unsigned* const*>(peer_flags), reinterpret_cast<unsigned*>(state), rank, world, channel, peer_timeout_ns()};
  const int grid = peer_gather_sim_grid(n_local * world);
  const size_t smem = (size_t)kQT * D * sizeof(float);
  peer_gather_sim_kernel<<<grid, kPgsThreads, smem, as_stream(stream)>>>(reinterpret_cast<const uint4* const*>(peer_src),
                                                                        reinterpret_cast<uint4*>(all), n_local, D,
                                                                        reinterpret_cast<const bf16*>(queries), Nq, inv_tau, scale, part, c);
  *nparts = grid;
  return check_launch("peer_gather_sim_kernel");
}

int cor_peer_gather_sim(const void* const* peer_src, void* all, long long n_local, int D, const void* queries, int Nq, float inv_tau,
                        float* part, int* nparts, void* const* peer_flags, void* state, int rank, int world, int channel,
                        cor_stream_t stream) {
  return peer_gather_sim_launch(peer_src, all, n_local, D, queries, Nq, inv_tau, nullptr, part, nparts, peer_flags, state, rank, world,
                                channel, stream);
}

int cor_peer_gather_sim_ls(const void* const* peer_src, void* all, long long n_local, int D, const void* queries, int Nq,
                           const float* logit_scale, float* part, int* nparts, void* const* peer_flags, void* state, int rank, int world,
                           int channel, cor_stream_t stream) {
  COR_REQUIRE(logit_scale, "cor_peer_gather_sim_ls: null logit_scale");
  return peer_gather_sim_launch(peer_src, all, n_local, D, queries, Nq, 0.f, logit_scale, part, nparts, peer_flags, state, rank, world,
                                channel, stream);
}

int cor_peer_reduce_rows(const void* const* peer_src, float* out, long long floats_per_rank, void* const* peer_flags, void* state,
                         int rank, int world, int channel, cor_stream_t stream) {
  COR_REQUIRE(peer_src && out && peer_flags && state, "cor_peer_reduce_rows: null pointer");
  COR_REQUIRE(world >= 1 && world <= kPeerMaxWorld && rank >= 0 && rank < world, "cor_peer_reduce_rows: rank %d / world %d (max %d)", rank,
              world, kPeerMaxWorld);
  COR_REQUIRE(channel == 0 || channel == 1, "cor_peer_reduce_rows: channel %d", channel);
  COR_REQUIRE(floats_per_rank > 0 && floats_per_rank % 4 == 0 && (uintptr_t)out % 16 == 0, "cor_peer_reduce_rows: %lld floats per rank must be a positive multiple of 4, 16-byte aligned", floats_per_rank);
  PeerCtl c{reinterpret_cast<unsigned* const*>(peer_flags), reinterpret_cast<unsigned*>(state), rank, world, channel, peer_timeout_ns()};
  const long long vecs = floats_per_rank / 4;
  peer_reduce_kernel<<<peer_grid(vecs), kPeerThreads, 0, as_stream(stream)>>>(reinterpret_cast<const uint4* const*>(peer_src),
                                                                             reinterpret_cast<float4*>(out), vecs, c);
  return check_launch("peer_reduce_kernel");
}

}  // extern "C"
