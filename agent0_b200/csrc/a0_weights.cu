// K8: versioned weight snapshots for actor processes -- a learner publishes the model's state into a device region,
// actors on the same GPU (CUDA IPC) or on a peer GPU (CUDA IPC over NVLink) pull the newest complete snapshot.
// Replaces the reference's state_dict() fetch from the trainer node at the start of every Actor.sample
// (agent0/deepq/launch.py:33-36,56-61) without a host round trip or a collective.
//
// The region is ONE cudaMalloc allocation, so one cudaIpcMemHandle_t covers it:
//   [0, 256)             control block A0WCtl: magic, layout hash, word count, latest, seq[2], the publish ticket
//   [256, 256 + S)       snapshot buffer 0, S = n_words * 4 rounded up to 256 B
//   [256 + S, 256 + 2S)  snapshot buffer 1
// Version v (1, 2, ...) goes into buffer v & 1.  seq[b] = 2v - 1 while version v is being written into b and 2v once
// it is complete; latest = the newest complete version (0: none yet).
//
// Publish (one launch, every CTA one chunk of the flat state):
//   open   thread 0 of every CTA stores seq[b] = 2v - 1 (all CTAs store the same value); bar.sync; every thread
//          executes fence.acq_rel.sys before its first data store.  The seq store is ordered before the barrier,
//          the barrier before each thread's fence, and each fence before that thread's data stores, so no data word of
//          buffer b can be observed (system scope) without seq[b] being odd already -- whichever CTA's seq store is
//          the first, every CTA stores its own before its own data.  (One CTA cannot order the stores of OTHER CTAs
//          behind its seq store, which is why each CTA opens the buffer for itself.)
//   copy   the CTA's words, gathered from the parameter segments, stored with st.relaxed.sys.
//   close  every thread: fence.acq_rel.sys after its stores; bar.sync; thread 0 takes a ticket.  The last CTA's
//          ticket observes every other CTA's fence, so after its own fence every data word of the version is visible
//          at system scope; it then stores seq[b] = 2v (release) and latest = v (release), in that order, so a reader
//          whose acquire load sees latest = v also sees seq[b] = 2v.  Every CTA read latest before its ticket, so no
//          CTA of this launch sees the new value.
//
// Fetch (subscriber side, never waits for the writer):
//   thread 0 of every CTA: v = latest (acquire), b = v & 1, s1 = seq[b] (acquire); the CTA copies its chunk only if
//   s1 == 2v; loads with ld.relaxed.sys into the subscriber's PRIVATE staging buffer; every thread fence.acq_rel.sys
//   after its loads; bar.sync; thread 0 re-reads seq[b].  A data load that saw a word of a later publish into b
//   (version v + 2) synchronises, through that writer's fence and this reader's fence, with the re-read, which then
//   sees seq[b] != s1.  CTAs fold (min v, max v, torn) into subscriber words and the last CTA (ticket) decides:
//   status = v when every CTA saw the same v, nothing was torn, v != 0 and v != the version last applied; else 0.
//   A second launch scatters the staging buffer into the actor's tensors only when status != 0, so a torn or empty
//   fetch leaves them exactly as they were.  With two buffers a fetch of latest can only be torn if two publishes
//   complete while it runs; the caller decides whether to retry.
#include "a0_common.cuh"

namespace {

constexpr uint32_t A0W_MAGIC = 0x57304130u;     // "0A0W"
constexpr uint32_t A0W_FORMAT = 1;
constexpr int A0W_THREADS = 256;
constexpr int A0W_ITERS = 8;                     // 16-byte groups per thread per chunk
constexpr int64_t A0W_CHUNK = (int64_t)A0W_THREADS * A0W_ITERS * 4;   // words per CTA (32 KB)
constexpr int64_t A0W_MAX_WORDS = (int64_t)1 << 34;
constexpr int32_t A0W_MAX_SEGMENTS = 1 << 24;

struct A0WCtl {                  // 256 B at the start of the region
  uint32_t magic;
  uint32_t format;               // A0W_FORMAT
  uint64_t layout_hash;
  uint64_t n_words;
  uint64_t latest;               // newest complete version, 0 = none
  uint64_t seq[2];
  uint32_t ticket;               // publish CTAs arrived (publisher-side; zero between launches)
  uint32_t pad0;
  uint64_t pad[25];
};
static_assert(sizeof(A0WCtl) == 256, "control block is 256 bytes");

struct A0WSub {                  // subscriber-private device words
  uint32_t ticket, torn;
  unsigned long long vmin, vmax;
  unsigned long long status;     // version the last fetch decided to apply, 0 = none
  unsigned long long applied;    // version last applied to the actor's tensors
  unsigned long long pad[27];
};
static_assert(sizeof(A0WSub) == 256, "subscriber words are 256 bytes");

int64_t a0w_buf_bytes(int64_t n_words) { return (n_words * 4 + 255) / 256 * 256; }

// The segment holding flat word i: the largest s in [lo, hi] with pre[s] <= i (pre = word-count prefix sums).
__device__ __forceinline__ int a0w_seg_find(const int64_t* __restrict__ pre, int lo, int hi, int64_t i) {
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(pre + mid) <= i) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// The CTA's range of segments: those that hold a word of [c0, c1).  Empty segments (0 words) are skipped by
// a0w_seg_find because it takes the LAST s with pre[s] <= i.
__device__ __forceinline__ void a0w_chunk_segments(const int64_t* pre, int n_seg, int64_t c0, int64_t c1, int* s_lo,
                                                   int* s_hi) {
  __shared__ int lo_hi[2];
  if (threadIdx.x == 0) {
    lo_hi[0] = a0w_seg_find(pre, 0, n_seg - 1, c0);
    lo_hi[1] = a0w_seg_find(pre, lo_hi[0], n_seg - 1, c1 - 1);
  }
  __syncthreads();
  *s_lo = lo_hi[0];
  *s_hi = lo_hi[1];
}

// Addresses of flat words i .. i+3 in the segments (nullptr past the end of the table).  Segment starts may sit at any
// 4-byte offset, so every word is addressed on its own.
__device__ __forceinline__ void a0w_word_ptrs(const unsigned long long* __restrict__ seg_ptr,
                                              const int64_t* __restrict__ pre, int s_lo, int s_hi, int64_t i,
                                              uint32_t* (&w)[4]) {
  int s = a0w_seg_find(pre, s_lo, s_hi, i);
  int64_t end = __ldg(pre + s + 1);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    while (i + k >= end && s < s_hi) { ++s; end = __ldg(pre + s + 1); }
    w[k] = i + k < end ? reinterpret_cast<uint32_t*>(__ldg(seg_ptr + s)) + (i + k - __ldg(pre + s)) : nullptr;
  }
}

__global__ void __launch_bounds__(A0W_THREADS) a0w_publish_kernel(A0WCtl* ctl, uint32_t* buf0, int64_t buf_words,
                                                                  int64_t n_words,
                                                                  const unsigned long long* __restrict__ seg_ptr,
                                                                  const int64_t* __restrict__ pre, int n_seg) {
  __shared__ uint64_t s_v;
  if (threadIdx.x == 0) {
    const uint64_t v = a0_sys_ld_relaxed(&ctl->latest) + 1;  // the previous publish on this stream has completed
    s_v = v;
    a0_sys_st_relaxed(&ctl->seq[v & 1], 2 * v - 1);          // open
  }
  __syncthreads();
  a0_sys_fence();
  const uint64_t v = s_v;
  uint4* dst = reinterpret_cast<uint4*>(buf0 + (v & 1) * buf_words);
  const int64_t c0 = (int64_t)blockIdx.x * A0W_CHUNK, c1 = min(c0 + A0W_CHUNK, n_words);
  int s_lo, s_hi;
  a0w_chunk_segments(pre, n_seg, c0, c1, &s_lo, &s_hi);
#pragma unroll 2
  for (int it = 0; it < A0W_ITERS; ++it) {
    const int64_t i = c0 + ((int64_t)it * A0W_THREADS + threadIdx.x) * 4;
    if (i >= c1) break;
    uint32_t* w[4];
    a0w_word_ptrs(seg_ptr, pre, s_lo, s_hi, i, w);
    uint4 x;
    x.x = w[0] ? *w[0] : 0u;
    x.y = w[1] ? *w[1] : 0u;
    x.z = w[2] ? *w[2] : 0u;
    x.w = w[3] ? *w[3] : 0u;
    a0_sys_st4_relaxed(dst + (i >> 2), x);
  }
  a0_sys_fence();                                            // close
  __syncthreads();
  if (threadIdx.x == 0) {
    if (atomicAdd(&ctl->ticket, 1u) == gridDim.x - 1) {
      a0_sys_fence();
      a0_sys_st_release(&ctl->seq[v & 1], 2 * v);
      a0_sys_st_release(&ctl->latest, v);
      ctl->ticket = 0u;
    }
  }
}

__global__ void __launch_bounds__(A0W_THREADS) a0w_fetch_kernel(const A0WCtl* ctl, const uint32_t* buf0,
                                                                int64_t buf_words, int64_t n_words, uint32_t* staging,
                                                                A0WSub* sub, unsigned long long* status_out) {
  __shared__ uint64_t s_v, s_seq;
  __shared__ int s_copy;
  if (threadIdx.x == 0) {
    const uint64_t v = a0_sys_ld_acquire(&ctl->latest);
    const uint64_t s1 = v ? a0_sys_ld_acquire(&ctl->seq[v & 1]) : 0;
    s_v = v;
    s_seq = s1;
    s_copy = v != 0 && v != sub->applied && s1 == 2 * v;
  }
  __syncthreads();
  const uint64_t v = s_v;
  if (s_copy) {
    const uint4* src = reinterpret_cast<const uint4*>(buf0 + (v & 1) * buf_words);
    uint4* dst = reinterpret_cast<uint4*>(staging);
    const int64_t g0 = (int64_t)blockIdx.x * (A0W_CHUNK / 4), g1 = min(g0 + A0W_CHUNK / 4, (n_words + 3) / 4);
#pragma unroll 4
    for (int it = 0; it < A0W_ITERS; ++it) {
      const int64_t g = g0 + (int64_t)it * A0W_THREADS + threadIdx.x;
      if (g < g1) dst[g] = a0_sys_ld4_relaxed(src + g);
    }
    a0_sys_fence();                                          // the loads above before the re-read below
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    bool ok = !s_copy || a0_sys_ld_relaxed(&ctl->seq[v & 1]) == s_seq;
    if (v != 0 && v != sub->applied && s_seq != 2 * v) ok = false;   // a version in flight or overtaken at the start
    atomicMin(&sub->vmin, (unsigned long long)v);
    atomicMax(&sub->vmax, (unsigned long long)v);
    if (!ok) atomicOr(&sub->torn, 1u);
    __threadfence();
    if (atomicAdd(&sub->ticket, 1u) == gridDim.x - 1) {
      __threadfence();
      const unsigned long long vmin = atomicAdd(&sub->vmin, 0ull), vmax = atomicAdd(&sub->vmax, 0ull);
      const uint32_t torn = atomicAdd(&sub->torn, 0u);
      const unsigned long long applied = sub->applied;
      const unsigned long long status = (vmin == vmax && !torn && vmin != 0 && vmin != applied) ? vmin : 0ull;
      sub->status = status;
      if (status) sub->applied = status;
      if (status_out) { *reinterpret_cast<volatile unsigned long long*>(status_out) = status; __threadfence_system(); }
      sub->vmin = ~0ull;
      sub->vmax = 0ull;
      sub->torn = 0u;
      sub->ticket = 0u;
    }
  }
}

// The untorn snapshot from the staging buffer into the actor's tensors; nothing when the fetch's status is 0.
__global__ void __launch_bounds__(A0W_THREADS) a0w_apply_kernel(const uint32_t* __restrict__ staging, int64_t n_words,
                                                                const A0WSub* sub,
                                                                const unsigned long long* __restrict__ seg_ptr,
                                                                const int64_t* __restrict__ pre, int n_seg) {
  if (*reinterpret_cast<const volatile unsigned long long*>(&sub->status) == 0ull) return;
  const int64_t c0 = (int64_t)blockIdx.x * A0W_CHUNK, c1 = min(c0 + A0W_CHUNK, n_words);
  int s_lo, s_hi;
  a0w_chunk_segments(pre, n_seg, c0, c1, &s_lo, &s_hi);
  const uint4* src = reinterpret_cast<const uint4*>(staging);
#pragma unroll 2
  for (int it = 0; it < A0W_ITERS; ++it) {
    const int64_t i = c0 + ((int64_t)it * A0W_THREADS + threadIdx.x) * 4;
    if (i >= c1) break;
    uint32_t* w[4];
    a0w_word_ptrs(seg_ptr, pre, s_lo, s_hi, i, w);
    const uint4 x = src[i >> 2];
    if (w[0]) *w[0] = x.x;
    if (w[1]) *w[1] = x.y;
    if (w[2]) *w[2] = x.z;
    if (w[3]) *w[3] = x.w;
  }
}

__global__ void a0w_init_sub(A0WSub* sub) {
  sub->ticket = 0u;
  sub->torn = 0u;
  sub->vmin = ~0ull;
  sub->vmax = 0ull;
  sub->status = 0ull;
  sub->applied = 0ull;
}

unsigned a0w_grid(int64_t n_words) { return (unsigned)((n_words + A0W_CHUNK - 1) / A0W_CHUNK); }

}  // namespace

struct a0_wpub {
  int32_t device;
  int64_t n_words, buf_words;
  uint64_t layout_hash;
  uint8_t* region;               // A0WCtl + 2 buffers
};

struct a0_wsub {
  int32_t device;
  int64_t n_words, buf_words;
  uint8_t* region;               // the publisher's region: IPC mapping or (attach) its own pointer
  bool mapped;                   // region came from a0_ipc_map
  uint32_t* staging;             // [buf_words] private
  A0WSub* sub;
};

extern "C" int a0_wp_create(a0_wpub_t** out, int64_t n_words, uint64_t layout_hash, int32_t device) {
  A0_REQUIRE(out != nullptr, "a0_wp_create: out is NULL");
  A0_REQUIRE(n_words >= 1 && n_words <= A0W_MAX_WORDS, "a0_wp_create: n_words %lld outside [1, 2^34]", (long long)n_words);
  A0_REQUIRE(device >= 0, "a0_wp_create: device %d is negative", device);
  A0DeviceGuard guard(device);
  A0WCtl ctl;
  memset(&ctl, 0, sizeof(ctl));
  ctl.magic = A0W_MAGIC;
  ctl.format = A0W_FORMAT;
  ctl.layout_hash = layout_hash;
  ctl.n_words = (uint64_t)n_words;
  uint8_t* region = nullptr;
  const int rc = a0_ipc_create("a0_wp_create", sizeof(A0WCtl) + 2 * (size_t)a0w_buf_bytes(n_words), &ctl, sizeof(ctl),
                               &region);
  if (rc != A0_OK) return rc;
  *out = new a0_wpub{device, n_words, a0w_buf_bytes(n_words) / 4, layout_hash, region};
  return A0_OK;
}

extern "C" int a0_wp_destroy(a0_wpub_t* wp) {
  if (!wp) return A0_OK;
  A0DeviceGuard guard(wp->device);
  cudaFree(wp->region);
  delete wp;
  return A0_OK;
}

extern "C" int a0_wp_handle(a0_wpub_t* wp, uint8_t* out64) {
  A0_REQUIRE(wp != nullptr && out64 != nullptr, "a0_wp_handle: NULL argument");
  A0DeviceGuard guard(wp->device);
  return a0_ipc_handle(wp->region, out64);
}

extern "C" void* a0_wp_ctl(a0_wpub_t* wp) { return wp ? wp->region : nullptr; }

extern "C" int a0_wp_publish(a0_wpub_t* wp, const uint64_t* seg_ptr, const int64_t* seg_words, int32_t n_seg,
                             a0_stream_t stream) {
  A0_REQUIRE(wp != nullptr, "a0_wp_publish: publisher is NULL");
  A0_REQUIRE(seg_ptr != nullptr && seg_words != nullptr, "a0_wp_publish: segment table is NULL");
  A0_REQUIRE(n_seg >= 1 && n_seg <= A0W_MAX_SEGMENTS, "a0_wp_publish: n_seg %d outside [1, 2^24]", n_seg);
  A0DeviceGuard guard(wp->device);
  a0w_publish_kernel<<<a0w_grid(wp->n_words), A0W_THREADS, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<A0WCtl*>(wp->region), reinterpret_cast<uint32_t*>(wp->region + sizeof(A0WCtl)), wp->buf_words,
      wp->n_words, reinterpret_cast<const unsigned long long*>(seg_ptr), seg_words, n_seg);
  A0_LAUNCH_CHECK();
  return A0_OK;
}

static int a0w_sub_alloc(a0_wsub* ws, const char* who) {
  cudaError_t e = cudaMalloc((void**)&ws->staging, (size_t)ws->buf_words * 4);
  if (e == cudaSuccess) e = cudaMalloc((void**)&ws->sub, sizeof(A0WSub));
  if (e != cudaSuccess) {
    a0_set_error("%s: cudaMalloc failed: %s", who, cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? A0_ENOMEM : (int)e;
  }
  a0w_init_sub<<<1, 1>>>(ws->sub);
  A0_LAUNCH_CHECK();
  A0_CUDA(cudaStreamSynchronize(nullptr));
  return A0_OK;
}

extern "C" int a0_ws_close(a0_wsub_t* ws) {
  if (!ws) return A0_OK;
  A0DeviceGuard guard(ws->device);
  if (ws->mapped) a0_ipc_unmap(ws->region);
  cudaFree(ws->staging);
  cudaFree(ws->sub);
  delete ws;
  return A0_OK;
}

// A subscriber of `region` (mapped: closing it unmaps the region); what is taken is given back on failure.
static int a0w_sub_new(a0_wsub_t** out, const char* who, int32_t device, int64_t n_words, uint8_t* region, bool mapped) {
  a0_wsub* ws = new a0_wsub{device, n_words, a0w_buf_bytes(n_words) / 4, region, mapped, nullptr, nullptr};
  const int rc = a0w_sub_alloc(ws, who);
  if (rc != A0_OK) { a0_ws_close(ws); return rc; }
  *out = ws;
  return A0_OK;
}

extern "C" int a0_ws_open(a0_wsub_t** out, const uint8_t* handle64, uint64_t layout_hash, int64_t n_words,
                          int32_t device) {
  A0_REQUIRE(out != nullptr && handle64 != nullptr, "a0_ws_open: NULL argument");
  A0_REQUIRE(n_words >= 1 && n_words <= A0W_MAX_WORDS, "a0_ws_open: n_words %lld outside [1, 2^34]", (long long)n_words);
  A0_REQUIRE(device >= 0, "a0_ws_open: device %d is negative", device);
  A0DeviceGuard guard(device);
  A0WCtl ctl;
  uint8_t* region = nullptr;
  const int rc = a0_ipc_map("a0_ws_open", handle64, A0W_MAGIC, A0W_FORMAT, "weight publisher's", &ctl, sizeof(ctl), &region);
  if (rc != A0_OK) return rc;
  const char* bad = ctl.layout_hash != layout_hash   ? "has another state layout (names, shapes, dtypes or strides differ)"
                    : ctl.n_words != (uint64_t)n_words ? "holds another number of words"
                                                       : nullptr;
  if (bad) {
    a0_ipc_unmap(region);
    a0_set_error("a0_ws_open: the handle's region %s (hash %016llx vs %016llx, %llu vs %lld words)", bad,
                 (unsigned long long)ctl.layout_hash, (unsigned long long)layout_hash, (unsigned long long)ctl.n_words,
                 (long long)n_words);
    return A0_EINVAL;
  }
  return a0w_sub_new(out, "a0_ws_open", device, n_words, region, true);
}

extern "C" int a0_ws_attach(a0_wsub_t** out, a0_wpub_t* wp) {
  A0_REQUIRE(out != nullptr && wp != nullptr, "a0_ws_attach: NULL argument");
  A0DeviceGuard guard(wp->device);
  return a0w_sub_new(out, "a0_ws_attach", wp->device, wp->n_words, wp->region, false);
}

extern "C" int a0_ws_fetch(a0_wsub_t* ws, const uint64_t* seg_ptr, const int64_t* seg_words, int32_t n_seg,
                           uint64_t* status_out, a0_stream_t stream) {
  A0_REQUIRE(ws != nullptr, "a0_ws_fetch: subscriber is NULL");
  A0_REQUIRE(seg_ptr != nullptr && seg_words != nullptr, "a0_ws_fetch: segment table is NULL");
  A0_REQUIRE(n_seg >= 1 && n_seg <= A0W_MAX_SEGMENTS, "a0_ws_fetch: n_seg %d outside [1, 2^24]", n_seg);
  A0DeviceGuard guard(ws->device);
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned grid = a0w_grid(ws->n_words);
  a0w_fetch_kernel<<<grid, A0W_THREADS, 0, st>>>(
      reinterpret_cast<const A0WCtl*>(ws->region), reinterpret_cast<const uint32_t*>(ws->region + sizeof(A0WCtl)),
      ws->buf_words, ws->n_words, ws->staging, ws->sub, reinterpret_cast<unsigned long long*>(status_out));
  A0_LAUNCH_CHECK();
  a0w_apply_kernel<<<grid, A0W_THREADS, 0, st>>>(ws->staging, ws->n_words, ws->sub,
                                                 reinterpret_cast<const unsigned long long*>(seg_ptr), seg_words, n_seg);
  A0_LAUNCH_CHECK();
  return A0_OK;
}
