// HBM-resident replay shard: frame ring + record ring.  K1 (append) and K3 (fused gather).
//
// Replaces the reference's host deque of lz4 blobs (agent0/deepq/replay.py:18,32-37,45-48) and
// the actor-side n-step tracker (agent0/deepq/agent.py:64-73).  Data layout in HBM:
//   frames    u8 [NF][F]      one 84x84 frame per slot, F = 7056 = 441 * 16 B (16-B aligned slots)
//   rec_slots i32[N][8]       frame slots of the observation stack [0..3] and next stack [4..7]
//   rec_info     [N] 16 B     {f64 reward, i32 action|done<<31, i32 successor link}
// A transition costs 7056 B of frame data (one new frame) + 48 B of record instead of the
// reference's self-contained 56 448 B blob.
#include <stdarg.h>
#include <stdlib.h>

#include <map>
#include <mutex>
#include <utility>

#include "a0_common.cuh"

static thread_local char g_err[512] = "";
void a0_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
extern "C" const char* a0_last_error(void) { return g_err; }

int a0_smem_at_least(const void* kernel, int device, size_t bytes, bool max_carveout) {
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> set;
  std::lock_guard<std::mutex> lock(mu);
  size_t& cur = set[{kernel, device}];
  if (cur >= bytes) return A0_OK;
  A0_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  if (max_carveout) A0_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  cur = bytes;
  return A0_OK;
}
extern "C" int a0_version(void) { return 101; }
#ifdef A0_TRACE
A0_TRACE_SETTER(a0_trace_set_replay)
int a0_trace_set_sumtree(void*, void*);
int a0_trace_set_targets(void*, void*);
extern "C" int a0_trace_set(void* buf, void* cur) {
  a0_trace_set_replay(buf, cur); a0_trace_set_sumtree(buf, cur); a0_trace_set_targets(buf, cur);
  return (int)cudaDeviceSynchronize();
}
#endif

static int g_pdl = -1;     // -1: not decided yet (environment); else a mask of A0_PDL_* classes
bool a0_pdl_enabled(int kernel_class) {
  if (g_pdl < 0) {
    const char* e = getenv("A0_PDL");
    g_pdl = e ? atoi(e) : A0_PDL_DEFAULT;
  }
  return (kernel_class & A0_PDL_FORCE) || (g_pdl & kernel_class) != 0;
}
static int g_k2b_levels = 0;
int a0_option_k2b_levels() {
  if (g_k2b_levels == 0) {
    const char* e = getenv("A0_K2B_LEVELS");
    g_k2b_levels = (e && e[0] == '4') ? 4 : 3;
  }
  return g_k2b_levels;
}
static int g_k2b_bulk_min = 0;
int a0_option_k2b_bulk_min() {
  if (g_k2b_bulk_min == 0) {
    const char* e = getenv("A0_K2B_BULK_MIN");
    g_k2b_bulk_min = e ? atoi(e) : A0_K2B_BULK_MIN_DEFAULT;
    if (g_k2b_bulk_min < 1) g_k2b_bulk_min = 1;
  }
  return g_k2b_bulk_min;
}
static int g_k3_l2 = -1;
// Measured (B200, profiles/): with 640 transitions per launch (68 MB, half the L2) evict_first on both
// directions shortens the batch-32 step by 6 % -- K4's inputs, the tree and the records stay in L2 -- and
// the gather itself by 4 %; at 10 240 transitions (1.1 GB per launch) nothing else survives in L2 either
// way and the hints cost 0.4 %.  "Auto" applies them while the launch moves less than the L2 holds.
static int a0_option_k3_l2(int64_t launch_bytes) {
  if (g_k3_l2 < 0) {
    const char* e = getenv("A0_K3_L2");
    g_k3_l2 = e ? atoi(e) : A0_K3_L2_DEFAULT;
    if (g_k3_l2 < 0 || g_k3_l2 > 4) g_k3_l2 = A0_K3_L2_DEFAULT;
  }
  if (g_k3_l2 == 4) return launch_bytes <= (int64_t)100 << 20 ? 3 : 0;
  return g_k3_l2;
}
static int64_t g_mail_timeout_us = -1;
uint64_t a0_option_mail_timeout_ns() {
  if (g_mail_timeout_us < 0) {
    const char* e = getenv("A0_MAIL_TIMEOUT_US");
    g_mail_timeout_us = e ? atoll(e) : 2000000;
    if (g_mail_timeout_us < 1) g_mail_timeout_us = 1;
  }
  return (uint64_t)g_mail_timeout_us * 1000ull;
}
int a0_check_fault(a0_replay* h, const char* who) {
  if (h && h->fault_host && *(volatile int32_t*)h->fault_host != 0) {
    const int32_t code = *(volatile int32_t*)h->fault_host;
    *(volatile int32_t*)h->fault_host = 0;
    a0_set_error("%s: an earlier launch on this shard reported device fault %d (%s)", who, code,
                 code == 1 ? "a gather CTA of a0_rb_sample_gather timed out waiting for its sampler: its outputs are invalid"
                 : code == 2 ? "a0_pt_sample_unique found fewer than B records with positive priority: the batch's last rows repeat its first record"
                             : "unknown");
    return A0_EFAULT;
  }
  return A0_OK;
}
extern "C" int a0_rb_check_fault(a0_replay_t* h) {
  A0_REQUIRE(h != nullptr, "a0_rb_check_fault: handle is NULL");
  return a0_check_fault(h, "a0_rb_check_fault");
}
static int g_fused_ingest = -1;
bool a0_option_fused_ingest() {
  if (g_fused_ingest < 0) {
    const char* e = getenv("A0_FUSED_INGEST");
    g_fused_ingest = e ? (atoi(e) != 0) : 1;
  }
  return g_fused_ingest != 0;
}
extern "C" int a0_get_option(int32_t option, int64_t* value) {
  A0_REQUIRE(value != nullptr, "a0_get_option: value is NULL");
  if (option == A0_OPT_PDL) { a0_pdl_enabled(0); *value = g_pdl; return A0_OK; }      // resolves the environment default first
  a0_set_error("a0_get_option: option %d cannot be read back", option);
  return A0_EINVAL;
}

extern "C" int a0_set_option(int32_t option, int64_t value) {
  if (option == A0_OPT_FUSED_INGEST) { g_fused_ingest = value != 0; return A0_OK; }
  if (option == A0_OPT_MAIL_TIMEOUT_US) {
    A0_REQUIRE(value >= 1, "a0_set_option: A0_OPT_MAIL_TIMEOUT_US must be positive");
    g_mail_timeout_us = value;
    return A0_OK;
  }
  if (option == A0_OPT_C51_FAST) { a0_set_c51_fast(value != 0); return A0_OK; }
  if (option == A0_OPT_K2B_SMALL) { a0_set_k2b_small(value != 0); return A0_OK; }
  if (option == A0_OPT_K2B_CHUNKS) { a0_set_k2b_chunks(value != 0); return A0_OK; }
  if (option == A0_OPT_K2A_ROUNDS) { a0_set_k2a_rounds(value != 0); return A0_OK; }
  if (option == A0_OPT_K2B_SPARSE) {
    A0_REQUIRE(value >= 0 && value <= 32, "a0_set_option: A0_OPT_K2B_SPARSE must be 0..32");
    a0_set_k2b_sparse((int)value);
    return A0_OK;
  }
  if (option == A0_OPT_K6_GLOBAL) { a0_set_k6_global(value != 0); return A0_OK; }
  if (option == A0_OPT_QH_SPEC) { a0_set_qh_spec(value != 0); return A0_OK; }
  if (option == A0_OPT_QH_SORTED) {
    A0_REQUIRE(value >= 0 && value <= 2, "a0_set_option: A0_OPT_QH_SORTED must be 0, 1 or 2");
    a0_set_qh_sorted((int)value);
    return A0_OK;
  }
  if (option == A0_OPT_K3_L2) {
    A0_REQUIRE(value >= 0 && value <= 4, "a0_set_option: A0_OPT_K3_L2 must be 0..4");
    g_k3_l2 = (int)value;
    return A0_OK;
  }
  if (option == A0_OPT_PDL) { g_pdl = (int)value & 15; return A0_OK; }
  if (option == A0_OPT_K2B_LEVELS) {
    A0_REQUIRE(value == 3 || value == 4, "a0_set_option: A0_OPT_K2B_LEVELS must be 3 or 4");
    g_k2b_levels = (int)value;
    return A0_OK;
  }
  if (option == A0_OPT_K2B_BULK_MIN) {
    A0_REQUIRE(value >= 1, "a0_set_option: A0_OPT_K2B_BULK_MIN must be positive");
    g_k2b_bulk_min = (int)(value > (1 << 30) ? (1 << 30) : value);
    return A0_OK;
  }
  a0_set_error("a0_set_option: unknown option %d", option);
  return A0_EINVAL;
}

// ------------------------------------------------------------------------------------------------
// typed joins of a captured step (hotloop.ReplayTargetLoop)
// ------------------------------------------------------------------------------------------------
// A kernel launched with the programmatic attribute after a cross-stream event wait gets programmatic edges from
// every predecessor, so it may start before the other stream's work is complete.  Instead the joining kernel is
// launched with its stream predecessor alone, and the edge from the other stream's node is added to the graph
// afterwards as a full edge: its type is then the one set here, whatever the launch attribute does to the others.
static int a0_capture_tail(cudaStream_t stream, cudaGraph_t* graph, cudaGraphNode_t* node) {
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  const cudaGraphNode_t* deps = nullptr;
  size_t n = 0;
  A0_CUDA(cudaStreamGetCaptureInfo_v3(stream, &st, nullptr, graph, &deps, nullptr, &n));
  A0_REQUIRE(st == cudaStreamCaptureStatusActive && n == 1,
             "the stream is not capturing (status %d) or its last captured work is not one node (%zu)", (int)st, n);
  *node = deps[0];
  return A0_OK;
}

extern "C" int a0_capture_node(a0_stream_t stream, void** node) {
  A0_REQUIRE(node != nullptr, "a0_capture_node: node is NULL");
  cudaGraphNode_t n;
  int rc = a0_capture_tail((cudaStream_t)stream, nullptr, &n);
  if (rc) return rc;
  *node = n;
  return A0_OK;
}

extern "C" int a0_capture_join(a0_stream_t stream, void* from) {
  A0_REQUIRE(from != nullptr, "a0_capture_join: from is NULL");
  cudaGraph_t g;
  cudaGraphNode_t to, f = (cudaGraphNode_t)from;
  int rc = a0_capture_tail((cudaStream_t)stream, &g, &to);
  if (rc) return rc;
  cudaGraphEdgeData full = {};      // cudaGraphDependencyTypeDefault from cudaGraphKernelNodePortDefault: on completion
  A0_CUDA(cudaGraphAddDependencies_v2(g, &f, &to, &full, 1));
  return A0_OK;
}

extern "C" int a0_graph_edges(void* graph, void** from, void** to, int32_t* type, int32_t* from_port, int64_t capacity,
                              int64_t* count) {
  A0_REQUIRE(graph != nullptr && count != nullptr && capacity >= 0, "a0_graph_edges: bad graph, count or capacity");
  size_t n = 0;
  A0_CUDA(cudaGraphGetEdges_v2((cudaGraph_t)graph, nullptr, nullptr, nullptr, &n));
  *count = (int64_t)n;
  if (n == 0 || capacity == 0) return A0_OK;
  A0_REQUIRE((int64_t)n <= capacity && from && to && type && from_port, "a0_graph_edges: %zu edges, room for %lld", n,
             (long long)capacity);
  std::vector<cudaGraphNode_t> f(n), t(n);
  std::vector<cudaGraphEdgeData> d(n);
  A0_CUDA(cudaGraphGetEdges_v2((cudaGraph_t)graph, f.data(), t.data(), d.data(), &n));
  for (size_t i = 0; i < n; ++i) {
    from[i] = f[i]; to[i] = t[i]; type[i] = d[i].type; from_port[i] = d[i].from_port;
  }
  return A0_OK;
}

// ------------------------------------------------------------------------------------------------
// lifetime
// ------------------------------------------------------------------------------------------------
__global__ void a0_fill_i32(int32_t* p, int64_t n, int32_t v) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = v;
}
__global__ void a0_init_scalars(float* max_p) {
  *max_p = 1.0f;
  for (int i = 1; i < 16; ++i) max_p[i] = 0.0f;              // padding up to the dyn words: defined, so shard states compare
  max_p[16] = 0.0f; max_p[17] = 1.0f; max_p[18] = 0.0f;     // dyn = {top, beta, sum_offset}
}

extern "C" int a0_rb_create(a0_replay_t** out, int64_t rec_capacity, int64_t frame_capacity,
                            int32_t frame_bytes, int32_t device) {
  A0_REQUIRE(out != nullptr, "a0_rb_create: out is NULL");
  // 2^24: record positions survive the reference's .float() round trip of indices (trainer.py:88-90)
  A0_REQUIRE(rec_capacity >= 2 && rec_capacity <= (1LL << 24), "a0_rb_create: rec_capacity %lld outside [2, 2^24]",
             (long long)rec_capacity);
  A0_REQUIRE(frame_capacity >= 8 && frame_capacity <= (1LL << 30), "a0_rb_create: frame_capacity %lld out of range",
             (long long)frame_capacity);
  A0_REQUIRE(frame_bytes > 0 && frame_bytes % 16 == 0, "a0_rb_create: frame_bytes %d must be a positive multiple of 16",
             frame_bytes);
  A0_REQUIRE((int64_t)frame_bytes * A0_SLOTS <= 200 * 1024,
             "a0_rb_create: frame_bytes %d is above 25 600 (the gather and the LZ4 kernels stage 8 frames in 200 KB of shared memory)",
             frame_bytes);
  A0DeviceGuard guard(device);
  a0_replay* h = new a0_replay();
  memset(h, 0, sizeof(*h));
  h->device = device;
  h->N = rec_capacity;
  h->NF = frame_capacity;
  h->F = frame_bytes;
  h->D = 1;
  while ((1LL << h->D) < rec_capacity) h->D++;
  h->P = 1LL << h->D;
  cudaError_t e = cudaSuccess;
  auto alloc = [&](void** p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); };
  alloc((void**)&h->frames, (size_t)h->NF * h->F);
  alloc((void**)&h->rec_slots, (size_t)h->N * A0_SLOTS * sizeof(int32_t));
  alloc((void**)&h->rec_info, (size_t)h->N * sizeof(A0RecInfo));
  alloc((void**)&h->tree, (size_t)2 * h->P * sizeof(float));
  alloc((void**)&h->max_p, 256);
  h->dyn = nullptr;
  alloc((void**)&h->winner, (size_t)h->N * sizeof(int32_t));
  alloc((void**)&h->dirty, (size_t)((h->P >> 12) + 1) * sizeof(int32_t));
  alloc((void**)&h->counter, (size_t)(2 * A0_MAX_BATCHES + 64) * sizeof(unsigned int));
  if (e != cudaSuccess) {
    a0_set_error("a0_rb_create: cudaMalloc failed: %s", cudaGetErrorString(e));
    a0_rb_destroy(h);
    return e == cudaErrorMemoryAllocation ? A0_ENOMEM : (int)e;
  }
  h->dyn = h->max_p + 16;     // same 256-byte allocation
  if (cudaHostAlloc((void**)&h->fault_host, 64, cudaHostAllocMapped) != cudaSuccess ||
      cudaHostGetDevicePointer((void**)&h->fault_dev, h->fault_host, 0) != cudaSuccess) {
    a0_set_error("a0_rb_create: cannot allocate the mapped fault word: %s", cudaGetErrorString(cudaGetLastError()));
    a0_rb_destroy(h);
    return A0_ENOMEM;
  }
  memset(h->fault_host, 0, 64);
  int rc = a0_rb_reset(h, nullptr);
  if (rc != 0) { a0_rb_destroy(h); return rc; }
  A0_CUDA(cudaStreamSynchronize(nullptr));
  *out = h;
  return A0_OK;
}

extern "C" int a0_rb_destroy(a0_replay_t* h) {
  if (!h) return A0_OK;
  A0DeviceGuard guard(h->device);
  cudaFree(h->frames); cudaFree(h->rec_slots); cudaFree(h->rec_info); cudaFree(h->tree);
  cudaFree(h->max_p); cudaFree(h->winner); cudaFree(h->dirty); cudaFree(h->counter); cudaFree(h->mail);
  if (h->fault_host) cudaFreeHost(h->fault_host);
  for (int t = 0; t < 2; ++t) {
    if (h->staging[t].event) { cudaEventSynchronize(h->staging[t].event); cudaEventDestroy(h->staging[t].event); }
    if (h->staging[t].copied) cudaEventDestroy(h->staging[t].copied);
    if (h->staging[t].host) cudaFreeHost(h->staging[t].host);
    if (h->staging[t].dev) cudaFree(h->staging[t].dev);
  }
  if (h->copy_stream) { cudaStreamSynchronize(h->copy_stream); cudaStreamDestroy(h->copy_stream); }
  delete h;
  return A0_OK;
}

extern "C" int a0_rb_reset(a0_replay_t* h, a0_stream_t stream_) {
  A0_REQUIRE(h != nullptr, "a0_rb_reset: handle is NULL");
  cudaStream_t stream = (cudaStream_t)stream_;
  A0DeviceGuard guard(h->device);
  A0_CUDA(cudaMemsetAsync(h->tree, 0, (size_t)2 * h->P * sizeof(float), stream));
  A0_CUDA(cudaMemsetAsync(h->rec_slots, 0, (size_t)h->N * A0_SLOTS * sizeof(int32_t), stream));
  A0_CUDA(cudaMemsetAsync(h->rec_info, 0xff, (size_t)h->N * sizeof(A0RecInfo), stream));
  a0_fill_i32<<<256, 256, 0, stream>>>(h->winner, h->N, -1);
  A0_LAUNCH_CHECK();
  A0_CUDA(cudaMemsetAsync(h->dirty, 0, (size_t)((h->P >> 12) + 1) * sizeof(int32_t), stream));
  A0_CUDA(cudaMemsetAsync(h->counter, 0, (size_t)(2 * A0_MAX_BATCHES + 64) * sizeof(unsigned int), stream));
  a0_init_scalars<<<1, 1, 0, stream>>>(h->max_p);
  A0_LAUNCH_CHECK();
  return A0_OK;
}

extern "C" void* a0_rb_ptr(a0_replay_t* h, int32_t which) {
  if (!h) return nullptr;
  switch (which) {
    case A0_PTR_FRAMES: return h->frames;
    case A0_PTR_REC_SLOTS: return h->rec_slots;
    case A0_PTR_REC_INFO: return h->rec_info;
    case A0_PTR_TREE: return h->tree;
    case A0_PTR_MAX_P: return h->max_p;
    default: return nullptr;
  }
}
extern "C" int64_t a0_rb_tree_leaves(a0_replay_t* h) { return h ? h->P : 0; }

// ------------------------------------------------------------------------------------------------
// K1: append.  Blocks [0, n_new) copy one staged frame each into its ring slot with 16-byte
// vector loads/stores (a 7056-B frame is 441 uint4, fully coalesced); the remaining blocks scatter
// record metadata, one thread per record.  HBM-bound: F read (staging) + F write per new frame.
// ------------------------------------------------------------------------------------------------
constexpr int K1_THREADS = 128;

__global__ void __launch_bounds__(K1_THREADS)
a0_k1_append(uint8_t* __restrict__ frames, int32_t F, int64_t NF, const uint8_t* __restrict__ staged,
             const int32_t* __restrict__ new_pos, const int32_t* __restrict__ src_idx, int32_t n_new,
             int32_t* __restrict__ rec_slots, A0RecInfo* __restrict__ rec_info, int64_t N, const int32_t* __restrict__ meta,
             int32_t m, const A0Dyn dyn) {
  A0_PDL_PROLOGUE();
  if (dyn.dyn && blockIdx.x == 0 && threadIdx.x == 0) {   // what a0_rb_set_dynamic would launch a kernel for
    dyn.dyn[0] = dyn.top; dyn.dyn[1] = dyn.beta; dyn.dyn[2] = dyn.sum_offset;
  }
  if ((int)blockIdx.x < n_new) {
    a0_k1_copy_frame(frames, F, NF, staged, new_pos, src_idx, blockIdx.x, threadIdx.x, K1_THREADS);
    return;
  }
  const int r = ((int)blockIdx.x - n_new) * K1_THREADS + threadIdx.x;
  if (r < m) a0_k1_write_record(rec_slots, rec_info, N, meta, r);
}

int a0_append_launch(a0_replay* h, const uint8_t* new_frames, const int32_t* new_frame_pos, const int32_t* src_idx,
                     int32_t n_new, const int32_t* rec_meta, int32_t m, const A0Dyn& dyn, cudaStream_t stream) {
  int blocks = n_new + (m + K1_THREADS - 1) / K1_THREADS;
  if (blocks == 0) {
    if (!dyn.dyn) return A0_OK;
    blocks = 1;                                   // nothing to append: the launch only publishes the scalars
  }
  A0_LAUNCH(a0_k1_append, (unsigned)blocks, K1_THREADS, 0, stream, 1, A0_PDL_K1, h->frames, h->F, h->NF, new_frames,
            new_frame_pos, src_idx, n_new, h->rec_slots, h->rec_info, h->N, rec_meta, m, dyn);
  return A0_OK;
}

extern "C" int a0_rb_append(a0_replay_t* h, const uint8_t* new_frames, const int32_t* new_frame_pos,
                            int32_t n_new, const int32_t* rec_meta, int32_t m, a0_stream_t stream_) {
  A0_REQUIRE(h != nullptr, "a0_rb_append: handle is NULL");
  A0_REQUIRE(n_new >= 0 && m >= 0, "a0_rb_append: negative count");
  if (n_new == 0 && m == 0) return A0_OK;
  A0_REQUIRE(n_new == 0 || (new_frames && new_frame_pos), "a0_rb_append: NULL frame arguments");
  A0_REQUIRE(m == 0 || rec_meta, "a0_rb_append: NULL rec_meta");
  A0_REQUIRE(((uintptr_t)new_frames & 15) == 0, "a0_rb_append: new_frames must be 16-byte aligned");
  A0DeviceGuard guard(h->device);
  const A0Dyn none = {nullptr, 0.0f, 0.0f, 0.0f};
  return a0_append_launch(h, new_frames, new_frame_pos, nullptr, n_new, rec_meta, m, none, (cudaStream_t)stream_);
}

// ------------------------------------------------------------------------------------------------
// K3: fused gather
// ------------------------------------------------------------------------------------------------
struct A0GatherArgs {
  const uint8_t* frames;
  const int32_t* rec_slots;
  const A0RecInfo* rec_info;
  const int64_t* idx;
  int64_t N, NF;
  int32_t F, count, n_step;
  int32_t stride_hint;   // expected distance between a record and its successor in the same stream (0: unknown)
  double gamma;
  uint8_t* frames_out;
  int64_t* action_out;
  double* reward64_out;
  float* reward32_out;
  uint8_t* done8_out;
  float* done32_out;
  int64_t* boot_out;
  long long* mail;       // != NULL: record positions arrive through the sampler's mailbox (a0_rb_sample_gather)
  int32_t* fault;        // mapped host word: set to 1 by a CTA whose mailbox word never arrived
  unsigned long long mail_timeout_ns;
  int32_t l2_hints;      // bit 0: frame reads evict_first, bit 1: output stores evict_first (A0_OPT_K3_L2)
  // ordered fetch (a0_rb_gather_mail with a window): draw gbase + blockIdx.x starts its frame traffic only when at most
  // `window` draws beyond the completed ones are in flight, so the FIRST batches of a draw complete first instead of all
  // resident CTAs sharing the bandwidth and finishing together.  progress counts completed draws of the whole sampler
  // call (gtotal); the last one re-arms it.
  unsigned int* progress;
  int32_t window, gbase, gtotal;
};

// Walks the n-step window that starts at record p0 (whose info word is already loaded), writes
// the scalar outputs of sample b and returns the last record of the window.  The return is
// evaluated as the reference does (agent.py:65-69): r = 0; for newest..oldest:
// r = r*gamma*(1-d) + r_t, every product and sum rounded separately in float64 (no FMA contraction).
__device__ __forceinline__ int64_t a0_walk_window(const A0GatherArgs& g, int b, int64_t p0, A0RecInfo info,
                                                  bool& ok) {
  double rew[A0_MAX_NSTEP];
  int dn[A0_MAX_NSTEP];
  int64_t p = p0;
  const int32_t action = info.action_done & 0x7fffffff;
  int32_t link = -1;
  int steps = 0;
#pragma unroll 1
  for (int i = 0; i < g.n_step; ++i) {
    if (i > 0) info = g.rec_info[p];
    rew[i] = info.reward;
    dn[i] = (info.action_done >> 31) & 1;
    link = info.link;
    steps = i + 1;
    if (i + 1 < g.n_step) {
      if (link < 0 || link >= g.N) { ok = false; break; }   // window not complete: caller error
      p = link;
    }
  }
  double r = 0.0;
  int d_any = 0;
#pragma unroll 1
  for (int i = steps - 1; i >= 0; --i) {
    d_any |= dn[i];
    r = __dadd_rn(__dmul_rn(__dmul_rn(r, g.gamma), (double)(1 - dn[i])), rew[i]);
  }
  if (g.action_out) g.action_out[b] = ok ? (int64_t)action : -1;
  if (g.reward64_out) g.reward64_out[b] = r;
  if (g.reward32_out) g.reward32_out[b] = (float)r;          // .float() in Trainer.step (trainer.py:88-90)
  if (g.done8_out) g.done8_out[b] = (uint8_t)d_any;
  if (g.done32_out) g.done32_out[b] = (float)d_any;
  if (g.boot_out) g.boot_out[b] = ok ? (int64_t)link : -1;
  return p;
}

// The same walk with the dependent chain speculated away.  Vector actors append one record per
// stream per step, so the successor of record p is almost always (p + stride) mod N, stride = the
// number of streams (the ingest path measures it: a0_replay::stride_hint).  The records and the
// next-stack slots of the guessed window are fetched together with the first record -- ONE
// memory round trip instead of n_step + 1 dependent ones -- and used only where the stored link
// confirms the guess; anything else falls back to the dependent load.  Results are identical.
constexpr int K3_SPEC_MAX = 4;         // speculate windows of up to this many records
struct A0Spec {
  int64_t pos[K3_SPEC_MAX];            // guessed record positions (pos[0] = p0)
  A0RecInfo info[K3_SPEC_MAX];
  int4 next_slots;                     // rec_slots[pos[n-1]][4..7]
  bool on;
};
__device__ __forceinline__ void a0_spec_fetch(const A0GatherArgs& g, int64_t p0, A0Spec& sp) {
  sp.on = g.n_step <= K3_SPEC_MAX && (g.n_step == 1 || g.stride_hint > 0);
  if (!sp.on) return;
  int64_t p = p0;
#pragma unroll
  for (int i = 0; i < K3_SPEC_MAX; ++i) {
    sp.pos[i] = p;
    if (i > 0 && i < g.n_step) sp.info[i] = g.rec_info[p];
    if (i == g.n_step - 1) sp.next_slots = reinterpret_cast<const int4*>(g.rec_slots + (size_t)p * A0_SLOTS)[1];
    p += g.stride_hint;
    if (p >= g.N) p -= g.N;
  }
}
__device__ __forceinline__ int64_t a0_walk_window_spec(const A0GatherArgs& g, int b, int64_t p0, A0RecInfo info,
                                                       const A0Spec& sp, bool& ok, int4& next_slots) {
  if (!sp.on) {
    const int64_t pl = a0_walk_window(g, b, p0, info, ok);
    next_slots = reinterpret_cast<const int4*>(g.rec_slots + (size_t)pl * A0_SLOTS)[1];
    return pl;
  }
  double rew[K3_SPEC_MAX];
  int dn[K3_SPEC_MAX];
  int64_t p = p0;
  const int32_t action = info.action_done & 0x7fffffff;
  int32_t link = -1;
  int steps = 0;
  bool guessed = true;                 // every record so far sits where the guess put it
#pragma unroll
  for (int i = 0; i < K3_SPEC_MAX; ++i) {
    if (i < g.n_step && steps == i) {
      if (i > 0) info = guessed ? sp.info[i] : g.rec_info[p];
      rew[i] = info.reward;
      dn[i] = (info.action_done >> 31) & 1;
      link = info.link;
      steps = i + 1;
      if (i + 1 < g.n_step) {
        if (link < 0 || link >= g.N) { ok = false; steps = -steps; }     // window not complete: stop here
        else {
          p = link;
          guessed = guessed && (i + 1 < K3_SPEC_MAX) && p == sp.pos[i + 1 < K3_SPEC_MAX ? i + 1 : 0];
        }
      }
    }
  }
  if (steps < 0) steps = -steps;
  double r = 0.0;
  int d_any = 0;
#pragma unroll
  for (int i = K3_SPEC_MAX - 1; i >= 0; --i) {
    if (i < steps) {
      d_any |= dn[i];
      r = __dadd_rn(__dmul_rn(__dmul_rn(r, g.gamma), (double)(1 - dn[i])), rew[i]);
    }
  }
  if (g.action_out) g.action_out[b] = ok ? (int64_t)action : -1;
  if (g.reward64_out) g.reward64_out[b] = r;
  if (g.reward32_out) g.reward32_out[b] = (float)r;          // .float() in Trainer.step (trainer.py:88-90)
  if (g.done8_out) g.done8_out[b] = (uint8_t)d_any;
  if (g.done32_out) g.done32_out[b] = (float)d_any;
  if (g.boot_out) g.boot_out[b] = ok ? (int64_t)link : -1;
  next_slots = (guessed && ok) ? sp.next_slots : reinterpret_cast<const int4*>(g.rec_slots + (size_t)p * A0_SLOTS)[1];
  return p;
}

// The 8 frame slots of sample b: observation stack of the first record, next stack of the last.
__device__ __forceinline__ bool a0_resolve_window(const A0GatherArgs& g, int b, int32_t (&slot)[A0_SLOTS]) {
  int64_t p0 = g.idx[b];
  bool ok = p0 >= 0 && p0 < g.N;
  if (!ok) p0 = 0;
  const int4 a = *reinterpret_cast<const int4*>(g.rec_slots + (size_t)p0 * A0_SLOTS);
  const int64_t p = a0_walk_window(g, b, p0, g.rec_info[p0], ok);
  const int4 c = reinterpret_cast<const int4*>(g.rec_slots + (size_t)p * A0_SLOTS)[1];
  slot[0] = a.x; slot[1] = a.y; slot[2] = a.z; slot[3] = a.w;
  slot[4] = c.x; slot[5] = c.y; slot[6] = c.z; slot[7] = c.w;
#pragma unroll
  for (int j = 0; j < A0_SLOTS; ++j)
    if (slot[j] < 0 || slot[j] >= g.NF) { slot[j] = 0; ok = false; }
  return ok;
}

// Distinct frames of the two stacks: uslot[u] = frame slot, dmask[u] = stack positions it fills.
// a0_unique_add registers stack position j (fully unrolled: the arrays stay in registers).
__device__ __forceinline__ void a0_unique_add(int32_t s, int j, int32_t (&uslot)[A0_SLOTS], uint32_t (&dmask)[A0_SLOTS],
                                              int& U) {
  bool found = false;
#pragma unroll
  for (int u = 0; u < A0_SLOTS; ++u)
    if (u < U && !found && uslot[u] == s) { dmask[u] |= 1u << j; found = true; }
  if (!found) {
#pragma unroll
    for (int u = 0; u < A0_SLOTS; ++u)
      if (u == U) { uslot[u] = s; dmask[u] = 1u << j; }
    ++U;
  }
}
__device__ __forceinline__ int a0_unique_frames(const int32_t (&slot)[A0_SLOTS], int32_t (&uslot)[A0_SLOTS],
                                                uint32_t (&dmask)[A0_SLOTS]) {
  int U = 0;
#pragma unroll
  for (int j = 0; j < A0_SLOTS; ++j) a0_unique_add(slot[j], j, uslot, dmask, U);
  return U;
}

// Variant 0 (default): one warp per sampled transition; lane 0 drives the TMA engine through a ring
// of K3_RING frame buffers.  Every *distinct* frame of the two stacks is fetched once with
// cp.async.bulk (global -> shared, completion on that buffer's mbarrier) and written with
// cp.async.bulk (shared -> global) to every stack position it occupies: (S+n)*F bytes read and
// 2S*F bytes written per transition, no register staging.  A buffer is refilled as soon as its
// stores have read it, so 28 KB of shared memory per CTA is enough and 7 CTAs fit on an SM: a
// 640-transition launch (20 batches of 32) is a single wave.  The loads of the observation stack
// are issued as soon as the first record is known, so the dependent walk along the n-step links
// (two more HBM round trips at n = 3) overlaps the first 28 KB of frame traffic.
constexpr int K3_RING = 4;
// (A ring of 8 -- every distinct frame of a transition in flight at once, 56 KB, 4 CTAs per SM -- was measured for the
// ordered waves of a small draw, where a CTA's own latency is what the first K4 waits for: no difference, 68.17 us per
// batch-32 step either way; the latency is the record fetch, the first loads and the store drain, not the refills.)
template <int RING>
__device__ __forceinline__ void a0_k3_gather_body(const A0GatherArgs& g) {
  extern __shared__ __align__(128) uint8_t a0_smem[];
  __shared__ __align__(8) uint64_t bars[RING];
  if (threadIdx.x != 0) return;
  A0_T0();
  const int b = blockIdx.x;
  const uint32_t F = (uint32_t)g.F;
  const uint32_t bar0 = a0_smem_u32(&bars[0]);
  const uint32_t buf0 = a0_smem_u32(a0_smem);
  int64_t p0;
  if (g.mail) {
    // Launched (programmatically) while the sampler is still running: everything older than the
    // sampler is complete -- it executed griddepcontrol.wait before it let this grid launch -- so
    // the shard may be read; the record position comes through the mailbox as soon as the draw's
    // warp has finished its descent.  The wait at the END of this kernel makes its completion
    // imply the sampler's (weights, priorities), which is what the successors rely on.
    asm volatile("griddepcontrol.launch_dependents;");
#pragma unroll
    for (int r = 0; r < RING; ++r) a0_mbar_init(bar0 + 8 * r, 1);
    a0_fence_barrier_init();
    // The poll is bounded: the paired sampler posts the word within microseconds; without it (a failed
    // launch, a mis-paired caller) the CTA gives up after mail_timeout_ns, raises the handle's fault word
    // (mapped host memory: the next host call reports it) and produces an invalid sample instead of hanging.
    long long v;
    unsigned long long t_start = 0;
    unsigned spins = 0;
    for (;;) {
      asm volatile("ld.relaxed.gpu.global.s64 %0, [%1];" : "=l"(v) : "l"(g.mail + b) : "memory");
      if (v != 0) break;
      if ((++spins & 255u) == 0) {
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (t_start == 0) t_start = now;
        else if (now - t_start > g.mail_timeout_ns) break;
      }
    }
    if (v != 0) {
      asm volatile("st.relaxed.gpu.global.s64 [%0], %1;" ::"l"(g.mail + b), "l"(0ll) : "memory");
      p0 = v - 1;
    } else {
      if (g.fault) { *reinterpret_cast<volatile int32_t*>(g.fault) = 1; __threadfence_system(); }
      p0 = -1;
    }
  } else {
    A0_PDL_PROLOGUE();
    p0 = g.idx[b];
  }
  A0_TMID();
  bool ok = p0 >= 0 && p0 < g.N;
  if (!ok) p0 = 0;
  const int4 sa = *reinterpret_cast<const int4*>(g.rec_slots + (size_t)p0 * A0_SLOTS);
  const A0RecInfo info0 = g.rec_info[p0];
  A0Spec sp;
  a0_spec_fetch(g, p0, sp);              // the guessed rest of the window, same round trip as the first record
  if (g.progress && g.window > 0) {
    // the record loads above are in flight; the frame traffic waits for this draw's turn.  Bounded like the mailbox
    // poll: giving up only costs the ordering, not the result.
    const int need = g.gbase + b - g.window + 1;
    if (need > 0) {
      unsigned long long t_start = 0;
      unsigned spins = 0;
      for (;;) {
        unsigned int done;
        asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(done) : "l"(g.progress) : "memory");
        if ((int)done >= need) break;
        __nanosleep(32);
        if ((++spins & 255u) == 0) {
          unsigned long long now;
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
          if (t_start == 0) t_start = now;
          else if (now - t_start > g.mail_timeout_ns) break;
        }
      }
    }
  }
  const uint64_t pol = a0_policy_evict_first();
  const bool hint_ld = g.l2_hints & 1, hint_st = g.l2_hints & 2;
  auto load = [&](uint32_t dst, const void* src, uint32_t bar) {
    if (hint_ld) a0_bulk_load_hint(dst, src, F, bar, pol);
    else a0_bulk_load(dst, src, F, bar);
  };
  auto store = [&](void* dst, uint32_t src) {
    if (hint_st) a0_bulk_store_hint(dst, src, F, pol);
    else a0_bulk_store(dst, src, F);
  };
  if (!g.mail) {
#pragma unroll
    for (int r = 0; r < RING; ++r) a0_mbar_init(bar0 + 8 * r, 1);
    a0_fence_barrier_init();
  }
  int32_t uslot[A0_SLOTS];
  uint32_t dmask[A0_SLOTS];
  int U = 0;
  {
    int32_t s4[A0_STACK] = {sa.x, sa.y, sa.z, sa.w};
#pragma unroll
    for (int j = 0; j < A0_STACK; ++j) {
      if (s4[j] < 0 || s4[j] >= g.NF) { s4[j] = 0; ok = false; }
      a0_unique_add(s4[j], j, uslot, dmask, U);
    }
  }
  const int U0 = U;                      // <= A0_STACK <= RING
#pragma unroll
  for (int u = 0; u < RING; ++u)
    if (u < U0) load(buf0 + u * F, g.frames + (size_t)uslot[u] * F, bar0 + 8 * u);
  // the n-step walk and the next stack, while those loads are in flight
  int4 sc;
  a0_walk_window_spec(g, b, p0, info0, sp, ok, sc);
  {
    int32_t s4[A0_STACK] = {sc.x, sc.y, sc.z, sc.w};
#pragma unroll
    for (int j = 0; j < A0_STACK; ++j) {
      if (s4[j] < 0 || s4[j] >= g.NF) { s4[j] = 0; ok = false; }
      a0_unique_add(s4[j], A0_STACK + j, uslot, dmask, U);
    }
  }
  if (!ok && g.action_out) g.action_out[b] = -1;
#pragma unroll
  for (int u = 0; u < RING; ++u)
    if (u >= U0 && u < U) load(buf0 + u * F, g.frames + (size_t)uslot[u] * F, bar0 + 8 * u);
  uint8_t* out = g.frames_out + (size_t)b * A0_SLOTS * F;
#pragma unroll
  for (int u = 0; u < A0_SLOTS; ++u) {
    if (u < U) {
      const int r = u % RING;
      a0_mbar_wait(bar0 + 8 * r, (u / RING) & 1);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
#pragma unroll
      for (int j = 0; j < A0_SLOTS; ++j)
        if (dmask[u] & (1u << j)) store(out + (size_t)j * F, buf0 + r * F);
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      if (u + RING < U) {
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        load(buf0 + r * F, g.frames + (size_t)uslot[u + RING] * F, bar0 + 8 * r);
      }
    }
  }
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  if (g.progress) {
    const unsigned int old = atomicAdd(g.progress, 1u);
    if (old == (unsigned int)g.gtotal - 1u) *reinterpret_cast<volatile unsigned int*>(g.progress) = 0u;   // every draw done: nobody polls any more
  }
#ifdef A0_TRACE
  _tx[0] = (unsigned long long)g.gbase + 1;     // which launch (gather wave) the record belongs to: its first draw + 1
#endif
  A0_TEND(3);
  if (g.mail) asm volatile("griddepcontrol.wait;" ::: "memory");
}

__global__ void __launch_bounds__(32) a0_k3_gather_tma(const A0GatherArgs g) { a0_k3_gather_body<K3_RING>(g); }

// Variant 3: the same data movement split over TWO CTAs per transition (even / odd distinct
// frames), each with a two-buffer ring (14 KB): 2x finer work units even out the SM load of a
// single-wave launch (640 transitions on 148 SMs is 4 or 5 CTAs per SM, 1280 half-transitions is
// 8 or 9) at the price of walking the record chain twice.  Scalar outputs come from the even CTA.
constexpr int K3S_RING = 2;
__global__ void __launch_bounds__(32) a0_k3_gather_tma_split(const A0GatherArgs g_in) {
  extern __shared__ __align__(128) uint8_t a0_smem[];
  __shared__ __align__(8) uint64_t bars[K3S_RING];
  if (threadIdx.x != 0) return;
  A0_PDL_PROLOGUE();
  const int b = blockIdx.x >> 1;
  const int half = blockIdx.x & 1;
  A0GatherArgs g = g_in;
  if (half) {
    g.action_out = nullptr; g.reward64_out = nullptr; g.reward32_out = nullptr; g.done8_out = nullptr;
    g.done32_out = nullptr; g.boot_out = nullptr;
  }
  const uint32_t F = (uint32_t)g.F;
  const uint32_t bar0 = a0_smem_u32(&bars[0]);
  const uint32_t buf0 = a0_smem_u32(a0_smem);
  int64_t p0 = g.idx[b];
  bool ok = p0 >= 0 && p0 < g.N;
  if (!ok) p0 = 0;
  const int4 sa = *reinterpret_cast<const int4*>(g.rec_slots + (size_t)p0 * A0_SLOTS);
  const A0RecInfo info0 = g.rec_info[p0];
#pragma unroll
  for (int r = 0; r < K3S_RING; ++r) a0_mbar_init(bar0 + 8 * r, 1);
  a0_fence_barrier_init();
  int32_t uslot[A0_SLOTS];
  uint32_t dmask[A0_SLOTS];
  int U = 0;
  {
    int32_t s4[A0_STACK] = {sa.x, sa.y, sa.z, sa.w};
#pragma unroll
    for (int j = 0; j < A0_STACK; ++j) {
      if (s4[j] < 0 || s4[j] >= g.NF) { s4[j] = 0; ok = false; }
      a0_unique_add(s4[j], j, uslot, dmask, U);
    }
  }
  const int U0 = U;
  // this CTA's frames are u = half, half + 2, ...; its i-th frame uses ring buffer i % 2
#pragma unroll
  for (int i = 0; i < K3S_RING; ++i) {
    const int u = half + 2 * i;
    if (u < U0) a0_bulk_load(buf0 + i * F, g.frames + (size_t)uslot[u] * F, F, bar0 + 8 * i);
  }
  const int64_t pl = a0_walk_window(g, b, p0, info0, ok);
  const int4 sc = reinterpret_cast<const int4*>(g.rec_slots + (size_t)pl * A0_SLOTS)[1];
  {
    int32_t s4[A0_STACK] = {sc.x, sc.y, sc.z, sc.w};
#pragma unroll
    for (int j = 0; j < A0_STACK; ++j) {
      if (s4[j] < 0 || s4[j] >= g.NF) { s4[j] = 0; ok = false; }
      a0_unique_add(s4[j], A0_STACK + j, uslot, dmask, U);
    }
  }
  if (!ok && g.action_out) g.action_out[b] = -1;
#pragma unroll
  for (int i = 0; i < K3S_RING; ++i) {
    const int u = half + 2 * i;
    if (u >= U0 && u < U) a0_bulk_load(buf0 + i * F, g.frames + (size_t)uslot[u] * F, F, bar0 + 8 * i);
  }
  uint8_t* out = g.frames_out + (size_t)b * A0_SLOTS * F;
#pragma unroll
  for (int i = 0; i < A0_SLOTS / 2; ++i) {
    const int u = half + 2 * i;
    if (u < U) {
      const int r = i % K3S_RING;
      a0_mbar_wait(bar0 + 8 * r, (i / K3S_RING) & 1);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      uint32_t dm = 0;
#pragma unroll
      for (int q = 0; q < A0_SLOTS; ++q)
        if (q == u) dm = dmask[q];
#pragma unroll
      for (int j = 0; j < A0_SLOTS; ++j)
        if (dm & (1u << j)) a0_bulk_store(out + (size_t)j * F, buf0 + r * F, F);
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      const int un = u + 2 * K3S_RING;
      if (un < U) {
        int32_t sl = 0;
#pragma unroll
        for (int q = 0; q < A0_SLOTS; ++q)
          if (q == un) sl = uslot[q];
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        a0_bulk_load(buf0 + r * F, g.frames + (size_t)sl * F, F, bar0 + 8 * r);
      }
    }
  }
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// Variant 2: all (up to 8) distinct frames staged at once behind one mbarrier (56 KB of shared
// memory, 4 CTAs per SM).  Kept as the measured alternative to the ring.
__global__ void __launch_bounds__(32) a0_k3_gather_tma_full(const A0GatherArgs g) {
  extern __shared__ __align__(128) uint8_t a0_smem[];
  __shared__ __align__(8) uint64_t bar;
  if (threadIdx.x != 0) return;
  A0_PDL_PROLOGUE();
  const int b = blockIdx.x;
  int32_t slot[A0_SLOTS];
  a0_resolve_window(g, b, slot);
  const uint32_t F = (uint32_t)g.F;
  int32_t uslot[A0_SLOTS];
  uint32_t dmask[A0_SLOTS];
  const int U = a0_unique_frames(slot, uslot, dmask);
  const uint32_t bar_a = a0_smem_u32(&bar);
  const uint32_t buf0 = a0_smem_u32(a0_smem);
  a0_mbar_init(bar_a, (uint32_t)U);
  a0_fence_barrier_init();
#pragma unroll
  for (int u = 0; u < A0_SLOTS; ++u)
    if (u < U) a0_bulk_load(buf0 + u * F, g.frames + (size_t)uslot[u] * F, F, bar_a);
  a0_mbar_wait(bar_a, 0);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  uint8_t* out = g.frames_out + (size_t)b * A0_SLOTS * F;
#pragma unroll
  for (int u = 0; u < A0_SLOTS; ++u)
    if (u < U) {
#pragma unroll
      for (int j = 0; j < A0_SLOTS; ++j)
        if (dmask[u] & (1u << j)) a0_bulk_store(out + (size_t)j * F, buf0 + u * F, F);
    }
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// Variant 1: same traffic with 16-byte LDG/STG through registers (no shared memory); kept as the
// measured alternative to the TMA path.
constexpr int K3_LDG_THREADS = 256;
__global__ void __launch_bounds__(K3_LDG_THREADS) a0_k3_gather_ldg(const A0GatherArgs g) {
  __shared__ int32_t s_slot[A0_SLOTS];
  A0_PDL_PROLOGUE();
  const int b = blockIdx.x;
  if (threadIdx.x == 0) {
    int32_t slot[A0_SLOTS];
    a0_resolve_window(g, b, slot);
#pragma unroll
    for (int j = 0; j < A0_SLOTS; ++j) s_slot[j] = slot[j];
  }
  __syncthreads();
  int32_t slot[A0_SLOTS];
#pragma unroll
  for (int j = 0; j < A0_SLOTS; ++j) slot[j] = s_slot[j];
  const int nvec = g.F >> 4;
  uint4* out = reinterpret_cast<uint4*>(g.frames_out + (size_t)b * A0_SLOTS * g.F);
#pragma unroll
  for (int j = 0; j < A0_SLOTS; ++j) {
    bool first = true;
#pragma unroll
    for (int k = 0; k < A0_SLOTS; ++k)
      if (k < j && slot[k] == slot[j]) first = false;
    if (!first) continue;
    const uint4* src = reinterpret_cast<const uint4*>(g.frames + (size_t)slot[j] * g.F);
    for (int i = threadIdx.x; i < nvec; i += K3_LDG_THREADS) {
      const uint4 v = __ldg(src + i);
#pragma unroll
      for (int k = 0; k < A0_SLOTS; ++k)
        if (k >= j && slot[k] == slot[j]) out[(size_t)k * nvec + i] = v;
    }
  }
}

// K3 with the learner's input conversion fused in (agent.py:129-135: frames.reshape(-1, 8, 84, 84)
// .float().div(255) and the split into obs / next_obs; trainer.py:88-90 is the .float()): every distinct
// frame is fetched ONCE with cp.async.bulk into the same 4-buffer shared-memory ring as variant 0, and
// the CTA's four warps turn it into normalised fp32 and write it to every stack position it occupies
// in the two contiguous outputs obs[B][4][F] and next_obs[B][4][F] with fully coalesced 16-byte
// stores.  (S+n)F bytes read + 8F*4 written per transition (39F at n = 3) instead of the 119F of
// gather-to-u8 + .float() + .div() as three passes.
//   norm_mode 0: x / 255 correctly rounded -- what torch computes on the CPU (the oracle);
//                q = x*r, e = fma(-q, 255, x), q' = fma(e, r, q) is exact for x in 0..255
//   norm_mode 1: x * fl(1/255)             -- what torch's CUDA div-by-scalar kernel computes
//   norm_mode 2: (float)x                  -- .float() only
constexpr int K3F_THREADS = 128;
__device__ __forceinline__ float a0_norm255(float x, int mode) {
  const float r = 1.0f / 255.0f;
  if (mode == 2) return x;
  const float q = __fmul_rn(x, r);
  if (mode == 1) return q;
  const float e = __fmaf_rn(-q, 255.0f, x);
  return __fmaf_rn(e, r, q);
}
// byte -> float without the conversion pipe: 0x4B000000 | byte is 2^23 + byte exactly
__device__ __forceinline__ float a0_byte_norm(uint32_t byte, int mode) {
  return a0_norm255(__uint_as_float(0x4B000000u | byte) - 8388608.0f, mode);
}
// bf16(fl32(norm(x))), round to nearest even: what .float().div(255).to(torch.bfloat16) gives.  Two
// values per 32-bit word, low half first (little endian: element 2i in the low half).
__device__ __forceinline__ uint32_t a0_bf16_pair(float lo, float hi) {
  auto rne = [](float v) -> uint32_t {
    const uint32_t u = __float_as_uint(v);               // finite, non-negative here (0..255 or 0..1)
    return (u + 0x7fffu + ((u >> 16) & 1u)) >> 16;
  };
  return rne(lo) | (rne(hi) << 16);
}

// One group of pixels of staged frame `src` into every stack position it fills.
//   OutT = float:    4 pixels  (one 32-bit shared-memory word)  -> one float4 (16 B) store per position
//   OutT = uint16_t: 8 pixels  (one 64-bit shared-memory word)  -> 8 bf16 = one uint4 (16 B) store
template <typename OutT> struct A0Conv;
template <> struct A0Conv<float> {
  static constexpr int PIX = 4;
  __device__ static __forceinline__ void run(const uint8_t* src, int i, uint32_t dm, float* obs_b, float* next_b, uint32_t F,
                                             int mode) {
    const uint32_t px = reinterpret_cast<const uint32_t*>(src)[i];
    float4 v;
    v.x = a0_byte_norm(px & 0xffu, mode);
    v.y = a0_byte_norm((px >> 8) & 0xffu, mode);
    v.z = a0_byte_norm((px >> 16) & 0xffu, mode);
    v.w = a0_byte_norm(px >> 24, mode);
#pragma unroll
    for (int j = 0; j < A0_SLOTS; ++j)
      if (dm & (1u << j)) {
        float* dst = (j < A0_STACK ? obs_b + (size_t)j * F : next_b + (size_t)(j - A0_STACK) * F);
        reinterpret_cast<float4*>(dst)[i] = v;
      }
  }
};
template <> struct A0Conv<uint16_t> {
  static constexpr int PIX = 8;
  __device__ static __forceinline__ void run(const uint8_t* src, int i, uint32_t dm, uint16_t* obs_b, uint16_t* next_b,
                                             uint32_t F, int mode) {
    const uint2 px = reinterpret_cast<const uint2*>(src)[i];
    uint4 v;
    v.x = a0_bf16_pair(a0_byte_norm(px.x & 0xffu, mode), a0_byte_norm((px.x >> 8) & 0xffu, mode));
    v.y = a0_bf16_pair(a0_byte_norm((px.x >> 16) & 0xffu, mode), a0_byte_norm(px.x >> 24, mode));
    v.z = a0_bf16_pair(a0_byte_norm(px.y & 0xffu, mode), a0_byte_norm((px.y >> 8) & 0xffu, mode));
    v.w = a0_bf16_pair(a0_byte_norm((px.y >> 16) & 0xffu, mode), a0_byte_norm(px.y >> 24, mode));
#pragma unroll
    for (int j = 0; j < A0_SLOTS; ++j)
      if (dm & (1u << j)) {
        uint16_t* dst = (j < A0_STACK ? obs_b + (size_t)j * F : next_b + (size_t)(j - A0_STACK) * F);
        reinterpret_cast<uint4*>(dst)[i] = v;
      }
  }
};

template <typename OutT>
__global__ void __launch_bounds__(K3F_THREADS)
a0_k3_gather_cvt(const A0GatherArgs g, OutT* __restrict__ obs_out, OutT* __restrict__ next_out, int norm_mode) {
  extern __shared__ __align__(128) uint8_t a0_smem[];
  __shared__ __align__(8) uint64_t bars[K3_RING];
  __shared__ int32_t s_uslot[A0_SLOTS];
  __shared__ uint32_t s_dmask[A0_SLOTS];
  __shared__ int s_U;
  A0_PDL_PROLOGUE();
  const int b = blockIdx.x;
  const uint32_t F = (uint32_t)g.F;
  const uint32_t bar0 = a0_smem_u32(&bars[0]);
  const uint32_t buf0 = a0_smem_u32(a0_smem);
  if (threadIdx.x == 0) {
    int64_t p0 = g.idx[b];
    bool ok = p0 >= 0 && p0 < g.N;
    if (!ok) p0 = 0;
    const int4 sa = *reinterpret_cast<const int4*>(g.rec_slots + (size_t)p0 * A0_SLOTS);
    const A0RecInfo info0 = g.rec_info[p0];
    A0Spec sp;
    a0_spec_fetch(g, p0, sp);
#pragma unroll
    for (int r = 0; r < K3_RING; ++r) a0_mbar_init(bar0 + 8 * r, 1);
    a0_fence_barrier_init();
    int32_t uslot[A0_SLOTS];
    uint32_t dmask[A0_SLOTS];
    int U = 0;
    {
      int32_t s4[A0_STACK] = {sa.x, sa.y, sa.z, sa.w};
#pragma unroll
      for (int j = 0; j < A0_STACK; ++j) {
        if (s4[j] < 0 || s4[j] >= g.NF) { s4[j] = 0; ok = false; }
        a0_unique_add(s4[j], j, uslot, dmask, U);
      }
    }
    const int U0 = U;
#pragma unroll
    for (int u = 0; u < K3_RING; ++u)
      if (u < U0) a0_bulk_load(buf0 + u * F, g.frames + (size_t)uslot[u] * F, F, bar0 + 8 * u);
    int4 sc;
    a0_walk_window_spec(g, b, p0, info0, sp, ok, sc);
    {
      int32_t s4[A0_STACK] = {sc.x, sc.y, sc.z, sc.w};
#pragma unroll
      for (int j = 0; j < A0_STACK; ++j) {
        if (s4[j] < 0 || s4[j] >= g.NF) { s4[j] = 0; ok = false; }
        a0_unique_add(s4[j], A0_STACK + j, uslot, dmask, U);
      }
    }
    if (!ok && g.action_out) g.action_out[b] = -1;
#pragma unroll
    for (int u = 0; u < K3_RING; ++u)
      if (u >= U0 && u < U) a0_bulk_load(buf0 + u * F, g.frames + (size_t)uslot[u] * F, F, bar0 + 8 * u);
#pragma unroll
    for (int u = 0; u < A0_SLOTS; ++u) { s_uslot[u] = uslot[u]; s_dmask[u] = u < U ? dmask[u] : 0u; }
    s_U = U;
  }
  __syncthreads();
  const int U = s_U;
  const int groups = (int)(F / A0Conv<OutT>::PIX);
  const size_t stack_elems = (size_t)A0_STACK * F;
  OutT* obs_b = obs_out + (size_t)b * stack_elems;
  OutT* next_b = next_out + (size_t)b * stack_elems;
  for (int u = 0; u < U; ++u) {
    const int r = u % K3_RING;
    a0_mbar_wait(bar0 + 8 * r, (u / K3_RING) & 1);
    const uint8_t* src = a0_smem + (size_t)r * F;
    const uint32_t dm = s_dmask[u];
    for (int i = threadIdx.x; i < groups; i += K3F_THREADS) A0Conv<OutT>::run(src, i, dm, obs_b, next_b, F, norm_mode);
    if (u + K3_RING < U) {
      __syncthreads();                                     // every thread has read buffer r
      if (threadIdx.x == 0) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        a0_bulk_load(buf0 + r * F, g.frames + (size_t)s_uslot[u + K3_RING] * F, F, bar0 + 8 * r);
      }
    }
  }
}

template <typename OutT>
static int a0_gather_cvt(a0_replay_t* h, const int64_t* idx, int32_t count, int32_t n_step, double gamma, OutT* obs_out,
                         OutT* next_out, int32_t norm_mode, int64_t* action_out, double* reward64_out, float* reward32_out,
                         uint8_t* done8_out, float* done32_out, int64_t* boot_out, a0_stream_t stream_, const char* who) {
  A0_REQUIRE(h != nullptr, "%s: handle is NULL", who);
  A0_REQUIRE(count >= 0, "%s: negative count", who);
  if (count == 0) return A0_OK;
  A0_REQUIRE(idx && obs_out && next_out, "%s: idx, obs_out and next_out are required", who);
  A0_REQUIRE(n_step >= 1 && n_step <= A0_MAX_NSTEP, "%s: n_step %d outside [1,%d]", who, n_step, A0_MAX_NSTEP);
  A0_REQUIRE((((uintptr_t)obs_out | (uintptr_t)next_out) & 15) == 0, "%s: outputs must be 16-byte aligned", who);
  A0_REQUIRE(norm_mode >= 0 && norm_mode <= 2, "%s: norm_mode %d outside [0,2]", who, norm_mode);
  A0DeviceGuard guard(h->device);
  A0GatherArgs g;
  g.frames = h->frames; g.rec_slots = h->rec_slots; g.rec_info = h->rec_info; g.idx = idx;
  g.N = h->N; g.NF = h->NF; g.F = h->F; g.count = count; g.n_step = n_step; g.gamma = gamma;
  g.stride_hint = (h->stride_hint > 0 && h->stride_hint < h->N) ? (int32_t)h->stride_hint : 0;
  g.frames_out = nullptr; g.action_out = action_out; g.reward64_out = reward64_out;
  g.reward32_out = reward32_out; g.done8_out = done8_out; g.done32_out = done32_out; g.boot_out = boot_out;
  g.mail = nullptr; g.fault = nullptr; g.mail_timeout_ns = 0;
  g.progress = nullptr; g.window = 0; g.gbase = 0; g.gtotal = 0;
  g.l2_hints = 0;
  const size_t smem = (size_t)K3_RING * h->F;
  int rc = a0_smem_at_least((const void*)a0_k3_gather_cvt<OutT>, h->device, smem);
  if (rc) return rc;
  A0_LAUNCH(a0_k3_gather_cvt<OutT>, (unsigned)count, K3F_THREADS, smem, (cudaStream_t)stream_, 1, A0_PDL_K3, g, obs_out, next_out,
            (int)norm_mode);
  return A0_OK;
}

extern "C" int a0_rb_gather_f32(a0_replay_t* h, const int64_t* idx, int32_t count, int32_t n_step, double gamma,
                                float* obs_out, float* next_out, int32_t norm_mode, int64_t* action_out,
                                double* reward64_out, float* reward32_out, uint8_t* done8_out, float* done32_out,
                                int64_t* boot_out, a0_stream_t stream_) {
  return a0_gather_cvt<float>(h, idx, count, n_step, gamma, obs_out, next_out, norm_mode, action_out, reward64_out,
                              reward32_out, done8_out, done32_out, boot_out, stream_, "a0_rb_gather_f32");
}

extern "C" int a0_rb_gather_bf16(a0_replay_t* h, const int64_t* idx, int32_t count, int32_t n_step, double gamma,
                                 uint16_t* obs_out, uint16_t* next_out, int32_t norm_mode, int64_t* action_out,
                                 double* reward64_out, float* reward32_out, uint8_t* done8_out, float* done32_out,
                                 int64_t* boot_out, a0_stream_t stream_) {
  return a0_gather_cvt<uint16_t>(h, idx, count, n_step, gamma, obs_out, next_out, norm_mode, action_out, reward64_out,
                                 reward32_out, done8_out, done32_out, boot_out, stream_, "a0_rb_gather_bf16");
}

static int a0_k3_smem_attr(a0_replay_t* h, size_t smem) {
  return a0_smem_at_least((const void*)a0_k3_gather_tma, h->device, smem, true);
}
// The gather half of a0_rb_sample_gather: variant 0 taking its record positions from the mailbox, always
// launched with programmatic stream serialization so that it becomes resident under the sampler.
int a0_gather_launch_mail(a0_replay* h, const int64_t* idx, long long* mail, int32_t count, int32_t n_step, double gamma,
                          const A0GatherOut& out, cudaStream_t stream, int64_t policy_count, int32_t window, int32_t gbase) {
  A0GatherArgs g;
  g.frames = h->frames; g.rec_slots = h->rec_slots; g.rec_info = h->rec_info; g.idx = idx;
  g.N = h->N; g.NF = h->NF; g.F = h->F; g.count = count; g.n_step = n_step; g.gamma = gamma;
  g.stride_hint = (h->stride_hint > 0 && h->stride_hint < h->N) ? (int32_t)h->stride_hint : 0;
  g.frames_out = out.frames; g.action_out = out.action; g.reward64_out = out.reward64;
  g.reward32_out = out.reward32; g.done8_out = out.done8; g.done32_out = out.done32; g.boot_out = out.boot;
  g.mail = mail;
  g.progress = window > 0 ? h->counter + A0_K3_PROGRESS : nullptr;
  g.window = window; g.gbase = gbase; g.gtotal = (int32_t)policy_count;
  g.fault = h->fault_dev;
  g.mail_timeout_ns = a0_option_mail_timeout_ns();
  // a wave of a larger draw (a0_rb_gather_mail) takes the L2 policy of the whole draw
  g.l2_hints = a0_option_k3_l2((policy_count > count ? policy_count : (int64_t)count) * 16 * h->F);
  const size_t smem = (size_t)K3_RING * h->F;
  int rc = a0_k3_smem_attr(h, smem);
  if (rc) return rc;
  A0_LAUNCH(a0_k3_gather_tma, (unsigned)count, 32, smem, stream, 1, A0_PDL_FORCE, g);
  return A0_OK;
}

extern "C" int a0_rb_gather_unpaired(a0_replay_t* h, int32_t count, uint8_t* frames_out, a0_stream_t stream_) {
  A0_REQUIRE(h && frames_out && count > 0, "a0_rb_gather_unpaired: bad argument");
  A0DeviceGuard guard(h->device);
  int rc = a0_mail_reserve(h, count, (cudaStream_t)stream_);
  if (rc) return rc;
  const A0GatherOut out = {frames_out, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  return a0_gather_launch_mail(h, nullptr, h->mail, count, 1, 0.99, out, (cudaStream_t)stream_);
}

extern "C" int a0_rb_gather(a0_replay_t* h, const int64_t* idx, int32_t count, int32_t n_step, double gamma,
                            uint8_t* frames_out, int64_t* action_out, double* reward64_out,
                            float* reward32_out, uint8_t* done8_out, float* done32_out,
                            int64_t* boot_out, int32_t variant, a0_stream_t stream_) {
  A0_REQUIRE(h != nullptr, "a0_rb_gather: handle is NULL");
  A0_REQUIRE(count >= 0, "a0_rb_gather: negative count");
  if (count == 0) return A0_OK;
  A0_REQUIRE(idx && frames_out, "a0_rb_gather: idx and frames_out are required");
  A0_REQUIRE(n_step >= 1 && n_step <= A0_MAX_NSTEP, "a0_rb_gather: n_step %d outside [1,%d]", n_step, A0_MAX_NSTEP);
  A0_REQUIRE(((uintptr_t)frames_out & 15) == 0, "a0_rb_gather: frames_out must be 16-byte aligned");
  A0_REQUIRE(variant >= 0 && variant <= 3, "a0_rb_gather: unknown variant %d", variant);
  { int frc = a0_check_fault(h, "a0_rb_gather"); if (frc) return frc; }
  A0DeviceGuard guard(h->device);
  cudaStream_t stream = (cudaStream_t)stream_;
  A0GatherArgs g;
  g.frames = h->frames; g.rec_slots = h->rec_slots; g.rec_info = h->rec_info; g.idx = idx;
  g.N = h->N; g.NF = h->NF; g.F = h->F; g.count = count; g.n_step = n_step; g.gamma = gamma;
  g.stride_hint = (h->stride_hint > 0 && h->stride_hint < h->N) ? (int32_t)h->stride_hint : 0;
  g.frames_out = frames_out; g.action_out = action_out; g.reward64_out = reward64_out;
  g.reward32_out = reward32_out; g.done8_out = done8_out; g.done32_out = done32_out; g.boot_out = boot_out;
  g.mail = nullptr; g.fault = nullptr; g.mail_timeout_ns = 0;
  g.progress = nullptr; g.window = 0; g.gbase = 0; g.gtotal = 0;
  g.l2_hints = a0_option_k3_l2((int64_t)count * 16 * h->F);
  if (variant == 3) {
    const size_t smem = (size_t)K3S_RING * h->F;
    int rc = a0_smem_at_least((const void*)a0_k3_gather_tma_split, h->device, smem);
    if (rc) return rc;
    A0_LAUNCH(a0_k3_gather_tma_split, (unsigned)count * 2, 32, smem, stream, 1, A0_PDL_K3, g);
  } else if (variant == 0 || variant == 2) {
    const size_t smem = (size_t)(variant == 0 ? K3_RING : A0_SLOTS) * h->F;
    int rc = variant == 0 ? a0_k3_smem_attr(h, smem) : a0_smem_at_least((const void*)a0_k3_gather_tma_full, h->device, smem);
    if (rc) return rc;
    if (variant == 0) A0_LAUNCH(a0_k3_gather_tma, (unsigned)count, 32, smem, stream, 1, A0_PDL_K3, g);
    else A0_LAUNCH(a0_k3_gather_tma_full, (unsigned)count, 32, smem, stream, 1, A0_PDL_K3, g);
  } else {
    A0_LAUNCH(a0_k3_gather_ldg, (unsigned)count, K3_LDG_THREADS, 0, stream, 1, A0_PDL_K3, g);
  }
  return A0_OK;
}
