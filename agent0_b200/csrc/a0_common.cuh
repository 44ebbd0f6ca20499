// Shared definitions for the agent0_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "../../include/agent0_b200.h"

// Per-record side data (16 B, one vector load).  Rewards stay float64 because the reference
// accumulates n-step returns in numpy float64 (agent0/deepq/agent.py:65-69).
struct __align__(16) A0RecInfo {
  double reward;
  int32_t action_done;   // action | (done << 31)
  int32_t link;          // ring position of the next record of the same stream, -1 if none yet
};

constexpr int A0_MAX_BATCHES = 4096;   // batches per a0_pt_sample call

struct A0Staging {        // one half of the double-buffered ingest staging area
  uint8_t* host;          // page-locked
  uint8_t* dev;
  size_t capacity;
  cudaEvent_t event;      // recorded after the kernels that consume `dev`
  cudaEvent_t copied;     // recorded on the copy stream after the H2D copies (A0_INGEST_COPY_STREAM)
};

struct a0_replay {
  int32_t device;
  int64_t N;             // record capacity
  int64_t NF;            // frame capacity
  int32_t F;             // bytes per frame (multiple of 16)
  int64_t P;             // tree leaves (power of two >= N)
  int32_t D;             // tree depth, P == 1 << D
  uint8_t* frames;       // [NF][F]
  int32_t* rec_slots;    // [N][8]
  A0RecInfo* rec_info;   // [N]
  float* tree;           // [2P], node 1 = root, leaf j at P + j
  float* max_p;          // device scalar
  float* dyn;            // device {top, beta, sum_offset}: a0_rb_set_dynamic / a0_pt_sample(top < 0)
  int32_t* winner;       // [N] scratch for last-writer-wins, kept at -1 between calls
  int32_t* dirty;        // [P >> 12] chunk needs its sub-tree recomputed
  unsigned int* counter; // [A0_MAX_BATCHES] per-batch tickets of the sampler epilogue, [16] rebuild ticket,
                         // [A0_MAX_BATCHES] per-batch max weight (float bits); all zero between launches;
                         // then the sampler's RNG words: CTA ticket and the 64-bit call counter
  A0Staging staging[2];
  int staging_turn;
  cudaStream_t copy_stream;   // lazily created; carries the ingest DMA under A0_INGEST_COPY_STREAM
  int64_t stride_hint;        // distance record -> successor of the same stream seen by the last appends
                              // (0: not uniform); lets K3 fetch an n-step window without chasing links
  long long* mail;            // [mail_cap] sampler -> gather mailbox of a0_rb_sample_gather: draw g's record
  int64_t mail_cap;           // position + 1, 0 = empty; every word is consumed (reset) by the gather CTA
  int64_t mail_total;         // draws of the last a0_rb_sample_mail (its gather waves pick their L2 policy by the whole draw)
  int32_t progress_dirty;     // a windowed gather wave failed to launch: the next a0_rb_sample_mail re-arms the progress word
  int32_t* fault_host;        // mapped page-locked word a kernel sets when it gives up (mailbox wait timed out);
  int32_t* fault_dev;         // the next host call on the handle reports and clears it (a0_check_fault)
};
// A0_EFAULT if a kernel of an earlier call on this handle reported a device-side fault
int a0_check_fault(a0_replay* h, const char* who);
uint64_t a0_option_mail_timeout_ns();
// Raises `kernel`'s dynamic shared-memory limit on `device` (the current device) to at least `bytes`, and with
// `max_carveout` asks for the largest shared-memory carveout.  The attribute belongs to the function for the whole
// process, so the record of what was set is process-wide too: one kept per shard or per thread would let a shard of
// small frames lower the limit that a shard of large frames still relies on.
int a0_smem_at_least(const void* kernel, int device, size_t bytes, bool max_carveout = false);

void a0_set_error(const char* fmt, ...);

#define A0_CUDA(expr)                                                          \
  do {                                                                         \
    cudaError_t _e = (expr);                                                   \
    if (_e != cudaSuccess) {                                                   \
      a0_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),     \
                   __FILE__, __LINE__);                                        \
      return (int)_e;                                                          \
    }                                                                          \
  } while (0)

#define A0_REQUIRE(cond, ...)                                                  \
  do {                                                                         \
    if (!(cond)) {                                                             \
      a0_set_error(__VA_ARGS__);                                               \
      return A0_EINVAL;                                                        \
    }                                                                          \
  } while (0)

#define A0_LAUNCH_CHECK()                                                      \
  do {                                                                         \
    cudaError_t _e = cudaGetLastError();                                       \
    if (_e != cudaSuccess) {                                                   \
      a0_set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), \
                   __FILE__, __LINE__);                                        \
      return (int)_e;                                                          \
    }                                                                          \
  } while (0)

// ---- optional device-side timeline (build with -DA0_TRACE: tools/trace_step.py) ----------------------
// Every traced CTA appends {kernel id, block, t_entry, t_mid, t_exit} (%globaltimer, ns) to a log; the
// production build compiles all of it away.
#ifdef A0_TRACE
struct A0TraceRec { unsigned long long t0, t1, t2; int kid, blk; unsigned long long x[8]; };
static __device__ A0TraceRec* a0_trace_buf;
static __device__ unsigned int* a0_trace_cur;
__device__ __forceinline__ unsigned long long a0_now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define A0_TRACE_SETTER(name)                                   \
  int name(void* buf, void* cur) {                              \
    cudaMemcpyToSymbol(a0_trace_buf, &buf, sizeof(buf));        \
    cudaMemcpyToSymbol(a0_trace_cur, &cur, sizeof(cur));        \
    return 0;                                                   \
  }
#define A0_T0() const unsigned long long _t0 = a0_now(); unsigned long long _t2 = 0, _tx[8] = {0, 0, 0, 0, 0, 0, 0, 0}
#define A0_TX(i) _tx[i] = (unsigned long long)clock64()      /* SM cycles: cheap, for phases inside one CTA */
#define A0_TMID() _t2 = a0_now()
#define A0_TEND(kid)                                                                       \
  do {                                                                                     \
    if (a0_trace_buf) {                                                                    \
      const unsigned _i = atomicAdd(a0_trace_cur, 1u);                                     \
      if (_i < (1u << 16)) a0_trace_buf[_i] = A0TraceRec{_t0, a0_now(), _t2, kid, (int)blockIdx.x, {_tx[0], _tx[1], _tx[2], _tx[3], _tx[4], _tx[5], _tx[6], _tx[7]}}; \
    }                                                                                      \
  } while (0)
#else
#define A0_T0() do {} while (0)
#define A0_TMID() do {} while (0)
#define A0_TX(i) do {} while (0)
#define A0_TEND(kid) do {} while (0)
#endif

// ---- launches ---------------------------------------------------------------------------------------
// Kernels can be launched with programmatic stream serialization (PDL): the kernel may become
// resident while its predecessor in the stream drains, executes griddepcontrol.wait as its first
// instruction (full completion + visibility of everything before it, so stream-order semantics
// are unchanged) and immediately lets its own successor start launching.  What this removes is
// part of the launch gap between the short dependent K4 kernels of one Trainer.step, eagerly and inside
// CUDA graphs.  a0_set_option(A0_OPT_PDL, mask) / A0_PDL=mask in the environment selects the kernel
// classes that use it (0 = none).
// kernel classes for the PDL mask (A0_OPT_PDL): which launches carry the attribute
enum { A0_PDL_K4 = 1, A0_PDL_K2 = 2, A0_PDL_K3 = 4, A0_PDL_K1 = 8, A0_PDL_FORCE = 1 << 30 };
constexpr int A0_PDL_DEFAULT = A0_PDL_K4;   // measured: K4-only is best at B=32 and B=512 (profiles/r01_kernel_options.json)
bool a0_pdl_enabled(int kernel_class);
int a0_option_k2b_levels();
constexpr int A0_K3_L2_DEFAULT = 4;              // L2 hints of the default gather (A0_OPT_K3_L2): auto
constexpr int A0_K2B_BULK_MIN_DEFAULT = 2048;    // from this many indices (and >= 4 per 4096-leaf chunk): leaf writes + chunk rebuild on all SMs
int a0_option_k2b_bulk_min();
bool a0_option_fused_ingest();
void a0_set_c51_fast(int on);
void a0_set_k2b_small(int on);
void a0_set_k2b_chunks(int on);
void a0_set_k2b_sparse(int max_paths);
void a0_set_k2a_rounds(int on);
void a0_set_qh_sorted(int on);
void a0_set_qh_spec(int on);
void a0_set_k6_global(int on);

// (Measured alternative: launch_dependents BEFORE the wait lets a whole chain of dependent kernels
// become resident launches ahead.  It does not lower the ~2.85 us per-link cost of the batch-32 K4
// chain -- that cost is the completion hand-over, not launch latency -- and the pre-launched CTAs
// take SM resources from a heavy predecessor: QR-200 K4 10.6 -> 16.7 us.  Not used.)
#define A0_PDL_PROLOGUE()                                   \
  do {                                                      \
    asm volatile("griddepcontrol.wait;" ::: "memory");      \
    asm volatile("griddepcontrol.launch_dependents;");      \
  } while (0)

template <typename... KArgs, typename... Args>
static inline cudaError_t a0_launch(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem,
                                    cudaStream_t stream, unsigned cluster, int kernel_class, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  unsigned n = 0;
  if (cluster > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  if (a0_pdl_enabled(kernel_class)) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

#define A0_LAUNCH(...)                                                          \
  do {                                                                          \
    cudaError_t _e = a0_launch(__VA_ARGS__);                                    \
    if (_e != cudaSuccess) {                                                    \
      a0_set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e),  \
                   __FILE__, __LINE__);                                         \
      return (int)_e;                                                           \
    }                                                                           \
  } while (0)

struct A0DeviceGuard {
  int prev;
  explicit A0DeviceGuard(int dev) { cudaGetDevice(&prev); if (dev != prev) cudaSetDevice(dev); else prev = -1; }
  ~A0DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ---- K1 building blocks (used by a0_k1_append and by the fused append + mark launch) -----------------
// One staged frame into its ring slot with 16-byte vector loads/stores (7056 B = 441 uint4).
__device__ __forceinline__ void a0_k1_copy_frame(uint8_t* __restrict__ frames, int32_t F, int64_t NF,
                                                 const uint8_t* __restrict__ staged, const int32_t* __restrict__ new_pos,
                                                 const int32_t* __restrict__ src_idx, int f, int tid, int nthreads) {
  const int32_t pos = new_pos[f];
  if (pos < 0 || pos >= NF) return;
  // src_idx (optional): frame f of the append sits at staged[src_idx[f]] (the decoded reference entries
  // of a0_ex_extend, where only the de-duplicated frames are stored) instead of staged[f]
  const uint4* src = reinterpret_cast<const uint4*>(staged + (size_t)(src_idx ? src_idx[f] : f) * F);
  uint4* dst = reinterpret_cast<uint4*>(frames + (size_t)pos * F);
  const int nvec = F >> 4;
  for (int i = tid; i < nvec; i += nthreads) dst[i] = __ldg(src + i);
}
// Record r of the append: slots, {reward, action|done, link}, and the predecessor's successor link.
__device__ __forceinline__ void a0_k1_write_record(int32_t* __restrict__ rec_slots, A0RecInfo* __restrict__ rec_info,
                                                   int64_t N, const int32_t* __restrict__ meta, int r) {
  const int32_t* mt = meta + (size_t)r * A0_REC_META_I32;
  const int32_t pos = mt[0], link_from = mt[1], link_to = mt[2], action_done = mt[3];
  if (pos < 0 || pos >= N) return;
  int4* s = reinterpret_cast<int4*>(rec_slots + (size_t)pos * A0_SLOTS);
  s[0] = make_int4(mt[4], mt[5], mt[6], mt[7]);
  s[1] = make_int4(mt[8], mt[9], mt[10], mt[11]);
  A0RecInfo info;
  info.reward = __hiloint2double(mt[13], mt[12]);
  info.action_done = action_done;
  info.link = link_to;
  rec_info[pos] = info;
  // predecessor written by an earlier append: only its link word is touched
  if (link_from >= 0 && link_from < N) rec_info[link_from].link = pos;
}
// {top, beta, sum_offset} for a0_pt_sample(top < 0); dyn == NULL: nothing to publish
struct A0Dyn {
  float* dyn;
  float top, beta, sum_offset;
};

// a0_sumtree.cu: marks (a0_pt_mark) and the append (a0_rb_append) of one small ingest in ONE launch.
// Returns A0_NOFIT when the sizes do not fit the fused kernel (the caller then launches the two separately).
constexpr int A0_NOFIT = -100;
int a0_launch_mark_append(a0_replay* h, const int32_t* marks, int32_t n_marks, float alpha, const uint8_t* new_frames,
                          const int32_t* new_frame_pos, const int32_t* src_idx, int32_t n_new, const int32_t* rec_meta,
                          int32_t m, const A0Dyn& dyn, cudaStream_t stream);
// a0_replay.cu: a0_rb_append that also publishes the sampler's dynamic scalars
int a0_append_launch(a0_replay* h, const uint8_t* new_frames, const int32_t* new_frame_pos, const int32_t* src_idx,
                     int32_t n_new, const int32_t* rec_meta, int32_t m, const A0Dyn& dyn, cudaStream_t stream);

// a0_ingest.cu: executes an index plan (staged upload + K2b marks + K1 append); with FRAMES_ON_DEVICE and
// new_frame_src the append reads frames[new_frame_src[j]] (the decoded entries of a0_ex_extend)
int a0_ingest_plan_impl(a0_replay_t* h, const a0_plan_t* plan, const uint8_t* frames, const int64_t* new_frame_src,
                        int32_t flags, float alpha, a0_stream_t stream, const A0Dyn& dyn);

// a0_sumtree.cu / a0_replay.cu: the two launches behind a0_rb_sample_gather (see there)
struct A0GatherOut {
  uint8_t* frames;
  int64_t* action;
  double* reward64;
  float* reward32;
  uint8_t* done8;
  float* done32;
  int64_t* boot;
};
int a0_gather_launch_mail(a0_replay* h, const int64_t* idx, long long* mail, int32_t count, int32_t n_step, double gamma,
                          const A0GatherOut& out, cudaStream_t stream, int64_t policy_count = 0, int32_t window = 0, int32_t gbase = 0);
constexpr int A0_K3_PROGRESS = 2 * A0_MAX_BATCHES + 40;      // counter[] word: completed draws of the current windowed gather
int a0_mail_reserve(a0_replay* h, int32_t total, cudaStream_t stream);

// a0_ckpt.cu's access to the other modules' state: the ring index (a0_ingest.cu) and the reference-tuple ingest
// (a0_extend.cu: the K6a decode of one batch of at most 2048 blobs into its scratch, and the stream tails)
void a0_ix_clear(a0_index* ix);
void a0_ix_stream_ids(a0_index* ix, std::vector<int64_t>& out);      // ascending
int a0_ex_decode_dev(a0_extend* ex, const uint8_t* blobs, const int64_t* blob_len, int32_t mb, cudaStream_t cs,
                     const uint8_t** dec, const unsigned long long** hash, const int32_t** status);
int a0_ex_tails_save(a0_extend* ex, std::vector<uint8_t>& out);
int a0_ex_tails_check(int32_t F, const uint8_t* p, int64_t len, int64_t head_fs);
int a0_ex_tails_load(a0_extend* ex, const uint8_t* p, int64_t len, cudaStream_t cs);
void a0_ex_tails_clear(a0_extend* ex);
a0_replay* a0_ex_shard(a0_extend* ex);
constexpr int A0_RNG_CALL_WORD = 2 * A0_MAX_BATCHES + 34;   // counter[] words of the sampler's 64-bit call counter

__device__ __forceinline__ uint32_t a0_smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

// ---- TMA helpers (cp.async.bulk + mbarrier, SASS: UBLKCP / SYNCS) -------------------------------
__device__ __forceinline__ void a0_mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void a0_fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void a0_bulk_load(uint32_t smem_dst, const void* gsrc, uint32_t bytes, uint32_t bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_dst), "l"(gsrc), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void a0_mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  }
}
__device__ __forceinline__ void a0_bulk_store(void* gdst, uint32_t smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_src), "r"(bytes) : "memory");
}
// The same copies with an L2 eviction-priority hint.  The gather streams: a sampled frame is read once
// out of a multi-GB ring (no reuse before it is evicted anyway), so its lines are marked evict_first
// and stop displacing what the step re-reads from L2 -- the sum-tree, the records, and the network
// outputs K4 consumes (device timeline: K4's first loads land in 850 cycles without the gather's
// traffic in L2 and 1500 with it).
__device__ __forceinline__ uint64_t a0_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void a0_bulk_load_hint(uint32_t smem_dst, const void* gsrc, uint32_t bytes, uint32_t bar, uint64_t pol) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               ::"r"(smem_dst), "l"(gsrc), "r"(bytes), "r"(bar), "l"(pol) : "memory");
}
__device__ __forceinline__ void a0_bulk_store_hint(void* gdst, uint32_t smem_src, uint32_t bytes, uint64_t pol) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
               ::"l"(gdst), "r"(smem_src), "r"(bytes), "l"(pol) : "memory");
}

// ---- system-scope memory order: the words of a region shared with other processes and peer GPUs (K8, K9) ---------
__device__ __forceinline__ void a0_sys_fence() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }
__device__ __forceinline__ uint64_t a0_sys_ld_acquire(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint64_t a0_sys_ld_relaxed(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void a0_sys_st_relaxed(uint64_t* p, uint64_t v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void a0_sys_st_release(uint64_t* p, uint64_t v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint4 a0_sys_ld4_relaxed(const uint4* p) {
  uint4 v;
  asm volatile("ld.relaxed.sys.global.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void a0_sys_st4_relaxed(uint4* p, uint4 v) {
  asm volatile("st.relaxed.sys.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}

// ---- a device region shared with other processes through CUDA IPC (K8 weight snapshots, K9 transition inbox) -----
// ONE cudaMalloc allocation, so one cudaIpcMemHandle_t covers it, starting with a control block whose first two words
// are {uint32_t magic, format}: what a0_ipc_map checks before the caller reads anything else of the block.  The
// caller sets the device.
// A zeroed region of `bytes` starting with the control block `ctl`; a failed allocation is A0_ENOMEM.
inline int a0_ipc_create(const char* who, size_t bytes, const void* ctl, size_t ctl_bytes, uint8_t** region) {
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) {
    a0_set_error("%s: cudaMalloc of %zu bytes failed: %s", who, bytes, cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? A0_ENOMEM : (int)e;
  }
  e = cudaMemset(p, 0, bytes);
  if (e == cudaSuccess) e = cudaMemcpy(p, ctl, ctl_bytes, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    cudaFree(p);
    a0_set_error("%s: initialising the region failed: %s", who, cudaGetErrorString(e));
    return (int)e;
  }
  *region = static_cast<uint8_t*>(p);
  return A0_OK;
}
inline int a0_ipc_handle(uint8_t* region, uint8_t* out64) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  cudaIpcMemHandle_t h;
  A0_CUDA(cudaIpcGetMemHandle(&h, region));
  memcpy(out64, &h, 64);
  return A0_OK;
}
inline void a0_ipc_unmap(uint8_t* region) { cudaIpcCloseMemHandle(region); }
// Maps another process's region (peer access enabled lazily: a peer GPU's region is read over NVLink) and copies its
// control block to `ctl`; a block of another kind (`kind`: the owner named in the error) is A0_EINVAL.  A failed
// mapping's error names cudaIpcOpenMemHandle: callers tell "this machine refuses CUDA IPC" by it.
inline int a0_ipc_map(const char* who, const uint8_t* handle64, uint32_t magic, uint32_t format, const char* kind,
                      void* ctl, size_t ctl_bytes, uint8_t** region) {
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  void* p = nullptr;
  A0_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  const cudaError_t e = cudaMemcpy(ctl, p, ctl_bytes, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) {
    a0_ipc_unmap(static_cast<uint8_t*>(p));
    a0_set_error("%s: reading the control block failed: %s", who, cudaGetErrorString(e));
    return (int)e;
  }
  const uint32_t* w = static_cast<const uint32_t*>(ctl);
  if (w[0] != magic || w[1] != format) {
    a0_ipc_unmap(static_cast<uint8_t*>(p));
    a0_set_error("%s: the handle's region is not a %s region (magic %08x format %u)", who, kind, w[0], w[1]);
    return A0_EINVAL;
  }
  *region = static_cast<uint8_t*>(p);
  return A0_OK;
}

// ---- 64-bit frame content hash of K6a / K7 ---------------------------------------------------------
__device__ __forceinline__ uint32_t a0_k6_rotl(uint32_t x, int r) { return (x << r) | (x >> (32 - r)); }
__device__ __forceinline__ uint32_t a0_k6_mix32(uint32_t h) {
  h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
  return h;
}
// 64-bit content hash of one frame held in shared memory (K6a computes it while decoding, K7 while
// encoding, and K6b uses it as a gate in front of the byte compare).  Four independent 32-bit multiply-rotate streams over 16-byte
// vector loads -- three instructions per word (the first version's 64-bit multiplies were a fifth of the
// kernel's instructions).  Lanes are seeded differently, so equal words in different places do not cancel
// in the final xor across the warp.
__device__ __forceinline__ unsigned long long a0_k6_frame_hash(const uint8_t* frame, int nvec, int lane) {
  uint32_t h0 = 0x9E3779B1u * (uint32_t)(lane + 1), h1 = 0x85EBCA77u * (uint32_t)(lane + 33);
  uint32_t h2 = 0xC2B2AE3Du * (uint32_t)(lane + 65), h3 = 0x27D4EB2Fu * (uint32_t)(lane + 97);
  const uint4* v4 = reinterpret_cast<const uint4*>(frame);
#pragma unroll 2
  for (int i = lane; i < nvec; i += 32) {
    const uint4 v = v4[i];
    h0 = a0_k6_rotl((h0 ^ v.x) * 0x9E3779B1u, 13);
    h1 = a0_k6_rotl((h1 ^ v.y) * 0x85EBCA77u, 15);
    h2 = a0_k6_rotl((h2 ^ v.z) * 0xC2B2AE3Du, 17);
    h3 = a0_k6_rotl((h3 ^ v.w) * 0x27D4EB2Fu, 11);
  }
  uint32_t lo = a0_k6_mix32(h0 + 0x165667B1u * h2), hi = a0_k6_mix32(h1 + 0x9E3779B1u * h3);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo ^= __shfl_xor_sync(0xffffffffu, lo, o);
    hi ^= __shfl_xor_sync(0xffffffffu, hi, o);
  }
  return ((unsigned long long)a0_k6_mix32(hi ^ 0x5bd1e995u) << 32) | a0_k6_mix32(lo);
}

// ---- small device helpers ------------------------------------------------------------------------
__device__ __forceinline__ float a0_warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float a0_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// ---- the arg-max rule of every kernel: torch.argmax / torch.max(dim) --------------------------------------
// NaN is greater than every number; among equal maxima (+0 == -0) and among NaNs the first index wins.
// Scan form: a scan over increasing indices takes v iff a0_argmax_takes(v, best).  Starting from -inf at index 0
// is the same as starting from element 0.
__device__ __forceinline__ bool a0_argmax_takes(float v, float best) { return v > best || (v != v && best == best); }
// (v, i) comes before (w, j).  A strict total order when the indices differ, so a butterfly over it is associative and
// every lane ends with the same answer (a plain '>' is not under NaN: [1, NaN, 5, 9] left lanes 0, 1 and 2-31 with
// three different answers).
__device__ __forceinline__ bool a0_argmax_before(float v, int i, float w, int j) {
  return a0_argmax_takes(v, w) || (!a0_argmax_takes(w, v) && i < j);
}
// Scan form over N values held in registers (pad with -inf): the index a scan with a0_argmax_takes finds, computed as
// the first NaN if there is one and otherwise the first maximum by '>'.  The NaN search does not depend on the running
// maximum, so the dependent chain is a plain '>' scan's plus one select (the selection is on the K4 chains; integer
// keys ordered as the rule orders the values put their conversion on that chain instead: QR-200 at batch 512 measured
// 0.5 % slower than the parent with them, 0.25-0.3 % with this form; NVIDIA B200, 1000 W power limit).
template <int N>
__device__ __forceinline__ int a0_argmax_regs(const float (&v)[N]) {
  int a = 0, an = N;
  float best = v[0];
#pragma unroll
  for (int i = 1; i < N; ++i)
    if (v[i] > best) { best = v[i]; a = i; }
#pragma unroll
  for (int i = N - 1; i >= 0; --i)
    if (v[i] != v[i]) an = i;
  return an < N ? an : a;
}
// Warp form: the index of the maximum over the lanes' (v, i), in every lane.  Lanes without an element pass -inf
// and an index above every real one.
__device__ __forceinline__ int a0_warp_argmax(float v, int i) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oi = __shfl_xor_sync(0xffffffffu, i, o);
    if (a0_argmax_before(ov, oi, v, i)) { v = ov; i = oi; }
  }
  return i;
}
__device__ __forceinline__ float a0_huber(float x) {
  float ax = fabsf(x);
  return ax < 1.0f ? 0.5f * x * x : ax - 0.5f;
}
__device__ __forceinline__ float a0_clamp1(float x) { return fminf(fmaxf(x, -1.0f), 1.0f); }
// (loss + eps)^alpha; sqrt when alpha == 0.5, which is what torch's CPU pow does (replay.py:56-58)
__device__ __forceinline__ float a0_priority(float loss, float eps, float alpha) {
  float x = loss + eps;
  return alpha == 0.5f ? sqrtf(x) : powf(x, alpha);
}
// A priority update with a loss that is NaN, infinite or negative leaves the old leaf in place: the
// reference skips the whole update when the loss is NaN (agent.py:150-152, SURVEY Q15); inside a captured
// CUDA graph there is no host guard, and one NaN leaf would poison every ancestor up to the root.
// The write-back's max_p takes only the losses that pass this test, filtered one by one before any reduction:
// a warp maximum that met an infinite loss would otherwise be dropped whole, finite losses beside it included.
__device__ __forceinline__ bool a0_loss_ok(float x) { return x >= 0.0f && x < __int_as_float(0x7f800000); }
__device__ __forceinline__ void a0_atomic_max_pos(float* addr, float v) {
  // valid for non-negative floats: the int ordering equals the float ordering
  if (v > 0.0f && v < __int_as_float(0x7f800000)) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
}
