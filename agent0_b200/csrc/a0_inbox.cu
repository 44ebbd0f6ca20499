// K9: an inbox through which actor processes append their transitions to the learner's shard.  The reference's actor
// nodes return their transitions to the trainer node over RPC at the end of every Actor.sample
// (agent0/deepq/launch.py:45-63); here an actor in its own process (CUDA IPC, on the same GPU or a peer GPU) stores
// them into a lane of a device region the learner owns, and the learner drains the lane into its shard with the
// native ingest (K1, frames read in place from the region).
//
// The region is ONE cudaMalloc allocation, so one cudaIpcMemHandle_t covers it:
//   [0, 256)                     control block A0XCtl: magic, format, frame bytes, lanes, slots, slot capacities,
//                                streams per lane, n_gather
//   [256 + l * lane_bytes, ...)  lane l: a 512-byte header A0XLane (claimed, committed, consumed, each on its own
//                                128-byte line), then S slots of slot_bytes.
// A slot (offsets from a0x_layout; every array 16-byte aligned, capacity T transitions and SF frames):
//   [0, 256)        header: n_transitions, n_steps, n_frames (i64)
//   step_count      i64[T]  transitions of vector step k (E_k)
//   step_reset      u8[T]   1: every transition of step k starts its stream; its 4-frame stack comes first
//   stream          i64[T]  local stream id (< streams per lane)
//   n_new           i64[T]  0..4
//   action          i64[T]
//   reward          f64[T]
//   done            u8[T]
//   frames          u8[SF][F], 256-byte aligned, in allocation order: per step the reset stacks, then the new frames
// Lane words count slots: the writer has committed slots [0, committed), the learner has consumed [0, consumed);
// slot q lives at q % S.  Only the lane's writer stores `committed`, only the learner stores `consumed`.
//
// Commit (K9a, writer side, one launch, never waits): thread 0 of every CTA loads `committed` (its own word) and
// `consumed` (acquire).  A CTA that sees committed - consumed == S copies nothing and marks the launch FULL; the others
// copy their chunk of the writer's private device staging into slot committed % S with st.relaxed.sys (that slot was
// released: its reads by K1 happened before the learner's release of `consumed`).  Every thread fences
// (fence.acq_rel.sys) after its stores; the last CTA (ticket) stores committed + 1 with st.release.sys unless some CTA
// saw FULL, and writes the status into the writer's mapped host word.  A writer that dies mid-commit leaves
// `committed` unchanged: its partial slot is never seen, and the next writer of the lane overwrites it.
//
// Scan (K9b, learner side): one CTA per lane.  Thread 0 loads `committed` (acquire); the CTA copies the header and
// the used prefix of every metadata array of slots [consumed, committed) into the inbox's page-locked mapped host
// memory and records the count taken.  The frames are not copied: K1 reads them from the slot.
// Release (K9c, learner side, stream-ordered after the ingest): consumed += taken with st.release.sys.
// Nothing on the device waits for another agent; every wait is on the host and has a timeout.
#include <unistd.h>

#include <atomic>

#include "a0_common.cuh"

namespace {

constexpr uint32_t A0X_MAGIC = 0x58304130u;      // "0A0X"
constexpr uint32_t A0X_FORMAT = 1;
constexpr int A0X_THREADS = 256;
constexpr int64_t A0X_CHUNK = 64 * 1024;         // bytes per commit CTA
constexpr int32_t A0X_MAX_LANES = 1024;
constexpr int32_t A0X_MAX_SLOTS = 64;
constexpr int64_t A0X_MAX_TRANSITIONS = 1 << 20;
constexpr int64_t A0X_MAX_FRAMES = 1 << 22;
constexpr int64_t A0X_MAX_FRAME_BYTES = 1 << 20;
constexpr int32_t A0X_MAX_STREAMS = 1 << 20;
constexpr int A0X_META_SEGS = 7;                 // arrays after the slot header

struct A0XCtl {                  // 256 B at the start of the region
  uint32_t magic, format;
  uint64_t frame_bytes;
  uint32_t lanes, slots;
  uint32_t slot_transitions, slot_frames;
  uint32_t streams_per_lane, n_gather;
  uint64_t slot_bytes, lane_bytes;
  uint64_t pad[25];
};
static_assert(sizeof(A0XCtl) == 256, "control block is 256 bytes");

struct A0XLane {                 // 512 B before the lane's slots
  unsigned long long claimed;    // 0: free, else claimed by a writer
  uint64_t pad0[15];
  uint64_t committed;
  uint64_t pad1[15];
  uint64_t consumed;
  uint64_t pad2[15];
  uint64_t pad3[16];
};
static_assert(sizeof(A0XLane) == 512, "lane header is 512 bytes");

struct A0XWriter {               // writer-private device words
  uint32_t ticket, full;
  uint64_t pad[31];
};
static_assert(sizeof(A0XWriter) == 256, "writer words are 256 bytes");

struct A0XLayout {               // byte offsets inside a slot, and the region's sizes
  int64_t seg[A0X_META_SEGS];    // step_count, step_reset, stream, n_new, action, reward, done
  int64_t frames;                // = bytes of the slot's header + metadata
  int64_t slot_bytes, lane_bytes, region_bytes, scan_meta, scan_bytes;
};

__host__ __device__ __forceinline__ int64_t a0x_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

A0XLayout a0x_layout(int64_t T, int64_t SF, int64_t F, int64_t lanes, int64_t slots) {
  A0XLayout L;
  const int64_t esz[A0X_META_SEGS] = {8, 1, 8, 8, 8, 8, 1};
  int64_t at = 256;
  for (int i = 0; i < A0X_META_SEGS; ++i) {
    L.seg[i] = at;
    at += a0x_up(esz[i] * T, 16);
  }
  L.frames = a0x_up(at, 256);
  L.slot_bytes = a0x_up(L.frames + SF * F, 256);
  L.lane_bytes = (int64_t)sizeof(A0XLane) + slots * L.slot_bytes;
  L.region_bytes = (int64_t)sizeof(A0XCtl) + lanes * L.lane_bytes;
  L.scan_meta = a0x_up(lanes * 32, 256);       // per lane {consumed, committed, taken, 0}, then the metadata copies
  L.scan_bytes = L.scan_meta + lanes * slots * L.frames;
  return L;
}

// K9a.  The staging buffer has the slot's layout; bytes [256, 256 + n16 * 16) (metadata and frames) are copied, the
// header is written from the arguments.
__global__ void __launch_bounds__(A0X_THREADS) a0x_commit_kernel(A0XLane* lane, uint8_t* slot0, int64_t slot_bytes,
                                                                 uint32_t S, const uint4* __restrict__ staging,
                                                                 int64_t n16, int64_t n_transitions, int64_t n_steps,
                                                                 int64_t n_frames, A0XWriter* w,
                                                                 unsigned long long* status_out) {
  __shared__ uint64_t s_c;
  __shared__ int s_full;
  if (threadIdx.x == 0) {
    const uint64_t c = a0_sys_ld_relaxed(&lane->committed);  // this writer's own word
    const uint64_t d = a0_sys_ld_acquire(&lane->consumed);
    s_c = c;
    s_full = c - d >= (uint64_t)S;
  }
  __syncthreads();
  const uint64_t c = s_c;
  if (!s_full) {
    a0_sys_fence();                                          // the acquire above before this thread's stores
    uint8_t* slot = slot0 + (int64_t)(c % S) * slot_bytes;
    uint4* dst = reinterpret_cast<uint4*>(slot + 256);
    const int64_t g0 = (int64_t)blockIdx.x * (A0X_CHUNK / 16), g1 = min(g0 + A0X_CHUNK / 16, n16);
    for (int64_t g = g0 + threadIdx.x; g < g1; g += A0X_THREADS) a0_sys_st4_relaxed(dst + g, __ldg(staging + g));
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      uint64_t* hdr = reinterpret_cast<uint64_t*>(slot);
      a0_sys_st_relaxed(hdr + 0, (uint64_t)n_transitions);
      a0_sys_st_relaxed(hdr + 1, (uint64_t)n_steps);
      a0_sys_st_relaxed(hdr + 2, (uint64_t)n_frames);
    }
    a0_sys_fence();                                          // close: this thread's stores before the ticket
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s_full) atomicOr(&w->full, 1u);
    __threadfence();
    if (atomicAdd(&w->ticket, 1u) == gridDim.x - 1) {
      __threadfence();
      const bool full = atomicAdd(&w->full, 0u) != 0u;
      if (!full) {
        a0_sys_fence();
        a0_sys_st_release(&lane->committed, c + 1);
      }
      *reinterpret_cast<volatile unsigned long long*>(status_out) = full ? A0_TX_FULL : A0_TX_COMMITTED;
      __threadfence_system();
      w->full = 0u;
      w->ticket = 0u;
    }
  }
}

// K9b.  One CTA per lane.  scan_head: per lane {consumed, committed, taken, 0} (i64); scan_meta: per lane S entries of
// `meta_bytes` (the slot's header and metadata), entry j = slot consumed + j.
__global__ void __launch_bounds__(A0X_THREADS) a0x_scan_kernel(const uint8_t* region, int64_t lane_bytes,
                                                               int64_t slot_bytes, uint32_t S, int64_t T,
                                                               A0XLayout L, int64_t max_slots, int64_t* scan_head,
                                                               uint8_t* scan_meta, int64_t* taken) {
  const int l = blockIdx.x;
  const A0XLane* lane = reinterpret_cast<const A0XLane*>(region + sizeof(A0XCtl) + (int64_t)l * lane_bytes);
  const uint8_t* slot0 = reinterpret_cast<const uint8_t*>(lane) + sizeof(A0XLane);
  __shared__ int64_t s_n;
  __shared__ int64_t s_first;
  if (threadIdx.x == 0) {
    const uint64_t c = a0_sys_ld_acquire(&lane->committed);
    const uint64_t d = a0_sys_ld_relaxed(&lane->consumed);  // stored only by K9c on this stream
    const int64_t avail = (int64_t)(c - d);
    const int64_t n = avail < 0 ? 0 : min(min(avail, max_slots), (int64_t)S);
    s_n = n;
    s_first = (int64_t)d;
    scan_head[4 * l + 0] = (int64_t)d;
    scan_head[4 * l + 1] = (int64_t)c;
    scan_head[4 * l + 2] = n;
    scan_head[4 * l + 3] = 0;
    taken[l] = n;
  }
  __syncthreads();
  __shared__ int64_t s_cnt[2];
  for (int64_t j = 0; j < s_n; ++j) {
    const uint8_t* slot = slot0 + (int64_t)((uint64_t)(s_first + j) % S) * slot_bytes;
    uint8_t* out = scan_meta + ((int64_t)l * S + j) * L.frames;
    if (threadIdx.x == 0) {
      const uint64_t* hdr = reinterpret_cast<const uint64_t*>(slot);
      s_cnt[0] = (int64_t)min(a0_sys_ld_relaxed(hdr + 0), (uint64_t)T);  // transitions (bounded: the host validates)
      s_cnt[1] = (int64_t)min(a0_sys_ld_relaxed(hdr + 1), (uint64_t)T);  // steps
    }
    __syncthreads();
    // the header, then the used prefix of every array, 16 bytes at a time
#pragma unroll
    for (int k = -1; k < A0X_META_SEGS; ++k) {
      const int64_t esz = (k == 1 || k == 6) ? 1 : 8;      // step_reset and done are u8
      const int64_t off = k < 0 ? 0 : L.seg[k];
      const int64_t bytes = k < 0 ? 256 : a0x_up(esz * s_cnt[k < 2 ? 1 : 0], 16);
      const uint4* src = reinterpret_cast<const uint4*>(slot + off);
      uint4* dst = reinterpret_cast<uint4*>(out + off);
      for (int64_t g = threadIdx.x; g < bytes / 16; g += A0X_THREADS) dst[g] = a0_sys_ld4_relaxed(src + g);
    }
    __syncthreads();
  }
}

// K9c.  consumed += taken for every lane (stream-ordered after the ingest that read the slots' frames).
__global__ void a0x_release_kernel(uint8_t* region, int64_t lane_bytes, int32_t lanes, int64_t* taken) {
  for (int l = threadIdx.x; l < lanes; l += blockDim.x) {
    const int64_t n = taken[l];
    if (n == 0) continue;
    A0XLane* lane = reinterpret_cast<A0XLane*>(region + sizeof(A0XCtl) + (int64_t)l * lane_bytes);
    const uint64_t d = a0_sys_ld_relaxed(&lane->consumed);
    a0_sys_fence();
    a0_sys_st_release(&lane->consumed, d + (uint64_t)n);
    taken[l] = 0;
  }
}

// claimed: 0 = free, else the token of the writer that holds the lane.  A writer hands the lane back only while it
// still holds its own token, so a writer that was unclaimed (presumed dead) cannot free its successor's lane.
__global__ void a0x_claim_kernel(A0XLane* lane, unsigned long long token, unsigned long long* out) {
  *out = atomicCAS_system(&lane->claimed, 0ull, token);
  __threadfence_system();
}

__global__ void a0x_hand_back_kernel(A0XLane* lane, unsigned long long token) {
  a0_sys_fence();                                  // the writer's earlier stores before the lane is free
  atomicCAS_system(&lane->claimed, token, 0ull);
}

__global__ void a0x_unclaim_kernel(A0XLane* lane) {
  a0_sys_fence();
  a0_sys_st_release(reinterpret_cast<uint64_t*>(&lane->claimed), 0ull);
}

int a0x_check_shape(const char* who, int64_t T, int64_t SF, int64_t F) {
  A0_REQUIRE(T >= 1 && T <= A0X_MAX_TRANSITIONS, "%s: slot_transitions %lld outside [1, 2^20]", who, (long long)T);
  A0_REQUIRE(SF >= 4 && SF <= A0X_MAX_FRAMES, "%s: slot_frames %lld outside [4, 2^22]", who, (long long)SF);
  A0_REQUIRE(F >= 16 && F <= A0X_MAX_FRAME_BYTES && F % 16 == 0,
             "%s: frame_bytes %lld is not a multiple of 16 in [16, 2^20]", who, (long long)F);
  return A0_OK;
}

}  // namespace

struct a0_txbox {
  int32_t device;
  int32_t lanes, slots, streams_per_lane, n_gather;
  int64_t T, SF, F;
  A0XLayout L;
  uint8_t* region;               // A0XCtl + lanes
  uint8_t* scan_host;            // page-locked, mapped: scan head + metadata copies
  uint8_t* scan_dev;             // its device alias
  int64_t* taken;                // device [lanes]
};

struct a0_txwriter {
  int32_t device, lane;
  uint32_t slots;
  int64_t T, SF, F;
  A0XLayout L;
  uint8_t* region;               // IPC mapping or (attach) the inbox's own pointer
  bool mapped;                   // region came from a0_ipc_map
  A0XWriter* w;
  unsigned long long* claim;     // device word for the claim's result; NULL when the lane was not claimed
  unsigned long long token;      // this writer's value of `claimed`
};

extern "C" int a0_tx_layout(int64_t slot_transitions, int64_t slot_frames, int64_t frame_bytes, int32_t lanes,
                            int32_t slots, int64_t* out) {
  A0_REQUIRE(out != nullptr, "a0_tx_layout: out is NULL");
  { int rc = a0x_check_shape("a0_tx_layout", slot_transitions, slot_frames, frame_bytes); if (rc) return rc; }
  A0_REQUIRE(lanes >= 1 && lanes <= A0X_MAX_LANES, "a0_tx_layout: lanes %d outside [1, 1024]", lanes);
  A0_REQUIRE(slots >= 1 && slots <= A0X_MAX_SLOTS, "a0_tx_layout: slots %d outside [1, 64]", slots);
  const A0XLayout L = a0x_layout(slot_transitions, slot_frames, frame_bytes, lanes, slots);
  for (int i = 0; i < A0X_META_SEGS; ++i) out[i] = L.seg[i];
  out[7] = L.frames;
  out[8] = L.slot_bytes;
  out[9] = L.lane_bytes;
  out[10] = L.region_bytes;
  out[11] = L.scan_meta;
  out[12] = L.scan_bytes;
  out[13] = (int64_t)sizeof(A0XCtl);
  out[14] = (int64_t)sizeof(A0XLane);
  return A0_OK;
}

extern "C" int a0_tx_destroy(a0_txbox_t* tx) {
  if (!tx) return A0_OK;
  A0DeviceGuard guard(tx->device);
  cudaFree(tx->region);
  if (tx->scan_host) cudaFreeHost(tx->scan_host);
  cudaFree(tx->taken);
  delete tx;
  return A0_OK;
}

extern "C" int a0_tx_create(a0_txbox_t** out, int32_t lanes, int32_t slots, int64_t slot_transitions,
                            int64_t slot_frames, int64_t frame_bytes, int32_t streams_per_lane, int32_t n_gather,
                            int32_t device) {
  A0_REQUIRE(out != nullptr, "a0_tx_create: out is NULL");
  { int rc = a0x_check_shape("a0_tx_create", slot_transitions, slot_frames, frame_bytes); if (rc) return rc; }
  A0_REQUIRE(lanes >= 1 && lanes <= A0X_MAX_LANES, "a0_tx_create: lanes %d outside [1, 1024]", lanes);
  A0_REQUIRE(slots >= 1 && slots <= A0X_MAX_SLOTS, "a0_tx_create: slots %d outside [1, 64]", slots);
  A0_REQUIRE(streams_per_lane >= 1 && streams_per_lane <= A0X_MAX_STREAMS,
             "a0_tx_create: streams_per_lane %d outside [1, 2^20]", streams_per_lane);
  A0_REQUIRE(n_gather >= 1 && n_gather <= A0_MAX_NSTEP, "a0_tx_create: n_gather %d outside [1, %d]", n_gather,
             A0_MAX_NSTEP);
  A0_REQUIRE(device >= 0, "a0_tx_create: device %d is negative", device);
  A0DeviceGuard guard(device);
  const A0XLayout L = a0x_layout(slot_transitions, slot_frames, frame_bytes, lanes, slots);
  A0XCtl ctl;
  memset(&ctl, 0, sizeof(ctl));
  ctl.magic = A0X_MAGIC;
  ctl.format = A0X_FORMAT;
  ctl.frame_bytes = (uint64_t)frame_bytes;
  ctl.lanes = (uint32_t)lanes;
  ctl.slots = (uint32_t)slots;
  ctl.slot_transitions = (uint32_t)slot_transitions;
  ctl.slot_frames = (uint32_t)slot_frames;
  ctl.streams_per_lane = (uint32_t)streams_per_lane;
  ctl.n_gather = (uint32_t)n_gather;
  ctl.slot_bytes = (uint64_t)L.slot_bytes;
  ctl.lane_bytes = (uint64_t)L.lane_bytes;
  uint8_t* region = nullptr;
  { int rc = a0_ipc_create("a0_tx_create", (size_t)L.region_bytes, &ctl, sizeof(ctl), &region); if (rc) return rc; }
  a0_txbox* tx = new a0_txbox{device, lanes, slots, streams_per_lane, n_gather, slot_transitions, slot_frames,
                              frame_bytes, L, region, nullptr, nullptr, nullptr};
  cudaError_t e = cudaMalloc((void**)&tx->taken, (size_t)lanes * 8);
  if (e == cudaSuccess) e = cudaMemset(tx->taken, 0, (size_t)lanes * 8);
  if (e == cudaSuccess) e = cudaHostAlloc((void**)&tx->scan_host, (size_t)L.scan_bytes, cudaHostAllocMapped);
  if (e == cudaSuccess) e = cudaHostGetDevicePointer((void**)&tx->scan_dev, tx->scan_host, 0);
  if (e != cudaSuccess) {
    a0_tx_destroy(tx);
    a0_set_error("a0_tx_create: allocating the scan buffers failed: %s", cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? A0_ENOMEM : (int)e;
  }
  memset(tx->scan_host, 0, (size_t)L.scan_bytes);
  *out = tx;
  return A0_OK;
}

extern "C" int a0_tx_handle(a0_txbox_t* tx, uint8_t* out64) {
  A0_REQUIRE(tx != nullptr && out64 != nullptr, "a0_tx_handle: NULL argument");
  A0DeviceGuard guard(tx->device);
  return a0_ipc_handle(tx->region, out64);
}

extern "C" void* a0_tx_ctl(a0_txbox_t* tx) { return tx ? tx->region : nullptr; }

extern "C" void* a0_tx_scan_host(a0_txbox_t* tx) { return tx ? tx->scan_host : nullptr; }

extern "C" void* a0_tx_slot_frames(a0_txbox_t* tx, int32_t lane, int32_t slot) {
  if (!tx || lane < 0 || lane >= tx->lanes || slot < 0 || slot >= tx->slots) return nullptr;
  return tx->region + sizeof(A0XCtl) + (int64_t)lane * tx->L.lane_bytes + sizeof(A0XLane) +
         (int64_t)slot * tx->L.slot_bytes + tx->L.frames;
}

extern "C" int a0_tx_scan(a0_txbox_t* tx, int32_t max_slots_per_lane, a0_stream_t stream) {
  A0_REQUIRE(tx != nullptr, "a0_tx_scan: inbox is NULL");
  A0_REQUIRE(max_slots_per_lane >= 1, "a0_tx_scan: max_slots_per_lane %d is below 1", max_slots_per_lane);
  A0DeviceGuard guard(tx->device);
  a0x_scan_kernel<<<tx->lanes, A0X_THREADS, 0, (cudaStream_t)stream>>>(
      tx->region, tx->L.lane_bytes, tx->L.slot_bytes, (uint32_t)tx->slots, tx->T, tx->L,
      (int64_t)max_slots_per_lane, reinterpret_cast<int64_t*>(tx->scan_dev), tx->scan_dev + tx->L.scan_meta,
      tx->taken);
  A0_LAUNCH_CHECK();
  return A0_OK;
}

extern "C" int a0_tx_release(a0_txbox_t* tx, a0_stream_t stream) {
  A0_REQUIRE(tx != nullptr, "a0_tx_release: inbox is NULL");
  A0DeviceGuard guard(tx->device);
  a0x_release_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(tx->region, tx->L.lane_bytes, tx->lanes, tx->taken);
  A0_LAUNCH_CHECK();
  return A0_OK;
}

extern "C" int a0_tx_unclaim(a0_txbox_t* tx, int32_t lane) {
  A0_REQUIRE(tx != nullptr, "a0_tx_unclaim: inbox is NULL");
  A0_REQUIRE(lane >= 0 && lane < tx->lanes, "a0_tx_unclaim: lane %d outside [0, %d)", lane, tx->lanes);
  A0DeviceGuard guard(tx->device);
  a0x_unclaim_kernel<<<1, 1>>>(reinterpret_cast<A0XLane*>(tx->region + sizeof(A0XCtl) + (int64_t)lane * tx->L.lane_bytes));
  A0_LAUNCH_CHECK();
  A0_CUDA(cudaStreamSynchronize(nullptr));
  return A0_OK;
}

extern "C" int a0_tw_close(a0_twriter_t* tw) {
  if (!tw) return A0_OK;
  A0DeviceGuard guard(tw->device);
  if (tw->claim) {                               // the lane is handed back if this writer still holds it
    a0x_hand_back_kernel<<<1, 1>>>(
        reinterpret_cast<A0XLane*>(tw->region + sizeof(A0XCtl) + (int64_t)tw->lane * tw->L.lane_bytes), tw->token);
    cudaStreamSynchronize(nullptr);
  }
  if (tw->mapped) a0_ipc_unmap(tw->region);
  cudaFree(tw->w);
  cudaFree(tw->claim);
  delete tw;
  return A0_OK;
}

// Claims the lane (atomicCAS 0 -> 1 on `claimed`); a lane that another writer holds fails the open.
static int a0x_writer_init(a0_txwriter* tw, const char* who) {
  cudaError_t e = cudaMalloc((void**)&tw->w, sizeof(A0XWriter));
  if (e == cudaSuccess) e = cudaMalloc((void**)&tw->claim, 8);
  if (e == cudaSuccess) e = cudaMemset(tw->w, 0, sizeof(A0XWriter));
  if (e == cudaSuccess) e = cudaMemset(tw->claim, 0xff, 8);
  if (e != cudaSuccess) {
    a0_set_error("%s: allocating the writer's words failed: %s", who, cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? A0_ENOMEM : (int)e;
  }
  static std::atomic<uint32_t> serial{0};
  tw->token = ((unsigned long long)getpid() << 32) | (unsigned long long)(++serial);
  a0x_claim_kernel<<<1, 1>>>(reinterpret_cast<A0XLane*>(tw->region + sizeof(A0XCtl) + (int64_t)tw->lane * tw->L.lane_bytes),
                             tw->token, tw->claim);
  A0_LAUNCH_CHECK();
  unsigned long long was = 1ull;
  A0_CUDA(cudaMemcpy(&was, tw->claim, 8, cudaMemcpyDeviceToHost));
  if (was != 0ull) {
    cudaFree(tw->claim);
    tw->claim = nullptr;                          // not ours: close must not hand it back
    a0_set_error("%s: lane %d is claimed by another writer (a0_tx_unclaim hands the lane of a dead one on)", who, tw->lane);
    return A0_EINVAL;
  }
  return A0_OK;
}

// A writer of lane `lane` of `region` (mapped: closing it unmaps the region); what is taken is given back on failure.
static int a0x_writer_new(a0_twriter_t** out, const char* who, int32_t device, int32_t lane, uint32_t slots, int64_t T,
                          int64_t SF, int64_t F, const A0XLayout& L, uint8_t* region, bool mapped) {
  a0_txwriter* tw = new a0_txwriter{device, lane, slots, T, SF, F, L, region, mapped, nullptr, nullptr, 0};
  const int rc = a0x_writer_init(tw, who);
  if (rc != A0_OK) { a0_tw_close(tw); return rc; }
  *out = tw;
  return A0_OK;
}

extern "C" int a0_tw_open(a0_twriter_t** out, const uint8_t* handle64, int32_t lane, int64_t frame_bytes,
                          int64_t slot_transitions, int64_t slot_frames, int32_t device) {
  A0_REQUIRE(out != nullptr && handle64 != nullptr, "a0_tw_open: NULL argument");
  { int rc = a0x_check_shape("a0_tw_open", slot_transitions, slot_frames, frame_bytes); if (rc) return rc; }
  A0_REQUIRE(lane >= 0, "a0_tw_open: lane %d is negative", lane);
  A0_REQUIRE(device >= 0, "a0_tw_open: device %d is negative", device);
  A0DeviceGuard guard(device);
  A0XCtl ctl;
  uint8_t* region = nullptr;
  const int rc = a0_ipc_map("a0_tw_open", handle64, A0X_MAGIC, A0X_FORMAT, "transition inbox's", &ctl, sizeof(ctl), &region);
  if (rc != A0_OK) return rc;
  const A0XLayout L = a0x_layout(slot_transitions, slot_frames, frame_bytes, ctl.lanes, ctl.slots);
  const char* bad = ctl.frame_bytes != (uint64_t)frame_bytes ? "holds frames of another size"
                    : ctl.slot_transitions != (uint64_t)slot_transitions || ctl.slot_frames != (uint64_t)slot_frames ||
                            ctl.slot_bytes != (uint64_t)L.slot_bytes || ctl.lane_bytes != (uint64_t)L.lane_bytes
                        ? "has slots of another layout"
                    : lane >= (int32_t)ctl.lanes ? "has fewer lanes"
                                                 : nullptr;
  if (bad) {
    a0_ipc_unmap(region);
    a0_set_error("a0_tw_open: the handle's region %s (frame bytes %llu vs %lld, slot %u x %u vs %lld x %lld, lane %d of %u)",
                 bad, (unsigned long long)ctl.frame_bytes, (long long)frame_bytes, ctl.slot_transitions, ctl.slot_frames,
                 (long long)slot_transitions, (long long)slot_frames, lane, ctl.lanes);
    return A0_EINVAL;
  }
  return a0x_writer_new(out, "a0_tw_open", device, lane, ctl.slots, slot_transitions, slot_frames, frame_bytes, L,
                        region, true);
}

extern "C" int a0_tw_attach(a0_twriter_t** out, a0_txbox_t* tx, int32_t lane) {
  A0_REQUIRE(out != nullptr && tx != nullptr, "a0_tw_attach: NULL argument");
  A0_REQUIRE(lane >= 0 && lane < tx->lanes, "a0_tw_attach: lane %d outside [0, %d)", lane, tx->lanes);
  A0DeviceGuard guard(tx->device);
  return a0x_writer_new(out, "a0_tw_attach", tx->device, lane, (uint32_t)tx->slots, tx->T, tx->SF, tx->F, tx->L,
                        tx->region, false);
}

extern "C" int a0_tw_commit(a0_twriter_t* tw, const uint8_t* staging_dev, int64_t n_transitions, int64_t n_steps,
                            int64_t n_frames, uint64_t* status_out, a0_stream_t stream) {
  A0_REQUIRE(tw != nullptr, "a0_tw_commit: writer is NULL");
  A0_REQUIRE(staging_dev != nullptr && status_out != nullptr, "a0_tw_commit: NULL staging or status");
  A0_REQUIRE(((uintptr_t)staging_dev & 15) == 0, "a0_tw_commit: the staging buffer must be 16-byte aligned");
  A0_REQUIRE(n_transitions >= 1 && n_transitions <= tw->T, "a0_tw_commit: n_transitions %lld outside [1, %lld]",
             (long long)n_transitions, (long long)tw->T);
  A0_REQUIRE(n_steps >= 1 && n_steps <= n_transitions, "a0_tw_commit: n_steps %lld outside [1, %lld]",
             (long long)n_steps, (long long)n_transitions);
  A0_REQUIRE(n_frames >= 0 && n_frames <= tw->SF, "a0_tw_commit: n_frames %lld outside [0, %lld]", (long long)n_frames,
             (long long)tw->SF);
  A0DeviceGuard guard(tw->device);
  const int64_t n16 = (tw->L.frames - 256 + n_frames * tw->F) / 16;
  const unsigned grid = (unsigned)((n16 * 16 + A0X_CHUNK - 1) / A0X_CHUNK);
  A0XLane* lane = reinterpret_cast<A0XLane*>(tw->region + sizeof(A0XCtl) + (int64_t)tw->lane * tw->L.lane_bytes);
  a0x_commit_kernel<<<grid, A0X_THREADS, 0, (cudaStream_t)stream>>>(
      lane, reinterpret_cast<uint8_t*>(lane) + sizeof(A0XLane), tw->L.slot_bytes, tw->slots,
      reinterpret_cast<const uint4*>(staging_dev + 256), n16, n_transitions, n_steps, n_frames, tw->w,
      reinterpret_cast<unsigned long long*>(status_out));
  A0_LAUNCH_CHECK();
  return A0_OK;
}
