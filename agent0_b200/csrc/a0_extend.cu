// K6: the reference-shaped ingest -- ReplayDataset.extend(list of (lz4 blob, a, r, d)) -- on the device.
//
// The reference's actor ships every transition as one python-lz4 block of concat(st, st_next), 8 frames =
// 56 448 B decoded (agent0/deepq/agent.py:78-81), and ReplayDataset.extend appends the blobs to a host deque
// (agent0/deepq/replay.py:45-53).  The shard stores single frames, so the drop-in has to decode the blocks
// and find out which of their frames it already holds.  Doing that on the host cost 20-28 ms per
// Trainer.step-sized call (1280 entries: liblz4 decode 16 ms, hash + memcmp 13 ms, 72 MB staged and copied).
// Here only the COMPRESSED bytes cross PCIe (~1 KB per entry for Atari-like frames) and the device does the
// byte work:
//
//   a0_k6_lz4_decode   one warp per entry: LZ4 block format decoded into shared memory (the 64 KB match
//                      window of the format is the entry itself, so every match is a shared-memory copy),
//                      a 64-bit hash per frame while the bytes are on chip, then ONE cp.async.bulk store of
//                      the 56 KB entry into a scratch buffer in HBM.
//   a0_k6_label        one CTA per entry, one warp per frame: the frame's canonical label = the first of
//                      {the 8 frames of the stream's previous entry, the earlier frames of its own entry}
//                      that is byte-identical (hash gate, then a full 16-byte-vector compare), else itself.
//   (host)             8 label bytes per entry come back; the host applies the residency / age rules of the
//                      ring index to them (a0_ex_resolve: the same decisions as a0_dd_resolve, which stays
//                      as the host specification) and plans the append;
//   K2b marks + K1     the append reads the new frames straight out of the scratch buffer (src_idx).
//   a0_k6_tails        keeps each stream's last entry (frames + hashes) for the next call.
//
// LZ4 block format (lz4 >= 4.3.3 is the reference's pinned dependency, pyproject.toml:14; the package is
// not part of /root/reference): python-lz4's block.compress prefixes a 4-byte little-endian decoded size;
// then sequences {token: literal length << 4 | match length - 4; length extension bytes (+255 ...);
// literals; 2-byte little-endian offset; match length extension}; the last sequence ends after its literals.
// oracle/lz4_block.py restates the decoder and is pinned to the system liblz4.
#include <stdlib.h>

#include <algorithm>
#include <chrono>
#include <new>
#include <unordered_map>
#include <vector>

#include "a0_common.cuh"

struct __align__(16) A0ExDesc {
  long long off;     // byte offset of the blob in the staged block (16-byte aligned)
  int32_t len;       // blob bytes; == 8 * F: a raw (uncompressed) entry
  int32_t prev;      // >= 0: previous entry of the same stream in this batch; -1: none; <= -2: tail slot -2 - prev
};

enum { A0_LZ_OK = 0, A0_LZ_BAD_SIZE = 1, A0_LZ_INPUT_OVERRUN = 2, A0_LZ_OUTPUT_OVERRUN = 3, A0_LZ_BAD_OFFSET = 4,
       A0_LZ_SHORT_OUTPUT = 5 };

// ------------------------------------------------------------------------------------------------
// device: copies inside one warp.  The decoded entry lives in the CTA's dynamic shared memory; the
// helpers index the array directly (a pointer parameter made the compiler rebuild the generic->shared
// address inside every loop iteration: S2R SR_CgaCtaId + LEA per byte, ncu source view).
// ------------------------------------------------------------------------------------------------
extern __shared__ __align__(128) uint8_t a0_k6_out[];
// K6_AT(i): byte i of the entry being decoded -- in the CTA's shared memory (GLOBAL = false, the default kernel) or
// straight in the scratch buffer in HBM/L2 (GLOBAL = true, the all-entries-resident variant below)
#define K6_AT(i) (*(GLOBAL ? gout + (i) : a0_k6_out + (i)))
#define K6_PTR(i) (GLOBAL ? gout + (i) : a0_k6_out + (i))

// `len` literal bytes from the compressed stream (global memory, any alignment) to out[op..]
template <bool GLOBAL>
__device__ __forceinline__ void a0_k6_copy_in(uint8_t* gout, int op, const uint8_t* __restrict__ src, int len, int lane) {
  if (len < 128) {
#pragma unroll 2
    for (int i = lane; i < len; i += 32) K6_AT(op + i) = src[i];
    return;
  }
  // destination-aligned 32-bit words; a source word is assembled from two aligned loads
  const int head = (4 - (op & 3)) & 3;
  if (lane < head) K6_AT(op + lane) = src[lane];
  const uint8_t* s2 = src + head;
  const int d2 = op + head, rem = len - head, nw = rem >> 2;
  const uintptr_t sa = (uintptr_t)s2;
  const uint32_t sh = (uint32_t)(sa & 3) * 8;
  const uint32_t* __restrict__ sw = reinterpret_cast<const uint32_t*>(sa & ~(uintptr_t)3);
  uint32_t* dw = reinterpret_cast<uint32_t*>(K6_PTR(d2));
  if (sh == 0) {
#pragma unroll 4
    for (int k = lane; k < nw; k += 32) dw[k] = sw[k];
  } else {
#pragma unroll 4
    for (int k = lane; k < nw; k += 32) dw[k] = __funnelshift_r(sw[k], sw[k + 1], sh);
  }
  const int tail = rem & 3;
  if (lane < tail) K6_AT(d2 + 4 * nw + lane) = s2[4 * nw + lane];
}

// LZ4 match: `ml` bytes from out[op - off ..] to out[op ..]; the ranges overlap when off < ml (the
// copy then repeats the last `off` bytes).  Everything before `op` is visible (the caller synchronised).
template <bool GLOBAL>
__device__ __forceinline__ void a0_k6_copy_match(uint8_t* gout, int op, int off, int ml, int lane) {
  const int sp = op - off;
  if (off >= ml) {
    // disjoint ranges: no ordering needed between iterations
    if (ml < 128) {
#pragma unroll 2
      for (int i = lane; i < ml; i += 32) K6_AT(op + i) = K6_AT(sp + i);
      return;
    }
    const int head = (4 - (op & 3)) & 3;
    if (lane < head) K6_AT(op + lane) = K6_AT(sp + lane);
    const int d2 = op + head, s2 = sp + head, rem = ml - head, nw = rem >> 2;
    const uint32_t sh = (uint32_t)(s2 & 3) * 8;
    const uint32_t* sw = reinterpret_cast<const uint32_t*>(K6_PTR((s2 & ~3)));
    uint32_t* dw = reinterpret_cast<uint32_t*>(K6_PTR(d2));
    // with sh != 0 the second source word of the last destination words may already be destination (off >= ml
    // only keeps the bytes that are USED in front of op): the bytes taken from it lie before op, the rest of
    // the word is shifted out, so reading it early or late is harmless
    if (sh == 0) {
#pragma unroll 4
      for (int k = lane; k < nw; k += 32) dw[k] = sw[k];
    } else {
#pragma unroll 2
      for (int k = lane; k < nw; k += 32) {
        const uint32_t lo = sw[k], hi = sw[k + 1];
        dw[k] = __funnelshift_r(lo, hi, sh);
      }
    }
    const int tail = rem & 3;
    if (lane < tail) K6_AT(d2 + 4 * nw + lane) = K6_AT(s2 + 4 * nw + lane);
    return;
  }
  // Overlapping match: the output repeats the `off` bytes in front of op, which are complete, so byte i
  // comes from out[sp + i mod off] and NO iteration depends on another (copying "what earlier iterations
  // wrote" needed a warp barrier per 32 bytes: 13 instructions per iteration, 16 % of the kernel on
  // Atari-like frames whose rows repeat with period 84).
  if (ml >= 32 && (off == 1 || off == 2 || off == 4)) {
    const int head = (4 - (op & 3)) & 3;
    uint32_t w = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) w |= (uint32_t)K6_AT(sp + ((head + q) & (off - 1))) << (8 * q);
    const int d2 = op + head, rem = ml - head, nw = rem >> 2;
    const int tail = rem & 3;
    if (lane < head) K6_AT(op + lane) = (uint8_t)(w >> (8 * ((lane + 4 - head) & 3)));
    uint32_t* dw = reinterpret_cast<uint32_t*>(K6_PTR(d2));
#pragma unroll 4
    for (int k = lane; k < nw; k += 32) dw[k] = w;
    if (lane < tail) K6_AT(d2 + 4 * nw + lane) = (uint8_t)(w >> (8 * lane));
    return;
  }
  int s, step;
  if (off >= 32) { s = lane; step = 32; if (step >= off) step -= off; }
  else { s = lane % off; step = 32 % off; }
#pragma unroll 4
  for (int i = lane; i < ml; i += 32) {
    K6_AT(op + i) = K6_AT(sp + s);
    s += step;
    if (s >= off) s -= off;
  }
}

// ------------------------------------------------------------------------------------------------
// K6a: LZ4 block decode, one warp per reference entry
// ------------------------------------------------------------------------------------------------
// GLOBAL = false (default): the entry is decoded in shared memory and leaves as one bulk copy.  GLOBAL = true
// (A0_OPT_K6_GLOBAL): it is decoded in place in the scratch buffer -- matches read back what the warp just wrote,
// through L1/L2 -- which needs no shared memory, so ALL entries of a call are resident at once (8-9 warps per SM
// instead of 4) at the price of a longer round trip per match.
template <bool GLOBAL>
__global__ void __launch_bounds__(32)
a0_k6_lz4_decode_t(const uint8_t* __restrict__ comp, const A0ExDesc* __restrict__ desc, int32_t F, uint8_t* __restrict__ dec,
                   unsigned long long* __restrict__ hash, int32_t* __restrict__ status) {
  const int t = blockIdx.x, lane = threadIdx.x;
  const A0ExDesc d = desc[t];
  const uint8_t* __restrict__ in = comp + d.off;
  const int n = d.len, total = A0_SLOTS * F;
  uint8_t* gout = dec + (size_t)t * total;
  int err = A0_LZ_OK;
  if (n == total) {
    // raw entry (ndarray / bytes of the decoded size): blob starts are 16-byte aligned in the staged block
    const uint4* s = reinterpret_cast<const uint4*>(in);
    uint4* o = reinterpret_cast<uint4*>(K6_PTR(0));
#pragma unroll 4
    for (int i = lane; i < (total >> 4); i += 32) o[i] = __ldg(s + i);
  } else {
    // pull the compressed block towards the SM: one 128-byte line per lane and round
#pragma unroll 1
    for (int o = lane * 128; o < n; o += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(in + o));
    if (n < 5) err = A0_LZ_BAD_SIZE;
    else {
      const uint32_t size = (uint32_t)in[0] | ((uint32_t)in[1] << 8) | ((uint32_t)in[2] << 16) | ((uint32_t)in[3] << 24);
      if (size != (uint32_t)total) err = A0_LZ_BAD_SIZE;
    }
    int ip = 4, op = 0;
#pragma unroll 1
    while (err == A0_LZ_OK) {
      if (ip >= n) { err = A0_LZ_INPUT_OVERRUN; break; }
      const uint32_t tok = in[ip++];
      int ll = (int)(tok >> 4);
      if (ll == 15) {
        uint32_t x;
        do {
          if (ip >= n) { err = A0_LZ_INPUT_OVERRUN; break; }
          x = in[ip++];
          ll += (int)x;
        } while (x == 255u);
        if (err) break;
      }
      if (ll > 0) {
        if (ll > n - ip) { err = A0_LZ_INPUT_OVERRUN; break; }
        if (ll > total - op) { err = A0_LZ_OUTPUT_OVERRUN; break; }
        a0_k6_copy_in<GLOBAL>(gout, op, in + ip, ll, lane);
        ip += ll;
        op += ll;
      }
      if (ip >= n) break;                        // the last sequence ends after its literals
      if (n - ip < 2) { err = A0_LZ_INPUT_OVERRUN; break; }
      const int off = (int)in[ip] | ((int)in[ip + 1] << 8);
      ip += 2;
      int ml = (int)(tok & 15u);
      if (ml == 15) {
        uint32_t x;
        do {
          if (ip >= n) { err = A0_LZ_INPUT_OVERRUN; break; }
          x = in[ip++];
          ml += (int)x;
        } while (x == 255u);
        if (err) break;
      }
      ml += 4;
      if (off == 0 || off > op) { err = A0_LZ_BAD_OFFSET; break; }
      if (ml > total - op) { err = A0_LZ_OUTPUT_OVERRUN; break; }
      __syncwarp();                              // everything written so far is visible to every lane
      a0_k6_copy_match<GLOBAL>(gout, op, off, ml, lane);
      op += ml;
    }
    if (err == A0_LZ_OK && op != total) err = A0_LZ_SHORT_OUTPUT;
  }
  __syncwarp();
  if (lane == 0) status[t] = err;
  const int nvec = F >> 4;
#pragma unroll 1
  for (int f = 0; f < A0_SLOTS; ++f) {
    const unsigned long long h = a0_k6_frame_hash(K6_PTR((size_t)f * F), nvec, lane);
    if (lane == 0) hash[(size_t)t * A0_SLOTS + f] = h;
  }
  if (GLOBAL) return;                              // decoded in place
  // the whole entry leaves the SM as one bulk copy (shared -> global through the async proxy)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncwarp();
  if (lane == 0) {
    a0_bulk_store(gout, a0_smem_u32(a0_k6_out), (uint32_t)total);
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
  }
}


// ------------------------------------------------------------------------------------------------
// K6b: canonical labels.  label[t][j] in 0..7: frame j equals frame `label` of the previous entry of its
// stream; 8..15: equals frame label-8 of its own entry (8+j: a frame seen for the first time).  The label
// is the FIRST byte-identical candidate in that order, so two frames are identical iff their labels are.
// ------------------------------------------------------------------------------------------------
constexpr int K6L_THREADS = 32 * A0_SLOTS;
__global__ void __launch_bounds__(K6L_THREADS)
a0_k6_label(const uint8_t* __restrict__ dec, const unsigned long long* __restrict__ hash, const A0ExDesc* __restrict__ desc,
            int32_t F, const uint8_t* __restrict__ tail_frames, const unsigned long long* __restrict__ tail_hash,
            uint8_t* __restrict__ label) {
  const int t = blockIdx.x, j = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t entry = (size_t)A0_SLOTS * F;
  const int prev = desc[t].prev;
  const uint8_t* pf = nullptr;
  const unsigned long long* ph = nullptr;
  if (prev >= 0) { pf = dec + (size_t)prev * entry; ph = hash + (size_t)prev * A0_SLOTS; }
  else if (prev <= -2) { pf = tail_frames + (size_t)(-2 - prev) * entry; ph = tail_hash + (size_t)(-2 - prev) * A0_SLOTS; }
  const unsigned long long* mh = hash + (size_t)t * A0_SLOTS;
  const unsigned long long hj = mh[j];
  bool cand = false;
  if (lane < A0_SLOTS) cand = ph != nullptr && ph[lane] == hj;
  else if (lane < A0_SLOTS + j) cand = mh[lane - A0_SLOTS] == hj;
  unsigned mask = __ballot_sync(0xffffffffu, cand);
  int lab = A0_SLOTS + j;
  const uint4* mine = reinterpret_cast<const uint4*>(dec + (size_t)t * entry + (size_t)j * F);
  const int nvec = F >> 4;
  while (mask) {
    const int x = __ffs(mask) - 1;
    mask &= mask - 1;
    const uint4* other = reinterpret_cast<const uint4*>(x < A0_SLOTS ? pf + (size_t)x * F
                                                                      : dec + (size_t)t * entry + (size_t)(x - A0_SLOTS) * F);
    bool eq = true;
#pragma unroll 2
    for (int i = lane; i < nvec; i += 32) {
      const uint4 a = mine[i], b = other[i];
      eq = eq && a.x == b.x && a.y == b.y && a.z == b.z && a.w == b.w;
    }
    if (__all_sync(0xffffffffu, eq)) { lab = x; break; }
  }
  if (lane == 0) label[(size_t)t * A0_SLOTS + j] = (uint8_t)lab;
}

// K6c: each touched stream's last entry of the call becomes its tail (frames + hashes)
__global__ void __launch_bounds__(128)
a0_k6_tails(const uint8_t* __restrict__ dec, const unsigned long long* __restrict__ hash, const int32_t* __restrict__ src_entry,
            const int32_t* __restrict__ slot, int32_t F, uint8_t* __restrict__ tail_frames,
            unsigned long long* __restrict__ tail_hash) {
  const int b = blockIdx.x, f = blockIdx.y;
  const size_t entry = (size_t)A0_SLOTS * F;
  const uint4* s = reinterpret_cast<const uint4*>(dec + (size_t)src_entry[b] * entry + (size_t)f * F);
  uint4* o = reinterpret_cast<uint4*>(tail_frames + (size_t)slot[b] * entry + (size_t)f * F);
  for (int i = threadIdx.x; i < (F >> 4); i += 128) o[i] = s[i];
  if (threadIdx.x == 0) tail_hash[(size_t)slot[b] * A0_SLOTS + f] = hash[(size_t)src_entry[b] * A0_SLOTS + f];
}

// ------------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------------
struct A0ExTail {
  int64_t seq[A0_SLOTS];      // frame sequence numbers of the stream's last entry
  uint8_t cls[A0_SLOTS];      // its labels: two of its frames are identical iff their labels are
  int32_t slot = -1;          // device tail slot
  bool valid = false;
};

struct a0_extend {
  a0_replay* h;
  a0_index* ix;
  int32_t F = 0;
  std::unordered_map<int64_t, A0ExTail> tail;
  int32_t n_slots = 0, slot_cap = 0;
  uint8_t* d_tail_frames = nullptr;
  unsigned long long* d_tail_hash = nullptr;
  int32_t cap = 0;                       // entries the per-batch buffers hold
  uint8_t* d_dec = nullptr;              // [cap][8][F]
  unsigned long long* d_hash = nullptr;  // [cap][8]
  uint8_t* d_back = nullptr;             // [cap][8] labels, then [cap] int32 status
  uint8_t* h_back = nullptr;             // page-locked mirror
  size_t stage_cap = 0;
  uint8_t* h_stage = nullptr;            // page-locked: descriptors, tail lists, compressed blobs
  uint8_t* d_stage = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::vector<int64_t> fs8, new_src;
  std::vector<int32_t> tail_src, tail_slot;
  float timing[6] = {0, 0, 0, 0, 0, 0};  // last call, microseconds: stage, wait (decode+label on the device), resolve+plan,
                                         // launches, device decode+label (CUDA events), entries
};

static int g_k6_global = -1;
static bool a0_option_k6_global() {
  if (g_k6_global < 0) {
    const char* e = getenv("A0_K6_GLOBAL");
    g_k6_global = e ? (atoi(e) != 0) : 0;
  }
  return g_k6_global != 0;
}
void a0_set_k6_global(int on) { g_k6_global = on != 0; }

constexpr int32_t A0_EX_BATCH = 2048;    // entries decoded per round (scratch: 2048 * 56 448 B = 116 MB)

extern "C" int a0_ex_create(a0_extend_t** out, a0_replay_t* h, a0_index_t* ix) {
  A0_REQUIRE(out && ix, "a0_ex_create: NULL argument");
  a0_extend* ex = new (std::nothrow) a0_extend();
  if (!ex) { a0_set_error("a0_ex_create: out of host memory"); return A0_ENOMEM; }
  ex->h = h;
  ex->ix = ix;
  ex->F = h ? h->F : 0;
  *out = ex;
  return A0_OK;
}

extern "C" int a0_ex_destroy(a0_extend_t* ex) {
  if (!ex) return A0_OK;
  if (ex->h) {
    A0DeviceGuard guard(ex->h->device);
    cudaFree(ex->d_tail_frames); cudaFree(ex->d_tail_hash); cudaFree(ex->d_dec); cudaFree(ex->d_hash);
    cudaFree(ex->d_back); cudaFree(ex->d_stage);
    if (ex->h_back) cudaFreeHost(ex->h_back);
    if (ex->h_stage) cudaFreeHost(ex->h_stage);
    if (ex->ev0) cudaEventDestroy(ex->ev0);
    if (ex->ev1) cudaEventDestroy(ex->ev1);
  }
  delete ex;
  return A0_OK;
}

// The decisions of a0_dd_resolve taken from labels instead of bytes.  Reads the index's head_fs /
// capacity / age limit as they are NOW, i.e. it resolves one chunk that a0_ix_plan commits next.
extern "C" int a0_ex_resolve(a0_extend_t* ex, const int64_t* stream, const uint8_t* labels, int32_t m, int64_t* fs8_out,
                             int64_t* new_src_out, int32_t* n_new_out) {
  A0_REQUIRE(ex && n_new_out, "a0_ex_resolve: NULL handle");
  A0_REQUIRE(m >= 0, "a0_ex_resolve: negative count");
  A0_REQUIRE(m == 0 || (stream && labels && fs8_out && new_src_out), "a0_ex_resolve: NULL array");
  int64_t st[A0_IX_STATE_WORDS];
  int rc = a0_ix_state(ex->ix, st);
  if (rc) return rc;
  const int64_t head_fs = st[A0_IX_HEAD_FS], NF = st[A0_IX_FRAME_CAPACITY], age_limit = st[A0_IX_AGE_LIMIT];
  int64_t next_fs = head_fs;
  const int64_t resident_from = head_fs - NF;
  int32_t n_new = 0;
  for (int32_t t = 0; t < m; ++t) {
    A0ExTail& tl = ex->tail[stream[t]];
    const uint8_t* lab = labels + (size_t)t * A0_SLOTS;
    int64_t* row = fs8_out + (size_t)t * A0_SLOTS;
    uint8_t pc[A0_SLOTS];                  // canonical (smallest identical) frame of the previous entry
    if (tl.valid) {
      for (int c = 0; c < A0_SLOTS; ++c) {
        pc[c] = (uint8_t)c;
        for (int e = 0; e < c; ++e)
          if (tl.cls[e] == tl.cls[c]) { pc[c] = (uint8_t)e; break; }
      }
    }
    for (int j = 0; j < A0_SLOTS; ++j) {
      A0_REQUIRE(lab[j] < 2 * A0_SLOTS && (lab[j] < A0_SLOTS ? tl.valid : lab[j] <= A0_SLOTS + j),
                 "a0_ex_resolve: label %d of entry %d frame %d is not a valid candidate", (int)lab[j], t, j);
      int64_t hit = -1;
      if (tl.valid && lab[j] < A0_SLOTS) {
        for (int c = 0; c < A0_SLOTS && hit < 0; ++c)
          if (pc[c] == lab[j] && next_fs - tl.seq[c] < age_limit && tl.seq[c] >= resident_from) hit = tl.seq[c];
      }
      for (int c = 0; c < j && hit < 0; ++c)
        if (lab[c] == lab[j]) hit = row[c];
      if (hit < 0) {
        hit = next_fs++;
        new_src_out[n_new++] = (int64_t)t * A0_SLOTS + j;
      }
      row[j] = hit;
    }
    for (int j = 0; j < A0_SLOTS; ++j) { tl.seq[j] = row[j]; tl.cls[j] = lab[j]; }
    tl.valid = true;
  }
  *n_new_out = n_new;
  return A0_OK;
}

static inline size_t a0_ex_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static int a0_ex_reserve(a0_extend* ex, int32_t mb, size_t stage_bytes, int32_t streams_needed) {
  const size_t entry = (size_t)A0_SLOTS * ex->F;
  if (!ex->ev0) {
    A0_CUDA(cudaEventCreate(&ex->ev0));
    A0_CUDA(cudaEventCreate(&ex->ev1));
  }
  if (ex->cap < mb) {
    const int32_t cap = (int32_t)std::min<int64_t>(A0_EX_BATCH, a0_ex_up((size_t)mb, 256));
    A0_CUDA(cudaDeviceSynchronize());
    cudaFree(ex->d_dec); cudaFree(ex->d_hash); cudaFree(ex->d_back);
    if (ex->h_back) cudaFreeHost(ex->h_back);
    ex->d_dec = nullptr; ex->d_hash = nullptr; ex->d_back = nullptr; ex->h_back = nullptr; ex->cap = 0;
    A0_CUDA(cudaMalloc((void**)&ex->d_dec, (size_t)cap * entry));
    A0_CUDA(cudaMalloc((void**)&ex->d_hash, (size_t)cap * A0_SLOTS * sizeof(unsigned long long)));
    A0_CUDA(cudaMalloc((void**)&ex->d_back, (size_t)cap * (A0_SLOTS + 4)));
    A0_CUDA(cudaMallocHost((void**)&ex->h_back, (size_t)cap * (A0_SLOTS + 4)));
    ex->cap = cap;
  }
  if (ex->stage_cap < stage_bytes) {
    const size_t cap = std::max<size_t>(stage_bytes + stage_bytes / 2, (size_t)4 << 20);
    A0_CUDA(cudaDeviceSynchronize());
    if (ex->h_stage) cudaFreeHost(ex->h_stage);
    cudaFree(ex->d_stage);
    ex->h_stage = nullptr; ex->d_stage = nullptr; ex->stage_cap = 0;
    A0_CUDA(cudaMallocHost((void**)&ex->h_stage, cap));
    A0_CUDA(cudaMalloc((void**)&ex->d_stage, cap));
    ex->stage_cap = cap;
  }
  if (ex->slot_cap < streams_needed) {
    const int32_t cap = std::max<int32_t>(64, 2 * streams_needed);
    uint8_t* nf = nullptr;
    unsigned long long* nh = nullptr;
    A0_CUDA(cudaMalloc((void**)&nf, (size_t)cap * entry));
    A0_CUDA(cudaMalloc((void**)&nh, (size_t)cap * A0_SLOTS * sizeof(unsigned long long)));
    A0_CUDA(cudaDeviceSynchronize());
    if (ex->n_slots) {
      A0_CUDA(cudaMemcpy(nf, ex->d_tail_frames, (size_t)ex->n_slots * entry, cudaMemcpyDeviceToDevice));
      A0_CUDA(cudaMemcpy(nh, ex->d_tail_hash, (size_t)ex->n_slots * A0_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToDevice));
    }
    cudaFree(ex->d_tail_frames); cudaFree(ex->d_tail_hash);
    ex->d_tail_frames = nf; ex->d_tail_hash = nh; ex->slot_cap = cap;
  }
  int dev = 0;
  A0_CUDA(cudaGetDevice(&dev));
  return a0_smem_at_least((const void*)a0_k6_lz4_decode_t<false>, dev, entry, true);
}

// Stages mb blobs (16-byte aligned each) behind their descriptors and launches the decode.
// Layout of the staged block: [desc mb*16][tail_src 4*mb][tail_slot 4*mb][blobs ...]
struct A0ExLayout { size_t desc, tsrc, tslot, blobs, end; };
static A0ExLayout a0_ex_layout(int32_t mb, const int64_t* blob_len) {
  A0ExLayout L;
  L.desc = 0;
  L.tsrc = a0_ex_up((size_t)mb * sizeof(A0ExDesc), 256);
  L.tslot = L.tsrc + a0_ex_up((size_t)mb * 4, 256);
  L.blobs = L.tslot + a0_ex_up((size_t)mb * 4, 256);
  size_t e = L.blobs;
  for (int32_t i = 0; i < mb; ++i) e += a0_ex_up((size_t)blob_len[i], 16);
  L.end = e + 64;                         // slack: the word copies may read up to 3 bytes past a literal run
  return L;
}

static const char* a0_lz_error(int code) {
  switch (code) {
    case A0_LZ_BAD_SIZE: return "size prefix does not match 8 frames";
    case A0_LZ_INPUT_OVERRUN: return "compressed block is truncated";
    case A0_LZ_OUTPUT_OVERRUN: return "block decodes to more than 8 frames";
    case A0_LZ_BAD_OFFSET: return "match offset points before the start of the block";
    case A0_LZ_SHORT_OUTPUT: return "block decodes to fewer than 8 frames";
    default: return "unknown";
  }
}

using a0_clock = std::chrono::steady_clock;
static inline float a0_us(a0_clock::time_point a, a0_clock::time_point b) {
  return std::chrono::duration<float, std::micro>(b - a).count();
}

// decode (+ label when `with_labels`) of one batch; on return the labels and statuses are on the host
static int a0_ex_run_batch(a0_extend* ex, const uint8_t* blobs, const uint8_t* const* blob_ptr, const int64_t* blob_len,
                           const int64_t* stream, int32_t mb, bool with_labels, cudaStream_t cs, const char* who) {
  const size_t entry = (size_t)A0_SLOTS * ex->F;
  for (int32_t i = 0; i < mb; ++i)
    A0_REQUIRE(blob_len[i] > 0 && blob_len[i] <= (int64_t)entry + entry / 255 + 64,
               "%s: entry %d has %lld bytes (a python-lz4 block of 8 frames has at most %lld)", who, i, (long long)blob_len[i],
               (long long)(entry + entry / 255 + 64));
  const auto t0 = a0_clock::now();
  const A0ExLayout L = a0_ex_layout(mb, blob_len);
  // tail slots for streams seen for the first time
  int32_t need = ex->n_slots;
  if (with_labels)
    for (int32_t i = 0; i < mb; ++i) {
      A0ExTail& tl = ex->tail[stream[i]];
      if (tl.slot < 0) tl.slot = need++;
    }
  int rc = a0_ex_reserve(ex, mb, L.end, need);
  if (rc) return rc;
  ex->n_slots = need;
  A0ExDesc* desc = reinterpret_cast<A0ExDesc*>(ex->h_stage + L.desc);
  size_t off = L.blobs;
  const uint8_t* src = blobs;
  std::unordered_map<int64_t, int32_t> last;      // stream -> its latest entry in this batch
  for (int32_t i = 0; i < mb; ++i) {
    const size_t len = (size_t)blob_len[i];
    memcpy(ex->h_stage + off, blob_ptr ? blob_ptr[i] : src, len);
    desc[i].off = (long long)off;
    desc[i].len = (int32_t)len;
    desc[i].prev = -1;
    if (with_labels) {
      auto it = last.find(stream[i]);
      if (it != last.end()) desc[i].prev = it->second;
      else {
        const A0ExTail& tl = ex->tail[stream[i]];
        if (tl.valid) desc[i].prev = -2 - tl.slot;
      }
      last[stream[i]] = i;
    }
    src += len;
    off += a0_ex_up(len, 16);
  }
  memset(ex->h_stage + off, 0, 64);
  ex->tail_src.clear();
  ex->tail_slot.clear();
  if (with_labels) {
    for (auto& kv : last) { ex->tail_src.push_back(kv.second); ex->tail_slot.push_back(ex->tail[kv.first].slot); }
    memcpy(ex->h_stage + L.tsrc, ex->tail_src.data(), ex->tail_src.size() * 4);
    memcpy(ex->h_stage + L.tslot, ex->tail_slot.data(), ex->tail_slot.size() * 4);
  }
  const auto t1 = a0_clock::now();
  A0_CUDA(cudaMemcpyAsync(ex->d_stage, ex->h_stage, L.end, cudaMemcpyHostToDevice, cs));
  A0_CUDA(cudaEventRecord(ex->ev0, cs));
  const A0ExDesc* d_desc = reinterpret_cast<const A0ExDesc*>(ex->d_stage + L.desc);
  int32_t* d_status = reinterpret_cast<int32_t*>(ex->d_back + (size_t)ex->cap * A0_SLOTS);
  if (a0_option_k6_global())
    A0_LAUNCH(a0_k6_lz4_decode_t<true>, (unsigned)mb, 32, 0, cs, 1, 0, ex->d_stage, d_desc, ex->F, ex->d_dec, ex->d_hash, d_status);
  else
    A0_LAUNCH(a0_k6_lz4_decode_t<false>, (unsigned)mb, 32, entry, cs, 1, 0, ex->d_stage, d_desc, ex->F, ex->d_dec, ex->d_hash, d_status);
  if (with_labels)
    A0_LAUNCH(a0_k6_label, (unsigned)mb, K6L_THREADS, 0, cs, 1, 0, ex->d_dec, ex->d_hash, d_desc, ex->F, ex->d_tail_frames,
              ex->d_tail_hash, ex->d_back);
  A0_CUDA(cudaEventRecord(ex->ev1, cs));
  A0_CUDA(cudaMemcpyAsync(ex->h_back, ex->d_back, (size_t)ex->cap * (A0_SLOTS + 4), cudaMemcpyDeviceToHost, cs));
  A0_CUDA(cudaStreamSynchronize(cs));
  const auto t2 = a0_clock::now();
  float dev_ms = 0.0f;
  cudaEventElapsedTime(&dev_ms, ex->ev0, ex->ev1);
  ex->timing[0] += a0_us(t0, t1);
  ex->timing[1] += a0_us(t1, t2);
  ex->timing[4] += dev_ms * 1e3f;
  ex->timing[5] += (float)mb;
  return A0_OK;
}

extern "C" int a0_ex_decode(a0_extend_t* ex, const uint8_t* blobs, const int64_t* blob_len, int32_t m,
                            uint8_t* frames_out, int32_t* status_out, a0_stream_t stream_) {
  A0_REQUIRE(ex && ex->h, "a0_ex_decode: handle without a shard");
  A0_REQUIRE(m >= 0, "a0_ex_decode: negative count");
  if (m == 0) return A0_OK;
  A0_REQUIRE(blobs && blob_len && frames_out && status_out, "a0_ex_decode: NULL argument");
  A0DeviceGuard guard(ex->h->device);
  cudaStream_t cs = (cudaStream_t)stream_;
  const size_t entry = (size_t)A0_SLOTS * ex->F;
  for (int i = 0; i < 6; ++i) ex->timing[i] = 0.0f;
  const uint8_t* src = blobs;
  for (int32_t lo = 0; lo < m; lo += A0_EX_BATCH) {
    const int32_t mb = std::min<int32_t>(A0_EX_BATCH, m - lo);
    int rc = a0_ex_run_batch(ex, src, nullptr, blob_len + lo, nullptr, mb, false, cs, "a0_ex_decode");
    if (rc) return rc;
    const int32_t* st = reinterpret_cast<const int32_t*>(ex->h_back + (size_t)ex->cap * A0_SLOTS);
    memcpy(status_out + lo, st, (size_t)mb * 4);
    A0_CUDA(cudaMemcpyAsync(frames_out + (size_t)lo * entry, ex->d_dec, (size_t)mb * entry, cudaMemcpyDeviceToDevice, cs));
    A0_CUDA(cudaStreamSynchronize(cs));
    for (int32_t i = 0; i < mb; ++i) src += blob_len[lo + i];
  }
  return A0_OK;
}

static int a0_ex_extend_impl(a0_extend_t* ex, const uint8_t* blobs, const uint8_t* const* blob_ptr, const int64_t* blob_len,
                             const int64_t* stream, const int64_t* action, const double* reward, const uint8_t* done, int32_t m,
                             float alpha, a0_stream_t stream_) {
  A0_REQUIRE(ex && ex->h && ex->ix, "a0_ex_extend: handle without a shard");
  A0_REQUIRE(m >= 0, "a0_ex_extend: negative count");
  if (m == 0) return A0_OK;
  A0_REQUIRE((blobs || blob_ptr) && blob_len && stream && action && reward && done, "a0_ex_extend: NULL argument");
  a0_replay* h = ex->h;
  { int frc = a0_check_fault(h, "a0_ex_extend"); if (frc) return frc; }
  A0DeviceGuard guard(h->device);
  cudaStream_t cs = (cudaStream_t)stream_;
  for (int i = 0; i < 6; ++i) ex->timing[i] = 0.0f;
  int64_t st[A0_IX_STATE_WORDS];
  int rc = a0_ix_state(ex->ix, st);
  if (rc) return rc;
  A0_REQUIRE(st[A0_IX_REC_CAPACITY] == h->N && st[A0_IX_FRAME_CAPACITY] == h->NF, "a0_ex_extend: index and shard capacities differ");
  A0_REQUIRE(st[A0_IX_NSTEP] == 1, "a0_ex_extend: reference entries are already n-step folded (agent.py:64-73); the index must "
                                   "gather 1-step windows, not %lld", (long long)st[A0_IX_NSTEP]);
  const int64_t chunk = st[A0_IX_MAX_CHUNK];
  const A0Dyn none = {nullptr, 0.0f, 0.0f, 0.0f};
  const uint8_t* src = blobs;
  for (int32_t lo = 0; lo < m; lo += A0_EX_BATCH) {
    const int32_t mb = std::min<int32_t>(A0_EX_BATCH, m - lo);
    // tails as they were before this batch: a failed batch leaves the host state untouched
    rc = a0_ex_run_batch(ex, src, blob_ptr ? blob_ptr + lo : nullptr, blob_len + lo, stream + lo, mb, true, cs, "a0_ex_extend");
    if (rc) return rc;
    const uint8_t* labels = ex->h_back;
    const int32_t* status = reinterpret_cast<const int32_t*>(ex->h_back + (size_t)ex->cap * A0_SLOTS);
    for (int32_t i = 0; i < mb; ++i)
      A0_REQUIRE(status[i] == A0_LZ_OK, "a0_ex_extend: entry %d is not a valid lz4 block of 8 frames (%s)", lo + i,
                 a0_lz_error(status[i]));
    const auto t2 = a0_clock::now();
    float plan_us = 0.0f;
    for (int32_t c0 = 0; c0 < mb; c0 += (int32_t)chunk) {
      const int32_t cnt = (int32_t)std::min<int64_t>(chunk, mb - c0);
      const auto ta = a0_clock::now();
      ex->fs8.resize((size_t)cnt * A0_SLOTS);
      ex->new_src.resize((size_t)cnt * A0_SLOTS);
      int32_t n_new = 0;
      rc = a0_ex_resolve(ex, stream + lo + c0, labels + (size_t)c0 * A0_SLOTS, cnt, ex->fs8.data(), ex->new_src.data(), &n_new);
      if (rc) return rc;
      for (int32_t j = 0; j < n_new; ++j) ex->new_src[j] += (int64_t)c0 * A0_SLOTS;      // relative to the batch scratch
      a0_plan_t plan;
      rc = a0_ix_plan(ex->ix, stream + lo + c0, ex->fs8.data(), cnt, n_new, action + lo + c0, reward + lo + c0, done + lo + c0, &plan);
      if (rc) return rc;
      const auto tb = a0_clock::now();
      plan_us += a0_us(ta, tb);
      rc = a0_ingest_plan_impl(h, &plan, ex->d_dec, n_new ? ex->new_src.data() : nullptr, A0_INGEST_FRAMES_ON_DEVICE, alpha, stream_, none);
      if (rc) return rc;
    }
    const int32_t nt = (int32_t)ex->tail_src.size();
    if (nt) {
      const A0ExLayout L = a0_ex_layout(mb, blob_len + lo);
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3((unsigned)nt, A0_SLOTS);
      cfg.blockDim = dim3(128);
      cfg.stream = cs;
      cudaError_t e = cudaLaunchKernelEx(&cfg, a0_k6_tails, (const uint8_t*)ex->d_dec, (const unsigned long long*)ex->d_hash,
                                         (const int32_t*)(ex->d_stage + L.tsrc), (const int32_t*)(ex->d_stage + L.tslot), ex->F,
                                         ex->d_tail_frames, ex->d_tail_hash);
      if (e != cudaSuccess) { a0_set_error("a0_ex_extend: tail launch failed: %s", cudaGetErrorString(e)); return (int)e; }
    }
    const auto t3 = a0_clock::now();
    ex->timing[2] += plan_us;
    ex->timing[3] += a0_us(t2, t3) - plan_us;
    if (src) for (int32_t i = 0; i < mb; ++i) src += blob_len[lo + i];
  }
  return A0_OK;
}

extern "C" int a0_ex_extend(a0_extend_t* ex, const uint8_t* blobs, const int64_t* blob_len, const int64_t* stream,
                            const int64_t* action, const double* reward, const uint8_t* done, int32_t m, float alpha,
                            a0_stream_t stream_) {
  A0_REQUIRE(m == 0 || blobs, "a0_ex_extend: blobs is NULL");
  return a0_ex_extend_impl(ex, blobs, nullptr, blob_len, stream, action, reward, done, m, alpha, stream_);
}

extern "C" int a0_ex_extend_v(a0_extend_t* ex, const uint8_t* const* blob_ptr, const int64_t* blob_len, const int64_t* stream,
                              const int64_t* action, const double* reward, const uint8_t* done, int32_t m, float alpha,
                              a0_stream_t stream_) {
  A0_REQUIRE(m == 0 || blob_ptr, "a0_ex_extend_v: blob_ptr is NULL");
  return a0_ex_extend_impl(ex, nullptr, blob_ptr, blob_len, stream, action, reward, done, m, alpha, stream_);
}

extern "C" int a0_ex_last_timing(a0_extend_t* ex, float* out6) {
  A0_REQUIRE(ex && out6, "a0_ex_last_timing: NULL argument");
  for (int i = 0; i < 6; ++i) out6[i] = ex->timing[i];
  return A0_OK;
}

// ------------------------------------------------------------------------------------------------
// checkpoints (a0_ckpt.cu): the decode kernel on one batch of blobs, and the stream tails.
// TAILS layout: count i64, then per stream in ascending id order {id i64, seq i64[8], cls u8[8], frames u8[8][F],
// hash u64[8]}.
// ------------------------------------------------------------------------------------------------
int a0_ex_decode_dev(a0_extend* ex, const uint8_t* blobs, const int64_t* blob_len, int32_t mb, cudaStream_t cs,
                     const uint8_t** dec, const unsigned long long** hash, const int32_t** status) {
  int rc = a0_ex_run_batch(ex, blobs, nullptr, blob_len, nullptr, mb, false, cs, "a0_ckpt_load");
  if (rc) return rc;
  *dec = ex->d_dec;
  *hash = ex->d_hash;
  *status = reinterpret_cast<const int32_t*>(ex->h_back + (size_t)ex->cap * A0_SLOTS);
  return A0_OK;
}

static inline size_t a0_ex_tail_bytes(int32_t F) { return 8 + 64 + 8 + (size_t)A0_SLOTS * F + 64; }

int a0_ex_tails_save(a0_extend* ex, std::vector<uint8_t>& out) {
  std::vector<int64_t> ids;
  for (auto& kv : ex->tail)
    if (kv.second.valid) ids.push_back(kv.first);
  std::sort(ids.begin(), ids.end());
  const size_t each = a0_ex_tail_bytes(ex->F);
  out.assign(8 + ids.size() * each, 0);
  const int64_t count = (int64_t)ids.size();
  memcpy(out.data(), &count, 8);
  uint8_t* p = out.data() + 8;
  for (int64_t id : ids) {
    const A0ExTail& tl = ex->tail[id];
    memcpy(p, &id, 8);
    memcpy(p + 8, tl.seq, 64);
    memcpy(p + 72, tl.cls, 8);
    A0_CUDA(cudaMemcpy(p + 80, ex->d_tail_frames + (size_t)tl.slot * A0_SLOTS * ex->F, (size_t)A0_SLOTS * ex->F, cudaMemcpyDeviceToHost));
    A0_CUDA(cudaMemcpy(p + 80 + (size_t)A0_SLOTS * ex->F, ex->d_tail_hash + (size_t)tl.slot * A0_SLOTS, 64, cudaMemcpyDeviceToHost));
    p += each;
  }
  return A0_OK;
}

// structure only: called before the shard is touched
int a0_ex_tails_check(int32_t F, const uint8_t* p, int64_t len, int64_t head_fs) {
  int64_t count = 0;
  A0_REQUIRE(len >= 8, "a0_ckpt_load: TAILS section truncated");
  memcpy(&count, p, 8);
  const size_t each = a0_ex_tail_bytes(F);
  A0_REQUIRE(count >= 0 && (uint64_t)count <= (uint64_t)(len - 8) / each && 8 + (int64_t)(count * each) == len,
             "a0_ckpt_load: TAILS section has the wrong length");
  int64_t prev = 0;
  for (int64_t i = 0; i < count; ++i) {
    const uint8_t* e = p + 8 + i * each;
    int64_t id, seq[A0_SLOTS];
    memcpy(&id, e, 8);
    memcpy(seq, e + 8, 64);
    A0_REQUIRE(i == 0 || id > prev, "a0_ckpt_load: TAILS stream ids out of order");
    prev = id;
    for (int j = 0; j < A0_SLOTS; ++j)
      A0_REQUIRE(seq[j] >= 0 && seq[j] < head_fs && e[72 + j] < 2 * A0_SLOTS, "a0_ckpt_load: TAILS entry of stream %lld is inconsistent",
                 (long long)id);
  }
  return A0_OK;
}

void a0_ex_tails_clear(a0_extend* ex) {
  ex->tail.clear();
  ex->n_slots = 0;
}

int a0_ex_tails_load(a0_extend* ex, const uint8_t* p, int64_t len, cudaStream_t cs) {
  (void)len;
  a0_ex_tails_clear(ex);
  int64_t count = 0;
  memcpy(&count, p, 8);
  int rc = a0_ex_reserve(ex, 0, 0, (int32_t)count);
  if (rc) return rc;
  const size_t each = a0_ex_tail_bytes(ex->F), entry = (size_t)A0_SLOTS * ex->F;
  for (int64_t i = 0; i < count; ++i) {
    const uint8_t* e = p + 8 + i * each;
    int64_t id;
    memcpy(&id, e, 8);
    A0ExTail& tl = ex->tail[id];
    memcpy(tl.seq, e + 8, 64);
    memcpy(tl.cls, e + 72, 8);
    tl.slot = (int32_t)i;
    tl.valid = true;
    A0_CUDA(cudaMemcpyAsync(ex->d_tail_frames + (size_t)i * entry, e + 80, entry, cudaMemcpyHostToDevice, cs));
    A0_CUDA(cudaMemcpyAsync(ex->d_tail_hash + (size_t)i * A0_SLOTS, e + 80 + entry, 64, cudaMemcpyHostToDevice, cs));
  }
  ex->n_slots = (int32_t)count;
  A0_CUDA(cudaStreamSynchronize(cs));
  return A0_OK;
}

a0_replay* a0_ex_shard(a0_extend* ex) { return ex->h; }
