// K7: LZ4 encode of 8-frame groups, one warp per group -- the frames of a checkpoint leave the device compressed.
//
// A group (8 * F bytes, the entry K6a decodes) comes into shared memory with one cp.async.bulk copy, next to a
// 4096-entry hash table (u16 entries while 8F <= 65536, u32 above).  The parse is the sequential greedy one of
// oracle/lz4_encode.py (encode_greedy), reproduced byte for byte:
//   * a step tests the 32 positions p .. p + 31, one per lane.  Lane i's candidate is what the sequential loop would
//     read at p + i: the latest earlier lane of the step with the same hash (__match_any_sync), else the table as it
//     stood before the step.  A ballot picks the first lane with a 4-byte match within the offset limit;
//   * the positions up to that lane (all 32 when none matched) go into the table, the highest lane winning a
//     collision, exactly as the sequential loop inserts them one after the other;
//   * the match is extended 32 bytes per ballot, the literals are copied out by the whole warp, e - 2 is inserted;
//   * the block-format end rules: no match starts within the last 12 bytes, the last 5 bytes are literals.
// The warp also hashes each frame while it is on chip (a0_k6_frame_hash, the hash K6a computes while decoding), so
// a loader can check every decoded frame.  A group whose block would not be shorter than 8F is stored raw.
#include "a0_common.cuh"

namespace {

constexpr int K7_HASH_LOG = 12;
constexpr int K7_TABLE = 1 << K7_HASH_LOG;
constexpr int K7_MIN_MATCH = 4, K7_LAST_LITERALS = 5, K7_MF_LIMIT = 12, K7_MAX_OFFSET = 65535;

__device__ __forceinline__ uint32_t k7_hash(uint32_t w) { return (w * 2654435761u) >> (32 - K7_HASH_LOG); }

// 4 bytes at p of the group in shared memory (the buffer has 16 bytes of slack behind the group)
__device__ __forceinline__ uint32_t k7_read32(const uint8_t* src, int p) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(src);
  const int i = p >> 2, sh = (p & 3) * 8;
  return sh ? __funnelshift_r(w[i], w[i + 1], sh) : w[i];
}

// LZ4 length extension bytes of `extra` (>= 0): 255 ... then the remainder; returns the next output position
__device__ __forceinline__ int k7_put_len(uint8_t* o, int op, int extra, int lane) {
  const int k = extra / 255;
  for (int i = lane; i < k; i += 32) o[op + i] = 255;
  if (lane == 0) o[op + k] = (uint8_t)(extra - 255 * k);
  return op + k + 1;
}
__device__ __forceinline__ int k7_len_bytes(int extra) { return extra >= 15 ? (extra - 15) / 255 + 1 : 0; }

// One sequence: literals src[anchor, anchor + ll), then (ml > 0) the match {off, ml}.  Returns the new output
// position, or -1 when the blob would reach `n` bytes (the group is then stored raw).
__device__ __forceinline__ int k7_sequence(uint8_t* o, int op, const uint8_t* src, int anchor, int ll, int off, int ml,
                                           int n, int lane) {
  const int need = 1 + k7_len_bytes(ll) + ll + (ml ? 2 + k7_len_bytes(ml - K7_MIN_MATCH) : 0);
  if (op + need >= n) return -1;
  if (lane == 0) o[op] = (uint8_t)((min(ll, 15) << 4) | (ml ? min(ml - K7_MIN_MATCH, 15) : 0));
  ++op;
  if (ll >= 15) op = k7_put_len(o, op, ll - 15, lane);
  for (int i = lane; i < ll; i += 32) o[op + i] = src[anchor + i];
  op += ll;
  if (ml) {
    if (lane == 0) { o[op] = (uint8_t)(off & 255); o[op + 1] = (uint8_t)(off >> 8); }
    op += 2;
    if (ml - K7_MIN_MATCH >= 15) op = k7_put_len(o, op, ml - K7_MIN_MATCH - 15, lane);
  }
  return op;
}

}  // namespace

template <typename T>
__global__ void __launch_bounds__(32)
a0_k7_lz4_encode(const uint8_t* __restrict__ frames, int32_t F, int64_t stride, uint8_t* __restrict__ out,
                 int32_t* __restrict__ out_len, unsigned long long* __restrict__ frame_hash) {
  extern __shared__ __align__(128) uint8_t k7_smem[];
  __shared__ __align__(8) unsigned long long bar;
  const int g = blockIdx.x, lane = threadIdx.x;
  const int n = A0_SLOTS * F;
  uint8_t* src = k7_smem;
  T* table = reinterpret_cast<T*>(k7_smem + n + 16);
  const uint32_t b = a0_smem_u32(&bar);
  if (lane == 0) {
    a0_mbar_init(b, 1);
    a0_fence_barrier_init();
    a0_bulk_load(a0_smem_u32(src), frames + (size_t)g * n, (uint32_t)n, b);
  }
  for (int i = lane; i < K7_TABLE; i += 32) table[i] = 0;
  if (lane < 4) reinterpret_cast<uint32_t*>(src + n)[lane] = 0u;
  __syncwarp();
  a0_mbar_wait(b, 0);

  const int nvec = F >> 4;
#pragma unroll 1
  for (int f = 0; f < A0_SLOTS; ++f) {
    const unsigned long long h = a0_k6_frame_hash(src + (size_t)f * F, nvec, lane);
    if (lane == 0) frame_hash[(size_t)g * A0_SLOTS + f] = h;
  }

  uint8_t* o = out + (size_t)g * stride;
  int op = 4, anchor = 0, p = 0;
  const int plimit = n - K7_MF_LIMIT;            // a match starts at p <= plimit
  const int elimit = n - K7_LAST_LITERALS;       // and ends at e <= elimit
  const unsigned below = (1u << lane) - 1u;
#pragma unroll 1
  while (p <= plimit && op >= 0) {
    const int q = p + lane;
    const bool valid = q <= plimit;
    const uint32_t w = valid ? k7_read32(src, q) : 0u;
    const uint32_t h = valid ? k7_hash(w) : 0xFFFFFFFFu;
    const unsigned peers = __match_any_sync(0xFFFFFFFFu, h);
    const unsigned earlier = peers & below;
    int c = earlier ? p + (31 - __clz(earlier)) : (valid ? (int)table[h] : 0);
    const bool ok = valid && c < q && q - c <= K7_MAX_OFFSET && k7_read32(src, c) == w;
    const unsigned ball = __ballot_sync(0xFFFFFFFFu, ok);
    const int j = ball ? __ffs(ball) - 1 : 31;
    const unsigned upto = j == 31 ? 0xFFFFFFFFu : ((2u << j) - 1u);
    // insert p .. p + j: the highest lane of each hash wins (the sequential loop's last write)
    if (valid && lane <= j && (peers & upto & ~below & ~(1u << lane)) == 0) table[h] = (T)q;
    __syncwarp();
    if (!ball) { p += 32; continue; }
    const int mstart = p + j;
    const int off = mstart - __shfl_sync(0xFFFFFFFFu, c, j);
    int e = mstart + K7_MIN_MATCH;
#pragma unroll 1
    while (true) {
      const int k = e + lane;
      const bool eq = k < elimit && src[k] == src[k - off];
      const unsigned miss = __ballot_sync(0xFFFFFFFFu, !eq);
      if (miss) { e += __ffs(miss) - 1; break; }
      e += 32;
    }
    op = k7_sequence(o, op, src, anchor, mstart - anchor, off, e - mstart, n, lane);
    if (lane == 0) table[k7_hash(k7_read32(src, e - 2))] = (T)(e - 2);
    __syncwarp();
    anchor = p = e;
  }
  if (op >= 0) op = k7_sequence(o, op, src, anchor, n - anchor, 0, 0, n, lane);
  if (op < 0) {
    // not shorter than the input: the group itself
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* o4 = reinterpret_cast<uint4*>(o);
    for (int i = lane; i < (n >> 4); i += 32) o4[i] = s4[i];
    op = n;
  } else if (lane == 0) {
    o[0] = (uint8_t)n; o[1] = (uint8_t)(n >> 8); o[2] = (uint8_t)(n >> 16); o[3] = (uint8_t)(n >> 24);
  }
  if (lane == 0) out_len[g] = op;
}

extern "C" int a0_lz4_encode(const uint8_t* frames, int32_t m, int32_t frame_bytes, uint8_t* out, int32_t* out_len,
                             uint64_t* frame_hash, a0_stream_t stream_) {
  A0_REQUIRE(m >= 0, "a0_lz4_encode: negative count");
  A0_REQUIRE(frame_bytes > 0 && frame_bytes % 16 == 0 && (int64_t)frame_bytes * A0_SLOTS <= 200 * 1024,
             "a0_lz4_encode: frame_bytes %d must be a positive multiple of 16 and at most 25 600", frame_bytes);
  if (m == 0) return A0_OK;
  A0_REQUIRE(frames && out && out_len && frame_hash, "a0_lz4_encode: NULL argument");
  A0_REQUIRE(((uintptr_t)frames & 15) == 0 && ((uintptr_t)out & 15) == 0, "a0_lz4_encode: frames and out must be 16-byte aligned");
  const int n = A0_SLOTS * frame_bytes;
  const bool wide = n > 65536;
  const size_t smem = (size_t)n + 16 + (size_t)K7_TABLE * (wide ? 4 : 2);
  int dev = 0;
  A0_CUDA(cudaGetDevice(&dev));
  static bool attr_set[64][2] = {};
  if (dev < 64 && !attr_set[dev][wide]) {
    // the largest group each variant takes: 64 KB (u16 table) or 200 KB (u32 table)
    if (wide) A0_CUDA(cudaFuncSetAttribute(a0_k7_lz4_encode<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024 + 16 + K7_TABLE * 4));
    else A0_CUDA(cudaFuncSetAttribute(a0_k7_lz4_encode<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536 + 16 + K7_TABLE * 2));
    attr_set[dev][wide] = true;
  }
  cudaStream_t cs = (cudaStream_t)stream_;
  const int64_t stride = A0_LZ4_STRIDE(frame_bytes);
  unsigned long long* fh = reinterpret_cast<unsigned long long*>(frame_hash);
  if (wide) A0_LAUNCH(a0_k7_lz4_encode<uint32_t>, (unsigned)m, 32, smem, cs, 1, 0, frames, frame_bytes, stride, out, out_len, fh);
  else A0_LAUNCH(a0_k7_lz4_encode<uint16_t>, (unsigned)m, 32, smem, cs, 1, 0, frames, frame_bytes, stride, out, out_len, fh);
  return A0_OK;
}
