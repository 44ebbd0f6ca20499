// Checkpoint of one replay shard: a0_ckpt_save / a0_ckpt_load (format: include/agent0_b200.h, DESIGN §3).
//
// Frames are 99 % of a shard's bytes, so they leave as K7 blobs (one python-lz4 block per 8 consecutive frame
// seqs) and come back through K6a, the decoder the reference-tuple ingest already uses.  Save runs batch by batch:
// the batch's frames are gathered from the ring (at most two copies: the ring may wrap), K7 encodes them, the
// blobs are compacted on the device and leave with ONE device-to-host copy into one of two page-locked buffers, so
// the encoder of the next batch runs while this one is written to the file.
#include <sys/stat.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <memory>
#include <string>
#include <vector>

#include "a0_common.cuh"

namespace {

constexpr char A0_CK_MAGIC[8] = {'A', '0', 'C', 'K', 'P', 'T', '0', '1'};
constexpr uint32_t A0_CK_VERSION = 1;
enum { CK_INDEX = 1, CK_RECORDS = 2, CK_LEAVES = 3, CK_SCALARS = 4, CK_TAILS = 5, CK_USER = 6, CK_FRAMES = 7, CK_BLOBS = 8 };
constexpr int32_t CK_BATCH = 1024;          // groups per encode / decode batch

struct CkHeader {
  char magic[8];
  uint32_t version, zero;
  int64_t N, NF, F, P, n_step, age_limit;
};
struct CkSection {
  uint32_t tag, zero;
  uint64_t len, hash;
};

// 64-bit hash of a section payload: four multiply-rotate lanes over 32-byte blocks, then the tail bytes and the
// length folded in.  Streaming, so the frames section is hashed as it is written or read.
struct CkHash {
  uint64_t h[4] = {0x9E3779B97F4A7C15ull, 0xC2B2AE3D27D4EB4Full, 0x165667B19E3779F9ull, 0x27D4EB2F165667C5ull};
  uint8_t buf[32];
  size_t nbuf = 0, total = 0;
  static inline uint64_t lane(uint64_t x, uint64_t w) { x = (x ^ w) * 0x9FB21C651E98DF25ull; return (x << 29) | (x >> 35); }
  void block(const uint8_t* p) {
    uint64_t w[4];
    memcpy(w, p, 32);
    for (int i = 0; i < 4; ++i) h[i] = lane(h[i], w[i]);
  }
  void update(const void* data, size_t n) {
    const uint8_t* p = static_cast<const uint8_t*>(data);
    total += n;
    if (nbuf) {
      const size_t k = std::min(n, 32 - nbuf);
      memcpy(buf + nbuf, p, k); nbuf += k; p += k; n -= k;
      if (nbuf < 32) return;
      block(buf); nbuf = 0;
    }
    for (; n >= 32; p += 32, n -= 32) block(p);
    memcpy(buf, p, n); nbuf = n;
  }
  uint64_t final() const {
    uint64_t x = h[0] ^ (h[1] * 3) ^ (h[2] * 5) ^ (h[3] * 7);
    for (size_t i = 0; i < nbuf; ++i) x = lane(x, buf[i]);
    x = lane(x, (uint64_t)total);
    x ^= x >> 32; x *= 0xD6E8FEB86659FD93ull; x ^= x >> 32;
    return x;
  }
};
uint64_t ck_hash(const void* p, size_t n) { CkHash h; h.update(p, n); return h.final(); }

using ck_clock = std::chrono::steady_clock;
double ck_us(ck_clock::time_point a, ck_clock::time_point b) { return std::chrono::duration<double, std::micro>(b - a).count(); }
double g_timing[8] = {0, 0, 0, 0, 0, 0, 0, 0};

struct CkFile {
  FILE* f = nullptr;
  ~CkFile() { if (f) fclose(f); }
};

int ck_write(FILE* f, const void* p, size_t n, const char* path) {
  if (n && fwrite(p, 1, n, f) != n) { a0_set_error("a0_ckpt_save: write to %s failed", path); return A0_EINVAL; }
  return A0_OK;
}
int ck_section(FILE* f, uint32_t tag, const void* p, size_t n, const char* path) {
  const CkSection s = {tag, 0, (uint64_t)n, ck_hash(p, n)};
  int rc = ck_write(f, &s, sizeof(s), path);
  return rc ? rc : ck_write(f, p, n, path);
}

struct CkPinned {                  // page-locked host memory, freed on scope exit
  uint8_t* p = nullptr;
  ~CkPinned() { if (p) cudaFreeHost(p); }
};
struct CkDev {
  void* p = nullptr;
  ~CkDev() { if (p) cudaFree(p); }
};
struct CkEvents {
  cudaEvent_t e[6] = {};
  ~CkEvents() { for (auto x : e) if (x) cudaEventDestroy(x); }
};

// frames of seqs [s0, s1) (s1 - s0 <= NF) from the ring to a contiguous device buffer, or back (to_ring)
int ck_ring_copy(a0_replay* h, uint8_t* buf, int64_t s0, int64_t s1, bool to_ring, cudaStream_t cs) {
  const size_t F = (size_t)h->F;
  int64_t s = s0;
  while (s < s1) {
    const int64_t pos = s % h->NF, k = std::min<int64_t>(s1 - s, h->NF - pos);
    uint8_t* ring = h->frames + (size_t)pos * F;
    uint8_t* lin = buf + (size_t)(s - s0) * F;
    A0_CUDA(cudaMemcpyAsync(to_ring ? ring : lin, to_ring ? lin : ring, (size_t)k * F, cudaMemcpyDeviceToDevice, cs));
    s += k;
  }
  return A0_OK;
}

}  // namespace

// group g's blob (length len[g], at scratch + g * stride) to dst + off[g]
__global__ void __launch_bounds__(128) a0_ck_compact(const uint8_t* __restrict__ scratch, int64_t stride, const int32_t* __restrict__ len,
                                                     const int64_t* __restrict__ off, uint8_t* __restrict__ dst) {
  const int g = blockIdx.x;
  const uint8_t* s = scratch + (size_t)g * stride;
  uint8_t* d = dst + off[g];
  const int n = len[g];
  for (int i = threadIdx.x; i < n; i += 128) d[i] = s[i];
}

extern "C" int a0_ckpt_save(a0_replay_t* h, a0_index_t* ix, a0_extend_t* ex, const char* path, const uint8_t* user,
                            int64_t user_len, a0_stream_t stream_) {
  A0_REQUIRE(h && ix && path, "a0_ckpt_save: NULL argument");
  A0_REQUIRE(user_len >= 0 && (user_len == 0 || user), "a0_ckpt_save: bad user bytes");
  A0_REQUIRE(!ex || a0_ex_shard(ex) == h, "a0_ckpt_save: the ingest handle belongs to another shard");
  const auto t0 = ck_clock::now();
  for (double& x : g_timing) x = 0.0;
  A0DeviceGuard guard(h->device);
  cudaStream_t cs = (cudaStream_t)stream_;
  cudaStreamCaptureStatus cst = cudaStreamCaptureStatusNone;
  A0_CUDA(cudaStreamIsCapturing(cs, &cst));
  A0_REQUIRE(cst == cudaStreamCaptureStatusNone, "a0_ckpt_save: the stream is being captured into a CUDA graph");
  A0_CUDA(cudaStreamSynchronize(cs));
  { int frc = a0_check_fault(h, "a0_ckpt_save"); if (frc) return frc; }
  int64_t st[A0_IX_STATE_WORDS];
  int rc = a0_ix_state(ix, st);
  if (rc) return rc;
  A0_REQUIRE(st[A0_IX_REC_CAPACITY] == h->N && st[A0_IX_FRAME_CAPACITY] == h->NF, "a0_ckpt_save: index and shard capacities differ");
  const int64_t N = h->N, F = h->F, head_fs = st[A0_IX_HEAD_FS];

  const std::string tmp = std::string(path) + ".tmp";
  CkFile file;
  file.f = fopen(tmp.c_str(), "wb");
  A0_REQUIRE(file.f, "a0_ckpt_save: cannot open %s for writing", tmp.c_str());
  FILE* f = file.f;
  CkHeader hd;
  memcpy(hd.magic, A0_CK_MAGIC, 8);
  hd.version = A0_CK_VERSION; hd.zero = 0;
  hd.N = N; hd.NF = h->NF; hd.F = F; hd.P = h->P; hd.n_step = st[A0_IX_NSTEP]; hd.age_limit = st[A0_IX_AGE_LIMIT];
  if ((rc = ck_write(f, &hd, sizeof(hd), path))) return rc;
  {
    int64_t len = 0;
    a0_ix_serialize(ix, nullptr, 0, &len);
    std::vector<uint8_t> b((size_t)len);
    if ((rc = a0_ix_serialize(ix, b.data(), len, &len))) return rc;
    if ((rc = ck_section(f, CK_INDEX, b.data(), b.size(), path))) return rc;
  }
  {
    std::vector<uint8_t> b((size_t)N * (A0_SLOTS * 4 + sizeof(A0RecInfo)));
    A0_CUDA(cudaMemcpy(b.data(), h->rec_slots, (size_t)N * A0_SLOTS * 4, cudaMemcpyDeviceToHost));
    A0_CUDA(cudaMemcpy(b.data() + (size_t)N * A0_SLOTS * 4, h->rec_info, (size_t)N * sizeof(A0RecInfo), cudaMemcpyDeviceToHost));
    if ((rc = ck_section(f, CK_RECORDS, b.data(), b.size(), path))) return rc;
    b.resize((size_t)N * 4);
    A0_CUDA(cudaMemcpy(b.data(), h->tree + h->P, (size_t)N * 4, cudaMemcpyDeviceToHost));
    if ((rc = ck_section(f, CK_LEAVES, b.data(), b.size(), path))) return rc;
  }
  {
    uint8_t b[32];
    A0_CUDA(cudaMemcpy(b, h->max_p, 4, cudaMemcpyDeviceToHost));
    A0_CUDA(cudaMemcpy(b + 4, h->dyn, 12, cudaMemcpyDeviceToHost));
    A0_CUDA(cudaMemcpy(b + 16, h->counter + A0_RNG_CALL_WORD, 8, cudaMemcpyDeviceToHost));
    memcpy(b + 24, &h->stride_hint, 8);
    if ((rc = ck_section(f, CK_SCALARS, b, sizeof(b), path))) return rc;
  }
  {
    std::vector<uint8_t> b(8, 0);
    if (ex && (rc = a0_ex_tails_save(ex, b))) return rc;
    if ((rc = ck_section(f, CK_TAILS, b.data(), b.size(), path))) return rc;
  }
  if ((rc = ck_section(f, CK_USER, user, (size_t)user_len, path))) return rc;

  // ---- frames: the group table is written once the blobs are known, into the room kept for it
  const int64_t lo = std::max<int64_t>(0, head_fs - h->NF), nfr = head_fs - lo, G = (nfr + 7) / 8;
  std::vector<int64_t> table((size_t)(3 + 2 * G));
  std::vector<uint64_t> fhash((size_t)G * A0_SLOTS);
  table[0] = lo; table[1] = nfr; table[2] = G;
  const long table_at = ftell(f);
  const size_t table_bytes = table.size() * 8 + fhash.size() * 8;
  {
    const CkSection s = {CK_FRAMES, 0, (uint64_t)table_bytes, 0};
    if ((rc = ck_write(f, &s, sizeof(s), path))) return rc;
    A0_REQUIRE(fseek(f, (long)table_bytes, SEEK_CUR) == 0, "a0_ckpt_save: seek in %s failed", path);
  }
  const long blobs_at = ftell(f);
  {
    const CkSection s = {CK_BLOBS, 0, 0, 0};
    if ((rc = ck_write(f, &s, sizeof(s), path))) return rc;
  }
  CkHash bh;
  uint64_t blob_total = 0;
  if (G > 0) {
    const int32_t B = (int32_t)std::min<int64_t>(CK_BATCH, G);
    const size_t group = (size_t)A0_SLOTS * F;
    const int64_t stride = A0_LZ4_STRIDE(F);
    CkDev d_in, d_out, d_len, d_hash, d_off, d_cmp;
    A0_CUDA(cudaMalloc(&d_in.p, (size_t)B * group));
    A0_CUDA(cudaMalloc(&d_out.p, (size_t)B * stride));
    A0_CUDA(cudaMalloc(&d_len.p, (size_t)B * 4));
    A0_CUDA(cudaMalloc(&d_hash.p, (size_t)B * A0_SLOTS * 8));
    A0_CUDA(cudaMalloc(&d_off.p, (size_t)B * 8));
    A0_CUDA(cudaMalloc(&d_cmp.p, (size_t)B * group));
    CkPinned big[2], small;
    A0_CUDA(cudaMallocHost((void**)&big[0].p, (size_t)B * group));
    A0_CUDA(cudaMallocHost((void**)&big[1].p, (size_t)B * group));
    A0_CUDA(cudaMallocHost((void**)&small.p, (size_t)B * (4 + 8 + A0_SLOTS * 8)));
    int32_t* h_len = reinterpret_cast<int32_t*>(small.p);
    int64_t* h_off = reinterpret_cast<int64_t*>(small.p + (size_t)B * 4);
    uint64_t* h_hash = reinterpret_cast<uint64_t*>(small.p + (size_t)B * 12);
    CkEvents ev;      // 0, 1: encode start / end; 2, 3: compaction + device-to-host copy start / end
    for (auto& x : ev.e) A0_CUDA(cudaEventCreate(&x));
    cudaEvent_t copied[2];
    A0_CUDA(cudaEventCreateWithFlags(&copied[0], cudaEventDisableTiming));
    A0_CUDA(cudaEventCreateWithFlags(&copied[1], cudaEventDisableTiming));
    size_t pending_bytes[2] = {0, 0};
    int pending = -1;                   // turn whose blobs are on their way into big[turn]
    auto flush = [&](int turn) -> int {
      const auto a = ck_clock::now();
      A0_CUDA(cudaEventSynchronize(copied[turn]));
      const auto b = ck_clock::now();
      float ms = 0.0f;
      cudaEventElapsedTime(&ms, ev.e[2], ev.e[3]);      // this batch's compaction + device-to-host copy
      g_timing[2] += ms * 1e3;
      bh.update(big[turn].p, pending_bytes[turn]);
      int r = ck_write(f, big[turn].p, pending_bytes[turn], path);
      g_timing[3] += ck_us(b, ck_clock::now());
      g_timing[6] += ck_us(a, b);
      return r;
    };
    int turn = 0;
    for (int64_t g0 = 0; g0 < G; g0 += B, turn ^= 1) {
      const int32_t mb = (int32_t)std::min<int64_t>(B, G - g0);
      const int64_t s0 = lo + 8 * g0, s1 = std::min<int64_t>(s0 + 8 * (int64_t)mb, head_fs);
      uint8_t* in = static_cast<uint8_t*>(d_in.p);
      if ((rc = ck_ring_copy(h, in, s0, s1, false, cs))) break;
      if (s1 - s0 < 8 * (int64_t)mb)
        A0_CUDA(cudaMemsetAsync(in + (size_t)(s1 - s0) * F, 0, (size_t)(8 * (int64_t)mb - (s1 - s0)) * F, cs));
      A0_CUDA(cudaEventRecord(ev.e[0], cs));
      if ((rc = a0_lz4_encode(in, mb, (int32_t)F, static_cast<uint8_t*>(d_out.p), static_cast<int32_t*>(d_len.p),
                              static_cast<uint64_t*>(d_hash.p), cs))) break;
      A0_CUDA(cudaEventRecord(ev.e[1], cs));
      A0_CUDA(cudaMemcpyAsync(h_len, d_len.p, (size_t)mb * 4, cudaMemcpyDeviceToHost, cs));
      A0_CUDA(cudaMemcpyAsync(h_hash, d_hash.p, (size_t)mb * A0_SLOTS * 8, cudaMemcpyDeviceToHost, cs));
      if (pending >= 0 && (rc = flush(pending))) break;      // the previous batch goes to the file while this one encodes
      pending = -1;
      A0_CUDA(cudaStreamSynchronize(cs));
      float ms = 0.0f;
      cudaEventElapsedTime(&ms, ev.e[0], ev.e[1]);
      g_timing[1] += ms * 1e3;
      int64_t off = 0;
      for (int32_t i = 0; i < mb; ++i) {
        A0_REQUIRE(h_len[i] > 0 && h_len[i] <= (int32_t)group, "a0_ckpt_save: encoder returned a bad length");
        h_off[i] = off;
        off += h_len[i];
        table[3 + 2 * (g0 + i)] = (s0 + 8 * (int64_t)i) % h->NF;
        table[4 + 2 * (g0 + i)] = h_len[i];
      }
      memcpy(fhash.data() + (size_t)g0 * A0_SLOTS, h_hash, (size_t)mb * A0_SLOTS * 8);
      A0_CUDA(cudaMemcpyAsync(d_off.p, h_off, (size_t)mb * 8, cudaMemcpyHostToDevice, cs));
      A0_CUDA(cudaEventRecord(ev.e[2], cs));
      a0_ck_compact<<<mb, 128, 0, cs>>>(static_cast<const uint8_t*>(d_out.p), stride, static_cast<const int32_t*>(d_len.p),
                                        static_cast<const int64_t*>(d_off.p), static_cast<uint8_t*>(d_cmp.p));
      A0_LAUNCH_CHECK();
      A0_CUDA(cudaMemcpyAsync(big[turn].p, d_cmp.p, (size_t)off, cudaMemcpyDeviceToHost, cs));
      A0_CUDA(cudaEventRecord(ev.e[3], cs));
      A0_CUDA(cudaEventRecord(copied[turn], cs));
      pending_bytes[turn] = (size_t)off;
      pending = turn;
      blob_total += (uint64_t)off;
    }
    if (!rc && pending >= 0) rc = flush(pending);
    A0_CUDA(cudaStreamSynchronize(cs));
    cudaEventDestroy(copied[0]);
    cudaEventDestroy(copied[1]);
    if (rc) return rc;
  }
  {
    // BLOBS header, then the group table into its room
    const CkSection s = {CK_BLOBS, 0, blob_total, bh.final()};
    A0_REQUIRE(fseek(f, blobs_at, SEEK_SET) == 0, "a0_ckpt_save: seek in %s failed", path);
    if ((rc = ck_write(f, &s, sizeof(s), path))) return rc;
    CkHash th;
    th.update(table.data(), table.size() * 8);
    th.update(fhash.data(), fhash.size() * 8);
    const CkSection t = {CK_FRAMES, 0, (uint64_t)table_bytes, th.final()};
    A0_REQUIRE(fseek(f, table_at, SEEK_SET) == 0, "a0_ckpt_save: seek in %s failed", path);
    if ((rc = ck_write(f, &t, sizeof(t), path))) return rc;
    if ((rc = ck_write(f, table.data(), table.size() * 8, path))) return rc;
    if ((rc = ck_write(f, fhash.data(), fhash.size() * 8, path))) return rc;
  }
  A0_REQUIRE(fflush(f) == 0, "a0_ckpt_save: write to %s failed", tmp.c_str());
  const int cl = fclose(f);
  file.f = nullptr;
  A0_REQUIRE(cl == 0 && rename(tmp.c_str(), path) == 0, "a0_ckpt_save: cannot finish %s", path);
  g_timing[0] = ck_us(t0, ck_clock::now());
  g_timing[4] = (double)nfr * F;
  g_timing[5] = (double)blob_total;
  return A0_OK;
}

namespace {
struct CkReader {
  FILE* f;
  const char* path;
  int64_t size;
  const char* who;
  int section(uint32_t tag, std::vector<uint8_t>& out, bool check_hash = true) {
    CkSection s;
    A0_REQUIRE(fread(&s, sizeof(s), 1, f) == 1, "%s: %s is truncated (section %u)", who, path, tag);
    A0_REQUIRE(s.tag == tag && s.zero == 0, "%s: %s: expected section %u, found %u", who, path, tag, s.tag);
    A0_REQUIRE(s.len <= (uint64_t)(size - ftell(f)), "%s: %s is truncated (section %u)", who, path, tag);
    out.resize((size_t)s.len);
    A0_REQUIRE(s.len == 0 || fread(out.data(), 1, (size_t)s.len, f) == (size_t)s.len, "%s: %s is truncated", who, path);
    A0_REQUIRE(!check_hash || ck_hash(out.data(), out.size()) == s.hash, "%s: %s: section %u is corrupt (hash)", who, path, tag);
    return A0_OK;
  }
};

// One checkpoint file, read and validated up to the BLOBS payload (where the file position stays).  a0_ckpt_load,
// a0_ckpt_merge and a0_ckpt_info share it, so every file is validated by the same code.
struct CkData {
  CkFile file;
  CkReader rd{nullptr, nullptr, 0, nullptr};
  CkHeader hd;
  std::vector<uint8_t> index_b, rec_b, leaf_b, sc_b, tail_b, user_b, frames_b;
  CkSection bs;
  std::vector<int64_t> tab;
  std::vector<uint64_t> fh;
  std::unique_ptr<a0_index_t, int (*)(a0_index_t*)> ix{nullptr, a0_ix_destroy};     // the file's index, validated
};

// the header: magic and version
int ck_open(const char* who, const char* path, CkData& d) {
  d.file.f = fopen(path, "rb");
  A0_REQUIRE(d.file.f, "%s: cannot open %s", who, path);
  struct stat sb;
  A0_REQUIRE(fstat(fileno(d.file.f), &sb) == 0, "%s: cannot stat %s", who, path);
  d.rd = CkReader{d.file.f, path, (int64_t)sb.st_size, who};
  CkHeader& hd = d.hd;
  A0_REQUIRE(fread(&hd, sizeof(hd), 1, d.file.f) == 1, "%s: %s is truncated (header)", who, path);
  A0_REQUIRE(memcmp(hd.magic, A0_CK_MAGIC, 8) == 0, "%s: %s is not a shard checkpoint (bad magic)", who, path);
  A0_REQUIRE(hd.version == A0_CK_VERSION && hd.zero == 0, "%s: %s has format version %u, this library reads %u", who, path,
             hd.version, A0_CK_VERSION);
  return A0_OK;
}

// a header read from a file that is not compared with a shard of the same shape: its sizes must at least fit the file
int ck_plausible(const char* who, CkData& d) {
  const CkHeader& hd = d.hd;
  A0_REQUIRE(hd.N >= 2 && hd.NF >= 8 && hd.F > 0 && hd.F % 16 == 0 && hd.n_step >= 1 && hd.n_step <= A0_MAX_NSTEP &&
                 hd.age_limit >= 0 && hd.N <= d.rd.size / 61,
             "%s: %s has an implausible header (N=%lld NF=%lld F=%lld n_step=%lld)", who, d.rd.path, (long long)hd.N,
             (long long)hd.NF, (long long)hd.F, (long long)hd.n_step);
  return A0_OK;
}

// the INDEX section into a scratch index of the header's parameters
int ck_read_index(CkData& d) {
  const CkHeader& hd = d.hd;
  int rc = d.rd.section(CK_INDEX, d.index_b);
  if (rc) return rc;
  a0_index_t* tix = nullptr;
  if ((rc = a0_ix_create(&tix, hd.N, hd.NF, (int32_t)hd.n_step, hd.age_limit))) return rc;
  d.ix.reset(tix);
  return a0_ix_deserialize(tix, d.index_b.data(), (int64_t)d.index_b.size());
}

// everything after the header, validated before anything is touched
int ck_read(const char* who, CkData& d) {
  const char* path = d.rd.path;
  FILE* f = d.file.f;
  CkReader& rd = d.rd;
  const int64_t N = d.hd.N, NF = d.hd.NF, F = d.hd.F;
  int rc;
  if ((rc = rd.section(CK_INDEX, d.index_b)) || (rc = rd.section(CK_RECORDS, d.rec_b)) || (rc = rd.section(CK_LEAVES, d.leaf_b)) ||
      (rc = rd.section(CK_SCALARS, d.sc_b)) || (rc = rd.section(CK_TAILS, d.tail_b)) || (rc = rd.section(CK_USER, d.user_b)) ||
      (rc = rd.section(CK_FRAMES, d.frames_b)))
    return rc;
  CkSection& bs = d.bs;
  A0_REQUIRE(fread(&bs, sizeof(bs), 1, f) == 1 && bs.tag == CK_BLOBS && bs.zero == 0, "%s: %s is truncated (blobs)", who, path);
  A0_REQUIRE(bs.len == (uint64_t)(rd.size - ftell(f)), "%s: %s has %lld blob bytes, the section says %llu", who, path,
             (long long)(rd.size - ftell(f)), (unsigned long long)bs.len);

  // the index, on a scratch copy
  a0_index_t* tix = nullptr;
  if ((rc = a0_ix_create(&tix, N, NF, (int32_t)d.hd.n_step, d.hd.age_limit))) return rc;
  d.ix.reset(tix);
  if ((rc = a0_ix_deserialize(tix, d.index_b.data(), (int64_t)d.index_b.size()))) return rc;
  int64_t ts[A0_IX_STATE_WORDS];
  a0_ix_state(tix, ts);
  const uint8_t* samp = a0_ix_sampleable(tix);
  const int64_t hq = ts[A0_IX_HEAD_Q], tq = ts[A0_IX_TAIL_Q], head_fs = ts[A0_IX_HEAD_FS];
  A0_REQUIRE(d.rec_b.size() == (size_t)N * (A0_SLOTS * 4 + sizeof(A0RecInfo)) && d.leaf_b.size() == (size_t)N * 4 && d.sc_b.size() == 32,
             "%s: %s: a section has the wrong size", who, path);
  const int32_t* slots = reinterpret_cast<const int32_t*>(d.rec_b.data());
  const A0RecInfo* info = reinterpret_cast<const A0RecInfo*>(d.rec_b.data() + (size_t)N * A0_SLOTS * 4);
  const int64_t resident = std::min(head_fs, NF);
  auto live = [&](int64_t pos) { return (pos - tq % N + N) % N < hq - tq; };
  for (int64_t q = tq; q < hq; ++q) {
    const int64_t pos = q % N;
    for (int j = 0; j < A0_SLOTS; ++j)
      A0_REQUIRE(slots[pos * A0_SLOTS + j] >= 0 && slots[pos * A0_SLOTS + j] < resident,
                 "%s: %s: record %lld names frame slot %d outside the resident window", who, path, (long long)pos,
                 slots[pos * A0_SLOTS + j]);
    const int32_t link = info[pos].link;
    A0_REQUIRE(link == -1 || (link >= 0 && link < N && live(link)), "%s: %s: record %lld links to %d, not a live record", who, path,
               (long long)pos, link);
  }
  const float* leaves = reinterpret_cast<const float*>(d.leaf_b.data());
  for (int64_t i = 0; i < N; ++i)
    A0_REQUIRE(std::isfinite(leaves[i]) && leaves[i] >= 0.0f && (samp[i] || leaves[i] == 0.0f),
               "%s: %s: priority %lld is %g (finite, >= 0, and 0 for a record that is not sampleable)", who, path, (long long)i,
               (double)leaves[i]);
  {
    float sc[4];
    int64_t sh;
    memcpy(sc, d.sc_b.data(), 16);
    memcpy(&sh, d.sc_b.data() + 24, 8);
    for (float x : sc) A0_REQUIRE(std::isfinite(x), "%s: %s: a saved scalar is not finite", who, path);
    A0_REQUIRE(sc[0] >= 0.0f && sh >= 0 && sh < N, "%s: %s: bad max_p or stride hint", who, path);
  }
  if ((rc = a0_ex_tails_check((int32_t)F, d.tail_b.data(), (int64_t)d.tail_b.size(), head_fs))) return rc;
  // the group table
  A0_REQUIRE(d.frames_b.size() >= 24, "%s: %s: frames section truncated", who, path);
  std::vector<int64_t>& tab = d.tab;
  tab.resize(3);
  memcpy(tab.data(), d.frames_b.data(), 24);
  const int64_t lo = std::max<int64_t>(0, head_fs - NF), nfr = head_fs - lo, G = (nfr + 7) / 8;
  A0_REQUIRE(tab[0] == lo && tab[1] == nfr && tab[2] == G && d.frames_b.size() == (size_t)(24 + 16 * G + 64 * G),
             "%s: %s: the frame table does not match the index", who, path);
  tab.resize((size_t)(3 + 2 * G));
  memcpy(tab.data(), d.frames_b.data(), (size_t)(3 + 2 * G) * 8);
  d.fh.resize((size_t)G * A0_SLOTS);
  memcpy(d.fh.data(), d.frames_b.data() + (size_t)(3 + 2 * G) * 8, d.fh.size() * 8);
  const int64_t maxlen = (int64_t)A0_SLOTS * F;
  uint64_t total = 0;
  for (int64_t g = 0; g < G; ++g) {
    A0_REQUIRE(tab[3 + 2 * g] == (lo + 8 * g) % NF && tab[4 + 2 * g] > 4 && tab[4 + 2 * g] <= maxlen,
               "%s: %s: frame group %lld has a bad table entry", who, path, (long long)g);
    total += (uint64_t)tab[4 + 2 * g];
  }
  A0_REQUIRE(total == bs.len, "%s: %s: the group table covers %llu blob bytes, the file holds %llu", who, path,
             (unsigned long long)total, (unsigned long long)bs.len);
  return A0_OK;
}
}  // namespace

// everything after the shard was touched: on failure, shard, index and tails go back to freshly created
static int ck_restore(a0_replay* h, a0_index_t* ix, a0_extend* ex, bool tails, CkData& d, cudaStream_t cs) {
  const int64_t N = h->N, F = h->F;
  CkReader& rd = d.rd;
  const std::vector<int64_t>& tab = d.tab;
  int rc = a0_rb_reset(h, cs);
  if (rc) return rc;
  if ((rc = a0_ix_deserialize(ix, d.index_b.data(), (int64_t)d.index_b.size()))) return rc;
  A0_CUDA(cudaMemcpyAsync(h->rec_slots, d.rec_b.data(), (size_t)N * A0_SLOTS * 4, cudaMemcpyHostToDevice, cs));
  A0_CUDA(cudaMemcpyAsync(h->rec_info, d.rec_b.data() + (size_t)N * A0_SLOTS * 4, (size_t)N * sizeof(A0RecInfo), cudaMemcpyHostToDevice, cs));
  {
    CkDev d_idx, d_val;
    std::vector<int64_t> idx((size_t)N);
    for (int64_t i = 0; i < N; ++i) idx[i] = i;
    A0_CUDA(cudaMalloc(&d_idx.p, (size_t)N * 8));
    A0_CUDA(cudaMalloc(&d_val.p, (size_t)N * 4));
    A0_CUDA(cudaMemcpyAsync(d_idx.p, idx.data(), (size_t)N * 8, cudaMemcpyHostToDevice, cs));
    A0_CUDA(cudaMemcpyAsync(d_val.p, d.leaf_b.data(), (size_t)N * 4, cudaMemcpyHostToDevice, cs));
    if ((rc = a0_pt_set(h, static_cast<const int64_t*>(d_idx.p), static_cast<const float*>(d_val.p), (int32_t)N, cs))) return rc;
    A0_CUDA(cudaStreamSynchronize(cs));
  }
  A0_CUDA(cudaMemcpyAsync(h->max_p, d.sc_b.data(), 4, cudaMemcpyHostToDevice, cs));
  A0_CUDA(cudaMemcpyAsync(h->dyn, d.sc_b.data() + 4, 12, cudaMemcpyHostToDevice, cs));
  A0_CUDA(cudaMemcpyAsync(h->counter + A0_RNG_CALL_WORD, d.sc_b.data() + 16, 8, cudaMemcpyHostToDevice, cs));
  memcpy(&h->stride_hint, d.sc_b.data() + 24, 8);
  A0_CUDA(cudaStreamSynchronize(cs));
  if (tails && (rc = a0_ex_tails_load(ex, d.tail_b.data(), (int64_t)d.tail_b.size(), cs))) return rc;
  // frames: K6a straight into the ring, batch by batch, every frame's hash compared with the saved one
  const int64_t lo = tab[0], nfr = tab[1], G = tab[2], head_fs = lo + nfr;
  CkHash bh;
  std::vector<uint8_t> blobs;
  std::vector<int64_t> lens;
  std::vector<unsigned long long> got((size_t)CK_BATCH * A0_SLOTS);
  for (int64_t g0 = 0; g0 < G; g0 += CK_BATCH) {
    const int32_t mb = (int32_t)std::min<int64_t>(CK_BATCH, G - g0);
    size_t bytes = 0;
    lens.resize((size_t)mb);
    for (int32_t i = 0; i < mb; ++i) { lens[i] = tab[4 + 2 * (g0 + i)]; bytes += (size_t)lens[i]; }
    blobs.resize(bytes);
    const auto a = ck_clock::now();
    A0_REQUIRE(fread(blobs.data(), 1, bytes, rd.f) == bytes, "a0_ckpt_load: %s is truncated (blobs)", rd.path);
    bh.update(blobs.data(), bytes);
    const auto b = ck_clock::now();
    const uint8_t* dec; const unsigned long long* dh; const int32_t* status;
    if ((rc = a0_ex_decode_dev(ex, blobs.data(), lens.data(), mb, cs, &dec, &dh, &status))) return rc;
    for (int32_t i = 0; i < mb; ++i)
      A0_REQUIRE(status[i] == 0, "a0_ckpt_load: %s: frame group %lld does not decode (status %d)", rd.path, (long long)(g0 + i), status[i]);
    A0_CUDA(cudaMemcpyAsync(got.data(), dh, (size_t)mb * A0_SLOTS * 8, cudaMemcpyDeviceToHost, cs));
    A0_CUDA(cudaStreamSynchronize(cs));
    A0_REQUIRE(memcmp(got.data(), d.fh.data() + (size_t)g0 * A0_SLOTS, (size_t)mb * A0_SLOTS * 8) == 0,
               "a0_ckpt_load: %s: a decoded frame of groups %lld.. differs from the saved one (hash)", rd.path, (long long)g0);
    const int64_t s0 = lo + 8 * g0, s1 = std::min<int64_t>(s0 + 8 * (int64_t)mb, head_fs);
    if ((rc = ck_ring_copy(h, const_cast<uint8_t*>(dec), s0, s1, true, cs))) return rc;
    A0_CUDA(cudaStreamSynchronize(cs));
    g_timing[2] += ck_us(a, b);
    g_timing[3] += ck_us(b, ck_clock::now());
    g_timing[5] += (double)bytes;
  }
  A0_REQUIRE(bh.final() == d.bs.hash && bh.total == d.bs.len, "a0_ckpt_load: %s: the frame blobs are corrupt (hash)", rd.path);
  g_timing[4] = (double)nfr * F;
  return A0_OK;
}

// a failure after the shard was touched: shard, index and tails back to freshly created
static int ck_reset_all(a0_replay* h, a0_index_t* ix, a0_extend* ex, cudaStream_t cs) {
  const std::string msg = a0_last_error();
  cudaStreamSynchronize(cs);
  a0_rb_reset(h, cs);
  cudaStreamSynchronize(cs);
  h->stride_hint = 0;
  a0_ix_clear(ix);
  if (ex) a0_ex_tails_clear(ex);
  a0_set_error("%s (the shard was reset to empty)", msg.c_str());
  return A0_EINVAL;
}

extern "C" int a0_ckpt_load(a0_replay_t* h, a0_index_t* ix, a0_extend_t* ex, const char* path, uint8_t* user_out,
                            int64_t user_cap, int64_t* user_len_out, a0_stream_t stream_) {
  A0_REQUIRE(h && ix && path, "a0_ckpt_load: NULL argument");
  A0_REQUIRE(!ex || a0_ex_shard(ex) == h, "a0_ckpt_load: the ingest handle belongs to another shard");
  const auto t0 = ck_clock::now();
  for (double& x : g_timing) x = 0.0;
  A0DeviceGuard guard(h->device);
  cudaStream_t cs = (cudaStream_t)stream_;
  cudaStreamCaptureStatus cst = cudaStreamCaptureStatusNone;
  A0_CUDA(cudaStreamIsCapturing(cs, &cst));
  A0_REQUIRE(cst == cudaStreamCaptureStatusNone, "a0_ckpt_load: the stream is being captured into a CUDA graph");
  A0_CUDA(cudaStreamSynchronize(cs));
  int64_t st[A0_IX_STATE_WORDS];
  int rc = a0_ix_state(ix, st);
  if (rc) return rc;
  A0_REQUIRE(st[A0_IX_REC_CAPACITY] == h->N && st[A0_IX_FRAME_CAPACITY] == h->NF, "a0_ckpt_load: index and shard capacities differ");
  CkData d;
  if ((rc = ck_open("a0_ckpt_load", path, d))) return rc;
  const CkHeader& hd = d.hd;
  const int64_t N = h->N, NF = h->NF, F = h->F;
  A0_REQUIRE(hd.N == N && hd.NF == NF && hd.F == F && hd.P == h->P && hd.n_step == st[A0_IX_NSTEP] && hd.age_limit == st[A0_IX_AGE_LIMIT],
             "a0_ckpt_load: %s holds a shard of N=%lld NF=%lld F=%lld n_step=%lld age_limit=%lld; this one has %lld %lld %lld %lld %lld",
             path, (long long)hd.N, (long long)hd.NF, (long long)hd.F, (long long)hd.n_step, (long long)hd.age_limit, (long long)N,
             (long long)NF, (long long)F, (long long)st[A0_IX_NSTEP], (long long)st[A0_IX_AGE_LIMIT]);
  if ((rc = ck_read("a0_ckpt_load", d))) return rc;
  A0_REQUIRE(d.user_b.empty() || (user_out && user_cap >= (int64_t)d.user_b.size()), "a0_ckpt_load: the user buffer needs %lld bytes",
             (long long)d.user_b.size());
  g_timing[1] = ck_us(t0, ck_clock::now());

  // ---- restore; from here a failure leaves everything as freshly created
  a0_extend_t* own = nullptr;
  if (!ex && (rc = a0_ex_create(&own, h, ix))) return rc;
  std::unique_ptr<a0_extend_t, int (*)(a0_extend_t*)> own_owner(own, a0_ex_destroy);
  rc = ck_restore(h, ix, ex ? ex : own, ex != nullptr, d, cs);
  if (rc) return ck_reset_all(h, ix, ex, cs);
  if (user_len_out) *user_len_out = (int64_t)d.user_b.size();
  if (!d.user_b.empty()) memcpy(user_out, d.user_b.data(), d.user_b.size());
  g_timing[0] = ck_us(t0, ck_clock::now());
  return A0_OK;
}

extern "C" int a0_ckpt_info(const char* path, int64_t* out8, int64_t* ids_out, int64_t ids_cap) {
  A0_REQUIRE(path && out8 && (ids_cap == 0 || ids_out), "a0_ckpt_info: NULL argument");
  CkData d;
  int rc = ck_open("a0_ckpt_info", path, d);
  if (rc || (rc = ck_plausible("a0_ckpt_info", d)) || (rc = ck_read_index(d))) return rc;
  int64_t st[A0_IX_STATE_WORDS];
  a0_ix_state(d.ix.get(), st);
  std::vector<int64_t> ids;
  a0_ix_stream_ids(d.ix.get(), ids);
  const int64_t v[8] = {d.hd.N, d.hd.NF, d.hd.F, d.hd.n_step, d.hd.age_limit, st[A0_IX_HEAD_Q] - st[A0_IX_TAIL_Q], st[A0_IX_TOP],
                        (int64_t)ids.size()};
  memcpy(out8, v, sizeof(v));
  A0_REQUIRE(ids_cap >= (int64_t)ids.size(), "a0_ckpt_info: %s has %lld streams, the id buffer takes %lld", path, (long long)ids.size(),
             (long long)ids_cap);
  if (!ids.empty()) memcpy(ids_out, ids.data(), ids.size() * 8);
  return A0_OK;
}

// ---- a0_ckpt_merge ---------------------------------------------------------------------------------------------
// the placed frames of one file: its BLOBS section read once, sequentially, and hashed whole; of each batch of
// CK_BATCH groups only those holding a placed frame are decoded (K6a into the ingest scratch), their hashes checked,
// and the placed frames copied to their target slots by K1's source-indexed copy
static int ck_place_file(a0_replay* h, a0_extend* ex, CkData& d, const std::vector<std::pair<int64_t, int32_t>>& place,
                         cudaStream_t cs, cudaEvent_t e0, cudaEvent_t e1) {
  const std::vector<int64_t>& tab = d.tab;
  const int64_t lo = tab[0], G = tab[2];
  CkHash bh;
  std::vector<uint8_t> raw, blobs;
  std::vector<int64_t> lens, src;
  std::vector<int32_t> pos, gsel;
  std::vector<unsigned long long> got((size_t)CK_BATCH * A0_SLOTS);
  size_t pi = 0;             // place: (source seq, target slot), ascending source seq
  for (int64_t g0 = 0; g0 < G; g0 += CK_BATCH) {
    const int32_t mb = (int32_t)std::min<int64_t>(CK_BATCH, G - g0);
    std::vector<size_t> off((size_t)mb + 1, 0);
    for (int32_t i = 0; i < mb; ++i) off[i + 1] = off[i] + (size_t)tab[4 + 2 * (g0 + i)];
    raw.resize(off[mb]);
    const auto a = ck_clock::now();
    A0_REQUIRE(fread(raw.data(), 1, raw.size(), d.rd.f) == raw.size(), "a0_ckpt_merge: %s is truncated (blobs)", d.rd.path);
    bh.update(raw.data(), raw.size());
    g_timing[7] += ck_us(a, ck_clock::now());
    // the groups of this batch that hold a placed frame
    gsel.clear(); blobs.clear(); lens.clear(); src.clear(); pos.clear();
    const int64_t s_end = lo + 8 * (g0 + mb);
    while (pi < place.size() && place[pi].first < s_end) {
      const int64_t g = (place[pi].first - lo) / 8 - g0;
      if (gsel.empty() || gsel.back() != (int32_t)g) {
        gsel.push_back((int32_t)g);
        blobs.insert(blobs.end(), raw.begin() + off[g], raw.begin() + off[g + 1]);
        lens.push_back((int64_t)(off[g + 1] - off[g]));
      }
      src.push_back((int64_t)(gsel.size() - 1) * A0_SLOTS + (place[pi].first - lo) % 8);
      pos.push_back(place[pi].second);
      ++pi;
    }
    if (gsel.empty()) continue;
    const int32_t nd = (int32_t)gsel.size();
    A0_CUDA(cudaEventRecord(e0, cs));
    const uint8_t* dec; const unsigned long long* dh; const int32_t* status;
    int rc = a0_ex_decode_dev(ex, blobs.data(), lens.data(), nd, cs, &dec, &dh, &status);
    if (rc) return rc;
    for (int32_t i = 0; i < nd; ++i)
      A0_REQUIRE(status[i] == 0, "a0_ckpt_merge: %s: frame group %lld does not decode (status %d)", d.rd.path, (long long)(g0 + gsel[i]),
                 status[i]);
    A0_CUDA(cudaMemcpyAsync(got.data(), dh, (size_t)nd * A0_SLOTS * 8, cudaMemcpyDeviceToHost, cs));
    A0_CUDA(cudaStreamSynchronize(cs));
    for (int32_t i = 0; i < nd; ++i)
      A0_REQUIRE(memcmp(got.data() + (size_t)i * A0_SLOTS, d.fh.data() + (size_t)(g0 + gsel[i]) * A0_SLOTS, A0_SLOTS * 8) == 0,
                 "a0_ckpt_merge: %s: a decoded frame of group %lld differs from the saved one (hash)", d.rd.path, (long long)(g0 + gsel[i]));
    a0_plan_t plan = {0, (int32_t)pos.size(), 0, pos.data(), nullptr, nullptr};
    const A0Dyn none = {nullptr, 0.0f, 0.0f, 0.0f};
    if ((rc = a0_ingest_plan_impl(h, &plan, dec, src.data(), A0_INGEST_FRAMES_ON_DEVICE, 0.0f, (a0_stream_t)cs, none))) return rc;
    A0_CUDA(cudaEventRecord(e1, cs));
    A0_CUDA(cudaStreamSynchronize(cs));
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, e0, e1);
    g_timing[3] += ms * 1e3;
    g_timing[5] += (double)nd * A0_SLOTS * h->F;
    g_timing[6] += (double)pos.size() * h->F;
  }
  A0_REQUIRE(pi == place.size(), "a0_ckpt_merge: %s: a placed frame lies outside the file's frame groups", d.rd.path);
  A0_REQUIRE(bh.final() == d.bs.hash && bh.total == d.bs.len, "a0_ckpt_merge: %s: the frame blobs are corrupt (hash)", d.rd.path);
  return A0_OK;
}

extern "C" int a0_ckpt_merge(a0_replay_t* h, a0_index_t* ix, a0_extend_t* ex, const char* const* paths, int32_t k,
                             const int64_t* map_old, const int64_t* map_new, const int64_t* map_len, uint8_t* user_out,
                             int64_t user_cap, int64_t* user_len_out, a0_stream_t stream_) {
  A0_REQUIRE(h && ix && paths && k >= 1 && map_len, "a0_ckpt_merge: NULL argument");
  A0_REQUIRE(!ex || a0_ex_shard(ex) == h, "a0_ckpt_merge: the ingest handle belongs to another shard");
  const auto t0 = ck_clock::now();
  for (double& x : g_timing) x = 0.0;
  A0DeviceGuard guard(h->device);
  cudaStream_t cs = (cudaStream_t)stream_;
  cudaStreamCaptureStatus cst = cudaStreamCaptureStatusNone;
  A0_CUDA(cudaStreamIsCapturing(cs, &cst));
  A0_REQUIRE(cst == cudaStreamCaptureStatusNone, "a0_ckpt_merge: the stream is being captured into a CUDA graph");
  A0_CUDA(cudaStreamSynchronize(cs));
  { int frc = a0_check_fault(h, "a0_ckpt_merge"); if (frc) return frc; }
  int64_t st[A0_IX_STATE_WORDS];
  int rc = a0_ix_state(ix, st);
  if (rc) return rc;
  A0_REQUIRE(st[A0_IX_REC_CAPACITY] == h->N && st[A0_IX_FRAME_CAPACITY] == h->NF, "a0_ckpt_merge: index and shard capacities differ");
  // ---- every file validated before anything is touched
  std::vector<std::unique_ptr<CkData>> files;
  int64_t user_total = 0;
  for (int32_t j = 0; j < k; ++j) {
    A0_REQUIRE(paths[j], "a0_ckpt_merge: path %d is NULL", j);
    files.emplace_back(new CkData());
    CkData& d = *files.back();
    if ((rc = ck_open("a0_ckpt_merge", paths[j], d)) || (rc = ck_plausible("a0_ckpt_merge", d))) return rc;
    A0_REQUIRE(d.hd.F == h->F && d.hd.n_step == st[A0_IX_NSTEP],
               "a0_ckpt_merge: %s holds frames of F=%lld gathered with n_step=%lld; this shard has F=%lld n_step=%lld", paths[j],
               (long long)d.hd.F, (long long)d.hd.n_step, (long long)h->F, (long long)st[A0_IX_NSTEP]);
    if ((rc = ck_read("a0_ckpt_merge", d))) return rc;
    user_total += (int64_t)d.user_b.size();
  }
  A0_REQUIRE(user_total == 0 || (user_out && user_cap >= user_total), "a0_ckpt_merge: the user buffer needs %lld bytes",
             (long long)user_total);
  g_timing[1] = ck_us(t0, ck_clock::now());
  // ---- the merge plan on a scratch index of the target's parameters
  const auto t1 = ck_clock::now();
  a0_index_t* tix = nullptr;
  if ((rc = a0_ix_create(&tix, h->N, h->NF, (int32_t)st[A0_IX_NSTEP], st[A0_IX_AGE_LIMIT]))) return rc;
  std::unique_ptr<a0_index_t, int (*)(a0_index_t*)> tix_owner(tix, a0_ix_destroy);
  std::vector<a0_index_t*> six;
  std::vector<const uint8_t*> recs;
  std::vector<const float*> leaves;
  std::vector<int64_t> tail_count, tail_ids, tail_seq;
  const size_t tail_each = 8 + 64 + 8 + (size_t)A0_SLOTS * h->F + 64;      // a0_ex_tails_check verified the layout
  for (auto& dp : files) {
    six.push_back(dp->ix.get());
    recs.push_back(dp->rec_b.data());
    leaves.push_back(reinterpret_cast<const float*>(dp->leaf_b.data()));
    int64_t cnt;
    memcpy(&cnt, dp->tail_b.data(), 8);
    tail_count.push_back(cnt);
    for (int64_t e = 0; e < cnt; ++e) {
      const uint8_t* p = dp->tail_b.data() + 8 + (size_t)e * tail_each;
      int64_t v[1 + A0_SLOTS];
      memcpy(v, p, sizeof(v));
      tail_ids.push_back(v[0]);
      tail_seq.insert(tail_seq.end(), v + 1, v + 1 + A0_SLOTS);
    }
  }
  std::vector<uint8_t> rec_out((size_t)h->N * (A0_SLOTS * 4 + sizeof(A0RecInfo)));
  std::vector<float> leaf_out((size_t)h->N);
  a0_merge_t mg;
  if ((rc = a0_ix_merge(tix, k, six.data(), recs.data(), leaves.data(), map_old, map_new, map_len, tail_count.data(),
                        tail_ids.data(), tail_seq.data(), rec_out.data(), leaf_out.data(), &mg)))
    return rc;
  std::vector<uint8_t> index_b;
  {
    int64_t len = 0;
    a0_ix_serialize(tix, nullptr, 0, &len);
    index_b.resize((size_t)len);
    if ((rc = a0_ix_serialize(tix, index_b.data(), len, &len))) return rc;
  }
  // scalars: max_p and the call counter the maxima over the files, dyn {top, file 0's beta, 0}
  float max_p = 0.0f, dyn[3];
  uint64_t calls = 0;
  for (auto& dp : files) {
    float mp;
    uint64_t c;
    memcpy(&mp, dp->sc_b.data(), 4);
    memcpy(&c, dp->sc_b.data() + 16, 8);
    max_p = std::max(max_p, mp);
    calls = std::max(calls, c);
  }
  int64_t tst[A0_IX_STATE_WORDS];
  a0_ix_state(tix, tst);
  dyn[0] = (float)tst[A0_IX_TOP];
  memcpy(&dyn[1], files[0]->sc_b.data() + 8, 4);
  dyn[2] = 0.0f;
  // tails: new ids and remapped seqs, the rest of each entry as saved
  std::vector<uint8_t> tails_b(8 + (size_t)mg.n_tail * tail_each);
  memcpy(tails_b.data(), &mg.n_tail, 8);
  for (int64_t i = 0; i < mg.n_tail; ++i) {
    const int64_t* o = mg.tails + i * (3 + A0_SLOTS);
    uint8_t* p = tails_b.data() + 8 + (size_t)i * tail_each;
    memcpy(p, files[(size_t)o[1]]->tail_b.data() + 8 + (size_t)o[2] * tail_each, tail_each);
    memcpy(p, &o[0], 8);
    memcpy(p + 8, o + 3, 64);
  }
  // placements per file, ascending source seq
  std::vector<std::vector<std::pair<int64_t, int32_t>>> place((size_t)k);
  for (int64_t i = 0; i < mg.n_place; ++i) place[(size_t)mg.place[3 * i]].push_back({mg.place[3 * i + 1], (int32_t)mg.place[3 * i + 2]});
  for (auto& p : place) std::sort(p.begin(), p.end());
  g_timing[2] = ck_us(t1, ck_clock::now());

  // ---- from here a failure leaves everything as freshly created
  a0_extend_t* own = nullptr;
  if (!ex && (rc = a0_ex_create(&own, h, ix))) return rc;
  std::unique_ptr<a0_extend_t, int (*)(a0_extend_t*)> own_owner(own, a0_ex_destroy);
  a0_extend* dx = ex ? ex : own;
  CkEvents ev;
  rc = [&]() -> int {
    const auto t2 = ck_clock::now();
    const int64_t N = h->N;
    int r = a0_rb_reset(h, cs);
    if (r) return r;
    if ((r = a0_ix_deserialize(ix, index_b.data(), (int64_t)index_b.size()))) return r;
    A0_CUDA(cudaMemcpyAsync(h->rec_slots, rec_out.data(), (size_t)N * A0_SLOTS * 4, cudaMemcpyHostToDevice, cs));
    A0_CUDA(cudaMemcpyAsync(h->rec_info, rec_out.data() + (size_t)N * A0_SLOTS * 4, (size_t)N * sizeof(A0RecInfo), cudaMemcpyHostToDevice, cs));
    {
      CkDev d_idx, d_val;
      std::vector<int64_t> idx((size_t)N);
      for (int64_t i = 0; i < N; ++i) idx[i] = i;
      A0_CUDA(cudaMalloc(&d_idx.p, (size_t)N * 8));
      A0_CUDA(cudaMalloc(&d_val.p, (size_t)N * 4));
      A0_CUDA(cudaMemcpyAsync(d_idx.p, idx.data(), (size_t)N * 8, cudaMemcpyHostToDevice, cs));
      A0_CUDA(cudaMemcpyAsync(d_val.p, leaf_out.data(), (size_t)N * 4, cudaMemcpyHostToDevice, cs));
      if ((r = a0_pt_set(h, static_cast<const int64_t*>(d_idx.p), static_cast<const float*>(d_val.p), (int32_t)N, cs))) return r;
      A0_CUDA(cudaStreamSynchronize(cs));
    }
    A0_CUDA(cudaMemcpyAsync(h->max_p, &max_p, 4, cudaMemcpyHostToDevice, cs));
    A0_CUDA(cudaMemcpyAsync(h->dyn, dyn, 12, cudaMemcpyHostToDevice, cs));
    A0_CUDA(cudaMemcpyAsync(h->counter + A0_RNG_CALL_WORD, &calls, 8, cudaMemcpyHostToDevice, cs));
    h->stride_hint = mg.stride_hint;
    A0_CUDA(cudaStreamSynchronize(cs));
    if (ex && (r = a0_ex_tails_load(ex, tails_b.data(), (int64_t)tails_b.size(), cs))) return r;
    g_timing[4] = ck_us(t2, ck_clock::now());
    for (auto& x : ev.e) A0_CUDA(cudaEventCreate(&x));
    for (int32_t j = 0; j < k; ++j)
      if ((r = ck_place_file(h, dx, *files[(size_t)j], place[(size_t)j], cs, ev.e[0], ev.e[1]))) return r;
    return A0_OK;
  }();
  if (rc) return ck_reset_all(h, ix, ex, cs);
  int64_t at = 0;
  for (int32_t j = 0; j < k; ++j) {
    const std::vector<uint8_t>& u = files[(size_t)j]->user_b;
    if (user_len_out) user_len_out[j] = (int64_t)u.size();
    if (!u.empty()) memcpy(user_out + at, u.data(), u.size());
    at += (int64_t)u.size();
  }
  g_timing[0] = ck_us(t0, ck_clock::now());
  return A0_OK;
}

extern "C" int a0_ckpt_last_timing(double* out8) {
  A0_REQUIRE(out8, "a0_ckpt_last_timing: NULL argument");
  for (int i = 0; i < 8; ++i) out8[i] = g_timing[i];
  return A0_OK;
}
