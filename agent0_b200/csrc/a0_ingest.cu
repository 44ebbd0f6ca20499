// Host side of the replay shard: the ring index (which incoming frames are new, where they go,
// which records become sampleable, which must be evicted) and the staged ingest that executes an
// index plan on the device (one pinned H2D copy, then K2b marks and K1 append).
//
// Replaces the host bookkeeping of the reference's ReplayDataset.extend (agent0/deepq/replay.py:45-53:
// deque.extend + top + tail priorities) and the actor-side n-step tracker's "entry k-n+1 is emitted
// at step k" rule (agent0/deepq/agent.py:64-73).  The rules are those of agent0_b200/ring_index.py,
// which stays as the executable specification: tests/test_ring_index.py runs both implementations
// on the same streams and requires identical plans.
//
//   * sequence numbers are monotone int64; ring position = seq % capacity;
//   * a frame seq f is resident while f >= head_fs - NF;
//   * evict record q iff its slot is being reused or fs_at_append[q] - age_limit < head_fs - NF
//     (conservative and monotone, so the live records are the window [tail_q, head_q));
//   * with n-step gathering a record becomes sampleable when its (n-1)-th successor in the same
//     stream has been appended.
#include <algorithm>
#include <new>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "a0_common.cuh"

struct A0Stream {
  int32_t last_pos = -1;
  int64_t last_seq = -1;
  std::vector<int64_t> pending;   // appended, waiting for their (n-1)-th successor
  int64_t stack[A0_STACK] = {0, 0, 0, 0};
  bool has_stack = false;
};

struct a0_index {
  int64_t N, NF, n, age_limit;
  int64_t head_q = 0, tail_q = 0, head_fs = 0, top = 0;
  std::vector<int64_t> fs_at_append;
  std::vector<uint8_t> sampleable;
  std::unordered_map<int64_t, A0Stream> streams;
  std::unordered_set<int64_t> stale;
  // plan storage, valid until the next call
  std::vector<int32_t> new_frame_pos, rec_meta, marks;
  std::vector<int32_t> order;
  std::vector<int64_t> fs8, ready;
  // a0_ix_merge output, valid until the next merge into this index
  std::vector<int64_t> merge_place, merge_rmap, merge_tails;

  int64_t max_chunk() const {
    const int64_t a = N / 2, b = (NF - 2 * age_limit) / (2 * A0_SLOTS);
    return std::max<int64_t>(1, std::min(a, b));
  }
};

extern "C" int a0_ix_create(a0_index_t** out, int64_t rec_capacity, int64_t frame_capacity, int32_t n_step,
                            int64_t age_limit) {
  A0_REQUIRE(out != nullptr, "a0_ix_create: out is NULL");
  A0_REQUIRE(rec_capacity >= 2 && frame_capacity >= 8, "a0_ix_create: capacities too small");
  A0_REQUIRE(n_step >= 1 && n_step <= A0_MAX_NSTEP, "a0_ix_create: n_step %d outside [1,%d]", n_step, A0_MAX_NSTEP);
  if (age_limit < 0) age_limit = std::max<int64_t>(8, std::min<int64_t>(32768, frame_capacity / 8));
  A0_REQUIRE(frame_capacity > 2 * age_limit, "a0_ix_create: frame ring (%lld) too small for the age limit (%lld)",
             (long long)frame_capacity, (long long)age_limit);
  a0_index* ix = new (std::nothrow) a0_index();
  if (!ix) { a0_set_error("a0_ix_create: out of host memory"); return A0_ENOMEM; }
  ix->N = rec_capacity; ix->NF = frame_capacity; ix->n = n_step; ix->age_limit = age_limit;
  ix->fs_at_append.assign((size_t)rec_capacity, 0);
  ix->sampleable.assign((size_t)rec_capacity, 0);
  *out = ix;
  return A0_OK;
}

extern "C" int a0_ix_destroy(a0_index_t* ix) {
  delete ix;
  return A0_OK;
}

extern "C" int a0_ix_state(a0_index_t* ix, int64_t* out) {
  A0_REQUIRE(ix && out, "a0_ix_state: NULL argument");
  out[A0_IX_HEAD_Q] = ix->head_q; out[A0_IX_TAIL_Q] = ix->tail_q; out[A0_IX_HEAD_FS] = ix->head_fs;
  out[A0_IX_TOP] = ix->top; out[A0_IX_REC_CAPACITY] = ix->N; out[A0_IX_FRAME_CAPACITY] = ix->NF;
  out[A0_IX_NSTEP] = ix->n; out[A0_IX_AGE_LIMIT] = ix->age_limit; out[A0_IX_MAX_CHUNK] = ix->max_chunk();
  return A0_OK;
}

extern "C" const uint8_t* a0_ix_sampleable(a0_index_t* ix) { return ix ? ix->sampleable.data() : nullptr; }

extern "C" int a0_ix_set_stack(a0_index_t* ix, int64_t stream, const int64_t* seq4) {
  A0_REQUIRE(ix && seq4, "a0_ix_set_stack: NULL argument");
  A0Stream& st = ix->streams[stream];
  for (int j = 0; j < A0_STACK; ++j) st.stack[j] = seq4[j];
  st.has_stack = true;
  return A0_OK;
}

extern "C" int a0_ix_get_stack(a0_index_t* ix, int64_t stream, int64_t* seq4) {
  A0_REQUIRE(ix && seq4, "a0_ix_get_stack: NULL argument");
  auto it = ix->streams.find(stream);
  if (it == ix->streams.end() || !it->second.has_stack) return 1;   // no stack yet (not an error)
  for (int j = 0; j < A0_STACK; ++j) seq4[j] = it->second.stack[j];
  return A0_OK;
}

// Groups of equal stream id in ascending id order, original order inside a group.
static void a0_group_by_stream(a0_index* ix, const int64_t* stream, int32_t m) {
  ix->order.resize((size_t)m);
  for (int32_t i = 0; i < m; ++i) ix->order[i] = i;
  std::stable_sort(ix->order.begin(), ix->order.end(), [&](int32_t a, int32_t b) { return stream[a] < stream[b]; });
}

extern "C" int a0_ix_resolve_shift(a0_index_t* ix, const int64_t* stream, const int64_t* n_new, int32_t m,
                                   int64_t* fs8_out) {
  A0_REQUIRE(ix && (m == 0 || (stream && n_new && fs8_out)), "a0_ix_resolve_shift: NULL argument");
  // new frames are numbered in (transition, frame) order from head_fs
  int64_t next = ix->head_fs;
  std::vector<int64_t>& off = ix->ready;     // scratch
  off.resize((size_t)m);
  for (int32_t i = 0; i < m; ++i) {
    A0_REQUIRE(n_new[i] >= 0 && n_new[i] <= A0_STACK, "a0_ix_resolve_shift: n_new[%d] = %lld outside [0,4]", i, (long long)n_new[i]);
    off[i] = next;
    next += n_new[i];
  }
  for (int32_t i = 0; i < m; ++i) {
    auto it = ix->streams.find(stream[i]);
    A0_REQUIRE(it != ix->streams.end() && it->second.has_stack,
               "a0_ix_resolve_shift: stream %lld has no observation stack yet (reset_streams first)", (long long)stream[i]);
  }
  // per stream, in commit order: obs stack = current stack, next stack = it shifted by the new frames
  for (int32_t i = 0; i < m; ++i) {
    A0Stream& st = ix->streams.find(stream[i])->second;
    int64_t* row = fs8_out + (size_t)i * A0_SLOTS;
    int64_t win[2 * A0_STACK];
    for (int j = 0; j < A0_STACK; ++j) { row[j] = st.stack[j]; win[j] = st.stack[j]; }
    const int c = (int)n_new[i];
    for (int j = 0; j < c; ++j) win[A0_STACK + j] = off[i] + j;
    for (int j = 0; j < A0_STACK; ++j) { row[A0_STACK + j] = win[c + j]; st.stack[j] = win[c + j]; }
  }
  return A0_OK;
}

extern "C" int a0_ix_plan(a0_index_t* ix, const int64_t* stream, const int64_t* fs8, int32_t m, int32_t n_new,
                          const int64_t* action, const double* reward, const uint8_t* done, a0_plan_t* out) {
  A0_REQUIRE(ix && out, "a0_ix_plan: NULL argument");
  A0_REQUIRE(m >= 0 && n_new >= 0, "a0_ix_plan: negative count");
  A0_REQUIRE(m == 0 || (stream && fs8 && action && reward && done), "a0_ix_plan: NULL array");
  A0_REQUIRE(m <= ix->max_chunk(), "a0_ix_plan: append of %d transitions is too large for the ring (max %lld): split it",
             m, (long long)ix->max_chunk());
  const int64_t N = ix->N, NF = ix->NF, n = ix->n;
  const int64_t q0 = ix->head_q;
  const int64_t new_head_fs = ix->head_fs + n_new, new_head_q = q0 + m;
  ix->marks.clear();
  // a record whose frames are already older than the age limit (an idle stream that resumes) can
  // never be a sampling start: the eviction bound below would not cover it
  for (int32_t i = 0; i < m; ++i) {
    int64_t mn = fs8[(size_t)i * A0_SLOTS];
    for (int j = 1; j < A0_SLOTS; ++j) mn = std::min(mn, fs8[(size_t)i * A0_SLOTS + j]);
    if (ix->head_fs - mn > ix->age_limit) ix->stale.insert(q0 + i);
  }
  // ---- evictions: a prefix of the live window ---------------------------------------------------
  const int64_t thr = new_head_fs - NF;
  while (ix->tail_q < q0) {
    const int64_t w = ix->tail_q, wp = w % N;
    if (!((w < new_head_q - N) || (ix->fs_at_append[wp] - ix->age_limit < thr))) break;
    ix->top -= ix->sampleable[wp];
    ix->sampleable[wp] = 0;
    ix->marks.push_back(~(int32_t)wp);
    ix->tail_q++;
  }
  // ---- links and sampleability, stream by stream ------------------------------------------------
  ix->rec_meta.resize((size_t)m * A0_REC_META_I32);
  int32_t* meta = ix->rec_meta.data();
  for (int32_t i = 0; i < m; ++i) {
    int32_t* mt = meta + (size_t)i * A0_REC_META_I32;
    mt[0] = (int32_t)((q0 + i) % N);
    mt[1] = -1;
    mt[2] = -1;
  }
  a0_group_by_stream(ix, stream, m);
  ix->ready.clear();
  bool any_newly = false;
  for (int32_t g0 = 0; g0 < m;) {
    int32_t g1 = g0;
    const int64_t sid = stream[ix->order[g0]];
    while (g1 < m && stream[ix->order[g1]] == sid) ++g1;
    A0Stream& st = ix->streams[sid];
    const int32_t first = ix->order[g0], last = ix->order[g1 - 1];
    if (st.last_seq >= std::max(ix->tail_q, q0 - N)) meta[(size_t)first * A0_REC_META_I32 + 1] = st.last_pos;
    for (int32_t g = g0; g + 1 < g1; ++g)
      meta[(size_t)ix->order[g] * A0_REC_META_I32 + 2] = meta[(size_t)ix->order[g + 1] * A0_REC_META_I32];
    if (n == 1) {
      for (int32_t g = g0; g < g1; ++g) ix->ready.push_back(q0 + ix->order[g]);
      any_newly = true;
    } else {
      for (int32_t g = g0; g < g1; ++g) st.pending.push_back(q0 + ix->order[g]);
      const int64_t nready = (int64_t)st.pending.size() - (n - 1);
      if (nready > 0) {
        ix->ready.insert(ix->ready.end(), st.pending.begin(), st.pending.begin() + nready);
        st.pending.erase(st.pending.begin(), st.pending.begin() + nready);
        any_newly = true;
      }
    }
    st.last_pos = meta[(size_t)last * A0_REC_META_I32];
    st.last_seq = q0 + last;
    g0 = g1;
  }
  for (int32_t i = 0; i < m; ++i) ix->fs_at_append[(size_t)((q0 + i) % N)] = ix->head_fs;
  ix->head_q = new_head_q;
  ix->head_fs = new_head_fs;
  if (any_newly) {
    const bool had_stale = !ix->stale.empty();
    std::unordered_set<int64_t> hit;
    for (int64_t r : ix->ready) {
      if (r < ix->tail_q) continue;                 // evicted before it ever became sampleable
      if (had_stale && ix->stale.count(r)) { hit.insert(r); continue; }
      const int64_t rp = r % N;
      ix->sampleable[rp] = 1;
      ix->top += 1;
      ix->marks.push_back((int32_t)rp);
    }
    if (had_stale) {
      for (auto it = ix->stale.begin(); it != ix->stale.end();) {
        if (*it < ix->tail_q || hit.count(*it)) it = ix->stale.erase(it);
        else ++it;
      }
    }
  }
  // ---- record metadata ----------------------------------------------------------------------------
  for (int32_t i = 0; i < m; ++i) {
    int32_t* mt = meta + (size_t)i * A0_REC_META_I32;
    mt[3] = (int32_t)(action[i] & 0x7fffffff) | (done[i] ? (int32_t)0x80000000 : 0);
    for (int j = 0; j < A0_SLOTS; ++j) {
      int64_t f = fs8[(size_t)i * A0_SLOTS + j] % NF;
      if (f < 0) f += NF;
      mt[4 + j] = (int32_t)f;
    }
    memcpy(mt + 12, reward + i, sizeof(double));
  }
  ix->new_frame_pos.resize((size_t)n_new);
  for (int32_t j = 0; j < n_new; ++j) ix->new_frame_pos[j] = (int32_t)((new_head_fs - n_new + j) % NF);
  out->m = m; out->n_new = n_new; out->n_marks = (int32_t)ix->marks.size();
  out->new_frame_pos = ix->new_frame_pos.data();
  out->rec_meta = ix->rec_meta.data();
  out->marks = ix->marks.data();
  return A0_OK;
}

// ------------------------------------------------------------------------------------------------
// content de-duplication for the reference-compatible ingest
// ------------------------------------------------------------------------------------------------
// The reference's entries are self-contained 8-frame blobs concat(st, st_next) (agent.py:78-81), 7 of
// which normally repeat frames of the same env's previous entry.  A frame is matched -- by a 64-bit
// hash first, then by full byte comparison, so a match is always bit-exact -- against the 8 frames of
// the stream's previous entry and the earlier frames of its own entry; unmatched frames are new.
// Specification: ring_index.ContentDeduper (numpy, 260 ms per 1280-transition extend); this is the
// same rule at memory speed (tests/test_ring_index.py drives both and requires identical output).
struct A0Tail {
  std::vector<uint8_t> frames;      // owned copy of the last entry's 8 frames (filled when a call ends)
  const uint8_t* cur = nullptr;     // the last entry's frames during a call (caller's buffer or `frames`)
  int64_t seq[A0_SLOTS];
  uint64_t hash[A0_SLOTS];
  bool valid = false;
};
struct a0_dedupe {
  int32_t F;
  std::unordered_map<int64_t, A0Tail> tail;
};

static inline uint64_t a0_frame_hash(const uint8_t* p, int32_t F) {
  // four independent multiply-rotate lanes over 64-bit words (frames are multiples of 16 bytes)
  uint64_t h0 = 0x9E3779B97F4A7C15ull, h1 = 0xC2B2AE3D27D4EB4Full, h2 = 0x165667B19E3779F9ull, h3 = 0x27D4EB2F165667C5ull;
  const int n = F / 8;
  int i = 0;
  for (; i + 4 <= n; i += 4) {
    uint64_t w0, w1, w2, w3;
    memcpy(&w0, p + 8 * i, 8); memcpy(&w1, p + 8 * i + 8, 8); memcpy(&w2, p + 8 * i + 16, 8); memcpy(&w3, p + 8 * i + 24, 8);
    h0 = (h0 ^ w0) * 0x9FB21C651E98DF25ull; h0 = (h0 << 29) | (h0 >> 35);
    h1 = (h1 ^ w1) * 0x9FB21C651E98DF25ull; h1 = (h1 << 29) | (h1 >> 35);
    h2 = (h2 ^ w2) * 0x9FB21C651E98DF25ull; h2 = (h2 << 29) | (h2 >> 35);
    h3 = (h3 ^ w3) * 0x9FB21C651E98DF25ull; h3 = (h3 << 29) | (h3 >> 35);
  }
  for (; i < n; ++i) {
    uint64_t w;
    memcpy(&w, p + 8 * i, 8);
    h0 = (h0 ^ w) * 0x9FB21C651E98DF25ull; h0 = (h0 << 29) | (h0 >> 35);
  }
  uint64_t h = h0 ^ (h1 * 3) ^ (h2 * 5) ^ (h3 * 7);
  h ^= h >> 32; h *= 0xD6E8FEB86659FD93ull; h ^= h >> 32;
  return h;
}

extern "C" int a0_dd_create(a0_dedupe_t** out, int32_t frame_bytes) {
  A0_REQUIRE(out != nullptr, "a0_dd_create: out is NULL");
  A0_REQUIRE(frame_bytes > 0 && frame_bytes % 8 == 0, "a0_dd_create: frame_bytes %d must be a positive multiple of 8", frame_bytes);
  a0_dedupe* dd = new (std::nothrow) a0_dedupe();
  if (!dd) { a0_set_error("a0_dd_create: out of host memory"); return A0_ENOMEM; }
  dd->F = frame_bytes;
  *out = dd;
  return A0_OK;
}

extern "C" int a0_dd_destroy(a0_dedupe_t* dd) {
  delete dd;
  return A0_OK;
}

extern "C" int a0_dd_resolve(a0_dedupe_t* dd, a0_index_t* ix, const int64_t* stream, const uint8_t* frames, int32_t m,
                             int64_t* fs8_out, int64_t* new_src_out, int32_t* n_new_out) {
  A0_REQUIRE(dd && ix && n_new_out, "a0_dd_resolve: NULL handle");
  A0_REQUIRE(m >= 0, "a0_dd_resolve: negative count");
  A0_REQUIRE(m == 0 || (stream && frames && fs8_out && new_src_out), "a0_dd_resolve: NULL array");
  const size_t F = (size_t)dd->F;
  int64_t next_fs = ix->head_fs;
  const int64_t resident_from = ix->head_fs - ix->NF;     // frame_resident(f): f >= head_fs - NF
  int32_t n_new = 0;
  std::vector<int64_t> touched;
  for (int32_t t = 0; t < m; ++t) {
    A0Tail& tl = dd->tail[stream[t]];
    const uint8_t* ent = frames + (size_t)t * A0_SLOTS * F;
    int64_t* row = fs8_out + (size_t)t * A0_SLOTS;
    uint64_t hs[A0_SLOTS];
    for (int j = 0; j < A0_SLOTS; ++j) hs[j] = a0_frame_hash(ent + j * F, dd->F);
    const uint8_t* prev = tl.valid ? (tl.cur ? tl.cur : tl.frames.data()) : nullptr;
    for (int j = 0; j < A0_SLOTS; ++j) {
      int64_t hit = -1;
      if (prev) {
        for (int c = 0; c < A0_SLOTS && hit < 0; ++c)
          if (tl.hash[c] == hs[j] && next_fs - tl.seq[c] < ix->age_limit && tl.seq[c] >= resident_from &&
              memcmp(prev + c * F, ent + j * F, F) == 0)
            hit = tl.seq[c];
      }
      for (int c = 0; c < j && hit < 0; ++c)
        if (hs[c] == hs[j] && memcmp(ent + c * F, ent + j * F, F) == 0) hit = row[c];
      if (hit < 0) {
        hit = next_fs++;
        new_src_out[n_new++] = (int64_t)t * A0_SLOTS + j;
      }
      row[j] = hit;
    }
    if (!tl.valid || tl.cur == nullptr) touched.push_back(stream[t]);
    tl.cur = ent;
    tl.valid = true;
    for (int j = 0; j < A0_SLOTS; ++j) { tl.seq[j] = row[j]; tl.hash[j] = hs[j]; }
  }
  // private copies of the stream tails: the caller may reuse its buffer after the call
  for (int64_t sid : touched) {
    A0Tail& tl = dd->tail[sid];
    if (tl.cur) {
      tl.frames.assign(tl.cur, tl.cur + A0_SLOTS * F);
      tl.cur = nullptr;
    }
  }
  *n_new_out = n_new;
  return A0_OK;
}

// ------------------------------------------------------------------------------------------------
// staged execution of a plan on the device
// ------------------------------------------------------------------------------------------------
static inline size_t a0_up256(size_t x) { return (x + 255) & ~(size_t)255; }

static int a0_stage_reserve(a0_replay* h, int turn, size_t bytes) {
  A0Staging& s = h->staging[turn];
  if (s.event) A0_CUDA(cudaEventSynchronize(s.event));     // the previous use of this buffer has been consumed
  if (s.capacity >= bytes) return A0_OK;
  const size_t cap = std::max<size_t>(bytes + bytes / 4, (size_t)1 << 20);
  if (s.host) { cudaFreeHost(s.host); s.host = nullptr; }
  if (s.dev) { cudaFree(s.dev); s.dev = nullptr; }
  s.capacity = 0;
  A0_CUDA(cudaMallocHost((void**)&s.host, cap));
  A0_CUDA(cudaMalloc((void**)&s.dev, cap));
  if (!s.event) A0_CUDA(cudaEventCreateWithFlags(&s.event, cudaEventDisableTiming));
  if (!s.copied) A0_CUDA(cudaEventCreateWithFlags(&s.copied, cudaEventDisableTiming));
  s.capacity = cap;
  return A0_OK;
}

// dyn.dyn != NULL: the launch that appends also publishes {top, beta, sum_offset} for the sampler
// (what a0_rb_set_dynamic would otherwise launch a kernel for).
int a0_ingest_plan_impl(a0_replay_t* h, const a0_plan_t* plan, const uint8_t* frames,
                        const int64_t* new_frame_src, int32_t flags, float alpha, a0_stream_t stream_,
                        const A0Dyn& dyn) {
  A0_REQUIRE(h && plan, "a0_rb_ingest_plan: NULL argument");
  const int32_t n_new = plan->n_new, m = plan->m, k = plan->n_marks;
  if (n_new == 0 && m == 0 && k == 0) {
    if (!dyn.dyn) return A0_OK;
    A0DeviceGuard guard(h->device);
    return a0_append_launch(h, nullptr, nullptr, nullptr, 0, nullptr, 0, dyn, (cudaStream_t)stream_);
  }
  A0_REQUIRE(n_new == 0 || frames, "a0_rb_ingest_plan: frames is NULL");
  const bool on_device = flags & A0_INGEST_FRAMES_ON_DEVICE;
  const bool pinned = flags & A0_INGEST_FRAMES_PINNED;
  A0_REQUIRE(!pinned || new_frame_src == nullptr, "a0_rb_ingest_plan: pinned frames must already be in allocation order");
  // device frames + new_frame_src: the picks are uploaded as int32 and K1 reads frames[src[j]] (a0_ex_extend)
  const bool dev_pick = on_device && new_frame_src != nullptr && n_new > 0;
  A0DeviceGuard guard(h->device);
  cudaStream_t stream = (cudaStream_t)stream_;
  const size_t F = (size_t)h->F;
  // successor stride of this append (rec_meta: {pos, link_from, ...}): the same for every record when
  // the actors step in lockstep; K3 uses it as a (verified) guess, see a0_spec_fetch
  if (m > 0) {
    int64_t stride = -1;
    for (int32_t i = 0; i < m && stride != 0; ++i) {
      const int32_t* mt = plan->rec_meta + (size_t)i * A0_REC_META_I32;
      if (mt[1] < 0) continue;                         // first record of its stream
      int64_t dlt = (int64_t)mt[0] - mt[1];
      if (dlt <= 0) dlt += h->N;
      stride = (stride < 0 || stride == dlt) ? dlt : 0;
    }
    if (stride >= 0) h->stride_hint = stride;
  }
  const bool stage_frames = n_new > 0 && !on_device && !pinned;
  size_t sec[6];
  sec[0] = 0;
  sec[1] = sec[0] + a0_up256(on_device ? 0 : (size_t)n_new * F);
  sec[2] = sec[1] + a0_up256((size_t)n_new * 4);
  sec[3] = sec[2] + a0_up256((size_t)m * A0_REC_META_I32 * 4);
  sec[5] = sec[3] + a0_up256((size_t)k * 4);
  sec[4] = sec[5] + a0_up256(dev_pick ? (size_t)n_new * 4 : 0);     // sec[4] stays "end of the upload"; [sec[5], sec[4]) = picks
  const int turn = h->staging_turn;
  h->staging_turn ^= 1;
  int rc = a0_stage_reserve(h, turn, sec[4]);
  if (rc) return rc;
  A0Staging& s = h->staging[turn];
  if (stage_frames) {
    for (int32_t j = 0; j < n_new; ++j) {
      const size_t src = new_frame_src ? (size_t)new_frame_src[j] : (size_t)j;
      memcpy(s.host + sec[0] + (size_t)j * F, frames + src * F, F);
    }
  }
  if (n_new) memcpy(s.host + sec[1], plan->new_frame_pos, (size_t)n_new * 4);
  if (m) memcpy(s.host + sec[2], plan->rec_meta, (size_t)m * A0_REC_META_I32 * 4);
  if (k) memcpy(s.host + sec[3], plan->marks, (size_t)k * 4);
  if (dev_pick) {
    int32_t* pick = reinterpret_cast<int32_t*>(s.host + sec[5]);
    for (int32_t j = 0; j < n_new; ++j) pick[j] = (int32_t)new_frame_src[j];
  }
  // The H2D copies may run on the shard's own copy stream, so that they overlap whatever `stream`
  // is still executing (the previous step's kernels); `stream` then waits for them.  The staging
  // buffer they fill was released by a0_stage_reserve (its last consumer has finished).
  cudaStream_t cs = stream;
  if (flags & A0_INGEST_COPY_STREAM) {
    if (!h->copy_stream) A0_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    cs = h->copy_stream;
  }
  if (stage_frames) {
    A0_CUDA(cudaMemcpyAsync(s.dev, s.host, sec[4], cudaMemcpyHostToDevice, cs));
  } else {
    if (pinned && n_new) A0_CUDA(cudaMemcpyAsync(s.dev + sec[0], frames, (size_t)n_new * F, cudaMemcpyHostToDevice, cs));
    A0_CUDA(cudaMemcpyAsync(s.dev + sec[1], s.host + sec[1], sec[4] - sec[1], cudaMemcpyHostToDevice, cs));
  }
  if (cs != stream) {
    A0_CUDA(cudaEventRecord(s.copied, cs));
    A0_CUDA(cudaStreamWaitEvent(stream, s.copied, 0));
  }
  const uint8_t* dev_frames = n_new ? (on_device ? frames : s.dev + sec[0]) : nullptr;
  const int32_t* dev_pos = n_new ? (const int32_t*)(s.dev + sec[1]) : nullptr;
  const int32_t* dev_meta = m ? (const int32_t*)(s.dev + sec[2]) : nullptr;
  const int32_t* dev_pick_idx = dev_pick ? (const int32_t*)(s.dev + sec[5]) : nullptr;
  A0_REQUIRE(((uintptr_t)dev_frames & 15) == 0, "a0_rb_ingest_plan: device frames must be 16-byte aligned");
  // A step-sized append (a few hundred marks, tens of frames) goes out as ONE launch: marks and
  // append touch disjoint state.  Bulk fills keep the two launches (cluster marks, 128-thread K1 CTAs).
  rc = (k && a0_option_fused_ingest()) ? a0_launch_mark_append(h, (const int32_t*)(s.dev + sec[3]), k, alpha, dev_frames, dev_pos, dev_pick_idx, n_new,
                                                               dev_meta, m, dyn, stream)
                                       : A0_NOFIT;
  if (rc == A0_NOFIT) {
    if (k) {
      rc = a0_pt_mark(h, (const int32_t*)(s.dev + sec[3]), k, alpha, stream_);
      if (rc) return rc;
    }
    rc = a0_append_launch(h, dev_frames, dev_pos, dev_pick_idx, n_new, dev_meta, m, dyn, stream);
  }
  if (rc) return rc;
  A0_CUDA(cudaEventRecord(s.event, stream));
  return A0_OK;
}

extern "C" int a0_rb_ingest_plan(a0_replay_t* h, const a0_plan_t* plan, const uint8_t* frames,
                                 const int64_t* new_frame_src, int32_t flags, float alpha, a0_stream_t stream) {
  const A0Dyn none = {nullptr, 0.0f, 0.0f, 0.0f};
  return a0_ingest_plan_impl(h, plan, frames, new_frame_src, flags, alpha, stream, none);
}

// beta == NULL: nothing is published.  Otherwise the LAST chunk's append publishes
// {ix->top after the append, *beta, compat_sum ? N - top : 0}.
static int a0_ingest_steps_impl(a0_replay_t* h, a0_index_t* ix, const int64_t* stream, const int64_t* n_new,
                                const uint8_t* new_frames, int32_t flags, const int64_t* action, const double* reward,
                                const uint8_t* done, int32_t m, float alpha, const float* beta, int32_t compat_sum,
                                a0_stream_t cuda_stream, const char* who) {
  A0_REQUIRE(h && ix, "%s: NULL handle", who);
  A0_REQUIRE(m >= 0, "%s: negative count", who);
  A0_REQUIRE(ix->N == h->N && ix->NF == h->NF, "%s: index and shard capacities differ", who);
  { int frc = a0_check_fault(h, who); if (frc) return frc; }
  const size_t F = (size_t)h->F;
  const int64_t step = ix->max_chunk();
  size_t frame_off = 0;
  A0Dyn dyn = {nullptr, 0.0f, 0.0f, 0.0f};
  for (int64_t lo = 0; lo < m || (lo == 0 && beta); lo += step) {
    const int32_t cnt = (int32_t)std::max<int64_t>(0, std::min<int64_t>(step, m - lo));
    ix->fs8.resize((size_t)cnt * A0_SLOTS);
    int rc = a0_ix_resolve_shift(ix, stream + lo, n_new + lo, cnt, ix->fs8.data());
    if (rc) return rc;
    int64_t total_new = 0;
    for (int32_t i = 0; i < cnt; ++i) total_new += n_new[lo + i];
    a0_plan_t plan;
    rc = a0_ix_plan(ix, stream + lo, ix->fs8.data(), cnt, (int32_t)total_new, action + lo, reward + lo, done + lo, &plan);
    if (rc) return rc;
    if (beta && lo + step >= m) {
      dyn.dyn = h->dyn;
      dyn.top = (float)ix->top;
      dyn.beta = *beta;
      dyn.sum_offset = compat_sum ? (float)(ix->N - ix->top) : 0.0f;
    }
    rc = a0_ingest_plan_impl(h, &plan, new_frames ? new_frames + frame_off * F : nullptr, nullptr, flags, alpha, cuda_stream,
                             dyn);
    if (rc) return rc;
    frame_off += (size_t)total_new;
    if (m == 0) break;
  }
  return A0_OK;
}

extern "C" int a0_rb_ingest_steps(a0_replay_t* h, a0_index_t* ix, const int64_t* stream, const int64_t* n_new,
                                  const uint8_t* new_frames, int32_t flags, const int64_t* action,
                                  const double* reward, const uint8_t* done, int32_t m, float alpha,
                                  a0_stream_t cuda_stream) {
  return a0_ingest_steps_impl(h, ix, stream, n_new, new_frames, flags, action, reward, done, m, alpha, nullptr, 0,
                              cuda_stream, "a0_rb_ingest_steps");
}

extern "C" int a0_rb_ingest_steps_dyn(a0_replay_t* h, a0_index_t* ix, const int64_t* stream, const int64_t* n_new,
                                      const uint8_t* new_frames, int32_t flags, const int64_t* action,
                                      const double* reward, const uint8_t* done, int32_t m, float alpha, float beta,
                                      int32_t compat_sum, a0_stream_t cuda_stream) {
  return a0_ingest_steps_impl(h, ix, stream, n_new, new_frames, flags, action, reward, done, m, alpha, &beta, compat_sum,
                              cuda_stream, "a0_rb_ingest_steps_dyn");
}

// ------------------------------------------------------------------------------------------------
// serialization of the ring index (checkpoints: a0_ckpt_save / a0_ckpt_load)
// ------------------------------------------------------------------------------------------------
// Layout, little-endian i64 words unless noted: magic "A0IX" u32, version u32, N, NF, n_step, age_limit, head_q,
// tail_q, head_fs, top, fs_at_append[N], sampleable u8[N], streams, per stream in ascending id order {id, last_pos,
// last_seq, has_stack, stack[4], pending count, pending[...]}, stale count, stale[...] ascending.
static constexpr uint32_t A0_IX_MAGIC = 0x58493041u;   // "A0IX"
static constexpr uint32_t A0_IX_VERSION = 1;

namespace {
struct A0IxWriter {
  uint8_t* out; int64_t cap, len = 0;
  void put(const void* p, size_t k) { if (out && len + (int64_t)k <= cap) memcpy(out + len, p, k); len += (int64_t)k; }
  void i64(int64_t v) { put(&v, 8); }
};
struct A0IxReader {
  const uint8_t* p; int64_t len, at = 0;
  bool get(void* d, size_t k) { if (at + (int64_t)k > len) return false; memcpy(d, p + at, k); at += (int64_t)k; return true; }
  bool i64(int64_t& v) { return get(&v, 8); }
};
}  // namespace

extern "C" int a0_ix_serialize(a0_index_t* ix, uint8_t* out, int64_t cap, int64_t* len_out) {
  A0_REQUIRE(ix && len_out, "a0_ix_serialize: NULL argument");
  A0IxWriter w{out, out ? cap : 0};
  const uint32_t hdr[2] = {A0_IX_MAGIC, A0_IX_VERSION};
  w.put(hdr, 8);
  for (int64_t v : {ix->N, ix->NF, ix->n, ix->age_limit, ix->head_q, ix->tail_q, ix->head_fs, ix->top}) w.i64(v);
  w.put(ix->fs_at_append.data(), (size_t)ix->N * 8);
  w.put(ix->sampleable.data(), (size_t)ix->N);
  std::vector<int64_t> ids;
  for (auto& kv : ix->streams) ids.push_back(kv.first);
  std::sort(ids.begin(), ids.end());
  w.i64((int64_t)ids.size());
  for (int64_t id : ids) {
    const A0Stream& st = ix->streams[id];
    w.i64(id); w.i64(st.last_pos); w.i64(st.last_seq); w.i64(st.has_stack ? 1 : 0);
    for (int j = 0; j < A0_STACK; ++j) w.i64(st.stack[j]);
    w.i64((int64_t)st.pending.size());
    w.put(st.pending.data(), st.pending.size() * 8);
  }
  std::vector<int64_t> stale(ix->stale.begin(), ix->stale.end());
  std::sort(stale.begin(), stale.end());
  w.i64((int64_t)stale.size());
  w.put(stale.data(), stale.size() * 8);
  *len_out = w.len;
  A0_REQUIRE(out && cap >= w.len, "a0_ix_serialize: the index needs %lld bytes", (long long)w.len);
  return A0_OK;
}

extern "C" int a0_ix_deserialize(a0_index_t* ix, const uint8_t* blob, int64_t len) {
  A0_REQUIRE(ix && blob && len >= 0, "a0_ix_deserialize: NULL argument");
  A0IxReader r{blob, len};
  uint32_t hdr[2];
  A0_REQUIRE(r.get(hdr, 8) && hdr[0] == A0_IX_MAGIC && hdr[1] == A0_IX_VERSION, "a0_ix_deserialize: not a ring index (bad magic or version)");
  int64_t N, NF, n, age, hq, tq, hfs, top;
  A0_REQUIRE(r.i64(N) && r.i64(NF) && r.i64(n) && r.i64(age) && r.i64(hq) && r.i64(tq) && r.i64(hfs) && r.i64(top),
             "a0_ix_deserialize: truncated header");
  A0_REQUIRE(N == ix->N && NF == ix->NF && n == ix->n && age == ix->age_limit,
             "a0_ix_deserialize: saved for N=%lld NF=%lld n_step=%lld age_limit=%lld, this index has %lld %lld %lld %lld",
             (long long)N, (long long)NF, (long long)n, (long long)age, (long long)ix->N, (long long)ix->NF, (long long)ix->n,
             (long long)ix->age_limit);
  A0_REQUIRE(0 <= tq && tq <= hq && hq - tq <= N && hfs >= 0 && 0 <= top && top <= hq - tq,
             "a0_ix_deserialize: inconsistent counters (head_q %lld, tail_q %lld, head_fs %lld, top %lld)", (long long)hq,
             (long long)tq, (long long)hfs, (long long)top);
  a0_index t;
  t.N = N; t.NF = NF; t.n = n; t.age_limit = age; t.head_q = hq; t.tail_q = tq; t.head_fs = hfs; t.top = top;
  t.fs_at_append.resize((size_t)N);
  t.sampleable.resize((size_t)N);
  A0_REQUIRE(r.get(t.fs_at_append.data(), (size_t)N * 8) && r.get(t.sampleable.data(), (size_t)N), "a0_ix_deserialize: truncated");
  int64_t count = 0;
  for (int64_t q = 0; q < N; ++q) {
    const bool live = (q - tq % N + N) % N < hq - tq;      // ring position of a record in [tail_q, head_q)
    A0_REQUIRE(t.sampleable[q] <= 1 && (live || t.sampleable[q] == 0), "a0_ix_deserialize: record %lld is sampleable but not live",
               (long long)q);
    A0_REQUIRE(!live || (t.fs_at_append[q] >= 0 && t.fs_at_append[q] <= hfs), "a0_ix_deserialize: record %lld has a bad frame key",
               (long long)q);
    count += t.sampleable[q];
  }
  A0_REQUIRE(count == top, "a0_ix_deserialize: %lld sampleable records, top says %lld", (long long)count, (long long)top);
  int64_t ns;
  A0_REQUIRE(r.i64(ns) && ns >= 0 && ns <= (len - r.at) / 72, "a0_ix_deserialize: truncated stream table");
  int64_t prev_id = 0;
  for (int64_t i = 0; i < ns; ++i) {
    int64_t id, lp, ls, hs, k;
    A0Stream st;
    A0_REQUIRE(r.i64(id) && r.i64(lp) && r.i64(ls) && r.i64(hs) && r.get(st.stack, sizeof(st.stack)) && r.i64(k),
               "a0_ix_deserialize: truncated stream %lld", (long long)i);
    A0_REQUIRE(i == 0 || id > prev_id, "a0_ix_deserialize: stream ids out of order");
    prev_id = id;
    A0_REQUIRE(ls >= -1 && ls < hq && (ls < 0 ? lp == -1 : lp == ls % N) && (hs == 0 || hs == 1),
               "a0_ix_deserialize: stream %lld has an inconsistent last record", (long long)id);
    A0_REQUIRE(k >= 0 && k < n && k <= (len - r.at) / 8, "a0_ix_deserialize: stream %lld has %lld pending records", (long long)id,
               (long long)k);
    st.pending.resize((size_t)k);
    A0_REQUIRE(r.get(st.pending.data(), (size_t)k * 8), "a0_ix_deserialize: truncated");
    for (int64_t j = 0; j < k; ++j)
      A0_REQUIRE(st.pending[j] >= 0 && st.pending[j] < hq && (j == 0 || st.pending[j] > st.pending[j - 1]),
                 "a0_ix_deserialize: stream %lld has a bad pending record", (long long)id);
    st.last_pos = (int32_t)lp; st.last_seq = ls; st.has_stack = hs != 0;
    t.streams.emplace(id, std::move(st));
  }
  int64_t nst;
  A0_REQUIRE(r.i64(nst) && nst >= 0 && nst <= (len - r.at) / 8, "a0_ix_deserialize: truncated stale set");
  for (int64_t i = 0; i < nst; ++i) {
    int64_t s;
    r.i64(s);
    A0_REQUIRE(s >= 0 && s < hq, "a0_ix_deserialize: stale record %lld out of range", (long long)s);
    t.stale.insert(s);
  }
  A0_REQUIRE(r.at == len, "a0_ix_deserialize: %lld trailing bytes", (long long)(len - r.at));
  ix->head_q = t.head_q; ix->tail_q = t.tail_q; ix->head_fs = t.head_fs; ix->top = t.top;
  ix->fs_at_append.swap(t.fs_at_append);
  // in place: a0_ix_sampleable hands out a pointer into this vector
  memcpy(ix->sampleable.data(), t.sampleable.data(), (size_t)N);
  ix->streams.swap(t.streams);
  ix->stale.swap(t.stale);
  return A0_OK;
}

// back to the state of a0_ix_create (a checkpoint load that failed after it touched the index)
void a0_ix_clear(a0_index* ix) {
  ix->head_q = ix->tail_q = ix->head_fs = ix->top = 0;
  std::fill(ix->fs_at_append.begin(), ix->fs_at_append.end(), 0);
  std::fill(ix->sampleable.begin(), ix->sampleable.end(), 0);
  ix->streams.clear();
  ix->stale.clear();
}

// ------------------------------------------------------------------------------------------------
// a0_ix_merge: k shard checkpoints into one empty index of any capacity (rules: ring_index.merge, which stays the
// executable specification; tests/test_ix_merge.py requires identical output)
// ------------------------------------------------------------------------------------------------
namespace {
struct MergeRec {
  int64_t age_key;        // q - head_q of its file (oldest first)
  int32_t file;
  int64_t q, pos, stream;
  bool stale;
};
}  // namespace

void a0_ix_stream_ids(a0_index* ix, std::vector<int64_t>& out) {
  out.clear();
  for (auto& kv : ix->streams) out.push_back(kv.first);
  std::sort(out.begin(), out.end());
}

extern "C" int a0_ix_merge(a0_index_t* t, int32_t k, a0_index_t* const* src, const uint8_t* const* records,
                           const float* const* leaves, const int64_t* map_old, const int64_t* map_new, const int64_t* map_len,
                           const int64_t* tail_count, const int64_t* tail_ids, const int64_t* tail_seq, uint8_t* records_out,
                           float* leaves_out, a0_merge_t* out) {
  A0_REQUIRE(t && k >= 1 && src && records && leaves && map_len && records_out && leaves_out && out, "a0_ix_merge: NULL argument");
  A0_REQUIRE(t->head_q == 0 && t->head_fs == 0 && t->streams.empty(), "a0_ix_merge: the target index is not empty");
  for (int32_t j = 0; j < k; ++j) {
    A0_REQUIRE(src[j] && records[j] && leaves[j], "a0_ix_merge: NULL source %d", j);
    A0_REQUIRE(src[j]->n == t->n, "a0_ix_merge: file %d gathers n_step=%lld, the target %lld", j, (long long)src[j]->n,
               (long long)t->n);
  }
  // ---- rule 5: stream maps (old id -> new id per file), collisions refused before anything changes
  std::vector<std::unordered_map<int64_t, int64_t>> maps((size_t)k);
  {
    std::vector<std::unordered_set<int64_t>> present((size_t)k);
    int64_t S = 0;
    const int64_t* tid = tail_ids;
    for (int32_t j = 0; j < k; ++j) {
      for (auto& kv : src[j]->streams) present[j].insert(kv.first);
      const int64_t nt = tail_count ? tail_count[j] : 0;
      for (int64_t e = 0; e < nt; ++e) present[j].insert(tid[e]);
      tid += nt;
      for (int64_t id : present[j]) S = std::max(S, id + 1);
    }
    const int64_t* mo = map_old;
    const int64_t* mn = map_new;
    std::unordered_set<int64_t> seen;
    for (int32_t j = 0; j < k; ++j) {
      if (map_len[j] < 0) {
        for (int64_t id : present[j]) maps[j][id] = id + (int64_t)j * S;
      } else {
        A0_REQUIRE(map_len[j] == 0 || (mo && mn), "a0_ix_merge: NULL stream map");
        for (int64_t e = 0; e < map_len[j]; ++e)
          if (present[j].count(mo[e])) maps[j][mo[e]] = mn[e];
        mo += map_len[j];
        mn += map_len[j];
      }
      for (auto& kv : maps[j]) {
        A0_REQUIRE(seen.insert(kv.second).second, "a0_ix_merge: two kept streams would both become stream %lld", (long long)kv.second);
      }
    }
  }
  // ---- rule 1: live records of the kept streams; a record's stream by walking the links backwards
  std::vector<MergeRec> recs;
  for (int32_t j = 0; j < k; ++j) {
    const a0_index* s = src[j];
    const int64_t N = s->N, hq = s->head_q, tq = s->tail_q;
    const A0RecInfo* info = reinterpret_cast<const A0RecInfo*>(records[j] + (size_t)N * A0_SLOTS * 4);
    std::vector<int64_t> pred((size_t)N, -1), owner((size_t)N, INT64_MIN);
    for (int64_t q = tq; q < hq; ++q) {
      const int32_t link = info[q % N].link;
      if (link < 0) continue;
      A0_REQUIRE(link < N && pred[link] < 0, "a0_ix_merge: file %d: two records link to record %d", j, link);
      pred[link] = q % N;
    }
    std::unordered_set<int64_t> pending;
    int64_t reached = 0;
    for (auto& kv : s->streams) {
      for (int64_t p : kv.second.pending) pending.insert(p);
      for (int64_t p = kv.second.last_seq >= tq ? kv.second.last_pos : -1; p >= 0; p = pred[p]) {
        A0_REQUIRE(owner[p] == INT64_MIN && reached < hq - tq, "a0_ix_merge: file %d: record %lld is reached twice", j, (long long)p);
        owner[p] = kv.first;
        ++reached;
      }
    }
    A0_REQUIRE(reached == hq - tq, "a0_ix_merge: file %d: %lld live records belong to no stream", j, (long long)(hq - tq - reached));
    for (int64_t q = tq; q < hq; ++q) {
      const int64_t pos = q % N;
      auto it = maps[j].find(owner[pos]);
      if (it == maps[j].end()) continue;
      const bool stale = !s->sampleable[pos] && (!pending.count(q) || s->stale.count(q));
      recs.push_back({q - hq, j, q, pos, it->second, stale});
    }
  }
  // ---- rule 2: oldest first, ties by file
  std::stable_sort(recs.begin(), recs.end(), [](const MergeRec& a, const MergeRec& b) {
    return a.age_key != b.age_key ? a.age_key < b.age_key : a.file < b.file;
  });
  // ---- rule 3: the target is fed the merged sequence through a0_ix_plan
  struct Ident {
    int32_t file;
    int64_t seq;
    bool operator==(const Ident& o) const { return file == o.file && seq == o.seq; }
  };
  struct IdentHash {
    size_t operator()(const Ident& x) const { return std::hash<int64_t>()(x.seq * 131 + x.file); }
  };
  std::unordered_map<Ident, int64_t, IdentHash> newest;
  struct Alloc { int64_t t; int32_t file; int64_t seq; };
  std::vector<Alloc> alloc;
  auto resolve = [&](const Ident& id, int64_t& next_fs, int64_t hf) -> int64_t {
    auto it = newest.find(id);
    if (it != newest.end() && it->second >= hf - t->NF && next_fs - it->second < t->age_limit) return it->second;
    const int64_t f = next_fs++;
    newest[id] = f;
    alloc.push_back({f, id.file, id.seq});
    return f;
  };
  auto src_seq = [&](int32_t j, int64_t pos) {
    const a0_index* s = src[j];
    const int64_t lo = std::max<int64_t>(0, s->head_fs - s->NF);
    return lo + ((pos - lo % s->NF) % s->NF + s->NF) % s->NF;
  };
  const int64_t N2 = t->N;
  int32_t* slots2 = reinterpret_cast<int32_t*>(records_out);
  A0RecInfo* info2 = reinterpret_cast<A0RecInfo*>(records_out + (size_t)N2 * A0_SLOTS * 4);
  memset(slots2, 0, (size_t)N2 * A0_SLOTS * 4);
  memset(info2, 0xff, (size_t)N2 * sizeof(A0RecInfo));
  int64_t hint = 0;
  const int64_t chunk = t->max_chunk();
  std::vector<int64_t> stream, fs8, action, tq_of(recs.size());
  std::vector<double> reward;
  std::vector<uint8_t> done;
  for (size_t c0 = 0; c0 < recs.size(); c0 += (size_t)chunk) {
    const int32_t m = (int32_t)std::min<size_t>((size_t)chunk, recs.size() - c0);
    const int64_t hf = t->head_fs, q0 = t->head_q;
    int64_t next_fs = hf;
    stream.resize((size_t)m); fs8.resize((size_t)m * A0_SLOTS); action.resize((size_t)m); reward.resize((size_t)m);
    done.resize((size_t)m);
    for (int32_t i = 0; i < m; ++i) {
      const MergeRec& r = recs[c0 + i];
      const int32_t* sl = reinterpret_cast<const int32_t*>(records[r.file]) + (size_t)r.pos * A0_SLOTS;
      for (int c = 0; c < A0_SLOTS; ++c) fs8[(size_t)i * A0_SLOTS + c] = resolve({r.file, src_seq(r.file, sl[c])}, next_fs, hf);
      const A0RecInfo& in = reinterpret_cast<const A0RecInfo*>(records[r.file] + (size_t)src[r.file]->N * A0_SLOTS * 4)[r.pos];
      stream[i] = r.stream;
      action[i] = in.action_done & 0x7fffffff;
      done[i] = in.action_done < 0;
      reward[i] = in.reward;
      if (r.stale) t->stale.insert(q0 + i);
      tq_of[c0 + i] = q0 + i;
    }
    a0_plan_t plan;
    int rc = a0_ix_plan(t, stream.data(), fs8.data(), m, (int32_t)(next_fs - hf), action.data(), reward.data(), done.data(), &plan);
    if (rc) return rc;
    int64_t stride = -1;
    for (int32_t i = 0; i < m; ++i) {
      const int32_t* mt = plan.rec_meta + (size_t)i * A0_REC_META_I32;
      const int32_t pos = mt[0];
      memcpy(slots2 + (size_t)pos * A0_SLOTS, mt + 4, A0_SLOTS * 4);
      memcpy(&info2[pos].reward, mt + 12, 8);
      info2[pos].action_done = mt[3];
      info2[pos].link = mt[2];
      if (mt[1] >= 0) info2[mt[1]].link = pos;
      if (stride == 0 || mt[1] < 0) continue;
      int64_t dlt = (int64_t)mt[0] - mt[1];
      if (dlt <= 0) dlt += N2;
      stride = (stride < 0 || stride == dlt) ? dlt : 0;
    }
    if (stride >= 0) hint = stride;
  }
  // ---- rule 6: stacks (frames-only plans, ascending new id), then the tails
  struct Todo { int64_t id; int32_t file; const int64_t* stack; };
  std::vector<Todo> todo;
  for (int32_t j = 0; j < k; ++j) {
    const a0_index* s = src[j];
    const int64_t lo = std::max<int64_t>(0, s->head_fs - s->NF);
    for (auto& kv : s->streams) {
      auto it = maps[j].find(kv.first);
      if (it == maps[j].end() || !kv.second.has_stack) continue;
      bool ok = true;
      for (int c = 0; c < A0_STACK; ++c) ok = ok && kv.second.stack[c] >= lo && kv.second.stack[c] < s->head_fs;
      if (ok) todo.push_back({it->second, j, kv.second.stack});
    }
  }
  std::sort(todo.begin(), todo.end(), [](const Todo& a, const Todo& b) { return a.id < b.id; });
  const size_t per = (size_t)std::max<int64_t>(1, 2 * chunk);
  for (size_t g0 = 0; g0 < todo.size(); g0 += per) {
    const size_t g1 = std::min(todo.size(), g0 + per);
    const int64_t hf = t->head_fs;
    int64_t next_fs = hf;
    std::vector<int64_t> seqs;
    for (size_t g = g0; g < g1; ++g)
      for (int c = 0; c < A0_STACK; ++c) seqs.push_back(resolve({todo[g].file, todo[g].stack[c]}, next_fs, hf));
    a0_plan_t plan;
    int rc = a0_ix_plan(t, nullptr, nullptr, 0, (int32_t)(next_fs - hf), nullptr, nullptr, nullptr, &plan);
    if (rc) return rc;
    for (size_t g = g0; g < g1; ++g) {
      A0Stream& st = t->streams[todo[g].id];
      for (int c = 0; c < A0_STACK; ++c) st.stack[c] = seqs[(g - g0) * A0_STACK + c];
      st.has_stack = true;
    }
  }
  const int64_t final_lo = t->head_fs - t->NF;
  t->merge_tails.clear();
  {
    struct TailOut { int64_t id; int32_t file; int64_t entry; int64_t seq[A0_SLOTS]; };
    std::vector<TailOut> tl;
    const int64_t* tid = tail_ids;
    const int64_t* tsq = tail_seq;
    for (int32_t j = 0; j < k; ++j) {
      const int64_t nt = tail_count ? tail_count[j] : 0;
      for (int64_t e = 0; e < nt; ++e) {
        auto it = maps[j].find(tid[e]);
        if (it == maps[j].end()) continue;
        TailOut o{it->second, j, e, {}};
        bool ok = true;
        for (int c = 0; c < A0_SLOTS && ok; ++c) {
          auto f = newest.find({j, tsq[e * A0_SLOTS + c]});
          ok = f != newest.end() && f->second >= final_lo;
          if (ok) o.seq[c] = f->second;
        }
        if (ok) tl.push_back(o);
      }
      tid += nt;
      tsq += nt * A0_SLOTS;
    }
    std::sort(tl.begin(), tl.end(), [](const TailOut& a, const TailOut& b) { return a.id < b.id; });
    for (const TailOut& o : tl) {
      t->merge_tails.push_back(o.id); t->merge_tails.push_back(o.file); t->merge_tails.push_back(o.entry);
      t->merge_tails.insert(t->merge_tails.end(), o.seq, o.seq + A0_SLOTS);
    }
  }
  // ---- rule 4: leaves of the records the target holds sampleable; the record map and the placements
  memset(leaves_out, 0, (size_t)N2 * 4);
  t->merge_rmap.clear();
  for (size_t i = 0; i < recs.size(); ++i) {
    const int64_t q = tq_of[i];
    const int64_t dst = q >= t->tail_q ? q % N2 : -1;
    if (dst >= 0 && t->sampleable[dst]) leaves_out[dst] = leaves[recs[i].file][recs[i].pos];
    t->merge_rmap.push_back(recs[i].file); t->merge_rmap.push_back(recs[i].pos); t->merge_rmap.push_back(dst);
  }
  t->merge_place.clear();
  for (const Alloc& a : alloc) {
    if (a.t < final_lo) continue;
    t->merge_place.push_back(a.file); t->merge_place.push_back(a.seq); t->merge_place.push_back(a.t % t->NF);
  }
  out->n_place = (int64_t)t->merge_place.size() / 3;
  out->place = t->merge_place.data();
  out->n_rec = (int64_t)t->merge_rmap.size() / 3;
  out->record_map = t->merge_rmap.data();
  out->n_tail = (int64_t)t->merge_tails.size() / (3 + A0_SLOTS);
  out->tails = t->merge_tails.data();
  out->stride_hint = hint;
  return A0_OK;
}
