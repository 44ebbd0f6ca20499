// GPU sum-tree for prioritized replay: K2a (batched stratified draws + IS weights) and K2b (leaf
// writes with bottom-up recomputation).
//
// Replaces the reference's flat CPU priority vector: the intended draw torch.multinomial(priority)
// (agent0/deepq/replay.py:39-43), priority[ids] = (loss+eps)^alpha and max_p (replay.py:55-59),
// priority[-k:] = max_p**alpha on extend (replay.py:52) and the IS-weight block of Trainer.step
// (agent0/deepq/trainer.py:91-94), which sums 1 M CPU floats per update.
//
// Arithmetic is defined by oracle/sumtree.py and must match it bit for bit:
//   node = fl32(left + right), recomputed from children;  t = fl32(fl32(fl32(b + u)/B) * root);
//   go left iff (t < left) || !(right > 0);  going right: t = fl32(t - left).
// The tree (2P floats, 8 MB at 1 M leaves, 16.8 MB at 2 M) is L2-resident: these kernels are
// latency-bound, not HBM-bound.
#include <stdlib.h>

#include "a0_common.cuh"
#ifdef A0_TRACE
A0_TRACE_SETTER(a0_trace_set_sumtree)
#endif

// ------------------------------------------------------------------------------------------------
// K2a.  One warp per draw.  Instead of one dependent L2 round trip per level, the warp fetches the
// whole 5-level sub-heap below the current node in two loads (lane i: sub-heap node 32+i; lane h-2:
// sub-heap node h for h = 2..31) and walks it through shuffles, with exactly the scalar arithmetic.
// ------------------------------------------------------------------------------------------------
constexpr int K2A_WARPS = 8;
constexpr int K2A_TOP = 10;         // tree levels every sampler CTA copies to shared memory (8 KB) before its descents

// Philox4x32-10 (Salmon et al., SC'11; the generator behind curand and torch's CUDA RNG), first
// output word.  The sampler's own uniforms: draw g of call c under seed s is
// u = (philox(counter = {g, 0, c_lo, c_hi}, key = {s_lo, s_hi}).x >> 8) * 2^-24  in [0, 1)
// (oracle/sumtree.py: philox_uniform), so a host without torch -- or a captured CUDA graph, which
// cannot take fresh host randoms per replay -- draws reproducible batches with no extra launch.
__device__ __forceinline__ uint32_t a0_philox_x0(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                 uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return c0;
}

struct A0Rng {
  unsigned long long seed;
  long long call;                  // >= 0: this call number; < 0: the device-resident counter, advanced by the launch
  unsigned long long* call_dev;    // device call counter (8-byte aligned)
  unsigned int* ticket;            // CTA arrivals of this launch (zero between launches)
  float* u_out;                    // optional copy of the uniforms (tests)
};

// One arrival per finished unit (`units` in the launch: batches on the prioritized path, whose
// last CTA reports for the whole batch -- 20 arrivals instead of 1280 same-address atomics at
// 20 x 512 draws; CTAs otherwise).  The last arrival advances the call counter and re-arms the ticket.
__device__ __forceinline__ void a0_rng_done(const A0Rng& rng, unsigned long long call, unsigned int units) {
  __threadfence();
  if (atomicAdd(rng.ticket, 1u) == units - 1u) {
    *rng.call_dev = call + 1ull;
    *rng.ticket = 0u;
  }
}

// One unit of the sampler: the 8 draws [8 * unit, 8 * unit + 8), one per warp (descent, mailbox, IS-weight epilogue).
// `units` = units of the whole launch (a CTA runs `rounds` of them, a0_k2a_sample below).
__device__ __forceinline__ void
a0_k2a_unit(const float* __restrict__ tree, int64_t P, int32_t D, const float* __restrict__ u, int32_t total,
            int32_t batch, float top, float beta, float sum_offset, int32_t uniform,
            int64_t* __restrict__ idx_out, float* __restrict__ prio_out, float* __restrict__ weight_out,
            unsigned int* counter, float* bmax, const A0Rng& rng, long long* __restrict__ mail, const bool rng_dev,
            const unsigned long long call, const float root, const int unit, const unsigned int units,
            const float* __restrict__ s_top, const int top_levels
#ifdef A0_TRACE
            , const unsigned long long _t0, const unsigned long long _t2, const unsigned long long (&_tx)[8]
#endif
            ) {
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int g = unit * K2A_WARPS + warp;
  float leaf_w = 0.0f;
  if (g < total) {
    const int b = g % batch;
    float ug;
    if (u) {
      ug = u[g];
    } else {
      const uint32_t x = a0_philox_x0((uint32_t)g, 0u, (uint32_t)call, (uint32_t)(call >> 32), (uint32_t)rng.seed,
                                      (uint32_t)(rng.seed >> 32));
      ug = __uint2float_rn(x >> 8) * 5.9604644775390625e-08f;      // exact: 24 bits * 2^-24
      if (rng.u_out && lane == 0) rng.u_out[g] = ug;
    }
    float t = __fmul_rn(__fdiv_rn(__fadd_rn((float)b, ug), (float)batch), root);
    int64_t v = 1;          // current node, warp-uniform
    float leaf = root;
    int left = D;
    if (top_levels > 0) {
      // the first levels from the CTA's shared-memory copy of the top of the tree: the same comparisons and
      // subtractions, one L2 round trip (the copy) instead of two
      int h = 1;
      for (int s = 0; s < top_levels; ++s) {
        const float L = s_top[2 * h], R = s_top[2 * h + 1];
        if (t < L || !(R > 0.0f)) { h = 2 * h; leaf = L; }
        else { t = __fsub_rn(t, L); h = 2 * h + 1; leaf = R; }
      }
      v = h;
      left = D - top_levels;
    }
    while (left > 0) {
      const int c = left < 5 ? left : 5;
      // sub-heap node h lives at tree[(v << l) + (h - (1 << l))], l = floor(log2 h)
      const int hB = lane + 2;
      const int lB = 31 - __clz(hB);
      float regB = 0.0f, regA = 0.0f;
      if (lB <= c && lB <= 4 && hB < 32) regB = __ldcg(tree + ((v << lB) + (hB - (1 << lB))));
      if (c == 5) regA = __ldcg(tree + ((v << 5) + lane));
      int h = 1;
      for (int s = 0; s < c; ++s) {
        const int hl = 2 * h;
        float L, R;
        if (hl < 32) {
          L = __shfl_sync(0xffffffffu, regB, hl - 2);
          R = __shfl_sync(0xffffffffu, regB, hl - 1);
        } else {
          L = __shfl_sync(0xffffffffu, regA, hl - 32);
          R = __shfl_sync(0xffffffffu, regA, hl - 31);
        }
        if (t < L || !(R > 0.0f)) { h = hl; leaf = L; }
        else { t = __fsub_rn(t, L); h = hl + 1; leaf = R; }
      }
      v = (v << c) + (h - (1 << c));
      left -= c;
    }
    if (lane == 0) {
      // the gather CTA of this draw may already be resident and polling (a0_rb_sample_gather): it
      // needs nothing but the position, so the mailbox word carries it (position + 1, 0 = empty)
      if (mail) asm volatile("st.relaxed.gpu.global.s64 [%0], %1;" ::"l"(mail + g), "l"((long long)(v - P) + 1ll) : "memory");
      idx_out[g] = v - P;
      prio_out[g] = leaf;
      if (warp == 0) A0_TEND(2);
    }
    leaf_w = leaf;
  }
  if (weight_out == nullptr || uniform) {
    if (uniform && weight_out && g < total && lane == 0) weight_out[g] = 1.0f;   // ReplayEnum.uniform: weights = 1 (trainer.py:95-96)
    if (rng_dev) {
      __syncthreads();                                  // every warp of this CTA has read the counter
      if (threadIdx.x == 0) a0_rng_done(rng, call, units);
    }
    return;
  }
  // ---- epilogue (trainer.py:91-94): every warp turns its own priority into the un-normalised
  //      weight; the batch maximum is folded with atomicMax on the bit pattern (w > 0) and the last
  //      arrival of each batch (ticket counter) divides the batch by (max + 1e-8).  All batches of
  //      a multi-batch draw finish in the same launch.  When the batch size is a multiple of the
  //      warps per CTA, a CTA lies inside one batch and aggregates in shared memory first (one
  //      atomic pair per CTA instead of per warp: 512 same-address atomics per batch become 64) and
  //      the last CTA normalises with all of its threads.
  const unsigned int nbatches = (unsigned int)(total / batch);
  const float denom = __fadd_rn(root, sum_offset);
  if (batch % K2A_WARPS == 0) {         // total % batch == 0, so every warp of the CTA has a draw
    __shared__ float s_w[K2A_WARPS];
    __shared__ int s_last;
    const int k = g / batch;
    float* w = weight_out + (size_t)k * batch;
    if (lane == 0) {
      const float wj = powf(__fmul_rn(top, __fdiv_rn(leaf_w, denom)), -beta);
      __stcg(weight_out + g, wj);
      s_w[warp] = wj;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      float mx = s_w[0];
#pragma unroll
      for (int i = 1; i < K2A_WARPS; ++i) mx = fmaxf(mx, s_w[i]);
      atomicMax(reinterpret_cast<int*>(bmax + k), __float_as_int(mx));
      __threadfence();
      s_last = atomicAdd(counter + k, (unsigned)K2A_WARPS) == (unsigned)(batch - K2A_WARPS);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const float inv = __fadd_rn(__ldcg(bmax + k), 1e-8f);
    for (int j = threadIdx.x; j < batch; j += K2A_WARPS * 32) w[j] = __fdiv_rn(__ldcg(w + j), inv);
    __syncthreads();                   // every warp has read the batch maximum before thread 0 re-arms it (a slow
                                       // warp would otherwise divide by 0 + 1e-8: seen under compute-sanitizer's timing)
    if (threadIdx.x == 0) {
      counter[k] = 0u; bmax[k] = 0.0f;
      if (rng_dev) a0_rng_done(rng, call, nbatches);    // this batch's CTAs have all arrived, hence all read the counter
    }
    return;
  }
  if (g >= total) return;
  const int k = g / batch;
  float* w = weight_out + (size_t)k * batch;
  unsigned ticket = 0;
  if (lane == 0) {
    const float wj = powf(__fmul_rn(top, __fdiv_rn(leaf_w, denom)), -beta);
    __stcg(weight_out + g, wj);
    atomicMax(reinterpret_cast<int*>(bmax + k), __float_as_int(wj));
    __threadfence();
    ticket = atomicAdd(counter + k, 1u);
  }
  ticket = __shfl_sync(0xffffffffu, ticket, 0);
  if (ticket != (unsigned)batch - 1u) return;
  __threadfence();
  const float inv = __fadd_rn(__ldcg(bmax + k), 1e-8f);
  for (int j0 = 0; j0 < batch; j0 += 32 * 8) {
    float v[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int j = j0 + q * 32 + lane;
      v[q] = j < batch ? __ldcg(w + j) : 0.0f;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int j = j0 + q * 32 + lane;
      if (j < batch) w[j] = __fdiv_rn(v[q], inv);
    }
  }
  __syncwarp();                        // every lane holds the batch maximum before lane 0 re-arms it
  if (lane == 0) {
    counter[k] = 0u; bmax[k] = 0.0f;
    if (rng_dev) a0_rng_done(rng, call, nbatches);
  }
}

// The launch: CTA c runs units c, c + gridDim.x, ... (`rounds` of them); one round by default.  A0_OPT_K2A_ROUNDS
// (measured alternative, off): 20 x 512 draws are 10 240 warps on 9 472 warp slots, and the gather that is launched
// under the sampler can only start once EVERY sampler CTA has started -- with one round its first CTAs enter 11 us
// after the sampler's (device timeline), with two rounds 1.3 us after.  The early CTAs only poll their mailbox
// sooner, though: the sampler itself takes 27 instead of 17 us and the batch-512 step does not get shorter (233.9
// against 231.8 us), so the option stays off.
__global__ void __launch_bounds__(K2A_WARPS * 32)
a0_k2a_sample(const float* __restrict__ tree, int64_t P, int32_t D, const float* __restrict__ u, int32_t total,
              int32_t batch, float top, float beta, float sum_offset, int32_t uniform,
              int64_t* __restrict__ idx_out, float* __restrict__ prio_out, float* __restrict__ weight_out,
              unsigned int* counter, float* bmax, const float* __restrict__ dyn, const A0Rng rng,
              long long* __restrict__ mail, int32_t rounds, int32_t top_levels) {
  A0_T0();
  A0_PDL_PROLOGUE();
  A0_TMID();
  if (dyn) {            // top / beta / sum_offset live on the device (a0_rb_set_dynamic): graph-replay safe
    top = __ldcg(dyn);
    beta = __ldcg(dyn + 1);
    sum_offset = __ldcg(dyn + 2);
  }
  // Device-resident call counter (rng.call < 0): every warp reads it before anything else; it is
  // advanced for the next launch / graph replay only after every unit has reported in
  // (a0_rng_done), i.e. after every warp of the launch has read it.
  const bool rng_dev = u == nullptr && rng.call < 0;
  const unsigned long long call = rng_dev ? __ldcg(rng.call_dev) : (unsigned long long)rng.call;
  // levels 0 .. top_levels of the tree (nodes 1 .. 2^(top_levels+1) - 1) into shared memory, once per CTA
  __shared__ __align__(16) float s_top[2 << K2A_TOP];
  if (top_levels > 0) {
    const int n4 = (2 << top_levels) >> 2;
    for (int i = threadIdx.x; i < n4; i += K2A_WARPS * 32)
      reinterpret_cast<float4*>(s_top)[i] = __ldcg(reinterpret_cast<const float4*>(tree) + i);
    __syncthreads();
  }
  const float root = top_levels > 0 ? s_top[1] : __ldcg(tree + 1);
  const unsigned int units = gridDim.x * (unsigned int)rounds;
  for (int r = 0; r < rounds; ++r) {
    a0_k2a_unit(tree, P, D, u, total, batch, top, beta, sum_offset, uniform, idx_out, prio_out, weight_out, counter, bmax, rng,
                mail, rng_dev, call, root, r * (int)gridDim.x + (int)blockIdx.x, units, s_top, top_levels
#ifdef A0_TRACE
                , _t0, _t2, _tx
#endif
                );
    if (r + 1 < rounds) __syncthreads();            // the unit's shared words are reused by the next one
  }
}

static int g_k2a_top = -1;         // A0_K2A_TOP=0: every level of the descent from L2 (the round-1/2 sampler)
static bool a0_option_k2a_top() {
  if (g_k2a_top < 0) {
    const char* e = getenv("A0_K2A_TOP");
    g_k2a_top = e ? (atoi(e) != 0) : 1;
  }
  return g_k2a_top != 0;
}
static int g_k2a_rounds = -1;      // A0_OPT_K2A_ROUNDS: a sampler launch too large to be resident at once runs several units per CTA
static bool a0_option_k2a_rounds() {
  if (g_k2a_rounds < 0) {
    const char* e = getenv("A0_K2A_ROUNDS");
    g_k2a_rounds = e ? (atoi(e) != 0) : 0;
  }
  return g_k2a_rounds != 0;
}
void a0_set_k2a_rounds(int on) { g_k2a_rounds = on != 0; }

__global__ void a0_set_dyn(float* dyn, float top, float beta, float sum_offset) {
  dyn[0] = top; dyn[1] = beta; dyn[2] = sum_offset;
}

extern "C" int a0_rb_set_dynamic(a0_replay_t* h, float top, float beta, float sum_offset, a0_stream_t stream_) {
  A0_REQUIRE(h != nullptr, "a0_rb_set_dynamic: handle is NULL");
  A0_REQUIRE(top >= 0.0f, "a0_rb_set_dynamic: top must be non-negative");
  A0DeviceGuard guard(h->device);
  a0_set_dyn<<<1, 1, 0, (cudaStream_t)stream_>>>(h->dyn, top, beta, sum_offset);
  A0_LAUNCH_CHECK();
  return A0_OK;
}

static int a0_sample_launch(a0_replay_t* h, const float* u, const A0Rng& rng, int32_t total, int32_t batch, float top,
                            float beta, float sum_offset, int32_t uniform, int64_t* idx_out, float* prio_out,
                            float* weight_out, a0_stream_t stream_, const char* who, long long* mail = nullptr) {
  A0_REQUIRE(h != nullptr, "%s: handle is NULL", who);
  A0_REQUIRE(total >= 0 && batch > 0 && total % batch == 0, "%s: total %d must be a multiple of batch %d", who, total, batch);
  if (total == 0) return A0_OK;
  A0_REQUIRE(idx_out && prio_out, "%s: NULL argument", who);
  A0_REQUIRE(total / batch <= A0_MAX_BATCHES, "%s: at most %d batches per call", who, A0_MAX_BATCHES);
  A0DeviceGuard guard(h->device);
  int blocks = (total + K2A_WARPS - 1) / K2A_WARPS;
  int rounds = 1;
  {
    // all CTAs resident at once (8 CTAs of 8 warps per SM), see a0_k2a_sample
    static thread_local int sms[64] = {0};
    int n_sm = 148;
    if (h->device < 64) {
      if (!sms[h->device]) A0_CUDA(cudaDeviceGetAttribute(&sms[h->device], cudaDevAttrMultiProcessorCount, h->device));
      n_sm = sms[h->device];
    }
    const int resident = n_sm * (2048 / (K2A_WARPS * 32));
    if (blocks > resident && a0_option_k2a_rounds()) {
      for (int r = 2; r <= 8; ++r)
        if (blocks % r == 0 && blocks / r <= resident) { rounds = r; break; }
    }
    blocks /= rounds;
  }
  if (mail) {
    // The gather's CTAs (28 KB of shared memory each) can only join an SM whose shared-memory carve-out
    // already fits them: an SM running sampler CTAs under the default (L1-heavy) carve-out is closed
    // to them until it drains -- device timeline: only (148 - 80) x 7 = 476 of 640 gather CTAs started
    // under the sampler, the rest 6 us later.  Same carve-out for both kernels: everything co-resides.
    static thread_local bool carved[64] = {false};
    if (h->device < 64 && !carved[h->device]) {
      A0_CUDA(cudaFuncSetAttribute(a0_k2a_sample, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
      carved[h->device] = true;
    }
  }
  A0_LAUNCH(a0_k2a_sample, (unsigned)blocks, K2A_WARPS * 32, 0, (cudaStream_t)stream_, 1, A0_PDL_K2, h->tree, h->P, h->D, u, total, batch,
            top, beta, sum_offset, uniform, idx_out, prio_out, weight_out, h->counter,
            reinterpret_cast<float*>(h->counter + A0_MAX_BATCHES + 16), (const float*)(top < 0.0f ? h->dyn : nullptr), rng, mail,
            (int32_t)rounds, (int32_t)(a0_option_k2a_top() ? (h->D < K2A_TOP ? (h->D >= 1 ? h->D : 0) : K2A_TOP) : 0));
  return A0_OK;
}

extern "C" int a0_pt_sample(a0_replay_t* h, const float* u, int32_t total, int32_t batch, float top, float beta,
                            float sum_offset, int32_t uniform, int64_t* idx_out, float* prio_out,
                            float* weight_out, a0_stream_t stream_) {
  A0_REQUIRE(total == 0 || u != nullptr, "a0_pt_sample: u is NULL (a0_pt_sample_rng draws its own uniforms)");
  A0Rng rng = {0ull, 0ll, nullptr, nullptr, nullptr};
  return a0_sample_launch(h, u, rng, total, batch, top, beta, sum_offset, uniform, idx_out, prio_out, weight_out, stream_,
                          "a0_pt_sample");
}

// counter[] words used by the sampler's own generator (the rest of the layout is in a0_common.cuh)
constexpr int K2A_RNG_TICKET = 2 * A0_MAX_BATCHES + 32;  // past the per-batch maxima at [MAXB+16, 2*MAXB+16)
constexpr int K2A_RNG_CALL = A0_RNG_CALL_WORD;           // two words, 8-byte aligned (a0_common.cuh)

extern "C" int a0_pt_sample_rng(a0_replay_t* h, uint64_t seed, int64_t call, int32_t total, int32_t batch, float top,
                                float beta, float sum_offset, int32_t uniform, int64_t* idx_out, float* prio_out,
                                float* weight_out, float* u_out, a0_stream_t stream_) {
  A0_REQUIRE(h != nullptr, "a0_pt_sample_rng: handle is NULL");
  A0Rng rng;
  rng.seed = seed;
  rng.call = call;
  rng.call_dev = reinterpret_cast<unsigned long long*>(h->counter + K2A_RNG_CALL);
  rng.ticket = h->counter + K2A_RNG_TICKET;
  rng.u_out = u_out;
  return a0_sample_launch(h, nullptr, rng, total, batch, top, beta, sum_offset, uniform, idx_out, prio_out, weight_out,
                          stream_, "a0_pt_sample_rng");
}

// Sample + gather as a producer/consumer pair.  Two launches, but the gather (K3, one CTA per draw)
// is launched with programmatic stream serialization and does NOT wait for the sampler to finish:
// it becomes resident while the sampler's warps are still descending the tree, and each gather CTA
// starts fetching frames the moment its own draw's position lands in the mailbox.  What disappears
// from the critical path of a step is the sampler's epilogue (IS-weight normalisation, tickets),
// its drain, and the launch hand-over between the two kernels.  The gather ends with
// griddepcontrol.wait, so "gather complete" still implies "sampler complete" for everything
// downstream (K4 reads the weights).  Results are those of a0_pt_sample[_rng] + a0_rb_gather.
// the mailbox of a0_rb_sample_gather: allocated on first use (or for a larger draw), not inside a graph capture
int a0_mail_reserve(a0_replay* h, int32_t total, cudaStream_t stream) {
  if (h->mail_cap >= total) return A0_OK;
  int64_t cap = h->mail_cap > 0 ? h->mail_cap : 1024;
  while (cap < total) cap *= 2;
  A0_CUDA(cudaStreamSynchronize(stream));
  if (h->mail) A0_CUDA(cudaFree(h->mail));
  h->mail = nullptr; h->mail_cap = 0;
  A0_CUDA(cudaMalloc((void**)&h->mail, (size_t)cap * sizeof(long long)));
  A0_CUDA(cudaMemset(h->mail, 0, (size_t)cap * sizeof(long long)));
  h->mail_cap = cap;
  return A0_OK;
}

extern "C" int a0_rb_sample_gather(a0_replay_t* h, const float* u, uint64_t seed, int64_t call, int32_t total,
                                   int32_t batch, float top, float beta, float sum_offset, int32_t uniform,
                                   int64_t* idx_out, float* prio_out, float* weight_out, int32_t n_step, double gamma,
                                   uint8_t* frames_out, int64_t* action_out, double* reward64_out, float* reward32_out,
                                   uint8_t* done8_out, float* done32_out, int64_t* boot_out, a0_stream_t stream_) {
  A0_REQUIRE(h != nullptr, "a0_rb_sample_gather: handle is NULL");
  A0_REQUIRE(total >= 0 && batch > 0 && total % batch == 0, "a0_rb_sample_gather: total %d must be a multiple of batch %d", total, batch);
  if (total == 0) return A0_OK;
  A0_REQUIRE(idx_out && prio_out && frames_out, "a0_rb_sample_gather: idx_out, prio_out and frames_out are required");
  A0_REQUIRE(n_step >= 1 && n_step <= A0_MAX_NSTEP, "a0_rb_sample_gather: n_step %d outside [1,%d]", n_step, A0_MAX_NSTEP);
  A0_REQUIRE(((uintptr_t)frames_out & 15) == 0, "a0_rb_sample_gather: frames_out must be 16-byte aligned");
  { int frc = a0_check_fault(h, "a0_rb_sample_gather"); if (frc) return frc; }
  A0DeviceGuard guard(h->device);
  cudaStream_t stream = (cudaStream_t)stream_;
  { int mrc = a0_mail_reserve(h, total, stream); if (mrc) return mrc; }
  A0Rng rng = {0ull, 0ll, nullptr, nullptr, nullptr};
  if (!u) {
    rng.seed = seed;
    rng.call = call;
    rng.call_dev = reinterpret_cast<unsigned long long*>(h->counter + K2A_RNG_CALL);
    rng.ticket = h->counter + K2A_RNG_TICKET;
  }
  int rc = a0_sample_launch(h, u, rng, total, batch, top, beta, sum_offset, uniform, idx_out, prio_out, weight_out, stream_,
                            "a0_rb_sample_gather", h->mail);
  if (rc) return rc;
  const A0GatherOut out = {frames_out, action_out, reward64_out, reward32_out, done8_out, done32_out, boot_out};
  rc = a0_gather_launch_mail(h, idx_out, h->mail, total, n_step, gamma, out, stream);
  if (rc) cudaMemsetAsync(h->mail, 0, (size_t)total * sizeof(long long), stream);   // nobody will consume the posted words
  return rc;
}

// The same pair with the gather cut into WAVES (consecutive ranges of the draw, one launch each), so that a
// consumer on another stream can start on the first batches while the later ones are still being fetched:
//   a0_rb_sample_mail            the sampler, posting every draw's record position to the mailbox
//   a0_rb_gather_mail (x waves)  draws [lo, lo + count): launched programmatically under its predecessor on the
//                                stream (the sampler or the previous wave), fed through the mailbox
// Every wave lets its successor launch at once and ends with griddepcontrol.wait, so waves complete in launch
// order and "wave j complete" implies "sampler complete" (weights) and "waves < j complete".
extern "C" int a0_rb_sample_mail(a0_replay_t* h, const float* u, uint64_t seed, int64_t call, int32_t total,
                                 int32_t batch, float top, float beta, float sum_offset, int32_t uniform,
                                 int64_t* idx_out, float* prio_out, float* weight_out, a0_stream_t stream_) {
  A0_REQUIRE(h != nullptr, "a0_rb_sample_mail: handle is NULL");
  A0_REQUIRE(total >= 0 && batch > 0 && total % batch == 0, "a0_rb_sample_mail: total %d must be a multiple of batch %d", total, batch);
  if (total == 0) return A0_OK;
  A0_REQUIRE(idx_out && prio_out, "a0_rb_sample_mail: idx_out and prio_out are required");
  { int frc = a0_check_fault(h, "a0_rb_sample_mail"); if (frc) return frc; }
  A0DeviceGuard guard(h->device);
  { int mrc = a0_mail_reserve(h, total, (cudaStream_t)stream_); if (mrc) return mrc; }
  {
    // The ordered fetch's progress word is re-armed by the last draw of every sampler call, which holds as long as every
    // draw is gathered exactly once.  An eagerly issued call can be left half done (an exception between two wave
    // launches, a failed launch), so outside a stream capture the word is cleared here; a captured graph launches all of
    // its waves or none.  A stale word could only cost the ordering and bounded polls, never a result.
    cudaStreamCaptureStatus cst = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing((cudaStream_t)stream_, &cst);
    if (cst == cudaStreamCaptureStatusNone || h->progress_dirty) {
      A0_CUDA(cudaMemsetAsync(h->counter + A0_K3_PROGRESS, 0, sizeof(unsigned int), (cudaStream_t)stream_));
      h->progress_dirty = 0;
    }
  }
  A0Rng rng = {0ull, 0ll, nullptr, nullptr, nullptr};
  if (!u) {
    rng.seed = seed;
    rng.call = call;
    rng.call_dev = reinterpret_cast<unsigned long long*>(h->counter + K2A_RNG_CALL);
    rng.ticket = h->counter + K2A_RNG_TICKET;
  }
  h->mail_total = total;
  return a0_sample_launch(h, u, rng, total, batch, top, beta, sum_offset, uniform, idx_out, prio_out, weight_out, stream_,
                          "a0_rb_sample_mail", h->mail);
}

extern "C" int a0_rb_gather_mail(a0_replay_t* h, int32_t lo, int32_t count, int32_t window, int32_t n_step, double gamma,
                                 uint8_t* frames_out, int64_t* action_out, double* reward64_out, float* reward32_out,
                                 uint8_t* done8_out, float* done32_out, int64_t* boot_out, a0_stream_t stream_) {
  A0_REQUIRE(h != nullptr, "a0_rb_gather_mail: handle is NULL");
  A0_REQUIRE(lo >= 0 && count >= 0, "a0_rb_gather_mail: negative range");
  A0_REQUIRE(window >= 0, "a0_rb_gather_mail: negative window");
  if (count == 0) return A0_OK;
  A0_REQUIRE(frames_out != nullptr, "a0_rb_gather_mail: frames_out is required");
  A0_REQUIRE(n_step >= 1 && n_step <= A0_MAX_NSTEP, "a0_rb_gather_mail: n_step %d outside [1,%d]", n_step, A0_MAX_NSTEP);
  A0_REQUIRE(((uintptr_t)frames_out & 15) == 0, "a0_rb_gather_mail: frames_out must be 16-byte aligned");
  A0_REQUIRE(h->mail != nullptr && (int64_t)lo + count <= h->mail_cap,
             "a0_rb_gather_mail: draws [%d, %d) lie outside the mailbox of the last a0_rb_sample_mail", lo, lo + count);
  A0DeviceGuard guard(h->device);
  cudaStream_t stream = (cudaStream_t)stream_;
  // the outputs are the bases of the whole draw's buffers: this wave writes rows [lo, lo + count)
  const A0GatherOut out = {frames_out + (size_t)lo * A0_SLOTS * h->F, action_out ? action_out + lo : nullptr,
                           reward64_out ? reward64_out + lo : nullptr, reward32_out ? reward32_out + lo : nullptr,
                           done8_out ? done8_out + lo : nullptr, done32_out ? done32_out + lo : nullptr,
                           boot_out ? boot_out + lo : nullptr};
  A0_REQUIRE((int64_t)lo + count <= h->mail_total, "a0_rb_gather_mail: draws [%d, %d) lie beyond the %lld draws of the last a0_rb_sample_mail",
             lo, lo + count, (long long)h->mail_total);
  int rc = a0_gather_launch_mail(h, nullptr, h->mail + lo, count, n_step, gamma, out, stream, h->mail_total, window, lo);
  if (rc) {
    cudaMemsetAsync(h->mail + lo, 0, (size_t)count * sizeof(long long), stream);   // nobody will consume the posted words
    if (window > 0) h->progress_dirty = 1;                                         // nor count these draws as complete
  }
  return rc;
}

__global__ void a0_set_u64(unsigned long long* p, unsigned long long v) { *p = v; }

extern "C" int a0_pt_rng_seek(a0_replay_t* h, uint64_t call, a0_stream_t stream_) {
  A0_REQUIRE(h != nullptr, "a0_pt_rng_seek: handle is NULL");
  A0DeviceGuard guard(h->device);
  a0_set_u64<<<1, 1, 0, (cudaStream_t)stream_>>>(reinterpret_cast<unsigned long long*>(h->counter + K2A_RNG_CALL),
                                                 (unsigned long long)call);
  A0_LAUNCH_CHECK();
  return A0_OK;
}

// ------------------------------------------------------------------------------------------------
// K2a-unique.  Prioritized batches WITHOUT replacement, the law of the reference's
// torch.multinomial(priority[:top], B, replacement=False) (agent0/deepq/replay.py:41-43).  Defined
// exactly by oracle/sample_unique.py, which this kernel matches bit for bit (indices, priorities, stats):
//   * a batch is the first B DISTINCT records of a stream of independent descents; candidate j of batch k
//     in call c takes u = ((x0 >> 5) * 2^26 + (x1 >> 6)) * 2^-53 (float64) from
//     Philox4x32-10(counter {j, 0x80000000 | k, c_lo, c_hi}, key {seed_lo, seed_hi});
//   * round r draws B - |F| candidates that descend in float64 against the accepted set F as it stood at
//     the start of the round: m(v) = max(0, tree[v] - (Pre[hi_v] - Pre[lo_v])) with Pre the sequential
//     float64 prefix sums of F's priorities in position order; t = u * m(1); go left iff
//     t < m(2v) || !(m(2v+1) > 0), else t -= m(2v).  A leaf in F or with p <= 0 is void.  The non-void
//     candidates are accepted in j order, each record once; the rows are F in acceptance order;
//   * m(1) <= 0 at the start of a round, or 8 consecutive rounds accepting nothing: fewer than B records
//     with positive priority.  The remaining rows repeat F[0] and the handle's fault word gets code 2.
// One CTA per batch owns the whole batch: thread c descends candidate c (float2 loads below the
// shared-memory top levels), a bitonic sort of (position, ordinal) keeps each record's first occurrence,
// a block scan turns acceptances into rows, and the IS-weight epilogue (trainer.py:91-94) needs no
// cross-CTA ticket.  A further round re-sorts F and forms Pre (one thread: the order of the sum is part
// of the law), and each level of its descents binary-searches F's range below the current node.
// ------------------------------------------------------------------------------------------------
constexpr int KU_MAX_BATCH = 1024;
constexpr int KU_MAX_IDLE = 8;
constexpr int KU_FAULT_SHORTFALL = 2;

// ascending sort of s_key[0, n) (n a power of two, n <= blockDim.x), every thread of the CTA calls it
__device__ __forceinline__ void a0_ku_bitonic(unsigned long long* s_key, int n) {
  for (int k = 2; k <= n; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      const int i = threadIdx.x;
      const int x = i ^ j;
      if (i < n && x > i) {
        const unsigned long long a = s_key[i], b = s_key[x];
        if ((a > b) == ((i & k) == 0)) { s_key[i] = b; s_key[x] = a; }
      }
      __syncthreads();
    }
}

// exclusive prefix sum of v over the CTA; *total = the sum (every thread)
__device__ __forceinline__ int a0_ku_scan(int v, int* s_warp, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) s_warp[warp] = x;
  __syncthreads();
  if (warp == 0) {
    int w = lane < nw ? s_warp[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    if (lane < nw) s_warp[lane] = w;          // inclusive over warps
  }
  __syncthreads();
  const int before = (warp > 0 ? s_warp[warp - 1] : 0) + x - v;
  *total = s_warp[nw - 1];
  __syncthreads();                            // s_warp is reused by the next scan
  return before;
}

__global__ void __launch_bounds__(KU_MAX_BATCH)
a0_k2a_unique(const float* __restrict__ tree, int32_t P, int32_t D, int32_t batch, int32_t nbatches, float top, float beta,
              float sum_offset, int32_t uniform, int64_t* __restrict__ idx_out, float* __restrict__ prio_out,
              float* __restrict__ weight_out, int32_t* __restrict__ stats_out, const float* __restrict__ dyn, const A0Rng rng,
              int32_t* fault, int32_t top_levels) {
  __shared__ __align__(16) float s_top[2 << K2A_TOP];
  __shared__ unsigned long long s_key[KU_MAX_BATCH];
  __shared__ int32_t s_apos[KU_MAX_BATCH];          // F in acceptance order
  __shared__ float s_apri[KU_MAX_BATCH];
  __shared__ int32_t s_fpos[KU_MAX_BATCH];          // F in position order
  __shared__ double s_pre[KU_MAX_BATCH + 1];        // its prefix sums
  __shared__ int32_t s_flag[KU_MAX_BATCH];
  __shared__ int s_warp[32];
  __shared__ unsigned long long s_call;
  A0_T0();
  A0_PDL_PROLOGUE();
  A0_TMID();
  if (dyn) {
    top = __ldcg(dyn);
    beta = __ldcg(dyn + 1);
    sum_offset = __ldcg(dyn + 2);
  }
  const int tid = threadIdx.x;
  const int k = blockIdx.x;
  const bool rng_dev = rng.call < 0;
  if (tid == 0) {
    s_call = rng_dev ? __ldcg(rng.call_dev) : (unsigned long long)rng.call;
    s_pre[0] = 0.0;
  }
  const int n4 = (2 << top_levels) >> 2;
  for (int i = tid; i < n4; i += blockDim.x) reinterpret_cast<float4*>(s_top)[i] = __ldcg(reinterpret_cast<const float4*>(tree) + i);
  __syncthreads();
  const unsigned long long call = s_call;
  const float root = s_top[1];
  int nF = 0, rounds = 0, cand = 0, idle = 0;
  bool shortfall = false;
  while (nF < batch) {
    const double m1 = fmax(0.0, __dsub_rn((double)root, s_pre[nF]));
    if (!(m1 > 0.0)) { shortfall = true; break; }
    const int need = batch - nF;
    int pos = -1;
    float leaf = 0.0f;
    if (tid < need) {
      const uint32_t j = (uint32_t)(cand + tid);
      uint32_t c0 = j, c1 = 0x80000000u | (uint32_t)k, c2 = (uint32_t)call, c3 = (uint32_t)(call >> 32);
      uint32_t k0 = (uint32_t)rng.seed, k1 = (uint32_t)(rng.seed >> 32);
#pragma unroll
      for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
      }
      const unsigned long long bits = ((unsigned long long)(c0 >> 5) << 26) | (unsigned long long)(c1 >> 6);
      double t = __dmul_rn(__dmul_rn(__ull2double_rn(bits), 1.1102230246251565e-16), m1);      // * 2^-53: exact
      int v = 1, a = 0, b = nF;
      leaf = root;
      for (int d = 0; d < D; ++d) {
        const int mid = ((2 * v + 1) << (D - d - 1)) - P;
        int lo = a, hi = b;                                   // first F position >= mid inside [a, b)
        while (lo < hi) {
          const int m = (lo + hi) >> 1;
          if (s_fpos[m] < mid) lo = m + 1; else hi = m;
        }
        float L, R;
        if (d < top_levels) { L = s_top[2 * v]; R = s_top[2 * v + 1]; }
        else { const float2 lr = __ldcg(reinterpret_cast<const float2*>(tree + 2 * v)); L = lr.x; R = lr.y; }
        const double mL = fmax(0.0, __dsub_rn((double)L, __dsub_rn(s_pre[lo], s_pre[a])));
        const double mR = fmax(0.0, __dsub_rn((double)R, __dsub_rn(s_pre[b], s_pre[lo])));
        if (t < mL || !(mR > 0.0)) { v = 2 * v; b = lo; leaf = L; }
        else { t = __dsub_rn(t, mL); v = 2 * v + 1; a = lo; leaf = R; }
      }
      if (b - a != 1 && leaf > 0.0f) pos = v - P;             // void: already accepted, or an empty leaf
    }
    // first occurrence of every record among this round's candidates, in draw order
    int n2 = 1;
    while (n2 < need) n2 <<= 1;
    if (tid < n2) s_key[tid] = pos >= 0 ? ((unsigned long long)pos << 32) | (unsigned)tid : ~0ull;
    if (tid < need) s_flag[tid] = 0;
    __syncthreads();
    a0_ku_bitonic(s_key, n2);
    if (tid < need) {
      const unsigned long long key = s_key[tid];
      if (key != ~0ull && (tid == 0 || (s_key[tid - 1] >> 32) != (key >> 32))) s_flag[(int)(key & 0xffffffffu)] = 1;
    }
    __syncthreads();
    const int acc = tid < need ? s_flag[tid] : 0;
    int accepted;
    const int row = nF + a0_ku_scan(acc, s_warp, &accepted);
    if (acc) { s_apos[row] = pos; s_apri[row] = leaf; }
    nF += accepted;
    rounds += 1;
    cand += need;
    idle = accepted ? 0 : idle + 1;
    if (nF == batch) break;
    if (idle == KU_MAX_IDLE) { shortfall = true; break; }
    // F in position order and its prefix sums for the next round's masked descents
    n2 = 1;
    while (n2 < nF) n2 <<= 1;
    __syncthreads();                                          // s_apos / s_apri complete
    if (tid < n2) s_key[tid] = tid < nF ? ((unsigned long long)s_apos[tid] << 32) | __float_as_uint(s_apri[tid]) : ~0ull;
    __syncthreads();
    a0_ku_bitonic(s_key, n2);
    if (tid < nF) s_fpos[tid] = (int32_t)(s_key[tid] >> 32);
    if (tid == 0) {
      double s = 0.0;
      for (int i = 0; i < nF; ++i) {
        s = __dadd_rn(s, (double)__uint_as_float((unsigned)(s_key[i] & 0xffffffffu)));
        s_pre[i + 1] = s;
      }
    }
    __syncthreads();
  }
  __syncthreads();
  if (tid == 0 && shortfall && fault) { *reinterpret_cast<volatile int32_t*>(fault) = KU_FAULT_SHORTFALL; __threadfence_system(); }
  if (tid == 0 && stats_out) { stats_out[2 * k] = rounds; stats_out[2 * k + 1] = cand; }
  // rows [nF, batch) of a shortfall repeat F[0]: every row is a valid position for the gather
  const int fill_pos = nF > 0 ? s_apos[0] : 0;
  const float fill_pri = nF > 0 ? s_apri[0] : __ldcg(tree + P);
  float p = 0.0f;
  if (tid < batch) {
    const int q = tid < nF ? s_apos[tid] : fill_pos;
    p = tid < nF ? s_apri[tid] : fill_pri;
    idx_out[(size_t)k * batch + tid] = q;
    prio_out[(size_t)k * batch + tid] = p;
  }
  if (weight_out) {
    float* w = weight_out + (size_t)k * batch;
    if (uniform) {
      if (tid < batch) w[tid] = 1.0f;                         // ReplayEnum.uniform: weights = 1 (trainer.py:95-96)
    } else {
      const float denom = __fadd_rn(root, sum_offset);
      const float wj = tid < batch ? powf(__fmul_rn(top, __fdiv_rn(p, denom)), -beta) : 0.0f;
      const float mx = a0_warp_max(wj);
      if ((tid & 31) == 0) reinterpret_cast<float*>(s_warp)[tid >> 5] = mx;
      __syncthreads();
      float bm = reinterpret_cast<float*>(s_warp)[0];
      for (int i = 1; i < (int)(blockDim.x >> 5); ++i) bm = fmaxf(bm, reinterpret_cast<float*>(s_warp)[i]);
      if (tid < batch) w[tid] = __fdiv_rn(wj, __fadd_rn(bm, 1e-8f));
    }
  }
  if (tid == 0) {
    A0_TEND(6);
    if (rng_dev) a0_rng_done(rng, call, (unsigned)nbatches);   // this CTA read the counter before it arrives
  }
}

extern "C" int a0_pt_sample_unique(a0_replay_t* h, uint64_t seed, int64_t call, int32_t total, int32_t batch, float top,
                                   float beta, float sum_offset, int32_t uniform, int64_t* idx_out, float* prio_out,
                                   float* weight_out, int32_t* stats_out, a0_stream_t stream_) {
  // the shape of the draw is checked before the handle: a malformed request is reported without a shard
  A0_REQUIRE(batch > 0 && batch <= KU_MAX_BATCH, "a0_pt_sample_unique: batch %d outside [1, %d]", batch, KU_MAX_BATCH);
  A0_REQUIRE(total >= 0 && total % batch == 0, "a0_pt_sample_unique: total %d must be a multiple of batch %d", total, batch);
  A0_REQUIRE(total / batch <= A0_MAX_BATCHES, "a0_pt_sample_unique: %d batches, at most %d per call", total / batch, A0_MAX_BATCHES);
  A0_REQUIRE(h != nullptr, "a0_pt_sample_unique: handle is NULL");
  if (total == 0) return A0_OK;
  A0_REQUIRE(idx_out && prio_out, "a0_pt_sample_unique: NULL argument");
  { int frc = a0_check_fault(h, "a0_pt_sample_unique"); if (frc) return frc; }
  A0DeviceGuard guard(h->device);
  A0Rng rng;
  rng.seed = seed;
  rng.call = call;
  rng.call_dev = reinterpret_cast<unsigned long long*>(h->counter + K2A_RNG_CALL);
  rng.ticket = h->counter + K2A_RNG_TICKET;
  rng.u_out = nullptr;
  int threads = 32;
  while (threads < batch) threads <<= 1;
  A0_LAUNCH(a0_k2a_unique, (unsigned)(total / batch), (unsigned)threads, 0, (cudaStream_t)stream_, 1, A0_PDL_K2, h->tree,
            (int32_t)h->P, h->D, batch, total / batch, top, beta, sum_offset, uniform, idx_out, prio_out, weight_out, stats_out,
            (const float*)(top < 0.0f ? h->dyn : nullptr), rng, h->fault_dev, (int32_t)(h->D < K2A_TOP ? h->D : K2A_TOP));
  return A0_OK;
}

// ------------------------------------------------------------------------------------------------
// K2b.  Leaves are written with a deterministic last-writer-wins rule:
//        mode 0: value = (loss+eps)^alpha, skipped when the leaf is 0; max_p = max(max_p, max loss)
//        mode 1: pos >= 0 -> max_p^alpha;  pos < 0 -> leaf ~pos = 0
//        mode 2: value = vals[k]
// and every touched ancestor is recomputed as fl32(left + right) -- never a delta, so the tree is
// bit-reproducible whatever the order of the updates.  Two implementations, same result:
//  * count <= K2P_MAX = 16384 (the training loop: B..20*B sampled indices, a few hundred marks per
//    append): a0_k2b_paths, ONE launch of one thread-block cluster (1..8 CTAs x 1024 threads, at
//    most two indices per thread, held in registers); the phases are separated by the hardware
//    cluster barrier.  After the leaf writes every index climbs three levels per phase up to
//    level 12: a thread loads the 8 siblings under its great-grandparent (two 16-byte L2 loads),
//    forms the 4 + 2 + 1 nodes above them and stores them; threads that share ancestors compute
//    identical values from identical inputs, so duplicate stores are benign -- but near the root
//    thousands of them would hit the same address, so levels 11..0 (4095 nodes) are instead
//    recomputed densely by CTA 0 in shared memory, one thread per node.  3 sparse phases + one
//    dense pass for a 1-2 M-leaf tree instead of 20-21 dependent levels.
//  * larger counts (bulk fills): a0_k2b_write (one CTA) marks the 4096-leaf chunks it touched and
//    a0_k2b_rebuild (one CTA per chunk) recomputes dirty chunks bottom-up in shared memory; the
//    last CTA to finish recomputes the levels above the chunk roots.  Work independent of count.
// ------------------------------------------------------------------------------------------------
constexpr int K2B_THREADS = 1024;

// Optional copy of the update's inputs for the host (a0_pt_update_report): the per-sample losses and
// indices are what BaseLearner.train hands back on the CPU (agent.py:163-169); writing them from the
// kernel that reads them anyway -- plain stores into mapped page-locked host memory -- replaces two
// device-to-host copies on the stream.
struct A0Report {
  int64_t* idx;
  float* loss;
};


__global__ void __launch_bounds__(K2B_THREADS)
a0_k2b_write(float* __restrict__ tree, int64_t P, int32_t chunk_log, int64_t N, const int64_t* __restrict__ idx64,
             const int32_t* __restrict__ idx32, const float* __restrict__ vals, int32_t count, int32_t mode,
             float alpha, float eps, float* __restrict__ max_p, int32_t* __restrict__ winner,
             int32_t* __restrict__ dirty, const A0Report rep) {
  __shared__ float red[K2B_THREADS / 32];
  A0_PDL_PROLOGUE();
  const int tid = threadIdx.x;
  const float maxp_in = *max_p;
  auto position = [&](int k) -> int64_t {
    if (mode == 1) { const int32_t p = idx32[k]; return p >= 0 ? p : ~p; }
    return idx64[k];
  };
  float local_max = 0.0f;
  for (int k = tid; k < count; k += K2B_THREADS) {          // claim
    const int64_t pos = position(k);
    if (rep.idx) { rep.idx[k] = pos; rep.loss[k] = vals[k]; }
    if (pos < 0 || pos >= N) continue;
    atomicMax(winner + pos, k);
    if (mode == 0 && a0_loss_ok(vals[k])) local_max = fmaxf(local_max, vals[k]);
  }
  __syncthreads();
  for (int k = tid; k < count; k += K2B_THREADS) {          // write
    const int64_t pos = position(k);
    if (pos < 0 || pos >= N) continue;
    if (__ldcg(winner + pos) != k) continue;
    float v;
    if (mode == 0) {
      if (!(__ldcg(tree + P + pos) > 0.0f) || !a0_loss_ok(vals[k])) continue;   // evicted since it was sampled / NaN loss
      v = a0_priority(vals[k], eps, alpha);
    } else if (mode == 1) {
      v = idx32[k] >= 0 ? (alpha == 0.5f ? sqrtf(maxp_in) : powf(maxp_in, alpha)) : 0.0f;
    } else {
      v = vals[k];
    }
    tree[P + pos] = v;
    dirty[pos >> chunk_log] = 1;
  }
  __syncthreads();
  for (int k = tid; k < count; k += K2B_THREADS) {          // release
    const int64_t pos = position(k);
    if (pos >= 0 && pos < N) winner[pos] = -1;
  }
  if (mode == 0) {
    local_max = a0_warp_max(local_max);
    if ((tid & 31) == 0) red[tid >> 5] = local_max;
    __syncthreads();
    if (tid == 0) {
      float mx = maxp_in;
      for (int i = 0; i < K2B_THREADS / 32; ++i) mx = fmaxf(mx, red[i]);
      *max_p = mx;
    }
  }
}

constexpr int K2R_THREADS = 512;
constexpr int K2R_MAXLOG = 12;      // chunk of up to 4096 leaves; up to 4096 chunk roots above

// Reduce `n = 1 << levels` values held in buf[0][0..n) up to one value, writing every level to the
// tree: the node at `levels - l` levels above the inputs, i-th of its row, goes to tree[base(l) + i].
__device__ __forceinline__ void a0_reduce_levels(float (*buf)[1 << K2R_MAXLOG], int levels, float* tree,
                                                 int64_t row0, int64_t first) {
  // inputs sit at tree row `row0 + levels` (depth), starting at column `first << levels`
  int cur = 0;
  for (int l = levels - 1; l >= 0; --l) {
    const int cnt = 1 << l;
    const int64_t base = ((int64_t)1 << (row0 + l)) + (first << l);
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
      const float v = __fadd_rn(buf[cur][2 * i], buf[cur][2 * i + 1]);
      buf[cur ^ 1][i] = v;
      tree[base + i] = v;
    }
    __syncthreads();
    cur ^= 1;
  }
}

__global__ void __launch_bounds__(K2R_THREADS)
a0_k2b_rebuild(float* __restrict__ tree, int32_t D, int32_t chunk_log, int32_t* __restrict__ dirty,
               unsigned int* __restrict__ ticket) {
  __shared__ float buf[2][1 << K2R_MAXLOG];
  __shared__ bool is_last;
  A0_PDL_PROLOGUE();
  const int c = blockIdx.x;
  const int top_levels = D - chunk_log;                  // depth of the chunk roots
  if (__ldcg(dirty + c) != 0) {
    const int n = 1 << chunk_log;
    const float* leaves = tree + ((int64_t)1 << D) + ((int64_t)c << chunk_log);
    for (int i = threadIdx.x; i < n; i += blockDim.x) buf[0][i] = __ldcg(leaves + i);
    __syncthreads();
    a0_reduce_levels(buf, chunk_log, tree, top_levels, c);
    if (threadIdx.x == 0) dirty[c] = 0;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  if (top_levels > 0) {
    const int n = 1 << top_levels;
    const float* roots = tree + ((int64_t)1 << top_levels);
    for (int i = threadIdx.x; i < n; i += blockDim.x) buf[0][i] = __ldcg(roots + i);
    __syncthreads();
    a0_reduce_levels(buf, top_levels, tree, 0, 0);
  }
  if (threadIdx.x == 0) *ticket = 0u;
}

constexpr int K2P_THREADS = 1024;
constexpr int K2P_CLUSTER = 8;                      // portable cluster size
constexpr int K2P_PER_THREAD = 2;
constexpr int K2P_MAX = K2P_THREADS * K2P_CLUSTER * K2P_PER_THREAD;   // 16384 indices per launch

// All CTAs of the launch form ONE thread-block cluster, so the hardware cluster barrier is a
// grid-wide barrier; release/acquire at cluster scope orders the L2-level (ld.cg/st.cg) accesses.
__device__ __forceinline__ void a0_cluster_sync(bool single_cta) {
  if (single_cta) { __syncthreads(); return; }
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// One climb of L levels for all of a thread's indices: load the 2^L siblings under the L-th
// ancestor (16-byte L2 loads, all issued before any arithmetic), reduce pairwise level by level
// with fl32 adds and store every level with the widest vectors that fit.
constexpr int K2P_TOP = 12;              // levels 0..11 (4095 nodes) are rebuilt densely in shared memory
constexpr int K2P_LEVELS_DEFAULT = 3;   // levels per phase: 8 (3) or 16 (4) siblings per index; A0_OPT_K2B_LEVELS

template <int L>
__device__ __forceinline__ void a0_climb_all(float* __restrict__ tree, int64_t P, const int64_t (&pos)[K2P_PER_THREAD],
                                             int shift) {
  constexpr int W = 1 << L;
  float v[K2P_PER_THREAD][W];
  int64_t x[K2P_PER_THREAD];
#pragma unroll
  for (int s = 0; s < K2P_PER_THREAD; ++s) {
    x[s] = ((P + (pos[s] < 0 ? 0 : pos[s])) >> shift) & ~(int64_t)(W - 1);
    if (pos[s] < 0) continue;
    if (L == 1) {
      const float2 t = __ldcg(reinterpret_cast<const float2*>(tree + x[s]));
      v[s][0] = t.x; v[s][1] = t.y;
    } else {
#pragma unroll
      for (int i = 0; i < W / 4; ++i) {
        const float4 t = __ldcg(reinterpret_cast<const float4*>(tree + x[s]) + i);
        v[s][4 * i] = t.x; v[s][4 * i + 1] = t.y; v[s][4 * i + 2] = t.z; v[s][4 * i + 3] = t.w;
      }
    }
  }
#pragma unroll
  for (int s = 0; s < K2P_PER_THREAD; ++s) {
    if (pos[s] < 0) continue;
#pragma unroll
    for (int l = 1; l <= L; ++l) {
      const int cnt = W >> l;
#pragma unroll
      for (int i = 0; i < cnt; ++i) v[s][i] = __fadd_rn(v[s][2 * i], v[s][2 * i + 1]);
      float* dst = tree + (x[s] >> l);
      if (cnt >= 4) {
#pragma unroll
        for (int i = 0; i < cnt / 4; ++i)
          __stcg(reinterpret_cast<float4*>(dst) + i, make_float4(v[s][4 * i], v[s][4 * i + 1], v[s][4 * i + 2], v[s][4 * i + 3]));
      } else if (cnt == 2) {
        __stcg(reinterpret_cast<float2*>(dst), make_float2(v[s][0], v[s][1]));
      } else {
        __stcg(dst, v[s][0]);
      }
    }
  }
}

// Reduces the 2^levels values in heap[n .. 2n) (n = 2^levels, heap in shared memory, heap[i] = node i of
// the sub-tree) down to heap[1]; every thread of a 1024-thread CTA calls it.  A 1024-thread barrier
// costs ~300 cycles here (device timeline), so levels are combined inside threads and by warp shuffles:
// two block barriers for 4096 inputs (four per thread: two levels in the thread, five by shuffles,
// barrier, five by warp 0), two for <= 1024 inputs, one per level only for 2048.
template <int T>
__device__ __forceinline__ void a0_heap_reduce(float* heap, int levels) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = 1 << levels;
  constexpr int PER = 4096 / T;                    // inputs per thread at 4096
  constexpr int LOGPER = PER == 4 ? 2 : PER == 8 ? 3 : PER == 16 ? 4 : 5;
  constexpr int WARPS = T / 32;
  constexpr int REM = WARPS == 32 ? 5 : WARPS == 16 ? 4 : WARPS == 8 ? 3 : 2;
  static_assert(PER >= 4 && PER <= 32 && WARPS >= 4, "a0_heap_reduce: 128..1024 threads");
  if (levels == 12) {
    float v[PER];
#pragma unroll
    for (int i = 0; i < PER / 4; ++i) {
      const float4 q4 = *reinterpret_cast<const float4*>(heap + n + PER * tid + 4 * i);
      v[4 * i] = q4.x; v[4 * i + 1] = q4.y; v[4 * i + 2] = q4.z; v[4 * i + 3] = q4.w;
    }
#pragma unroll
    for (int lev = 1; lev <= LOGPER; ++lev) {      // levels inside the thread
      const int cnt = PER >> lev;
#pragma unroll
      for (int i = 0; i < cnt; ++i) v[i] = __fadd_rn(v[2 * i], v[2 * i + 1]);
      float* dst = heap + (n >> lev) + cnt * tid;
#pragma unroll
      for (int i = 0; i < cnt; ++i) dst[i] = v[i];
    }
    float x = v[0];
#pragma unroll
    for (int j = 1; j <= 5; ++j) {                 // five levels by warp shuffles
      x = __fadd_rn(x, __shfl_down_sync(0xffffffffu, x, 1 << (j - 1)));       // left child + right child
      if ((lane & ((1 << j) - 1)) == 0) heap[(n >> (LOGPER + j)) + (tid >> j)] = x;
    }
    __syncthreads();
    if (warp == 0) {                               // the last REM levels: WARPS values
      x = lane < WARPS ? heap[WARPS + lane] : 0.0f;
#pragma unroll
      for (int j = 1; j <= REM; ++j) {
        x = __fadd_rn(x, __shfl_down_sync(0xffffffffu, x, 1 << (j - 1)));
        if (lane < WARPS && (lane & ((1 << j) - 1)) == 0) heap[(WARPS >> j) + (lane >> j)] = x;
      }
    }
    __syncthreads();
  } else if (n <= T) {
    float v = tid < n ? heap[n + tid] : 0.0f;
    const int first = levels < 5 ? levels : 5;
#pragma unroll
    for (int j = 1; j <= 5; ++j) {
      if (j <= first) {
        v = __fadd_rn(v, __shfl_down_sync(0xffffffffu, v, 1 << (j - 1)));
        if (tid < n && (lane & ((1 << j) - 1)) == 0) heap[(n >> j) + (tid >> j)] = v;
      }
    }
    __syncthreads();
    const int rem = levels - first;                        // <= 5 levels left, 2^rem <= 32 values
    if (warp == 0 && rem > 0) {
      const int m = 1 << rem;
      v = lane < m ? heap[m + lane] : 0.0f;
#pragma unroll
      for (int j = 1; j <= 5; ++j) {
        if (j <= rem) {
          v = __fadd_rn(v, __shfl_down_sync(0xffffffffu, v, 1 << (j - 1)));
          if (lane < m && (lane & ((1 << j) - 1)) == 0) heap[(m >> j) + (lane >> j)] = v;
        }
      }
    }
    __syncthreads();
  } else {
    for (int l = levels - 1; l >= 0; --l) {
      const int cnt = 1 << l;
      for (int i = cnt + tid; i < 2 * cnt; i += T) heap[i] = __fadd_rn(heap[2 * i], heap[2 * i + 1]);
      __syncthreads();
    }
  }
}
// Levels top-1 .. 0 of the whole tree from its 2^top level-`top` nodes in heap[n .. 2n): reduce, write out.
template <int T>
__device__ __forceinline__ void a0_dense_top(float* heap, int top, float* __restrict__ tree) {
  a0_heap_reduce<T>(heap, top);
  const int n = 1 << top;
  for (int i = threadIdx.x; i < n; i += T)
    if (i >= 1) tree[i] = heap[i];
}

// `cta` of `nctas` CTAs (one cluster when nctas > 1) run this body; the caller has executed the PDL prologue.
template <int K2P_LEVELS>
__device__ __forceinline__ void
a0_paths_body(float* __restrict__ tree, int64_t P, int32_t D, int64_t N, const int64_t* __restrict__ idx64,
              const int32_t* __restrict__ idx32, const float* __restrict__ vals, int32_t count, int32_t mode,
              float alpha, float eps, float* __restrict__ max_p, int32_t* __restrict__ winner,
              int32_t* __restrict__ dirty, int32_t chunk_log, const int cta, const int nctas, const A0Report rep,
              unsigned long long* _tx = nullptr) {
#ifdef A0_TRACE
#define K2B_TX(i) do { if (_tx) _tx[i] = (unsigned long long)clock64(); } while (0)
#else
#define K2B_TX(i) do {} while (0)
#endif
  const bool single = nctas == 1;
  const int gtid = cta * K2P_THREADS + threadIdx.x;
  const int gstride = nctas * K2P_THREADS;
  const float maxp_in = __ldcg(max_p);
  // this thread's (at most K2P_PER_THREAD) indices, kept in registers for all phases
  int64_t pos[K2P_PER_THREAD];
  int kk[K2P_PER_THREAD];
  float val[K2P_PER_THREAD];
#pragma unroll
  for (int s = 0; s < K2P_PER_THREAD; ++s) {
    const int k = gtid + s * gstride;
    kk[s] = k;
    pos[s] = -1;
    val[s] = 0.0f;
    if (k < count) {
      int64_t p;
      bool set = true;
      if (mode == 1) { const int32_t q = idx32[k]; set = q >= 0; p = set ? q : ~q; }
      else p = idx64[k];
      if (rep.idx) { rep.idx[k] = p; rep.loss[k] = vals[k]; }
      if (p >= 0 && p < N) {
        pos[s] = p;
        if (mode == 0) val[s] = vals[k];
        else if (mode == 1) val[s] = set ? 1.0f : 0.0f;
        else val[s] = vals[k];
      }
    }
  }
  // the leaf's current value is only compared with 0 (evicted since it was sampled?): nothing in this
  // launch can turn a live leaf into 0 or back (mode 0), so it is fetched here, in the same memory round
  // trip as the claim, instead of after the winner is known
  float old_leaf[K2P_PER_THREAD];
#pragma unroll
  for (int s = 0; s < K2P_PER_THREAD; ++s) old_leaf[s] = (mode == 0 && pos[s] >= 0) ? __ldcg(tree + P + pos[s]) : 1.0f;
#pragma unroll
  for (int s = 0; s < K2P_PER_THREAD; ++s)                   // claim
    if (pos[s] >= 0) atomicMax(winner + pos[s], kk[s]);
  if (mode == 0) {
    float mx = 0.0f;
#pragma unroll
    for (int s = 0; s < K2P_PER_THREAD; ++s) mx = fmaxf(mx, pos[s] >= 0 && a0_loss_ok(val[s]) ? val[s] : 0.0f);
    mx = a0_warp_max(mx);
    if ((threadIdx.x & 31) == 0) a0_atomic_max_pos(max_p, mx);   // max_p = max(max_p, max loss), replay.py:59
  }
  a0_cluster_sync(single);
  K2B_TX(0);
#pragma unroll
  for (int s = 0; s < K2P_PER_THREAD; ++s) {                 // write (the highest k wins)
    if (pos[s] < 0 || __ldcg(winner + pos[s]) != kk[s]) continue;
    float v;
    if (mode == 0) {
      if (!(old_leaf[s] > 0.0f) || !a0_loss_ok(val[s])) continue;   // evicted since it was sampled / NaN loss
      v = a0_priority(val[s], eps, alpha);
    } else if (mode == 1) {
      v = val[s] != 0.0f ? (alpha == 0.5f ? sqrtf(maxp_in) : powf(maxp_in, alpha)) : 0.0f;
    } else {
      v = val[s];
    }
    __stcg(tree + P + pos[s], v);
    if (dirty) dirty[pos[s] >> chunk_log] = 1;               // hybrid: a0_k2b_rebuild recomputes the touched chunks
  }
  a0_cluster_sync(single);
  K2B_TX(1);
#pragma unroll
  for (int s = 0; s < K2P_PER_THREAD; ++s)                   // release
    if (pos[s] >= 0) winner[pos[s]] = -1;
  if (dirty) return;
  // ---- propagate, sparse part: climb from the leaves (level D) to level `top` ---------------------
  // Near the root every index shares its ancestors with every other one (10 240 stores to the
  // root per phase serialise in L2), so the per-index climb stops at level `top` <= K2P_TOP and the
  // levels above are recomputed densely below, one thread per node and no duplicate stores.
  const int top = D < K2P_TOP ? D : K2P_TOP;
  int depth = D;
  int shift = 0;                 // node of an index at `depth` = (P + pos) >> shift
  const int first = (D - top) % K2P_LEVELS;      // a short climb first, then whole groups of K2P_LEVELS
  if (first) {
    switch (first) {
      case 1: a0_climb_all<1>(tree, P, pos, shift); break;
      case 2: a0_climb_all<2>(tree, P, pos, shift); break;
      default: if (K2P_LEVELS > 3) a0_climb_all<3>(tree, P, pos, shift); break;
    }
    depth -= first;
    shift += first;
    a0_cluster_sync(single);
    K2B_TX(2);
  }
  while (depth > top) {
    a0_climb_all<K2P_LEVELS>(tree, P, pos, shift);
    depth -= K2P_LEVELS;
    shift += K2P_LEVELS;
    a0_cluster_sync(single);
    K2B_TX(3);
  }
  // ---- dense part: CTA 0 rebuilds levels top-1 .. 0 from the 2^top nodes of level `top` -----------
  if (cta != 0 || top == 0) return;
  __shared__ __align__(16) float heap[2 << K2P_TOP];         // heap[i] = node i, i < 2n
  const int n = 1 << top;
  K2B_TX(4);
  for (int i = threadIdx.x; i < n; i += K2P_THREADS) heap[n + i] = __ldcg(tree + n + i);
  __syncthreads();
  K2B_TX(5);
  a0_dense_top<1024>(heap, top, tree);
  K2B_TX(6);
}

template <int K2P_LEVELS>
__global__ void __launch_bounds__(K2P_THREADS)
a0_k2b_paths(float* __restrict__ tree, int64_t P, int32_t D, int64_t N, const int64_t* __restrict__ idx64,
             const int32_t* __restrict__ idx32, const float* __restrict__ vals, int32_t count, int32_t mode,
             float alpha, float eps, float* __restrict__ max_p, int32_t* __restrict__ winner,
             int32_t* __restrict__ dirty, int32_t chunk_log, const A0Report rep) {
  A0_T0();
  A0_PDL_PROLOGUE();
  A0_TMID();
#ifdef A0_TRACE
  const long long _c0 = clock64();
  a0_paths_body<K2P_LEVELS>(tree, P, D, N, idx64, idx32, vals, count, mode, alpha, eps, max_p, winner, dirty, chunk_log,
                            (int)blockIdx.x, (int)gridDim.x, rep, threadIdx.x == 0 ? _tx : nullptr);
  _tx[7] = (unsigned long long)_c0;
#else
  a0_paths_body<K2P_LEVELS>(tree, P, D, N, idx64, idx32, vals, count, mode, alpha, eps, max_p, winner, dirty, chunk_log,
                            (int)blockIdx.x, (int)gridDim.x, rep);
#endif
  if (threadIdx.x == 0) A0_TEND(5);
}

// ------------------------------------------------------------------------------------------------
// K2b for small counts (<= 1024 indices: the 640 sampled indices of a batch-32 Trainer.step, the marks
// of a step's append).  The cluster path climb above communicates between its phases through global
// memory: every phase is a store, a barrier and a dependent load -- two L2 traversals -- and the device
// timeline (tools/trace_step.py) shows ~3000 SM cycles per phase, 20 000 for a 640-index update.
// Here ONE CTA keeps everything it produces in shared memory:
//   * the kernel's global LOADS are issued in two batches at the start (indices; then old leaf + the
//     sibling of every node on the sparse part of the path + the 4096 nodes of level 12): two L2 round
//     trips in total, nothing loaded later depends on anything stored by this kernel;
//   * a shared-memory hash map node -> value holds every node this launch has recomputed.  Duplicate
//     indices meet in the map (atomicMax ticket: the highest k wins, as `priority[ids] = ...` does);
//     per level an index combines its node with the sibling's value -- from the map if this launch
//     changed it, else the prefetched one -- and publishes the parent; phases are separated by
//     __syncthreads() only;
//   * levels 11..0 are rebuilt densely in a shared-memory heap and written out in one sweep; all
//     global STORES are fire-and-forget.
// Every node is still fl32(left + right) of its two children: the tree is bit-identical to the other
// schedules' (tests).
// ------------------------------------------------------------------------------------------------
constexpr int K2S_THREADS = 1024;
constexpr int K2S_SLOT_LOG = 14;
constexpr int K2S_SLOTS = 1 << K2S_SLOT_LOG;          // 1024 indices x (<= 12 sparse levels + leaf) at load <= 0.81
constexpr int K2S_MAX_SPARSE = 12;                    // D - 12 <= 12: trees of up to 2^24 leaves (the handle's limit)
constexpr size_t K2S_SMEM = (size_t)K2S_SLOTS * 8;    // keys + values (128 KB); the dense heap (32 KB) reuses it

__device__ __forceinline__ uint32_t a0_k2s_hash(uint32_t id) { return (id * 2654435761u) >> (32 - K2S_SLOT_LOG); }
// slot of node `id`, claiming an empty one when it is not in the map yet (node ids are >= 1; 0 = empty)
__device__ __forceinline__ uint32_t a0_k2s_insert(uint32_t* keys, uint32_t id) {
  uint32_t s = a0_k2s_hash(id);
  while (true) {
    const uint32_t prev = atomicCAS(keys + s, 0u, id);
    if (prev == 0u || prev == id) return s;
    s = (s + 1) & (K2S_SLOTS - 1);
  }
}
// slot of node `id`, or -1.  Entries are never removed, so a key inserted before the last barrier is
// found before the probe reaches an empty slot, whatever is being inserted concurrently.
__device__ __forceinline__ int a0_k2s_find(const volatile uint32_t* keys, uint32_t id) {
  uint32_t s = a0_k2s_hash(id);
  while (true) {
    const uint32_t k = keys[s];
    if (k == id) return (int)s;
    if (k == 0u) return -1;
    s = (s + 1) & (K2S_SLOTS - 1);
  }
}

// A load the compiler may not sink to its first use: these are issued up front on purpose.
__device__ __forceinline__ float a0_ld_now(const float* p) {
  float v;
  asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ void
a0_small_body(float* __restrict__ tree, int64_t P, int32_t D, int64_t N, const int64_t* __restrict__ idx64,
              const int32_t* __restrict__ idx32, const float* __restrict__ vals, int32_t count, int32_t mode,
              float alpha, float eps, float* __restrict__ max_p, const A0Report rep, uint8_t* smem,
              unsigned long long* _tx = nullptr) {
  uint32_t* keys = reinterpret_cast<uint32_t*>(smem);
  uint32_t* tval = keys + K2S_SLOTS;
  float* heap = reinterpret_cast<float*>(smem);         // after the sparse levels: heap[i] = node i, i < 2n
  const int tid = threadIdx.x;
  const int top = D < K2P_TOP ? D : K2P_TOP;
  const int S = D - top;                                // sparse levels D .. top+1 climb through the map
  const int n = 1 << top;
  // ---- loads that do not depend on the indices ------------------------------------------------------
  const float maxp_in = __ldcg(max_p);
  float dn[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) dn[q] = (4 * tid + q < n) ? a0_ld_now(tree + n + 4 * tid + q) : 0.0f;
  int64_t pos = -1;
  float val = 0.0f;
  if (tid < count) {
    int64_t p;
    bool set = true;
    if (mode == 1) { const int32_t q = idx32[tid]; set = q >= 0; p = set ? q : ~q; }
    else p = idx64[tid];
    if (rep.idx) { rep.idx[tid] = p; rep.loss[tid] = vals[tid]; }
    if (p >= 0 && p < N) {
      pos = p;
      val = mode == 1 ? (set ? 1.0f : 0.0f) : vals[tid];
    }
  }
  {   // clear the map while those loads are in flight
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
    uint4* t4 = reinterpret_cast<uint4*>(smem);
    for (int i = tid; i < (int)(K2S_SMEM / 16); i += K2S_THREADS) t4[i] = z;
  }
  const bool valid = pos >= 0;
  const uint32_t leaf = (uint32_t)(P + (valid ? pos : 0));
  // ---- loads that depend on the index: the old leaf and the siblings along the sparse path -----------
  float old_leaf = 0.0f, sib[K2S_MAX_SPARSE];
#pragma unroll
  for (int s = 0; s < K2S_MAX_SPARSE; ++s) sib[s] = 0.0f;
  if (valid) {
    old_leaf = a0_ld_now(tree + leaf);
#pragma unroll
    for (int s = 0; s < K2S_MAX_SPARSE; ++s)
      if (s < S) sib[s] = a0_ld_now(tree + ((leaf >> s) ^ 1u));
  }
  if (mode == 0) {
    const float mx = a0_warp_max(valid && a0_loss_ok(val) ? val : 0.0f);
    if ((tid & 31) == 0) a0_atomic_max_pos(max_p, mx);      // max_p = max(max_p, max loss), replay.py:59
  }
  __syncthreads();                                          // the map is empty
  K2B_TX(0);
  uint32_t slot = 0;
  if (valid) {
    slot = a0_k2s_insert(keys, leaf);
    atomicMax(tval + slot, (uint32_t)tid + 1u);             // duplicates: the highest k wins
  }
  __syncthreads();
  const bool active = valid && tval[slot] == (uint32_t)tid + 1u;
  __syncthreads();                                          // every ticket has been read
  K2B_TX(1);
  float myv = 0.0f;
  if (active) {
    bool store = true;
    if (mode == 0) {
      store = old_leaf > 0.0f && a0_loss_ok(val);           // evicted since it was sampled (the leaf stays 0) / NaN loss
      myv = store ? a0_priority(val, eps, alpha) : old_leaf;
    } else if (mode == 1) {
      myv = val != 0.0f ? (alpha == 0.5f ? sqrtf(maxp_in) : powf(maxp_in, alpha)) : 0.0f;
    } else {
      myv = val;
    }
    tval[slot] = __float_as_uint(myv);
    if (store) __stcg(tree + leaf, myv);
  }
  __syncthreads();
  K2B_TX(2);
  // ---- sparse levels: parent = fl32(node + sibling), sibling from the map when this launch changed it --
  uint32_t cur = leaf;
  uint32_t onode[K2S_MAX_SPARSE];
  float oval[K2S_MAX_SPARSE];
#pragma unroll
  for (int s = 0; s < K2S_MAX_SPARSE; ++s) {
    if (s < S) {
      if (active) {
        const int f = a0_k2s_find(keys, cur ^ 1u);
        const float sv = f >= 0 ? __uint_as_float(tval[f]) : sib[s];
        myv = __fadd_rn(myv, sv);
        cur >>= 1;
        tval[a0_k2s_insert(keys, cur)] = __float_as_uint(myv);    // indices that share the parent store the same bits
        onode[s] = cur;
        oval[s] = myv;
      }
      __syncthreads();
    }
  }
  if (active) {
#pragma unroll
    for (int s = 0; s < K2S_MAX_SPARSE; ++s)
      if (s < S) __stcg(tree + onode[s], oval[s]);
  }
  K2B_TX(3);
  // ---- dense part: levels top-1 .. 0 in a shared-memory heap (the map is dead: same memory) ----------
  __syncthreads();
#pragma unroll
  for (int q = 0; q < 4; ++q)
    if (4 * tid + q < n) heap[n + 4 * tid + q] = dn[q];
  __syncthreads();
  if (active) heap[cur] = myv;                              // cur is the index's level-`top` ancestor, in [n, 2n)
  __syncthreads();
  K2B_TX(4);
  a0_dense_top<1024>(heap, top, tree);
  K2B_TX(6);
}

__global__ void __launch_bounds__(K2S_THREADS)
a0_k2b_small(float* __restrict__ tree, int64_t P, int32_t D, int64_t N, const int64_t* __restrict__ idx64,
             const int32_t* __restrict__ idx32, const float* __restrict__ vals, int32_t count, int32_t mode,
             float alpha, float eps, float* __restrict__ max_p, const A0Report rep) {
  extern __shared__ __align__(16) uint8_t a0_k2s_smem[];
  A0_T0();
  A0_PDL_PROLOGUE();
  A0_TMID();
#ifdef A0_TRACE
  const long long _c0 = clock64();
  a0_small_body(tree, P, D, N, idx64, idx32, vals, count, mode, alpha, eps, max_p, rep, a0_k2s_smem, threadIdx.x == 0 ? _tx : nullptr);
  _tx[7] = (unsigned long long)_c0;
#else
  a0_small_body(tree, P, D, N, idx64, idx32, vals, count, mode, alpha, eps, max_p, rep, a0_k2s_smem);
#endif
  if (threadIdx.x == 0) A0_TEND(5);
}

static int g_k2b_small = -1;
static bool a0_option_k2b_small() {
  if (g_k2b_small < 0) {
    const char* e = getenv("A0_K2B_SMALL");
    g_k2b_small = e ? (atoi(e) != 0) : 0;      // measured slower at 640 indices (shared-memory CAS throughput), see DESIGN.md
  }
  return g_k2b_small != 0;
}
void a0_set_k2b_small(int on) { g_k2b_small = on != 0; }

template <typename K>
static int a0_k2s_smem_attr(a0_replay_t* h, K kernel, bool* done) {
  if (h->device < 64 && !done[h->device]) {
    A0_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K2S_SMEM));
    done[h->device] = true;
  }
  return A0_OK;
}

// A small ingest in ONE launch: CTA 0 applies the marks to the tree (the shared-memory update above),
// CTAs 1..n_new copy one new frame each, the rest scatter the record metadata (K1).  The two halves
// touch disjoint state (tree / max_p vs frames / records), so they need no ordering inside the
// launch; everything that samples runs after it in stream order.  Thread 0 also publishes the
// sampler's dynamic scalars when asked to.
constexpr int K1M_MAX_MARKS = K2S_THREADS;                      // one mark per thread of CTA 0
constexpr int K1M_MAX_FRAMES = 140;                             // one wave of CTAs (each reserves CTA 0's 128 KB); larger appends: K1's own launch
__global__ void __launch_bounds__(K2S_THREADS)
a0_k1_append_mark(float* __restrict__ tree, int64_t P, int32_t D, int64_t N, const int32_t* __restrict__ marks,
                  int32_t n_marks, float alpha, float* __restrict__ max_p,
                  uint8_t* __restrict__ frames, int32_t F, int64_t NF, const uint8_t* __restrict__ staged,
                  const int32_t* __restrict__ new_pos, const int32_t* __restrict__ src_idx, int32_t n_new,
                  int32_t* __restrict__ rec_slots, A0RecInfo* __restrict__ rec_info, const int32_t* __restrict__ meta,
                  int32_t m, const A0Dyn dyn) {
  extern __shared__ __align__(16) uint8_t a0_k2s_smem[];
  A0_PDL_PROLOGUE();
  if (blockIdx.x == 0) {
    if (dyn.dyn && threadIdx.x == 0) { dyn.dyn[0] = dyn.top; dyn.dyn[1] = dyn.beta; dyn.dyn[2] = dyn.sum_offset; }
    const A0Report none = {nullptr, nullptr};
    a0_small_body(tree, P, D, N, nullptr, marks, nullptr, n_marks, 1, alpha, 0.0f, max_p, none, a0_k2s_smem);
    return;
  }
  const int blk = (int)blockIdx.x - 1;
  if (blk < n_new) {
    a0_k1_copy_frame(frames, F, NF, staged, new_pos, src_idx, blk, threadIdx.x, K2S_THREADS);
    return;
  }
  const int r = (blk - n_new) * K2S_THREADS + threadIdx.x;
  if (r < m) a0_k1_write_record(rec_slots, rec_info, N, meta, r);
}

int a0_launch_mark_append(a0_replay* h, const int32_t* marks, int32_t n_marks, float alpha, const uint8_t* new_frames,
                          const int32_t* new_frame_pos, const int32_t* src_idx, int32_t n_new, const int32_t* rec_meta,
                          int32_t m, const A0Dyn& dyn, cudaStream_t stream) {
  if (n_marks <= 0 || n_marks > K1M_MAX_MARKS || n_new > K1M_MAX_FRAMES || h->D - K2P_TOP > K2S_MAX_SPARSE) return A0_NOFIT;
  static thread_local bool attr[64] = {false};
  int rc = a0_k2s_smem_attr(h, a0_k1_append_mark, attr);
  if (rc) return rc;
  const int blocks = 1 + n_new + (m + K2S_THREADS - 1) / K2S_THREADS;
  A0_LAUNCH(a0_k1_append_mark, (unsigned)blocks, K2S_THREADS, K2S_SMEM, stream, 1, A0_PDL_K1, h->tree, h->P, h->D, h->N, marks, n_marks,
            alpha, h->max_p, h->frames, h->F, h->NF, new_frames, new_frame_pos, src_idx, n_new, h->rec_slots, h->rec_info,
            rec_meta, m, dyn);
  return A0_OK;
}

// ------------------------------------------------------------------------------------------------
// K2b, one CTA per 4096-leaf chunk of the tree (trees of up to 2 M leaves: <= 512 CTAs, all resident).
// The schedules above pay one L2 round trip and one barrier per PHASE (claim / write / release / three
// climbs / dense top: ~3000 cycles each on the device timeline, 19 000 for 640 indices) because their
// threads hand values to each other through global memory.  Here nothing a CTA needs is produced by
// another CTA until the very end:
//   * every CTA scans the whole index list (640 .. 16 384 entries, a few KB from L2) and keeps the
//     entries that fall into its chunk; duplicates meet in a shared-memory ticket array (atomicMax:
//     the highest k wins, as `priority[ids] = ...`);
//   * it loads its 4096 leaves (one coalesced round trip, overlapped with the scan), overlays the new
//     values, recomputes the chunk's 12 levels in shared memory (two block barriers) and writes back
//     only the nodes on the updated paths;
//   * the last CTA to finish (ticket) recomputes the levels above the chunk roots.
// Two dependent L2 round trips + one grid-wide ticket for any number of indices.  Every node is
// fl32(left + right) of its children, as everywhere else: the same tree, bit for bit (tests).
// ------------------------------------------------------------------------------------------------
constexpr int K2C_THREADS = 1024;                             // (256 fatter threads measured the same: 75.4 vs 74.9 us per step)
constexpr int K2C_LOG = 12;                                  // leaves per chunk = 4096
constexpr int K2C_MAX_COUNT_DEFAULT = 16384;                 // A0_K2B_CHUNK_MAX: largest index list this schedule takes (2048 before the match list)
constexpr int K2C_MAX_CHUNKS = 592;                          // 148 SMs x 4: beyond that (> 2 M leaves) the other schedules run
constexpr int K2C_MATCH_CAP = 1024;                          // entries of the index list a chunk remembers from its one scan
constexpr size_t K2C_SMEM = ((size_t)2 << K2C_LOG) * 4 + ((size_t)1 << K2C_LOG) * 4 + (size_t)K2C_MATCH_CAP * 8;    // heap + tickets + match list = 56 KB
constexpr int K2C_SPARSE_MAX = 32;                           // updated leaves per chunk climbed path by path (one lane each)

__global__ void __launch_bounds__(K2C_THREADS)
a0_k2b_chunks(float* __restrict__ tree, int64_t P, int32_t D, int64_t N, const int64_t* __restrict__ idx64,
              const int32_t* __restrict__ idx32, const float* __restrict__ vals, int32_t count, int32_t mode,
              float alpha, float eps, float* __restrict__ max_p, unsigned int* __restrict__ ticket, const A0Report rep,
              int32_t early, int32_t sparse_max) {
  extern __shared__ __align__(16) uint8_t a0_k2c_smem[];
  __shared__ int s_dirty;
  __shared__ bool s_last;
  __shared__ int s_nwin;                                     // distinct leaves of this chunk in the index list
  __shared__ int s_nmatch;                                   // entries of the index list that fall into this chunk
  __shared__ int s_list[K2C_SPARSE_MAX];
  float* heap = reinterpret_cast<float*>(a0_k2c_smem);                      // heap[i] = node i of the chunk's sub-tree
  int* win = reinterpret_cast<int*>(a0_k2c_smem + ((size_t)2 << K2C_LOG) * 4);
  int* m_k = win + ((size_t)1 << K2C_LOG);                   // the chunk's entries, remembered by the one scan of the list:
  int* m_l = m_k + K2C_MATCH_CAP;                            // index k, leaf l (bit 31: an "unset" mark)
  A0_T0();
  // early (a0_pt_update_overlapped): launched programmatically under its predecessor -- the last K4 of a step -- the
  // kernel loads its leaves and builds its tickets (positions only) while that kernel is still running, and waits
  // for it only where the loss values are first needed.  Everything OLDER than the predecessor is complete when
  // this grid starts (the predecessor triggered after its own wait), which is what the caller guarantees for idx.
  if (!early) A0_PDL_PROLOGUE();
  A0_TMID();
#ifdef A0_TRACE
  const long long _c0 = clock64();
#define K2C_TX(i) _tx[i] = (unsigned long long)clock64()
#else
#define K2C_TX(i) do {} while (0)
#endif
  const int tid = threadIdx.x;
  const int c = blockIdx.x;
  const int clog = D < K2C_LOG ? D : K2C_LOG;
  const int n = 1 << clog;
  const int top_levels = D - clog;                           // depth of the chunk roots
  const int64_t lo = (int64_t)c << clog;                    // first leaf of the chunk
  if (tid == 0) { s_dirty = 0; s_nwin = 0; s_nmatch = 0; }
  if (n >= 4) {
    const float4* src = reinterpret_cast<const float4*>(tree + P + lo);
    for (int i = tid; i < (n >> 2); i += K2C_THREADS) {
      reinterpret_cast<float4*>(heap + n)[i] = __ldcg(src + i);
      reinterpret_cast<int4*>(win)[i] = make_int4(-1, -1, -1, -1);
    }
  } else {
    for (int i = tid; i < n; i += K2C_THREADS) {
      heap[n + i] = __ldcg(tree + P + lo + i);
      win[i] = -1;
    }
  }
  auto position = [&](int k, bool& set) -> int64_t {
    set = true;
    if (mode == 1) { const int32_t q = idx32[k]; set = q >= 0; return set ? q : ~q; }
    return idx64[k];
  };
  __syncthreads();
  K2C_TX(0);
  // ---- pass 1: the ONE scan of the index list: tickets for the entries of this chunk (positions only), and the
  //      entries themselves into the match list, so that the later passes walk a few dozen entries instead of
  //      re-reading the whole list (three scans of 10 240 indices by each of 256 CTAs were what kept this schedule
  //      behind the leaf-write + rebuild pair at batch 512).  A chunk with more entries than the list holds falls
  //      back to re-scanning.
  for (int k = tid; k < count; k += K2C_THREADS) {
    bool set;
    const int64_t p = position(k, set);
    if (p >= lo && p < lo + n && p < N) {
      const int l = (int)(p - lo);
      atomicMax(win + l, k);
      const int slot = atomicAdd(&s_nmatch, 1);
      if (slot < K2C_MATCH_CAP) { m_k[slot] = k; m_l[slot] = set ? l : (l | (int)0x80000000); }
    }
  }
  __syncthreads();                                           // tickets and match list final
  const int nmatch = s_nmatch;
  const bool listed = nmatch <= K2C_MATCH_CAP;               // CTA-uniform
  // body(k, l, set) for every entry of this chunk that holds its leaf's ticket (the highest k of its duplicates)
  auto for_each_winner = [&](auto&& body) {
    if (listed) {
      for (int i = tid; i < nmatch; i += K2C_THREADS) {
        const int k = m_k[i], lw = m_l[i], l = lw & 0x7fffffff;
        if (win[l] == k) body(k, l, lw >= 0);
      }
    } else {
      for (int k = tid; k < count; k += K2C_THREADS) {
        bool set;
        const int64_t p = position(k, set);
        if (!(p >= lo && p < lo + n && p < N)) continue;
        const int l = (int)(p - lo);
        if (win[l] == k) body(k, l, set);
      }
    }
  };
  // ---- few updated leaves (the usual case: 640 indices over 256 chunks): instead of recomputing the chunk's 4095
  //      inner nodes, each updated path is climbed on its own -- 12 adds -- from the siblings along it.  The sibling
  //      leaf is in shared memory already; the inner siblings are fetched from the tree here, one round trip for
  //      all paths and levels at once (thread = (path, level)), into their places in the chunk heap.  A sibling that
  //      lies on ANOTHER updated path is overwritten by that path's climb before it is read (levels are separated
  //      by a warp barrier).  The tree's invariant (node == fl32(left + right)) makes the fetched values exactly
  //      what the full recomputation would produce: the same tree, bit for bit.
  bool sparse = false;
  if (sparse_max > 0) {
    for_each_winner([&](int, int l, bool) {
      const int slot = atomicAdd(&s_nwin, 1);
      if (slot < K2C_SPARSE_MAX) s_list[slot] = l;
    });
    __syncthreads();
    const int nwin = s_nwin;
    sparse = nwin <= sparse_max;                             // CTA-uniform
    if (sparse && nwin > 0) {
      for (int t = tid; t < nwin * 16; t += K2C_THREADS) {
        const int j = t & 15;                                // level of the sibling: 1 .. clog-1 (level clog = leaves)
        if (j < 1 || j >= clog) continue;
        const int l = s_list[t >> 4];
        const int sib = ((n + l) >> (clog - j)) ^ 1;
        heap[sib] = __ldcg(tree + (((int64_t)1 << (top_levels + j)) + ((int64_t)c << j) + (sib - (1 << j))));
      }
    }
  }
  if (early) A0_PDL_PROLOGUE();                              // from here on the values (losses, max_p) are read
  const float maxp_in = __ldcg(max_p);
  if (c == 0) {                                              // CTA 0 also: running max of the losses, report
    float mx = 0.0f;
    for (int k = tid; k < count; k += K2C_THREADS) {
      bool set;
      const int64_t p = position(k, set);
      if (rep.idx) { rep.idx[k] = p; rep.loss[k] = vals[k]; }
      if (mode == 0 && p >= 0 && p < N && a0_loss_ok(vals[k])) mx = fmaxf(mx, vals[k]);
    }
    if (mode == 0) {
      mx = a0_warp_max(mx);
      if ((tid & 31) == 0) a0_atomic_max_pos(max_p, mx);    // max_p = max(max_p, max loss), replay.py:59
    }
  }
  __syncthreads();
  K2C_TX(1);
  // ---- pass 2: the winners overlay their leaves ----------------------------------------------------------
  for_each_winner([&](int k, int l, bool set) {
    float v;
    if (mode == 0) {
      if (!(heap[n + l] > 0.0f) || !a0_loss_ok(vals[k])) return;     // evicted since it was sampled / NaN loss
      v = a0_priority(vals[k], eps, alpha);
    } else if (mode == 1) {
      v = set ? (alpha == 0.5f ? sqrtf(maxp_in) : powf(maxp_in, alpha)) : 0.0f;
    } else {
      v = vals[k];
    }
    heap[n + l] = v;
    __stcg(tree + P + lo + l, v);
    s_dirty = 1;
  });
  __syncthreads();
  K2C_TX(2);
  if (s_dirty && sparse) {
    // every listed path (its leaf rewritten or not: an unchanged path recomputes the values it already holds),
    // one lane each, level by level; two lanes that share an ancestor write it the same value
    if (tid < 32) {
      const int nwin = s_nwin;
      const int l = tid < nwin ? s_list[tid] : -1;
      for (int j = clog - 1; j >= 0; --j) {
        if (l >= 0) {
          const int h = (n + l) >> (clog - j);
          const float v = __fadd_rn(heap[2 * h], heap[2 * h + 1]);
          heap[h] = v;
          __stcg(tree + (((int64_t)1 << (top_levels + j)) + ((int64_t)c << j) + (h - (1 << j))), v);
        }
        __syncwarp();
      }
    }
    K2C_TX(3);
  } else if (s_dirty) {
    a0_heap_reduce<K2C_THREADS>(heap, clog);
    K2C_TX(3);
    // ---- pass 3: the nodes on the updated paths (chunk-local node h at local level j) ------------------
    for_each_winner([&](int, int l, bool) {
      for (int j = clog - 1; j >= 0; --j) {
        const int h = (n + l) >> (clog - j);
        const int64_t g = ((int64_t)1 << (top_levels + j)) + ((int64_t)c << j) + (h - (1 << j));
        __stcg(tree + g, heap[h]);
      }
    });
  }
  K2C_TX(4);
  if (top_levels == 0) return;                               // a single chunk: its root is the tree's root
  // ---- the last CTA to finish recomputes the levels above the chunk roots --------------------------------
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  K2C_TX(5);
  __threadfence();
  const int nt = 1 << top_levels;                            // == gridDim.x chunk roots, <= K2C_MAX_CHUNKS rounded up
  for (int i = tid; i < nt; i += K2C_THREADS) heap[nt + i] = __ldcg(tree + nt + i);
  __syncthreads();
  K2C_TX(6);
  a0_dense_top<K2C_THREADS>(heap, top_levels, tree);
  if (tid == 0) *ticket = 0u;
#ifdef A0_TRACE
  _tx[7] = (unsigned long long)_c0;
#endif
  if (tid == 0) A0_TEND(5);
}

// ------------------------------------------------------------------------------------------------
// K2b in two halves, for the end of a training step (a0_pt_update_plan + a0_pt_update_apply).
// Everything the write-back needs but the losses is known once the draw has run: the positions, the
// duplicate winners, the paths and the values of the off-path siblings (nothing else writes the tree
// during a step).  a0_k2b_plan works that out in one CTA off the critical path; a0_k2b_apply runs under
// the step's last K4, reads the plan before griddepcontrol.wait and after it only reads the losses, forms
// the leaves and climbs.  The climb is short arithmetic; in one CTA it is bound by issuing the ~5 800
// scattered node stores of 640 paths on 1 M leaves from one SM (device timeline: 5 100 cycles).  So each of
// K2Q_APPLY_CTAS CTAs runs the whole apply and stores only its share of the nodes (slots d with
// d % K2Q_APPLY_CTAS == cta, and a slice of the dense top): the CTAs need nothing from each other, so there
// is no fence and no grid ticket.
//
// The tree splits at level t = min(D, 12): the 2^t level-t nodes are the inputs of a dense top (as in
// a0_k2b_chunks, two block barriers), the s = D - t levels below are climbed path by path.  Slot d holds
// the d-th distinct valid leaf in ascending order.  Paths d-1 and d of one level-t subtree meet at height
// lca = bit length of (p[d-1] ^ p[d]); slot d owns its path up to height top = lca - 1 and hands that value
// to the slot r that owns the left child there (the last slot before d whose own path joins above that
// height) -- r's right neighbour at that level is on a path, every other neighbour is an off-path sibling
// the plan has read.  The first slot of a subtree owns its path up to level t.  Hand-overs inside a warp
// need a warp barrier; the plan marks the heights where one crosses warps (xmask), and only those take a
// block barrier.  Every node is fl32(left + right) of its children: the tree a0_pt_update writes, bit for bit.
// ------------------------------------------------------------------------------------------------
constexpr int K2Q_THREADS = A0_K2B_PLAN_MAX;                  // indices (and so distinct leaves) of one planned update
constexpr int K2Q_TOP = 12;                                   // dense top from up to 4096 level-t nodes
constexpr int K2Q_SMAX = 16;                                  // levels climbed below it: trees of up to 2^28 leaves
struct A0K2bPlan {
  int32_t nd, s, xmask, pad_[13];
  int32_t pos[K2Q_THREADS];                                  // distinct valid leaves, ascending
  int32_t k[K2Q_THREADS];                                    // each one's winning index (the highest k of its duplicates)
  float old[K2Q_THREADS];                                    // the leaf before the update (0: evicted, stays)
  int32_t top[K2Q_THREADS];                                  // height up to which the slot owns its path
  int32_t recv[K2Q_THREADS];                                 // slot that receives the value at `top` (top < s)
  int32_t rmask[K2Q_THREADS];                                // heights at which the slot receives its right child
  float sib[K2Q_SMAX][K2Q_THREADS];                          // off-path sibling at heights 0 .. top-1
};
static_assert(sizeof(A0K2bPlan) == A0_K2B_PLAN_BYTES, "A0_K2B_PLAN_BYTES");
constexpr int K2Q_ROOT = 1 << 30;                            // lca of a subtree's first slot
constexpr int K2Q_APPLY_CTAS = 8;                            // power of two

__global__ void __launch_bounds__(K2Q_THREADS)
a0_k2b_plan(const float* __restrict__ tree, int64_t P, int32_t D, int64_t N, const int64_t* __restrict__ idx, int32_t count,
            A0K2bPlan* __restrict__ plan) {
  __shared__ unsigned long long s_key[K2Q_THREADS];
  __shared__ int s_pos[K2Q_THREADS];
  __shared__ int s_lca[K2Q_THREADS];
  __shared__ unsigned s_rmask[K2Q_THREADS];
  __shared__ int s_warp[32];
  __shared__ unsigned s_xmask;
  A0_T0();
  A0_PDL_PROLOGUE();
  A0_TMID();
  const int tid = threadIdx.x;
  const int s = D - (D < K2Q_TOP ? D : K2Q_TOP);
  unsigned long long key = ~0ull;                            // (leaf << 10 | k); invalid positions sort last
  if (tid < count) {
    const int64_t p = idx[tid];
    if (p >= 0 && p < N) key = ((unsigned long long)p << 10) | (unsigned)tid;
  }
  s_key[tid] = key;
  s_rmask[tid] = 0u;
  if (tid == 0) s_xmask = 0u;
  __syncthreads();
  a0_ku_bitonic(s_key, K2Q_THREADS);
  A0_TX(0);
  key = s_key[tid];
  const unsigned long long nxt = tid + 1 < K2Q_THREADS ? s_key[tid + 1] : ~0ull;
  const bool win = key != ~0ull && (nxt == ~0ull || (nxt >> 10) != (key >> 10));     // last of its run: highest k
  int nd;
  const int d = a0_ku_scan(win ? 1 : 0, s_warp, &nd);
  const int p = (int)(key >> 10);
  if (win) s_pos[d] = p;
  __syncthreads();
  int lca = K2Q_ROOT;
  if (win && d > 0) {
    const int q = s_pos[d - 1];
    if ((q >> s) == (p >> s)) lca = 32 - __clz(q ^ p);
  }
  if (win) s_lca[d] = lca;
  __syncthreads();
  A0_TX(1);
  if (win) {
    const int top = lca == K2Q_ROOT ? s : lca - 1;
    if (lca != K2Q_ROOT) {
      int r = d - 1;
      while (s_lca[r] <= top) --r;                           // stops at the subtree's first slot at the latest
      atomicOr(&s_rmask[r], 1u << top);
      if ((r >> 5) != (d >> 5)) atomicOr(&s_xmask, 1u << top);
      plan->recv[d] = r;
    }
    const int64_t leaf = P + p;
    for (int h = 0; h < top; ++h) plan->sib[h][d] = __ldcg(tree + ((leaf >> h) ^ 1));
    plan->pos[d] = p;
    plan->k[d] = (int)(key & 1023u);
    plan->old[d] = __ldcg(tree + leaf);
    plan->top[d] = top;
  }
  __syncthreads();
  if (win) plan->rmask[d] = (int)s_rmask[d];
  if (tid == 0) { plan->nd = nd; plan->s = s; plan->xmask = (int)s_xmask; }
  A0_TX(2);
  if (tid == 0) A0_TEND(7);
}

__global__ void __launch_bounds__(K2Q_THREADS)
a0_k2b_apply(float* __restrict__ tree, int64_t P, int32_t D, int64_t N, const int64_t* __restrict__ idx,
             const float* __restrict__ vals, int32_t count, float alpha, float eps, float* __restrict__ max_p,
             const A0K2bPlan* __restrict__ plan, const A0Report rep) {
  extern __shared__ __align__(16) float a0_k2q_smem[];
  A0_T0();
#ifdef A0_TRACE
  const long long _c0 = clock64();
#endif
  const int tid = threadIdx.x, lane = tid & 31, cta = blockIdx.x;
  const bool mine = (tid & (K2Q_APPLY_CTAS - 1)) == cta;      // this CTA stores slot tid's nodes
  const int t = D < K2Q_TOP ? D : K2Q_TOP;
  const int n = 1 << t;
  float* heap = a0_k2q_smem;                                 // heap[i] = node i of the top, level t in [n, 2n)
  float* xch = a0_k2q_smem + (2 << K2Q_TOP);                // xch[h * K2Q_THREADS + r]: r's right child at height h
  // ---- before the wait: the plan, the positions and the level-t nodes (written by launches older than the last K4)
  const int nd = __ldcg(&plan->nd), s = __ldcg(&plan->s);
  const unsigned xmask = (unsigned)__ldcg(&plan->xmask);
  for (int i = tid; i < n; i += K2Q_THREADS) heap[n + i] = __ldcg(tree + n + i);
  __syncthreads();                                           // the heap is final before the climb overlays its paths
  const bool live = tid < nd;
  int p = 0, k = 0, top = -1, recv = 0;
  unsigned rmask = 0u;
  float old = 0.0f, sib[K2Q_SMAX];
  if (live) {
    p = __ldcg(&plan->pos[tid]); k = __ldcg(&plan->k[tid]); old = __ldcg(&plan->old[tid]);
    top = __ldcg(&plan->top[tid]); recv = __ldcg(&plan->recv[tid]); rmask = (unsigned)__ldcg(&plan->rmask[tid]);
  }
#pragma unroll
  for (int h = 0; h < K2Q_SMAX; ++h) sib[h] = h < top ? __ldcg(&plan->sib[h][tid]) : 0.0f;
  const int64_t pos_k = tid < count ? idx[tid] : -1;
  A0_TX(0);
  A0_PDL_PROLOGUE();                                         // the last K4 is complete: the losses
  A0_TMID();
  A0_TX(1);
  const float loss_k = tid < count ? __ldcg(vals + tid) : 0.0f;
  const float loss_w = live ? __ldcg(vals + k) : 0.0f;
  if (cta == 0 && rep.idx && tid < count) { rep.idx[tid] = pos_k; rep.loss[tid] = loss_k; }
  const int64_t leaf = P + p;
  float v = old;
  if (live && old > 0.0f && a0_loss_ok(loss_w)) {            // evicted since it was sampled / NaN loss: the leaf stays
    v = a0_priority(loss_w, eps, alpha);
    if (mine) __stcg(tree + leaf, v);
  }
  A0_TX(2);
#pragma unroll
  for (int h = 0; h < K2Q_SMAX; ++h) {
    if (h >= s) break;
    if (live && top == h && h < s) xch[h * K2Q_THREADS + recv] = v;
    if ((xmask >> h) & 1u) __syncthreads(); else __syncwarp();
    if (live && h < top) {
      const float o = ((rmask >> h) & 1u) ? xch[h * K2Q_THREADS + tid] : sib[h];
      v = ((p >> h) & 1) ? __fadd_rn(o, v) : __fadd_rn(v, o);
      if (mine) __stcg(tree + (leaf >> (h + 1)), v);
    }
  }
  if (live && top == s) heap[n + (p >> s)] = v;
  __syncthreads();
  A0_TX(3);
  a0_heap_reduce<K2Q_THREADS>(heap, t);
  const int share = (n + K2Q_APPLY_CTAS - 1) / K2Q_APPLY_CTAS;
  for (int i = cta * share + tid; i < n && i < (cta + 1) * share; i += K2Q_THREADS)
    if (i >= 1) tree[i] = heap[i];
  if (cta == 0) {                                            // off the climb's path: nothing here waits for max_p
    float mx = pos_k >= 0 && pos_k < N && a0_loss_ok(loss_k) ? loss_k : 0.0f;
    mx = a0_warp_max(mx);
    if (lane == 0) a0_atomic_max_pos(max_p, mx);            // max_p = max(max_p, max loss), replay.py:59
  }
  A0_TX(4);
#ifdef A0_TRACE
  _tx[7] = (unsigned long long)_c0;
#endif
  if (tid == 0) A0_TEND(8);
}

static int g_k2b_chunk_max = -1;   // largest index list the one-launch chunk schedule takes (A0_K2B_CHUNK_MAX)
static int a0_option_k2b_chunk_max() {
  if (g_k2b_chunk_max < 0) {
    const char* e = getenv("A0_K2B_CHUNK_MAX");
    g_k2b_chunk_max = e ? atoi(e) : K2C_MAX_COUNT_DEFAULT;
    if (g_k2b_chunk_max < 0) g_k2b_chunk_max = K2C_MAX_COUNT_DEFAULT;
  }
  return g_k2b_chunk_max;
}
static int g_k2b_sparse = -1;      // updated leaves per chunk up to which a0_k2b_chunks climbs path by path (0: always the full chunk)
static int a0_option_k2b_sparse() {
  if (g_k2b_sparse < 0) {
    const char* e = getenv("A0_K2B_SPARSE");
    g_k2b_sparse = e ? atoi(e) : K2C_SPARSE_MAX;
    if (g_k2b_sparse < 0 || g_k2b_sparse > K2C_SPARSE_MAX) g_k2b_sparse = K2C_SPARSE_MAX;
  }
  return g_k2b_sparse;
}
void a0_set_k2b_sparse(int v) { g_k2b_sparse = v < 0 ? 0 : (v > K2C_SPARSE_MAX ? K2C_SPARSE_MAX : v); }
static int g_k2b_chunks = -1;
static bool a0_option_k2b_chunks() {
  if (g_k2b_chunks < 0) {
    const char* e = getenv("A0_K2B_CHUNKS");
    g_k2b_chunks = e ? (atoi(e) != 0) : 1;
  }
  return g_k2b_chunks != 0;
}
void a0_set_k2b_chunks(int on) { g_k2b_chunks = on != 0; }

static int a0_launch_paths(a0_replay_t* h, const int64_t* idx64, const int32_t* idx32, const float* vals,
                           int32_t count, int32_t mode, float alpha, float eps, cudaStream_t stream,
                           const A0Report& rep, int32_t* dirty = nullptr, int32_t chunk_log = 0) {
  int ctas = (count + K2P_THREADS - 1) / K2P_THREADS;
  ctas = ctas < 1 ? 1 : (ctas > K2P_CLUSTER ? K2P_CLUSTER : ctas);
  if (ctas > 1 && (ctas & (ctas - 1))) {            // cluster sizes: powers of two
    int p2 = 1;
    while (p2 < ctas) p2 <<= 1;
    ctas = p2;
  }
  if (a0_option_k2b_levels() == 4)
    A0_LAUNCH(a0_k2b_paths<4>, (unsigned)ctas, K2P_THREADS, 0, stream, (unsigned)ctas, A0_PDL_K2, h->tree, h->P, h->D, h->N, idx64, idx32,
              vals, count, mode, alpha, eps, h->max_p, h->winner, dirty, chunk_log, rep);
  else
    A0_LAUNCH(a0_k2b_paths<3>, (unsigned)ctas, K2P_THREADS, 0, stream, (unsigned)ctas, A0_PDL_K2, h->tree, h->P, h->D, h->N, idx64, idx32,
              vals, count, mode, alpha, eps, h->max_p, h->winner, dirty, chunk_log, rep);
  return A0_OK;
}

static int a0_launch_update(a0_replay_t* h, const int64_t* idx64, const int32_t* idx32, const float* vals,
                            int32_t count, int32_t mode, float alpha, float eps, a0_stream_t stream_,
                            const A0Report rep = {nullptr, nullptr}, bool early = false) {
  if (count == 0) return A0_OK;
  A0DeviceGuard guard(h->device);
  cudaStream_t stream = (cudaStream_t)stream_;
  const int chunk_log = h->D < K2R_MAXLOG ? h->D : K2R_MAXLOG;
  const int64_t chunks = h->P >> chunk_log;
  // Three schedules, same tree.  Few indices: one cluster climbs the paths.  Many indices relative to
  // the tree (10 240 updates on a 1 M-leaf tree touch nearly every 4096-leaf chunk): the cluster only
  // writes the leaves (claim / write / release, two cluster barriers) and the chunk rebuild runs on
  // all SMs -- measured 29 -> see DESIGN.md.  More than one cluster can hold: one CTA writes.
  if (count <= a0_option_k2b_chunk_max() && chunks <= K2C_MAX_CHUNKS && a0_option_k2b_chunks()) {
    // one CTA per 4096-leaf chunk in a single launch.  Measured: 640 indices on 1 M leaves 9.5 -> 8 us against
    // the cluster climb.  With three scans of the index list per CTA the leaf write + rebuild pair was faster at
    // 10 240 indices (16.9 vs 21.5 us), so this schedule stopped at 2048; with ONE scan and a match list it takes
    // 11.9 us there and is the default up to 16 384 indices (A0_K2B_CHUNK_MAX)
    static thread_local bool attr[64] = {false};
    if (h->device < 64 && !attr[h->device]) {
      A0_CUDA(cudaFuncSetAttribute(a0_k2b_chunks, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K2C_SMEM));
      attr[h->device] = true;
    }
    A0_LAUNCH(a0_k2b_chunks, (unsigned)chunks, K2C_THREADS, K2C_SMEM, stream, 1, early ? A0_PDL_FORCE : A0_PDL_K2, h->tree, h->P, h->D, h->N,
              idx64, idx32, vals, count, mode, alpha, eps, h->max_p, h->counter + A0_MAX_BATCHES, rep, (int32_t)(early ? 1 : 0),
              (int32_t)a0_option_k2b_sparse());
    return A0_OK;
  }
  const bool hybrid = count >= a0_option_k2b_bulk_min() && (int64_t)count >= 4 * chunks;
  if (count <= K2S_THREADS && !hybrid && h->D - K2P_TOP <= K2S_MAX_SPARSE && a0_option_k2b_small()) {
    static thread_local bool attr[64] = {false};
    int rc = a0_k2s_smem_attr(h, a0_k2b_small, attr);
    if (rc) return rc;
    A0_LAUNCH(a0_k2b_small, 1, K2S_THREADS, K2S_SMEM, stream, 1, A0_PDL_K2, h->tree, h->P, h->D, h->N, idx64, idx32, vals, count, mode,
              alpha, eps, h->max_p, rep);
    return A0_OK;
  }
  if (count <= K2P_MAX && !hybrid) return a0_launch_paths(h, idx64, idx32, vals, count, mode, alpha, eps, stream, rep);
  if (count <= K2P_MAX) {
    int rc = a0_launch_paths(h, idx64, idx32, vals, count, mode, alpha, eps, stream, rep, h->dirty, chunk_log);
    if (rc) return rc;
  } else {
    A0_LAUNCH(a0_k2b_write, 1, K2B_THREADS, 0, stream, 1, A0_PDL_K2, h->tree, h->P, chunk_log, h->N, idx64, idx32, vals, count, mode, alpha,
              eps, h->max_p, h->winner, h->dirty, rep);
  }
  A0_LAUNCH(a0_k2b_rebuild, (unsigned)chunks, K2R_THREADS, 0, stream, 1, A0_PDL_K2, h->tree, h->D, chunk_log, h->dirty,
            h->counter + A0_MAX_BATCHES);
  return A0_OK;
}

extern "C" int a0_pt_update(a0_replay_t* h, const int64_t* idx, const float* loss, int32_t count, float alpha,
                            float eps, a0_stream_t stream) {
  A0_REQUIRE(h != nullptr && count >= 0, "a0_pt_update: bad handle or count");
  A0_REQUIRE(count == 0 || (idx && loss), "a0_pt_update: NULL argument");
  { int frc = a0_check_fault(h, "a0_pt_update"); if (frc) return frc; }
  return a0_launch_update(h, idx, nullptr, loss, count, 0, alpha, eps, stream);
}
extern "C" int a0_pt_update_overlapped(a0_replay_t* h, const int64_t* idx, const float* loss, int32_t count, float alpha,
                                       float eps, int64_t* idx_report, float* loss_report, a0_stream_t stream) {
  A0_REQUIRE(h != nullptr && count >= 0, "a0_pt_update_overlapped: bad handle or count");
  A0_REQUIRE(count == 0 || (idx && loss), "a0_pt_update_overlapped: NULL argument");
  A0_REQUIRE((idx_report == nullptr) == (loss_report == nullptr), "a0_pt_update_overlapped: give both report buffers or none");
  { int frc = a0_check_fault(h, "a0_pt_update_overlapped"); if (frc) return frc; }
  const A0Report rep = {idx_report, loss_report};
  return a0_launch_update(h, idx, nullptr, loss, count, 0, alpha, eps, stream, rep, true);
}
// Device-visible alias of page-locked host memory (mapped under unified addressing: what cudaHostAlloc
// and torch's pin_memory give), for the report buffers of a0_pt_update_report.  Not a stream
// operation; call it once per buffer, outside any graph capture.
extern "C" int a0_host_map(const void* host_ptr, void** dev_ptr_out) {
  A0_REQUIRE(host_ptr && dev_ptr_out, "a0_host_map: NULL argument");
  cudaPointerAttributes at;
  A0_CUDA(cudaPointerGetAttributes(&at, host_ptr));
  A0_REQUIRE(at.type != cudaMemoryTypeUnregistered && at.devicePointer != nullptr,
             "a0_host_map: pageable host memory; the buffer must be page-locked (cudaHostAlloc / pin_memory)");
  *dev_ptr_out = at.devicePointer;
  return A0_OK;
}

extern "C" int a0_pt_update_report(a0_replay_t* h, const int64_t* idx, const float* loss, int32_t count, float alpha,
                                   float eps, int64_t* idx_report, float* loss_report, a0_stream_t stream) {
  A0_REQUIRE(h != nullptr && count >= 0, "a0_pt_update_report: bad handle or count");
  A0_REQUIRE(count == 0 || (idx && loss), "a0_pt_update_report: NULL argument");
  A0_REQUIRE(idx_report && loss_report, "a0_pt_update_report: NULL report buffer (a0_pt_update reports nothing)");
  const A0Report rep = {idx_report, loss_report};
  { int frc = a0_check_fault(h, "a0_pt_update_report"); if (frc) return frc; }
  return a0_launch_update(h, idx, nullptr, loss, count, 0, alpha, eps, stream, rep);
}
extern "C" int a0_pt_mark(a0_replay_t* h, const int32_t* pos, int32_t count, float alpha, a0_stream_t stream) {
  A0_REQUIRE(h != nullptr && count >= 0, "a0_pt_mark: bad handle or count");
  A0_REQUIRE(count == 0 || pos, "a0_pt_mark: NULL argument");
  return a0_launch_update(h, nullptr, pos, nullptr, count, 1, alpha, 0.0f, stream);
}
extern "C" int a0_pt_set(a0_replay_t* h, const int64_t* idx, const float* value, int32_t count, a0_stream_t stream) {
  A0_REQUIRE(h != nullptr && count >= 0, "a0_pt_set: bad handle or count");
  A0_REQUIRE(count == 0 || (idx && value), "a0_pt_set: NULL argument");
  return a0_launch_update(h, idx, nullptr, value, count, 2, 1.0f, 0.0f, stream);
}

// The planned write-back (see a0_k2b_plan): idx must not change, and nothing may write the tree, between the two calls.
extern "C" int a0_pt_update_plan(a0_replay_t* h, const int64_t* idx, int32_t count, void* plan, a0_stream_t stream) {
  A0_REQUIRE(h != nullptr && count >= 0 && count <= A0_K2B_PLAN_MAX, "a0_pt_update_plan: bad handle or count (at most %d)",
             A0_K2B_PLAN_MAX);
  A0_REQUIRE(idx && plan, "a0_pt_update_plan: NULL argument");
  A0_REQUIRE(h->D >= 1 && h->D <= K2Q_TOP + K2Q_SMAX, "a0_pt_update_plan: tree depth %d outside 1..%d", (int)h->D,
             K2Q_TOP + K2Q_SMAX);
  { int frc = a0_check_fault(h, "a0_pt_update_plan"); if (frc) return frc; }
  A0DeviceGuard guard(h->device);
  A0_LAUNCH(a0_k2b_plan, 1, K2Q_THREADS, 0, (cudaStream_t)stream, 1, A0_PDL_K2, (const float*)h->tree, h->P, h->D, h->N, idx,
            count, (A0K2bPlan*)plan);
  return A0_OK;
}
extern "C" int a0_pt_update_apply(a0_replay_t* h, const int64_t* idx, const float* loss, int32_t count, float alpha, float eps,
                                  const void* plan, int64_t* idx_report, float* loss_report, a0_stream_t stream) {
  A0_REQUIRE(h != nullptr && count >= 0 && count <= A0_K2B_PLAN_MAX, "a0_pt_update_apply: bad handle or count (at most %d)",
             A0_K2B_PLAN_MAX);
  A0_REQUIRE(idx && loss && plan, "a0_pt_update_apply: NULL argument");
  A0_REQUIRE((idx_report == nullptr) == (loss_report == nullptr), "a0_pt_update_apply: give both report buffers or none");
  A0_REQUIRE(h->D >= 1 && h->D <= K2Q_TOP + K2Q_SMAX, "a0_pt_update_apply: tree depth %d outside 1..%d", (int)h->D,
             K2Q_TOP + K2Q_SMAX);
  { int frc = a0_check_fault(h, "a0_pt_update_apply"); if (frc) return frc; }
  A0DeviceGuard guard(h->device);
  const int s = h->D - (h->D < K2Q_TOP ? h->D : K2Q_TOP);
  const size_t smem = ((size_t)(2 << K2Q_TOP) + (size_t)s * K2Q_THREADS) * sizeof(float);
  static thread_local bool attr[64] = {false};
  if (h->device < 64 && !attr[h->device]) {
    A0_CUDA(cudaFuncSetAttribute(a0_k2b_apply, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)(((size_t)(2 << K2Q_TOP) + (size_t)K2Q_SMAX * K2Q_THREADS) * sizeof(float))));
    attr[h->device] = true;
  }
  A0_LAUNCH(a0_k2b_apply, K2Q_APPLY_CTAS, K2Q_THREADS, smem, (cudaStream_t)stream, 1, A0_PDL_FORCE, h->tree, h->P, h->D, h->N, idx, loss, count,
            alpha, eps, h->max_p, (const A0K2bPlan*)plan, A0Report{idx_report, loss_report});
  return A0_OK;
}
