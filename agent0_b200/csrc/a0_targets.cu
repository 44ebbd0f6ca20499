// K4: fused target + loss + IS weighting + new-priority kernels for the six deepq learners.
//
// Each kernel consumes the *network outputs* the reference's train_step consumes and produces, in
// one launch: the per-sample loss (what the reference returns as q_loss), the gradient of
// (loss * weight).sum() with respect to the online-network output (agent0/deepq/agent.py:152-155;
// the loss is SUM-reduced, SURVEY Q7), and the new priority (loss+eps)^alpha with a device-side
// running max (agent0/deepq/replay.py:55-59).  The reference runs 10-30 eager ATen kernels per rule
// and, for the quantile family, materialises [B,N,N] tensors several times (agent.py:110-114);
// here the pair loop stays in registers.  Inputs are <= 2.4 KB per transition: these kernels are
// launch/ALU-bound, not HBM-bound (SURVEY section 8d).
#include <stdlib.h>

#include "a0_common.cuh"
#ifdef A0_TRACE
A0_TRACE_SETTER(a0_trace_set_targets)
#endif

struct A0Common {
  int32_t B, A;
  const int64_t* action;
  const float* reward;
  const float* done;
  const float* weight;
  float gamma_n, alpha, eps;
  float* loss;
  float* prio;
  float* max_p;
};

static inline A0Common a0_unpack(const a0_loss_common_t* c) {
  A0Common k;
  k.B = c->B; k.A = c->A; k.action = c->action; k.reward = c->reward; k.done = c->done;
  k.weight = c->weight; k.gamma_n = c->gamma_n; k.alpha = c->alpha; k.eps = c->eps;
  k.loss = c->loss; k.prio = c->prio; k.max_p = c->max_p;
  return k;
}

static int a0_check_common(const a0_loss_common_t* c, const char* who) {
  A0_REQUIRE(c != nullptr, "%s: common block is NULL", who);
  A0_REQUIRE(c->B >= 0, "%s: negative batch", who);
  A0_REQUIRE(c->A >= 1 && c->A <= A0_MAX_ACTIONS, "%s: action_dim %d outside [1,%d]", who, c->A, A0_MAX_ACTIONS);
  A0_REQUIRE(c->action && c->reward && c->done && c->weight && c->loss, "%s: NULL tensor in common block", who);
  return A0_OK;
}

__device__ __forceinline__ void a0_emit(const A0Common& c, int b, float loss) {
  c.loss[b] = loss;
  if (c.prio) c.prio[b] = a0_priority(loss, c.eps, c.alpha);
  if (c.max_p) a0_atomic_max_pos(c.max_p, loss);
}

// T = r + (gamma_n * (1 - d)) * boot, each op rounded (agent.py:181-186)
__device__ __forceinline__ float a0_td_target(float r, float d, float gamma_n, float boot) {
  return __fadd_rn(r, __fmul_rn(__fmul_rn(gamma_n, __fsub_rn(1.0f, d)), boot));
}

// ------------------------------------------------------------------------------------------------
// DQN (agent.py:173-190) and M-DQN (agent.py:194-215): one warp per sample, lane = action.
// ------------------------------------------------------------------------------------------------
constexpr int K4S_WARPS = 4;

// Every global load of the sample is issued up front (the taken action's Q-value comes from a shuffle of
// the row, not from a second, action-dependent load), and M-DQN's independent reductions are advanced
// together -- the two row maxima, then the three sums: 15 dependent shuffle steps instead of 30.  One
// warp per sample: as for C51, the launch lasts as long as one warp's dependent chain.
__global__ void __launch_bounds__(K4S_WARPS * 32)
a0_k4_dqn(const A0Common c, const float* __restrict__ q, const float* __restrict__ qt_next,
          const float* __restrict__ qsel, const float* __restrict__ qt_cur, int32_t munchausen, float tau,
          float lo, float* __restrict__ grad) {
  A0_PDL_PROLOGUE();
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * K4S_WARPS + (threadIdx.x >> 5);
  if (b >= c.B) return;
  const int A = c.A;
  const bool valid = lane < A;
  const size_t off = (size_t)b * A + lane;
  const float tn = valid ? qt_next[off] : 0.0f;
  const float qv = valid ? q[off] : 0.0f;
  const float sel_in = (!munchausen && qsel && valid) ? qsel[off] : 0.0f;
  const float tc = (munchausen && valid) ? qt_cur[off] : 0.0f;
  const int a = (int)c.action[b];
  const float r = c.reward[b], d = c.done[b], w = c.weight[b];
  float boot, bonus = 0.0f;
  if (!munchausen) {
    const float sel = valid ? (qsel ? sel_in : tn) : -INFINITY;
    const int a_star = a0_warp_argmax(sel, lane);
    boot = __shfl_sync(0xffffffffu, tn, a_star);
  } else {
    // log_softmax_stable (agent.py:116-119) of both target rows: (l - max) - tau * logsumexp((l - max)/tau)
    float mxn = valid ? tn : -INFINITY, mxc = valid ? tc : -INFINITY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float x_ = __shfl_xor_sync(0xffffffffu, mxn, o), y_ = __shfl_xor_sync(0xffffffffu, mxc, o);
      mxn = fmaxf(mxn, x_);
      mxc = fmaxf(mxc, y_);
    }
    const float zn = tn - mxn, zc = tc - mxc;
    float sen = valid ? expf(__fdiv_rn(zn, tau)) : 0.0f;     // max over lanes of z/tau is 0
    float sec = valid ? expf(__fdiv_rn(zc, tau)) : 0.0f;
    const float e = valid ? expf(zn) : 0.0f;
    float es = e;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float x_ = __shfl_xor_sync(0xffffffffu, sen, o), y_ = __shfl_xor_sync(0xffffffffu, sec, o);
      const float z_ = __shfl_xor_sync(0xffffffffu, es, o);
      sen += x_;
      sec += y_;
      es += z_;
    }
    const float tlp = zn - tau * logf(sen);                  // tau * log pi(.|s')
    const float tlp_cur = zc - tau * logf(sec);
    const float p = __fdiv_rn(e, es);                        // softmax at temperature 1 (SURVEY Q11)
    boot = a0_warp_sum(valid ? p * (tn - tlp) : 0.0f);
    const float at_a = __shfl_sync(0xffffffffu, tlp_cur, a);
    bonus = __fmul_rn(tau, fminf(fmaxf(at_a, lo), 0.0f));
  }
  const float qa = __shfl_sync(0xffffffffu, qv, a);
  const float T = munchausen
      ? __fadd_rn(__fadd_rn(r, bonus), __fmul_rn(__fmul_rn(c.gamma_n, __fsub_rn(1.0f, d)), boot))
      : a0_td_target(r, d, c.gamma_n, boot);
  const float x = qa - T;
  if (valid) grad[off] = lane == a ? w * a0_clamp1(x) : 0.0f;
  if (lane == 0) a0_emit(c, b, a0_huber(x));
}

extern "C" int a0_loss_dqn(const a0_loss_common_t* c, const float* q, const float* qt_next, const float* qsel,
                           float* grad, a0_stream_t stream) {
  int rc = a0_check_common(c, "a0_loss_dqn");
  if (rc) return rc;
  A0_REQUIRE(q && qt_next && grad, "a0_loss_dqn: NULL tensor");
  if (c->B == 0) return A0_OK;
  A0_LAUNCH(a0_k4_dqn, (unsigned)((c->B + K4S_WARPS - 1) / K4S_WARPS), K4S_WARPS * 32, 0, (cudaStream_t)stream, 1, A0_PDL_K4,
            a0_unpack(c), q, qt_next, qsel, (const float*)nullptr, 0, 0.0f, 0.0f, grad);
  return A0_OK;
}

extern "C" int a0_loss_mdqn(const a0_loss_common_t* c, const float* q, const float* qt_next, const float* qt_cur,
                            float tau, float lo, float* grad, a0_stream_t stream) {
  int rc = a0_check_common(c, "a0_loss_mdqn");
  if (rc) return rc;
  A0_REQUIRE(q && qt_next && qt_cur && grad, "a0_loss_mdqn: NULL tensor");
  A0_REQUIRE(tau > 0.0f, "a0_loss_mdqn: tau must be positive");
  if (c->B == 0) return A0_OK;
  A0_LAUNCH(a0_k4_dqn, (unsigned)((c->B + K4S_WARPS - 1) / K4S_WARPS), K4S_WARPS * 32, 0, (cudaStream_t)stream, 1, A0_PDL_K4,
            a0_unpack(c), q, qt_next, (const float*)nullptr, qt_cur, 1, tau, lo, grad);
  return A0_OK;
}

// ------------------------------------------------------------------------------------------------
// C51 (agent.py:219-269): one warp per sample, lane l owns atoms l, l+32, ... (M <= 128).
// The projection replaces two index_add_ calls (atomicAdd scatter on CUDA, agent.py:258-264).
// b_j = (clamp(r + g z_j) - vmin)/delta is non-decreasing in j, so the sources that fall into one
// bin are consecutive atoms: a segmented warp scan over the lanes (keys = destination bin, five
// shuffle steps) sums every run, and the last lane of a run adds the run total to that bin in
// shared memory.  Four such phases (lo/up terms x two 32-atom chunks) in a fixed order give a
// result that does not depend on scheduling; the summation order inside a run is a tree instead
// of the CPU's left-to-right, which moves a bin by a few ulp (all terms are non-negative).
// ------------------------------------------------------------------------------------------------
constexpr int C51_WARPS = 4;
constexpr int C51_MAXR = 4;     // atoms per lane: M <= 128
constexpr int C51_FAST_WARPS = 4;  // samples per CTA of the short-chain kernel
constexpr int C51_SPEC_A = 6;   // speculative all-action row fetch up to this many actions

// Adds v (keyed by destination bin) into bins[]: runs of equal adjacent keys are reduced with
// shuffles first.  key < 0 marks a lane without a term.  NP independent (key, value) streams are
// scanned together -- their shuffles are issued back to back, so the five dependent steps cost one
// shuffle latency each instead of NP -- and then added stream by stream in a fixed order.
template <int NP>
__device__ __forceinline__ void a0_c51_scatter(float* bins, const int (&key)[NP], float (&v)[NP], int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    float vu[NP];
    int ku[NP];
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      vu[p] = __shfl_up_sync(0xffffffffu, v[p], d);
      ku[p] = __shfl_up_sync(0xffffffffu, key[p], d);
    }
#pragma unroll
    for (int p = 0; p < NP; ++p)
      if (lane >= d && ku[p] == key[p]) v[p] = __fadd_rn(v[p], vu[p]);
  }
  int kn[NP];
#pragma unroll
  for (int p = 0; p < NP; ++p) kn[p] = __shfl_down_sync(0xffffffffu, key[p], 1);
#pragma unroll
  for (int p = 0; p < NP; ++p) {
    if (key[p] >= 0 && (lane == 31 || kn[p] != key[p])) atomicAdd(bins + key[p], v[p]);   // one writer per bin when keys are sorted
    __syncwarp();
  }
}

__global__ void __launch_bounds__(C51_WARPS * 32)
a0_k4_c51(const A0Common c, const float* __restrict__ logits, const float* __restrict__ tgt_logits,
          const float* __restrict__ qsel, const float* __restrict__ atoms, int32_t M, float vmin, float vmax,
          float* __restrict__ grad, float* __restrict__ target_prob) {
  __shared__ float s_m[C51_WARPS][C51_MAXR * 32];      // projected distribution of this warp's sample
  A0_T0();
  A0_PDL_PROLOGUE();
  A0_TMID();
#ifdef A0_TRACE
  const long long _c0 = clock64();
#endif
  const int lane = threadIdx.x & 31;
  const int wid = threadIdx.x >> 5;
  const int b = blockIdx.x * C51_WARPS + wid;
  if (b >= c.B) return;
  const int A = c.A;
  const int R = (M + 31) / 32;
  // Every global load of this sample is issued up front.  With few actions and <= 64 atoms (the
  // Atari case: A = 4..6 after the minimal action set, M = 51) the rows of ALL actions are fetched
  // speculatively -- A*M*4 B <= 1.2 KB per network output -- so neither the taken action nor the
  // arg-max action adds a second dependent memory round trip to this latency-bound kernel.
  const bool spec = A <= C51_SPEC_A && R <= 2;
  float lo_all[C51_SPEC_A][2], tg_all[C51_SPEC_A][2];
  if (spec) {
#pragma unroll
    for (int a2 = 0; a2 < C51_SPEC_A; ++a2)
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const bool in = a2 < A && lane + 32 * k < M;
        const size_t off = ((size_t)b * A + a2) * M + lane + 32 * k;
        lo_all[a2][k] = in ? logits[off] : -INFINITY;
        tg_all[a2][k] = in ? tgt_logits[off] : -INFINITY;
      }
  }
  const int a = (int)c.action[b];
  const float r = c.reward[b], d = c.done[b], w = c.weight[b];
  const float qs = (qsel && lane < A) ? qsel[(size_t)b * A + lane] : -INFINITY;
  float z[C51_MAXR], l[C51_MAXR];
  const float* orow = logits + ((size_t)b * A + a) * M;
#pragma unroll
  for (int k = 0; k < C51_MAXR; ++k) {
    const bool in = k < R && lane + 32 * k < M;
    z[k] = in ? atoms[lane + 32 * k] : 0.0f;
    l[k] = -INFINITY;
    if (!spec) l[k] = in ? orow[lane + 32 * k] : -INFINITY;
    s_m[wid][lane + 32 * k] = 0.0f;
  }
  if (spec) {
#pragma unroll
    for (int a2 = 0; a2 < C51_SPEC_A; ++a2)
      if (a2 == a) { l[0] = lo_all[a2][0]; l[1] = lo_all[a2][1]; }
  }

  // ---- action selection + the reductions of both softmaxes ---------------------------------------
  // This kernel is one warp per sample and latency-bound: every warp reduction is five dependent
  // shuffle steps.  Independent reductions are therefore advanced together, one shuffle latency
  // per step for the pair: (arg-max of qsel | max of the online row), then (max of the selected
  // target row | sum-exp of the online row).
  float omx = -INFINITY;
#pragma unroll
  for (int k = 0; k < C51_MAXR; ++k) omx = fmaxf(omx, l[k]);
#ifdef A0_TRACE
  if (omx == 12345.678f) printf("x");     // forces the loads to have landed before the timestamp
#endif
  A0_TX(0);
  int a_star;
  if (qsel) {
    float v = qs;
    int vi = lane;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, v, o);
      const int oi = __shfl_xor_sync(0xffffffffu, vi, o);
      const float om = __shfl_xor_sync(0xffffffffu, omx, o);
      if (a0_argmax_before(ov, oi, v, vi)) { v = ov; vi = oi; }
      omx = fmaxf(omx, om);
    }
    a_star = vi;
  } else {
    omx = a0_warp_max(omx);
    // argmax_a sum_j softmax(tgt[b,a,:])_j * z_j (agent.py:226)
    float best = -INFINITY;
    a_star = 0;
    for (int a2 = 0; a2 < A; ++a2) {
      const float* row = tgt_logits + ((size_t)b * A + a2) * M;
      float v[C51_MAXR], mx = -INFINITY;
#pragma unroll
      for (int k = 0; k < C51_MAXR; ++k) {
        v[k] = (k < R && lane + 32 * k < M) ? row[lane + 32 * k] : -INFINITY;   // L1/L2 hit when spec
        mx = fmaxf(mx, v[k]);
      }
      mx = a0_warp_max(mx);
      float se = 0.0f;
#pragma unroll
      for (int k = 0; k < C51_MAXR; ++k) { v[k] = (k < R && lane + 32 * k < M) ? expf(v[k] - mx) : 0.0f; se += v[k]; }
      se = a0_warp_sum(se);
      float ev = 0.0f;
#pragma unroll
      for (int k = 0; k < C51_MAXR; ++k) ev += __fdiv_rn(v[k], se) * z[k];
      ev = a0_warp_sum(ev);
      if (a0_argmax_takes(ev, best)) { best = ev; a_star = a2; }
    }
  }

  A0_TX(1);
  // ---- softmax of the selected target row | sum-exp of the online row -----------------------------
  const float* trow = tgt_logits + ((size_t)b * A + a_star) * M;
  float p[C51_MAXR], mx = -INFINITY;
#pragma unroll
  for (int k = 0; k < C51_MAXR; ++k) p[k] = -INFINITY;
  if (spec) {
#pragma unroll
    for (int a2 = 0; a2 < C51_SPEC_A; ++a2)
      if (a2 == a_star) { p[0] = tg_all[a2][0]; p[1] = tg_all[a2][1]; }
  } else {
#pragma unroll
    for (int k = 0; k < C51_MAXR; ++k)
      if (k < R && lane + 32 * k < M) p[k] = trow[lane + 32 * k];
  }
#pragma unroll
  for (int k = 0; k < C51_MAXR; ++k) mx = fmaxf(mx, p[k]);
  float ose = 0.0f;
#pragma unroll
  for (int k = 0; k < C51_MAXR; ++k) ose += (k < R && lane + 32 * k < M) ? expf(l[k] - omx) : 0.0f;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const float os = __shfl_xor_sync(0xffffffffu, ose, o);
    mx = fmaxf(mx, om);
    ose += os;
  }
  float se = 0.0f;
#pragma unroll
  for (int k = 0; k < C51_MAXR; ++k) { p[k] = (k < R && lane + 32 * k < M) ? expf(p[k] - mx) : 0.0f; se += p[k]; }
  se = a0_warp_sum(se);

  A0_TX(2);
  // ---- projection (agent.py:230-264) ------------------------------------------------------------
  const float gm = __fmul_rn(c.gamma_n, __fsub_rn(1.0f, d));
  const float delta = (vmax - vmin) / (float)(M - 1);
  int lo[C51_MAXR], up[C51_MAXR];
  float wlo[C51_MAXR], wup[C51_MAXR];
#pragma unroll
  for (int k = 0; k < C51_MAXR; ++k) {
    lo[k] = up[k] = -1;
    wlo[k] = wup[k] = 0.0f;
    if (k < R && lane + 32 * k < M) {
      const float pj = __fdiv_rn(p[k], se);
      float tz = __fadd_rn(r, __fmul_rn(gm, z[k]));
      tz = fminf(fmaxf(tz, vmin), vmax);
      const float base = __fdiv_rn(__fsub_rn(tz, vmin), delta);
      int lo_ = (int)floorf(base), up_ = (int)ceilf(base);
      if (up_ > 0 && lo_ == up_) lo_ -= 1;
      if (lo_ < M - 1 && lo_ == up_) up_ += 1;
      // delta is rounded to fp32, so an atom clamped at vmax can get a base just above M-1 (M = 128, vmin = -10,
      // vmax = 25: 127.0000076) and up_ = M.  That upper term is dropped, as in a0_k4_c51_fast: bin M is past the
      // sample's row, and at M = 128 it is bin 0 of the next warp's sample.
      lo[k] = lo_; up[k] = up_ < M ? up_ : -1;
      wlo[k] = __fmul_rn(pj, __fsub_rn((float)up_, base));
      wup[k] = __fmul_rn(pj, __fsub_rn(base, (float)lo_));
    }
  }
  __syncwarp();
  A0_TX(3);
  if (R <= 2) {
    // M <= 64 (the 51-atom case): lower and upper terms of both atom chunks in one scan
    const int key4[4] = {lo[0], lo[1], up[0], up[1]};
    float val4[4] = {wlo[0], wlo[1], wup[0], wup[1]};
    a0_c51_scatter<4>(s_m[wid], key4, val4, lane);
  } else {
    a0_c51_scatter<C51_MAXR>(s_m[wid], lo, wlo, lane);
    a0_c51_scatter<C51_MAXR>(s_m[wid], up, wup, lane);
  }
  float m[C51_MAXR];
#pragma unroll
  for (int k = 0; k < C51_MAXR; ++k) m[k] = s_m[wid][lane + 32 * k];

  A0_TX(4);
  // ---- cross-entropy with the online row, gradient through log_softmax (agent.py:266-268) ------
  const float lse = logf(ose);
  float ce = 0.0f, msum = 0.0f;
#pragma unroll
  for (int k = 0; k < C51_MAXR; ++k)
    if (k < R && lane + 32 * k < M) { ce += m[k] * ((l[k] - omx) - lse); msum += m[k]; }
  ce = a0_warp_sum(ce);
  msum = a0_warp_sum(msum);
  A0_TX(5);
  float* grow = grad + (size_t)b * A * M;
  for (int a2 = 0; a2 < A; ++a2) {
    if (a2 == a) continue;
    for (int j = lane; j < M; j += 32) grow[(size_t)a2 * M + j] = 0.0f;
  }
#pragma unroll
  for (int k = 0; k < C51_MAXR; ++k) {
    const int j = lane + 32 * k;
    if (k < R && j < M) {
      const float sm = expf((l[k] - omx) - lse);
      grow[(size_t)a * M + j] = w * (sm * msum - m[k]);
      if (target_prob) target_prob[(size_t)b * M + j] = m[k];
    }
  }
  A0_TX(6);
  if (lane == 0) a0_emit(c, b, -ce);
  A0_TX(7);
#ifdef A0_TRACE
  _t2 = _t2 * 0 + (unsigned long long)_c0;      // phases are reported in SM cycles relative to the wait's return
#endif
  if (threadIdx.x == 0) A0_TEND(4);
}

// ------------------------------------------------------------------------------------------------
// C51, the Atari shape (A <= 6 actions, M <= 64 atoms, double-Q action selection given): the same
// arithmetic as a0_k4_c51 -- bit for bit -- with the dependent instruction chain cut down.  A batch of
// 32 is one warp per sample on 8 SMs: the kernel's duration IS the length of one warp's dependent
// chain (device timeline, tools/trace_step.py: 3.5 us of a 3.9 us launch-to-launch period, 20 of them
// per Trainer.step), so what counts is instructions on that chain, not throughput:
//   * arg-max over the A selection values computed by every lane from broadcast loads (no shuffles);
//   * each row maximum is one warp-reduction instruction (redux.sync.max.f32), the two sum-exps are
//     reduced together: 5 shuffle steps before the projection, not 15;
//   * u = l + 1 always holds after the reference's two adjustments (agent.py:246-250), so
//     l = max(ceil(b) - 1, 0) and one key per atom drives the scan of both terms;
//   * everything of the projection that does not depend on the softmax -- the bin positions b_j (a
//     division without IEEE division's slow path, a0_c51_div_delta), the keys, the scan's run masks,
//     the fractions of both terms -- is computed under the latency of the sum-exp reduction, so after
//     it only p_j / sum, two multiplies and the scan of the values are left;
//   * each term of a bin goes to its own shared-memory row (one writer per row and bin by construction)
//     and a bin is then the sum of its four rows in the order of a0_k4_c51's four phases: one store /
//     load round trip instead of four read-modify-writes;
//   * log-sum-exp of the online row and the gradient's softmax are computed as soon as its sum is
//     known; cross-entropy and mass reduced together; the zeros of the sample's [A, M] gradient block
//     (every row but the taken action's) are stored as soon as the action is known, under the latency
//     of the input loads, so only row a is left after the arithmetic.
// ------------------------------------------------------------------------------------------------

// Maximum over the warp in one instruction.  Without .NaN a NaN operand is ignored, as fmaxf does, so this is the
// fmaxf butterfly's result whatever the order of the lanes.
__device__ __forceinline__ float a0_warp_max_redux(float v) {
  float m;
  asm("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(m) : "f"(v));
  return m;
}

// fl32(nu / delta) for 0 <= nu <= fl32(vmax - vmin), equal to __fdiv_rn(nu, delta) and without its slow-path call:
// a float64 quotient by one Markstein correction from rdelta = RN64(1/delta), then rounded to float32.  Every float32
// operand is a normal float64, so the correction step's premises hold (q0 = RN64(nu * rdelta) is within one ulp of
// nu/delta, the remainder is exact) and the float64 quotient is correctly rounded; rounding that to float32 is exact
// too, because a quotient of 24-bit operands is never within 2^-53 relative of a float32 rounding boundary without
// being on it (53 >= 2 * 24 + 2).  tests/test_gpu_c51_chain.py checks every float32 nu of the tested supports.
__device__ __forceinline__ float a0_c51_div_delta(float nu, float delta, double rdelta) {
  const double q0 = __dmul_rn((double)nu, rdelta);
  const double rem = __fma_rn(-q0, (double)delta, (double)nu);
  return __double2float_rn(__fma_rn(rem, rdelta, q0));
}

// delta and 1/delta of a launch: delta is the same float division the kernels' rule uses (oracle/losses.py).
static void a0_c51_delta(float vmin, float vmax, int32_t M, float* delta, double* rdelta) {
  *delta = (vmax - vmin) / (float)(M - 1);
  *rdelta = 1.0 / (double)*delta;
}

// EARLY (a0_loss_c51_linked, A0_C51_EARLY): one link of a chain of dependent launches whose batch-side inputs were
// complete before the link ahead of it passed its own wait.  The CTAs of such a link are resident for the whole
// dependent chain of that link (it lets this one launch right after its wait), so everything that reads only the
// batch side -- action, reward, done, weight, atoms, the projection's geometry, the zeros of the gradient block --
// runs before griddepcontrol.wait; the network outputs are still read after it, and of the online rows only the
// taken action's (known by then).  launch_dependents stays after the wait, so the chain stays one launch deep.
template <int WARPS, bool EARLY>
__global__ void __launch_bounds__(WARPS * 32)
a0_k4_c51_fast(const A0Common c, const float* __restrict__ logits, const float* __restrict__ tgt_logits,
               const float* __restrict__ qsel, const float* __restrict__ atoms, int32_t M, float vmin, float vmax,
               float delta, double rdelta, float* __restrict__ grad, float* __restrict__ target_prob) {
  // the four terms of the projection, one row each: lower terms of atoms lane and lane + 32, then upper terms.  Index
  // M may be written when b rounds above M-1 (never read: that upper term is dropped, as in a0_k4_c51 and
  // oracle.losses.c51_project)
  __shared__ float s_t[WARPS][4][72];
  A0_T0();
#ifdef A0_TRACE
  _tx[7] = (unsigned long long)clock64();      // entry: with EARLY, the batch-side phase is x[7] .. the wait
#endif
  if (!EARLY) {
    A0_PDL_PROLOGUE();
    A0_TMID();
  }
#ifdef A0_TRACE
  long long _c0 = clock64();
#endif
  const int lane = threadIdx.x & 31;
  const int wid = threadIdx.x >> 5;
  const int b = blockIdx.x * WARPS + wid;
  if (b >= c.B) return;       // never the whole CTA: warp 0 always has a sample, and it waits
  const int A = c.A;
  const bool in0 = lane < M, in1 = lane + 32 < M;
  float(*terms)[72] = s_t[wid];
  // ---- the batch side: scalars of the sample, atoms, zeros of the shared rows and of the gradient block ----
  int a, r0;
  float r, d, w, z0, z1;
  float* gb;
  auto batch_side = [&] {
    a = (int)c.action[b];
    r = c.reward[b], d = c.done[b], w = c.weight[b];
    z0 = in0 ? atoms[lane] : 0.0f, z1 = in1 ? atoms[lane + 32] : 0.0f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      terms[t][lane] = 0.0f;
      terms[t][lane + 32] = 0.0f;
    }
    // The gradient block [A, M] of the sample is zero outside row a: those stores depend on nothing but
    // `a`, so they go out now, under the latency of the loads, and only row a is left for the end.
    const int AM = A * M;
    r0 = a * M;
    gb = grad + (size_t)b * AM;
    for (int e = lane; e < AM; e += 32)
      if (e < r0 || e >= r0 + M) gb[e] = 0.0f;
  };
  // ---- the projection's geometry (agent.py:230-250), which needs neither softmax: bin positions, keys of the
  // segmented scan and its run masks, fractions of the lower and upper terms --------------------------------------
  int k0, k1;
  float fl0, fu0, fl1, fu1;
  unsigned join0 = 0, join1 = 0;
  unsigned tail0, tail1;       // run tails (0 / 1)
  auto geometry = [&] {
    const float gm = __fmul_rn(c.gamma_n, __fsub_rn(1.0f, d));
    const float tz0 = fminf(fmaxf(__fadd_rn(r, __fmul_rn(gm, z0)), vmin), vmax);
    const float tz1 = fminf(fmaxf(__fadd_rn(r, __fmul_rn(gm, z1)), vmin), vmax);
    const float bs0 = a0_c51_div_delta(__fsub_rn(tz0, vmin), delta, rdelta);
    const float bs1 = a0_c51_div_delta(__fsub_rn(tz1, vmin), delta, rdelta);
    const int c0 = max((int)ceilf(bs0) - 1, 0), c1 = max((int)ceilf(bs1) - 1, 0);
    k0 = in0 ? c0 : -1, k1 = in1 ? c1 : -1;   // lower bin of atoms lane and lane + 32; the upper one is k + 1
    fl0 = __fsub_rn((float)(c0 + 1), bs0), fu0 = __fsub_rn(bs0, (float)c0);
    fl1 = __fsub_rn((float)(c1 + 1), bs1), fu1 = __fsub_rn(bs1, (float)c1);
    // segmented inclusive scan over the lanes, keyed by the lower bin (bins are non-decreasing in the atom index, so
    // the sources of one bin are adjacent lanes); step s adds the partial sum 2^s lanes up where the keys agree
#pragma unroll
    for (int s = 0; s < 5; ++s) {
      const int q0 = __shfl_up_sync(0xffffffffu, k0, 1 << s), q1 = __shfl_up_sync(0xffffffffu, k1, 1 << s);
      if (lane >= (1 << s) && q0 == k0) join0 |= 1u << s;
      if (lane >= (1 << s) && q1 == k1) join1 |= 1u << s;
    }
    const int n0 = __shfl_down_sync(0xffffffffu, k0, 1), n1 = __shfl_down_sync(0xffffffffu, k1, 1);
    tail0 = k0 >= 0 && (lane == 31 || n0 != k0), tail1 = k1 >= 0 && (lane == 31 || n1 != k1);
  };
  if (EARLY) {
    batch_side();
    geometry();
    // the wait orders memory accesses only: without this the compiler would sink the geometry's arithmetic below it
    asm volatile("" : "+r"(k0), "+r"(k1), "+f"(fl0), "+f"(fu0), "+f"(fl1), "+f"(fu1), "+r"(join0), "+r"(join1),
                 "+r"(tail0), "+r"(tail1), "+r"(a), "+f"(w));
    A0_PDL_PROLOGUE();        // from here on the network outputs are read
    A0_TMID();
#ifdef A0_TRACE
    _c0 = clock64();
#endif
  }
  // ---- every global load of the network outputs, issued up front ---------------------------------------
  float lo_all[C51_SPEC_A][2], tg_all[C51_SPEC_A][2], qs[C51_SPEC_A];
  float l0 = -INFINITY, l1 = -INFINITY, p0 = -INFINITY, p1 = -INFINITY;
  const float* lrow = logits + (size_t)b * A * M + lane;
  const float* trow = tgt_logits + (size_t)b * A * M + lane;
  const float* qrow = qsel + (size_t)b * A;
  if (EARLY) {                // the action is known: only its online row (an action outside [0, A) selects none)
    const bool on = a >= 0 && a < A;
    l0 = (on && in0) ? lrow[a * M] : -INFINITY;
    l1 = (on && in1) ? lrow[a * M + 32] : -INFINITY;
  }
#pragma unroll
  for (int a2 = 0; a2 < C51_SPEC_A; ++a2) {
    const bool on = a2 < A;
    if (!EARLY) {
      lo_all[a2][0] = (on && in0) ? lrow[a2 * M] : -INFINITY;
      lo_all[a2][1] = (on && in1) ? lrow[a2 * M + 32] : -INFINITY;
    }
    tg_all[a2][0] = (on && in0) ? trow[a2 * M] : -INFINITY;
    tg_all[a2][1] = (on && in1) ? trow[a2 * M + 32] : -INFINITY;
    qs[a2] = on ? qrow[a2] : -INFINITY;                 // same address in every lane: one broadcast transaction
  }
  if (!EARLY) batch_side();
  // ---- action selection: torch.argmax's rule (agent.py:224) ---------------------------------------------
  const int a_star = a0_argmax_regs(qs);
#pragma unroll
  for (int a2 = 0; a2 < C51_SPEC_A; ++a2) {
    if (!EARLY && a2 == a) { l0 = lo_all[a2][0]; l1 = lo_all[a2][1]; }
    if (a2 == a_star) { p0 = tg_all[a2][0]; p1 = tg_all[a2][1]; }
  }
  A0_TX(0);
  // ---- both softmaxes: the maxima, then the sum-exps together --------------------------------------------
  const float omx = a0_warp_max_redux(fmaxf(l0, l1)), mx = a0_warp_max_redux(fmaxf(p0, p1));
  A0_TX(1);
  // an idle atom's exponential is expf(-inf) = +0: the arguments are selected, the calls are not branched around
  const float eo0 = expf(in0 ? l0 - omx : -INFINITY), eo1 = expf(in1 ? l1 - omx : -INFINITY);
  p0 = expf(in0 ? p0 - mx : -INFINITY);
  p1 = expf(in1 ? p1 - mx : -INFINITY);
  float ose = eo0 + eo1, se = p0 + p1;
  if (!EARLY) geometry();     // under the latency of the sum-exp reduction
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float a_ = __shfl_xor_sync(0xffffffffu, ose, o);
    const float b_ = __shfl_xor_sync(0xffffffffu, se, o);
    ose += a_;
    se += b_;
  }
  // log-softmax of the online row and its exponential (the gradient's softmax, agent.py:266-268)
  const float lse = logf(ose);
  const float ls0 = (l0 - omx) - lse, ls1 = (l1 - omx) - lse;
  float sm0 = expf(ls0), sm1 = expf(ls1);
  A0_TX(2);
  // ---- projection (agent.py:252-264) -------------------------------------------------------------------
  // The warp pays for IEEE division's slow path (a subroutine) if ANY lane's operands need it -- a zero
  // numerator does: the idle lanes of the second atom chunk (p = 0).  Those lanes divide a harmless
  // stand-in (1) instead and select the exact answer (0) afterwards: same bits.
  float wl0 = 0.0f, wu0 = 0.0f, wl1 = 0.0f, wu1 = 0.0f;
  {
    const float q0 = __fdiv_rn(p0 != 0.0f ? p0 : 1.0f, se), q1 = __fdiv_rn(p1 != 0.0f ? p1 : 1.0f, se);
    const float pj0 = p0 != 0.0f ? q0 : 0.0f, pj1 = p1 != 0.0f ? q1 : 0.0f;
    if (in0) { wl0 = __fmul_rn(pj0, fl0); wu0 = __fmul_rn(pj0, fu0); }
    if (in1) { wl1 = __fmul_rn(pj1, fl1); wu1 = __fmul_rn(pj1, fu1); }
  }
  A0_TX(3);
  // the same combination order as a0_c51_scatter
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    const float a0_ = __shfl_up_sync(0xffffffffu, wl0, 1 << s), b0_ = __shfl_up_sync(0xffffffffu, wu0, 1 << s);
    const float a1_ = __shfl_up_sync(0xffffffffu, wl1, 1 << s), b1_ = __shfl_up_sync(0xffffffffu, wu1, 1 << s);
    if (join0 >> s & 1u) { wl0 = __fadd_rn(wl0, a0_); wu0 = __fadd_rn(wu0, b0_); }
    if (join1 >> s & 1u) { wl1 = __fadd_rn(wl1, a1_); wu1 = __fadd_rn(wu1, b1_); }
  }
  // sm0 and sm1 are needed only by the last stores: without this the compiler would compute them there, after the
  // cross-entropy reduction, instead of under the latency of the scan
  asm volatile("" : "+f"(sm0), "+f"(sm1));
  // A run tail holds its run's total; every row has at most one writer per bin.  a0_k4_c51 adds the four terms of
  // a bin into a zeroed bin in this order (lower terms of both chunks, then upper terms); the absent ones are +0
  // here and there (every term is >= +0), so the sum below has the same bits.
  __syncwarp();                                // the zeros above are visible
  if (tail0) { terms[0][k0] = wl0; terms[2][k0 + 1] = wu0; }
  if (tail1) { terms[1][k1] = wl1; terms[3][k1 + 1] = wu1; }
  __syncwarp();
  const float m0 = __fadd_rn(__fadd_rn(__fadd_rn(terms[0][lane], terms[1][lane]), terms[2][lane]), terms[3][lane]);
  const float m1 = __fadd_rn(__fadd_rn(__fadd_rn(terms[0][lane + 32], terms[1][lane + 32]), terms[2][lane + 32]),
                             terms[3][lane + 32]);
  A0_TX(4);
  // ---- cross-entropy with the online row, gradient through log_softmax (agent.py:266-268) -----------------
  float ce = 0.0f, msum = 0.0f;
  if (in0) { ce += m0 * ls0; msum += m0; }
  if (in1) { ce += m1 * ls1; msum += m1; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float a_ = __shfl_xor_sync(0xffffffffu, ce, o);
    const float b_ = __shfl_xor_sync(0xffffffffu, msum, o);
    ce += a_;
    msum += b_;
  }
  A0_TX(5);
  if (lane == 0) a0_emit(c, b, -ce);           // loss / priority / max_p leave before the gradient block does
  const float g0 = w * (sm0 * msum - m0), g1 = w * (sm1 * msum - m1);
  if (in0) gb[r0 + lane] = g0;
  if (in1) gb[r0 + lane + 32] = g1;
  if (target_prob) {
    if (in0) target_prob[(size_t)b * M + lane] = m0;
    if (in1) target_prob[(size_t)b * M + lane + 32] = m1;
  }
  A0_TX(6);
#ifdef A0_TRACE
  _t2 = _t2 * 0 + (unsigned long long)_c0;
#endif
  if (threadIdx.x == 0) A0_TEND(4);
}

static int g_c51_fast = -1;
static bool a0_option_c51_fast() {
  if (g_c51_fast < 0) {
    const char* e = getenv("A0_C51_FAST");
    g_c51_fast = e ? (atoi(e) != 0) : 1;
  }
  return g_c51_fast != 0;
}
void a0_set_c51_fast(int on) { g_c51_fast = on != 0; }

static int a0_loss_c51_launch(const char* fn, const a0_loss_common_t* c, const float* logits, const float* tgt_logits,
                              const float* qsel, const float* atoms, int32_t M, float vmin, float vmax, float* grad,
                              float* target_prob, bool early, a0_stream_t stream) {
  int rc = a0_check_common(c, fn);
  if (rc) return rc;
  A0_REQUIRE(logits && tgt_logits && atoms && grad, "%s: NULL tensor", fn);
  A0_REQUIRE(M >= 2 && M <= C51_MAXR * 32, "%s: num_atoms %d outside [2,%d]", fn, M, C51_MAXR * 32);
  A0_REQUIRE(vmax > vmin, "%s: vmax must exceed vmin", fn);
  if (c->B == 0) return A0_OK;
  float delta;
  double rdelta;
  a0_c51_delta(vmin, vmax, M, &delta, &rdelta);
  // a0_c51_div_delta needs a finite, nonzero delta (not so when vmax - vmin overflows or underflows)
  if (qsel && c->A <= C51_SPEC_A && M <= 64 && delta > 0.0f && delta < INFINITY && a0_option_c51_fast()) {
    static int warps = 0;                                     // samples (= warps) per CTA: A0_C51_WARPS, measured default
    if (!warps) {
      const char* e = getenv("A0_C51_WARPS");
      warps = e ? atoi(e) : C51_FAST_WARPS;
      if (warps != 1 && warps != 2 && warps != 4 && warps != 8 && warps != 16 && warps != 32) warps = C51_FAST_WARPS;
    }
    const unsigned grid = (unsigned)((c->B + warps - 1) / warps);
#define A0_C51_FAST_LAUNCH(W)                                                                                              \
    if (early)                                                                                                             \
      A0_LAUNCH(a0_k4_c51_fast<W, true>, grid, W * 32, 0, (cudaStream_t)stream, 1, A0_PDL_K4, a0_unpack(c), logits,         \
                tgt_logits, qsel, atoms, M, vmin, vmax, delta, rdelta, grad, target_prob);                                 \
    else                                                                                                                   \
      A0_LAUNCH(a0_k4_c51_fast<W, false>, grid, W * 32, 0, (cudaStream_t)stream, 1, A0_PDL_K4, a0_unpack(c), logits,        \
                tgt_logits, qsel, atoms, M, vmin, vmax, delta, rdelta, grad, target_prob)
    if (warps == 1) { A0_C51_FAST_LAUNCH(1); }
    else if (warps == 2) { A0_C51_FAST_LAUNCH(2); }
    else if (warps == 4) { A0_C51_FAST_LAUNCH(4); }
    else if (warps == 8) { A0_C51_FAST_LAUNCH(8); }
    else if (warps == 16) { A0_C51_FAST_LAUNCH(16); }
    else { A0_C51_FAST_LAUNCH(32); }
#undef A0_C51_FAST_LAUNCH
    return A0_OK;
  }
  A0_LAUNCH(a0_k4_c51, (unsigned)((c->B + C51_WARPS - 1) / C51_WARPS), C51_WARPS * 32, 0, (cudaStream_t)stream, 1, A0_PDL_K4,
            a0_unpack(c), logits, tgt_logits, qsel, atoms, M, vmin, vmax, grad, target_prob);
  return A0_OK;
}

extern "C" int a0_loss_c51(const a0_loss_common_t* c, const float* logits, const float* tgt_logits,
                           const float* qsel, const float* atoms, int32_t M, float vmin, float vmax, float* grad,
                           float* target_prob, a0_stream_t stream) {
  return a0_loss_c51_launch("a0_loss_c51", c, logits, tgt_logits, qsel, atoms, M, vmin, vmax, grad, target_prob, false,
                            stream);
}

extern "C" int a0_loss_c51_linked(const a0_loss_common_t* c, const float* logits, const float* tgt_logits,
                                  const float* qsel, const float* atoms, int32_t M, float vmin, float vmax, float* grad,
                                  float* target_prob, int32_t flags, a0_stream_t stream) {
  A0_REQUIRE((flags & ~A0_C51_EARLY) == 0, "a0_loss_c51_linked: unknown flags 0x%x", (unsigned)flags);
  return a0_loss_c51_launch("a0_loss_c51_linked", c, logits, tgt_logits, qsel, atoms, M, vmin, vmax, grad, target_prob,
                            (flags & A0_C51_EARLY) != 0, stream);
}

// Every float32 nu in [0, hi] (by bit pattern): a0_c51_div_delta against __fdiv_rn.  out[0] += mismatches,
// out[1] = min(bit pattern of a mismatching nu).
__global__ void a0_c51_div_check_kernel(uint32_t hi, float delta, double rdelta, unsigned long long* out) {
  unsigned long long bad = 0, first = ~0ull;
  for (unsigned long long u = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; u <= hi;
       u += (unsigned long long)gridDim.x * blockDim.x) {
    const float nu = __uint_as_float((uint32_t)u);
    if (__float_as_uint(a0_c51_div_delta(nu, delta, rdelta)) != __float_as_uint(__fdiv_rn(nu, delta))) {
      ++bad;
      first = min(first, u);
    }
  }
  if (bad) {
    atomicAdd(out, bad);
    atomicMin(out + 1, first);
  }
}

extern "C" int a0_c51_div_check(float vmin, float vmax, int32_t M, unsigned long long* out, a0_stream_t stream) {
  A0_REQUIRE(out != nullptr, "a0_c51_div_check: NULL output");
  A0_REQUIRE(M >= 2 && vmax > vmin, "a0_c51_div_check: M %d, vmin %g, vmax %g", M, (double)vmin, (double)vmax);
  float delta;
  double rdelta;
  a0_c51_delta(vmin, vmax, M, &delta, &rdelta);
  A0_REQUIRE(delta > 0.0f && delta < INFINITY, "a0_c51_div_check: delta %g is zero or infinite", (double)delta);
  const float hi = vmax - vmin;
  A0_REQUIRE(hi < INFINITY, "a0_c51_div_check: vmax - vmin overflows");
  uint32_t hb;
  memcpy(&hb, &hi, sizeof(hb));
  a0_c51_div_check_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(hb, delta, rdelta, out);
  A0_LAUNCH_CHECK();
  return A0_OK;
}

// ------------------------------------------------------------------------------------------------
// Quantile-Huber family (agent.py:110-114; QR :273-293, IQN :297-327, FQF :340-388).
// One CTA per sample, thread j owns online quantile q_j and loops over the Ni targets held in
// shared memory: Ni*Nj pairs (40 000 for QR-200) never leave registers.
//   loss_b = (1/Ni) sum_i sum_j |tau_j - 1[T_i < q_j]| * huber(q_j - T_i)
//   grad_j = (w/Ni) sum_i |tau_j - 1[q_j - T_i > 0]| * clamp(q_j - T_i, -1, 1)
// ------------------------------------------------------------------------------------------------
constexpr int QH_SPEC_A = 8;     // all-action fetch of the quantile kernel (IQN/FQF layout) up to this many actions

__device__ __forceinline__ float a0_block_sum(float v, float* red, int nwarps) {
  v = a0_warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float s = 0.0f;
  for (int i = 0; i < nwarps; ++i) s += red[i];
  return s;
}

// SPEC: the all-action fetch for IQN/FQF-sized samples (a separate instantiation, so that QR-200's
// issue-bound pair loop keeps its register allocation: with both paths in one kernel it spilled inside
// the loop and QR went from 10.6 to 14.6 us)
template <bool SPEC>
__global__ void __launch_bounds__(A0_MAX_QUANTILES)
a0_k4_quantile(const A0Common c, int32_t layout, const float* __restrict__ q, const float* __restrict__ qt,
               const float* __restrict__ taus, const float* __restrict__ qsel, int32_t Ni, int32_t Nj,
               float* __restrict__ grad, const float* __restrict__ q_bar, const float* __restrict__ taus_full,
               float* __restrict__ fraction_loss, float* __restrict__ grad_taus) {
  __shared__ float sT[A0_MAX_QUANTILES];
  __shared__ float sQ[A0_MAX_QUANTILES];
  __shared__ float sMean[A0_MAX_ACTIONS];
  __shared__ float red[A0_MAX_QUANTILES / 32];
  __shared__ int s_astar;
  A0_PDL_PROLOGUE();
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nwarps = blockDim.x >> 5;
  const int A = c.A;
  // element (b, n, a) of an online/target tensor
  const size_t sN_q = layout == 0 ? 1 : (size_t)A, sA_q = layout == 0 ? (size_t)Nj : 1;
  const size_t sN_t = layout == 0 ? 1 : (size_t)A, sA_t = layout == 0 ? (size_t)Ni : 1;
  const float* qb = q + (size_t)b * A * Nj;
  const float* tb = qt + (size_t)b * A * Ni;

  float qj = 0.0f, tau = 0.0f, w;
  int a;
  if (SPEC) {
    a = (int)c.action[b];
    const float r = c.reward[b], d = c.done[b];
    w = c.weight[b];
    // IQN / FQF with few actions (64 x 64 or 32 x 32 pairs per sample: latency-bound, unlike QR-200):
    // every thread fetches its quantile of ALL actions from both networks -- one [A]-row each in this
    // layout -- and the A selection values (broadcast) in one batch of loads, then picks the taken and
    // the arg-max action in registers: no second, action-dependent memory round trip, no shared-memory
    // hand-off of the arg-max.
    float qs[QH_SPEC_A], tv[QH_SPEC_A], qv[QH_SPEC_A];
#pragma unroll
    for (int a2 = 0; a2 < QH_SPEC_A; ++a2) {
      const bool on = a2 < A;
      qs[a2] = on ? qsel[(size_t)b * A + a2] : -INFINITY;
      tv[a2] = (on && tid < Ni) ? tb[(size_t)tid * A + a2] : 0.0f;
      qv[a2] = (on && tid < Nj) ? qb[(size_t)tid * A + a2] : 0.0f;
    }
    if (tid < Nj) tau = taus[(size_t)b * Nj + tid];
    const int a_star = a0_argmax_regs(qs);
    float tsel = 0.0f;
#pragma unroll
    for (int a2 = 0; a2 < QH_SPEC_A; ++a2) {
      if (a2 == a_star) tsel = tv[a2];
      if (a2 == a) qj = qv[a2];
    }
    if (tid < Ni) sT[tid] = a0_td_target(r, d, c.gamma_n, tsel);
    if (tid < Nj) sQ[tid] = qj;
    __syncthreads();
  } else {
  // ---- action selection ------------------------------------------------------------------------
  if (qsel) {
    if (wid == 0) {
      const int as = a0_warp_argmax(lane < A ? qsel[(size_t)b * A + lane] : -INFINITY, lane);
      if (lane == 0) s_astar = as;
    }
  } else {
    // QR without double_q: argmax_a mean_i theta'[a][i] (agent.py:279)
    for (int a2 = wid; a2 < A; a2 += nwarps) {
      float s = 0.0f;
      for (int i = lane; i < Ni; i += 32) s += tb[a2 * sA_t + i * sN_t];
      s = a0_warp_sum(s);
      if (lane == 0) sMean[a2] = __fdiv_rn(s, (float)Ni);
    }
    __syncthreads();
    if (wid == 0) {
      const int as = a0_warp_argmax(lane < A ? sMean[lane] : -INFINITY, lane);
      if (lane == 0) s_astar = as;
    }
  }
  __syncthreads();
  const int a_star = s_astar;
  a = (int)c.action[b];
  const float r = c.reward[b], d = c.done[b];
  w = c.weight[b];
  if (tid < Ni) sT[tid] = a0_td_target(r, d, c.gamma_n, tb[a_star * sA_t + tid * sN_t]);
  if (tid < Nj) {
    qj = qb[a * sA_q + tid * sN_q];
    tau = taus ? taus[(size_t)b * Nj + tid] : __fdiv_rn((float)(2 * tid + 1), 2.0f * (float)Nj);
    sQ[tid] = qj;
  }
  __syncthreads();
  }

  // ---- pair loop ---------------------------------------------------------------------------------
  // With a = |u|, c = min(a, 1):  huber(u) = c * (a - c/2),  clamp(u, -1, 1) = copysign(c, u),
  // |tau - 1[u > 0]| = u > 0 ? 1 - tau : tau   -- nine FP32 instructions per pair.
  float lsum = 0.0f, gsum = 0.0f;
  if (tid < Nj) {
    // the weight is (1 - tau) on the pairs with u > 0 and tau on the others: accumulate the two groups
    // separately (predicated FFMA/FADD, 8 instructions per pair of which 2 on the half-rate ALU
    // pipe, instead of two selects: 9 and 4) and weight them once at the end
    float lp = 0.0f, ln = 0.0f, gp = 0.0f, gn = 0.0f;
#pragma unroll 8
    for (int i = 0; i < Ni; ++i) {
      const float uij = qj - sT[i];
      const float a_ = fabsf(uij);
      const float c_ = fminf(a_, 1.0f);
      const float x_ = fmaf(-0.5f, c_, a_);
      if (uij > 0.0f) { lp = fmaf(c_, x_, lp); gp += c_; }
      else { ln = fmaf(c_, x_, ln); gn += c_; }
    }
    const float k_pos = 1.0f - tau;
    lsum = fmaf(k_pos, lp, tau * ln);
    gsum = fmaf(k_pos, gp, -tau * gn);
  }
  const float total = a0_block_sum(lsum, red, nwarps);
  // zero the whole [A, Nj] gradient block of this sample, then fill the taken action's column/row
  float* gb = grad + (size_t)b * A * Nj;
  for (int i = tid; i < A * Nj; i += blockDim.x) gb[i] = 0.0f;
  __syncthreads();
  if (tid < Nj) gb[a * sA_q + tid * sN_q] = __fdiv_rn(w, (float)Ni) * gsum;
  if (tid == 0) a0_emit(c, b, __fdiv_rn(total, (float)Ni));

  // ---- FQF fraction loss (agent.py:371-387) ----------------------------------------------------
  if (q_bar) {
    const int F = Nj;
    float gi = 0.0f, contrib = 0.0f;
    if (tid < F - 1) {
      const float* qbar_b = q_bar + (size_t)b * (F - 1) * A;
      const float qi = qbar_b[(size_t)tid * A + a];
      const float prev = tid == 0 ? sQ[0] : qbar_b[(size_t)(tid - 1) * A + a];
      const float next = tid == F - 2 ? sQ[F - 1] : qbar_b[(size_t)(tid + 1) * A + a];
      const float v1 = qi - sQ[tid], v2 = qi - sQ[tid + 1];
      gi = (qi > prev ? v1 : -v1) + (qi < next ? v2 : -v2);
      contrib = gi * taus_full[(size_t)b * (F + 1) + tid + 1];
    }
    const float fl = a0_block_sum(contrib, red, nwarps);
    if (tid == 0 && fraction_loss) fraction_loss[b] = fl;
    if (grad_taus) {
      float* gt = grad_taus + (size_t)b * (F + 1);
      if (tid < F - 1) gt[tid + 1] = w * gi;
      if (tid == 0) { gt[0] = 0.0f; gt[F] = 0.0f; }
    }
  }
}

// ---- QR-sized samples: the same pair sums in O(N log N) ------------------------------------------------------
// 200 x 200 pairs at 8 issue slots each made QR-200 the one kernel of the path bound by arithmetic (10.4 us per
// batch of 512, 0.32 of the FP32 peak).  For a fixed online quantile q the targets split, once SORTED, into four
// contiguous ranges of u = q - T:
//     A: T <= q-1  (u >= 1,  |u| - 1/2, weight 1-tau)      B: q-1 < T < q   (0 < u < 1,  u^2/2, weight 1-tau)
//     C: q <= T < q+1 (-1 < u <= 0, u^2/2, weight tau)      D: T >= q+1      (u <= -1, |u| - 1/2, weight tau)
// and over a range the Huber terms are polynomials in q whose coefficients are the range's count, sum T and
// sum T^2 -- differences of prefix sums.  (At u = +-1 and u = 0 neighbouring ranges give the same value and the
// same clamp, so which side a boundary target falls on does not matter.)  Per sample: sort the Ni targets (warp
// bitonic networks in registers, then three merge levels in shared memory where every element finds its rank in
// the sibling run by binary search -- no compare-exchange stages, three barriers), prefix sums of T and T^2, and
// per online quantile three binary searches plus ~25 flops.  The prefix sums and the polynomial are evaluated in
// float64 and centred on the median target c (sums of T-c and (T-c)^2, q-c): the quadratic ranges subtract numbers of
// size N*(T-c)^2 to get terms of size (q-T)^2 <= 1, and uncentred sums of size N*T^2 lost the 1e-5 contract from
// |T| ~ 1e5 (8e-5 relative; 8e-3 at 1e6).  The summation
// order differs from the reference's pairwise sum, so this kernel lives under the 1e-5 relative contract (it is
// closer to the exact sum than the fp32 pairwise form); oracle.losses.huber_qr_sorted is its specification.
constexpr int QS_MAX = A0_MAX_QUANTILES;         // 256 = 8 sorted runs of one warp each
static_assert(QS_MAX == 256, "the merge tree below is written for 8 runs of 32");

// smallest float greater than x (x finite): "v <= x" becomes "v < next_up(x)", so both tie rules of the merge are
// one comparison
__device__ __forceinline__ float a0_qs_next_up(float x) {
  const uint32_t b = __float_as_uint(x);
  if (x == 0.0f) return __uint_as_float(1u);
  return __uint_as_float((b >> 31) ? b - 1u : b + 1u);
}
// Padding above the Ni real targets: finite, larger than any real target, DISTINCT and increasing with the index,
// so that pads never tie with each other (tied elements of a right run count "<=", which a pad run would not
// survive) and always sort to the end in index order.
__device__ __forceinline__ float a0_qs_pad(int idx) { return __uint_as_float(0x7f7fff00u + (uint32_t)idx); }

// One merge level: the thread's element x, currently at src[pos] (runs of S sorted values), finds how many
// elements of its sibling run precede it -- binary search with a running pointer: LDS [p + imm], FSETP, predicated
// add per step -- and moves to its rank in the merged run of 2S (returned: the thread keeps its element in a
// register and follows its position, so no level re-reads it).  x_up = next_up(x).
// (Indices, not pointers: with 32-bit indices into the static shared arrays every step is LDS [R + imm], FSETP and a
// predicated add; generic 64-bit pointers cost two more instructions per step -- ncu source view.)
template <int S_LOG>
__device__ __forceinline__ int a0_qs_merge(const float* __restrict__ src, float* __restrict__ dst, int pos, float x, float x_up) {
  constexpr int S = 1 << S_LOG;
  const int r = pos >> S_LOG, p = pos & (S - 1);
  const int sib = (r ^ 1) << S_LOG;
  const float xc = (r & 1) ? x_up : x;            // ties: the left run's elements go first (unique ranks)
  int lo = sib;
#pragma unroll
  for (int step = S >> 1; step > 0; step >>= 1)
    lo += (src[lo + step - 1] < xc) ? step : 0;
  lo += (src[lo] < xc) ? 1 : 0;
  const int out = ((r >> 1) << (S_LOG + 1)) + p + (lo - sib);
  dst[out] = x;
  return out;
}

// SPEC (qsel given, A <= QH_SPEC_A): every thread fetches its quantile of ALL actions from both networks together with
// the selection values, the taken action and the scalars in ONE batch of loads and picks in registers -- no arg-max
// hand-off through shared memory, no second (action-dependent) memory round trip -- and the sample's gradient block is
// zeroed under the latency of those loads.  Under the gather's traffic (the K4 launches of a batch-512 step run while
// the later batches are being fetched) a dependent round trip costs several microseconds, not 0.4.
template <bool SPEC, int AMAX>
__global__ void __launch_bounds__(QS_MAX)
a0_k4_quantile_sorted(const A0Common c, int32_t layout, const float* __restrict__ q, const float* __restrict__ qt,
                      const float* __restrict__ taus, const float* __restrict__ qsel, int32_t Ni, int32_t Nj,
                      float* __restrict__ grad) {
  __shared__ float bufA[QS_MAX], bufB[QS_MAX];
  __shared__ __align__(16) double S1[QS_MAX + 2], S2[QS_MAX + 2];
  __shared__ __align__(16) double ws1[QS_MAX / 32], ws2[QS_MAX / 32];
  __shared__ float sMean[A0_MAX_ACTIONS];
  __shared__ float red[QS_MAX / 32];
  __shared__ int s_astar;
  A0_PDL_PROLOGUE();
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nthreads = blockDim.x, nwarps = nthreads >> 5;      // 32 * ceil(max(Ni, Nj) / 32): 7 warps for QR-200
  const int A = c.A;
  const int sN_q = layout == 0 ? 1 : A, sA_q = layout == 0 ? Nj : 1;       // 32-bit strides inside one sample's block
  const int sN_t = layout == 0 ? 1 : A, sA_t = layout == 0 ? Ni : 1;
  const float* qb = q + (size_t)b * A * Nj;
  const float* tb = qt + (size_t)b * A * Ni;
  // runs without threads (beyond blockDim) hold pads in both buffers: they are never moved and never counted
  for (int i = nthreads + tid; i < QS_MAX; i += nthreads) { bufA[i] = a0_qs_pad(i); bufB[i] = a0_qs_pad(i); }
  float* gb = grad + (size_t)b * A * Nj;
  int a;
  float w, qj = 0.0f, tau = 0.0f, x;
  if (SPEC) {
    float qs[AMAX], tv[AMAX], qv[AMAX];
#pragma unroll
    for (int a2 = 0; a2 < AMAX; ++a2) {
      const bool on = a2 < A;
      qs[a2] = on ? qsel[(size_t)b * A + a2] : -INFINITY;
      tv[a2] = (on && tid < Ni) ? tb[a2 * sA_t + tid * sN_t] : 0.0f;
      qv[a2] = (on && tid < Nj) ? qb[a2 * sA_q + tid * sN_q] : 0.0f;
    }
    a = (int)c.action[b];
    const float r = c.reward[b], d = c.done[b];
    w = c.weight[b];
    if (tid < Nj) tau = taus ? taus[(size_t)b * Nj + tid] : __fdiv_rn((float)(2 * tid + 1), 2.0f * (float)Nj);
    for (int i = tid; i < A * Nj; i += nthreads) gb[i] = 0.0f;      // the taken action's entries are rewritten after the barriers below
    const int a_star = a0_argmax_regs(qs);
    float tsel = 0.0f;
#pragma unroll
    for (int a2 = 0; a2 < AMAX; ++a2) {
      if (a2 == a_star) tsel = tv[a2];
      if (a2 == a) qj = qv[a2];
    }
    x = tid < Ni ? a0_td_target(r, d, c.gamma_n, tsel) : a0_qs_pad(tid);
  } else {
  // ---- action selection (as a0_k4_quantile) ------------------------------------------------------------
  if (qsel) {
    if (wid == 0) {
      const int as = a0_warp_argmax(lane < A ? qsel[(size_t)b * A + lane] : -INFINITY, lane);
      if (lane == 0) s_astar = as;
    }
  } else {
    for (int a2 = wid; a2 < A; a2 += nwarps) {
      float s = 0.0f;
      for (int i = lane; i < Ni; i += 32) s += tb[a2 * sA_t + i * sN_t];
      s = a0_warp_sum(s);
      if (lane == 0) sMean[a2] = __fdiv_rn(s, (float)Ni);
    }
    __syncthreads();
    if (wid == 0) {
      const int as = a0_warp_argmax(lane < A ? sMean[lane] : -INFINITY, lane);
      if (lane == 0) s_astar = as;
    }
  }
  a = (int)c.action[b];
  const float r = c.reward[b], d = c.done[b];
  w = c.weight[b];
  if (tid < Nj) {
    qj = qb[a * sA_q + tid * sN_q];
    tau = taus ? taus[(size_t)b * Nj + tid] : __fdiv_rn((float)(2 * tid + 1), 2.0f * (float)Nj);
  }
  __syncthreads();
  const int a_star = s_astar;
  x = tid < Ni ? a0_td_target(r, d, c.gamma_n, tb[a_star * sA_t + tid * sN_t]) : a0_qs_pad(tid);
  }
  // ---- sort the targets: one bitonic network per warp, then merge 32 -> 64 -> 128 -> 256 ------------------
#pragma unroll
  for (int lk = 1; lk <= 5; ++lk) {
#pragma unroll
    for (int lj = lk - 1; lj >= 0; --lj) {
      const float y = __shfl_xor_sync(0xffffffffu, x, 1 << lj);
      // keep the minimum iff bit lj and bit lk of the lane agree (ascending blocks of 2^lk; lk = 5: the whole warp)
      const bool keep_min = (((lane ^ (lane >> (lk - lj))) >> lj) & 1) == 0;
      x = keep_min ? fminf(x, y) : fmaxf(x, y);
    }
  }
  const float x_up = a0_qs_next_up(x);
  bufA[tid] = x;
  __syncthreads();
  int pos = a0_qs_merge<5>(bufA, bufB, tid, x, x_up);
  __syncthreads();
  pos = a0_qs_merge<6>(bufB, bufA, pos, x, x_up);
  __syncthreads();
  a0_qs_merge<7>(bufA, bufB, pos, x, x_up);
  __syncthreads();
  // ---- prefix sums of T-c and (T-c)^2 over the sorted targets (float64) --------------------------------------
  // c = the sorted target at Ni/2.  Centring keeps the sums of size N*(T-c)^2 instead of N*T^2, so the quadratic
  // ranges lose no precision as |T| grows; T - c and q - c are exact in float64 (T, q and c are fp32).
  const double cen = (double)bufB[Ni >> 1];
  {
    const double y = tid < Ni ? (double)bufB[tid] - cen : 0.0;
    double p1 = y, p2 = y * y;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double t1 = __shfl_up_sync(0xffffffffu, p1, o), t2 = __shfl_up_sync(0xffffffffu, p2, o);
      if (lane >= o) { p1 += t1; p2 += t2; }
    }
    if (lane == 31) { ws1[wid] = p1; ws2[wid] = p2; }
    __syncthreads();
    double b1 = 0.0, b2 = 0.0;
#pragma unroll
    for (int w2 = 0; w2 < QS_MAX / 32 - 1; ++w2)
      if (w2 < wid) { b1 += ws1[w2]; b2 += ws2[w2]; }
    S1[tid + 1] = p1 + b1;
    S2[tid + 1] = p2 + b2;
    if (tid == 0) { S1[0] = 0.0; S2[0] = 0.0; }
  }
  __syncthreads();
  // ---- per online quantile: the three range boundaries, then the closed form ---------------------------------
  float lsum = 0.0f, gsum = 0.0f;
  if (tid < Nj) {
    const float qm_up = a0_qs_next_up(qj - 1.0f), qp = qj + 1.0f;
    int ia = 0, ib = 0, ic = 0;                       // -> #{T <= q-1}, #{T < q}, #{T < q+1}
#pragma unroll
    for (int step = QS_MAX >> 1; step > 0; step >>= 1) {
      ia += (bufB[ia + step - 1] < qm_up) ? step : 0;
      ib += (bufB[ib + step - 1] < qj) ? step : 0;
      ic += (bufB[ic + step - 1] < qp) ? step : 0;
    }
    ia += (bufB[ia] < qm_up) ? 1 : 0;
    ib += (bufB[ib] < qj) ? 1 : 0;
    ic += (bufB[ic] < qp) ? 1 : 0;
    ia = min(ia, Ni); ib = min(max(ib, ia), Ni); ic = min(max(ic, ib), Ni);
    const double qd = (double)qj - cen, td = (double)tau;       // the range boundaries above use the uncentred fp32 values
    const double nA = (double)ia, nB = (double)(ib - ia), nC = (double)(ic - ib), nD = (double)(Ni - ic);
    const double s1a = S1[ia], s1b = S1[ib], s1c = S1[ic];
    const double s1B = s1b - s1a, s2B = S2[ib] - S2[ia];
    const double s1C = s1c - s1b, s2C = S2[ic] - S2[ib];
    const double s1D = S1[Ni] - s1c;
    const double A_ = nA * (qd - 0.5) - s1a;
    const double B_ = 0.5 * ((nB * qd - 2.0 * s1B) * qd + s2B);
    const double C_ = 0.5 * ((nC * qd - 2.0 * s1C) * qd + s2C);
    const double D_ = s1D - nD * (qd + 0.5);
    lsum = (float)((1.0 - td) * (A_ + B_) + td * (C_ + D_));
    gsum = (float)((1.0 - td) * (nA + nB * qd - s1B) + td * (nC * qd - s1C - nD));
  }
  const float total = a0_block_sum(lsum, red, nwarps);
  if (!SPEC) {
    for (int i = tid; i < A * Nj; i += nthreads) gb[i] = 0.0f;
    __syncthreads();
  }
  if (tid < Nj) gb[a * sA_q + tid * sN_q] = __fdiv_rn(w, (float)Ni) * gsum;
  if (tid == 0) a0_emit(c, b, __fdiv_rn(total, (float)Ni));
}

// ---- the sorted form with ONE WARP per sample (measured alternative, A0_OPT_QH_SORTED = 2) -----------------------
// The CTA-per-sample kernel above spends ~1000 instructions in each of its 7 warps: a rank-by-binary-search merge
// costs every element log2(run) shared-memory probes per level, and prefix sums, barriers and the action selection are
// paid per warp.  With the whole sample in ONE warp the 256 (padded) targets sit in registers, 8 per lane (element
// e = 8*lane + r), and are sorted by a plain bitonic network: the 21 stages whose partner distance is below 8 are
// register-to-register min/max, the 15 others one shuffle per element -- no shared memory, no barrier.  Prefix sums are
// 8 local adds plus one warp scan of the lane totals; each lane then evaluates the closed form for its 7 online
// quantiles.  2900 warp-instructions per sample instead of 7200 (ncu) -- and yet 7.4 us per batch of 512 against 6.9:
// a batch of 512 is 512 warps on 592 schedulers, so the launch lasts as long as ONE warp's dependent chain (17 % issue
// utilisation), which is longer here than the CTA form's per-warp chain.  It would win from ~2000 samples per launch.
constexpr int QW_R = 8;                            // targets per lane
__device__ __forceinline__ void a0_qw_sort256(float (&x)[QW_R], int lane) {
#pragma unroll
  for (int k = 2; k <= 256; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j < QW_R) {
        // partner inside the lane; the direction of an ascending block of k depends on r (k <= 8) or on the lane
#pragma unroll
        for (int r = 0; r < QW_R; ++r) {
          if (r & j) continue;
          const float a = x[r], b = x[r | j];
          const float lo = fminf(a, b), hi = fmaxf(a, b);
          const bool up = k < QW_R ? ((r & k) == 0) : (((lane * QW_R) & k) == 0);      // bit log2(k) of e = 8*lane + r
          x[r] = up ? lo : hi;
          x[r | j] = up ? hi : lo;
        }
      } else {
        const int jl = j / QW_R;
        const bool keep_min = ((lane & jl) == 0) == (((lane * QW_R) & k) == 0);
#pragma unroll
        for (int r = 0; r < QW_R; ++r) {
          const float y = __shfl_xor_sync(0xffffffffu, x[r], jl);
          x[r] = keep_min ? fminf(x[r], y) : fmaxf(x[r], y);
        }
      }
    }
  }
}

__global__ void __launch_bounds__(32)
a0_k4_quantile_warp(const A0Common c, int32_t layout, const float* __restrict__ q, const float* __restrict__ qt,
                    const float* __restrict__ taus, const float* __restrict__ qsel, int32_t Ni, int32_t Nj,
                    float* __restrict__ grad) {
  __shared__ __align__(16) float sT[QS_MAX];
  __shared__ __align__(16) double S1[QS_MAX + 2], S2[QS_MAX + 2];
  A0_PDL_PROLOGUE();
  const int b = blockIdx.x, lane = threadIdx.x;
  const int A = c.A;
  const int sN_q = layout == 0 ? 1 : A, sA_q = layout == 0 ? Nj : 1;
  const int sN_t = layout == 0 ? 1 : A, sA_t = layout == 0 ? Ni : 1;
  const float* qb = q + (size_t)b * A * Nj;
  const float* tb = qt + (size_t)b * A * Ni;
  float* gb = grad + (size_t)b * A * Nj;
  // zeros of the sample's whole [A, Nj] gradient block first (under the latency of the loads); the taken action's
  // entries are written at the end by other lanes, ordered by the warp barriers in between
  for (int i = lane; i < A * Nj; i += 32) gb[i] = 0.0f;
  // ---- action selection ----------------------------------------------------------------------------------
  int a_star;
  if (qsel) {
    a_star = a0_warp_argmax(lane < A ? qsel[(size_t)b * A + lane] : -INFINITY, lane);
  } else {
    // QR without double_q: argmax_a mean_i theta'[a][i] (agent.py:279)
    float best = -INFINITY;
    a_star = 0;
    for (int a2 = 0; a2 < A; ++a2) {
      float s = 0.0f;
      for (int i = lane; i < Ni; i += 32) s += tb[a2 * sA_t + i * sN_t];
      s = __fdiv_rn(a0_warp_sum(s), (float)Ni);
      if (a0_argmax_takes(s, best)) { best = s; a_star = a2; }
    }
  }
  a_star = __shfl_sync(0xffffffffu, a_star, 0);
  const int a = (int)c.action[b];
  const float r = c.reward[b], d = c.done[b], w = c.weight[b];
  // ---- the targets, 8 per lane, sorted in registers ----------------------------------------------------------
  float x[QW_R];
#pragma unroll
  for (int i = 0; i < QW_R; ++i) {
    const int e = lane * QW_R + i;
    x[i] = e < Ni ? a0_td_target(r, d, c.gamma_n, tb[a_star * sA_t + e * sN_t]) : a0_qs_pad(e);
  }
  a0_qw_sort256(x, lane);
  // ---- sorted targets and their float64 prefix sums, centred on the target at Ni/2 (as a0_k4_quantile_sorted) --
  {
    float4* dst = reinterpret_cast<float4*>(sT + lane * QW_R);
    dst[0] = make_float4(x[0], x[1], x[2], x[3]);
    dst[1] = make_float4(x[4], x[5], x[6], x[7]);
  }
  __syncwarp();
  const double cen = (double)sT[Ni >> 1];
  {
    double c1[QW_R], c2[QW_R];
    double p1 = 0.0, p2 = 0.0;
#pragma unroll
    for (int i = 0; i < QW_R; ++i) {
      const double y = (lane * QW_R + i) < Ni ? (double)x[i] - cen : 0.0;      // sorted position >= Ni: a pad
      p1 += y;
      p2 += y * y;
      c1[i] = p1;
      c2[i] = p2;
    }
    double t1 = p1, t2 = p2;                        // inclusive scan of the lane totals
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double u1 = __shfl_up_sync(0xffffffffu, t1, o), u2 = __shfl_up_sync(0xffffffffu, t2, o);
      if (lane >= o) { t1 += u1; t2 += u2; }
    }
    const double e1 = t1 - p1, e2 = t2 - p2;        // exclusive: everything in front of this lane
#pragma unroll
    for (int i = 0; i < QW_R; ++i) {
      S1[lane * QW_R + i + 1] = e1 + c1[i];
      S2[lane * QW_R + i + 1] = e2 + c2[i];
    }
    if (lane == 0) { S1[0] = 0.0; S2[0] = 0.0; }
  }
  __syncwarp();
  // ---- per online quantile: the three range boundaries, then the closed form -----------------------------------
  float lsum = 0.0f;
  const float wn = __fdiv_rn(w, (float)Ni);
  const double s1N = S1[Ni];
#pragma unroll 2
  for (int j = lane; j < Nj; j += 32) {
    const float qj = qb[a * sA_q + j * sN_q];
    const float tau = taus ? taus[(size_t)b * Nj + j] : __fdiv_rn((float)(2 * j + 1), 2.0f * (float)Nj);
    const float qm_up = a0_qs_next_up(qj - 1.0f), qp = qj + 1.0f;
    int ia = 0, ib = 0, ic = 0;                       // -> #{T <= q-1}, #{T < q}, #{T < q+1}
#pragma unroll
    for (int step = QS_MAX >> 1; step > 0; step >>= 1) {
      ia += (sT[ia + step - 1] < qm_up) ? step : 0;
      ib += (sT[ib + step - 1] < qj) ? step : 0;
      ic += (sT[ic + step - 1] < qp) ? step : 0;
    }
    ia += (sT[ia] < qm_up) ? 1 : 0;
    ib += (sT[ib] < qj) ? 1 : 0;
    ic += (sT[ic] < qp) ? 1 : 0;
    ia = min(ia, Ni); ib = min(max(ib, ia), Ni); ic = min(max(ic, ib), Ni);
    const double qd = (double)qj - cen, td = (double)tau;
    const double nA = (double)ia, nB = (double)(ib - ia), nC = (double)(ic - ib), nD = (double)(Ni - ic);
    const double s1a = S1[ia], s1b = S1[ib], s1c = S1[ic];
    const double s1B = s1b - s1a, s2B = S2[ib] - S2[ia];
    const double s1C = s1c - s1b, s2C = S2[ic] - S2[ib];
    const double s1D = s1N - s1c;
    const double A_ = nA * (qd - 0.5) - s1a;
    const double B_ = 0.5 * ((nB * qd - 2.0 * s1B) * qd + s2B);
    const double C_ = 0.5 * ((nC * qd - 2.0 * s1C) * qd + s2C);
    const double D_ = s1D - nD * (qd + 0.5);
    lsum += (float)((1.0 - td) * (A_ + B_) + td * (C_ + D_));
    const float gsum = (float)((1.0 - td) * (nA + nB * qd - s1B) + td * (nC * qd - s1C - nD));
    gb[a * sA_q + j * sN_q] = wn * gsum;
  }
  const float total = a0_warp_sum(lsum);
  if (lane == 0) a0_emit(c, b, __fdiv_rn(total, (float)Ni));
}

static int g_qh_spec = -1;         // A0_OPT_QH_SPEC = 0: the quantile kernels without the all-action fetch (measured alternative)
static bool a0_option_qh_spec() {
  if (g_qh_spec < 0) {
    const char* e = getenv("A0_QH_SPEC");
    g_qh_spec = e ? (atoi(e) != 0) : 1;
  }
  return g_qh_spec != 0;
}
void a0_set_qh_spec(int on) { g_qh_spec = on != 0; }
static int g_qh_sorted = -1;
static int a0_option_qh_sorted() {
  if (g_qh_sorted < 0) {
    const char* e = getenv("A0_QH_SORTED");
    g_qh_sorted = e ? atoi(e) : 1;
    if (g_qh_sorted < 0 || g_qh_sorted > 2) g_qh_sorted = 1;
  }
  return g_qh_sorted;
}
void a0_set_qh_sorted(int mode) { g_qh_sorted = (mode < 0 || mode > 2) ? 1 : mode; }

extern "C" int a0_loss_quantile(const a0_loss_common_t* c, int32_t layout, const float* q, const float* qt,
                                const float* taus, const float* qsel, int32_t Ni, int32_t Nj, float* grad,
                                const float* q_bar, const float* taus_full, float* fraction_loss,
                                float* grad_taus, a0_stream_t stream) {
  int rc = a0_check_common(c, "a0_loss_quantile");
  if (rc) return rc;
  A0_REQUIRE(layout == 0 || layout == 1, "a0_loss_quantile: layout must be 0 ([B,A,N]) or 1 ([B,N,A])");
  A0_REQUIRE(q && qt && grad, "a0_loss_quantile: NULL tensor");
  A0_REQUIRE(Ni >= 1 && Ni <= A0_MAX_QUANTILES && Nj >= 1 && Nj <= A0_MAX_QUANTILES,
             "a0_loss_quantile: Ni=%d Nj=%d outside [1,%d]", Ni, Nj, A0_MAX_QUANTILES);
  A0_REQUIRE(layout == 0 || taus, "a0_loss_quantile: layout 1 needs per-sample taus");
  A0_REQUIRE(layout == 0 || qsel, "a0_loss_quantile: layout 1 (IQN/FQF) needs qsel (head.qval)");
  if (q_bar) {
    A0_REQUIRE(layout == 1 && Ni == Nj && Nj >= 2 && taus_full, "a0_loss_quantile: fraction term needs layout 1, Ni == Nj >= 2 and taus_full");
  }
  if (c->B == 0) return A0_OK;
  int threads = Ni > Nj ? Ni : Nj;
  threads = ((threads + 31) / 32) * 32;
  if (!q_bar && Ni > 64 && Nj > 64 && a0_option_qh_sorted() == 2) { // measured alternative: one warp per sample (7.4 us against 6.9)
    A0_LAUNCH(a0_k4_quantile_warp, (unsigned)c->B, 32, 0, (cudaStream_t)stream, 1, A0_PDL_K4, a0_unpack(c), layout, q, qt, taus, qsel,
              Ni, Nj, grad);
    return A0_OK;
  }
  if (!q_bar && Ni > 64 && Nj > 64 && a0_option_qh_sorted() == 1) { // QR-sized: O(N log N) sorted-target form, one CTA per sample
    if (qsel && c->A <= 4 && a0_option_qh_spec())
      A0_LAUNCH((a0_k4_quantile_sorted<true, 4>), (unsigned)c->B, (unsigned)threads, 0, (cudaStream_t)stream, 1, A0_PDL_K4, a0_unpack(c), layout, q, qt,
                taus, qsel, Ni, Nj, grad);
    else if (qsel && c->A <= QH_SPEC_A && a0_option_qh_spec())
      A0_LAUNCH((a0_k4_quantile_sorted<true, QH_SPEC_A>), (unsigned)c->B, (unsigned)threads, 0, (cudaStream_t)stream, 1, A0_PDL_K4, a0_unpack(c), layout, q, qt,
                taus, qsel, Ni, Nj, grad);
    else
      A0_LAUNCH((a0_k4_quantile_sorted<false, 1>), (unsigned)c->B, (unsigned)threads, 0, (cudaStream_t)stream, 1, A0_PDL_K4, a0_unpack(c), layout, q, qt,
                taus, qsel, Ni, Nj, grad);
    return A0_OK;
  }
  if (layout == 1 && qsel && c->A <= QH_SPEC_A && threads <= 64 && a0_option_qh_spec())
    A0_LAUNCH(a0_k4_quantile<true>, (unsigned)c->B, (unsigned)threads, 0, (cudaStream_t)stream, 1, A0_PDL_K4, a0_unpack(c), layout, q, qt,
              taus, qsel, Ni, Nj, grad, q_bar, taus_full, fraction_loss, grad_taus);
  else
    A0_LAUNCH(a0_k4_quantile<false>, (unsigned)c->B, (unsigned)threads, 0, (cudaStream_t)stream, 1, A0_PDL_K4, a0_unpack(c), layout, q, qt,
              taus, qsel, Ni, Nj, grad, q_bar, taus_full, fraction_loss, grad_taus);
  return A0_OK;
}

// ------------------------------------------------------------------------------------------------
// K5: batched epsilon-greedy action selection for the actors that feed the shard (SURVEY 8f item 4).
// Replaces Actor.act's tail (agent0/deepq/agent.py:30-39): qt.max(dim=-1), .cpu() of the arg-max,
// np.where(rand > epsilon, greedy, random) and qt_max.mean().item() -- two host syncs per env step --
// with one launch whose results (E actions + the mean of the per-env max) are read back in one copy.
// The random draws stay the caller's (the reference takes them from numpy's global generator in
// the order randint, rand), so a seeded run picks the same actions.  One warp per env, lane = action.
// ------------------------------------------------------------------------------------------------
constexpr int K5_WARPS = 4;
__global__ void __launch_bounds__(K5_WARPS * 32)
a0_k5_act(const float* __restrict__ q, int32_t E, int32_t A, double epsilon, const double* __restrict__ u,
          const int64_t* __restrict__ action_random, int64_t* __restrict__ action_out, float* __restrict__ qmax_out,
          unsigned int* __restrict__ ticket, float* __restrict__ qmax_mean) {
  __shared__ bool is_last;
  __shared__ float red[K5_WARPS];
  A0_PDL_PROLOGUE();
  const int lane = threadIdx.x & 31;
  const int e = blockIdx.x * K5_WARPS + (threadIdx.x >> 5);
  if (e < E) {
    const float v = lane < A ? q[(size_t)e * A + lane] : -INFINITY;
    const int arg = a0_warp_argmax(v, lane);
    if (lane == 0) {
      action_out[e] = (u[e] > epsilon) ? (int64_t)arg : action_random[e];
      if (qmax_out) qmax_out[e] = q[(size_t)e * A + arg];
    }
  }
  // The last CTA to finish computes mean_e q[e, a*_e] in a fixed order (thread-strided partial sums,
  // shuffle tree, warps in order), so the result does not depend on scheduling; it then re-arms the ticket.
  // a*_e is found again by the scan form of the same rule, so each term is the value qmax_out holds (a NaN row
  // makes the mean NaN, as qt_max.mean() does).
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!is_last) return;
  float s = 0.0f;
  for (int i = threadIdx.x; i < E; i += K5_WARPS * 32) {
    float m = -INFINITY;
    for (int a2 = 0; a2 < A; ++a2) {
      const float v = q[(size_t)i * A + a2];
      if (a0_argmax_takes(v, m)) m = v;
    }
    s += m;
  }
  s = a0_warp_sum(s);
  if (lane == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.0f;
#pragma unroll
    for (int w = 0; w < K5_WARPS; ++w) t += red[w];
    *qmax_mean = __fdiv_rn(t, (float)E);
    *ticket = 0u;
  }
}

extern "C" int a0_act_epsilon_greedy(const float* q, int32_t E, int32_t A, double epsilon, const double* u,
                                     const int64_t* action_random, int64_t* action_out, float* qmax_out,
                                     float* scratch, float* qmax_mean, a0_stream_t stream) {
  A0_REQUIRE(E >= 0, "a0_act_epsilon_greedy: negative env count");
  A0_REQUIRE(A >= 1 && A <= A0_MAX_ACTIONS, "a0_act_epsilon_greedy: action_dim %d outside [1,%d]", A, A0_MAX_ACTIONS);
  if (E == 0) return A0_OK;
  A0_REQUIRE(q && u && action_random && action_out && scratch && qmax_mean, "a0_act_epsilon_greedy: NULL argument");
  A0_LAUNCH(a0_k5_act, (unsigned)((E + K5_WARPS - 1) / K5_WARPS), K5_WARPS * 32, 0, (cudaStream_t)stream, 1, A0_PDL_K4, q, E, A, epsilon,
            u, action_random, action_out, qmax_out, reinterpret_cast<unsigned int*>(scratch), qmax_mean);
  return A0_OK;
}

// u8 -> f32 of the actors' observations with the same three normalisations as a0_rb_gather_f32
// (agent.py:27: torch.from_numpy(obs).to(device).float().div(255.0)); 16 pixels per thread.
__global__ void __launch_bounds__(256) a0_k5_u8_to_f32(const uint4* __restrict__ in, float4* __restrict__ out, int64_t nvec,
                                                       int norm_mode) {
  A0_PDL_PROLOGUE();
  const float r = 1.0f / 255.0f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    const uint4 px = __ldg(in + i);
    const uint32_t w[4] = {px.x, px.y, px.z, px.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float f[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float x = __uint_as_float(0x4B000000u | ((w[k] >> (8 * j)) & 0xffu)) - 8388608.0f;
        float y = x;
        if (norm_mode != 2) {
          const float qv = __fmul_rn(x, r);
          y = norm_mode == 1 ? qv : __fmaf_rn(__fmaf_rn(-qv, 255.0f, x), r, qv);
        }
        f[j] = y;
      }
      out[i * 4 + k] = make_float4(f[0], f[1], f[2], f[3]);
    }
  }
}

extern "C" int a0_u8_to_f32(const uint8_t* in, float* out, int64_t count, int32_t norm_mode, a0_stream_t stream) {
  A0_REQUIRE(count >= 0 && count % 16 == 0, "a0_u8_to_f32: count %lld must be a non-negative multiple of 16", (long long)count);
  if (count == 0) return A0_OK;
  A0_REQUIRE(in && out, "a0_u8_to_f32: NULL argument");
  A0_REQUIRE((((uintptr_t)in | (uintptr_t)out) & 15) == 0, "a0_u8_to_f32: pointers must be 16-byte aligned");
  A0_REQUIRE(norm_mode >= 0 && norm_mode <= 2, "a0_u8_to_f32: norm_mode %d outside [0,2]", norm_mode);
  const int64_t nvec = count / 16;
  const unsigned blocks = (unsigned)((nvec + 255) / 256 < 148 * 8 ? (nvec + 255) / 256 : 148 * 8);
  A0_LAUNCH(a0_k5_u8_to_f32, blocks, 256, 0, (cudaStream_t)stream, 1, A0_PDL_K4, reinterpret_cast<const uint4*>(in),
            reinterpret_cast<float4*>(out), nvec, (int)norm_mode);
  return A0_OK;
}
