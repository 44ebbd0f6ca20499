/*
 * agent0_b200 -- C ABI of the B200-native replay-and-target path for zhoubin-me/agent0's deepq.
 *
 * Every entry point is `extern "C"`, takes plain pointers and sizes (no torch types), launches on
 * the caller's CUDA stream, never synchronises and never allocates on the hot path.  Return value:
 * 0 on success, a positive cudaError_t on a CUDA failure, a negative A0_E* code on a bad argument;
 * a0_last_error() gives the message of the calling thread's last failure.
 *
 * All `const T* x /\* dev *\/` arguments are DEVICE pointers; batch outputs are caller-allocated.
 * The ring, the records and the sum-tree are owned by the handle (cudaMalloc once, in a0_rb_create).
 *
 * Reference interfaces replaced (paths relative to the reference repo):
 *   agent0/deepq/replay.py:15-27   ReplayDataset.__init__          -> a0_rb_create / a0_rb_destroy
 *   agent0/deepq/replay.py:45-53   ReplayDataset.extend            -> a0_ex_extend (the reference's lz4 entries,
 *                                                                     decoded and de-duplicated on the device),
 *                                                                     a0_ix_plan + a0_rb_ingest_plan
 *                                                                     (= a0_pt_mark + a0_rb_append), or
 *                                                                     a0_rb_ingest_steps for 1-step actors
 *   agent0/deepq/replay.py:39-43   ReplayDataset.__iter__ (draw)   -> a0_pt_sample
 *   agent0/deepq/replay.py:32-37   ReplayDataset.__getitem__ + default_collate, and
 *   agent0/deepq/agent.py:64-73    Actor.sample's n-step tracker   -> a0_rb_gather
 *   agent0/deepq/agent.py:129-135  BaseLearner.train: /255 + split -> a0_rb_gather_f32
 *   agent0/deepq/trainer.py:91-94  IS weights in Trainer.step      -> a0_pt_sample (epilogue)
 *   agent0/deepq/replay.py:55-59   ReplayDataset.update_priority   -> a0_pt_update
 *   agent0/deepq/agent.py:163-169  BaseLearner.train: loss/indices .cpu() -> a0_pt_update_report
 *   agent0/deepq/agent.py:173-190  DQNLearner.train_step           -> a0_loss_dqn
 *   agent0/deepq/agent.py:194-215  MDQNLearner.train_step          -> a0_loss_mdqn
 *   agent0/deepq/agent.py:219-269  C51Learner.train_step           -> a0_loss_c51
 *   agent0/deepq/agent.py:110-114,273-327 huber_qr_loss, QR/IQN    -> a0_loss_quantile
 *   agent0/deepq/agent.py:340-388  FQFLearner.train_step           -> a0_loss_quantile (+fraction)
 *   agent0/deepq/agent.py:25-39    Actor.act (actor side, "next")  -> a0_u8_to_f32 + a0_act_epsilon_greedy
 */
#ifndef AGENT0_B200_H
#define AGENT0_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct a0_replay a0_replay_t;    /* opaque shard handle (device state) */
typedef struct a0_index a0_index_t;      /* opaque ring index (host state, no CUDA calls) */
typedef void* a0_stream_t;               /* cudaStream_t */

#define A0_OK 0
#define A0_EINVAL (-1)
#define A0_ENOMEM (-2)
#define A0_EFAULT (-3)      /* a kernel of an EARLIER call on this handle gave up (see A0_OPT_MAIL_TIMEOUT_US) */
#define A0_STACK 4          /* frames per observation stack (FrameStack(4), atari_wrappers.py:62) */
#define A0_SLOTS 8          /* obs stack + next-obs stack */
#define A0_MAX_NSTEP 16
#define A0_MAX_ACTIONS 32
#define A0_MAX_QUANTILES 256
#define A0_REC_META_I32 14  /* int32 words per appended record, see a0_rb_append */

int a0_version(void);
const char* a0_last_error(void);
/* A0_OPT_PDL: mask of kernel classes launched with programmatic stream serialization (1 = K4
 * target/loss kernels, 2 = K2 sum-tree, 4 = K3 gather, 8 = K1 append; default 1, A0_PDL=<mask> in
 * the environment overrides).  Every kernel waits for its predecessor with griddepcontrol.wait
 * first, so stream-order semantics are unchanged; what overlaps is launch latency.             */
#define A0_OPT_PDL 1
/* A0_OPT_K2B_LEVELS (3 or 4, default 3; A0_K2B_LEVELS in the environment): tree levels a priority
 * update climbs per barrier phase (8 or 16 siblings loaded per index).  Same tree either way.   */
#define A0_OPT_K2B_LEVELS 2
/* A0_OPT_K2B_BULK_MIN (default 2048; A0_K2B_BULK_MIN in the environment): sum-tree writes of at
 * least this many indices -- and at least 4 per 4096-leaf chunk of the tree -- write the leaves in
 * one cluster launch and rebuild the touched chunks on all SMs in a second one, instead of the
 * single-cluster path climb.  Same tree either way.                                              */
#define A0_OPT_K2B_BULK_MIN 3
/* A0_OPT_FUSED_INGEST (default 1; A0_FUSED_INGEST in the environment): a step-sized ingest (at most
 * 2048 marks and 2048 new frames) applies its marks and its append in ONE launch instead of
 * a0_pt_mark followed by a0_rb_append.  Same shard state either way.                              */
#define A0_OPT_FUSED_INGEST 4
/* A0_OPT_C51_FAST (default 1; A0_C51_FAST in the environment): a0_loss_c51 with qsel given, at most 6
 * actions, at most 64 atoms and a finite, nonzero fl32(vmax - vmin) / (M - 1) runs the
 * short-dependent-chain kernel; 0 forces the general kernel.
 * Bit-identical outputs.                                                                         */
#define A0_OPT_C51_FAST 5
/* A0_OPT_K3_L2 (A0_K3_L2 in the environment): L2 eviction hints of the default gather's bulk copies.
 * 0..3: bit 0 = frame reads marked evict_first, bit 1 = output stores marked evict_first;
 * 4 (default) = both while one launch moves less than 100 MB (it then leaves the sum-tree, the
 * records and the learner's tensors in L2), none for larger launches.  Results do not change.    */
#define A0_OPT_K3_L2 6
/* A0_OPT_K2B_SMALL (default 0; A0_K2B_SMALL in the environment): sum-tree writes of at most 1024
 * indices run as one CTA that keeps the recomputed nodes in a shared-memory hash map.  A measured
 * alternative that lost (shared-memory CAS throughput); same tree either way.                     */
#define A0_OPT_K2B_SMALL 7
/* A0_OPT_K2B_CHUNKS (default 1; A0_K2B_CHUNKS in the environment): sum-tree writes of up to 16 384
 * indices (A0_K2B_CHUNK_MAX in the environment) on trees of up to 2 M leaves run as ONE launch with one CTA
 * per 4096-leaf chunk (each scans the index list once, remembers its own entries, recomputes its chunk -- or
 * only the updated paths, A0_OPT_K2B_SPARSE -- in shared memory; the last CTA finishes the top levels); 0
 * falls back to the cluster schedules selected by A0_OPT_K2B_BULK_MIN.  Same tree either way.       */
#define A0_OPT_K2B_CHUNKS 8
/* A0_OPT_K2B_SPARSE (0..32, default 32; A0_K2B_SPARSE in the environment): a chunk CTA of the schedule above whose
 * chunk holds at most this many updated leaves climbs each updated path on its own (12 adds per path, the inner
 * siblings fetched from the tree in one round trip) instead of recomputing all 4095 inner nodes of the chunk in
 * shared memory; 0 = always recompute the whole chunk.  Same tree either way (node == fl32(left + right)).     */
#define A0_OPT_K2B_SPARSE 12
/* A0_OPT_K2A_ROUNDS (default 0; A0_K2A_ROUNDS in the environment): a sampler launch with more CTAs than the device
 * holds at once (20 x 512 draws: 1280 CTAs on 1184 slots) runs two or more 8-draw units per CTA so that the whole
 * grid -- and with it the gather launched under it -- is resident from the start.  Same draws and weights; a
 * measured alternative that did not shorten the batch-512 step.                                          */
#define A0_OPT_K2A_ROUNDS 13
/* A0_OPT_QH_SORTED (default 1; A0_QH_SORTED in the environment): a0_loss_quantile with more than 64 target
 * and more than 64 online quantiles and no FQF fraction term (QR-200) evaluates the pair sums in
 * O(N log N) from the sorted targets (float64 prefix sums): 1 = one CTA per sample, merge sort in shared
 * memory; 2 = one warp per sample, the targets sorted in registers (measured alternative: fewer instructions,
 * longer chain, slower at batch 512); 0 forces the O(N^2) pair loop.  All
 * agree to ~1e-6 relative (different summation order), within the 1e-5 contract.                      */
#define A0_OPT_QH_SORTED 10
/* A0_OPT_QH_SPEC (default 1; A0_QH_SPEC in the environment): a0_loss_quantile with qsel given and at most 8
 * actions fetches every action's quantiles and the selection values in one batch of loads and selects in
 * registers (the sorted form, and the pair loop of IQN / FQF with at most 64 quantiles); 0 selects the
 * action first and then fetches its row.  Bit-identical outputs.                                          */
#define A0_OPT_QH_SPEC 14
/* A0_OPT_K6_GLOBAL (default 0; A0_K6_GLOBAL in the environment): the LZ4 decode of a0_ex_extend / a0_ex_decode
 * writes its output in place in the scratch buffer (matches read back through L1/L2) instead of staging the
 * entry in shared memory: no shared memory, so every entry of a call is resident at once.  Same bytes, hashes
 * and status codes.                                                                                    */
#define A0_OPT_K6_GLOBAL 11
/* A0_OPT_MAIL_TIMEOUT_US (default 2 000 000; A0_MAIL_TIMEOUT_US in the environment): how long a gather CTA of
 * a0_rb_sample_gather polls its mailbox word before it gives up.  The paired sampler posts every word
 * within microseconds; a CTA that still has nothing after this long was launched without its sampler
 * (a failed launch, a mis-paired caller), sets the handle's fault word and exits instead of spinning
 * forever.  The next a0_rb_sample_gather / a0_rb_gather / a0_pt_sample / a0_pt_update on the handle
 * returns A0_EFAULT (and clears the word).                                                          */
#define A0_OPT_MAIL_TIMEOUT_US 9
int a0_set_option(int32_t option, int64_t value);
/* Reads an option back (A0_OPT_PDL only: a caller that launches ONE kernel without the programmatic attribute --
 * the K4 that joins a gather wave from another stream -- restores the mask it found).                     */
int a0_get_option(int32_t option, int64_t* value);

/* ---- shard lifetime -------------------------------------------------------------------------
 * rec_capacity   transitions kept (cfg.replay.size); indices returned by a0_pt_sample are record
 *                ring positions in [0, rec_capacity)
 * frame_capacity 84x84 frames kept in the HBM frame ring (>= rec_capacity + slack)
 * frame_bytes    bytes per frame, a multiple of 16 (84*84 = 7056 = 441*16)                    */
int a0_rb_create(a0_replay_t** out, int64_t rec_capacity, int64_t frame_capacity,
                 int32_t frame_bytes, int32_t device);
int a0_rb_destroy(a0_replay_t* h);
/* zero the tree, max_p = 1 (ReplayDataset.__init__: priority state, replay.py:19-27) */
int a0_rb_reset(a0_replay_t* h, a0_stream_t stream);

/* device pointers to handle-owned state (tests, checkpointing, zero-copy views) */
enum { A0_PTR_FRAMES = 0, A0_PTR_REC_SLOTS = 1, A0_PTR_REC_INFO = 2, A0_PTR_TREE = 3,
       A0_PTR_MAX_P = 4 };
void* a0_rb_ptr(a0_replay_t* h, int32_t which);
int64_t a0_rb_tree_leaves(a0_replay_t* h);      /* P = next_pow2(rec_capacity) */

/* ---- K1: append ---------------------------------------------------------------------------------
 * Copies n_new staged frames into the ring with coalesced 16-byte stores and scatters m records.
 * new_frames    [n_new][frame_bytes]  staged frames (device)
 * new_frame_pos [n_new]               destination frame-ring positions
 * rec_meta      [m][14] int32   {pos, link_from, link_to, action_done, slot[8], reward_lo, reward_hi}
 *                 pos         record ring position to write
 *                 link_from   position of the previous record of the same stream, written by an
 *                             EARLIER append, whose successor link must now point at `pos` (-1: none)
 *                 link_to     position of the next record of the same stream when it is part of
 *                             this same append (-1: not known yet)
 *                 action_done action | done << 31
 *                 slot[0..3]  frame positions of the observation stack, slot[4..7] of the next one
 *                 reward      float64 bit pattern (the reference keeps rewards in float64)       */
int a0_rb_append(a0_replay_t* h, const uint8_t* new_frames /* dev */,
                 const int32_t* new_frame_pos /* dev */, int32_t n_new,
                 const int32_t* rec_meta /* dev */, int32_t m, a0_stream_t stream);

/* ---- host ring index ------------------------------------------------------------------------------
 * Pure host code (usable without a GPU).  Decides, for every appended transition, where its new
 * frames go, which records become sampleable and which must be evicted because their slot or
 * their frames are about to be overwritten; the device only executes the plan.  Replaces the
 * bookkeeping of ReplayDataset.extend (replay.py:45-53) and the "entry k-n+1 is emitted at step k"
 * rule of the actor's n-step tracker (agent.py:64-73).
 * n_step: records gathered per sample (1 when the caller appends already-folded reference entries).
 * age_limit: frames older than this are never referenced by a new record (< 0: default).        */
int a0_ix_create(a0_index_t** out, int64_t rec_capacity, int64_t frame_capacity, int32_t n_step,
                 int64_t age_limit);
int a0_ix_destroy(a0_index_t* ix);
enum { A0_IX_HEAD_Q = 0, A0_IX_TAIL_Q = 1, A0_IX_HEAD_FS = 2, A0_IX_TOP = 3, A0_IX_REC_CAPACITY = 4,
       A0_IX_FRAME_CAPACITY = 5, A0_IX_NSTEP = 6, A0_IX_AGE_LIMIT = 7, A0_IX_MAX_CHUNK = 8,
       A0_IX_STATE_WORDS = 9 };
int a0_ix_state(a0_index_t* ix, int64_t* out /* [A0_IX_STATE_WORDS] */);
const uint8_t* a0_ix_sampleable(a0_index_t* ix);          /* host u8[rec_capacity], 1 = sampleable */
/* current observation stack of a stream, as frame sequence numbers */
int a0_ix_set_stack(a0_index_t* ix, int64_t stream, const int64_t* seq4);
int a0_ix_get_stack(a0_index_t* ix, int64_t stream, int64_t* seq4);   /* returns 1 if none yet */
/* Structural description of m transitions: the observation of transition i is its stream's
 * current stack, the next observation that stack shifted by n_new[i] (0..4) new frames; new
 * frames are numbered from head_fs in (transition, frame) order.  fs8_out i64[m][8].            */
int a0_ix_resolve_shift(a0_index_t* ix, const int64_t* stream, const int64_t* n_new, int32_t m,
                        int64_t* fs8_out);
typedef struct {
  int32_t m, n_new, n_marks;
  const int32_t* new_frame_pos;   /* [n_new]  frame-ring positions of the new frames            */
  const int32_t* rec_meta;        /* [m][14]  a0_rb_append layout                               */
  const int32_t* marks;           /* [n_marks] a0_pt_mark layout: >= 0 sampleable, < 0 ~evicted */
} a0_plan_t;                      /* arrays are owned by the index, valid until its next call   */
/* Commit m transitions whose 8 frame sequence numbers are resolved (fs8 i64[m][8]; the n_new
 * new ones numbered upwards from head_fs).  m must not exceed A0_IX_MAX_CHUNK.                  */
int a0_ix_plan(a0_index_t* ix, const int64_t* stream, const int64_t* fs8, int32_t m, int32_t n_new,
               const int64_t* action, const double* reward, const uint8_t* done, a0_plan_t* out);

/* ---- content de-duplication for the reference-compatible ingest (host code) ------------------------
 * ReplayDataset.extend receives self-contained 8-frame entries concat(st, st_next) (agent.py:78-81).
 * a0_dd_resolve decides which of their frames are new: a frame is matched -- 64-bit hash, then full
 * byte comparison, so a match is always bit-exact -- against the 8 frames of the stream's previous
 * entry (if still resident and younger than the index's age limit) and the earlier frames of its
 * own entry.  frames: host u8[m][8][frame_bytes]; fs8_out i64[m][8] frame sequence numbers (new
 * ones numbered upwards from the index's head_fs) for a0_ix_plan; new_src_out i64[<= 8m] flat
 * indices t*8+j of the new frames in allocation order (a0_rb_ingest_plan's new_frame_src).       */
typedef struct a0_dedupe a0_dedupe_t;
int a0_dd_create(a0_dedupe_t** out, int32_t frame_bytes);
int a0_dd_destroy(a0_dedupe_t* dd);
int a0_dd_resolve(a0_dedupe_t* dd, a0_index_t* ix, const int64_t* stream, const uint8_t* frames,
                  int32_t m, int64_t* fs8_out, int64_t* new_src_out, int32_t* n_new_out);

/* ---- K6: ReplayDataset.extend with the entries still compressed (agent0/deepq/replay.py:45-53) --------
 * The reference actor ships every transition as (lz4.block.compress(concat(st, st_next)), a, r, d)
 * (agent0/deepq/agent.py:78-81): a python-lz4 block = 4-byte little-endian decoded size + one raw LZ4
 * block of 8 frames.  a0_ex_extend takes m such entries exactly as they arrive -- `blobs` is their
 * concatenation in host memory, blob_len[i] the length of entry i (an entry of exactly 8*frame_bytes is
 * taken as uncompressed) -- copies only the COMPRESSED bytes to the device, decodes them there (one warp
 * per entry, output staged in shared memory), labels every frame with the first byte-identical frame of
 * its stream's previous entry / its own entry (hash gate + full compare, so a match is always
 * bit-exact), reads 8 label bytes per entry back, resolves them against the ring index on the host
 * (a0_ex_resolve: the decisions of a0_dd_resolve) and appends the new frames straight from the decoded
 * scratch (K2b marks + K1).  stream[i] = the actor env entry i comes from (entry order inside a stream is
 * its time order); action / reward / done as a0_ix_plan.  The index must have been created with
 * n_step = 1: reference entries are already n-step folded.  Synchronises `cuda_stream` once per 2048
 * entries (the labels); the appends themselves are stream-ordered.  A malformed block fails the call
 * with A0_EINVAL before anything of its batch is committed.
 * a0_ex_create: h may be NULL for host-only use of a0_ex_resolve (tests of the rule without a GPU).   */
typedef struct a0_extend a0_extend_t;
int a0_ex_create(a0_extend_t** out, a0_replay_t* h, a0_index_t* ix);
int a0_ex_destroy(a0_extend_t* ex);
int a0_ex_extend(a0_extend_t* ex, const uint8_t* blobs /* host */, const int64_t* blob_len /* host [m] */,
                 const int64_t* stream, const int64_t* action, const double* reward, const uint8_t* done,
                 int32_t m, float alpha, a0_stream_t cuda_stream);
/* The same call with the entries where they lie: blob_ptr[i] points at entry i (e.g. the bytes objects of the
 * reference's list), so the only copy on the host is the one into the page-locked staging block.        */
int a0_ex_extend_v(a0_extend_t* ex, const uint8_t* const* blob_ptr /* host [m] */,
                   const int64_t* blob_len /* host [m] */, const int64_t* stream, const int64_t* action,
                   const double* reward, const uint8_t* done, int32_t m, float alpha,
                   a0_stream_t cuda_stream);
/* The decode kernel alone: frames_out dev u8[m][8][frame_bytes], status_out host i32[m] (0 = ok,
 * 1 bad size prefix, 2 truncated input, 3 output overrun, 4 bad match offset, 5 short output).      */
int a0_ex_decode(a0_extend_t* ex, const uint8_t* blobs /* host */, const int64_t* blob_len /* host [m] */,
                 int32_t m, uint8_t* frames_out /* dev */, int32_t* status_out /* host */,
                 a0_stream_t cuda_stream);
/* Host rule: labels u8[m][8] (0..7 = identical to that frame of the stream's previous entry, 8+c =
 * identical to frame c <= j of its own entry; always the FIRST identical candidate in that order)
 * -> fs8_out / new_src_out / n_new_out exactly as a0_dd_resolve produces them from the bytes.        */
int a0_ex_resolve(a0_extend_t* ex, const int64_t* stream, const uint8_t* labels, int32_t m,
                  int64_t* fs8_out, int64_t* new_src_out, int32_t* n_new_out);
/* microseconds of the last a0_ex_extend / a0_ex_decode call: {host staging, wait for decode + label,
 * host resolve + plan, append launches, device time of decode + label (CUDA events), entries}       */
int a0_ex_last_timing(a0_extend_t* ex, float* out6);

/* ---- K7: LZ4 encode of 8-frame groups on the device ---------------------------------------------------
 * frames dev u8[m][8][frame_bytes] (16-byte aligned); group g becomes one python-lz4 block (4-byte little-endian
 * decoded size + one raw LZ4 block, no dictionary shared across groups) at out + g * A0_LZ4_STRIDE(frame_bytes),
 * or the 8 * frame_bytes input bytes themselves when that block would not be shorter (K6a takes a blob of exactly
 * the decoded size as uncompressed).  out_len dev i32[m]: blob lengths; frame_hash dev u64[m][8]: the 64-bit content
 * hash K6a computes for each decoded frame.  The parse is the greedy one defined by oracle/lz4_encode.py
 * (encode_greedy), byte for byte: one warp per group, the group in shared memory.                              */
#define A0_LZ4_STRIDE(frame_bytes) \
  ((((int64_t)8 * (frame_bytes) + (int64_t)8 * (frame_bytes) / 255 + 20) + 15) / 16 * 16)
int a0_lz4_encode(const uint8_t* frames /* dev */, int32_t m, int32_t frame_bytes, uint8_t* out /* dev */,
                  int32_t* out_len /* dev */, uint64_t* frame_hash /* dev */, a0_stream_t stream);

/* ---- checkpoint: one shard (+ its ring index and reference-ingest state) to a file and back ---------------
 * a0_ix_serialize writes the ring index's whole state (head_q, tail_q, head_fs, top, fs_at_append, sampleable,
 * per stream last_pos / last_seq / pending / stack / has_stack, the stale set) into out[cap]; *len_out receives
 * the length (also when out is NULL or cap is too small, which then fails with A0_EINVAL).  a0_ix_deserialize
 * replaces the state of an index created with the same capacities, n_step and age limit; a blob that is
 * truncated, inconsistent or made for other parameters is rejected with A0_EINVAL and the index is unchanged.
 * Host code only.                                                                                          */
int a0_ix_serialize(a0_index_t* ix, uint8_t* out, int64_t cap, int64_t* len_out);
int a0_ix_deserialize(a0_index_t* ix, const uint8_t* blob, int64_t len);
/* a0_ckpt_save synchronises `stream`, refuses during a CUDA-graph capture and on a shard whose fault word is set,
 * and writes the shard h, its index ix and (ex != NULL) the stream tails of the reference-tuple ingest to `path`
 * (through path + ".tmp", renamed when complete), with `user` (user_len bytes) stored alongside.  Frames leave as
 * K7 blobs.  File format (little-endian; section hash: the 64-bit streaming hash of a0_ckpt.cu):
 *   header   "A0CKPT01" magic (8 B), version u32 (= 1), 0 u32, N i64, NF i64, F i64, P i64, n_step i64, age_limit i64
 *   sections {tag u32, 0 u32, length u64, hash u64 of the payload} + payload, in this order:
 *   INDEX    (1) a0_ix_serialize
 *   RECORDS  (2) rec_slots i32[N][8], then rec_info {reward f64, action|done<<31 i32, link i32}[N]
 *   LEAVES   (3) f32[N] tree leaves (the inner nodes are rebuilt on load: node = fl32(left + right))
 *   SCALARS  (4) max_p f32, dyn {top, beta, sum_offset} f32[3], sampler call counter u64, stride_hint i64
 *   TAILS    (5) count i64, then per stream {id i64, seq i64[8], cls u8[8], frames u8[8][F], hash u64[8]}
 *   USER     (6) the caller's bytes
 *   FRAMES   (7) lo i64 (first frame seq: max(0, head_fs - NF)), frames i64 (head_fs - lo), groups i64, then
 *                {first ring position i64, blob length i64}[groups] and the frame hashes u64[groups][8].  Group g
 *                holds seqs lo + 8g .. lo + 8g + 7 (the last group padded with zero frames)
 *   BLOBS    (8) the groups' K7 blobs, back to back
 * a0_ckpt_load reads such a file into an existing shard + index (+ ex, or NULL) of the same N, NF, F, n_step and
 * age limit, into the buffers they already own (CUDA graphs captured on the shard stay valid).  It validates
 * everything it can before touching the shard (header, section hashes, index invariants, finite non-negative
 * leaves that are 0 where a record is not sampleable, slots and links of live records, the group table); a file
 * that fails there leaves shard and index unchanged.  Frames are then decoded by K6a into the ring and every
 * frame's hash is compared with the saved one; a failure from there on leaves shard, index and tails as freshly
 * created.  Both return A0_EINVAL with a message for a bad file.  user_out[user_cap] receives the USER bytes and
 * *user_len_out their length (NULLs allowed).                                                              */
int a0_ckpt_save(a0_replay_t* h, a0_index_t* ix, a0_extend_t* ex, const char* path, const uint8_t* user,
                 int64_t user_len, a0_stream_t stream);
int a0_ckpt_load(a0_replay_t* h, a0_index_t* ix, a0_extend_t* ex, const char* path, uint8_t* user_out,
                 int64_t user_cap, int64_t* user_len_out, a0_stream_t stream);
/* Phases of the last a0_ckpt_save / a0_ckpt_load / a0_ckpt_merge of the process.  Save: {total us, K7 device us
 * (CUDA events), blob compaction + device-to-host copy device us (CUDA events), file write us, raw frame bytes, blob
 * bytes, host wait for the copies us, 0}.  Load: {total us, header + small sections + validation us, blob file read
 * us, decode + hash check + restore us (host clock, K6a included), raw frame bytes, blob bytes, 0, 0}.  Merge: {total
 * us, header + small sections + validation us of all files, host merge plan (a0_ix_merge) us, decode + place device
 * us (CUDA events around K6a and K1), records + leaves + scalars + tails us, bytes decoded, bytes placed, blob file
 * read + hash us}.                                                                                               */
int a0_ckpt_last_timing(double* out8);

/* ---- merging shard checkpoints into a shard of another capacity or world size ----------------------------------
 * a0_ix_merge (host code only) fills the EMPTY index `target` (any record capacity, frame capacity and age limit;
 * the same n_step) from k checkpoint files, given each file's index (a0_ix_deserialize of its INDEX section), its
 * RECORDS and LEAVES sections and, optionally, its TAILS ids and seq[8] (tail_count[k], tail_ids and tail_seq[][8]
 * concatenated over the files; tail_count NULL = none).  The rule (specification: agent0_b200/ring_index.py, merge):
 *   1. from each file the live records of the kept streams; a record's stream is found by walking the link words
 *      backwards from the stream's last record;
 *   2. ages head_q - 1 - q inside each file; all records oldest first, ties by file index;
 *   3. fed to a0_ix_plan in chunks of the target's max_chunk; a frame is (file, source seq) and reuses its newest
 *      target seq t when t is resident and next_fs - t < age_limit, otherwise it takes the next new seq in (record,
 *      slot) order; the target's eviction rule keeps the newest suffix;
 *   4. a record sampleable in the target keeps its source leaf bit for bit; a record stale in its file (live,
 *      neither sampleable nor pending) enters the target's stale set and stays unsampleable;
 *   5. map_len[j] < 0: every stream of file j, id + j * S (S = 1 + the largest id of any file); otherwise the
 *      map_len[j] pairs (map_old, map_new; concatenated over such files) name the streams taken and their new ids.
 *      Two kept streams with one new id fail the call before the target is touched;
 *   6. stacks whose frames are resident in their file are placed after the records (frames-only plans, ascending new
 *      id, the rule of 3); a tail takes the newest target seq of each of its frames and is dropped when one of them is
 *      not resident in the target at the end.
 * records_out receives the target's RECORDS (N'*48 bytes: what K1 writes for the plans on a freshly reset shard),
 * leaves_out f32[N'] its leaves (0 where not sampleable).  *out: arrays owned by the target index until its next
 * merge.  Every target ring slot receives at most one placement, so they may run in any order.                    */
typedef struct {
  int64_t n_place;
  const int64_t* place;           /* [n_place][3] {file, source frame seq, target ring slot}                    */
  int64_t n_rec;
  const int64_t* record_map;      /* [n_rec][3] {file, source position, target position or -1 if evicted}     */
  int64_t n_tail;
  const int64_t* tails;           /* [n_tail][11] {new id, file, TAILS entry, target seq[8]}, ascending new id   */
  int64_t stride_hint;            /* K3's successor stride after the target's records (as the ingest sets it)  */
} a0_merge_t;
int a0_ix_merge(a0_index_t* target, int32_t k, a0_index_t* const* src, const uint8_t* const* records,
                const float* const* leaves, const int64_t* map_old, const int64_t* map_new, const int64_t* map_len,
                const int64_t* tail_count, const int64_t* tail_ids, const int64_t* tail_seq, uint8_t* records_out,
                float* leaves_out, a0_merge_t* out);
/* a0_ckpt_info reads only the header and the INDEX section of a checkpoint: out8 = {N, NF, F, n_step, age_limit,
 * live records, sampleable records, streams}; ids_out[ids_cap] receives the stream ids in ascending order.       */
int a0_ckpt_info(const char* path, int64_t* out8, int64_t* ids_out, int64_t ids_cap);
/* a0_ckpt_merge fills the shard h + index ix (+ ex, or NULL) from k checkpoint files of the same F and n_step by
 * the rule of a0_ix_merge (map_old / map_new / map_len as there).  Every file is validated as a0_ckpt_load
 * validates it before anything is touched; then the shard is reset, records, leaves (inner nodes fl32(left +
 * right)), max_p (the maximum over the files), the sampler's call counter (the maximum), dyn {top, file 0's beta,
 * 0} and the stride hint are written, and the frames are placed file by file: the BLOBS section is read once,
 * hashed whole, and only the groups that hold a placed frame are decoded by K6a (at most 1024 groups at a time,
 * every decoded frame's hash compared with the saved one) and copied to their target slots by K1.  A failure from
 * the reset on leaves shard, index and tails as freshly created.  user_out[user_cap] receives the files' USER
 * bytes back to back, user_len_out[k] their lengths.                                                            */
int a0_ckpt_merge(a0_replay_t* h, a0_index_t* ix, a0_extend_t* ex, const char* const* paths, int32_t k,
                  const int64_t* map_old, const int64_t* map_new, const int64_t* map_len, uint8_t* user_out,
                  int64_t user_cap, int64_t* user_len_out, a0_stream_t stream);

/* ---- staged ingest: execute a plan on the device ------------------------------------------------
 * One pinned H2D copy of {frames, positions, record metadata, marks} from a double-buffered
 * staging area owned by the handle, then a0_pt_mark and a0_rb_append on `stream`.  frames:
 * host u8[*][frame_bytes]; new_frame_src (host, optional) picks the n_new frames to store, in
 * allocation order, out of it (NULL: the first n_new).  Flags: FRAMES_ON_DEVICE = frames is a
 * device pointer (with new_frame_src: K1 reads frames[new_frame_src[j]]; without: allocation order); FRAMES_PINNED = frames is page-locked host memory
 * in allocation order that stays untouched until `stream` has passed this call (it is copied by
 * DMA straight from there, no staging memcpy); COPY_STREAM = the H2D copies are issued on a
 * copy stream owned by the handle and `stream` waits for them, so the DMA overlaps the kernels
 * `stream` is still running (not usable while `stream` is being captured into a CUDA graph).      */
#define A0_INGEST_FRAMES_ON_DEVICE 1
#define A0_INGEST_FRAMES_PINNED 2
#define A0_INGEST_COPY_STREAM 4
int a0_rb_ingest_plan(a0_replay_t* h, const a0_plan_t* plan, const uint8_t* frames,
                      const int64_t* new_frame_src, int32_t flags, float alpha, a0_stream_t stream);
/* a0_ix_resolve_shift + a0_ix_plan + a0_rb_ingest_plan for m 1-step transitions (any m: split
 * into chunks internally); all arrays are host arrays except new_frames under FRAMES_ON_DEVICE. */
int a0_rb_ingest_steps(a0_replay_t* h, a0_index_t* ix, const int64_t* stream, const int64_t* n_new,
                       const uint8_t* new_frames, int32_t flags, const int64_t* action,
                       const double* reward, const uint8_t* done, int32_t m, float alpha,
                       a0_stream_t cuda_stream);
/* The same ingest, which also publishes the sampler's device-resident scalars (a0_rb_set_dynamic:
 * top = sampleable records after this append, beta, sum_offset = compat_sum ? capacity - top : 0)
 * from inside its append launch: no separate launch per Trainer.step for a graph-captured draw.
 * beta is the value ReplayDataset.extend leaves in self.beta (replay.py:53).  m == 0 only publishes. */
int a0_rb_ingest_steps_dyn(a0_replay_t* h, a0_index_t* ix, const int64_t* stream,
                           const int64_t* n_new, const uint8_t* new_frames, int32_t flags,
                           const int64_t* action, const double* reward, const uint8_t* done,
                           int32_t m, float alpha, float beta, int32_t compat_sum,
                           a0_stream_t cuda_stream);

/* ---- K2b: sum-tree leaf writes ---------------------------------------------------------------------
 * a0_pt_mark: pos[k] >= 0 -> leaf = max_p^alpha (a newly sampleable record, replay.py:52);
 *             pos[k] <  0 -> leaf ~pos[k] = 0   (a record whose frames are being overwritten).
 * a0_pt_update: leaf[idx[k]] = (loss[k]+eps)^alpha, max_p = max(max_p, max loss) (replay.py:55-59);
 *             duplicated indices: the last one wins, as in `priority[ids] = ...` on the CPU;
 *             indices whose leaf is currently 0 (evicted since they were sampled) are skipped.
 * a0_pt_set:  leaf[idx[k]] = value[k] (restore / tests).
 * All three recompute every touched ancestor as fl32(left+right), level by level.               */
int a0_pt_mark(a0_replay_t* h, const int32_t* pos /* dev */, int32_t count, float alpha,
               a0_stream_t stream);
int a0_pt_update(a0_replay_t* h, const int64_t* idx /* dev */, const float* loss /* dev */,
                 int32_t count, float alpha, float eps, a0_stream_t stream);
int a0_pt_set(a0_replay_t* h, const int64_t* idx /* dev */, const float* value /* dev */,
              int32_t count, a0_stream_t stream);
/* a0_pt_update that also hands the step's result to the host: idx[k] and loss[k] are stored to
 * idx_report / loss_report by the kernel that reads them anyway.  With report buffers in mapped
 * page-locked host memory (device-visible aliases from a0_host_map) this is the `.cpu()` of
 * BaseLearner.train's return value (agent.py:163-169: q_loss and indices on the CPU) without two
 * device-to-host copies on the stream; the data is valid on the host once an event recorded after
 * the call has completed.  Device memory works too.                                             */
int a0_pt_update_report(a0_replay_t* h, const int64_t* idx /* dev */, const float* loss /* dev */,
                        int32_t count, float alpha, float eps, int64_t* idx_report /* dev-visible */,
                        float* loss_report /* dev-visible */, a0_stream_t stream);
/* a0_pt_update[_report] for the end of a Trainer.step, where the kernel launched immediately before this call on
 * `stream` is the last K4 and idx was written several launches earlier (by the draw): the update is launched
 * programmatically under that kernel, loads its leaves and sorts out duplicates (positions only) while it is
 * still running, and waits for it only where the loss values are first read.  THE CALLER GUARANTEES that idx is
 * not produced by the immediately preceding launch on the stream (loss may be).  Report buffers optional (both
 * or none).  Same tree, same max_p, same reports as a0_pt_update_report.                                  */
int a0_pt_update_overlapped(a0_replay_t* h, const int64_t* idx /* dev */, const float* loss /* dev */,
                            int32_t count, float alpha, float eps, int64_t* idx_report, float* loss_report,
                            a0_stream_t stream);
/* The write-back of a Trainer.step in two halves, for counts up to A0_K2B_PLAN_MAX.  a0_pt_update_plan reads idx and
 * the tree (one CTA; run it any time after the draw) and writes into `plan` (A0_K2B_PLAN_BYTES of device memory owned
 * by the caller) the distinct valid leaves with their winning index (the highest k of each leaf's duplicates), the old
 * leaves, the off-path siblings of every path and where the paths meet.  a0_pt_update_apply (8 CTAs) is launched
 * programmatically under its predecessor on `stream`, like a0_pt_update_overlapped: it reads the plan before it waits
 * and after the wait only the losses.  THE CALLER GUARANTEES that idx and the tree do not change between the two
 * calls, and that the plan and idx were written by launches older than the one immediately preceding the apply.
 * Same tree, same max_p, same reports as a0_pt_update_report / a0_pt_update.  Trees of 2 .. 2^28 leaves.        */
#define A0_K2B_PLAN_MAX 1024
#define A0_K2B_PLAN_BYTES 90176
int a0_pt_update_plan(a0_replay_t* h, const int64_t* idx /* dev */, int32_t count, void* plan /* dev */,
                      a0_stream_t stream);
int a0_pt_update_apply(a0_replay_t* h, const int64_t* idx /* dev */, const float* loss /* dev */, int32_t count,
                       float alpha, float eps, const void* plan /* dev */, int64_t* idx_report, float* loss_report,
                       a0_stream_t stream);
/* Device-visible alias of page-locked host memory (cudaHostAlloc / cudaHostRegister with mapping,
 * torch's pin_memory); fails for pageable memory.  Not a stream operation: call it once per
 * buffer, outside CUDA-graph capture.                                                          */
int a0_host_map(const void* host_ptr, void** dev_ptr_out);

/* ---- K2a: batched stratified prioritized draws + IS weights ------------------------------------------
 * total = k_batches * batch draws; draw j of a batch uses t = ((j + u)/batch) * root and descends
 * the tree (warp-cooperative, five levels per memory round trip).  Epilogue (trainer.py:91-94):
 *   w = (top * p / (root + sum_offset))^(-beta);  w /= max_over_the_batch(w) + 1e-8
 * uniform != 0 writes w = 1 (ReplayEnum.uniform: weights = priorities = 1, trainer.py:95-96).
 * sum_offset reproduces the reference's denominator over never-written slots (SURVEY Q3) when the
 * caller asks for compat mode; 0 otherwise.
 * top < 0: take top, beta and sum_offset from the device-resident values last written by
 * a0_rb_set_dynamic (stream-ordered), so that a captured CUDA graph of the draw stays correct
 * while the shard grows and beta anneals.                                                       */
int a0_rb_set_dynamic(a0_replay_t* h, float top, float beta, float sum_offset, a0_stream_t stream);
int a0_pt_sample(a0_replay_t* h, const float* u /* dev [total] */, int32_t total, int32_t batch,
                 float top, float beta, float sum_offset, int32_t uniform,
                 int64_t* idx_out /* dev [total] */, float* prio_out /* dev [total] */,
                 float* weight_out /* dev [total] */, a0_stream_t stream);

/* The same draw with the sampler's own uniforms (no torch / host RNG, no extra launch): draw g of
 * call c under `seed` uses u = (Philox4x32-10(counter {g, 0, c_lo, c_hi}, key {seed_lo, seed_hi}).x >> 8)
 * * 2^-24.  call >= 0 gives the call number explicitly; call < 0 uses a device-resident counter
 * that the launch itself advances, so every replay of a captured CUDA graph draws fresh batches
 * (a0_rb_reset zeroes it, a0_pt_rng_seek sets it).  u_out (optional, dev [total]) receives the
 * uniforms.                                                                                      */
int a0_pt_sample_rng(a0_replay_t* h, uint64_t seed, int64_t call, int32_t total, int32_t batch,
                     float top, float beta, float sum_offset, int32_t uniform, int64_t* idx_out,
                     float* prio_out, float* weight_out, float* u_out, a0_stream_t stream);
int a0_pt_rng_seek(a0_replay_t* h, uint64_t call, a0_stream_t stream);

/* Batches WITHOUT replacement (K2a-unique): the law of the reference's torch.multinomial(priority[:top], B,
 * replacement=False) (agent0/deepq/replay.py:41-43), no record twice in a batch.  A batch is the first B
 * distinct records of a stream of descents; later rounds descend with the records already taken masked out.
 * Candidate j of batch k in call c under `seed` uses u = ((x0 >> 5) * 2^26 + (x1 >> 6)) * 2^-53 from
 * Philox4x32-10(counter {j, 0x80000000 | k, c_lo, c_hi}, key {seed_lo, seed_hi}); the arithmetic is defined by
 * oracle/sample_unique.py.  Rows are in draw order.  call, top (< 0: device-resident values), uniform and the
 * IS weights as a0_pt_sample_rng; batch <= 1024.  stats_out (optional, dev i32 [total / batch][2]) receives
 * {rounds, candidates drawn} per batch.  A batch with fewer than `batch` records of positive priority fills
 * its remaining rows with its first record and sets device fault code 2, which the next call on the handle
 * that checks faults (this one included) reports as A0_EFAULT.                                           */
int a0_pt_sample_unique(a0_replay_t* h, uint64_t seed, int64_t call, int32_t total, int32_t batch,
                        float top, float beta, float sum_offset, int32_t uniform, int64_t* idx_out,
                        float* prio_out, float* weight_out, int32_t* stats_out, a0_stream_t stream);

/* ---- K3: fused gather ---------------------------------------------------------------------------------
 * For each sampled record position: walk n_step-1 successor links, rebuild the two 4-frame stacks
 * (each distinct frame is read from HBM once and written to every place it appears), and compute
 *   Rn = sum_i gamma^i prod_{j<i}(1-d_j) r_i   in float64, Horner newest->oldest, separately rounded
 *        mul/mul/add (agent.py:65-69), Dn = OR d_i, boot = position of the record that follows the
 *        window (-1 if not appended yet).
 * frames_out [count][8][frame_bytes]: the reference's `frames` layout, concat(st, st_next)
 * (agent.py:80); action i64; reward f64 and f32; done u8 and f32; boot i64.  Any output but
 * frames_out may be NULL.  variant: 0 = TMA bulk copies through a 4-buffer shared-memory ring
 * (default), 1 = LDG/STG through registers, 2 = TMA with all distinct frames staged at once,
 * 3 = TMA, transition split over two CTAs (even/odd distinct frames).                            */
int a0_rb_gather(a0_replay_t* h, const int64_t* idx /* dev */, int32_t count, int32_t n_step,
                 double gamma, uint8_t* frames_out, int64_t* action_out, double* reward64_out,
                 float* reward32_out, uint8_t* done8_out, float* done32_out, int64_t* boot_out,
                 int32_t variant, a0_stream_t stream);

/* a0_pt_sample[_rng] + a0_rb_gather (variant 0) as an overlapped producer/consumer pair: the gather
 * is launched with programmatic stream serialization, becomes resident while the sampler is still
 * descending the tree, and each of its CTAs starts fetching frames as soon as its own draw's record
 * position arrives through a handle-owned mailbox -- the sampler's IS-weight epilogue, its drain and
 * the launch hand-over between the two kernels leave the critical path of a step.  The gather ends
 * with griddepcontrol.wait, so work queued after this call sees both kernels complete.  Same results
 * as the two separate calls.  u != NULL: caller-supplied uniforms (seed, call ignored); u == NULL:
 * the sampler's own Philox stream as a0_pt_sample_rng.  The first call (and any call with a larger
 * total) allocates the mailbox and must not be inside a CUDA-graph capture.                        */
int a0_rb_sample_gather(a0_replay_t* h, const float* u /* dev [total] or NULL */, uint64_t seed,
                        int64_t call, int32_t total, int32_t batch, float top, float beta,
                        float sum_offset, int32_t uniform, int64_t* idx_out, float* prio_out,
                        float* weight_out, int32_t n_step, double gamma, uint8_t* frames_out,
                        int64_t* action_out, double* reward64_out, float* reward32_out,
                        uint8_t* done8_out, float* done32_out, int64_t* boot_out, a0_stream_t stream);

/* The same pair with the gather cut into WAVES -- consecutive ranges of the draw, one launch each -- so that
 * the consumer of the first batches (the K4 launches of Trainer.step's inner loop, trainer.py:82-104, on another
 * stream) starts while the later batches are still being fetched: the reference's DataPrefetcher does the same
 * with its 3-deep queue (utils.py:45-61).
 *   a0_rb_sample_mail   the sampler of a0_rb_sample_gather alone: every draw's record position is posted to the
 *                       handle's mailbox (same arguments and results as a0_pt_sample / a0_pt_sample_rng)
 *   a0_rb_gather_mail   the gather of draws [lo, lo + count) of that sampler call; the output pointers are the
 *                       bases of the WHOLE draw's buffers (this wave writes rows [lo, lo + count)).  Must be queued
 *                       on the sampler's stream, directly after it or after the previous wave, and every draw must
 *                       be covered by exactly one wave before the next a0_rb_sample_mail.
 * window > 0 (the same value for every wave of a draw): ORDERED fetch -- a draw starts its frame traffic only when
 * at most `window` draws beyond the completed ones are in flight, so the first batches complete first (a consumer
 * that needs ~2 us per batch is fed in order) instead of every resident CTA sharing the bandwidth and all batches
 * finishing together; 0: no limit (launches too large to be resident at once are ordered by the hardware anyway).
 * Waves complete in launch order, and a complete wave implies a complete sampler (weights, priorities): an
 * event recorded after wave j is what the consumer of its batches waits for.  Same results as
 * a0_rb_sample_gather.  The first a0_rb_sample_mail (and any with a larger total) allocates the mailbox and must
 * not be inside a CUDA-graph capture.                                                                    */
int a0_rb_sample_mail(a0_replay_t* h, const float* u /* dev [total] or NULL */, uint64_t seed, int64_t call,
                      int32_t total, int32_t batch, float top, float beta, float sum_offset, int32_t uniform,
                      int64_t* idx_out, float* prio_out, float* weight_out, a0_stream_t stream);
int a0_rb_gather_mail(a0_replay_t* h, int32_t lo, int32_t count, int32_t window, int32_t n_step, double gamma,
                      uint8_t* frames_out, int64_t* action_out, double* reward64_out, float* reward32_out,
                      uint8_t* done8_out, float* done32_out, int64_t* boot_out, a0_stream_t stream);

/* TEST HOOK: the gather half of a0_rb_sample_gather launched WITHOUT its sampler -- what a failed sampler
 * launch or a mis-paired caller would leave behind.  Every CTA times out (A0_OPT_MAIL_TIMEOUT_US), the
 * kernel ends, and the next call on the handle returns A0_EFAULT.  Never call it on a production path. */
int a0_rb_gather_unpaired(a0_replay_t* h, int32_t count, uint8_t* frames_out, a0_stream_t stream);
/* A0_EFAULT (once) if a kernel of an earlier call reported a fault, else A0_OK.  Reads a mapped host word:
 * no synchronisation, so synchronise the stream first to observe the kernels queued on it.           */
int a0_rb_check_fault(a0_replay_t* h);

/* K3 with the learner's input conversion fused in (agent.py:129-135: reshape, .float(), .div(255),
 * split into obs / next_obs).  obs_out, next_out: f32 [count][4][frame_bytes], contiguous, ready
 * for the CNN.  norm_mode 0: x/255 correctly rounded (torch on the CPU); 1: x * fl(1/255) (torch's
 * CUDA div-by-scalar); 2: (float)x.  Scalar outputs as a0_rb_gather.                               */
int a0_rb_gather_f32(a0_replay_t* h, const int64_t* idx /* dev */, int32_t count, int32_t n_step,
                     double gamma, float* obs_out, float* next_out, int32_t norm_mode,
                     int64_t* action_out, double* reward64_out, float* reward32_out,
                     uint8_t* done8_out, float* done32_out, int64_t* boot_out, a0_stream_t stream);
/* The same with bfloat16 outputs (bit patterns in uint16_t), for a learner that runs its CNN in
 * mixed precision (SURVEY 8f-2): each value is bf16(fl32(norm(x))) rounded to nearest even, i.e.
 * what `.float().div(255).to(torch.bfloat16)` gives for the chosen norm_mode.  obs_out, next_out:
 * bf16 [count][4][frame_bytes]; 23 frame-sizes of traffic per transition at n = 3 instead of 39. */
int a0_rb_gather_bf16(a0_replay_t* h, const int64_t* idx /* dev */, int32_t count, int32_t n_step,
                      double gamma, uint16_t* obs_out, uint16_t* next_out, int32_t norm_mode,
                      int64_t* action_out, double* reward64_out, float* reward32_out,
                      uint8_t* done8_out, float* done32_out, int64_t* boot_out, a0_stream_t stream);

/* ---- K4: fused target + loss + IS weighting + new priority -----------------------------------------------
 * Common arguments: B samples; A actions; action i64[B]; reward f32[B] (n-step return); done f32[B]
 * in {0,1}; weight f32[B]; gamma_n = float(discount**n_step).  Outputs: loss f32[B] (unweighted,
 * what the reference returns as q_loss), grad = d[(loss*weight).sum()]/d[online output] (same
 * shape as the online output, zero outside the taken action), prio f32[B] = (loss+eps)^alpha,
 * and *max_p = max(*max_p, loss) when max_p != NULL.  qsel f32[B,A] are the action-selection
 * values (model.qval(next_obs) under double_q); NULL selects from the target output itself.      */
typedef struct {
  int32_t B, A;
  const int64_t* action;
  const float* reward;
  const float* done;
  const float* weight;
  float gamma_n;
  float alpha, eps;      /* priority exponent and offset (ReplayConfig) */
  float* loss;
  float* prio;           /* may be NULL */
  float* max_p;          /* may be NULL */
} a0_loss_common_t;

/* q, qt_next, grad: f32[B,A] */
int a0_loss_dqn(const a0_loss_common_t* c, const float* q, const float* qt_next, const float* qsel,
                float* grad, a0_stream_t stream);
/* qt_next = target(next_obs), qt_cur = target(obs): f32[B,A] */
int a0_loss_mdqn(const a0_loss_common_t* c, const float* q, const float* qt_next,
                 const float* qt_cur, float tau, float lo, float* grad, a0_stream_t stream);
/* logits, tgt_logits, grad: f32[B,A,M]; atoms f32[M]; target_prob (optional) f32[B,M] */
int a0_loss_c51(const a0_loss_common_t* c, const float* logits, const float* tgt_logits,
                const float* qsel, const float* atoms, int32_t M, float vmin, float vmax,
                float* grad, float* target_prob, a0_stream_t stream);
/* a0_loss_c51 as one link of a chain of dependent launches on one stream (hotloop.ReplayTargetLoop: one launch per
 * batch, each behind the previous one).  flags = 0: a0_loss_c51 exactly.  A0_C51_EARLY: the short-chain kernel (qsel
 * given, A <= 6, M <= 64) reads action, reward, done, weight and atoms, computes the projection's geometry and stores
 * the zeros of the sample's gradient block outside the taken action's row BEFORE it waits for its stream predecessor
 * (griddepcontrol.wait); logits, tgt_logits and qsel are still read after the wait.  The caller guarantees: those
 * batch-side inputs and atoms are complete, and no kernel that can still run once this launch's stream predecessor
 * has passed its own wait writes them or reads this batch's gradient rows.  That holds when the stream predecessor
 * is the previous link of the chain and its own only predecessor joined every writer of this batch's inputs; a link
 * that itself joins another stream or event must not set the flag.  Other kernels ignore it.  Same results.     */
#define A0_C51_EARLY 1
int a0_loss_c51_linked(const a0_loss_common_t* c, const float* logits, const float* tgt_logits,
                       const float* qsel, const float* atoms, int32_t M, float vmin, float vmax,
                       float* grad, float* target_prob, int32_t flags, a0_stream_t stream);
/* Test hook of a0_loss_c51's bin arithmetic: for every float32 nu in [0, fl32(vmax - vmin)], the division
 * nu / delta of the short-chain kernel against the correctly rounded one, delta = fl32(vmax - vmin) / (M - 1).
 * out: 2 device words; out[0] += the number of mismatches, out[1] = min(out[1], bit pattern of the first). */
int a0_c51_div_check(float vmin, float vmax, int32_t M, unsigned long long* out, a0_stream_t stream);
/* Quantile-Huber family.  layout 0: q f32[B,A,Nj], qt f32[B,A,Ni], taus implicit (2j+1)/2Nj (QR).
 * layout 1: q f32[B,Nj,A], qt f32[B,Ni,A], taus f32[B,Nj] (IQN, FQF).
 * FQF fraction term (optional, layout 1, Ni == Nj == F): q_bar f32[B,F-1,A] = quantile values at the
 * interior fractions, taus_full f32[B,F+1]; outputs fraction_loss f32[B] and grad_taus f32[B,F+1]
 * = d[(fraction_loss*weight).sum()]/d taus_full.                                                 */
int a0_loss_quantile(const a0_loss_common_t* c, int32_t layout, const float* q, const float* qt,
                     const float* taus, const float* qsel, int32_t Ni, int32_t Nj, float* grad,
                     const float* q_bar, const float* taus_full, float* fraction_loss,
                     float* grad_taus, a0_stream_t stream);

/* ---- K5: actor-side helpers (SURVEY 8f: actor inference batching) ----------------------------------
 * a0_act_epsilon_greedy replaces the tail of Actor.act (agent.py:30-39): per env e,
 *   action[e] = u[e] > epsilon ? argmax_a q[e,a] : action_random[e]   (np.where(rand > eps, greedy, random))
 *   qmax_out[e] = q[e, argmax_a q[e,a]] (optional), *qmax_mean = mean_e of that value (qt_max.mean()).
 * The arg-max is torch's (qt.max(dim=-1)): NaN is greater than every number, and among equal maxima
 * (+0 == -0) or among NaNs the first index wins.  So action, qmax_out and the mean agree: a row with a
 * NaN picks its first NaN, stores NaN and makes the mean NaN.
 * q f32[E,A] = model.qval(obs); u f64[E] and action_random i64[E] are the caller's draws (numpy's
 * generator in the reference: randint first, then rand).  scratch: 8 bytes of device memory, zero
 * before the first call (the kernel re-arms it).  The mean is summed in a fixed order: the same
 * inputs give the same bits on every launch and every GPU.
 * a0_u8_to_f32 is Actor.act's input conversion (agent.py:27), count a multiple of 16 bytes,
 * norm_mode as a0_rb_gather_f32.                                                                  */
int a0_act_epsilon_greedy(const float* q /* dev */, int32_t E, int32_t A, double epsilon,
                          const double* u /* dev */, const int64_t* action_random /* dev */,
                          int64_t* action_out, float* qmax_out, float* scratch, float* qmax_mean,
                          a0_stream_t stream);
int a0_u8_to_f32(const uint8_t* in /* dev */, float* out /* dev */, int64_t count, int32_t norm_mode,
                 a0_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* AGENT0_B200_H */
