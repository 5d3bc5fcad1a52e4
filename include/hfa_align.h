/*
 * hfa_align.h -- C ABI of libhfa_align.so, the B200 (sm_100a) forced-alignment decoder.
 *
 * This is the drop-in boundary for ONE path of yjzxkxdn/HubertFA: tools/alignment_decoder.py
 * (AlignmentDecoder.decode :26-143, ._decode :232-294, .forward_pass :170-230).  The reference
 * has no FFI of its own (it is pure Python + numba), so each entry point below names the
 * reference lines it replaces; INTEGRATION.md shows the ctypes stub a maintainer would add.
 *
 * Conventions
 *   - plain C types only; every pointer marked [dev] is device memory owned by the caller, [host]
 *     is host memory owned by the caller.  The library never allocates device memory and never
 *     synchronises the stream; kernels are enqueued on the cudaStream_t passed as void*.  The one
 *     resource it creates itself: a few non-blocking side streams and timing-free events per host
 *     thread and device, made on first use (independent kernels of one call are forked onto them and
 *     joined back into the caller's stream before the call returns; capturable into a CUDA graph) and
 *     destroyed by hfa_release_thread_resources().
 *   - every function returns HFA_OK (0) or a negative HFA_ERR_* code and never throws;
 *     hfa_last_error() returns a thread-local message for the last failure.
 *   - a batch is ragged: utterance b has T[b] frames and S[b] phoneme states.  Per-frame arrays
 *     are indexed through hfa_plan_frame_offsets(), per-state / per-segment arrays through
 *     hfa_plan_seg_offsets() (both [n_utt + 1], host, int64).
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef HFA_ALIGN_H
#define HFA_ALIGN_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HFA_ABI_VERSION 2

enum {
    HFA_OK = 0,
    HFA_ERR_ARG = -1,         /* bad argument (null pointer, negative size, ...)                  */
    HFA_ERR_CUDA = -2,        /* a CUDA runtime call failed; see hfa_last_error()                 */
    HFA_ERR_UNSUPPORTED = -3, /* shape outside what the kernels cover (S > HFA_MAX_STATES)        */
    HFA_ERR_NOMEM = -4        /* host allocation for the plan failed                              */
};

/* per-utterance status codes written to the result blob (mirror the reference's exceptions) */
enum {
    HFA_UTT_OK = 0,
    HFA_UTT_EMPTY = 1,       /* T < 1: reference raises IndexError at alignment_decoder.py:250     */
    HFA_UTT_BAD_ID = 2,      /* phoneme id outside [0, V): reference raises IndexError at :38/:239 */
    HFA_UTT_NO_STATES = 3,   /* S < 1: reference raises IndexError at :250                         */
    HFA_UTT_INFEASIBLE = 4,  /* best path has score -inf (T too short); outputs still follow the
                                reference (single segment, NaN confidence), flagged for callers    */
    HFA_UTT_TOO_MANY_STATES = 5 /* S > HFA_MAX_STATES (see there)                                  */
};

/* element type of the logits handed to hfa_emission (the reference applies .float(), :57,:63,:69) */
enum { HFA_DTYPE_F32 = 0, HFA_DTYPE_F16 = 1, HFA_DTYPE_BF16 = 2 };

/* Largest S the library aligns (2^20).  Utterances with S <= HFA_CTA_MAX_S (8192: one CTA of 1024 threads x 8
 * states) may run in any forward kernel; longer ones always run in the skewed-wavefront strips (halo bands without
 * TMA tensor maps), whose shared memory does not depend on S.  The bound is what every index provably handles:
 * state indices, strip / band counts per utterance and the emission, backpointer and exchange row strides
 * (Sp, 16-frame words x Sp) are int32 and stay below 2^21 here; every offset that multiplies a frame index by
 * a state count or stride is int64 (cells, emissions, backpointer words, kept dp); the per-utterance kept-dp /
 * exchange sizes of one utterance (T < 2^31 frames x 2^20 states) fit int64 with room to spare.  Larger S ->
 * HFA_UTT_TOO_MANY_STATES. */
#define HFA_MAX_STATES (1 << 20)
#define HFA_CTA_MAX_S 8192

typedef struct hfa_plan hfa_plan; /* opaque, host side: collation + bucketing of one ragged batch */

/* Where each result lives inside the result blob (byte offsets from its start).  The blob is one
 * contiguous device buffer so that a single D2H copy returns everything the host needs. */
typedef struct HfaResultLayout {
    int64_t total_bytes;
    int64_t status;       /* int32 [n_utt]            HFA_UTT_*                                    */
    int64_t n_seg;        /* int32 [n_utt]            K = number of segments on the best path      */
    int64_t end_state;    /* int32 [n_utt]            state chosen at T-1 (:269-272)               */
    int64_t final_score;  /* float [n_utt]            dp[T-1, end_state]                           */
    int64_t total_conf;   /* float [n_utt]            :97                                          */
    int64_t ph_idx_seq;   /* int32 [sum S]            :278, utterance b at seg_off[b], K entries   */
    int64_t ph_time_int;  /* int32 [sum S]            :279                                         */
    int64_t intervals;    /* double[sum S][2]         :104-113 seconds, before SP filter / clip    */
} HfaResultLayout;

/* ---- library ------------------------------------------------------------------------------ */
int hfa_abi_version(void);
const char *hfa_last_error(void);
/* destroys the side streams / events the calling host thread made (see the conventions above); no
 * library call of this thread may be in flight.  They are re-created on the next use. */
void hfa_release_thread_resources(void);

/* ---- collation (host only; replaces the reference's one-utterance-per-call loop, infer.py:60) */
/* T, S: [n_utt] host.  ph_ids: concatenated phoneme ids of all utterances, [sum S] host
 * (alignment_decoder.py:35).  frame_length = hop_length / sample_rate (:12).
 * Utterances are bucketed by the number of states per lane (S class) and ordered by T inside a
 * bucket; invalid utterances get a per-utterance status and are skipped by the kernels. */
int hfa_plan_create(int32_t n_utt, int32_t vocab_size, const int32_t *T, const int32_t *S,
                    const int32_t *ph_ids, double frame_length, hfa_plan **out);
void hfa_plan_destroy(hfa_plan *plan);

int64_t hfa_plan_workspace_bytes(const hfa_plan *plan); /* device scratch the caller must provide */
int64_t hfa_plan_total_frames(const hfa_plan *plan);    /* sum T over valid utterances            */
int64_t hfa_plan_total_states(const hfa_plan *plan);    /* sum S (all utterances)                 */
int64_t hfa_plan_total_cells(const hfa_plan *plan);     /* sum T*S over valid utterances          */
const int64_t *hfa_plan_frame_offsets(const hfa_plan *plan); /* [n_utt+1] host                    */
const int64_t *hfa_plan_seg_offsets(const hfa_plan *plan);   /* [n_utt+1] host                    */
int hfa_plan_result_layout(const hfa_plan *plan, HfaResultLayout *out);
/* algorithmic HBM bytes of each kernel for this batch (DESIGN.md "roofline"): [0] emission,
 * [1] DP forward, [2] backtrace+finalize */
int hfa_plan_algorithmic_bytes(const hfa_plan *plan, int32_t dtype, int64_t out[3]);

/* Which forward-pass kernels this plan uses (filled at hfa_plan_create from the batch shape):
 * out[0] utterances in the one-warp-per-utterance kernel, out[1] warps (bands) and out[2] states per
 * lane of the banded kernel for S <= 256 (small batches: several warps per utterance), out[3] / out[4]
 * the same for S > 256, out[5] utterances in the CTA-per-utterance kernels, out[6] 1 if the banded
 * forward pass keeps dp for the backtrace, out[7] > 0: those lists run in the skewed-wavefront kernel
 * (one state per lane, out[2] / out[4] == 1) with that many frames of skew per state. */
int hfa_plan_routing(const hfa_plan *plan, int32_t out[8]);
/* How many of the out[0] utterances run in the warp kernel's SP-aware pair layout (the state axis regrouped into
 * {SP, phoneme} pairs so that the advance out of an SP needs no f64 arithmetic; tools/alignment_decoder.py:182-187
 * with curr == 0 at :226-228).  Chosen per utterance at hfa_plan_create. */
int32_t hfa_plan_pair_utterances(const hfa_plan *plan);
/* Strips of the skewed-wavefront kernel resident per SM (4 or 5), chosen per plan from a list schedule of the strips
 * of one forward list: list 0 = the small-batch list (hfa_plan_routing out[1]), 1 = the long-sequence list (out[3]).
 * 0 when that list does not run in the skewed kernel. */
int32_t hfa_plan_skew_ctas_per_sm(const hfa_plan *plan, int32_t list);
/* Bytes of emissions hfa_emission stores for this plan.  For the utterances of the pair layout the rows are
 * compacted to one column per DISTINCT phoneme id (states with the same id have the same emission,
 * prob_log[t, ids[s]], tools/alignment_decoder.py:239): fewer than the 4 bytes per DP cell of SURVEY 8(d). */
int64_t hfa_plan_stored_emission_bytes(const hfa_plan *plan);

/* Copies the plan's tables (descriptors, ids, bucket order) into the head of the workspace, zeroes
 * the banded kernel's exchange table and writes the TMA tensor maps of its emission windows (they
 * hold addresses inside THIS workspace).
 * Must be enqueued once per (plan, workspace) before any compute call. */
int hfa_plan_upload(const hfa_plan *plan, void *workspace /*[dev]*/, void *stream);

/* ---- stage 1: logits -> emissions (alignment_decoder.py:35-40,53-71,83-84,239,241-242) ------- */
/* hfa_set_inputs: frame_ptrs[b] -> logits of utterance b addressed as
 * base[t*frame_stride_t[b] + v*frame_stride_v[b]] (elements; the reference receives strided views of
 * the [1,T,V+2] head output, networks/task/forced_alignment.py:288-291); edge_ptrs[b][t*edge_stride[b]].
 * When every utterance has unit column stride the rows travel by TMA in 16-byte units: the logits
 * must then be readable from the 16-byte boundary below a block's first logit to the one above its
 * last (always true for views of a larger tensor and for allocator-aligned buffers).
 * The tables are [host] arrays of [dev] pointers; this call copies them into the workspace (a
 * pageable-memory H2D copy, so it is NOT capturable into a CUDA graph; every other compute entry
 * point only launches kernels and is).  What is recorded is per (plan, workspace): one plan may be
 * uploaded to several workspaces, each with its own inputs. */
int hfa_set_inputs(const hfa_plan *plan, void *workspace, const void *const *frame_ptrs,
                   const int64_t *frame_stride_t, const int64_t *frame_stride_v,
                   const void *const *edge_ptrs, const int64_t *edge_stride, void *stream);

/* The same table, already in device memory: [dev] HfaInputDesc[n_utt].  A device-to-device copy, so the
 * whole step (this call, hfa_align_batch, the caller's D2H copy) can be captured into a CUDA graph and
 * replayed while the caller rewrites the table between replays.  The library cannot look into the table:
 * max_row_stride > 0 promises that every utterance has frame_stride_v == 1, a 4-byte aligned frame
 * pointer and vocab_size <= frame_stride_t <= max_row_stride (the TMA-fed emission kernel is used then);
 * pass 0 for anything else. */
typedef struct HfaInputDesc {
    const void *frame;        /* [dev] logits of the utterance, element (t, v) at frame[t*frame_stride_t + v*frame_stride_v] */
    const void *edge;         /* [dev] edge logits, element t at edge[t*edge_stride]                                          */
    int64_t frame_stride_t, frame_stride_v, edge_stride;   /* in elements */
} HfaInputDesc;
int hfa_set_inputs_device(const hfa_plan *plan, void *workspace, const HfaInputDesc *table /*[dev]*/,
                          int64_t max_row_stride, void *stream);
int hfa_emission(const hfa_plan *plan, void *workspace, int32_t dtype, void *stream);

/* ---- stage 1': the reference's forward_pass inputs, given directly (parity tests) ----------- */
/* prob_log: ragged dense [T_b][S_b] f32 blocks concatenated in utterance order (:239);
 * edge_log / not_edge_log: f32 [sum T] (:241-242); edge_pred: f32 [sum T] (:68-71) or NULL
 * (NULL -> boundaries are not refined, i.e. edge_diff == 0).  All [dev]. */
int hfa_pack_emissions(const hfa_plan *plan, void *workspace, const float *prob_log,
                       const float *edge_log, const float *not_edge_log, const float *edge_pred,
                       void *stream);

/* ---- stage 2: the stay/advance/skip recurrence (alignment_decoder.py:170-230,245-257) -------- */
/* dp_dump: NULL, or [dev] f32 [sum T*S] receiving every dp cell (ragged dense, for tests).      */
int hfa_viterbi_forward(const hfa_plan *plan, void *workspace, float *dp_dump, void *stream);

/* ---- stage 3: end state, backtrace, confidence, intervals (:264-288,:97,:104-113) ----------- */
/* result: [dev] blob of hfa_plan_result_layout().total_bytes.  frame_conf / dp_path: NULL or
 * [dev] f32 [sum T] (frame_confidence :284-288 and dp along the path :276). */
int hfa_backtrace(const hfa_plan *plan, void *workspace, void *result, float *frame_conf,
                  float *dp_path, void *stream);

/* ---- all stages, logits -> result blob (what AlignmentDecoder.decode_batch calls) ----------- */
/* = hfa_emission + hfa_viterbi_forward + hfa_backtrace on the inputs of the last hfa_set_inputs. */
int hfa_align_batch(const hfa_plan *plan, void *workspace, int32_t dtype, void *result,
                    float *frame_conf, void *stream);

/* ---- the fused forward pass (small batches) -------------------------------------------------- */
/* Stages 1+2 in one go for plans whose utterances are all in the banded kernel (hfa_plan_routing:
 * out[0] == out[5] == 0, out[6] == 1), f32 logits with contiguous rows and V <= 256: the edge stream
 * is computed up front, the emissions (alignment_decoder.py:53-65,239) are produced inside the DP
 * kernel by its producer warps and never written to HBM.  hfa_align_batch takes this route on its
 * own when it applies; this entry point exists so that the route can be timed and tested by stage.
 * Returns HFA_ERR_UNSUPPORTED when the plan / inputs do not qualify.  Follow with hfa_backtrace. */
int hfa_forward_fused(const hfa_plan *plan, void *workspace, int32_t dtype, void *stream);
/* algorithmic HBM bytes of that pass: logits + edge logits in, edge logs + backpointers + dp out */
int64_t hfa_plan_algorithmic_bytes_fused(const hfa_plan *plan, int32_t dtype);

/* ---- greedy CTC decode (alignment_decoder.py:145-150, the validation-time ctc()) ------------ */
/* logits: [dev] [T][V] addressed as base[t*stride_t + v*stride_v] (elements), dtype HFA_DTYPE_*.
 * scratch / out_ids: [dev] int32 [T] each; out_len: [dev] int32.  out_ids[0 .. *out_len) = the
 * argmax ids of the frames where the argmax changes (the frame before frame 0 counts as id 0) and
 * is not 0 -- what ctc() returns.  Ties in the argmax go to the lowest id (numpy). */
int hfa_ctc_greedy(const void *logits, int32_t dtype, int64_t T, int64_t V, int64_t stride_t,
                   int64_t stride_v, int32_t *scratch, int32_t *out_ids, int32_t *out_len, void *stream);

/* ---- introspection for tests: unpacked backpointers of one utterance ------------------------ */
/* out: [dev] int8 [T_b][S_b], codes 0/1/2 (row 0 is -1 like the reference, :247). */
int hfa_debug_unpack_backptr(const hfa_plan *plan, const void *workspace, int32_t utt, int8_t *out,
                             void *stream);

/* out: [dev] f32 [T_b][S_b]: the dp cells the forward pass KEPT for the table backtrace (latency plans,
 * hfa_plan_routing out[6]) -- the production kernels' own values, unlike hfa_viterbi_forward's dp_dump.
 * HFA_ERR_UNSUPPORTED when the plan keeps no dp for this utterance. */
int hfa_debug_unpack_dp(const hfa_plan *plan, const void *workspace, int32_t utt, float *out, void *stream);

/* out: [dev] f32, dense ragged [T_b][S_b] for every utterance (the layout hfa_pack_emissions takes): the
 * emissions the workspace currently holds (tools/alignment_decoder.py:239 prob_log[:, ph_seq_id]), whichever
 * way the last writer stored them (plain or compacted rows). */
int hfa_debug_unpack_emissions(const hfa_plan *plan, const void *workspace, float *out, void *stream);

/* byte offset of a workspace region (tests peek at intermediate buffers through this):
 * which = 0 emissions f32 [sum T*Sp] (Sp = S rounded up to 4), 1 edge pairs f32x2 (per utterance
 * padded to a multiple of 16 frames), 2 edge_pred f32 (same padding), 3 backpointer words, 4 the strips' and
 * bands' exchange table (all-zero between calls).
 * Returns -1 for an unknown region. */
int64_t hfa_plan_debug_region(const hfa_plan *plan, int32_t which, int64_t *n_bytes);

/* number of kernel launches the library has enqueued since load (bench.py's gpu_launches) */
int64_t hfa_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* HFA_ALIGN_H */
