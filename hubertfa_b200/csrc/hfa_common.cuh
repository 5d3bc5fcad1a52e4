// hfa_common.cuh -- shared declarations of the sm_100a forced-alignment kernels.
//
// Data layout in HBM (one "plan" = one ragged batch, see hfa_api.cu):
//   emissions  emis[utt][t][s]  f32, row stride Sp = round_up(S, 4) so every row and every 8-frame
//              tile starts 16-byte aligned -> a tile is ONE contiguous 1-D bulk (TMA) copy.
//              Columns S..Sp-1 hold -inf (inert pad states to the right of the last real state).
//   edge pair  edge2[utt][t]    {log(edge_prob+1e-6), log(1-edge_prob+1e-6)} f32x2, frame count
//              padded to a multiple of 16 per utterance so every tile copy is 64 / 128 bytes.
//   edge_p     edge_p[utt][t]   f32 clamp((sigmoid-0.1)/0.8) (same padded indexing as edge2).
//   backptr    bp[utt][t/16][s] u32: bit tt = "advanced by one" and bit 16+tt = "jumped over an
//              SP" for frame t = 16*(t/16)+tt  (2 bits per DP cell, written once per 16 frames).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>

#define HFA_TILE_T 16            // frames per emission tile == frames per backpointer word
#define HFA_WARP_MAX_K 8         // states per lane in the warp-per-utterance kernel
#define HFA_WARP_MAX_S (32 * HFA_WARP_MAX_K)
#define HFA_CTA_K 8              // states per thread in the CTA-per-utterance kernel
#define HFA_PAIR_MAX_K 4         // pairs per lane in the warp kernel's SP-aware pair layout (hfa_dp_pair_body)
#define HFA_NUM_CLASSES 8        // K = 1..8 for the warp kernel (index K-1); class 8 -> CTA kernel

struct HfaUtt {                  // 96 bytes, one per utterance, device copy lives in the workspace
    int32_t T, S, Sp, status;
    int64_t seg_off;             // into ids / per-segment outputs (ints)
    int64_t emis_off;            // floats, multiple of 4
    int64_t edge_off;            // frames, multiple of 16 (edge2 / edge_p index)
    int64_t bp_off;              // u32 words
    int64_t frame_off;           // frames, unpadded (frame_conf / dp_path / path_state / dense in)
    int64_t cell_off;            // sum of T*S of the previous utterances (dense ragged dumps)
    int64_t dp_off;              // floats into dp_store when the forward pass keeps dp for this utterance
                                 // (banded routing; one [T][32 K] block per band, hfa_dp_store_index), else -1
    int32_t band_k;              // states per lane of that banded pass (2 / 4 / 8; 1 = skewed kernel)
    int32_t tmap;                // index of the utterance's emission tensor map (banded / skewed routing), else -1
    int32_t skew_d;              // > 0: the skewed-wavefront kernel ran this utterance with this many frames of
                                 // skew per state; its kept dp uses the skewed layout (hfa_skew_dp_index)
    int32_t pair_k;              // > 0: the warp kernel runs this utterance in the SP-aware pair layout with this
                                 // many {SP, phoneme} pairs per lane (hfa_dp_pair_body); 0: K states per lane
    int32_t Dp;                  // > 0: the emission kernels may store this utterance's rows COMPACTED to one column
                                 // per distinct phoneme id (row stride Dp floats instead of Sp; see HfaWs::colmap)
    int32_t pad_;
};
static_assert(sizeof(HfaUtt) == 96, "HfaUtt is 96 bytes (16-byte multiple)");

struct HfaInput {                // per-utterance logits descriptor (changes per call)
    const void *frame;
    const void *edge;
    int64_t frame_st, frame_sv, edge_st;
};

// one band of one utterance in the banded (halo) DP kernel: consecutive table entries are
// consecutive bands of one utterance
struct HfaBandItem {
    int32_t utt, band;
    int64_t xoff;                // uint4 index of this band's exchange slots [n_tiles][32][2] (0 if unused)
};

// device-side view of the workspace (pointers computed on the host from the plan's layout)
struct HfaWs {
    const HfaUtt *utt;
    const int32_t *ids;          // concatenated phoneme ids
    const int32_t *order;        // bucket order lists (see plan)
    const int32_t *row_blocks;   // exclusive prefix of emission row-blocks per utterance [n+1]
    const int32_t *block_utt;    // utterance of every 64-frame emission row-block [total blocks]
    HfaInput *inputs;
    float *emis;
    float2 *edge2;
    float *edge_p;
    uint32_t *bp;
    int32_t *path_state;         // [sum T]
    int32_t *rev_idx;            // [sum S] segments in backward order
    int32_t *rev_t;              // [sum S]
    float *dp_last;              // end-of-forward scores: [n_utt][2] = dp[T-1][S-1], dp[T-1][S-2]
    float *dp_store;             // dp[t][s] of the utterances with dp_off >= 0 (small-batch routing only)
    // backtrace jump tables of those utterances (same indexing as bp: one entry per backpointer word)
    uint8_t *jump;               // states the path drops while it crosses the 16-frame row, entered at s
    uint8_t *moves;              // segments it opens on the way
    int32_t *row_entry;          // [sum ceil(T/16)] state of the best path at the last frame of each row
    const int32_t *jblk_utt;     // utterance of every 256-word block of the jump-table kernel
    const int32_t *jblk_first;   // [n_utt + 1] first such block of every utterance
    // 128-byte TMA tensor maps (CUtensorMap) over emis[t][s] of the banded utterances: box = 16 frames
    // x one band window; NULL when the driver entry point is unavailable (row copies are used then)
    const void *tmaps;
    // Compacted emission rows (utterances with Dp > 0, i.e. the warp kernel's pair layout): states with the same
    // phoneme id have the same emission (prob_log[t, ids[s]], alignment_decoder.py:239), and 40 % of a
    // dictionary-style sequence is the one id 0 -- so hfa_emission stores one column per DISTINCT id,
    // emis[t][colmap[s]], about half the bytes written and read back.  hfa_pack_emissions takes per-state values
    // and stores the plain [T][Sp] rows; emis_mode[u] says which of the two the last writer left (1 = compacted).
    const int32_t *col_ids;      // [seg_off + 4 u + c]: phoneme id of column c (ascending; pads = vocab -> -inf)
    const uint8_t *colmap;       // [seg_off + s]: column of state s
    int32_t *emis_mode;          // [n_utt]
    const HfaBandItem *band_items;   // banded kernel work list (see hfa_dp_band_kernel)
    int32_t *band_ticket;        // [2] work-item tickets of the two band lists (self-resetting)
    uint4 *band_xchg;            // 16-byte slots of tagged 64-bit words (hfa_ld_xchg): per band, tile and state of
                                 // its last 32, {dp | tag << 32, p.lo | tag << 32}{p.hi | tag << 32, tag << 32};
                                 // per strip and frame, {adv31 | tag << 32, adv30 | tag << 32}.
                                 // All-zero between calls (zeroed by hfa_plan_upload, then by its readers)
};

#define HFA_NEG_INF __uint_as_float(0xff800000u)

// index of dp[t][s] inside an utterance's part of the dp store (floats from dp_off).  The banded kernel
// with K states per lane has windows of W = 32 K states at a stride of W - 32, and every band keeps its
// whole window as a [T][W] block; state s is OWNED by band 0 if s < W, else by band 1 + (s - W) / (W - 32).
__host__ __device__ __forceinline__ int64_t hfa_dp_store_index(int K, int T, int t, int s)
{
    const int W = 32 * K, OWN = W - 32;
    const int b = (s < W) ? 0 : 1 + (s - W) / OWN;
    return ((int64_t)b * T + t) * W + (s - b * OWN);
}

// Skewed-wavefront kernel (hfa_dp_skew.cu): one warp = one STRIP of the state axis, one state per lane.
// Strip 0 covers states 0..31; strip w > 0 starts at column 30 w: its lanes 0 and 1 are GHOSTS that replay the
// advance scores of the left strip's last two states, lanes 2..31 own states 30 w + 2 .. 30 w + 31.
#define HFA_SKEW_OWN 30
#define HFA_SKEW_BOX 36          // columns of its TMA box: the box starts at (30 w) & ~3, a 16-byte boundary
#define HFA_SKEW_BLK 32          // frames per block (TMA tile rows, exchange batch, dp staging tile)
__host__ __device__ __forceinline__ int hfa_skew_strips(int Sp)
{
    return Sp <= 32 ? 1 : 1 + (Sp - 32 + HFA_SKEW_OWN - 1) / HFA_SKEW_OWN;
}
// blocks of HFA_SKEW_BLK iterations a strip runs: lane p handles frame t at iteration t + p D, the last
// lane finishes frame T-1 at iteration T - 1 + 31 D
__host__ __device__ __forceinline__ int hfa_skew_blocks(int D, int T)
{
    return (T + 31 * D + HFA_SKEW_BLK - 1) / HFA_SKEW_BLK;
}
// The kept dp of a skewed pass: every strip stores what its 32 lanes hold after each iteration, one
// 128-byte row per iteration (so dp[t][s] sits at row t + p D of its strip, p = lane of state s).
__host__ __device__ __forceinline__ int64_t hfa_skew_dp_index(int D, int T, int t, int s)
{
    const int w = (s < 32) ? 0 : 1 + (s - 32) / HFA_SKEW_OWN;
    const int p = s - HFA_SKEW_OWN * w;
    return ((int64_t)w * hfa_skew_blocks(D, T) * HFA_SKEW_BLK + t + p * D) * 32 + p;
}

// ---------------------------------------------------------------------------------------------
// PTX primitives.  Shared memory is addressed through 32-bit shared::cta window addresses: a generic
// pointer costs an S2UR + ULEA at every use on sm_100, so a kernel converts once (hfa_smem_u32) and
// works on offsets from there.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t hfa_smem_u32(const void *p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ float hfa_lds_f32(uint32_t addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ float2 hfa_lds_f2(uint32_t addr)
{
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ int hfa_lds_s32(uint32_t addr)
{
    int v;
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void hfa_sts_f32(uint32_t addr, float v)
{
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void hfa_sts_s32(uint32_t addr, int v)
{
    asm volatile("st.shared.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// mbarriers
__device__ __forceinline__ void hfa_mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void hfa_fence_mbar_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void hfa_mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void hfa_mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// non-blocking: has the phase of this parity completed?
__device__ __forceinline__ bool hfa_mbar_test_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// Poll bounds of the spin waits (DESIGN §8 item 4).  A phase that never completes is a bug: fail loudly
// rather than hang the GPU.  Every bound counts the polls of ONE wait and none grows with T.
constexpr uint32_t HFA_POLLS_COPY = 1u << 24;      // one TMA copy of one tile
constexpr uint32_t HFA_POLLS_EXCHANGE = 1u << 26;  // one exchange with the left neighbour (an L2 round trip per poll)
// try_wait suspends the thread for a hardware time slice per poll; `limit` polls, then trap
__device__ __forceinline__ void hfa_mbar_wait(uint32_t bar, uint32_t parity, uint32_t limit)
{
    uint32_t spins = 0;
    for (;;) {
        uint32_t ok;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
        if (ok) return;
        if (++spins > limit) __trap();
    }
}

// bulk async copies (TMA engine): 1-D global -> shared (SASS UBLKCP), completing on an mbarrier
__device__ __forceinline__ void hfa_bulk_load(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// 2-D tensor tile global -> shared (SASS UTMALDG): box position {x = column, y = row}
__device__ __forceinline__ void hfa_tensor_load_2d(uint32_t dst, const void *tmap, int x, int y, uint32_t bar)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cta.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
        "l"(tmap), "r"(x), "r"(y), "r"(bar)
        : "memory");
}
// shared -> global (TMA store), tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void hfa_bulk_store(void *dst, uint32_t src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void hfa_bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// at most N committed stores may still be reading their shared-memory source
template <int N> __device__ __forceinline__ void hfa_bulk_wait_read()
{
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void hfa_bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (a bulk store, a later TMA refill)
__device__ __forceinline__ void hfa_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// one lane of a CONVERGED warp (ptxas then emits TMA / bulk instructions once, from uniform registers, instead of
// an ELECT / R2UR / BRA.U.ANY loop of ~20 instructions per copy)
__device__ __forceinline__ bool hfa_elect_one()
{
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}

// Scattered 4-byte gathers (one value out of a row or a column per frame): by default the L2 fetches the whole
// 128-byte line from HBM; the 64-byte fetch-granularity hint (SASS: LDG.E.LTC64B) is the smallest PTX offers.
__device__ __forceinline__ float hfa_ldg_f32_64B(const float *p)
{
    float v;
    asm volatile("ld.global.L2::64B.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

// Exchange words between the CTAs of one utterance (band and strip kernels, HfaWs::band_xchg): every 64-bit
// word is {payload bits | tag << 32} and is read and written as ONE access, so it is single-copy atomic and
// valid iff its tag matches -- no flag, no fence.  Readers zero what they consumed: the table is all-zero
// between calls.
__device__ __forceinline__ ulonglong2 hfa_ld_xchg(const ulonglong2 *p)
{
    ulonglong2 v;
    asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(v.x), "=l"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void hfa_st_xchg(ulonglong2 *p, unsigned long long a, unsigned long long b)
{
    asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}
__device__ __forceinline__ void hfa_st_xchg_word(unsigned long long *p, unsigned long long a)
{
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(a) : "memory");
}
__device__ __forceinline__ unsigned long long hfa_tagged(uint32_t bits, uint32_t tag)
{
    return (unsigned long long)bits | ((unsigned long long)tag << 32);
}

// the one mixed-precision operation of the recurrence (alignment_decoder.py:182-187):
// f32( f64(a) + f64(curr) * ratio ), multiply and add rounded separately (no FMA contraction).
__device__ __forceinline__ float hfa_advance(float a, float curr, double ratio)
{
    return __double2float_rn(__dadd_rn((double)a, __dmul_rn((double)curr, ratio)));
}

template <typename T> __device__ __forceinline__ float hfa_to_float(T v);
template <> __device__ __forceinline__ float hfa_to_float<float>(float v) { return v; }
template <> __device__ __forceinline__ float hfa_to_float<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float hfa_to_float<__nv_bfloat16>(__nv_bfloat16 v)
{
    return __bfloat162float(v);
}

// {max, log-sum} of one emission row from the max and the sum of exp(x - max) over the logits the
// normaliser reads; every emission is then (x[id] - max) - log-sum.  A max of -inf means every logit read
// is -inf: exp(-inf - -inf) made the sum NaN, so the row takes {0, 0} and every emission stays the
// logit itself, -inf (the reference's masked logits are finite there and its emissions are -inf as well).
__device__ __forceinline__ float2 hfa_row_stat(float mx, float sum)
{
    return mx == HFA_NEG_INF ? make_float2(0.0f, 0.0f) : make_float2(mx, logf(sum));
}

// typed views of the caller's result blob (layout: HfaResultLayout in include/hfa_align.h)
struct HfaResultPtrs {
    int32_t *status, *n_seg, *end_state;
    float *final_score, *total_conf;
    int32_t *ph_idx_seq, *ph_time_int;
    double *intervals;
};

// host-side launchers implemented in the .cu files (all enqueue on `stream`, return cudaError_t)
struct HfaLaunchCtx {
    HfaWs ws;
    int32_t n_utt;
    int32_t vocab;
    double frame_length;
    cudaStream_t stream;
};
