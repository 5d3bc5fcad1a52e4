// hfa_dp.cu -- the stay / advance / skip log-max recurrence over T frames x S states.
//
// Reference semantics: tools/alignment_decoder.py:170-230 (forward_pass) and :245-257 (init).
// For every frame t >= 1 and state i (all f32 unless noted, ratio = f64(T)/f64(S)):
//     stay[i] = (dp[i] + e[t,i]) + not_edge[t]
//     adv[j]  = f32( f64( (dp[j] + e[t,j]) + edge[t] ) + f64(curr[j]) * ratio )     (source state j)
//     dp'[i]  = max(stay[i], adv[i-1], adv[i-2] if ids[i-1]==0)   strict '>' in that order (ties ->
//               the earlier candidate), backpointer = which one won
//     curr[i] = stayed ? max(curr[i], e[t,i]) : e[t,i];   curr[i] = 0 for id-0 (SP) states
// The recurrence is serial in t (curr depends on the path history, so there is no associative scan)
// and embarrassingly parallel across utterances, which is how it is mapped to the GPU:
//
//   hfa_dp_warp_kernel<K>  S <= 32*K <= 256: ONE WARP per utterance, K consecutive states per lane
//       held in registers (dp, curr, backpointer bits); per frame only the last two advance scores
//       of the left neighbour lane cross lanes (2 warp shuffles).  Emission rows are streamed
//       HBM -> smem by the TMA engine as contiguous 8-frame tiles (1-D bulk copy + mbarrier,
//       3 stages); backpointers leave as one bit-packed u32 per state per 16 frames.
//   hfa_dp_cta_kernel      S <= 8192: ONE CTA per utterance, 8 states per thread, the two boundary
//       scores cross warps through shared memory with one __syncthreads per frame.
//
// HBM traffic per DP cell: 4 B emission read + 2 bits backpointer write (+ 8 B per frame of edge
// logs) = the 4.25 B/cell "algorithmic bytes" of DESIGN.md.
#include <algorithm>
#include <cstdlib>
#include <type_traits>

#include "hfa_common.cuh"

namespace {

// one frame of the recurrence for the K states owned by this lane/thread.
// up1 / up2: advance scores of states (first-1) and (first-2) (up1 already -inf where that state
// does not exist).  sp_and[k] = 0 for id-0 (SP) states else ~0 (curr is zeroed by an AND, :226-228);
// jump_cap[k] = +inf where state first+k may be entered by a two-state jump, else -inf (:191-202).
template <int K>
__device__ __forceinline__ void hfa_select(const float (&e)[K], const float (&stay)[K],
                                           const float (&adv)[K], float up1, float up2,
                                           const uint32_t (&sp_and)[K], const float (&jump_cap)[K],
                                           uint32_t m1, uint32_t m2, float (&dp)[K], float (&cu)[K],
                                           uint32_t (&bits)[K])
{
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const float p2 = (k == 0) ? up1 : adv[k - 1];
        const float p3 = (k == 0) ? up2 : ((k == 1) ? up1 : adv[k - 2]);
        // Written as PTX so that the two backpointer bits become predicated ORs and the selects
        // stay selects.  Semantics (alignment_decoder.py:210-228): strict '>' scanned in the order
        // stay, +1, +2 (ties keep the earlier candidate); curr = moved ? e : max(curr, e); curr of
        // an id-0 state is 0 (AND with 0); a two-state jump is only a candidate where jump_cap is
        // +inf (min with -inf removes it).
        asm("{\n\t"
            ".reg .pred q1, q2, q3;\n\t"
            ".reg .f32 m, j, h;\n\t"
            "min.f32 j, %5, %6;\n\t"
            "setp.gt.f32 q1, %3, %4;\n\t"
            "selp.f32 m, %3, %4, q1;\n\t"
            "setp.gt.f32 q2, j, m;\n\t"
            "selp.f32 %0, j, m, q2;\n\t"
            "@q1 or.b32 %2, %2, %9;\n\t"
            "@q2 or.b32 %2, %2, %10;\n\t"
            "max.f32 h, %1, %7;\n\t"
            "or.pred q3, q1, q2;\n\t"
            "selp.f32 h, %7, h, q3;\n\t"
            "and.b32 %1, h, %8;\n\t"
            "}"
            : "=&f"(dp[k]), "+f"(cu[k]), "+r"(bits[k])
            : "f"(p2), "f"(stay[k]), "f"(p3), "f"(jump_cap[k]), "f"(e[k]), "r"(sp_and[k]), "r"(m1),
              "r"(m2));
    }
}

template <int K> __device__ __forceinline__ void hfa_load_row(const float *row, float (&e)[K])
{
    // row is 8-byte (K even) / 16-byte (K % 4 == 0) aligned: Sp % 4 == 0 and first = lane * K
    if constexpr (K % 4 == 0) {
#pragma unroll
        for (int q = 0; q < K / 4; ++q) {
            const float4 v = reinterpret_cast<const float4 *>(row)[q];
            e[4 * q] = v.x; e[4 * q + 1] = v.y; e[4 * q + 2] = v.z; e[4 * q + 3] = v.w;
        }
    } else if constexpr (K % 2 == 0) {
#pragma unroll
        for (int q = 0; q < K / 2; ++q) {
            const float2 v = reinterpret_cast<const float2 *>(row)[q];
            e[2 * q] = v.x; e[2 * q + 1] = v.y;
        }
    } else {
#pragma unroll
        for (int k = 0; k < K; ++k) e[k] = row[k];
    }
}

template <int K>
__device__ __forceinline__ void hfa_store_bits(uint32_t *dst, const uint32_t (&bits)[K], int first,
                                               int Sp)
{
    // dst = &bp[word_row * Sp + first]; Sp % 4 == 0, so for K % 4 == 0 a lane is all-in or all-out
    if constexpr (K % 4 == 0) {
        if (first < Sp) {
#pragma unroll
            for (int q = 0; q < K / 4; ++q)
                if (first + 4 * q < Sp)
                    reinterpret_cast<uint4 *>(dst)[q] =
                        make_uint4(bits[4 * q], bits[4 * q + 1], bits[4 * q + 2], bits[4 * q + 3]);
        }
    } else if constexpr (K % 2 == 0) {
#pragma unroll
        for (int q = 0; q < K / 2; ++q)
            if (first + 2 * q < Sp)
                reinterpret_cast<uint2 *>(dst)[q] = make_uint2(bits[2 * q], bits[2 * q + 1]);
    } else {
#pragma unroll
        for (int k = 0; k < K; ++k)
            if (first + k < Sp) dst[k] = bits[k];
    }
}

// per-thread static state flags (alignment_decoder.py:194,227)
template <int K>
__device__ __forceinline__ void hfa_state_masks(const int32_t *ids, int first, int S,
                                                uint32_t (&sp_and)[K], float (&jump_cap)[K])
{
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int i = first + k;
        sp_and[k] = 0xffffffffu;
        jump_cap[k] = HFA_NEG_INF;
        if (i < S) {
            if (ids[i] == 0) sp_and[k] = 0u;
            if (i >= 2 && ids[i - 1] == 0) jump_cap[k] = __uint_as_float(0x7f800000u);
        }
    }
}

// shared-memory loads by 32-bit shared address (keeps generic->shared address arithmetic out of
// the per-frame loop)
template <int K> __device__ __forceinline__ void hfa_lds_row(uint32_t addr, float (&e)[K])
{
    if constexpr (K % 4 == 0) {
#pragma unroll
        for (int q = 0; q < K / 4; ++q)
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                         : "=f"(e[4 * q]), "=f"(e[4 * q + 1]), "=f"(e[4 * q + 2]), "=f"(e[4 * q + 3])
                         : "r"(addr + 16u * q));
    } else if constexpr (K % 2 == 0) {
#pragma unroll
        for (int q = 0; q < K / 2; ++q)
            asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];"
                         : "=f"(e[2 * q]), "=f"(e[2 * q + 1])
                         : "r"(addr + 8u * q));
    } else {
#pragma unroll
        for (int k = 0; k < K; ++k)
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(e[k]) : "r"(addr + 4u * k));
    }
}

// One frame of K states with curr carried as p = f64(curr) * ratio (see above).
//   e / pe : this frame's emissions and f64(e) * ratio;  ed = {edge_log, not_edge_log}
//   cap1   : +inf, or -inf where state first-1 does not exist (lane 0)
//   sp_hi  : 0 for id-0 (SP) states else ~0 -- ANDed into the high word of p: a zero high word makes
//            p a non-negative subnormal below 2^-1042, which adds to any f64(f32) exactly like +0.0
template <int K>
__device__ __forceinline__ void hfa_frame_p(const float (&e)[K], const double (&pe)[K], const float2 ed,
                                            const uint32_t (&sp_hi)[K], const float (&jump_cap)[K],
                                            const float cap1, const uint32_t m1, const uint32_t m2,
                                            float (&dp)[K], double (&p)[K], uint32_t (&bits)[K])
{
    float stay[K], adv[K];
    // the last state's advance score crosses lanes (shuffle): with two states per lane its conversion
    // chain goes first
#pragma unroll
    for (int kk = 0; kk < K; ++kk) {
        const int k = (K <= 2) ? K - 1 - kk : kk;     // measured: descending only pays for K = 2
        const float base = __fadd_rn(dp[k], e[k]);
        adv[k] = __double2float_rn(__dadd_rn((double)__fadd_rn(base, ed.x), p[k]));
        stay[k] = __fadd_rn(base, ed.y);
    }
    float up1 = __shfl_up_sync(0xffffffffu, adv[K - 1], 1);
    const float up2 = __shfl_up_sync(0xffffffffu, adv[K - 2], 1);   // capped by jump_cap on lane 0
    up1 = fminf(up1, cap1);
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const float p2 = (k == 0) ? up1 : adv[k - 1];
        const float p3 = (k == 0) ? up2 : ((k == 1) ? up1 : adv[k - 2]);
        // alignment_decoder.py:210-228.  Value: max of the three candidates.  Backpointer: strict
        // '>' scanned in the order stay, +1, +2 (ties keep the earlier candidate).  curr: moved ?
        // e : max(curr, e), 0 for id-0 states -- all on p.
        asm("{\n\t"
            ".reg .pred q1, q2, q3;\n\t"
            ".reg .f32 j, m;\n\t"
            ".reg .f64 pn;\n\t"
            ".reg .b32 lo, hi;\n\t"
            "min.f32 j, %5, %6;\n\t"
            "max.f32 m, %4, %3;\n\t"
            "max.f32 %0, m, j;\n\t"
            "setp.gt.f32 q1, %3, %4;\n\t"
            "setp.gt.f32 q2, j, m;\n\t"
            "@q1 or.b32 %2, %2, %9;\n\t"
            "@q2 or.b32 %2, %2, %10;\n\t"
            "or.pred q3, q1, q2;\n\t"
            "setp.gt.or.f64 q3, %7, %1, q3;\n\t"
            "selp.f64 pn, %7, %1, q3;\n\t"
            "mov.b64 {lo, hi}, pn;\n\t"
            "and.b32 hi, hi, %8;\n\t"
            "mov.b64 %1, {lo, hi};\n\t"
            "}"
            : "=&f"(dp[k]), "+d"(p[k]), "+r"(bits[k])
            : "f"(p2), "f"(stay[k]), "f"(p3), "f"(jump_cap[k]), "d"(pe[k]), "r"(sp_hi[k]), "r"(m1),
              "r"(m2));
    }
}

// ---------------------------------------------------------------------------------------------
// warp per utterance
// ---------------------------------------------------------------------------------------------
constexpr int HFA_WARP_TILE = 8;      // frames per TMA stage (two stages = one backpointer word)
// 2 stages, measured on config 4 (B200) against 3: 13 -> 20 resident warps per SM, DP stage 0.370 -> 0.362 ms
// (pairs), 0.480 -> 0.457 ms (plain); the next tile still has a whole tile time (~1 us) to land.  The copy of
// tile i + 2 is issued when tile i has been consumed.
constexpr int HFA_WARP_STAGES = 2;

template <int K> constexpr size_t hfa_warp_smem_bytes()
{
    constexpr int nst = HFA_WARP_STAGES;
    // [stages x 8 rows x 32K floats][one slack row: the prefetch of "row 8" of the last stage]
    // [stages x 8 edge pairs][one slack pair][stages mbarriers]
    // ... [pair tables of hfa_dp_pair_body, which shares this layout]
    return (size_t)(nst * HFA_WARP_TILE + 1) * 32 * K * sizeof(float) +
           (size_t)(nst * HFA_WARP_TILE + 1) * sizeof(float2) + nst * sizeof(uint64_t) +
           (size_t)2 * 32 * HFA_PAIR_MAX_K * sizeof(int16_t);
}

template <int K, bool DUMP>
__device__ __forceinline__ void hfa_dp_warp_body(const HfaWs &ws, const int u,
                                                 float *__restrict__ dp_dump,
                                                 unsigned char *smem_raw)
{
    constexpr int TT = HFA_WARP_TILE, NST = HFA_WARP_STAGES;
    constexpr int ROW_MAX = 32 * K;                       // floats per smem tile row (upper bound)
    constexpr int TILE_FLOATS = TT * ROW_MAX;
    float *tile0 = reinterpret_cast<float *>(smem_raw);
    float2 *edge0 = reinterpret_cast<float2 *>(tile0 + NST * TILE_FLOATS + ROW_MAX);
    uint64_t *bar = reinterpret_cast<uint64_t *>(edge0 + NST * TT + 1);

    const int lane = threadIdx.x & 31;
    const HfaUtt m = ws.utt[u];
    const int T = m.T, S = m.S, Sp = m.Sp;
    const int first = lane * K;
    const int n_tiles = (T + TT - 1) / TT;
    const float *g_emis = ws.emis + m.emis_off;
    const float2 *g_edge = ws.edge2 + m.edge_off;
    uint32_t *g_bp = ws.bp + m.bp_off;
    const double ratio = __ddiv_rn((double)T, (double)S);     // T / S (:186)

    auto issue = [&](int i) {                                  // lane 0 only
        const int st = i % NST;
        const int t0 = i * TT;
        const int rows = min(TT, T - t0);
        const uint32_t bytes = (uint32_t)rows * (uint32_t)Sp * 4u;
        const uint32_t tx = bytes + TT * (uint32_t)sizeof(float2);
        hfa_mbar_expect_tx(hfa_smem_u32(&bar[st]), tx);
        const float *src = g_emis + (int64_t)t0 * Sp;
        hfa_bulk_load(hfa_smem_u32(tile0 + st * TILE_FLOATS), src, bytes, hfa_smem_u32(&bar[st]));
        const float2 *esrc = g_edge + t0;
        hfa_bulk_load(hfa_smem_u32(edge0 + st * TT), esrc, TT * (uint32_t)sizeof(float2), hfa_smem_u32(&bar[st]));
    };

    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < NST; ++s) hfa_mbar_init(hfa_smem_u32(&bar[s]), 1);
        hfa_fence_mbar_init();
        for (int i = 0; i < NST && i < n_tiles; ++i) issue(i);
    }
    uint32_t sp_and[K];
    float jump_cap[K];
    hfa_state_masks<K>(ws.ids + m.seg_off, first, S, sp_and, jump_cap);
    const bool lead_sp = (ws.ids[m.seg_off] == 0) && (S > 1);
    __syncwarp();

    float dp[K], cu[K];
    uint32_t bits[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        dp[k] = HFA_NEG_INF;
        cu[k] = HFA_NEG_INF;
        bits[k] = 0;
    }
    const uint32_t tile_sa = hfa_smem_u32(tile0) + (uint32_t)first * 4u;
    const uint32_t edge_sa = hfa_smem_u32(edge0);
    const uint32_t row_bytes = (uint32_t)Sp * 4u;

    int st = 0;
    uint32_t phase = 0;
    for (int i = 0; i < n_tiles; ++i) {
        hfa_mbar_wait(hfa_smem_u32(&bar[st]), phase, HFA_POLLS_COPY);
        const uint32_t tl = tile_sa + (uint32_t)st * (TILE_FLOATS * 4u);
        const uint32_t et = edge_sa + (uint32_t)st * (TT * 8u);
        const int rows = min(TT, T - i * TT);
        const int sh = (i & 1) * TT;                         // bit position of this tile's frame 0
        uint32_t mbit = 1u << sh;                             // backpointer bit of the current frame
        // one frame; operands of the NEXT frame (en / edn) are fetched before this frame's dependent
        // chain -- for the last row of a stage that reads the next stage / the slack row (discarded)
        auto frame = [&](int tt, const float (&e)[K], const float2 ed, float (&en)[K], float2 &edn) {
            hfa_lds_row<K>(tl + (uint32_t)(tt + 1) * row_bytes, en);
            edn = hfa_lds_f2(et + (uint32_t)(tt + 1) * 8u);
            if (tt == 0 && i == 0) {
                // t = 0 (:250-254): state 0 is seeded, and state 1 too behind a leading SP
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    const int s = first + k;
                    if (s == 0 || (s == 1 && lead_sp)) {
                        dp[k] = e[k];
                        cu[k] = e[k];
                    }
                }
            } else {
                float stay[K], adv[K];
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    const float base = __fadd_rn(dp[k], e[k]);
                    stay[k] = __fadd_rn(base, ed.y);
                    adv[k] = hfa_advance(__fadd_rn(base, ed.x), cu[k], ratio);
                }
                float up1 = __shfl_up_sync(0xffffffffu, adv[K - 1], 1);
                float up2;
                if constexpr (K >= 2) up2 = __shfl_up_sync(0xffffffffu, adv[K - 2], 1);
                else up2 = __shfl_up_sync(0xffffffffu, adv[0], 2);
                if (lane == 0) up1 = HFA_NEG_INF;  // state -1 does not exist; up2 is capped by jump_cap
                hfa_select<K>(e, stay, adv, up1, up2, sp_and, jump_cap, mbit, mbit << 16, dp, cu, bits);
            }
            mbit <<= 1;
            if constexpr (DUMP) {
                const int64_t o = m.cell_off + (int64_t)(i * TT + tt) * S;
#pragma unroll
                for (int k = 0; k < K; ++k)
                    if (first + k < S) dp_dump[o + first + k] = dp[k];
            }
        };
        float ea[K], eb[K];
        float2 da, db;
        hfa_lds_row<K>(tl, ea);
        da = hfa_lds_f2(et);
        if (rows == TT) {
            // full tile: the two operand sets ping-pong without copies.  NOT unrolled further: the
            // merged kernel keeps up to 8 code paths hot per SM and must fit the instruction cache
            // (ncu: stall_no_instruction dominated when this loop was fully unrolled).
#pragma unroll 1
            for (int tt = 0; tt < TT; tt += 2) {
                frame(tt, ea, da, eb, db);
                frame(tt + 1, eb, db, ea, da);
            }
        } else {
            for (int tt = 0; tt < rows; ++tt) {               // last, partial tile
                frame(tt, ea, da, eb, db);
#pragma unroll
                for (int k = 0; k < K; ++k) ea[k] = eb[k];
                da = db;
            }
        }
        if ((i & 1) || i == n_tiles - 1) {                   // 16 frames done (or the end): flush
            hfa_store_bits<K>(g_bp + (int64_t)(i >> 1) * Sp + first, bits, first, Sp);
#pragma unroll
            for (int k = 0; k < K; ++k) bits[k] = 0;
        }
        __syncwarp();                                        // every lane is done reading stage `st`
        if (lane == 0 && i + NST < n_tiles) issue(i + NST);
        if (++st == NST) {
            st = 0;
            phase ^= 1u;
        }
    }

    // scores of the last two states at T-1 for the end-state rule (:269-272)
#pragma unroll
    for (int k = 0; k < K; ++k) {
        if (first + k == S - 1) ws.dp_last[2 * u] = dp[k];
        if (first + k == S - 2) ws.dp_last[2 * u + 1] = dp[k];
    }
}

// ---------------------------------------------------------------------------------------------
// warp per utterance, SP-aware PAIR layout (big batches; SURVEY 7: "skip the f64 op when the source
// state is SP")
// ---------------------------------------------------------------------------------------------
// An id-0 (SP) state never keeps a running maximum: curr is zeroed after every update (:226-228), so
// for every frame t >= 2 its advance score is f32(f64(a) + 0.0 * ratio) = a (+0.0 for a = -0.0) -- no
// conversion, no f64 op.  It also has only two candidates (stay / +1: the two-state jump needs an SP at
// i-1, and in a sequence without adjacent SPs that is a phoneme).  To make that saving warp-uniform the
// state axis is regrouped into PAIRS {B = the SP in front of phoneme n (if there is one), A = phoneme n};
// a trailing SP is the B of one more pair without an A.  Every lane owns KP consecutive pairs:
//     B[n]  = max(stayB, advA[n-1])                                  bit: +1
//     A[n]  = max(stayA, advB[n], advA[n-1])   strict '>' in this order.  With a B the two candidates are
//             "+1" and "+2 over the SP"; without one advB is -inf and advA[n-1] is the "+1" -- the bits
//             are sorted out when a backpointer word is stored, once per 16 frames.
// ~27 instructions per pair instead of ~21 per state, one lane exchange per frame instead of two, a third of
// the conversions, and a dictionary-style sequence has ~1.67 states per pair.  Nothing else changes: the
// emission tile is the same contiguous bulk copy into the same shared-memory ring as in hfa_dp_warp_body,
// every slot reads its column through its own address register plus the frame's (uniform) row offset, and
// the backpointer words keep their state order.  A pair without an SP reads its phoneme's column for B and
// caps B's only candidate at -inf, so that B stays at -inf; a slot without a phoneme (the trailing pair,
// the lanes past the last pair) computes garbage that only flows to the right, where nothing exists.
// Frame 0 (:250-254) and frame 1 (the one frame where the curr of a leading SP is not 0, quirk q1) go
// through the guarded body.
// Eligibility (hfa_plan_create): no two adjacent SPs, pairs <= 32 * HFA_PAIR_MAX_K, cheaper than the
// K-states-per-lane body.

template <int KP, bool DUMP>
__device__ __forceinline__ void hfa_dp_pair_body(const HfaWs &ws, const int u, float *__restrict__ dp_dump,
                                                 unsigned char *smem_raw)
{
    constexpr int TT = HFA_WARP_TILE, NST = HFA_WARP_STAGES;
    // frames per unrolled chunk: measured on config 4 (B200, every utterance in pairs), DP stage 0.382 / 0.390 /
    // 0.370 ms with 2 / 4 / 8
    constexpr int UNR = 8;
    const int lane = threadIdx.x & 31;
    const HfaUtt m = ws.utt[u];
    const int T = m.T, S = m.S, Sp = m.Sp;
    // the shared-memory layout of hfa_dp_warp_body<K> for this utterance's class, K = ceil(Sp / 32): rows of Sp
    // floats, NST tiles of TT rows and one slack row; then the pair tables
    const int row_max = (Sp + 31) & ~31;
    float *tile0 = reinterpret_cast<float *>(smem_raw);
    float2 *edge0 = reinterpret_cast<float2 *>(tile0 + (NST * TT + 1) * row_max);
    uint64_t *bar = reinterpret_cast<uint64_t *>(edge0 + NST * TT + 1);
    int16_t *tabA = reinterpret_cast<int16_t *>(bar + NST);     // state of every pair's phoneme / SP, or -1
    int16_t *tabB = tabA + 32 * KP;

    const int n_tiles = (T + TT - 1) / TT;
    const float *g_emis = ws.emis + m.emis_off;
    const float2 *g_edge = ws.edge2 + m.edge_off;
    uint32_t *g_bp = ws.bp + m.bp_off;
    const int32_t *ids = ws.ids + m.seg_off;
    const double ratio = __ddiv_rn((double)T, (double)S);     // T / S (:186)
    // emission rows: plain [T][Sp], or compacted to one column per distinct id (HfaWs::colmap) -- then several
    // slots simply hold the same column address
    const bool compact = m.Dp > 0 && ws.emis_mode[u] != 0;
    const int Ep = compact ? m.Dp : Sp;
    const uint8_t *cmap = ws.colmap + m.seg_off;
    const uint32_t row_bytes = (uint32_t)Ep * 4u;
    const uint32_t tile_bytes = TT * row_bytes;

    auto issue = [&](int i) {                                  // one elected lane
        const int st = i % NST;
        const int t0 = i * TT;
        const int rows = min(TT, T - t0);
        const uint32_t bytes = (uint32_t)rows * row_bytes;
        const uint32_t tx = bytes + TT * (uint32_t)sizeof(float2);
        hfa_mbar_expect_tx(hfa_smem_u32(&bar[st]), tx);
        const float *src = g_emis + (int64_t)t0 * Ep;
        hfa_bulk_load(hfa_smem_u32(tile0 + st * TT * Ep), src, bytes, hfa_smem_u32(&bar[st]));
        const float2 *esrc = g_edge + t0;
        hfa_bulk_load(hfa_smem_u32(edge0 + st * TT), esrc, TT * (uint32_t)sizeof(float2), hfa_smem_u32(&bar[st]));
    };

    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < NST; ++s) hfa_mbar_init(hfa_smem_u32(&bar[s]), 1);
        hfa_fence_mbar_init();
    }
    for (int q = lane; q < 32 * KP; q += 32) {
        tabA[q] = -1;
        tabB[q] = -1;
    }
    __syncwarp();
    if (hfa_elect_one())
        for (int i = 0; i < NST && i < n_tiles; ++i) issue(i);
    {
        int before = 0;                                        // phonemes in front of this chunk of 32 states
        for (int c0 = 0; c0 < S; c0 += 32) {
            const int i = c0 + lane;
            const bool is_ph = i < S && ids[i] != 0;
            const uint32_t mask = __ballot_sync(0xffffffffu, is_ph);
            const int pr = before + __popc(mask & ((1u << lane) - 1u));
            if (i < S) (is_ph ? tabA : tabB)[pr] = (int16_t)i;
            before += __popc(mask);
        }
    }
    const bool sp0 = ids[0] == 0;
    __syncwarp();

    float dpA[KP], cuA[KP], dpB[KP], capB[KP];
    uint32_t X[KP], Y[KP], Z[KP];                              // A: won by advB / by advA[n-1];  B: advanced
    uint32_t aA[KP], aB[KP];                                   // shared address of the slot's column in ring row 0
    const uint32_t tile_sa = hfa_smem_u32(tile0);
#pragma unroll
    for (int k = 0; k < KP; ++k) {
        dpA[k] = HFA_NEG_INF; cuA[k] = HFA_NEG_INF; dpB[k] = HFA_NEG_INF;
        X[k] = 0; Y[k] = 0; Z[k] = 0;
        const int sa = tabA[lane * KP + k], sb = tabB[lane * KP + k];
        // a slot that does not exist reads its partner's column (any valid address): B is then capped below,
        // A is garbage that nothing real ever reads
        const int ca = sa >= 0 ? sa : max(sb, 0), cb = sb >= 0 ? sb : max(sa, 0);
        aA[k] = tile_sa + 4u * (uint32_t)(compact ? cmap[ca] : ca);
        aB[k] = tile_sa + 4u * (uint32_t)(compact ? cmap[cb] : cb);
        capB[k] = sb >= 0 ? __uint_as_float(0x7f800000u) : HFA_NEG_INF;
    }
    float cuB0 = 0.f;                                          // curr of a leading SP during frame 1 (q1)
    const uint32_t edge_sa = hfa_smem_u32(edge0);

    auto load = [&](uint32_t off, uint32_t eoff, float (&eA)[KP], float (&eB)[KP], float2 &ed) {
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            eA[k] = hfa_lds_f32(aA[k] + off);
            eB[k] = hfa_lds_f32(aB[k] + off);
        }
        ed = hfa_lds_f2(edge_sa + eoff);
    };
    // one frame t >= 1.  GUARD: frame 1 -- the leading SP still carries curr = e[0][0]
    auto step = [&](auto guard, const int t, const uint32_t mbit, const float (&eA)[KP], const float (&eB)[KP],
                    const float2 ed) {
        float stayA[KP], stayB[KP], advA[KP], advB[KP];
        const float xc = __fadd_rn(ed.x, 0.0f);               // -0.0 -> +0.0: f32(f64(a) + 0.0) without the f64
#pragma unroll
        for (int kk = 0; kk < KP; ++kk) {
            const int k = KP - 1 - kk;                         // the last pair's score crosses lanes: first
            const float baseA = __fadd_rn(dpA[k], eA[k]);
            advA[k] = hfa_advance(__fadd_rn(baseA, ed.x), cuA[k], ratio);
            stayA[k] = __fadd_rn(baseA, ed.y);
            const float baseB = __fadd_rn(dpB[k], eB[k]);
            advB[k] = __fadd_rn(baseB, xc);
            stayB[k] = __fadd_rn(baseB, ed.y);
            if constexpr (decltype(guard)::value) {
                if (k == 0 && t == 1 && lane == 0 && sp0) advB[0] = hfa_advance(__fadd_rn(baseB, ed.x), cuB0, ratio);
            }
        }
        float up = __shfl_up_sync(0xffffffffu, advA[KP - 1], 1);
        if (lane == 0) up = HFA_NEG_INF;                       // no phoneme in front of pair 0
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            const float p3 = (k == 0) ? up : advA[k - 1];
            const float p3b = fminf(p3, capB[k]);              // a B that does not exist stays at -inf
            // alignment_decoder.py:210-228 on the pair: strict '>' scanned in the reference's order; curr of the
            // phoneme = moved ? e : max(curr, e); the SP has no curr.
            // Three predicates per pair (a fourth one for "moved" made ptxas spill predicates from two pairs per
            // lane on; masks instead of predicates -- set.gt.u32 -- cost an FSETP + SEL each).
            asm("{\n\t"
                ".reg .pred qb, q1, q2;\n\t"
                ".reg .f32 m, h;\n\t"
                "setp.gt.f32 qb, %12, %7;\n\t"
                "selp.f32 %0, %12, %7, qb;\n\t"
                "@qb or.b32 %3, %3, %11;\n\t"
                "setp.gt.f32 q1, %8, %9;\n\t"
                "selp.f32 m, %8, %9, q1;\n\t"
                "setp.gt.f32 q2, %6, m;\n\t"
                "selp.f32 %1, %6, m, q2;\n\t"
                "@q1 or.b32 %4, %4, %11;\n\t"
                "@q2 or.b32 %5, %5, %11;\n\t"
                "max.f32 h, %2, %10;\n\t"
                "selp.f32 h, %10, h, q1;\n\t"
                "selp.f32 %2, %10, h, q2;\n\t"
                "}"
                : "=&f"(dpB[k]), "=&f"(dpA[k]), "+f"(cuA[k]), "+r"(Z[k]), "+r"(X[k]), "+r"(Y[k])
                : "f"(p3), "f"(stayB[k]), "f"(advB[k]), "f"(stayA[k]), "f"(eA[k]), "r"(mbit), "f"(p3b));
        }
        if constexpr (DUMP) {
            const int64_t o = m.cell_off + (int64_t)t * S;
#pragma unroll
            for (int k = 0; k < KP; ++k) {
                const int sa = tabA[lane * KP + k], sb = tabB[lane * KP + k];
                if (sa >= 0) dp_dump[o + sa] = dpA[k];
                if (sb >= 0) dp_dump[o + sb] = dpB[k];
            }
        }
    };
    // frame 0 (:250-254): state 0 is seeded, and state 1 too behind a leading SP
    auto seed = [&](const float (&eA)[KP], const float (&eB)[KP]) {
        if (lane == 0) {
            if (sp0) {
                dpB[0] = eB[0];
                cuB0 = eB[0];
            }
            if (!sp0 || S > 1) {
                dpA[0] = eA[0];
                cuA[0] = eA[0];
            }
        }
        if constexpr (DUMP) {
#pragma unroll
            for (int k = 0; k < KP; ++k) {
                const int sa = tabA[lane * KP + k], sb = tabB[lane * KP + k];
                if (sa >= 0) dp_dump[m.cell_off + sa] = dpA[k];
                if (sb >= 0) dp_dump[m.cell_off + sb] = dpB[k];
            }
        }
    };

    int st = 0;
    uint32_t phase = 0;
    for (int i = 0; i < n_tiles; ++i) {
        hfa_mbar_wait(hfa_smem_u32(&bar[st]), phase, HFA_POLLS_COPY);
        const uint32_t tl = (uint32_t)st * tile_bytes;        // row 0 of this stage (uniform)
        const uint32_t et = (uint32_t)st * (TT * 8u);
        const int rows = min(TT, T - i * TT);
        const uint32_t mb0 = 1u << ((i & 1) * TT);             // backpointer bit of this tile's frame 0
        float ea[KP], eb[KP], fa[KP], fb[KP];
        float2 da, db;
        load(tl, et, ea, eb, da);
        if (rows == TT && i > 0) {
            // full tile: two operand sets ping-pong, the next frame's operands are fetched before this
            // frame's dependent chain (row 8 = the next stage's row 0 or the slack row: discarded).  Unrolled
            // in chunks of UNR frames.  The merged kernel keeps one body hot per class present and the
            // instruction cache is 32 KB: with pair AND plain bodies in one launch no_instruction was the top
            // stall on config 4, which is why the plan moves a whole batch to pairs or none of it
            uint32_t ro = tl, ec = et, mb = mb0;
#pragma unroll 1
            for (int c = 0; c < TT / UNR; ++c) {
#pragma unroll
                for (int tt = 0; tt < UNR; tt += 2) {
                    load(ro + (uint32_t)(tt + 1) * row_bytes, ec + (uint32_t)(tt + 1) * 8u, fa, fb, db);
                    step(std::false_type{}, i * TT + c * UNR + tt, mb << tt, ea, eb, da);
                    load(ro + (uint32_t)(tt + 2) * row_bytes, ec + (uint32_t)(tt + 2) * 8u, ea, eb, da);
                    step(std::false_type{}, i * TT + c * UNR + tt + 1, mb << (tt + 1), fa, fb, db);
                }
                ro += UNR * row_bytes;
                ec += UNR * 8u;
                mb <<= UNR;
            }
        } else {
            for (int tt = 0; tt < rows; ++tt) {                // first tile / last, partial tile
                if (tt > 0) load(tl + (uint32_t)tt * row_bytes, et + (uint32_t)tt * 8u, ea, eb, da);
                if (i == 0 && tt == 0) seed(ea, eb);
                else step(std::true_type{}, i * TT + tt, mb0 << tt, ea, eb, da);
            }
        }
        if ((i & 1) || i == n_tiles - 1) {                     // 16 frames done (or the end): flush
            uint32_t *row = g_bp + (int64_t)(i >> 1) * Sp;
#pragma unroll
            for (int k = 0; k < KP; ++k) {
                const int sa = tabA[lane * KP + k], sb = tabB[lane * KP + k];
                // with an SP in front: X = "+1", Y = "+2"; without: Y = "+1" (X is empty)
                if (sa >= 0) row[sa] = sb >= 0 ? (X[k] | (Y[k] << 16)) : Y[k];
                if (sb >= 0) row[sb] = Z[k];
                X[k] = 0; Y[k] = 0; Z[k] = 0;
            }
        }
        __syncwarp();                                          // every lane is done reading stage `st`
        if (i + NST < n_tiles) {
            if (hfa_elect_one()) issue(i + NST);
        }
        if (++st == NST) {
            st = 0;
            phase ^= 1u;
        }
    }

    // scores of the last two states at T-1 for the end-state rule (:269-272)
#pragma unroll
    for (int k = 0; k < KP; ++k) {
        const int sa = tabA[lane * KP + k], sb = tabB[lane * KP + k];
        if (sa >= 0 && sa >= S - 2) ws.dp_last[2 * u + (S - 1 - sa)] = dpA[k];
        if (sb >= 0 && sb >= S - 2) ws.dp_last[2 * u + (S - 1 - sb)] = dpB[k];
    }
}

// every state class in ONE launch: each warp picks the code path of its utterance.  All warps get
// the shared memory of the largest class present, the block scheduler sees one globally
// longest-first ordered grid, and nothing depends on concurrent-kernel scheduling.  WPC warps per
// CTA (one utterance each, no interaction between them); HFA_DP_WPC=4 packs four per CTA.
template <bool DUMP, int MAXK>
__global__ void __launch_bounds__(32)
hfa_dp_warp_any_kernel(HfaWs ws, const int32_t *__restrict__ order, int n,
                       float *__restrict__ dp_dump)
{
    // MAXK = largest states-per-lane class in this launch: the register allocation (and with it the
    // number of resident warps per SM) follows the widest code path that can actually run
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int item = blockIdx.x;
    if (item >= n) return;
    const int u = order[item];
    const int kp = ws.utt[u].pair_k;                    // > 0: the SP-aware pair layout was chosen for it
    if (kp > 0) {
        if (kp == 1) hfa_dp_pair_body<1, DUMP>(ws, u, dp_dump, smem_raw);
        else if (kp == 2) hfa_dp_pair_body<2, DUMP>(ws, u, dp_dump, smem_raw);
        else if (kp == 3) hfa_dp_pair_body<3, DUMP>(ws, u, dp_dump, smem_raw);
        else hfa_dp_pair_body<4, DUMP>(ws, u, dp_dump, smem_raw);
        return;
    }
    const int k = (ws.utt[u].Sp + 31) >> 5;
    if (k <= 1) hfa_dp_warp_body<1, DUMP>(ws, u, dp_dump, smem_raw);
    else if (k == 2) hfa_dp_warp_body<2, DUMP>(ws, u, dp_dump, smem_raw);
    if constexpr (MAXK >= 3) { if (k == 3) hfa_dp_warp_body<3, DUMP>(ws, u, dp_dump, smem_raw); }
    if constexpr (MAXK >= 4) { if (k == 4) hfa_dp_warp_body<4, DUMP>(ws, u, dp_dump, smem_raw); }
    if constexpr (MAXK >= 5) { if (k == 5) hfa_dp_warp_body<5, DUMP>(ws, u, dp_dump, smem_raw); }
    if constexpr (MAXK >= 6) { if (k == 6) hfa_dp_warp_body<6, DUMP>(ws, u, dp_dump, smem_raw); }
    if constexpr (MAXK >= 8) {
        if (k == 7) hfa_dp_warp_body<7, DUMP>(ws, u, dp_dump, smem_raw);
        if (k >= 8) hfa_dp_warp_body<8, DUMP>(ws, u, dp_dump, smem_raw);
    }
}

// ---------------------------------------------------------------------------------------------
// CTA per utterance (256 < S <= 8192)
// ---------------------------------------------------------------------------------------------
constexpr int HFA_CTA_STAGES = 3;

template <int K, int NT>
__global__ void __launch_bounds__(NT)
hfa_dp_cta_kernel(HfaWs ws, const int32_t *__restrict__ order, int tile_t, int stage_floats,
                  float *__restrict__ dp_dump)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // [stages x stage_floats f32][stages x 16 float2][stages mbarriers][2 x 32 float2 exchange]
    float *tile0 = reinterpret_cast<float *>(smem_raw);
    float2 *edge0 = reinterpret_cast<float2 *>(tile0 + HFA_CTA_STAGES * stage_floats);
    uint64_t *bar = reinterpret_cast<uint64_t *>(edge0 + HFA_CTA_STAGES * HFA_TILE_T);
    float2 *xch = reinterpret_cast<float2 *>(bar + HFA_CTA_STAGES);   // [2][32]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int u = order[blockIdx.x];
    const HfaUtt m = ws.utt[u];
    const int T = m.T, S = m.S, Sp = m.Sp;
    // the launch is sized for the longest phoneme sequence of the list: warps that own no state of
    // THIS utterance leave, the rest synchronise on a barrier sized to the warps that stay
    const int n_active = (((Sp + K - 1) / K) + 31) & ~31;
    if (tid >= n_active) return;
    auto cta_sync = [&]() { asm volatile("bar.sync 0, %0;" ::"r"(n_active) : "memory"); };
    const int first = tid * K;
    const int n_tiles = (T + tile_t - 1) / tile_t;
    const float *g_emis = ws.emis + m.emis_off;
    const float2 *g_edge = ws.edge2 + m.edge_off;
    uint32_t *g_bp = ws.bp + m.bp_off;
    const double ratio = __ddiv_rn((double)T, (double)S);
    // the edge pair always travels as the whole 16-frame (128 B) block that contains the tile
    constexpr uint32_t edge_bytes = HFA_TILE_T * (uint32_t)sizeof(float2);

    auto issue = [&](int i) {                                  // thread 0 only
        const int st = i % HFA_CTA_STAGES;
        const int t0 = i * tile_t;
        const int rows = min(tile_t, T - t0);
        const uint32_t bytes = (uint32_t)rows * (uint32_t)Sp * 4u;
        const uint32_t tx = bytes + edge_bytes;
        hfa_mbar_expect_tx(hfa_smem_u32(&bar[st]), tx);
        const float *src = g_emis + (int64_t)t0 * Sp;
        hfa_bulk_load(hfa_smem_u32(tile0 + st * stage_floats), src, bytes, hfa_smem_u32(&bar[st]));
        const float2 *esrc = g_edge + (t0 & ~(HFA_TILE_T - 1));
        hfa_bulk_load(hfa_smem_u32(edge0 + st * HFA_TILE_T), esrc, edge_bytes, hfa_smem_u32(&bar[st]));
    };

    if (tid == 0) {
        for (int s = 0; s < HFA_CTA_STAGES; ++s) hfa_mbar_init(hfa_smem_u32(&bar[s]), 1);
        hfa_fence_mbar_init();
        for (int i = 0; i < HFA_CTA_STAGES && i < n_tiles; ++i) issue(i);
    }
    uint32_t sp_and[K];
    float jump_cap[K];
    hfa_state_masks<K>(ws.ids + m.seg_off, first, S, sp_and, jump_cap);
    const bool lead_sp = (ws.ids[m.seg_off] == 0) && (S > 1);
    cta_sync();

    float dp[K], cu[K];
    uint32_t bits[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        dp[k] = HFA_NEG_INF;
        cu[k] = HFA_NEG_INF;
        bits[k] = 0;
    }

    for (int i = 0; i < n_tiles; ++i) {
        const int st = i % HFA_CTA_STAGES;
        const uint32_t parity = (i / HFA_CTA_STAGES) & 1;
        hfa_mbar_wait(hfa_smem_u32(&bar[st]), parity, HFA_POLLS_COPY);
        // threads past the last padded state still run the loop (they take part in the barriers)
        // but read row 0 of the stage instead of running off its end
        const float *tl = tile0 + st * stage_floats + (first < Sp ? first : 0);
        const float2 *et = edge0 + st * HFA_TILE_T;
        const int rows = min(tile_t, T - i * tile_t);
        for (int tt = 0; tt < rows; ++tt) {
            const int t = i * tile_t + tt;
            float e[K];
            hfa_load_row<K>(tl + tt * Sp, e);
            if (t == 0) {
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    const int s = first + k;
                    if (s == 0 || (s == 1 && lead_sp)) {
                        dp[k] = e[k];
                        cu[k] = e[k];
                    }
                    if (dp_dump != nullptr && s < S) dp_dump[m.cell_off + s] = dp[k];
                }
                continue;
            }
            const float2 ed = et[t & (HFA_TILE_T - 1)];
            float stay[K], adv[K];
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const float base = __fadd_rn(dp[k], e[k]);
                stay[k] = __fadd_rn(base, ed.y);
                adv[k] = hfa_advance(__fadd_rn(base, ed.x), cu[k], ratio);
            }
            float up1 = __shfl_up_sync(0xffffffffu, adv[K - 1], 1);
            float up2 = __shfl_up_sync(0xffffffffu, adv[K - 2], 1);
            float2 *slot = xch + (t & 1) * 32;
            if (lane == 31) slot[warp] = make_float2(adv[K - 1], adv[K - 2]);
            cta_sync();
            if (lane == 0) {
                if (warp == 0) {
                    up1 = HFA_NEG_INF;
                    up2 = HFA_NEG_INF;
                } else {
                    const float2 v = slot[warp - 1];
                    up1 = v.x;
                    up2 = v.y;
                }
            }
            const int b = t & 15;
            hfa_select<K>(e, stay, adv, up1, up2, sp_and, jump_cap, 1u << b, 0x10000u << b, dp, cu,
                          bits);
            if (dp_dump != nullptr) {
                const int64_t o = m.cell_off + (int64_t)t * S;
#pragma unroll
                for (int k = 0; k < K; ++k)
                    if (first + k < S) dp_dump[o + first + k] = dp[k];
            }
            if (b == 15 || t == T - 1) {
                hfa_store_bits<K>(g_bp + (int64_t)(t >> 4) * Sp + first, bits, first, Sp);
#pragma unroll
                for (int k = 0; k < K; ++k) bits[k] = 0;
            }
        }
        // Every thread has read its last row of stage `st` before the barrier of that frame (or,
        // for a tile that only holds frame 0, before this point): one more barrier frees the stage.
        cta_sync();
        if (tid == 0 && i + HFA_CTA_STAGES < n_tiles) issue(i + HFA_CTA_STAGES);
    }
    if (T == 1) hfa_store_bits<K>(g_bp + first, bits, first, Sp);   // row 0 word (all zero)

#pragma unroll
    for (int k = 0; k < K; ++k) {
        if (first + k == S - 1) ws.dp_last[2 * u] = dp[k];
        if (first + k == S - 2) ws.dp_last[2 * u + 1] = dp[k];
    }
}

// ---------------------------------------------------------------------------------------------
// Banded (halo) kernel: SEVERAL WARPS PER UTTERANCE ON DIFFERENT SMs, one exchange per 16 frames.
//
// State i at frame t only depends on states i, i-1, i-2 at frame t-1 (alignment_decoder.py:177-202),
// so over a 16-frame tile a state is a function of the 32 states to its left at the start of the
// tile.  A band is one compute warp that holds a window of W = 32 K consecutive states, K per
// lane; windows of neighbouring bands overlap by 32 states: band b covers [b (W-32), b (W-32) + W).
// The first 32 states of a window (b > 0) are the HALO: they are recomputed from the left
// neighbour's values at the start of every tile, go stale from the left edge at two states per
// frame, and the stale region reaches the first owned state exactly when the tile ends.  After each
// tile the left band publishes {dp, curr*ratio} of its last 32 states (= the halo of its right
// neighbour); neighbours never talk inside a tile, so the bands of one utterance run as a pipeline
// skewed by 1-2 tiles across SMs instead of a serial chain on one lane set.
//   * small batches (latency regime): K = 2 -- every utterance with more than 64 states becomes
//     ceil((Sp-32)/32) warps whose per-frame dependent chain is as short as it gets;
//   * long phoneme sequences (S > 256, BASELINE config 3): K = 2/4 -- 2000 states = 62/21 warps on
//     as many SMs instead of one CTA with a barrier per frame.
// CTA = 2 warps.  Warp 1 is the PRODUCER: it issues the TMA row copies of the emission window
// (16 bulk copies + the edge pairs per tile, 3 stages, full/empty mbarriers) and polls the left
// neighbour's exchange slots into shared memory; both complete on the stage's "full" barrier.
// Warp 0 is the CONSUMER: it only waits on that barrier, runs the recurrence, stores backpointer
// words and publishes its own last 32 states.  Work items are claimed through an atomic ticket, so
// a band's left neighbour has always started before the band itself; band 0 never waits.
// Exchange slot of one state after tile i: two 16-byte halves of tagged 64-bit words (hfa_ld_xchg),
// {dp | tag << 32, p.lo | tag << 32} {p.hi | tag << 32, tag << 32}, tag = i + 1.  Every word is
// read and written as ONE access (single-copy atomic), so a word is valid iff its tag matches: no
// flag, no fence.  The reader zeroes the slot after use, so the table is all-zero between calls
// (zeroed once by hfa_plan_upload).
//
// The serial chain per frame is  FADD, FADD, F2F, DADD, F2F, SHFL, 3 x FMNMX  (~85 cycles):
//   * curr[] is carried as the f64 product p = f64(curr) * ratio.  ratio > 0 and rounding is
//     monotone, so max(curr, e) * ratio == max(p, f64(e) * ratio) bit for bit, and f64(e) * ratio
//     only depends on the emission: it is computed one frame ahead, off the chain.
//   * dp' = max(stay, adv1, adv2) is taken with FMNMX (value identical to the reference's strict-'>'
//     scan, ties included); the two comparisons that define the backpointer run beside it.
// Extra HBM/L2 traffic: 1 KB per band per tile each way.
// ---------------------------------------------------------------------------------------------
constexpr int HFA_BAND_STAGES = 3;

template <int K> constexpr size_t hfa_band_smem_bytes()
{
    // [stages x 16 rows x 32K floats][slack row][stages x 16 edge pairs][slack pair]
    // [stages x 32 halo entries {dp, pad, p}][full, empty mbarriers][ticket]
    return (size_t)(HFA_BAND_STAGES * HFA_TILE_T + 1) * 32 * K * sizeof(float) +
           (size_t)(HFA_BAND_STAGES * HFA_TILE_T + 2) * sizeof(float2) +
           (size_t)HFA_BAND_STAGES * 32 * 16 + 2 * HFA_BAND_STAGES * sizeof(uint64_t) + 16;
}
// fused emission: [keep mask 8 u32][kept ids 256 i32][16 x {max, lse}][2 mbarriers][2 shifts + pad]
// [2 logits stages of lstage_bytes]
constexpr size_t HFA_FUSED_FIXED_BYTES = 8 * 4 + 256 * 4 + 16 * 8 + 2 * 8 + 16;

template <int K, bool DUMP, bool KEEP, bool FUSED>
__global__ void __launch_bounds__(64)
hfa_dp_band_kernel(HfaWs ws, int item_begin, int32_t *ticket, float *__restrict__ dp_dump, int V,
                   int lstage_bytes)
{
    static_assert(32 % K == 0 && K >= 2, "the halo (32 states) must be a whole number of lanes");
    constexpr int TT = HFA_TILE_T, NST = HFA_BAND_STAGES;
    constexpr int W = 32 * K, OWN = W - 32, HL = 32 / K;     // HL = halo lanes = publishing lanes
    constexpr int TILE_FLOATS = TT * W;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *tile0 = reinterpret_cast<float *>(smem_raw);
    float2 *edge0 = reinterpret_cast<float2 *>(tile0 + NST * TILE_FLOATS + W);
    uint4 *halo0 = reinterpret_cast<uint4 *>(edge0 + NST * TT + 2);   // 16-byte aligned
    uint64_t *full = reinterpret_cast<uint64_t *>(halo0 + NST * 32);
    uint64_t *empty = full + NST;
    int *slot = reinterpret_cast<int *>(empty + NST);

    // Which of the two warps computes?  The warps of a 2-warp CTA land on an aligned pair of warp
    // slots, and slot % 4 is the scheduler partition, so "warp 0 computes" would put every compute
    // warp of the SM on partitions 0 and 2 (tools/ubench_warpid.cu).  Swapping the roles in every
    // other pair spreads them over all four.
    const int lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        unsigned hw_slot;
        asm volatile("mov.u32 %0, %%warpid;" : "=r"(hw_slot));
        slot[1] = (int)((hw_slot >> 2) & 1u);
    }
    if (threadIdx.x == 0) {
        *slot = (int)atomicInc(reinterpret_cast<unsigned int *>(ticket), gridDim.x - 1);   // self-resetting
#pragma unroll
        for (int s = 0; s < NST; ++s) {
            hfa_mbar_init(hfa_smem_u32(&full[s]), 2);    // the copy issuer + the halo relay
            hfa_mbar_init(hfa_smem_u32(&empty[s]), 1);   // the compute warp
        }
        hfa_fence_mbar_init();
    }
    __syncthreads();
    const int warp = (int)(threadIdx.x >> 5) ^ slot[1];        // 0 = compute, 1 = producer
    const int item = item_begin + *slot;
    const HfaBandItem bi = ws.band_items[item];
    const int u = bi.utt, band = bi.band;
    const HfaUtt m = ws.utt[u];
    const int T = m.T, S = m.S, Sp = m.Sp;
    const int c0 = band * OWN;                                 // first state of the window
    const int n_bands = Sp <= W ? 1 : (Sp - 32 + OWN - 1) / OWN;
    const bool has_left = band > 0, has_right = band + 1 < n_bands;
    const int n_tiles = (T + TT - 1) / TT;

    if (warp == 1) {
        // ---------------- producer: TMA row copies + halo relay ----------------
        const int cols = min(W, Sp - c0);                      // window columns that exist (% 4 == 0)
        const uint32_t row_b = (uint32_t)cols * 4u;
        const float *g_emis = ws.emis + m.emis_off + c0;
        const float2 *g_edge = ws.edge2 + m.edge_off;
        // ---- fused emission (FUSED): the producer computes the emission window itself.  The
        // logits rows of a tile arrive by ONE bulk copy ([16][row stride] f32, contiguous in the
        // [T, V+2] head output) into a double-buffered logits stage; the masked log-softmax and
        // the gather by phoneme id follow hfa_emission_stream_kernel instruction for instruction
        // (4 lanes per frame over the kept ids, xor-shuffle combine, (x - max) - lse), so a fused
        // and an unfused run produce the same bits.  No emission ever touches HBM.
        uint32_t *mask_sm = reinterpret_cast<uint32_t *>(slot + 4);
        int32_t *kept_sm = reinterpret_cast<int32_t *>(mask_sm + 8);
        float2 *stat_sm = reinterpret_cast<float2 *>(kept_sm + 256);
        uint64_t *lbar = reinterpret_cast<uint64_t *>(stat_sm + 16);
        int32_t *shift_sm = reinterpret_cast<int32_t *>(lbar + 2);
        unsigned char *lstage0 = reinterpret_cast<unsigned char *>(shift_sm + 4);
        int n_kept = 0, row_st = 0;
        uint32_t gid[K];
        int kreg[16];
        const unsigned char *g_logits = nullptr;
        auto issue_logits = [&](int i) {                       // lane 0 only
            const int ls = i & 1;
            const int t0 = i * TT;
            const int rows = min(TT, T - t0);
            const unsigned char *src = g_logits + (int64_t)t0 * row_st * 4;
            const uint32_t shift = (uint32_t)(reinterpret_cast<uintptr_t>(src) & 15u);
            const uint32_t bytes = (shift + (uint32_t)(((int64_t)(rows - 1) * row_st + V) * 4) + 15u) & ~15u;
            shift_sm[ls] = (int32_t)shift;
            hfa_mbar_expect_tx(hfa_smem_u32(&lbar[ls]), bytes);
            hfa_bulk_load(hfa_smem_u32(lstage0 + (size_t)ls * lstage_bytes), src - shift, bytes,
                          hfa_smem_u32(&lbar[ls]));
        };
        if constexpr (FUSED) {
            const HfaInput in = ws.inputs[u];
            g_logits = reinterpret_cast<const unsigned char *>(in.frame);
            row_st = (int)in.frame_st;
            const int32_t *ids = ws.ids + m.seg_off;
            if (lane < 8) mask_sm[lane] = (lane == 0) ? 1u : 0u;             // id 0 always kept (:39)
            if (lane == 0) {
                hfa_mbar_init(hfa_smem_u32(&lbar[0]), 1);
                hfa_mbar_init(hfa_smem_u32(&lbar[1]), 1);
                hfa_fence_mbar_init();
            }
            __syncwarp();
            for (int q = lane; q < S; q += 32) atomicOr(&mask_sm[ids[q] >> 5], 1u << (ids[q] & 31));
            __syncwarp();
            const int mask_words = (V + 31) >> 5;
#pragma unroll
            for (int w = 0; w < 8; ++w) n_kept += (w < mask_words) ? __popc(mask_sm[w]) : 0;
            for (int v = lane; v < V; v += 32) {
                if ((mask_sm[v >> 5] >> (v & 31)) & 1u) {
                    int pos = __popc(mask_sm[v >> 5] & ((1u << (v & 31)) - 1u));
                    for (int w = 0; w < (v >> 5); ++w) pos += __popc(mask_sm[w]);
                    kept_sm[pos] = v;
                }
            }
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int sgl = c0 + lane * K + k;
                gid[k] = (sgl < S) ? (uint32_t)ids[sgl] : (uint32_t)V;       // pad columns: -inf
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int k = (lane & 3) + 4 * j;
                kreg[j] = (k < n_kept && k < 256) ? kept_sm[k] : 0;
            }
            if (lane == 0) issue_logits(0);
        }
        const unsigned char *tmap = (ws.tmaps != nullptr && m.tmap >= 0)
                                        ? static_cast<const unsigned char *>(ws.tmaps) + (size_t)m.tmap * 128 : nullptr;
        ulonglong2 *left_x =
            reinterpret_cast<ulonglong2 *>(ws.band_xchg) + (has_left ? ws.band_items[item - 1].xoff : 0) + 2 * lane;
        // dp store: the compute warp leaves dp[t][.] of a tile in the stage it has just consumed (in
        // place of the emissions); before the stage is refilled the tile goes out as one bulk store.
        // every band keeps its WHOLE window ([T][W] block of its own, the halo columns included --
        // they hold stale values and are never read) so that a tile leaves as one bulk store
        float *g_dp = (KEEP && m.dp_off >= 0) ? ws.dp_store + m.dp_off + (int64_t)band * T * W : nullptr;
        for (int i = 0; i < n_tiles + NST; ++i) {
            const int st = i % NST;
            if (i >= NST) {
                hfa_mbar_wait(hfa_smem_u32(&empty[st]), (uint32_t)(((i / NST) - 1) & 1), HFA_POLLS_COPY);
                const int j = i - NST;                         // the tile that sat in this stage
                if (g_dp != nullptr && lane == 0) {
                    hfa_bulk_store(g_dp + (int64_t)j * TT * W, hfa_smem_u32(tile0 + st * TILE_FLOATS),
                                   (uint32_t)min(TT, T - j * TT) * (uint32_t)W * 4u);
                    hfa_bulk_commit();
                    hfa_bulk_wait_read<0>();                   // the stage may be overwritten
                }
                __syncwarp();
            }
            if (i >= n_tiles) continue;
            const int t0 = i * TT;
            const int rows = min(TT, T - t0);
            const uint32_t full_sa = hfa_smem_u32(&full[st]), edge_sa = hfa_smem_u32(edge0 + st * TT);
            constexpr uint32_t edge_bytes = TT * (uint32_t)sizeof(float2);
            if constexpr (FUSED) {
                if (lane == 0) {
                    hfa_mbar_expect_tx(full_sa, edge_bytes);
                    hfa_bulk_load(edge_sa, g_edge + t0, edge_bytes, full_sa);
                    if (i + 1 < n_tiles) issue_logits(i + 1);     // its stage was read during tile i-1
                }
                const int ls = i & 1;
                hfa_mbar_wait(hfa_smem_u32(&lbar[ls]), (uint32_t)((i >> 1) & 1), HFA_POLLS_COPY);
                const float *xs = reinterpret_cast<const float *>(lstage0 + (size_t)ls * lstage_bytes + shift_sm[ls]);
                // normaliser: lane -> (row = 8 * pass + lane / 4, part = lane % 4), kept ids only.
                // The lane's kept ids sit in registers (kreg, <= 16 of them: up to 64 kept ids) so
                // that its loads go out back to back; the max / sum chains keep the standalone
                // kernel's order (k = part, part + 4, ...).
#pragma unroll
                for (int pass = 0; pass < 2; ++pass) {
                    const int rr = 8 * pass + (lane >> 2);
                    const float *row = xs + rr * row_st;
                    const int part = lane & 3;
                    float mx = HFA_NEG_INF, sum = 0.0f;
                    if (n_kept <= 64) {                                       // warp-uniform
                        float xv[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {   // unconditional load (kreg is 0 past the end) + select
                            const float x = row[kreg[j]];
                            xv[j] = (part + 4 * j < n_kept) ? x : HFA_NEG_INF;
                        }
#pragma unroll
                        for (int j = 0; j < 16; ++j) mx = fmaxf(mx, xv[j]);
                        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
                        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
#pragma unroll
                        for (int j = 0; j < 16; ++j)     // entries past the end are -inf: exp = +0, sum unchanged
                            sum = __fadd_rn(sum, expf(__fsub_rn(xv[j], mx)));
                    } else {
                        for (int k = part; k < n_kept; k += 4) mx = fmaxf(mx, row[kept_sm[k]]);
                        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
                        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
                        for (int k = part; k < n_kept; k += 4)
                            sum = __fadd_rn(sum, expf(__fsub_rn(row[kept_sm[k]], mx)));
                    }
                    sum = __fadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, 1));
                    sum = __fadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, 2));
                    if (part == 0) stat_sm[rr] = hfa_row_stat(mx, sum);
                }
                __syncwarp();
                // gather by phoneme id: K window columns per lane, the layout the compute warp reads;
                // four rows at a time so that their loads overlap
                float *dst = tile0 + st * TILE_FLOATS + lane * K;
                auto put_row = [&](int r, const float (&o)[K]) {
                    if constexpr (K % 4 == 0) {
#pragma unroll
                        for (int q = 0; q < K / 4; ++q)
                            reinterpret_cast<float4 *>(dst + r * W)[q] =
                                make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
                    } else {
#pragma unroll
                        for (int q = 0; q < K / 2; ++q)
                            reinterpret_cast<float2 *>(dst + r * W)[q] = make_float2(o[2 * q], o[2 * q + 1]);
                    }
                };
                for (int r0 = 0; r0 < rows; r0 += 4) {
                    float o[4][K];
                    float2 sv[4];
#pragma unroll
                    for (int d = 0; d < 4; ++d) {
                        const int r = min(r0 + d, TT - 1);
                        sv[d] = stat_sm[r];
                        const float *row = xs + r * row_st;
#pragma unroll
                        for (int k = 0; k < K; ++k) o[d][k] = (gid[k] < (uint32_t)V) ? row[gid[k]] : HFA_NEG_INF;
                    }
#pragma unroll
                    for (int d = 0; d < 4; ++d) {
#pragma unroll
                        for (int k = 0; k < K; ++k) o[d][k] = __fsub_rn(__fsub_rn(o[d][k], sv[d].x), sv[d].y);
                        if (r0 + d < rows) put_row(r0 + d, o[d]);
                    }
                }
            } else if (tmap != nullptr) {
                // ONE tensor-tile copy per stage: box = 16 frames x W columns at {c0, t0} of emis[t][s]
                // (rows past T and columns past Sp are zero-filled and never used)
                if (lane == 0) {
                    hfa_mbar_expect_tx(full_sa, (uint32_t)(TILE_FLOATS * 4) + edge_bytes);
                    hfa_bulk_load(edge_sa, g_edge + t0, edge_bytes, full_sa);
                    hfa_tensor_load_2d(hfa_smem_u32(tile0 + st * TILE_FLOATS), tmap, c0, t0, full_sa);
                }
            } else {
                if (lane == 0) {
                    hfa_mbar_expect_tx(full_sa, (uint32_t)rows * row_b + edge_bytes);
                    hfa_bulk_load(edge_sa, g_edge + t0, edge_bytes, full_sa);
                }
                __syncwarp();
                if (lane < rows)
                    hfa_bulk_load(hfa_smem_u32(tile0 + st * TILE_FLOATS + lane * W), g_emis + (int64_t)(t0 + lane) * Sp, row_b,
                                  full_sa);
            }
            if (has_left && i > 0) {
                // the window's first 32 states at the start of tile i = the left band's last 32
                // after its tile i-1: lane j relays state j
                ulonglong2 *src = left_x + (int64_t)(i - 1) * 64;
                const uint32_t tag = (uint32_t)i;
                ulonglong2 a = hfa_ld_xchg(src), b = hfa_ld_xchg(src + 1);
                uint32_t spins = 0;
                while ((uint32_t)(a.x >> 32) != tag || (uint32_t)(a.y >> 32) != tag || (uint32_t)(b.x >> 32) != tag ||
                       (uint32_t)(b.y >> 32) != tag) {
                    if (++spins > HFA_POLLS_EXCHANGE) __trap();
                    a = hfa_ld_xchg(src);
                    b = hfa_ld_xchg(src + 1);
                }
                halo0[st * 32 + lane] = make_uint4((uint32_t)a.x, 0u, (uint32_t)a.y, (uint32_t)b.x);
                hfa_st_xchg(src, 0ull, 0ull);   // leave the table clean for the next call
                hfa_st_xchg(src + 1, 0ull, 0ull);
            }
            __syncwarp();
            if (lane == 0) hfa_mbar_arrive(full_sa);
        }
        hfa_bulk_wait_all();
        return;
    }

    // ---------------- consumer: the recurrence ----------------
    const int first = c0 + lane * K;                           // first state of this lane
    const bool owner = !has_left || lane >= HL;                // lanes whose states this band owns
    uint32_t *g_bp = ws.bp + m.bp_off;
    const double ratio = __ddiv_rn((double)T, (double)S);
    ulonglong2 *my_x = reinterpret_cast<ulonglong2 *>(ws.band_xchg) + bi.xoff + 2 * ((lane - (32 - HL)) * K);

    uint32_t sp_hi[K];
    float jump_cap[K];
    hfa_state_masks<K>(ws.ids + m.seg_off, first, S, sp_hi, jump_cap);
    const bool lead_sp = (ws.ids[m.seg_off] == 0) && (S > 1);
    // lane 0: nothing to the left of state 0 (band 0) / stale halo edge (other bands, value unused)
    const float cap1 = lane == 0 ? HFA_NEG_INF : __uint_as_float(0x7f800000u);

    float dp[K];
    double p[K];
    uint32_t bits[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        dp[k] = HFA_NEG_INF;
        p[k] = __longlong_as_double(0xfff0000000000000ll);     // curr = -inf
        bits[k] = 0;
    }
    const uint32_t tile_sa = hfa_smem_u32(tile0) + (uint32_t)(lane * K) * 4u;
    const uint32_t edge_sa = hfa_smem_u32(edge0);
    constexpr uint32_t row_bytes = (uint32_t)W * 4u;

    // dp[t][.] replaces the emissions of frame t in the stage (picked up by the producer warp)
    constexpr bool keep = KEEP;      // compiled out when the plan keeps no dp: even a predicated-off store
                                     // in the frame loop costs 8 % (measured)
    auto put = [&](uint32_t row_sa, int t) {
        if (keep) {
            if constexpr (K % 4 == 0) {
#pragma unroll
                for (int q = 0; q < K / 4; ++q)
                    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(row_sa + 16u * q), "f"(dp[4 * q]),
                                 "f"(dp[4 * q + 1]), "f"(dp[4 * q + 2]), "f"(dp[4 * q + 3])
                                 : "memory");
            } else {
#pragma unroll
                for (int q = 0; q < K / 2; ++q)
                    asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(row_sa + 8u * q), "f"(dp[2 * q]),
                                 "f"(dp[2 * q + 1])
                                 : "memory");
            }
        }
        if constexpr (DUMP) {
            const int64_t o = m.cell_off + (int64_t)t * S;
#pragma unroll
            for (int k = 0; k < K; ++k)
                if (owner && first + k < S) dp_dump[o + first + k] = dp[k];
        }
    };

    int st = 0;
    uint32_t phase = 0;
    for (int i = 0; i < n_tiles; ++i) {
        hfa_mbar_wait(hfa_smem_u32(&full[st]), phase, HFA_POLLS_COPY);
        const uint32_t tl = tile_sa + (uint32_t)st * (TILE_FLOATS * 4u);
        const uint32_t et = edge_sa + (uint32_t)st * (TT * 8u);
        const int rows = min(TT, T - i * TT);
        if (has_left && i > 0 && lane < HL) {                 // halo: the left band's values
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const uint4 h = halo0[st * 32 + lane * K + k];
                dp[k] = __uint_as_float(h.x);
                p[k] = __hiloint2double((int)h.w, (int)h.z);
            }
        }
        float ea[K], eb[K];
        double pa[K], pb[K];
        float2 da, db;
        hfa_lds_row<K>(tl, ea);
        da = hfa_lds_f2(et);
#pragma unroll
        for (int k = 0; k < K; ++k) pa[k] = __dmul_rn((double)ea[k], ratio);
        int tt0 = 0;
        if (i == 0) {
            // t = 0 (:250-254): state 0 is seeded, and state 1 too behind a leading SP; curr keeps
            // the emission even for an id-0 state until the first step has run
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int s = first + k;
                if (s == 0 || (s == 1 && lead_sp)) {
                    dp[k] = ea[k];
                    p[k] = pa[k];
                }
            }
            put(tl, 0);
            tt0 = 1;
        }
        if (tt0 == 0 && rows == TT) {
            // full tile: operands of the next frame (emissions, their f64 products, edge pair) are
            // fetched / converted while the current frame's chain runs; two frames per iteration
            // (unrolling the whole tile measured slower: 0.157 vs 0.154 ms on config 2)
            uint32_t mbit = 1u;
#pragma unroll 1
            for (int tt = 0; tt < TT; tt += 2) {
                hfa_lds_row<K>(tl + (uint32_t)(tt + 1) * row_bytes, eb);
                db = hfa_lds_f2(et + (uint32_t)(tt + 1) * 8u);
                hfa_frame_p<K>(ea, pa, da, sp_hi, jump_cap, cap1, mbit, mbit << 16, dp, p, bits);
#pragma unroll
                for (int k = 0; k < K; ++k) pb[k] = __dmul_rn((double)eb[k], ratio);
                put(tl + (uint32_t)tt * row_bytes, i * TT + tt);
                hfa_lds_row<K>(tl + (uint32_t)(tt + 2) * row_bytes, ea);     // slack row after the last
                da = hfa_lds_f2(et + (uint32_t)(tt + 2) * 8u);
                hfa_frame_p<K>(eb, pb, db, sp_hi, jump_cap, cap1, mbit << 1, mbit << 17, dp, p, bits);
#pragma unroll
                for (int k = 0; k < K; ++k) pa[k] = __dmul_rn((double)ea[k], ratio);
                put(tl + (uint32_t)(tt + 1) * row_bytes, i * TT + tt + 1);
                mbit <<= 2;
            }
        } else {
            for (int tt = tt0; tt < rows; ++tt) {            // first and last (partial) tile
                hfa_lds_row<K>(tl + (uint32_t)tt * row_bytes, ea);
                da = hfa_lds_f2(et + (uint32_t)tt * 8u);
#pragma unroll
                for (int k = 0; k < K; ++k) pa[k] = __dmul_rn((double)ea[k], ratio);
                hfa_frame_p<K>(ea, pa, da, sp_hi, jump_cap, cap1, 1u << tt, 0x10000u << tt, dp, p, bits);
                put(tl + (uint32_t)tt * row_bytes, i * TT + tt);
            }
        }
        // one backpointer word per owned state per tile
        if (owner) hfa_store_bits<K>(g_bp + (int64_t)i * Sp + first, bits, first, Sp);
#pragma unroll
        for (int k = 0; k < K; ++k) bits[k] = 0;
        if (has_right && i + 1 < n_tiles && lane >= 32 - HL) {   // publish the right neighbour's halo
            const uint32_t tag = (uint32_t)i + 1u;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                ulonglong2 *dst = my_x + (int64_t)i * 64 + 2 * k;
                hfa_st_xchg(dst, hfa_tagged(__float_as_uint(dp[k]), tag),
                            hfa_tagged((uint32_t)__double2loint(p[k]), tag));
                hfa_st_xchg(dst + 1, hfa_tagged((uint32_t)__double2hiint(p[k]), tag), hfa_tagged(0u, tag));
            }
        }
        if (keep) hfa_fence_async_smem();                    // dp rows -> visible to the bulk store
        __syncwarp();                                        // every lane is done with stage `st`
        if (lane == 0) hfa_mbar_arrive(hfa_smem_u32(&empty[st]));
        if (++st == NST) {
            st = 0;
            phase ^= 1u;
        }
    }

#pragma unroll
    for (int k = 0; k < K; ++k) {
        if (owner && first + k == S - 1) ws.dp_last[2 * u] = dp[k];
        if (owner && first + k == S - 2) ws.dp_last[2 * u + 1] = dp[k];
    }
}

}  // namespace

template <bool DUMP, int MAXK>
static cudaError_t launch_any(const HfaLaunchCtx &c, size_t smem, const int32_t *order, int n, float *dp_dump)
{
    cudaError_t e = cudaFuncSetAttribute(hfa_dp_warp_any_kernel<DUMP, MAXK>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    hfa_dp_warp_any_kernel<DUMP, MAXK><<<n, 32, smem, c.stream>>>(c.ws, order, n, dp_dump);
    return cudaGetLastError();
}

// all warp-kernel classes in one launch; max_k = largest states-per-lane class present, ceil(Sp / 32) (the pair
// layout uses the shared-memory layout of its utterance's class), max_pair_k = largest pairs-per-lane class
cudaError_t hfa_launch_dp_warp_any(const HfaLaunchCtx &c, int max_k, int max_pair_k, const int32_t *order, int n,
                                   float *dp_dump)
{
    if (n <= 0) return cudaSuccess;
    if (max_k < 1 || max_k > 8 || max_pair_k < 0 || max_pair_k > HFA_PAIR_MAX_K) return cudaErrorInvalidValue;

    static const size_t bytes[9] = {0, hfa_warp_smem_bytes<1>(), hfa_warp_smem_bytes<2>(),
                                    hfa_warp_smem_bytes<3>(), hfa_warp_smem_bytes<4>(),
                                    hfa_warp_smem_bytes<5>(), hfa_warp_smem_bytes<6>(),
                                    hfa_warp_smem_bytes<7>(), hfa_warp_smem_bytes<8>()};
    size_t smem = (bytes[max_k] + 127) & ~(size_t)127;
    // HFA_DP_WARPS_PER_SM=n caps the resident warps per SM by padding the shared-memory request
    // (experiment knob; measured on config 4: flat from 13 warps per SM upwards)
    static const int cap = [] { const char *e = getenv("HFA_DP_WARPS_PER_SM"); return e ? atoi(e) : 0; }();
    if (cap > 0) smem = std::max(smem, ((size_t)(227 * 1024) / (size_t)cap - 1024) & ~(size_t)127);
    // (register-leaner variants compiled for the largest class present -- 72 registers for K <= 5 --
    // and 2 instead of 3 emission stages were measured on config 4: no gain, 0.465 vs 0.459 ms)
    if (dp_dump != nullptr) return launch_any<true, 8>(c, smem, order, n, dp_dump);
    return launch_any<false, 8>(c, smem, order, n, dp_dump);
}

// all utterances of the CTA-per-utterance list share one launch; max_sp = largest padded S among them
// (8 states per thread, one bar.sync per frame).  Round 1 also had a flag-synchronised wavefront variant of this
// kernel and a 2-states-per-thread "latency" variant: both lost to the strips of hfa_dp_skew.cu (config 3:
// 16.9 / 17.8 ms against 1.62 ms) and were removed in round 2.
cudaError_t hfa_launch_dp_cta(const HfaLaunchCtx &c, const int32_t *order, int n, int max_sp, float *dp_dump)
{
    if (n <= 0) return cudaSuccess;
    int threads = (max_sp + HFA_CTA_K - 1) / HFA_CTA_K;
    threads = ((threads + 31) / 32) * 32;
    if (threads > 1024) return cudaErrorInvalidValue;
    // frames per stage: largest power of two <= 16 whose stage stays under ~64 KB
    int tile_t = HFA_TILE_T;
    while (tile_t > 1 && (size_t)tile_t * max_sp * sizeof(float) > 64 * 1024) tile_t >>= 1;
    const int stage_floats = tile_t * max_sp;
    const size_t smem = (size_t)HFA_CTA_STAGES * stage_floats * sizeof(float) +
                        HFA_CTA_STAGES * HFA_TILE_T * sizeof(float2) +
                        HFA_CTA_STAGES * sizeof(uint64_t) + 2 * 32 * sizeof(float2);
    cudaError_t e;
#define HFA_CTA_LAUNCH(NT)                                                                         \
    e = cudaFuncSetAttribute(hfa_dp_cta_kernel<HFA_CTA_K, NT>,                                     \
                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);              \
    if (e != cudaSuccess) return e;                                                                \
    hfa_dp_cta_kernel<HFA_CTA_K, NT><<<n, threads, smem, c.stream>>>(c.ws, order, tile_t, stage_floats, dp_dump)
    if (threads <= 256) { HFA_CTA_LAUNCH(256); }
    else if (threads <= 512) { HFA_CTA_LAUNCH(512); }
    else { HFA_CTA_LAUNCH(1024); }
#undef HFA_CTA_LAUNCH
    return cudaGetLastError();
}

// banded kernel: items [item_begin, item_begin + n_items) of the plan's band table, one CTA each
template <int K, bool DUMP, bool KEEP, bool FUSED>
static cudaError_t launch_band(const HfaLaunchCtx &c, int item_begin, int n_items, int32_t *ticket,
                               float *dp_dump, int64_t row_stride)
{
    size_t smem = hfa_band_smem_bytes<K>();
    int lstage = 0;
    if (FUSED) {
        lstage = (int)(((int64_t)HFA_TILE_T * row_stride * 4 + 32 + 15) & ~(int64_t)15);
        smem = ((smem + 15) & ~(size_t)15) + HFA_FUSED_FIXED_BYTES + 2 * (size_t)lstage;
    }
    cudaError_t e = cudaFuncSetAttribute(hfa_dp_band_kernel<K, DUMP, KEEP, FUSED>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    hfa_dp_band_kernel<K, DUMP, KEEP, FUSED><<<n_items, 64, smem, c.stream>>>(c.ws, item_begin, ticket, dp_dump,
                                                                            c.vocab, lstage);
    return cudaGetLastError();
}

// keep_dp: the plan reserved a dp store for the utterances of this list (all or none).
// fused_row_stride > 0: compute the emissions inside the kernel from f32 logits whose rows are
// contiguous with at most this stride (requires keep_dp: nothing else holds what the backtrace needs)
cudaError_t hfa_launch_dp_band(const HfaLaunchCtx &c, int k, int item_begin, int n_items, int32_t *ticket,
                               bool keep_dp, int64_t fused_row_stride, float *dp_dump)
{
    if (n_items <= 0) return cudaSuccess;
    const bool fused = fused_row_stride > 0 && keep_dp && dp_dump == nullptr;
#define HFA_BAND_CASE(KK)                                                                              \
    case KK:                                                                                           \
        if (fused) return launch_band<KK, false, true, true>(c, item_begin, n_items, ticket, nullptr,  \
                                                             fused_row_stride);                        \
        if (dp_dump != nullptr)                                                                        \
            return keep_dp ? launch_band<KK, true, true, false>(c, item_begin, n_items, ticket, dp_dump, 0)   \
                           : launch_band<KK, true, false, false>(c, item_begin, n_items, ticket, dp_dump, 0); \
        return keep_dp ? launch_band<KK, false, true, false>(c, item_begin, n_items, ticket, dp_dump, 0)      \
                       : launch_band<KK, false, false, false>(c, item_begin, n_items, ticket, dp_dump, 0)
    switch (k) {
        HFA_BAND_CASE(2);
        HFA_BAND_CASE(4);
        HFA_BAND_CASE(8);
        default: return cudaErrorInvalidValue;
    }
#undef HFA_BAND_CASE
}
