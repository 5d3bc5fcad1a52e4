// hfa_backtrace.cu -- end state, backtrace, path rescoring, confidence and frame->interval, on device.
//
// Reference: tools/alignment_decoder.py:264-288 (end state, backward walk, frame_confidence),
// :97 (total_confidence), :104-113 (fractional boundary refinement, seconds).
//
// One warp per utterance, three phases:
//  1. backward walk over the bit-packed backpointers.  A word covers 16 frames of one state and the
//     path moves down at most 2 states per frame, so one 16-frame word-row only ever needs the 32
//     states below the state it was entered in: lane j keeps word(row, s_hi - j) in a register, the
//     walk is shuffle lookups + clz jumps from move to move, and the band of the next row (64 states
//     wide, it is not yet known where this row ends) is prefetched before the walk starts.
//  2. forward rescoring of the path.  The reference reads dp[t, s_t] out of the T x S matrix it kept;
//     we never store dp, and rebuild those T numbers bit-exactly from the path alone: on the best
//     path curr[] of the state being left equals the running max of its emissions since the path
//     entered it (0 for SP states, except that nothing is zeroed at t = 0).  Lanes gather the
//     per-frame operands in parallel, the f32/f64 chain itself runs once per frame (uniform).
//  3. segments -> seconds (f64), lane-parallel.
#include "hfa_common.cuh"

#define HFA_BT_WARPS 4

namespace {

__device__ __forceinline__ double seg_time(const float *p, int t, int T, double frame_length)
{
    // :83 edge_diff[t] = f64(f32(p[t+1] - p[t])), 0 for the last frame; :104 clip(diff / 2, +-0.5)
    double d = (t + 1 < T) ? (double)__fsub_rn(p[t + 1], p[t]) : 0.0;
    d = fmin(fmax(__dmul_rn(d, 0.5), -0.5), 0.5);
    return __dmul_rn(frame_length, __dadd_rn((double)(float)t, d));   // :105-108
}

// One 16-frame row of the backward walk, entered at state `cur` in its last frame `tt`.
// word(s) = backpointer word of state s in this row; bit f = "advanced by one at frame f", bit 16+f =
// "jumped over an SP".  The walk hops from move to move (clz); on_move(state, f) is called for every
// move met (latest first), on_span(state, f_lo, f_hi) for every run of frames spent in one state.
// Row 0 ends with the segment that frame 0 always opens (:277).  Returns the state the path has
// before the row's first frame.
template <typename FMove, typename FSpan>
__device__ __forceinline__ int hfa_walk_row(const uint32_t *__restrict__ row_words, int cur, int tt, bool row0,
                                            FMove on_move, FSpan on_span)
{
    while (tt >= 0) {
        const uint32_t wc = row_words[cur];
        uint32_t nz = (wc | (wc >> 16)) & 0xffffu & ((2u << tt) - 1u);
        if (row0) nz |= 1u;
        if (nz == 0u) {
            on_span(cur, 0, tt);
            break;
        }
        const int tp = 31 - __clz(nz);
        on_span(cur, tp, tt);
        on_move(cur, tp);
        if (row0 && tp == 0) break;
        cur -= ((wc >> (16 + tp)) & 1u) ? 2 : 1;
        tt = tp - 1;
    }
    return cur;
}

// Jump tables (latency plans): for every row w and every state s, where does a path that is in s at
// the row's last frame come from, and how many segments does it open on the way?  One thread per
// backpointer word; the serial part of the backtrace then takes ONE table lookup per 16 frames.
__global__ void __launch_bounds__(256)
hfa_jump_table_kernel(HfaWs ws)
{
    const int u = ws.jblk_utt[blockIdx.x];
    const HfaUtt m = ws.utt[u];
    const int n_rows = (m.T + 15) >> 4;
    const int64_t idx = (int64_t)(blockIdx.x - ws.jblk_first[u]) * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)n_rows * m.Sp) return;
    const int w = (int)(idx / m.Sp), s = (int)(idx - (int64_t)w * m.Sp);
    const int tt = (w == n_rows - 1) ? ((m.T - 1) & 15) : 15;
    int n_moves = 0;
    const int from = hfa_walk_row(ws.bp + m.bp_off + (int64_t)w * m.Sp, s, tt, false,
                                  [&](int, int) { ++n_moves; }, [](int, int, int) {});
    ws.jump[m.bp_off + idx] = (uint8_t)(s - from);
    ws.moves[m.bp_off + idx] = (uint8_t)n_moves;
}

__global__ void __launch_bounds__(HFA_BT_WARPS * 32)
hfa_backtrace_kernel(HfaWs ws, const int32_t *__restrict__ order, int n, HfaResultPtrs res,
                     float *__restrict__ frame_conf, float *__restrict__ dp_path,
                     double frame_length)
{
    __shared__ float4 stage_sm[HFA_BT_WARPS][32];
    __shared__ float dpath_sm[HFA_BT_WARPS][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int item = blockIdx.x * HFA_BT_WARPS + warp;
    if (item >= n) return;
    const int u = order[item];
    const HfaUtt m = ws.utt[u];
    if (m.status != 0) {                       // invalid utterance: report, produce nothing
        if (lane == 0) {
            res.status[u] = m.status;
            res.n_seg[u] = 0;
            res.end_state[u] = -1;
            res.final_score[u] = HFA_NEG_INF;
            res.total_conf[u] = __uint_as_float(0x7fc00000u);
        }
        return;
    }
    if (m.dp_off >= 0) return;                 // kept dp: hfa_backtrace_walk_kernel / hfa_backtrace_tables_kernel
    const int T = m.T, S = m.S, Sp = m.Sp;
    const int32_t *ids = ws.ids + m.seg_off;
    const uint32_t *bp = ws.bp + m.bp_off;
    int32_t *rev_idx = ws.rev_idx + m.seg_off;
    int32_t *rev_t = ws.rev_t + m.seg_off;
    int32_t *path_state = ws.path_state + m.frame_off;

    // ---- end state (:269-272) ----
    const float last1 = ws.dp_last[2 * u];
    const float last2 = (S >= 2) ? ws.dp_last[2 * u + 1] : HFA_NEG_INF;
    int s = S - 1;
    float final_score = last1;
    if (S >= 2 && last2 > last1 && ids[S - 1] == 0) {
        s = S - 2;
        final_score = last2;
    }
    const int s_end = s;

    // ---- phase 1: backward walk ----
    // Lane j holds word(row, s_hi - j) of the row being walked.  Rows are fetched LEAD rows ahead
    // as 64-state bands below the state the path has at fetch time: the path drops ~T/S... a few
    // states per 16-frame row, so LEAD rows later the wanted 32 states are almost always inside the
    // band (otherwise: one exposed reload).  This keeps the load latency off the serial walk.
    constexpr int LEAD = 4;
    const int n_rows = (T + 15) >> 4;
    int n_seg = 0;
    int s_hi = s;
    uint32_t q[LEAD][2];                                 // q[d]: band of row (w - 1 - d)
    int qref[LEAD];
    auto fetch = [&](int row, int ref, uint32_t (&w2)[2]) {
        w2[0] = w2[1] = 0u;
        if (row >= 0) {
            const uint32_t *r = bp + (int64_t)row * Sp;
            if (ref - lane >= 0) w2[0] = r[ref - lane];
            if (ref - lane - 32 >= 0) w2[1] = r[ref - lane - 32];
        }
    };
    uint32_t W = (s_hi - lane >= 0) ? bp[(int64_t)(n_rows - 1) * Sp + (s_hi - lane)] : 0u;
#pragma unroll
    for (int dd = 0; dd < LEAD; ++dd) {
        fetch(n_rows - 2 - dd, s_hi, q[dd]);
        qref[dd] = s_hi;
    }
    for (int w = n_rows - 1; w >= 0; --w) {
        uint32_t f[2];
        fetch(w - 1 - LEAD, s_hi, f);                    // LEAD rows ahead, below the current state
        const int fref = s_hi;
        int tt = (w == n_rows - 1) ? ((T - 1) & 15) : 15;
        int my_state = 0;
        while (tt >= 0) {
            const uint32_t wc = __shfl_sync(0xffffffffu, W, (s_hi - s) & 31);
            uint32_t nz = (wc | (wc >> 16)) & 0xffffu & ((2u << tt) - 1u);
            if (w == 0) nz |= 1u;                       // frame 0 always opens a segment (:277)
            if (nz == 0u) {
                if (lane <= tt) my_state = s;
                break;
            }
            const int tp = 31 - __clz(nz);              // latest frame <= tt where the path moved
            if (lane <= tt && lane >= tp) my_state = s;
            if (lane == 0 && n_seg < S) {
                rev_idx[n_seg] = s;
                rev_t[n_seg] = 16 * w + tp;
            }
            ++n_seg;
            if (w == 0 && tp == 0) break;
            s -= ((wc >> (16 + tp)) & 1u) ? 2 : 1;
            tt = tp - 1;
        }
        if (lane < 16 && 16 * w + lane < T) path_state[16 * w + lane] = my_state;
        if (w > 0) {
            const int o = (qref[0] - s) + lane;         // offset of state (s - lane) inside band q[0]
            if (qref[0] - s + 31 < 64) {                 // warp-uniform: the band covers it
                const uint32_t x0 = __shfl_sync(0xffffffffu, q[0][0], o & 31);
                const uint32_t x1 = __shfl_sync(0xffffffffu, q[0][1], o & 31);
                W = (o < 32) ? x0 : x1;
            } else {                                     // the path dropped > 32 states in LEAD rows
                W = (s - lane >= 0) ? bp[(int64_t)(w - 1) * Sp + (s - lane)] : 0u;
            }
            s_hi = s;
#pragma unroll
            for (int dd = 0; dd + 1 < LEAD; ++dd) {
                q[dd][0] = q[dd + 1][0];
                q[dd][1] = q[dd + 1][1];
                qref[dd] = qref[dd + 1];
            }
            q[LEAD - 1][0] = f[0];
            q[LEAD - 1][1] = f[1];
            qref[LEAD - 1] = fref;
        }
    }
    if (n_seg > S) n_seg = S;                           // cannot happen with valid backpointers
    __syncwarp();

    // ---- phase 2: forward rescoring, frame confidence ----
    // 32 frames per round: lanes gather the operands of their frame (software-pipelined: path
    // states two rounds ahead, emissions one round ahead), then the f32/f64 chain itself runs once
    // per frame, uniformly, over operands parked in shared memory.
    double log_sum = 0.0;
    {
    const float *emis = ws.emis + m.emis_off;
    const float2 *edge2 = ws.edge2 + m.edge_off;
    const double ratio = __ddiv_rn((double)T, (double)S);
    const bool lead_sp = (ids[0] == 0) && (S > 1);
    // emission rows: plain [T][Sp], or compacted to one column per distinct id (HfaWs::colmap)
    const bool compact = m.Dp > 0 && ws.emis_mode[u] != 0;
    const int Ep = compact ? m.Dp : Sp;
    const uint8_t *cmap = ws.colmap + m.seg_off;
    float4 *stage = stage_sm[warp];
    float *dpath = dpath_sm[warp];
    float d = 0.0f, cu = 0.0f, carry_d = 0.0f;          // dp_path[-1] := 0 (:286)
    const int n_rounds = (T + 31) >> 5;
    auto load_state = [&](int round) {
        const int t = round * 32 + lane;
        return (round < n_rounds && t < T) ? path_state[t] : 0;
    };
    // flags: 1 = the path moved into this frame's state, 2 = that state is an id-0 (SP) state,
    //        4 = frame past T (no-op), 8 = frame 0 (seed, :250-254)
    // Raw operands of one frame: nothing here touches a loaded value, so the loads stay in flight
    // until `finish` turns them into the staged tuple two rounds later.
    struct Raw { float x, y; float2 ed; int id, st, sprev; };
    auto gather = [&](int round, int st, int sprev) {
        const int t = min(round * 32 + lane, T - 1);         // clamped: always a valid address
        const float *row = emis + (int64_t)t * Ep;
        Raw g;
        g.x = hfa_ldg_f32_64B(row + (compact ? (int)cmap[st] : st));
        g.y = hfa_ldg_f32_64B(row + (compact ? (int)cmap[sprev] : sprev));
        g.ed = edge2[t];
        g.id = ids[st];
        g.st = st;
        g.sprev = sprev;
        return g;
    };
    auto finish = [&](int round, const Raw &g) {
        const int t = round * 32 + lane;
        float4 v = make_float4(0.f, 0.f, 0.f, __int_as_float(4));
        if (t < T) {
            const bool moved = (t > 0) && (g.sprev != g.st);
            v.x = g.x;
            v.y = g.y;
            v.z = moved ? g.ed.x : g.ed.y;
            int fl = (moved ? 1 : 0) | ((g.id == 0) ? 2 : 0);
            if (t == 0) {
                const bool seeded = (g.st == 0) || (g.st == 1 && lead_sp);
                v.x = seeded ? v.x : HFA_NEG_INF;
                fl = 8;
            }
            v.w = __int_as_float(fl);
        }
        return v;
    };
    // software pipeline: path states three rounds ahead, gathered operands two rounds ahead
    int st_a = load_state(0), st_b = load_state(1), st_c = load_state(2);
    Raw g_cur = gather(0, st_a, __shfl_up_sync(0xffffffffu, st_a, 1));
    Raw g_nxt;
    {
        int sp1 = __shfl_up_sync(0xffffffffu, st_b, 1);
        const int last0 = __shfl_sync(0xffffffffu, st_a, 31);
        if (lane == 0) sp1 = last0;
        g_nxt = gather(1, st_b, sp1);
    }
    for (int r = 0; r < n_rounds; ++r) {
        // issue the loads of the following rounds before touching this round's results
        const int st_d = load_state(r + 3);
        int sp2 = __shfl_up_sync(0xffffffffu, st_c, 1);
        const int last1 = __shfl_sync(0xffffffffu, st_b, 31);
        if (lane == 0) sp2 = last1;
        const Raw g_nn = gather(r + 2, st_c, sp2);
        const float4 v_cur = finish(r, g_cur);

        stage[lane] = v_cur;
        // frames that are not a plain "stay" (moved / seed / past T): one bit per frame, uniform
        const uint32_t special = __ballot_sync(0xffffffffu, (__float_as_int(v_cur.w) & 13) != 0);
        __syncwarp();
        // Runs of stay frames are a pure two-add chain (curr: running max, or 0 in an SP state, which
        // is constant over a run); only the frames flagged in `special` take the branchy path.
        int j = 0;
        while (j < 32) {
            if ((special >> j) & 1u) {
                const float4 q = stage[j];
                const int fl = __float_as_int(q.w);
                if (fl & 1) {
                    d = hfa_advance(__fadd_rn(__fadd_rn(d, q.y), q.z), cu, ratio);
                    cu = (fl & 2) ? 0.0f : q.x;
                } else if (fl & 8) {
                    d = q.x;
                    cu = d;
                }
                if (lane == 0) dpath[j] = d;
                ++j;
                continue;
            }
            const uint32_t rest = special >> j;
            const int run = rest ? (__ffs(rest) - 1) : (32 - j);
            const bool sp_state = (__float_as_int(stage[j].w) & 2) != 0;
            int k = 0;
            for (; k + 4 <= run; k += 4) {
                const float4 q0 = stage[j + k], q1 = stage[j + k + 1], q2 = stage[j + k + 2],
                             q3 = stage[j + k + 3];
                const float d0 = __fadd_rn(__fadd_rn(d, q0.x), q0.z);
                const float d1 = __fadd_rn(__fadd_rn(d0, q1.x), q1.z);
                const float d2 = __fadd_rn(__fadd_rn(d1, q2.x), q2.z);
                d = __fadd_rn(__fadd_rn(d2, q3.x), q3.z);
                cu = fmaxf(fmaxf(cu, q0.x), fmaxf(fmaxf(q1.x, q2.x), q3.x));
                if (lane == 0) {
                    dpath[j + k] = d0; dpath[j + k + 1] = d1; dpath[j + k + 2] = d2; dpath[j + k + 3] = d;
                }
            }
            for (; k < run; ++k) {
                const float4 q = stage[j + k];
                d = __fadd_rn(__fadd_rn(d, q.x), q.z);
                cu = fmaxf(cu, q.x);
                if (lane == 0) dpath[j + k] = d;
            }
            if (sp_state) cu = 0.0f;
            j += run;
        }
        __syncwarp();
        const int t = r * 32 + lane;
        if (t < T) {
            const float cur = dpath[lane];
            const float prev = (lane == 0) ? carry_d : dpath[lane - 1];
            const float fc = expf(__fsub_rn(cur, prev));                 // :284-288
            if (frame_conf != nullptr) frame_conf[m.frame_off + t] = fc;
            if (dp_path != nullptr) dp_path[m.frame_off + t] = cur;
            log_sum += (double)logf(__fadd_rn(fc, 1e-6f));               // :97
        }
        carry_d = d;
        __syncwarp();
        st_b = st_c;
        st_c = st_d;
        g_cur = g_nxt;
        g_nxt = g_nn;
    }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) log_sum += __shfl_xor_sync(0xffffffffu, log_sum, o);
    const float mean = (float)(log_sum / (double)T);
    const float total = expf(__fdiv_rn(mean, 3.0f));

    // ---- phase 3: segments in forward order, seconds ----
    const float *p = ws.edge_p + m.edge_off;
    int32_t *out_idx = res.ph_idx_seq + m.seg_off;
    int32_t *out_t = res.ph_time_int + m.seg_off;
    double *out_iv = res.intervals + 2 * m.seg_off;
    for (int k = lane; k < n_seg; k += 32) {
        const int tk = rev_t[n_seg - 1 - k];
        out_idx[k] = rev_idx[n_seg - 1 - k];
        out_t[k] = tk;
        out_iv[2 * k] = seg_time(p, tk, T, frame_length);
        out_iv[2 * k + 1] = (k + 1 < n_seg) ? seg_time(p, rev_t[n_seg - 2 - k], T, frame_length)
                                            : __dmul_rn(frame_length, (double)T);
    }
    if (lane == 0) {
        res.status[u] = (final_score == HFA_NEG_INF) ? 4 : 0;
        res.n_seg[u] = n_seg;
        res.end_state[u] = s_end;
        res.final_score[u] = final_score;
        res.total_conf[u] = total;
    }
}

// ---------------------------------------------------------------------------------------------
// Backtrace of the utterances whose forward pass kept dp (latency plans): ONE CTA per utterance.
// Everything except the row-to-row chain is data parallel; the kernel is bound by the number of
// dependent memory round trips, so every phase is as wide as the CTA:
//   1a (warp 0)  entry state of every 16-frame row: one jump-table lookup per row, 16 rows per round
//                (lane l prefetches jump[w - r][s - l] and jump[w - r][s - l - 32] for the next 16 rows,
//                the rows are then chained with shuffles);
//   1b (thread = row)  segment counts from the move table, a CTA-wide scan for their positions, then
//                every thread re-walks its own row, writes its segments straight in forward order and
//                gathers dp[t, s_t] of its 16 frames;
//   2  (thread = frame)  frame confidence, log-sum;   3 (thread = segment)  seconds.
// ---------------------------------------------------------------------------------------------
#define HFA_BTT_THREADS 256
#define HFA_BTW_CHUNKS 8         // bulk copies (and mbarriers) the walk kernel stages an utterance's words in

// Phases 2 and 3 of the kept-dp backtraces, for a CTA of HFA_BTT_THREADS threads: frame confidence, log-sum and
// total confidence from dp[t, s_t] (dp_at(t)), segment seconds from the segment frames in forward order
// (seg_t(k)), then the utterance's scalar results.  Both kernels call this, so their results are the same bits.
template <typename FDp, typename FSegT>
__device__ __forceinline__ void hfa_bt_finish(const HfaUtt &m, int u, int n_seg, int s_end, float final_score,
                                              const float *p, const HfaResultPtrs &res, float *frame_conf,
                                              float *dp_path, double frame_length, double *warp_log, FDp dp_at,
                                              FSegT seg_t)
{
    constexpr int NW = HFA_BTT_THREADS / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int T = m.T;

    // ---- 2: frame confidence (:284-288), total confidence (:97) ----
    double log_sum = 0.0;
    for (int t = tid; t < T; t += HFA_BTT_THREADS) {
        const float cur = dp_at(t);
        const float prev = (t > 0) ? dp_at(t - 1) : 0.0f;          // dp_path[-1] := 0 (:286)
        const float fc = expf(__fsub_rn(cur, prev));
        if (frame_conf != nullptr) frame_conf[m.frame_off + t] = fc;
        if (dp_path != nullptr) dp_path[m.frame_off + t] = cur;
        log_sum += (double)logf(__fadd_rn(fc, 1e-6f));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) log_sum += __shfl_xor_sync(0xffffffffu, log_sum, o);
    if (lane == 0) warp_log[warp] = log_sum;

    // ---- 3: segments -> seconds ----
    double *out_iv = res.intervals + 2 * m.seg_off;
    for (int k = tid; k < n_seg; k += HFA_BTT_THREADS) {
        out_iv[2 * k] = seg_time(p, seg_t(k), T, frame_length);
        out_iv[2 * k + 1] = (k + 1 < n_seg) ? seg_time(p, seg_t(k + 1), T, frame_length)
                                            : __dmul_rn(frame_length, (double)T);
    }
    __syncthreads();
    if (tid == 0) {
        double tot = 0.0;
        for (int q = 0; q < NW; ++q) tot += warp_log[q];
        const float mean = (float)(tot / (double)T);
        res.status[u] = (final_score == HFA_NEG_INF) ? 4 : 0;
        res.n_seg[u] = n_seg;
        res.end_state[u] = s_end;
        res.final_score[u] = final_score;
        res.total_conf[u] = expf(__fdiv_rn(mean, 3.0f));
    }
}


__global__ void __launch_bounds__(HFA_BTT_THREADS)
hfa_backtrace_tables_kernel(HfaWs ws, const int32_t *__restrict__ order, int n, HfaResultPtrs res,
                            float *__restrict__ frame_conf, float *__restrict__ dp_path, double frame_length)
{
    constexpr int NW = HFA_BTT_THREADS / 32;
    __shared__ int warp_sum[NW];
    __shared__ double warp_log[NW];
    __shared__ int carry_sm;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int u = order[blockIdx.x];
    const HfaUtt m = ws.utt[u];
    if (m.status != 0 || m.dp_off < 0) return;
    const int T = m.T, S = m.S, Sp = m.Sp;
    const int32_t *ids = ws.ids + m.seg_off;
    const uint32_t *bp = ws.bp + m.bp_off;
    int32_t *path_state = ws.path_state + m.frame_off;
    int32_t *out_idx = res.ph_idx_seq + m.seg_off;
    int32_t *out_t = res.ph_time_int + m.seg_off;
    const int n_rows = (T + 15) >> 4;
    int32_t *entry = ws.row_entry + m.edge_off / HFA_TILE_T;

    // ---- end state (:269-272) ----
    const float last1 = ws.dp_last[2 * u];
    const float last2 = (S >= 2) ? ws.dp_last[2 * u + 1] : HFA_NEG_INF;
    int s_end = S - 1;
    float final_score = last1;
    if (S >= 2 && last2 > last1 && ids[S - 1] == 0) {
        s_end = S - 2;
        final_score = last2;
    }

    // ---- 1a ----
    if (warp == 0) {
        const uint8_t *J = ws.jump + m.bp_off;
        int sr = s_end;
        int w = n_rows - 1;
        while (w >= 0) {
            uint32_t c0[16], c1[16];
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const bool row_ok = w - r >= 1;                  // row 0 has no predecessor row
                c0[r] = (row_ok && sr - lane >= 0) ? J[(int64_t)(w - r) * Sp + (sr - lane)] : 0u;
                c1[r] = (row_ok && sr - lane - 32 >= 0) ? J[(int64_t)(w - r) * Sp + (sr - lane - 32)] : 0u;
            }
            const int s_ref = sr;
            int done = 0;
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const int d = s_ref - sr;
                if (w - r < 0 || d >= 64) break;                 // uniform: out of rows / out of the band
                if (lane == 0) entry[w - r] = sr;
                const uint32_t x0 = __shfl_sync(0xffffffffu, c0[r], d & 31);
                const uint32_t x1 = __shfl_sync(0xffffffffu, c1[r], d & 31);
                sr -= (int)(d < 32 ? x0 : x1);
                ++done;
            }
            w -= done;
        }
    }
    if (tid == 0) carry_sm = 0;
    __syncthreads();

    // ---- 1b ----
    const uint8_t *M = ws.moves + m.bp_off;
    const float *dps = ws.dp_store + m.dp_off;
    for (int base = 0; base < n_rows; base += HFA_BTT_THREADS) {
        const int wr = base + tid;
        int e = 0, c = 0;
        if (wr < n_rows) {
            e = entry[wr];
            c = (int)M[(int64_t)wr * Sp + e] + (wr == 0 ? 1 : 0);
        }
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        int pos = carry_sm + incl;                               // segments of the rows <= wr
        for (int q = 0; q < warp; ++q) pos += warp_sum[q];
        __syncthreads();
        if (tid == HFA_BTT_THREADS - 1) carry_sm = pos;
        if (wr < n_rows) {
            const int tt = (wr == n_rows - 1) ? ((T - 1) & 15) : 15;
            hfa_walk_row(bp + (int64_t)wr * Sp, e, tt, wr == 0,
                         [&](int st, int f) {
                             --pos;
                             if (pos < S) {
                                 out_idx[pos] = st;
                                 out_t[pos] = 16 * wr + f;
                             }
                         },
                         [&](int st, int f_lo, int f_hi) {
                             for (int f = f_lo; f <= f_hi; ++f) path_state[16 * wr + f] = st;
                         });
            // dp[t, s_t] of the row's frames: sixteen independent gathers, parked where the
            // per-frame state was (phase 2 only needs the dp values)
            float dv[16];
#pragma unroll
            for (int f = 0; f < 16; ++f) {
                const int t = min(16 * wr + f, T - 1);
                dv[f] = hfa_ldg_f32_64B(dps + (m.skew_d > 0 ? hfa_skew_dp_index(m.skew_d, T, t, path_state[t])
                                                            : hfa_dp_store_index(m.band_k, T, t, path_state[t])));
            }
#pragma unroll
            for (int f = 0; f < 16; ++f)
                if (16 * wr + f < T) path_state[16 * wr + f] = __float_as_int(dv[f]);
        }
        __syncthreads();
    }
    const int n_seg = min(carry_sm, S);
    hfa_bt_finish(m, u, n_seg, s_end, final_score, ws.edge_p + m.edge_off, res, frame_conf, dp_path, frame_length,
                  warp_log, [&](int t) { return __int_as_float(path_state[t]); }, [&](int k) { return out_t[k]; });
}

// ---------------------------------------------------------------------------------------------
// Backtrace of the kept-dp utterances whose backpointers fit in shared memory: ONE CTA per utterance,
// no jump tables.  The utterance's ceil(T/16) x Sp backpointer words are staged by bulk copies, last
// rows first (one mbarrier per chunk of rows), and warp 0 walks the path from move to move straight out
// of shared memory (hfa_walk_row: one LDS + clz per move, one per row without a move), all 32 lanes in
// lock step: lane f writes the state of frame f of the row.  Then every thread gathers dp[t, s_t] of its
// frames and hfa_bt_finish does the rest exactly as in the table backtrace.
// Dynamic shared memory (hfa_bt_walk_smem): [n_rows][Sp] words, [16 n_rows] frame state -> dp bits,
// [S] segment states and [S] segment frames in backward order.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(HFA_BTT_THREADS)
hfa_backtrace_walk_kernel(HfaWs ws, const int32_t *__restrict__ order, HfaResultPtrs res,
                          float *__restrict__ frame_conf, float *__restrict__ dp_path, double frame_length)
{
    constexpr int NW = HFA_BTT_THREADS / 32;
    extern __shared__ __align__(16) unsigned char walk_sm[];
    __shared__ __align__(8) uint64_t bars[HFA_BTW_CHUNKS];
    __shared__ double warp_log[NW];
    __shared__ int n_seg_sm;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int u = order[blockIdx.x];
    const HfaUtt m = ws.utt[u];                  // the planner sends valid utterances with kept dp only
    const int T = m.T, S = m.S, Sp = m.Sp;
    const int n_rows = (T + 15) >> 4;
    const uint32_t *words = reinterpret_cast<const uint32_t *>(walk_sm);
    int32_t *fr = reinterpret_cast<int32_t *>(walk_sm + (size_t)n_rows * Sp * 4);
    int32_t *rev_idx = fr + 16 * n_rows;
    int32_t *rev_t = rev_idx + S;
    const int rows_per = (n_rows + HFA_BTW_CHUNKS - 1) / HFA_BTW_CHUNKS;
    const uint32_t bar0 = hfa_smem_u32(bars);

    if (tid == 0) {
        for (int c = 0; c < HFA_BTW_CHUNKS; ++c) hfa_mbar_init(bar0 + 8 * c, 1);
        hfa_fence_mbar_init();
        // chunk c = rows [hi - rows_per, hi), hi = n_rows - c rows_per: the walk needs the last rows first
        for (int c = 0; c * rows_per < n_rows; ++c) {
            const int hi = n_rows - c * rows_per, lo = max(hi - rows_per, 0);
            const uint32_t bytes = (uint32_t)(hi - lo) * Sp * 4;
            hfa_mbar_expect_tx(bar0 + 8 * c, bytes);
            hfa_bulk_load(hfa_smem_u32(words) + (uint32_t)lo * Sp * 4, ws.bp + m.bp_off + (int64_t)lo * Sp, bytes,
                          bar0 + 8 * c);
        }
    }

    // ---- end state (:269-272) ----
    const int32_t *ids = ws.ids + m.seg_off;
    const float last1 = ws.dp_last[2 * u];
    const float last2 = (S >= 2) ? ws.dp_last[2 * u + 1] : HFA_NEG_INF;
    int s_end = S - 1;
    float final_score = last1;
    if (S >= 2 && last2 > last1 && ids[S - 1] == 0) {
        s_end = S - 2;
        final_score = last2;
    }
    __syncthreads();                             // the barriers are initialised

    // ---- 1: the walk (warp 0) ----
    if (warp == 0) {
        int cur = s_end, n_seg = 0, c = 0;
        hfa_mbar_wait(bar0, 0, HFA_POLLS_COPY);
        for (int w = n_rows - 1; w >= 0; --w) {
            if (w < n_rows - (c + 1) * rows_per) {
                ++c;
                hfa_mbar_wait(bar0 + 8 * c, 0, HFA_POLLS_COPY);
            }
            const int tt = (w == n_rows - 1) ? ((T - 1) & 15) : 15;
            cur = hfa_walk_row(words + (size_t)w * Sp, cur, tt, w == 0,
                               [&](int st, int f) {
                                   if (lane == 0 && n_seg < S) {
                                       rev_idx[n_seg] = st;
                                       rev_t[n_seg] = 16 * w + f;
                                   }
                                   ++n_seg;
                               },
                               [&](int st, int f_lo, int f_hi) {
                                   if (lane >= f_lo && lane <= f_hi) fr[16 * w + lane] = st;
                               });
        }
        if (lane == 0) n_seg_sm = min(n_seg, S);   // n_seg > S cannot happen with valid backpointers
    }
    __syncthreads();
    const int n_seg = n_seg_sm;

    // ---- dp[t, s_t] in place of s_t, segments in forward order ----
    const float *dps = ws.dp_store + m.dp_off;
    constexpr int G = 8;                         // independent gathers in flight per thread
    for (int base = 0; base < T; base += G * HFA_BTT_THREADS) {
        float dv[G];
#pragma unroll
        for (int j = 0; j < G; ++j) {
            const int t = min(base + j * HFA_BTT_THREADS + tid, T - 1);
            const int st = fr[t];
            dv[j] = hfa_ldg_f32_64B(dps + (m.skew_d > 0 ? hfa_skew_dp_index(m.skew_d, T, t, st)
                                                        : hfa_dp_store_index(m.band_k, T, t, st)));
        }
        __syncthreads();                         // every state of this batch is read before any is replaced
#pragma unroll
        for (int j = 0; j < G; ++j) {
            const int t = base + j * HFA_BTT_THREADS + tid;
            if (t < T) fr[t] = __float_as_int(dv[j]);
        }
    }
    int32_t *out_idx = res.ph_idx_seq + m.seg_off;
    int32_t *out_t = res.ph_time_int + m.seg_off;
    for (int k = tid; k < n_seg; k += HFA_BTT_THREADS) {
        out_idx[k] = rev_idx[n_seg - 1 - k];
        out_t[k] = rev_t[n_seg - 1 - k];
    }
    __syncthreads();
    hfa_bt_finish(m, u, n_seg, s_end, final_score, ws.edge_p + m.edge_off, res, frame_conf, dp_path, frame_length,
                  warp_log, [&](int t) { return __int_as_float(fr[t]); },
                  [&](int k) { return rev_t[n_seg - 1 - k]; });
}

// test helper: unpack one utterance's backpointers to int8 [T][S] (row 0 = -1, :247)
__global__ void hfa_unpack_bp_kernel(HfaWs ws, int u, int8_t *__restrict__ out)
{
    const HfaUtt m = ws.utt[u];
    const int64_t n = (int64_t)m.T * m.S;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int t = (int)(i / m.S), s = (int)(i - (int64_t)t * m.S);
        const uint32_t w = ws.bp[m.bp_off + (int64_t)(t >> 4) * m.Sp + s];
        const int b = t & 15;
        const int code = ((w >> (16 + b)) & 1u) ? 2 : (int)((w >> b) & 1u);
        out[i] = (int8_t)((t == 0) ? -1 : code);
    }
}

// test helper: the dp the forward pass kept for one utterance (latency plans), as f32 [T][S]
__global__ void hfa_unpack_dp_kernel(HfaWs ws, int u, float *__restrict__ out)
{
    const HfaUtt m = ws.utt[u];
    const float *dps = ws.dp_store + m.dp_off;
    const int64_t n = (int64_t)m.T * m.S;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int t = (int)(i / m.S), s = (int)(i - (int64_t)t * m.S);
        out[i] = dps[m.skew_d > 0 ? hfa_skew_dp_index(m.skew_d, m.T, t, s) : hfa_dp_store_index(m.band_k, m.T, t, s)];
    }
}

}  // namespace

cudaError_t hfa_launch_unpack_dp(const HfaLaunchCtx &c, int utt, float *out)
{
    hfa_unpack_dp_kernel<<<148, 256, 0, c.stream>>>(c.ws, utt, out);
    return cudaGetLastError();
}

cudaError_t hfa_launch_backtrace(const HfaLaunchCtx &c, const int32_t *order, int n,
                                 const HfaResultPtrs &res, float *frame_conf, float *dp_path)
{
    if (n <= 0) return cudaSuccess;
    const int blocks = (n + HFA_BT_WARPS - 1) / HFA_BT_WARPS;
    hfa_backtrace_kernel<<<blocks, HFA_BT_WARPS * 32, 0, c.stream>>>(c.ws, order, n, res, frame_conf,
                                                                    dp_path, c.frame_length);
    return cudaGetLastError();
}

cudaError_t hfa_launch_jump_tables(const HfaLaunchCtx &c, int n_blocks)
{
    if (n_blocks <= 0) return cudaSuccess;
    hfa_jump_table_kernel<<<n_blocks, 256, 0, c.stream>>>(c.ws);
    return cudaGetLastError();
}

// one CTA per utterance of the list; utterances without kept dp are left to hfa_launch_backtrace
cudaError_t hfa_launch_backtrace_tables(const HfaLaunchCtx &c, const int32_t *order, int n,
                                        const HfaResultPtrs &res, float *frame_conf, float *dp_path)
{
    if (n <= 0) return cudaSuccess;
    hfa_backtrace_tables_kernel<<<n, HFA_BTT_THREADS, 0, c.stream>>>(c.ws, order, n, res, frame_conf, dp_path,
                                                                    c.frame_length);
    return cudaGetLastError();
}

cudaError_t hfa_launch_backtrace_walk(const HfaLaunchCtx &c, const int32_t *order, int n, int64_t smem,
                                      const HfaResultPtrs &res, float *frame_conf, float *dp_path)
{
    if (n <= 0) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(hfa_backtrace_walk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return e;
    hfa_backtrace_walk_kernel<<<n, HFA_BTT_THREADS, (size_t)smem, c.stream>>>(c.ws, order, res, frame_conf, dp_path,
                                                                             c.frame_length);
    return cudaGetLastError();
}

cudaError_t hfa_launch_unpack_bp(const HfaLaunchCtx &c, int utt, int8_t *out)
{
    hfa_unpack_bp_kernel<<<148, 256, 0, c.stream>>>(c.ws, utt, out);
    return cudaGetLastError();
}
