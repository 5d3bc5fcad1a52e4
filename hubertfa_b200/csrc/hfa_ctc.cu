// hfa_ctc.cu -- greedy CTC decode on the device, and the per-frame path state of an aligned batch.
//
// Reference: AlignmentDecoder.ctc(), tools/alignment_decoder.py:145-150 (used by validation_step,
// networks/task/forced_alignment.py:413):
//     ctc = argmax(ctc_logits, -1);  keep frame t iff ctc[t] != ctc[t-1] (ctc[-1] := 0) and ctc[t] != 0
// One utterance (hfa_ctc_greedy_kernel): one CTA, every warp takes frames round-robin for the argmax (first
// maximum wins, like numpy), then the CTA compacts the kept ids in frame order with a running prefix sum.
// A ragged batch (hfa_ctc_batch_kernel): the frames of the whole batch are spread over the grid, one CTA per
// 64-frame row block of the plan, so that a batch of very different T keeps every SM streaming logits; the
// last CTA to finish an utterance compacts it.  Index work: bit-exact.
//
// AlignmentDecoder.plot(), :152-168, builds the state the best path occupies at every frame with a cumsum over
// the segments; hfa_frame_state_kernel writes the same from the result blob, one thread per frame.
#include "../../include/hfa_align.h"
#include "hfa_common.cuh"

namespace {

constexpr int HFA_CTC_THREADS = 1024;
constexpr int HFA_CTC_BATCH_THREADS = 256;                       // one CTA per row block of HFA_EMIS_ROWS frames
constexpr int HFA_CTC_ROWS_PER_WARP = HFA_EMIS_ROWS / (HFA_CTC_BATCH_THREADS / 32);
constexpr int HFA_CTC_ROWS_IN_FLIGHT = 4;                        // rows one warp reads at once (memory parallelism)
constexpr int HFA_CTC_FRAMES_PER_THREAD = 4;                     // compaction: consecutive frames per thread

// argmax over the V columns of R rows, one warp, every lane gets the results.  f32 compare after .float()
// (:77), ties -> the lowest index, an all -inf row -> 0.  Each lane reads its columns lane, lane + 32, ... in
// groups of U for all R rows at once, so that R * U loads are in flight per lane before the first compare; the
// compares then run in column order, so each row's result depends on neither R nor U.
template <typename TIn, int R, int U = 4>
__device__ __forceinline__ void hfa_warp_row_argmax(const TIn *const (&row)[R], int V, int64_t st_v, int lane,
                                                    int (&out)[R])
{
    float best[R];
    int bi[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        best[r] = HFA_NEG_INF;
        bi[r] = 0x7fffffff;
    }
    for (int v0 = lane; v0 < V; v0 += 32 * U) {
        float x[U][R];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int v = v0 + 32 * j;
#pragma unroll
            for (int r = 0; r < R; ++r) x[j][r] = (v < V) ? hfa_to_float<TIn>(row[r][(int64_t)v * st_v]) : 0.0f;
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int v = v0 + 32 * j;
            if (v < V) {
#pragma unroll
                for (int r = 0; r < R; ++r)
                    if (x[j][r] > best[r] || bi[r] == 0x7fffffff) {   // the first element always enters (all -inf rows -> 0)
                        best[r] = x[j][r];
                        bi[r] = v;
                    }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best[r], o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi[r], o);
            if (oi != 0x7fffffff && (bi[r] == 0x7fffffff || ob > best[r] || (ob == best[r] && oi < bi[r]))) {
                best[r] = ob;
                bi[r] = oi;
            }
        }
        out[r] = bi[r];
    }
}

template <typename TIn>
__global__ void __launch_bounds__(HFA_CTC_THREADS)
hfa_ctc_greedy_kernel(const TIn *__restrict__ logits, int T, int V, int64_t st_t, int64_t st_v,
                      int32_t *__restrict__ arg, int32_t *__restrict__ out_ids, int32_t *__restrict__ out_len)
{
    __shared__ int warp_sum[HFA_CTC_THREADS / 32];
    __shared__ int carry_sm;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // 1. argmax per frame
    for (int t = warp; t < T; t += HFA_CTC_THREADS / 32) {
        const TIn *row[1] = {logits + (int64_t)t * st_t};
        int bi[1];
        hfa_warp_row_argmax<TIn, 1>(row, V, st_v, lane, bi);
        if (lane == 0) arg[t] = bi[0];
    }
    if (tid == 0) carry_sm = 0;
    __syncthreads();
    // 2. keep / compact in frame order
    for (int base = 0; base < T; base += HFA_CTC_THREADS) {
        const int t = base + tid;
        int id = 0, keep = 0;
        if (t < T) {
            id = arg[t];
            const int prev = (t > 0) ? arg[t - 1] : 0;
            keep = (id != prev && id != 0) ? 1 : 0;
        }
        int incl = keep;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        int pos = carry_sm + incl;
        for (int q = 0; q < warp; ++q) pos += warp_sum[q];
        __syncthreads();
        if (keep) out_ids[pos - 1] = id;
        if (tid == HFA_CTC_THREADS - 1) carry_sm = pos;
        __syncthreads();
    }
    if (tid == 0) *out_len = carry_sm;
}

// One CTA per row block (the plan's HfaWs::block_utt / row_blocks: 64 frames of one valid utterance).
//  1. every warp takes 8 consecutive frames, 4 rows in flight, and stores their argmax into arg (= scratch) at
//     the utterance's frame offset;
//  2. thread 0 adds the block's frame count to out_len[u], zeroed before the launch.  The CTA whose addition
//     reaches T owns the utterance: every other block of it has published its argmax (barrier, then a fence
//     before the add), so it reads arg[] back through L2 and compacts the kept ids into out_ids in frame order
//     (a CTA-wide prefix sum over 1024 frames per pass), then overwrites out_len[u] with the count.
// Utterances the plan did not accept have no row block: their out_len stays 0.
template <typename TIn>
__global__ void __launch_bounds__(HFA_CTC_BATCH_THREADS)
hfa_ctc_batch_kernel(HfaWs ws, const HfaCtcDesc *__restrict__ table, int V, int32_t *__restrict__ arg,
                     int32_t *__restrict__ out_ids, int32_t *__restrict__ out_len)
{
    constexpr int NW = HFA_CTC_BATCH_THREADS / 32;
    constexpr int RPW = HFA_CTC_ROWS_PER_WARP, RIF = HFA_CTC_ROWS_IN_FLIGHT, FPT = HFA_CTC_FRAMES_PER_THREAD;
    __shared__ int warp_sum[NW];
    __shared__ int last_sm;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int u = ws.block_utt[blockIdx.x];
    const int T = ws.utt[u].T;
    const int64_t f0 = ws.utt[u].frame_off;
    const int t_base = (blockIdx.x - ws.row_blocks[u]) * HFA_EMIS_ROWS;
    const int rows = min(HFA_EMIS_ROWS, T - t_base);
    const HfaCtcDesc d = table[u];
    const TIn *logits = static_cast<const TIn *>(d.logits);

    // 1. argmax of this block's frames
#pragma unroll
    for (int p = 0; p < RPW; p += RIF) {
        const TIn *row[RIF];
        int bi[RIF];
#pragma unroll
        for (int r = 0; r < RIF; ++r)      // rows past the end re-read the block's last row (never stored)
            row[r] = logits + (int64_t)(t_base + min(warp * RPW + p + r, rows - 1)) * d.stride_t;
        hfa_warp_row_argmax<TIn, RIF>(row, V, d.stride_v, lane, bi);
        if (lane < RIF && warp * RPW + p + lane < rows) {
            int v = bi[0];
#pragma unroll
            for (int r = 1; r < RIF; ++r) v = (lane == r) ? bi[r] : v;
            arg[f0 + t_base + warp * RPW + p + lane] = v;
        }
    }
    __syncthreads();
    if (tid == 0) {                        // the barrier orders the block's stores before thread 0's fence
        __threadfence();
        last_sm = (atomicAdd(out_len + u, rows) + rows == T);
    }
    __syncthreads();
    if (!last_sm) return;
    __threadfence();

    // 2. the utterance's last block: keep / compact all of its frames in order
    const int32_t *a = arg + f0;
    int32_t *o = out_ids + f0;
    int carry = 0;
    for (int base = 0; base < T; base += HFA_CTC_BATCH_THREADS * FPT) {
        const int t0 = base + tid * FPT;
        int id[FPT], cnt = 0;
        int prev = (t0 > 0 && t0 <= T) ? __ldcg(a + t0 - 1) : 0;
#pragma unroll
        for (int j = 0; j < FPT; ++j) {
            id[j] = (t0 + j < T) ? __ldcg(a + t0 + j) : 0;
            const bool keep = id[j] != prev && id[j] != 0;
            prev = id[j];
            if (!keep) id[j] = 0;                   // a kept id is never 0
            cnt += keep;
        }
        int incl = cnt;
#pragma unroll
        for (int o2 = 1; o2 < 32; o2 <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o2);
            if (lane >= o2) incl += v;
        }
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        int pos = carry + incl - cnt, total = 0;
#pragma unroll
        for (int q = 0; q < NW; ++q) {
            pos += (q < warp) ? warp_sum[q] : 0;
            total += warp_sum[q];
        }
#pragma unroll
        for (int j = 0; j < FPT; ++j)
            if (id[j] != 0) o[pos++] = id[j];
        carry += total;
        __syncthreads();                            // warp_sum is rewritten by the next pass
    }
    if (tid == 0) out_len[u] = carry;
}

// frame_state[frame_off + t] = ph_idx_seq[k] for the largest k with ph_time_int[k] <= t (0 before the first
// segment): the state plot() reaches at frame t with its cumsum of index steps (:156-161).  One thread per
// frame, a binary search over the utterance's n_seg segment starts (non-decreasing).
__global__ void __launch_bounds__(HFA_EMIS_ROWS)
hfa_frame_state_kernel(HfaWs ws, HfaResultPtrs res, int32_t *__restrict__ out)
{
    const int u = ws.block_utt[blockIdx.x];
    const int T = ws.utt[u].T, S = ws.utt[u].S;
    const int t = (blockIdx.x - ws.row_blocks[u]) * HFA_EMIS_ROWS + threadIdx.x;
    if (t >= T) return;
    const int64_t so = ws.utt[u].seg_off;
    const int32_t *tim = res.ph_time_int + so;
    int lo = 0, hi = min(max(res.n_seg[u], 0), S);   // first k with tim[k] > t
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (tim[mid] <= t) lo = mid + 1;
        else hi = mid;
    }
    out[ws.utt[u].frame_off + t] = lo > 0 ? res.ph_idx_seq[so + lo - 1] : 0;
}

}  // namespace

cudaError_t hfa_launch_ctc_greedy(const void *logits, int dtype, int T, int V, int64_t st_t, int64_t st_v,
                                  int32_t *arg, int32_t *out_ids, int32_t *out_len, cudaStream_t stream)
{
    if (dtype == 0)
        hfa_ctc_greedy_kernel<float><<<1, HFA_CTC_THREADS, 0, stream>>>(static_cast<const float *>(logits), T, V,
                                                                        st_t, st_v, arg, out_ids, out_len);
    else if (dtype == 1)
        hfa_ctc_greedy_kernel<__half><<<1, HFA_CTC_THREADS, 0, stream>>>(static_cast<const __half *>(logits), T, V,
                                                                         st_t, st_v, arg, out_ids, out_len);
    else if (dtype == 2)
        hfa_ctc_greedy_kernel<__nv_bfloat16><<<1, HFA_CTC_THREADS, 0, stream>>>(
            static_cast<const __nv_bfloat16 *>(logits), T, V, st_t, st_v, arg, out_ids, out_len);
    else
        return cudaErrorInvalidValue;
    return cudaGetLastError();
}

// out_len must be zero on entry (the caller enqueues the memset)
cudaError_t hfa_launch_ctc_batch(const HfaLaunchCtx &c, int total_row_blocks, const HfaCtcDesc *table, int V,
                                 int dtype, int32_t *arg, int32_t *out_ids, int32_t *out_len)
{
    if (dtype == 0)
        hfa_ctc_batch_kernel<float><<<total_row_blocks, HFA_CTC_BATCH_THREADS, 0, c.stream>>>(c.ws, table, V, arg,
                                                                                            out_ids, out_len);
    else if (dtype == 1)
        hfa_ctc_batch_kernel<__half><<<total_row_blocks, HFA_CTC_BATCH_THREADS, 0, c.stream>>>(c.ws, table, V, arg,
                                                                                             out_ids, out_len);
    else if (dtype == 2)
        hfa_ctc_batch_kernel<__nv_bfloat16><<<total_row_blocks, HFA_CTC_BATCH_THREADS, 0, c.stream>>>(
            c.ws, table, V, arg, out_ids, out_len);
    else
        return cudaErrorInvalidValue;
    return cudaGetLastError();
}

cudaError_t hfa_launch_frame_states(const HfaLaunchCtx &c, int total_row_blocks, const HfaResultPtrs &res,
                                    int32_t *out)
{
    hfa_frame_state_kernel<<<total_row_blocks, HFA_EMIS_ROWS, 0, c.stream>>>(c.ws, res, out);
    return cudaGetLastError();
}
