// hfa_emission.cu -- logits -> emission matrix and edge logs, one fused pass.
//
// Reference: tools/alignment_decoder.py:35-40 (mask = ids of ph_seq U {0}), :53 (others pushed down
// by 1e9 in f32), :62-65 (log_softmax), :239 (gather columns by ph_seq_id), :68-71 (edge sigmoid,
// rescale, clamp), :84 (edge_prob = clip(p[t] + p[t-1], 0, 1) in f64), :241-242 (f64 log -> f32).
//
// One CTA = 64 consecutive frames of one utterance (see hfa_emission_block_kernel below).
// Algorithmic HBM bytes per frame: V*sizeof(in) + sizeof(in) (edge logit) read, 4*S + 12 written.
#include "hfa_common.cuh"

#define HFA_EMIS_ROWS 64
#define HFA_EMIS_WARPS 8

namespace {

__device__ __forceinline__ float warp_max(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// clamp((sigmoid(x) - 0.1) / 0.8, 0, 1), all f32 (:68-71)
__device__ __forceinline__ float edge_pred(float x)
{
    const float sg = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x)));
    const float v = __fdiv_rn(__fsub_rn(sg, 0.1f), 0.8f);
    return fminf(fmaxf(v, 0.0f), 1.0f);
}

__device__ __forceinline__ void edge_logs(float p, float p_prev, float2 &out)
{
    double ep = __dadd_rn((double)p, (double)p_prev);                 // :84 (f64 sum of f32 values)
    ep = fmin(fmax(ep, 0.0), 1.0);
    out.x = (float)log(__dadd_rn(ep, 1e-6));                          // :241
    out.y = (float)log(__dadd_rn(__dsub_rn(1.0, ep), 1e-6));          // :242  (1 - ep) + 1e-6
}

// The emission kernels stage an utterance's ids in shared memory for at most this many states (sp_cap =
// min(largest Sp of the batch, HFA_EMIS_ID_CAP)), so one long utterance cannot lower the occupancy of its whole
// batch.  The ids of the states past the staged ones (S > HFA_CTA_MAX_S only) are read from global memory.
#define HFA_EMIS_ID_CAP 8192

// ids of states s4 .. s4 + 3 (pads past S -> V), straight from global memory
__device__ __forceinline__ int4 hfa_ids4(const int32_t *ids, int S, int V, int s4)
{
    return make_int4(s4 < S ? __ldg(ids + s4) : V, s4 + 1 < S ? __ldg(ids + s4 + 1) : V,
                     s4 + 2 < S ? __ldg(ids + s4 + 2) : V, s4 + 3 < S ? __ldg(ids + s4 + 3) : V);
}

// One edge logit per frame out of a [T, V+2] head output is a 4-byte load every row stride: by default the L2
// fetches the whole 128-byte line around it from HBM (ncu, config 4: 460 MB read for 3.7 M frames).  The 64-byte
// fetch-granularity hint is the smallest PTX offers; the rest of the line belongs to the emission kernel's copy.
template <typename TIn> __device__ __forceinline__ float hfa_ld_edge(const TIn *p);
template <> __device__ __forceinline__ float hfa_ld_edge<float>(const float *p) { return hfa_ldg_f32_64B(p); }
template <> __device__ __forceinline__ float hfa_ld_edge<__half>(const __half *p)
{
    unsigned short v;
    asm volatile("ld.global.L2::64B.u16 %0, [%1];" : "=h"(v) : "l"(p));
    return __half2float(__ushort_as_half(v));
}
template <> __device__ __forceinline__ float hfa_ld_edge<__nv_bfloat16>(const __nv_bfloat16 *p)
{
    unsigned short v;
    asm volatile("ld.global.L2::64B.u16 %0, [%1];" : "=h"(v) : "l"(p));
    return __bfloat162float(__ushort_as_bfloat16(v));
}

// edge stream of one CTA's 64 frames, one thread per frame (:68-71,:84,:241-242)
template <typename TIn>
__device__ __forceinline__ void edge_block(const HfaWs &ws, const HfaUtt &m, const HfaInput &in,
                                           int t_base, int tid)
{
    if (tid < HFA_EMIS_ROWS) {
        const int t = t_base + tid;
        if (t < m.T) {
            const TIn *edge = reinterpret_cast<const TIn *>(in.edge);
            const float p = edge_pred(hfa_ld_edge<TIn>(edge + (int64_t)t * in.edge_st));
            const float pp = (t > 0) ? edge_pred(hfa_ld_edge<TIn>(edge + (int64_t)(t - 1) * in.edge_st)) : 0.0f;
            float2 lg;
            edge_logs(p, pp, lg);
            ws.edge2[m.edge_off + t] = lg;
            ws.edge_p[m.edge_off + t] = p;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Main emission kernel (V <= HFA_EMIS_BLOCK_MAX_V).  One CTA = 64 frames of one utterance:
//   A. the 8 warps load the 64 x V logits block coalesced (strided-view aware) into shared memory,
//      row stride VP odd -> a thread walking one row and a warp walking a column are conflict-free;
//   B. phoneme ids -> smem (pads -> slot V, which holds -inf), keep-mask, compacted list of the kept
//      vocabulary ids (ids of ph_seq U {0}, alignment_decoder.py:37-39);
//   C. normaliser: 4 threads per frame walk the KEPT ids only (max, then sum of exp) and combine
//      with two shuffles -- no 32-lane butterfly per row, no exp for the masked entries (the
//      reference pushes those down by 1e9, so their exp is exactly 0 and they never win the max
//      for |logit| < 5e8, :53);
//   D. each warp gathers its 8 rows by phoneme id (byte offsets held in registers) and stores the
//      [Sp] emission rows as float4: out = (x[id] - max) - log(sum), the reference's order (:63).
// ---------------------------------------------------------------------------------------------
#define HFA_EMIS_BLOCK_MAX_V 255

template <typename TIn>
__global__ void __launch_bounds__(HFA_EMIS_WARPS * 32, 5)
hfa_emission_block_kernel(HfaWs ws, int n_utt, int V, int sp_cap)
{
    constexpr int RPW = HFA_EMIS_ROWS / HFA_EMIS_WARPS;                      // rows per warp
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int VP = (V + 1) | 1;                                              // odd, >= V + 1
    const int mask_words = (V + 31) >> 5;
    int32_t *ids_sm = reinterpret_cast<int32_t *>(smem_raw);                 // [sp_cap]
    uint32_t *mask_sm = reinterpret_cast<uint32_t *>(ids_sm + sp_cap);       // [8]
    int32_t *kept_sm = reinterpret_cast<int32_t *>(mask_sm + 8);             // [256]
    float2 *stat_sm = reinterpret_cast<float2 *>(kept_sm + 256);             // [64] {max, lse}
    float *xs = reinterpret_cast<float *>(stat_sm + HFA_EMIS_ROWS);          // [64][VP]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int u = ws.block_utt[blockIdx.x];
    const HfaUtt m = ws.utt[u];
    const HfaInput in = ws.inputs[u];
    const bool compact = m.Dp > 0;                                           // see the stream kernel
    const int T = m.T, S = compact ? m.Dp : m.S, Sp = compact ? m.Dp : m.Sp;
    const int t_base = (blockIdx.x - ws.row_blocks[u]) * HFA_EMIS_ROWS;
    const TIn *frame = reinterpret_cast<const TIn *>(in.frame);
    if (compact && t_base == 0 && threadIdx.x == 0) ws.emis_mode[u] = 1;

    // A. logits block -> smem (rows past T re-read row T-1: valid memory, results never stored)
    {
        const TIn *rowp[RPW];
#pragma unroll
        for (int r = 0; r < RPW; ++r)
            rowp[r] = frame + (int64_t)min(t_base + warp + HFA_EMIS_WARPS * r, T - 1) * in.frame_st +
                      (int64_t)lane * in.frame_sv;
        const int64_t vstep = 32 * in.frame_sv;
        float *xw = xs + warp * VP + lane;
        for (int v = lane; v < V; v += 32) {
            float xv[RPW];
#pragma unroll
            for (int r = 0; r < RPW; ++r) {
                xv[r] = hfa_to_float<TIn>(*rowp[r]);
                rowp[r] += vstep;
            }
#pragma unroll
            for (int r = 0; r < RPW; ++r) xw[r * HFA_EMIS_WARPS * VP] = xv[r];
            xw += 32;
        }
    }
    if (lane < RPW) xs[(warp + HFA_EMIS_WARPS * lane) * VP + V] = HFA_NEG_INF;   // pad sentinel

    // B. ids, keep mask, kept list
    if (tid < 8) mask_sm[tid] = (tid == 0) ? 1u : 0u;                        // id 0 always kept (:39)
    __syncthreads();
    const int32_t *ids = compact ? ws.col_ids + m.seg_off + 4 * (int64_t)u : ws.ids + m.seg_off;
    for (int s = tid; s < Sp; s += blockDim.x) {
        const int id = (s < S) ? ids[s] : V;
        if (s < sp_cap) ids_sm[s] = id;
        if (id < V) atomicOr(&mask_sm[id >> 5], 1u << (id & 31));
    }
    __syncthreads();
    int n_kept = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) n_kept += (w < mask_words) ? __popc(mask_sm[w]) : 0;
    if (tid < V && ((mask_sm[tid >> 5] >> (tid & 31)) & 1u)) {
        int pos = __popc(mask_sm[tid >> 5] & ((1u << (tid & 31)) - 1u));
        for (int w = 0; w < (tid >> 5); ++w) pos += __popc(mask_sm[w]);
        kept_sm[pos] = tid;
    }
    __syncthreads();

    // C. normaliser: thread -> (row = tid / 4, part = tid % 4)
    {
        const float *row = xs + (tid >> 2) * VP;
        const int part = tid & 3;
        float mx = HFA_NEG_INF;
        for (int k = part; k < n_kept; k += 4) mx = fmaxf(mx, row[kept_sm[k]]);
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
        float sum = 0.0f;
        for (int k = part; k < n_kept; k += 4) sum = __fadd_rn(sum, expf(__fsub_rn(row[kept_sm[k]], mx)));
        sum = __fadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, 1));
        sum = __fadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, 2));
        if (part == 0) stat_sm[tid >> 2] = hfa_row_stat(mx, sum);
    }
    __syncthreads();

    // D. gather by phoneme id and store
    {
        uint32_t goff[2][4];
#pragma unroll
        for (int it = 0; it < 2; ++it) {
            const int s4 = min(lane * 4 + 128 * it, Sp - 4);
            const int4 id4 = *reinterpret_cast<const int4 *>(ids_sm + s4);
            goff[it][0] = (uint32_t)id4.x * 4u; goff[it][1] = (uint32_t)id4.y * 4u;
            goff[it][2] = (uint32_t)id4.z * 4u; goff[it][3] = (uint32_t)id4.w * 4u;
        }
        const uint32_t xs_sa = hfa_smem_u32(xs);
        const int rows_here = min(RPW, (T - t_base - warp + HFA_EMIS_WARPS - 1) / HFA_EMIS_WARPS);
        float *dst = ws.emis + m.emis_off + (int64_t)(t_base + warp) * Sp + lane * 4;
        const int dst_step = HFA_EMIS_WARPS * Sp;
        const bool st0 = lane * 4 < Sp, st1 = lane * 4 + 128 < Sp;
#pragma unroll
        for (int r = 0; r < RPW; ++r) {
            if (r >= rows_here) break;                                       // warp-uniform
            const int rr = warp + HFA_EMIS_WARPS * r;
            const float2 st = stat_sm[rr];
            const uint32_t rb = xs_sa + (uint32_t)(rr * VP) * 4u;
            float4 o;
            o.x = __fsub_rn(__fsub_rn(hfa_lds_f32(rb + goff[0][0]), st.x), st.y);
            o.y = __fsub_rn(__fsub_rn(hfa_lds_f32(rb + goff[0][1]), st.x), st.y);
            o.z = __fsub_rn(__fsub_rn(hfa_lds_f32(rb + goff[0][2]), st.x), st.y);
            o.w = __fsub_rn(__fsub_rn(hfa_lds_f32(rb + goff[0][3]), st.x), st.y);
            if (st0) *reinterpret_cast<float4 *>(dst + r * dst_step) = o;
            if (Sp > 128) {                                                  // warp-uniform
                o.x = __fsub_rn(__fsub_rn(hfa_lds_f32(rb + goff[1][0]), st.x), st.y);
                o.y = __fsub_rn(__fsub_rn(hfa_lds_f32(rb + goff[1][1]), st.x), st.y);
                o.z = __fsub_rn(__fsub_rn(hfa_lds_f32(rb + goff[1][2]), st.x), st.y);
                o.w = __fsub_rn(__fsub_rn(hfa_lds_f32(rb + goff[1][3]), st.x), st.y);
                if (st1) *reinterpret_cast<float4 *>(dst + r * dst_step + 128) = o;
            }
        }
        if (Sp > 256) {                                                      // long phoneme sequences
            const int s_sm = min(Sp, sp_cap);
            for (int r = 0; r < rows_here; ++r) {
                const int rr = warp + HFA_EMIS_WARPS * r;
                const float2 st = stat_sm[rr];
                for (int s4 = lane * 4 + 256; s4 < s_sm; s4 += 128) {
                    const int4 id4 = *reinterpret_cast<const int4 *>(ids_sm + s4);
                    float4 o;
                    o.x = __fsub_rn(__fsub_rn(xs[rr * VP + id4.x], st.x), st.y);
                    o.y = __fsub_rn(__fsub_rn(xs[rr * VP + id4.y], st.x), st.y);
                    o.z = __fsub_rn(__fsub_rn(xs[rr * VP + id4.z], st.x), st.y);
                    o.w = __fsub_rn(__fsub_rn(xs[rr * VP + id4.w], st.x), st.y);
                    *reinterpret_cast<float4 *>(dst + r * dst_step + (s4 - lane * 4)) = o;
                }
                for (int s4 = lane * 4 + s_sm; s4 < Sp; s4 += 128) {        // past the staged ids
                    const int4 id4 = hfa_ids4(ids, S, V, s4);
                    float4 o;
                    o.x = __fsub_rn(__fsub_rn(xs[rr * VP + id4.x], st.x), st.y);
                    o.y = __fsub_rn(__fsub_rn(xs[rr * VP + id4.y], st.x), st.y);
                    o.z = __fsub_rn(__fsub_rn(xs[rr * VP + id4.z], st.x), st.y);
                    o.w = __fsub_rn(__fsub_rn(xs[rr * VP + id4.w], st.x), st.y);
                    *reinterpret_cast<float4 *>(dst + r * dst_step + (s4 - lane * 4)) = o;
                }
            }
        }
    }
    edge_block<TIn>(ws, m, in, t_base, tid);
}

// The edge stream on its own (one thread per frame), used next to the persistent emission kernel:
// its two f64 logs per frame are ~250 instructions for a quarter of a CTA and would otherwise sit
// between that kernel's barriers.
template <typename TIn>
__global__ void __launch_bounds__(HFA_EMIS_ROWS)
hfa_edge_kernel(HfaWs ws)
{
    const int u = ws.block_utt[blockIdx.x];
    const HfaUtt m = ws.utt[u];
    const HfaInput in = ws.inputs[u];
    edge_block<TIn>(ws, m, in, (blockIdx.x - ws.row_blocks[u]) * HFA_EMIS_ROWS, threadIdx.x);
}

// max and sum of exp over the kept ids of one row, the part of one of the row's 4 lanes: kept id `part + 4 j` sits
// in kreg[j].  The two 2-step butterflies that combine the 4 lanes follow in the caller.
template <int NJ, typename TIn>
__device__ __forceinline__ void hfa_row_stats(const TIn *row, const int (&kreg)[16], int part, int n_kept,
                                              float &mx, float &sum)
{
    float xv[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {           // unconditional load (kreg is 0 past the end) + select:
        const float x = hfa_to_float<TIn>(row[kreg[j]]);          // no divergent branches
        xv[j] = (part + 4 * j < n_kept) ? x : HFA_NEG_INF;
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) mx = fmaxf(mx, xv[j]);
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
#pragma unroll
    for (int j = 0; j < NJ; ++j)             // entries past the end are -inf: exp = +0, sum unchanged
        sum = __fadd_rn(sum, expf(__fsub_rn(xv[j], mx)));
}

// ---------------------------------------------------------------------------------------------
// Persistent, TMA-fed variant of the kernel above -- the default whenever the logits rows of an
// utterance are contiguous (unit column stride, which is what the [T, V+2] head-output views are).
// A CTA owns a contiguous range of 64-frame row blocks and streams them through two shared-memory
// stages: while block i is normalised and gathered, the TMA engine already copies block i+1 (one
// 1-D bulk copy of 64 x row_stride elements, mbarrier-signalled; SASS UBLKCP).  No thread ever
// loads a logit itself, no registers hold loads in flight, and the per-utterance setup (ids,
// keep-mask, kept list, gather offsets) is reused by the consecutive blocks of one utterance.
// The copy starts at the 16-byte boundary below the first logit (a view of the head output starts
// 2 elements in) and is rounded up to 16 bytes; both stay inside the allocation the view lives in.
// ---------------------------------------------------------------------------------------------
template <typename TIn>
__global__ void __launch_bounds__(HFA_EMIS_WARPS * 32)      // (.., 4) caps it at 64 registers: measured slower
hfa_emission_stream_kernel(HfaWs ws, int n_blocks, int V, int sp_cap, int stage_bytes)
{
    constexpr int RPW = HFA_EMIS_ROWS / HFA_EMIS_WARPS;                      // rows per warp
    extern __shared__ __align__(128) unsigned char smem_raw[];
    unsigned char *stage0 = smem_raw;                                        // [2][stage_bytes]
    int32_t *ids_sm = reinterpret_cast<int32_t *>(smem_raw + 2 * stage_bytes);   // [sp_cap]
    uint32_t *mask_sm = reinterpret_cast<uint32_t *>(ids_sm + sp_cap);       // [8]
    int32_t *kept_sm = reinterpret_cast<int32_t *>(mask_sm + 8);             // [256]
    float2 *stat_sm = reinterpret_cast<float2 *>(kept_sm + 256);             // [64] {max, lse}
    uint64_t *bar = reinterpret_cast<uint64_t *>(stat_sm + HFA_EMIS_ROWS);   // [2]
    int32_t *shift_sm = reinterpret_cast<int32_t *>(bar + 2);                // [2] byte shift of a stage

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int blk0 = (int)(((int64_t)blockIdx.x * n_blocks) / gridDim.x);
    const int blk1 = (int)(((int64_t)(blockIdx.x + 1) * n_blocks) / gridDim.x);
    if (blk0 >= blk1) return;

    // thread 0: start the copy of row block `blk` into stage `s`
    auto issue = [&](int blk, int s) {
        const int u = ws.block_utt[blk];
        const HfaUtt m = ws.utt[u];
        const HfaInput in = ws.inputs[u];
        const int t_base = (blk - ws.row_blocks[u]) * HFA_EMIS_ROWS;
        const int rows = min(HFA_EMIS_ROWS, m.T - t_base);
        const unsigned char *src = reinterpret_cast<const unsigned char *>(in.frame) +
                                   (int64_t)t_base * in.frame_st * (int64_t)sizeof(TIn);
        const uint32_t shift = (uint32_t)(reinterpret_cast<uintptr_t>(src) & 15u);
        // rows-1 full strides plus the V logits of the last row, from the aligned address
        const uint32_t bytes =
            (shift + (uint32_t)(((int64_t)(rows - 1) * in.frame_st + V) * (int64_t)sizeof(TIn)) + 15u) & ~15u;
        shift_sm[s] = (int32_t)shift;
        hfa_mbar_expect_tx(hfa_smem_u32(&bar[s]), bytes);
        hfa_bulk_load(hfa_smem_u32(stage0 + (size_t)s * stage_bytes), src - shift, bytes, hfa_smem_u32(&bar[s]));
    };
    if (tid == 0) {
        hfa_mbar_init(hfa_smem_u32(&bar[0]), 1);
        hfa_mbar_init(hfa_smem_u32(&bar[1]), 1);
        hfa_fence_mbar_init();
        issue(blk0, 0);
    }
    __syncthreads();

    int cur_u = -1;
    int S = 0, Sp = 4, T = 0, n_kept = 0;
    uint32_t goff[2][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}};
    int lpr = 32;
    int kreg[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) kreg[j] = 0;
    HfaUtt m;
    HfaInput in;
    for (int blk = blk0; blk < blk1; ++blk) {
        const int s = (blk - blk0) & 1;
        if (tid == 0 && blk + 1 < blk1) issue(blk + 1, s ^ 1);     // stage s^1 was released by the
                                                                   // barrier that ended block blk-1
        const int u = ws.block_utt[blk];
        if (u != cur_u) {
            // B. per-utterance setup: ids, keep mask, kept list, gather offsets
            cur_u = u;
            m = ws.utt[u];
            in = ws.inputs[u];
            // compacted rows (m.Dp > 0, HfaWs::colmap): one column per distinct id instead of one per state --
            // the column ids take the place of the phoneme ids, the row stride is Dp
            const bool compact = m.Dp > 0;
            S = compact ? m.Dp : m.S; Sp = compact ? m.Dp : m.Sp; T = m.T;
            const int mask_words = (V + 31) >> 5;
            if (tid < 8) mask_sm[tid] = (tid == 0) ? 1u : 0u;                // id 0 always kept (:39)
            __syncthreads();
            const int32_t *ids = compact ? ws.col_ids + m.seg_off + 4 * (int64_t)u : ws.ids + m.seg_off;
            for (int q = tid; q < Sp; q += blockDim.x) {
                const int id = (q < S) ? ids[q] : V;
                if (q < sp_cap) ids_sm[q] = id;
                if (id < V) atomicOr(&mask_sm[id >> 5], 1u << (id & 31));
            }
            if (compact && tid == 0 && blk == ws.row_blocks[u]) ws.emis_mode[u] = 1;
            __syncthreads();
            n_kept = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) n_kept += (w < mask_words) ? __popc(mask_sm[w]) : 0;
            if (tid < V && ((mask_sm[tid >> 5] >> (tid & 31)) & 1u)) {
                int pos = __popc(mask_sm[tid >> 5] & ((1u << (tid & 31)) - 1u));
                for (int w = 0; w < (tid >> 5); ++w) pos += __popc(mask_sm[w]);
                kept_sm[pos] = tid;
            }
            // lanes per stored row in the gather (D): a row of <= 32 / <= 64 columns (the compacted rows of big
            // batches, short phoneme sequences) takes 8 / 16 lanes x float4, so a warp gathers 4 / 2 rows per pass
            lpr = (Sp <= 32) ? 8 : (Sp <= 64) ? 16 : 32;
#pragma unroll
            for (int it = 0; it < 2; ++it) {
                const int s4 = min((lane & (lpr - 1)) * 4 + 128 * it, Sp - 4);
                const int4 id4 = *reinterpret_cast<const int4 *>(ids_sm + s4);
                goff[it][0] = (uint32_t)id4.x; goff[it][1] = (uint32_t)id4.y;
                goff[it][2] = (uint32_t)id4.z; goff[it][3] = (uint32_t)id4.w;
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int k = (lane & 3) + 4 * j;
                kreg[j] = (k < n_kept && k < 256) ? kept_sm[k] : 0;
            }
        }
        const int t_base = (blk - ws.row_blocks[u]) * HFA_EMIS_ROWS;
        const int row_st = (int)in.frame_st;

        const uint32_t parity = ((blk - blk0) >> 1) & 1;
        hfa_mbar_wait(hfa_smem_u32(&bar[s]), parity, HFA_POLLS_COPY);
        const TIn *xs = reinterpret_cast<const TIn *>(stage0 + (size_t)s * stage_bytes + shift_sm[s]);

        // C. normaliser, warp-local: lane -> (row = 8 * warp + lane / 4, part = lane % 4), kept ids
        //    only.  A warp normalises exactly the 8 consecutive rows it gathers below, so C -> D needs
        //    no CTA barrier (consecutive rows: their shared-memory banks differ).
        {
            const int rr = RPW * warp + (lane >> 2);
            const TIn *row = xs + rr * row_st;
            const int part = lane & 3;
            float mx = HFA_NEG_INF, sum = 0.0f;
            if (n_kept <= 64) {                                              // CTA-uniform
                // the lane's kept ids sit in registers (kreg, set up per utterance): one load per logit, reused
                // by both passes; same order of operations as the loop below.  Only as many slots as the
                // utterance has kept ids (4 lanes x NJ): slots past the end would add exp(-inf) = +0, the sums
                // are bit-identical -- the kernel is issue-bound, a typical utterance keeps 40-50 ids.
                const int nj = (n_kept + 3) >> 2;
                if (nj <= 8) hfa_row_stats<8, TIn>(row, kreg, part, n_kept, mx, sum);
                else if (nj <= 10) hfa_row_stats<10, TIn>(row, kreg, part, n_kept, mx, sum);
                else if (nj <= 12) hfa_row_stats<12, TIn>(row, kreg, part, n_kept, mx, sum);
                else if (nj <= 14) hfa_row_stats<14, TIn>(row, kreg, part, n_kept, mx, sum);
                else hfa_row_stats<16, TIn>(row, kreg, part, n_kept, mx, sum);
            } else {
                for (int k = part; k < n_kept; k += 4) mx = fmaxf(mx, hfa_to_float<TIn>(row[kept_sm[k]]));
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
                for (int k = part; k < n_kept; k += 4)
                    sum = __fadd_rn(sum, expf(__fsub_rn(hfa_to_float<TIn>(row[kept_sm[k]]), mx)));
            }
            sum = __fadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, 1));
            sum = __fadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, 2));
            if (part == 0) stat_sm[rr] = hfa_row_stat(mx, sum);
        }
        __syncwarp();

        // D. gather by phoneme id and store (pad columns: id V -> -inf)
        {
            const int rows_here = max(0, min(RPW, T - t_base - RPW * warp));
            float *dst = ws.emis + m.emis_off + (int64_t)(t_base + RPW * warp) * Sp + lane * 4;
            const int dst_step = Sp;
            const bool st0 = lane * 4 < Sp, st1 = lane * 4 + 128 < Sp;
            auto val = [&](const TIn *row, uint32_t id, const float2 st) {
                const float x = (id < (uint32_t)V) ? hfa_to_float<TIn>(row[id]) : HFA_NEG_INF;
                return __fsub_rn(__fsub_rn(x, st.x), st.y);
            };
            if (lpr < 32) {                                                  // CTA-uniform: narrow rows
                // lane -> (row r0 + lane / lpr, columns 4 (lane % lpr) ..): 4 or 2 rows per pass; same values, same
                // order of operations per element as the one-row-per-pass loop below
                const int sub = (lpr == 8) ? (lane >> 3) : (lane >> 4);
                const int col = (lane & (lpr - 1)) * 4;
                const int rpp = 32 / lpr;
                const bool stc = col < Sp;
                float *dst_n = ws.emis + m.emis_off + (int64_t)(t_base + RPW * warp) * Sp + col;
#pragma unroll
                for (int r0 = 0; r0 < RPW; r0 += 2) {
                    if (r0 >= rows_here) break;                              // warp-uniform
                    if (rpp == 4 && (r0 & 2)) continue;                      // uniform: 4 rows per pass -> r0 = 0, 4
                    const int r = r0 + sub;
                    const int rr = RPW * warp + r;
                    const float2 st = stat_sm[rr];
                    const TIn *row = xs + rr * row_st;
                    float4 o;
                    o.x = val(row, goff[0][0], st); o.y = val(row, goff[0][1], st);
                    o.z = val(row, goff[0][2], st); o.w = val(row, goff[0][3], st);
                    if (stc && r < rows_here) *reinterpret_cast<float4 *>(dst_n + r * dst_step) = o;
                }
            } else {
#pragma unroll
            for (int r = 0; r < RPW; ++r) {
                if (r >= rows_here) break;                                   // warp-uniform
                const int rr = RPW * warp + r;
                const float2 st = stat_sm[rr];
                const TIn *row = xs + rr * row_st;
                float4 o;
                o.x = val(row, goff[0][0], st); o.y = val(row, goff[0][1], st);
                o.z = val(row, goff[0][2], st); o.w = val(row, goff[0][3], st);
                if (st0) *reinterpret_cast<float4 *>(dst + r * dst_step) = o;
                if (Sp > 128) {                                              // warp-uniform
                    o.x = val(row, goff[1][0], st); o.y = val(row, goff[1][1], st);
                    o.z = val(row, goff[1][2], st); o.w = val(row, goff[1][3], st);
                    if (st1) *reinterpret_cast<float4 *>(dst + r * dst_step + 128) = o;
                }
            }
            }
            if (Sp > 256) {                                                  // long phoneme sequences
                const int s_sm = min(Sp, sp_cap);
                for (int r = 0; r < rows_here; ++r) {
                    const int rr = RPW * warp + r;
                    const float2 st = stat_sm[rr];
                    const TIn *row = xs + rr * row_st;
                    for (int s4 = lane * 4 + 256; s4 < s_sm; s4 += 128) {
                        const int4 id4 = *reinterpret_cast<const int4 *>(ids_sm + s4);
                        float4 o;
                        o.x = val(row, (uint32_t)id4.x, st); o.y = val(row, (uint32_t)id4.y, st);
                        o.z = val(row, (uint32_t)id4.z, st); o.w = val(row, (uint32_t)id4.w, st);
                        *reinterpret_cast<float4 *>(dst + r * dst_step + (s4 - lane * 4)) = o;
                    }
                    if (Sp > s_sm) {                                         // past the staged ids
                        const int32_t *ids = m.Dp > 0 ? ws.col_ids + m.seg_off + 4 * (int64_t)cur_u
                                                      : ws.ids + m.seg_off;
                        for (int s4 = lane * 4 + s_sm; s4 < Sp; s4 += 128) {
                            const int4 id4 = hfa_ids4(ids, S, V, s4);
                            float4 o;
                            o.x = val(row, (uint32_t)id4.x, st); o.y = val(row, (uint32_t)id4.y, st);
                            o.z = val(row, (uint32_t)id4.z, st); o.w = val(row, (uint32_t)id4.w, st);
                            *reinterpret_cast<float4 *>(dst + r * dst_step + (s4 - lane * 4)) = o;
                        }
                    }
                }
            }
        }
        __syncthreads();                           // everyone is done with stage s and stat_sm
    }
}

// ---------------------------------------------------------------------------------------------
// Wide vocabularies (V > HFA_EMIS_BLOCK_MAX_V): one warp per row, rows streamed through a per-warp
// shared-memory buffer, full masked softmax exactly as the reference spells it.
// ---------------------------------------------------------------------------------------------
template <typename TIn>
__global__ void __launch_bounds__(HFA_EMIS_WARPS * 32)
hfa_emission_wide_kernel(HfaWs ws, int n_utt, int V, int sp_cap)
{
    constexpr int RPW = HFA_EMIS_ROWS / HFA_EMIS_WARPS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int32_t *ids_sm = reinterpret_cast<int32_t *>(smem_raw);                 // [sp_cap]
    uint32_t *mask_sm = reinterpret_cast<uint32_t *>(ids_sm + sp_cap);       // [ceil(V/32)] keep bits
    const int mask_words = (V + 31) >> 5;
    float *rows_sm = reinterpret_cast<float *>(mask_sm + ((mask_words + 3) & ~3));
    const int VS = V + 1;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int u = ws.block_utt[blockIdx.x];
    const HfaUtt m = ws.utt[u];
    const HfaInput in = ws.inputs[u];
    const bool compact = m.Dp > 0;                                           // see the stream kernel
    const int T = m.T, S = compact ? m.Dp : m.S, Sp = compact ? m.Dp : m.Sp;
    const int t_base = (blockIdx.x - ws.row_blocks[u]) * HFA_EMIS_ROWS;
    const TIn *frame = reinterpret_cast<const TIn *>(in.frame);
    float *g_out = ws.emis + m.emis_off;
    if (compact && t_base == 0 && threadIdx.x == 0) ws.emis_mode[u] = 1;

    for (int w = tid; w < mask_words; w += blockDim.x) mask_sm[w] = (w == 0) ? 1u : 0u;  // id 0 (:39)
    __syncthreads();
    const int32_t *ids = compact ? ws.col_ids + m.seg_off + 4 * (int64_t)u : ws.ids + m.seg_off;
    for (int s = tid; s < Sp; s += blockDim.x) {
        const int id = (s < S) ? ids[s] : V;
        if (s < sp_cap) ids_sm[s] = id;
        if (id < V) atomicOr(&mask_sm[id >> 5], 1u << (id & 31));
    }
    __syncthreads();

    float *rowbuf = rows_sm + (size_t)warp * VS;
    if (lane == 0) rowbuf[V] = HFA_NEG_INF;
    __syncwarp();
    for (int j = 0; j < RPW; ++j) {
        const int t = t_base + warp + HFA_EMIS_WARPS * j;
        if (t >= T) continue;
        const TIn *src = frame + (int64_t)t * in.frame_st;
        float mr = HFA_NEG_INF;
        for (int v = lane; v < V; v += 32) {
            float xv = hfa_to_float<TIn>(src[(int64_t)v * in.frame_sv]);
            if (!((mask_sm[v >> 5] >> (v & 31)) & 1u)) xv = __fsub_rn(xv, 1e9f);          // :53
            rowbuf[v] = xv;
            mr = fmaxf(mr, xv);
        }
        mr = warp_max(mr);
        float sum = 0.0f;
        for (int v = lane; v < V; v += 32) sum = __fadd_rn(sum, expf(__fsub_rn(rowbuf[v], mr)));
        // every logit of the row -inf: the reference's rows are NaN, ours -inf (hfa_row_stat, DESIGN 4.1)
        const float2 st = hfa_row_stat(mr, warp_sum(sum));
        mr = st.x;
        const float l = st.y;
        __syncwarp();
        float *dst = g_out + (int64_t)t * Sp;
        for (int s4 = lane * 4; s4 < Sp; s4 += 128) {
            const int4 id4 = s4 < sp_cap ? *reinterpret_cast<const int4 *>(ids_sm + s4)
                                         : hfa_ids4(ids, S, V, s4);           // past the staged ids
            float4 o;
            o.x = __fsub_rn(__fsub_rn(rowbuf[id4.x], mr), l);
            o.y = __fsub_rn(__fsub_rn(rowbuf[id4.y], mr), l);
            o.z = __fsub_rn(__fsub_rn(rowbuf[id4.z], mr), l);
            o.w = __fsub_rn(__fsub_rn(rowbuf[id4.w], mr), l);
            *reinterpret_cast<float4 *>(dst + s4) = o;
        }
        __syncwarp();
    }
    edge_block<TIn>(ws, m, in, t_base, tid);
}

// the reference's forward_pass inputs given directly (dense ragged), repacked into the workspace
__global__ void __launch_bounds__(256)
hfa_pack_kernel(HfaWs ws, int n_utt, const float *__restrict__ prob_log,
                const float *__restrict__ edge_log, const float *__restrict__ not_edge_log,
                const float *__restrict__ edge_pred_in)
{
    const int tid = threadIdx.x;
    const int u = ws.block_utt[blockIdx.x];
    const HfaUtt m = ws.utt[u];
    const int T = m.T, S = m.S, Sp = m.Sp;
    const int t_base = (blockIdx.x - ws.row_blocks[u]) * HFA_EMIS_ROWS;
    const int rows = min(HFA_EMIS_ROWS, T - t_base);
    const float *src = prob_log + m.cell_off + (int64_t)t_base * S;
    float *dst = ws.emis + m.emis_off + (int64_t)t_base * Sp;
    if (m.Dp > 0 && t_base == 0 && tid == 0) ws.emis_mode[u] = 0;     // per-state values: plain rows
    for (int64_t i = tid; i < (int64_t)rows * Sp; i += blockDim.x) {
        const int r = (int)(i / Sp), s = (int)(i - (int64_t)r * Sp);
        dst[i] = (s < S) ? src[(int64_t)r * S + s] : HFA_NEG_INF;
    }
    if (tid < rows) {
        const int t = t_base + tid;
        ws.edge2[m.edge_off + t] = make_float2(edge_log[m.frame_off + t], not_edge_log[m.frame_off + t]);
        ws.edge_p[m.edge_off + t] = edge_pred_in ? edge_pred_in[m.frame_off + t] : 0.0f;
    }
}

// debug: emis[t][s] of every utterance as dense ragged [T_b][S_b] (cell_off), whatever the stored layout
__global__ void __launch_bounds__(256)
hfa_unpack_emis_kernel(HfaWs ws, float *__restrict__ out)
{
    const int u = ws.block_utt[blockIdx.x];
    const HfaUtt m = ws.utt[u];
    const bool compact = m.Dp > 0 && ws.emis_mode[u] != 0;
    const int Ep = compact ? m.Dp : m.Sp, S = m.S;
    const int t_base = (blockIdx.x - ws.row_blocks[u]) * HFA_EMIS_ROWS;
    const int rows = min(HFA_EMIS_ROWS, m.T - t_base);
    const uint8_t *cm = ws.colmap + m.seg_off;
    for (int64_t i = threadIdx.x; i < (int64_t)rows * S; i += blockDim.x) {
        const int r = (int)(i / S), s = (int)(i - (int64_t)r * S);
        out[m.cell_off + (int64_t)(t_base + r) * S + s] =
            ws.emis[m.emis_off + (int64_t)(t_base + r) * Ep + (compact ? cm[s] : s)];
    }
}

}  // namespace

cudaError_t hfa_launch_unpack_emissions(const HfaLaunchCtx &c, int total_row_blocks, float *out)
{
    if (total_row_blocks <= 0) return cudaSuccess;
    hfa_unpack_emis_kernel<<<total_row_blocks, 256, 0, c.stream>>>(c.ws, out);
    return cudaGetLastError();
}

template <typename TIn>
static cudaError_t launch_emission_t(const HfaLaunchCtx &c, int blocks, int max_sp, int64_t max_row_stride,
                                     int *n_launched)
{
    *n_launched = 1;
    const int V = c.vocab;
    max_sp = max_sp < HFA_EMIS_ID_CAP ? max_sp : HFA_EMIS_ID_CAP;      // = sp_cap of the kernels
    cudaError_t e;
    // max_row_stride > 0: every utterance has unit column stride and rows at most that many elements
    // apart -> a 64-row block is one contiguous range and can travel by TMA
    const int64_t stage = max_row_stride > 0
        ? ((HFA_EMIS_ROWS * max_row_stride * (int64_t)sizeof(TIn) + 32 + 127) & ~(int64_t)127) : 0;
    if (V <= HFA_EMIS_BLOCK_MAX_V && stage > 0 && stage <= 48 * 1024) {
        const size_t smem = 2 * (size_t)stage + (size_t)max_sp * 4 + 8 * 4 + 256 * 4 + HFA_EMIS_ROWS * 8 +
                            2 * 8 + 2 * 4 + 16;
        e = cudaFuncSetAttribute(hfa_emission_stream_kernel<TIn>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        // persistent CTAs: exactly as many as are resident at once (registers and shared memory)
        int per_sm = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hfa_emission_stream_kernel<TIn>,
                                                          HFA_EMIS_WARPS * 32, smem);
        if (e != cudaSuccess) return e;
        per_sm = per_sm < 1 ? 1 : (per_sm > 4 ? 4 : per_sm);
        int dev = 0, n_sm = 148;
        if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        const int grid = blocks < n_sm * per_sm ? blocks : n_sm * per_sm;
        *n_launched = 2;     // tells the caller to launch hfa_launch_edge as well (on a forked stream)
        hfa_emission_stream_kernel<TIn><<<grid, HFA_EMIS_WARPS * 32, smem, c.stream>>>(
            c.ws, blocks, V, max_sp, (int)stage);
        return cudaGetLastError();
    }
    if (V <= HFA_EMIS_BLOCK_MAX_V) {
        const int VP = (V + 1) | 1;
        const size_t smem = (size_t)max_sp * 4 + 8 * 4 + 256 * 4 + HFA_EMIS_ROWS * 8 +
                            (size_t)HFA_EMIS_ROWS * VP * 4;
        e = cudaFuncSetAttribute(hfa_emission_block_kernel<TIn>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        hfa_emission_block_kernel<TIn><<<blocks, HFA_EMIS_WARPS * 32, smem, c.stream>>>(c.ws, c.n_utt,
                                                                                    V, max_sp);
    } else {
        const int mask_words = (V + 31) >> 5;
        const size_t smem = (size_t)max_sp * 4 + (size_t)((mask_words + 3) & ~3) * 4 +
                            (size_t)HFA_EMIS_WARPS * (V + 1) * 4;
        e = cudaFuncSetAttribute(hfa_emission_wide_kernel<TIn>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        hfa_emission_wide_kernel<TIn><<<blocks, HFA_EMIS_WARPS * 32, smem, c.stream>>>(c.ws, c.n_utt,
                                                                                   V, max_sp);
    }
    return cudaGetLastError();
}

cudaError_t hfa_launch_emission(const HfaLaunchCtx &c, int total_row_blocks, int max_sp, int dtype,
                                int64_t max_row_stride, int *n_launched)
{
    *n_launched = 0;
    if (total_row_blocks <= 0) return cudaSuccess;
    if (dtype == 0) return launch_emission_t<float>(c, total_row_blocks, max_sp, max_row_stride, n_launched);
    if (dtype == 1) return launch_emission_t<__half>(c, total_row_blocks, max_sp, max_row_stride, n_launched);
    if (dtype == 2)
        return launch_emission_t<__nv_bfloat16>(c, total_row_blocks, max_sp, max_row_stride, n_launched);
    return cudaErrorInvalidValue;
}

// the edge stream as its own launch (needed when hfa_launch_emission reported 2 launches)
cudaError_t hfa_launch_edge(const HfaLaunchCtx &c, int total_row_blocks, int dtype)
{
    if (total_row_blocks <= 0) return cudaSuccess;
    if (dtype == 0) hfa_edge_kernel<float><<<total_row_blocks, HFA_EMIS_ROWS, 0, c.stream>>>(c.ws);
    else if (dtype == 1) hfa_edge_kernel<__half><<<total_row_blocks, HFA_EMIS_ROWS, 0, c.stream>>>(c.ws);
    else if (dtype == 2) hfa_edge_kernel<__nv_bfloat16><<<total_row_blocks, HFA_EMIS_ROWS, 0, c.stream>>>(c.ws);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}

cudaError_t hfa_launch_pack(const HfaLaunchCtx &c, int total_row_blocks, const float *prob_log,
                            const float *edge_log, const float *not_edge_log, const float *edge_pred)
{
    if (total_row_blocks <= 0) return cudaSuccess;
    hfa_pack_kernel<<<total_row_blocks, 256, 0, c.stream>>>(c.ws, c.n_utt, prob_log, edge_log,
                                                            not_edge_log, edge_pred);
    return cudaGetLastError();
}
