// hfa_api.cu -- host side of libhfa_align.so: length-bucketed collation ("plan") and the C ABI
// declared in include/hfa_align.h.  No torch types, no device allocation, no stream sync.
#include <algorithm>
#include <atomic>
#include <climits>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <numeric>
#include <queue>
#include <unordered_map>
#include <vector>

#include <cuda.h>      // CUtensorMap types only: the encoder is fetched through cudaGetDriverEntryPoint

#include "../../include/hfa_align.h"
#include "hfa_common.cuh"

cudaError_t hfa_launch_unpack_emissions(const HfaLaunchCtx &c, int total_row_blocks, float *out);
cudaError_t hfa_launch_dp_warp_any(const HfaLaunchCtx &c, int max_k, int max_pair_k, const int32_t *order, int n,
                                   float *dp_dump);
cudaError_t hfa_launch_dp_cta(const HfaLaunchCtx &c, const int32_t *order, int n, int max_sp, float *dp_dump);
cudaError_t hfa_launch_dp_band(const HfaLaunchCtx &c, int k, int item_begin, int n_items, int32_t *ticket,
                               bool keep_dp, int64_t fused_row_stride, float *dp_dump);
cudaError_t hfa_launch_dp_skew(const HfaLaunchCtx &c, int d, int ctas_per_sm, int item_begin, int n_items,
                               int32_t *ticket, bool keep_dp, int force_slow, float *dp_dump);
cudaError_t hfa_launch_emission(const HfaLaunchCtx &c, int total_row_blocks, int max_sp, int dtype,
                                int64_t max_row_stride, int *n_launched);
cudaError_t hfa_launch_edge(const HfaLaunchCtx &c, int total_row_blocks, int dtype);
cudaError_t hfa_launch_pack(const HfaLaunchCtx &c, int total_row_blocks, const float *prob_log,
                            const float *edge_log, const float *not_edge_log,
                            const float *edge_pred);
cudaError_t hfa_launch_backtrace(const HfaLaunchCtx &c, const int32_t *order, int n,
                                 const HfaResultPtrs &res, float *frame_conf, float *dp_path);
cudaError_t hfa_launch_unpack_bp(const HfaLaunchCtx &c, int utt, int8_t *out);
cudaError_t hfa_launch_unpack_dp(const HfaLaunchCtx &c, int utt, float *out);
cudaError_t hfa_launch_ctc_greedy(const void *logits, int dtype, int T, int V, int64_t st_t, int64_t st_v,
                                  int32_t *arg, int32_t *out_ids, int32_t *out_len, cudaStream_t stream);
cudaError_t hfa_launch_ctc_batch(const HfaLaunchCtx &c, int total_row_blocks, const HfaCtcDesc *table, int V,
                                 int dtype, int32_t *arg, int32_t *out_ids, int32_t *out_len);
cudaError_t hfa_launch_frame_states(const HfaLaunchCtx &c, int total_row_blocks, const HfaResultPtrs &res,
                                    int32_t *out);
cudaError_t hfa_launch_jump_tables(const HfaLaunchCtx &c, int n_blocks);
cudaError_t hfa_launch_backtrace_tables(const HfaLaunchCtx &c, const int32_t *order, int n,
                                        const HfaResultPtrs &res, float *frame_conf, float *dp_path);
cudaError_t hfa_launch_backtrace_walk(const HfaLaunchCtx &c, const int32_t *order, int n, int64_t smem,
                                      const HfaResultPtrs &res, float *frame_conf, float *dp_path);

namespace {

thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
int cuda_fail(cudaError_t e, const char *what)
{
    return fail(HFA_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

// cuTensorMapEncodeTiled without linking libcuda: resolved once through the runtime
typedef CUresult (*HfaEncodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                   const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
HfaEncodeTiled tensor_map_encoder()
{
    static const HfaEncodeTiled fn = [] {
        void *f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            return (HfaEncodeTiled) nullptr;
        return reinterpret_cast<HfaEncodeTiled>(f);
    }();
    return fn;
}

// side streams for the concurrent per-class DP launches: one set per (host thread, device)
struct HfaSideStreams {
    int device = -1;
    cudaStream_t stream[HFA_NUM_CLASSES] = {};
    cudaEvent_t fork = nullptr, join[HFA_NUM_CLASSES] = {};
};
std::vector<HfaSideStreams *> &side_pool()
{
    thread_local std::vector<HfaSideStreams *> pool;
    return pool;
}
HfaSideStreams *side_streams()
{
    std::vector<HfaSideStreams *> &pool = side_pool();
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    for (HfaSideStreams *s : pool)
        if (s->device == dev) return s;
    HfaSideStreams *s = new (std::nothrow) HfaSideStreams();
    if (!s) return nullptr;
    s->device = dev;
    bool ok = cudaEventCreateWithFlags(&s->fork, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; ok && i < HFA_NUM_CLASSES; ++i) {
        ok = cudaStreamCreateWithFlags(&s->stream[i], cudaStreamNonBlocking) == cudaSuccess &&
             cudaEventCreateWithFlags(&s->join[i], cudaEventDisableTiming) == cudaSuccess;
    }
    if (!ok) { delete s; return nullptr; }
    try {
        pool.push_back(s);
    } catch (const std::bad_alloc &) {
        delete s;
        return nullptr;
    }
    return s;
}

int sm_count()
{
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n < 1)
        return 148;                                            // B200
    return n;
}

// Length in blocks of a launch of the skewed kernel when `slots` CTAs are resident: a list schedule of the strips in
// ticket order (each claims the first slot that frees up) in which every block takes the same time and a strip's
// blocks trail its left neighbour's by ceil(31 d / 32) + 1 blocks (block j waits for the left strip's block
// j + ceil(31 d / 32) to be published).
int64_t skew_makespan(const std::vector<HfaBandItem> &items, int begin, int count, const std::vector<HfaUtt> &utt,
                      int d, int64_t slots)
{
    const int64_t lag = (31 * d + HFA_SKEW_BLK - 1) / HFA_SKEW_BLK + 1;
    std::priority_queue<int64_t, std::vector<int64_t>, std::greater<int64_t>> free_at;
    int64_t makespan = 0, left_start = 0;
    for (int i = begin; i < begin + count; ++i) {
        int64_t start = 0;
        if ((int64_t)free_at.size() == slots) {
            start = free_at.top();
            free_at.pop();
        }
        if (items[i].band > 0) start = std::max(start, left_start + lag);
        const int64_t end = start + hfa_skew_blocks(d, utt[items[i].utt].T);
        free_at.push(end);
        left_start = start;
        makespan = std::max(makespan, end);
    }
    return makespan;
}

}  // namespace

// Workspace layout (byte offsets from the workspace base, every region 256-byte aligned):
//   [utt table][ids][order lists][row_blocks][inputs]   <- "head", uploaded from the plan
//   [emis][edge2][edge_p][bp][path_state][rev_idx][rev_t][dp_last]
struct hfa_plan {
    int32_t n_utt = 0, vocab = 0;
    double frame_length = 0.0;
    std::vector<HfaUtt> utt;
    std::vector<int32_t> ids;
    std::vector<int32_t> col_ids;              // compacted emission columns (HfaWs::col_ids / colmap)
    std::vector<uint8_t> colmap;
    int32_t n_compact = 0;
    int64_t stored_emis = 0;                   // floats the emission kernels write (compacted where possible)
    std::vector<int64_t> frame_off, seg_off;   // [n+1]
    // bucket lists: class c = K-1 for the warp kernel (K states per lane), class 8 = CTA kernel,
    // then the backtrace list (valid utterances by descending T, then the invalid ones)
    std::vector<int32_t> order;                // concatenation of all lists
    int32_t class_begin[HFA_NUM_CLASSES + 2] = {0};
    int32_t class_count[HFA_NUM_CLASSES + 1] = {0};
    int32_t cta_max_sp = 0, max_sp = 4;
    int32_t warp_all_begin = 0, warp_all_count = 0, warp_max_k = 0;   // merged warp-kernel list
    int32_t warp_max_pair_k = 0, pair_count = 0;                     // ... of which in the SP-aware pair layout
    // banded (halo) kernel work lists: [0] S <= 256 utterances of a small batch (latency regime,
    // 2 states per lane), [1] long phoneme sequences (S > 256, band_k[1] states per lane)
    std::vector<HfaBandItem> band_items;
    int32_t band_begin[2] = {0, 0}, band_count[2] = {0, 0}, band_k[2] = {2, 4};
    // > 0: the list runs in the skewed-wavefront kernel (hfa_dp_skew.cu) with this many frames of skew
    // per state -- 32 / 30-state strips, one state per lane -- instead of the halo bands
    int32_t band_skew[2] = {0, 0};
    // strips of the skewed kernel resident per SM (4 or 5: the kernel's ring has 6 or 5 stages)
    int32_t skew_ctas[2] = {5, 5};
    int32_t skew_slow = 0;                     // 1: every block of the skewed kernel through its guarded body
    // true: the strips and bands read their emission tiles through TMA tensor maps, which hfa_plan_upload writes;
    // false: the halo bands take the strips' place and their producers copy one frame row at a time
    bool use_tmaps = false;
    int64_t band_xchg_elems = 0, dp_store_elems = 0;
    std::vector<int32_t> jblk_utt, jblk_first; // jump-table kernel: 256-word blocks per utterance of the table set
    int32_t n_kept = 0;                        // utterances that keep dp
    int32_t bt_begin = 0;
    // the kept-dp utterances split into the walk set (backpointers staged in shared memory, hfa_backtrace_walk_kernel)
    // and the table set (jump tables + hfa_backtrace_tables_kernel); both lists follow the backtrace list in `order`
    int32_t walk_begin = 0, n_walk = 0, tab_begin = 0, n_tab = 0;
    int64_t walk_smem = 0;                     // dynamic shared memory of the walk launch: its largest utterance
    std::vector<int32_t> row_blocks;           // [n+1]
    std::vector<int32_t> block_utt;            // [row_blocks[n]]
    int64_t total_frames = 0, total_states = 0, total_cells = 0, padded_cells = 0;
    int64_t total_words = 0, total_edge = 0;
    // byte offsets
    int64_t o_colids = 0, o_colmap = 0, o_emode = 0;
    int64_t o_utt = 0, o_ids = 0, o_order = 0, o_rowblk = 0, o_blkutt = 0, o_inputs = 0, head_bytes = 0;
    int64_t o_emis = 0, o_edge2 = 0, o_edgep = 0, o_bp = 0, o_path = 0, o_revi = 0, o_revt = 0,
            o_last = 0, o_dpst = 0, o_jump = 0, o_moves = 0, o_rowent = 0, o_band_items = 0, o_jblk_utt = 0, o_jblk_first = 0, o_band_ticket = 0, o_band_xchg = 0, band_bytes = 0, o_tmaps = 0, ws_bytes = 0;
    int32_t n_tmaps = 0;                       // banded utterances (one emission tensor map each)
    std::vector<unsigned char> head;           // host image of the head (without inputs)
    HfaResultLayout res{};
    // What hfa_set_inputs / hfa_set_inputs_device last stored in each workspace this plan was used with
    // (one plan may serve several workspaces, from several host threads): > 0 when every utterance's
    // logits have unit column stride, element-aligned base pointers and positive row strides of at most
    // this many elements -- then the logits rows can travel by TMA.  A per-workspace record, not plan state.
    mutable std::mutex layout_mu;
    mutable std::unordered_map<const void *, int64_t> layout_of;
    int64_t row_stride_of(const void *workspace) const
    {
        std::lock_guard<std::mutex> g(layout_mu);
        auto it = layout_of.find(workspace);
        return it == layout_of.end() ? 0 : it->second;
    }
    void set_row_stride(const void *workspace, int64_t v) const
    {
        std::lock_guard<std::mutex> g(layout_mu);
        layout_of[workspace] = v;
    }
};

namespace {

HfaWs make_ws(const hfa_plan *p, void *workspace)
{
    unsigned char *b = static_cast<unsigned char *>(workspace);
    HfaWs w;
    w.utt = reinterpret_cast<const HfaUtt *>(b + p->o_utt);
    w.ids = reinterpret_cast<const int32_t *>(b + p->o_ids);
    w.order = reinterpret_cast<const int32_t *>(b + p->o_order);
    w.row_blocks = reinterpret_cast<const int32_t *>(b + p->o_rowblk);
    w.block_utt = reinterpret_cast<const int32_t *>(b + p->o_blkutt);
    w.inputs = reinterpret_cast<HfaInput *>(b + p->o_inputs);
    w.emis = reinterpret_cast<float *>(b + p->o_emis);
    w.edge2 = reinterpret_cast<float2 *>(b + p->o_edge2);
    w.edge_p = reinterpret_cast<float *>(b + p->o_edgep);
    w.bp = reinterpret_cast<uint32_t *>(b + p->o_bp);
    w.path_state = reinterpret_cast<int32_t *>(b + p->o_path);
    w.rev_idx = reinterpret_cast<int32_t *>(b + p->o_revi);
    w.rev_t = reinterpret_cast<int32_t *>(b + p->o_revt);
    w.dp_last = reinterpret_cast<float *>(b + p->o_last);
    w.dp_store = reinterpret_cast<float *>(b + p->o_dpst);
    w.jump = reinterpret_cast<uint8_t *>(b + p->o_jump);
    w.moves = reinterpret_cast<uint8_t *>(b + p->o_moves);
    w.row_entry = reinterpret_cast<int32_t *>(b + p->o_rowent);
    w.jblk_utt = reinterpret_cast<const int32_t *>(b + p->o_jblk_utt);
    w.jblk_first = reinterpret_cast<const int32_t *>(b + p->o_jblk_first);
    w.tmaps = (p->n_tmaps > 0 && p->use_tmaps) ? b + p->o_tmaps : nullptr;
    w.col_ids = reinterpret_cast<const int32_t *>(b + p->o_colids);
    w.colmap = reinterpret_cast<const uint8_t *>(b + p->o_colmap);
    w.emis_mode = reinterpret_cast<int32_t *>(b + p->o_emode);
    w.band_items = reinterpret_cast<const HfaBandItem *>(b + p->o_band_items);
    w.band_ticket = reinterpret_cast<int32_t *>(b + p->o_band_ticket);
    w.band_xchg = reinterpret_cast<uint4 *>(b + p->o_band_xchg);
    return w;
}

HfaLaunchCtx make_ctx(const hfa_plan *p, void *workspace, void *stream)
{
    HfaLaunchCtx c;
    c.ws = make_ws(p, workspace);
    c.n_utt = p->n_utt;
    c.vocab = p->vocab;
    c.frame_length = p->frame_length;
    c.stream = static_cast<cudaStream_t>(stream);
    return c;
}

HfaResultPtrs make_res(const hfa_plan *p, void *result)
{
    unsigned char *b = static_cast<unsigned char *>(result);
    HfaResultPtrs r;
    r.status = reinterpret_cast<int32_t *>(b + p->res.status);
    r.n_seg = reinterpret_cast<int32_t *>(b + p->res.n_seg);
    r.end_state = reinterpret_cast<int32_t *>(b + p->res.end_state);
    r.final_score = reinterpret_cast<float *>(b + p->res.final_score);
    r.total_conf = reinterpret_cast<float *>(b + p->res.total_conf);
    r.ph_idx_seq = reinterpret_cast<int32_t *>(b + p->res.ph_idx_seq);
    r.ph_time_int = reinterpret_cast<int32_t *>(b + p->res.ph_time_int);
    r.intervals = reinterpret_cast<double *>(b + p->res.intervals);
    return r;
}

}  // namespace

extern "C" {

int hfa_abi_version(void) { return HFA_ABI_VERSION; }
const char *hfa_last_error(void) { return g_err; }
int64_t hfa_launch_count(void) { return g_launches.load(); }

int hfa_plan_create(int32_t n_utt, int32_t vocab_size, const int32_t *T, const int32_t *S,
                    const int32_t *ph_ids, double frame_length, hfa_plan **out)
{
    if (out == nullptr) return fail(HFA_ERR_ARG, "hfa_plan_create: out is NULL");
    *out = nullptr;
    if (n_utt < 0 || vocab_size < 1 || (n_utt > 0 && (!T || !S || !ph_ids)))
        return fail(HFA_ERR_ARG, "hfa_plan_create: bad arguments (n_utt=%d, V=%d)", n_utt,
                    vocab_size);
    hfa_plan *p = new (std::nothrow) hfa_plan();
    if (!p) return fail(HFA_ERR_NOMEM, "hfa_plan_create: out of host memory");

    // Routing overrides (DESIGN §4.6), read here and nowhere else: the plan keeps what it read, and no call made
    // with it looks at the environment again.  Unset, each leaves the planner's own choice.
    // HFA_LATENCY_MODE: 0 never cut utterances with S <= 256 into strips / bands, 2 always, -1: by the budget below
    int lat_mode = -1;
    if (const char *e = std::getenv("HFA_LATENCY_MODE")) lat_mode = e[0] - '0';
    // HFA_BAND_MAX: strip / band budget of the latency route and of the S > 256 list (3072: the measured crossover)
    int64_t band_max = 3072;
    if (const char *e = std::getenv("HFA_BAND_MAX")) band_max = std::atoll(e);
    // HFA_SKEW_D = 2 | 3: frames of skew per state of the skewed kernel; HFA_LAT_KERNEL = band: halo bands instead
    int skew_d = 2;
    if (const char *e = std::getenv("HFA_SKEW_D")) skew_d = (std::atoi(e) == 3) ? 3 : 2;
    if (const char *e = std::getenv("HFA_LAT_KERNEL")) { if (e[0] == 'b') skew_d = 0; }
    // HFA_SKEW_SLOW = 1: every block of the skewed kernel through its guarded body
    if (const char *e = std::getenv("HFA_SKEW_SLOW")) p->skew_slow = e[0] == '1' ? 1 : 0;
    // HFA_SKEW_CTAS = 4 | 5: strips resident per SM, instead of the list schedule's choice
    int force_ctas = 0;
    if (const char *e = std::getenv("HFA_SKEW_CTAS")) force_ctas = std::atoi(e);
    // HFA_BIG_KERNEL = cta | band: kernel of the S > 256 list (-1: by the budget); HFA_BIG_K = 2 | 4 | 8: states
    // per lane of its halo bands
    int big_mode = -1;
    if (const char *e = std::getenv("HFA_BIG_KERNEL")) big_mode = (e[0] == 'b');
    int big_k = 0;
    if (const char *e = std::getenv("HFA_BIG_K")) big_k = std::atoi(e);
    // HFA_KEEP_DP = 0: the strips and bands keep no dp (the backtrace re-scores the path)
    bool keep_dp = true;
    if (const char *e = std::getenv("HFA_KEEP_DP")) keep_dp = (e[0] != '0');
    // HFA_BT_WALK = 0: jump tables instead of the shared-memory walk for every kept-dp utterance
    int bt_walk = 2;
    if (const char *e = std::getenv("HFA_BT_WALK")) bt_walk = std::atoi(e);
    // HFA_PAIR = 0: never the SP-aware pair layout, 2: wherever possible, 1: where the cost rule picks it
    int pair_mode = 1;
    if (const char *e = std::getenv("HFA_PAIR")) pair_mode = std::atoi(e);
    // HFA_COMPACT = 0: plain [T][Sp] emission rows for the pair layout
    bool compact = true;
    if (const char *e = std::getenv("HFA_COMPACT")) compact = e[0] != '0';
    // HFA_NO_TENSORMAP = 1: no TMA tensor maps, as when the driver lacks cuTensorMapEncodeTiled
    p->use_tmaps = tensor_map_encoder() != nullptr;
    if (const char *e = std::getenv("HFA_NO_TENSORMAP")) { if (e[0] == '1') p->use_tmaps = false; }

    try {
        p->n_utt = n_utt;
        p->vocab = vocab_size;
        p->frame_length = frame_length;
        p->utt.resize((size_t)n_utt);
        p->frame_off.assign((size_t)n_utt + 1, 0);
        p->seg_off.assign((size_t)n_utt + 1, 0);
        p->row_blocks.assign((size_t)n_utt + 1, 0);
        for (int32_t b = 0; b < n_utt; ++b)
            p->seg_off[b + 1] = p->seg_off[b] + std::max<int32_t>(S[b], 0);
        p->total_states = p->seg_off[n_utt];
        p->ids.assign(ph_ids, ph_ids + p->total_states);

        // giant: S > HFA_CTA_MAX_S, beyond the CTA kernel -- always in the skewed strips (or halo bands), routed
        // after everything else so that the other utterances of the batch are placed as if it were not there
        std::vector<int32_t> lists[HFA_NUM_CLASSES + 1], invalid, giant;
        int64_t emis = 0, edge = 0, words = 0, cells = 0, frames = 0;
        for (int32_t b = 0; b < n_utt; ++b) {
            HfaUtt &m = p->utt[b];
            std::memset(&m, 0, sizeof(m));
            const int32_t t = T[b], s = S[b];
            int32_t st = HFA_UTT_OK;
            if (s < 1) st = HFA_UTT_NO_STATES;
            else if (t < 1) st = HFA_UTT_EMPTY;
            else if (s > HFA_MAX_STATES) st = HFA_UTT_TOO_MANY_STATES;
            else {
                const int32_t *id = ph_ids + p->seg_off[b];
                for (int32_t i = 0; i < s; ++i)
                    if (id[i] < 0 || id[i] >= vocab_size) { st = HFA_UTT_BAD_ID; break; }
            }
            m.status = st;
            m.seg_off = p->seg_off[b];
            m.frame_off = frames;
            m.cell_off = cells;
            m.emis_off = emis;
            m.edge_off = edge;
            m.bp_off = words;
            m.dp_off = -1;
            m.tmap = -1;
            p->frame_off[b] = frames;
            if (st == HFA_UTT_OK) {
                m.T = t;
                m.S = s;
                m.Sp = (s + 3) & ~3;
                frames += t;
                cells += (int64_t)t * s;
                emis += (int64_t)t * m.Sp;
                edge += align_up(t, HFA_TILE_T);
                words += (int64_t)((t + 15) / 16) * m.Sp;
                p->row_blocks[b + 1] = p->row_blocks[b] + (t + HFA_EMIS_ROWS - 1) / HFA_EMIS_ROWS;
                p->max_sp = std::max(p->max_sp, m.Sp);
                if (m.Sp <= HFA_WARP_MAX_S) lists[(m.Sp + 31) / 32 - 1].push_back(b);
                else if (s > HFA_CTA_MAX_S) giant.push_back(b);
                else {
                    lists[HFA_NUM_CLASSES].push_back(b);
                    p->cta_max_sp = std::max(p->cta_max_sp, m.Sp);
                }
            } else {
                p->row_blocks[b + 1] = p->row_blocks[b];
                invalid.push_back(b);
            }
        }
        p->frame_off[n_utt] = frames;
        p->total_frames = frames;
        p->total_cells = cells;
        p->padded_cells = emis;
        p->total_words = words;
        p->total_edge = edge;

        // longest utterances first inside every bucket (they bound the tail of the launch)
        auto by_len = [&](int32_t a, int32_t b) {
            return p->utt[a].T != p->utt[b].T ? p->utt[a].T > p->utt[b].T : a < b;
        };
        std::vector<int32_t> all;
        for (int c = 0; c <= HFA_NUM_CLASSES; ++c) {
            std::sort(lists[c].begin(), lists[c].end(), by_len);
            p->class_begin[c] = (int32_t)p->order.size();
            p->class_count[c] = (int32_t)lists[c].size();
            p->order.insert(p->order.end(), lists[c].begin(), lists[c].end());
            all.insert(all.end(), lists[c].begin(), lists[c].end());
        }
        all.insert(all.end(), giant.begin(), giant.end());
        // Routing.  The recurrence is a serial chain in t, so a batch that cannot fill the machine
        // with one warp per utterance (BASELINE configs 1-3) is bounded by the per-frame latency of
        // its longest utterances.  Such batches go to the banded kernel (hfa_dp_band_kernel): every
        // utterance becomes several 2-states-per-lane warps on different SMs.  Big batches keep
        // one warp per utterance (no redundant halo work).
        // Latency-regime kernel: the skewed wavefront (default; needs the TMA tensor maps) or the halo bands.
        if (!p->use_tmaps) skew_d = 0;
        auto n_bands = [&](int32_t b, int k) {
            if (k == 1) return hfa_skew_strips(p->utt[b].Sp);
            const int w = 32 * k, own = w - 32, sp = p->utt[b].Sp;
            return sp <= w ? 1 : (sp - 32 + own - 1) / own;
        };
        // measured crossover (profiles/r2_routing_crossover.json, B200): strips win for 256 / 512 utterances
        // (820 / 1674 strips: 0.22 vs 0.44 ms, 0.33 vs 0.48 ms per step), tie at 1024 (3310 strips: 0.550 vs
        // 0.553 ms), one warp per utterance wins at 2048 (6582 strips: 1.03 vs 0.73 ms)
        std::vector<int32_t> lat_band;
        if (lat_mode != 0) {
            int64_t nb = 0;
            for (int c = 0; c < HFA_NUM_CLASSES; ++c)
                for (int32_t b : lists[c]) nb += n_bands(b, skew_d > 0 ? 1 : 2);
            if (skew_d > 0) {
                p->band_k[0] = 1;
                p->band_skew[0] = skew_d;
            }
            if (lat_mode == 2 || (nb > 0 && nb <= band_max)) {
                for (int c = 0; c < HFA_NUM_CLASSES; ++c) {
                    lat_band.insert(lat_band.end(), lists[c].begin(), lists[c].end());
                    lists[c].clear();
                    p->class_count[c] = 0;
                }
                std::sort(lat_band.begin(), lat_band.end(), by_len);
            }
        }
        std::vector<int32_t> big_band;
        {
            // states per lane of the long-sequence bands: as few as the band budget allows (measured on
            // config 3: 2.5 ms with 2, 3.8 ms with 4, 9.9 ms with 8, 17 ms in the CTA kernel)
            auto count = [&](int k) {
                int64_t nb = 0;
                for (int32_t b : lists[HFA_NUM_CLASSES]) nb += n_bands(b, k);
                return nb;
            };
            if (big_k != 2 && big_k != 4 && big_k != 8) {
                big_k = 8;
                for (int k : {2, 4, 8})
                    if (count(k) <= band_max) { big_k = k; break; }
                if (skew_d > 0 && count(1) <= band_max) big_k = 1;      // strips of the skewed kernel
            }
            p->band_k[1] = big_k;
            if (big_k == 1) p->band_skew[1] = skew_d;
            if (big_mode == 1 || (big_mode == -1 && count(big_k) <= band_max)) {
                big_band = lists[HFA_NUM_CLASSES];
                lists[HFA_NUM_CLASSES].clear();
                p->class_count[HFA_NUM_CLASSES] = 0;
            }
            // The giants join that list whatever the budget.  When it is otherwise empty (the other long
            // utterances, if any, stay in the CTA kernel) it becomes strips, or 2-states-per-lane halo bands
            // without tensor maps.  When it already holds the batch's other long utterances it keeps their kernel:
            // strips, or halo bands if those won the budget or HFA_BIG_K / the missing tensor maps chose them.
            if (!giant.empty()) {
                if (big_band.empty()) {
                    p->band_k[1] = skew_d > 0 ? 1 : 2;
                    p->band_skew[1] = skew_d;
                }
                big_band.insert(big_band.end(), giant.begin(), giant.end());
                std::sort(big_band.begin(), big_band.end(), by_len);
            }
        }
        auto add_bands = [&](const std::vector<int32_t> &utts, int which) {
            const int k = p->band_k[which];
            const int sd = p->band_skew[which];
            p->band_begin[which] = (int32_t)p->band_items.size();
            for (int32_t b : utts) {
                const int nb = n_bands(b, k);
                const int64_t tiles = (p->utt[b].T + 15) / 16;
                p->utt[b].skew_d = sd;
                // the banded routing is the latency regime: the forward pass also keeps dp (4 B per
                // cell more HBM traffic, irrelevant there) so that the backtrace reads dp[t, s_t]
                // instead of re-running the serial chain along the path
                p->utt[b].band_k = k;
                p->utt[b].tmap = p->n_tmaps++;
                if (keep_dp) {
                    p->utt[b].dp_off = p->dp_store_elems;
                    // bands: one [T][32 k] block per band; strips: one 128-byte row per iteration
                    p->dp_store_elems += sd > 0 ? (int64_t)nb * hfa_skew_blocks(sd, p->utt[b].T) * HFA_SKEW_BLK * 32
                                                : (int64_t)nb * p->utt[b].T * 32 * k;
                }
                for (int j = 0; j < nb; ++j) {
                    const bool has_right = j + 1 < nb;
                    p->band_items.push_back(HfaBandItem{b, j, has_right ? p->band_xchg_elems : 0});
                    // exchange slots (16 bytes each): bands 32 states x 2 per tile, strips one per frame
                    if (has_right) p->band_xchg_elems += sd > 0 ? (tiles + 1) / 2 * 32 : tiles * 64;
                }
            }
            p->band_count[which] = (int32_t)p->band_items.size() - p->band_begin[which];
        };
        add_bands(lat_band, 0);
        add_bands(big_band, 1);
        // Strips per SM.  Five 2-warp CTAs put two compute warps on one scheduler partition; four give each its
        // own partition, which shortens the block period of the critical chain (DESIGN §4.3), but fewer strips
        // start in the first wave.  Four when the list schedule is not longer with them (configs 1-3: the
        // strips that miss the first wave belong to short utterances), five otherwise (512 utterances and up).
        // HFA_SKEW_CTAS = 4 | 5 forces one residency (tests run both ring sizes on the same batches).
        for (int wh = 0; wh < 2; ++wh) {
            if (p->band_skew[wh] <= 0 || p->band_count[wh] == 0) continue;
            if (force_ctas == 4 || force_ctas == 5) {
                p->skew_ctas[wh] = force_ctas;
                continue;
            }
            const int64_t m4 = skew_makespan(p->band_items, p->band_begin[wh], p->band_count[wh], p->utt,
                                             p->band_skew[wh], 4LL * sm_count());
            const int64_t m5 = skew_makespan(p->band_items, p->band_begin[wh], p->band_count[wh], p->utt,
                                             p->band_skew[wh], 5LL * sm_count());
            p->skew_ctas[wh] = m4 <= m5 ? 4 : 5;
        }
        // Backtrace of the utterances that keep dp.  The walk stages an utterance's backpointer words in shared
        // memory and walks them serially, one CTA per utterance; the jump tables make the serial part one lookup
        // per 16 frames but cost a kernel that walks every word.  Measured (profiles/r5_bt_routes.jsonl, B200): the
        // walk wins on every batch it fits, 256 utterances of T = 500-6000 and S = 40-256 up to 192 KB of words
        // at one CTA per SM, so an utterance takes it whenever its words fit in one CTA's shared memory; giants
        // (S > 8192) keep the tables.  HFA_BT_WALK = 0: never (tests compare the two routes).
        std::vector<int32_t> walk_list, tab_list;
        std::vector<char> walks((size_t)n_utt, 0);
        for (int32_t b : all) {
            const HfaUtt &m = p->utt[b];
            if (m.dp_off < 0) continue;
            p->n_kept += 1;
            const bool walk = bt_walk != 0 && m.S <= HFA_CTA_MAX_S &&
                              hfa_bt_walk_smem(m.T, m.S, m.Sp) <= HFA_BT_WALK_SMEM_LIMIT;
            (walk ? walk_list : tab_list).push_back(b);
            if (walk) {
                walks[(size_t)b] = 1;
                p->walk_smem = std::max(p->walk_smem, hfa_bt_walk_smem(m.T, m.S, m.Sp));
            }
        }
        p->n_walk = (int32_t)walk_list.size();
        p->n_tab = (int32_t)tab_list.size();
        // jump-table kernel (the table set): one thread per backpointer word
        p->jblk_first.assign((size_t)n_utt + 1, 0);
        for (int32_t b = 0; b < n_utt; ++b) {
            const HfaUtt &m = p->utt[b];
            const int64_t w = (m.status == 0 && m.dp_off >= 0 && !walks[(size_t)b]) ? (int64_t)((m.T + 15) / 16) * m.Sp : 0;
            const int32_t nblk = (int32_t)((w + 255) / 256);
            p->jblk_first[b + 1] = p->jblk_first[b] + nblk;
            p->jblk_utt.insert(p->jblk_utt.end(), (size_t)nblk, b);
        }
        // merged warp-kernel list: longest expected run time first (frames x per-frame cost, which
        // grows with the states per lane)
        // SP-aware pair layout (hfa_dp_pair_body): the state axis regrouped into {SP, phoneme} pairs, KP pairs per
        // lane.  Possible when no two SPs are adjacent and KP <= 4.  Decided for the BATCH, not per utterance: the
        // merged kernel keeps one code path hot per class present, and a launch that mixes pair and plain bodies
        // runs out of instruction cache (B200, config 4, DP stage: 0.462 ms all plain, 0.433 ms pairs only where
        // they are cheaper (5 + 3 bodies hot, no_instruction the top stall), 0.370 ms every utterance in pairs).
        // So: if the frames-weighted instruction count of the possible utterances is lower in pairs, all of them
        // go there.  Instructions per frame counted in the SASS (loop bodies + the per-tile work / 8):
        // 16 + 21 K plain, 17 + 25 KP in pairs.   HFA_PAIR = 0: never | 2: whenever possible | unset: as above.
        std::vector<int32_t> warp_all;
        std::vector<std::pair<int32_t, int>> pairable;          // (utterance, pairs per lane)
        int64_t sum_pair = 0, sum_plain = 0;
        for (int c = 0; c < HFA_NUM_CLASSES; ++c) {
            warp_all.insert(warp_all.end(), lists[c].begin(), lists[c].end());
            for (int32_t b : lists[c]) {
                const HfaUtt &m = p->utt[b];
                const int32_t *id = ph_ids + m.seg_off;
                int phon = 0;
                bool ok = pair_mode > 0;
                for (int32_t i = 0; i < m.S && ok; ++i) {
                    phon += id[i] != 0;
                    if (i > 0 && id[i] == 0 && id[i - 1] == 0) ok = false;
                }
                const int kp = (phon + (id[m.S - 1] == 0) + 31) / 32;
                if (ok && kp <= HFA_PAIR_MAX_K) {
                    pairable.push_back({b, kp});
                    sum_pair += (int64_t)m.T * (17 + 25 * kp);
                    sum_plain += (int64_t)m.T * (16 + 21 * (c + 1));
                }
                p->warp_max_k = std::max(p->warp_max_k, c + 1);
            }
        }
        // Compacted emission rows for those utterances (HfaWs::colmap): every slot of the pair layout reads its
        // column through its own address register, so pointing states with the same id at ONE column is free.
        // HFA_COMPACT=0 keeps the plain [T][Sp] rows, and so does V > 255 (a colmap entry is one byte).
        compact = compact && vocab_size <= 255;
        p->col_ids.assign((size_t)(p->total_states + 4 * (int64_t)n_utt), vocab_size);
        p->colmap.assign((size_t)p->total_states, 0);
        if (pair_mode >= 2 || sum_pair < sum_plain)
            for (const auto &bk : pairable) {
                HfaUtt &m = p->utt[bk.first];
                m.pair_k = bk.second;
                p->warp_max_pair_k = std::max(p->warp_max_pair_k, bk.second);
                p->pair_count += 1;
                if (!compact) continue;
                const int32_t *id = ph_ids + m.seg_off;
                int col_of[256];
                std::fill(col_of, col_of + 256, -1);
                for (int32_t i = 0; i < m.S; ++i) col_of[id[i]] = 0;
                int d = 0;
                for (int v = 0; v < vocab_size; ++v)
                    if (col_of[v] == 0) col_of[v] = d++;
                const int dp = (d + 3) & ~3;
                if (dp >= m.Sp) continue;                              // nothing to gain
                m.Dp = dp;
                p->n_compact += 1;
                int32_t *ci = p->col_ids.data() + m.seg_off + 4 * (int64_t)bk.first;
                for (int v = 0; v < vocab_size; ++v)
                    if (col_of[v] >= 0) ci[col_of[v]] = v;
                for (int32_t i = 0; i < m.S; ++i) p->colmap[(size_t)(m.seg_off + i)] = (uint8_t)col_of[id[i]];
            }
        for (const HfaUtt &m : p->utt)
            if (m.status == 0) p->stored_emis += (int64_t)m.T * (m.Dp > 0 ? m.Dp : m.Sp);
        // launch order = expected run time, longest first.  Measured on config 4 (B200, DP stage): all-plain batch
        // 0.462 ms with round 1's weights T (2 + K) against 0.485 ms with the instruction counts; batch in pairs
        // 0.388 ms with the instruction counts against 0.405 ms with T (2 + K) -- each layout keeps its winner.
        const bool old_order = p->pair_count == 0;
        auto cost = [&](int32_t b) {
            const HfaUtt &m = p->utt[b];
            if (old_order) return (int64_t)m.T * (2 + (m.Sp + 31) / 32);
            return (int64_t)m.T * (m.pair_k > 0 ? 17 + 25 * m.pair_k : 16 + 21 * ((m.Sp + 31) / 32));
        };
        std::sort(warp_all.begin(), warp_all.end(),
                  [&](int32_t a, int32_t b) { return cost(a) != cost(b) ? cost(a) > cost(b) : a < b; });
        p->warp_all_begin = (int32_t)p->order.size();
        p->warp_all_count = (int32_t)warp_all.size();
        p->order.insert(p->order.end(), warp_all.begin(), warp_all.end());
        std::sort(all.begin(), all.end(), by_len);
        p->bt_begin = (int32_t)p->order.size();
        p->order.insert(p->order.end(), all.begin(), all.end());
        p->order.insert(p->order.end(), invalid.begin(), invalid.end());
        p->walk_begin = (int32_t)p->order.size();
        p->order.insert(p->order.end(), walk_list.begin(), walk_list.end());
        p->tab_begin = (int32_t)p->order.size();
        p->order.insert(p->order.end(), tab_list.begin(), tab_list.end());

        // workspace layout
        int64_t o = 0;
        auto region = [&](int64_t bytes) { const int64_t at = o; o = align_up(o + bytes, 256); return at; };
        p->o_utt = region((int64_t)n_utt * sizeof(HfaUtt));
        p->o_ids = region(p->total_states * 4);
        p->o_order = region((int64_t)p->order.size() * 4);
        p->o_rowblk = region((int64_t)(n_utt + 1) * 4);
        p->block_utt.reserve((size_t)p->row_blocks[n_utt]);
        for (int32_t b = 0; b < n_utt; ++b)
            p->block_utt.insert(p->block_utt.end(), (size_t)(p->row_blocks[b + 1] - p->row_blocks[b]), b);
        p->o_blkutt = region((int64_t)p->block_utt.size() * 4);
        p->o_band_items = region((int64_t)p->band_items.size() * sizeof(HfaBandItem));
        p->o_jblk_utt = region((int64_t)p->jblk_utt.size() * 4);
        p->o_jblk_first = region((int64_t)p->jblk_first.size() * 4);
        p->o_colids = region(p->n_compact > 0 ? (int64_t)p->col_ids.size() * 4 : 0);
        p->o_colmap = region(p->n_compact > 0 ? (int64_t)p->colmap.size() : 0);
        p->head_bytes = o;
        p->o_inputs = region((int64_t)n_utt * sizeof(HfaInput));
        p->o_emis = region(emis * 4);
        p->o_edge2 = region(edge * 8);
        p->o_edgep = region(edge * 4 + 4);      // +1: seg_time reads p[t+1] only when t+1 < T
        p->o_bp = region(words * 4);
        p->o_path = region(frames * 4);
        p->o_revi = region(p->total_states * 4);
        p->o_revt = region(p->total_states * 4);
        p->o_last = region((int64_t)n_utt * 8);
        p->o_emode = region(p->n_compact > 0 ? (int64_t)n_utt * 4 : 0);
        p->o_dpst = region(p->dp_store_elems * 4);
        const bool jump_tables = p->n_tab > 0;              // kept-dp utterances the walk does not take
        p->o_jump = region(jump_tables ? words : 0);
        p->o_moves = region(jump_tables ? words : 0);
        p->o_rowent = region(jump_tables ? edge / 16 * 4 : 0);

        p->o_tmaps = region((int64_t)p->n_tmaps * 128);
        p->o_band_ticket = region(p->band_items.empty() ? 0 : 8);
        p->o_band_xchg = region(p->band_xchg_elems * 16);
        p->band_bytes = o - p->o_band_ticket;
        p->ws_bytes = std::max<int64_t>(o, 256);

        p->head.assign((size_t)p->head_bytes, 0);
        if (n_utt > 0) {
            std::memcpy(p->head.data() + p->o_utt, p->utt.data(), (size_t)n_utt * sizeof(HfaUtt));
            if (p->total_states)
                std::memcpy(p->head.data() + p->o_ids, p->ids.data(), (size_t)p->total_states * 4);
            std::memcpy(p->head.data() + p->o_order, p->order.data(), p->order.size() * 4);
        }
        if (!p->band_items.empty())
            std::memcpy(p->head.data() + p->o_band_items, p->band_items.data(),
                        p->band_items.size() * sizeof(HfaBandItem));
        if (!p->jblk_utt.empty())
            std::memcpy(p->head.data() + p->o_jblk_utt, p->jblk_utt.data(), p->jblk_utt.size() * 4);
        std::memcpy(p->head.data() + p->o_jblk_first, p->jblk_first.data(), p->jblk_first.size() * 4);
        if (p->n_compact > 0) {
            std::memcpy(p->head.data() + p->o_colids, p->col_ids.data(), p->col_ids.size() * 4);
            if (!p->colmap.empty()) std::memcpy(p->head.data() + p->o_colmap, p->colmap.data(), p->colmap.size());
        }
        std::memcpy(p->head.data() + p->o_rowblk, p->row_blocks.data(), (size_t)(n_utt + 1) * 4);
        if (!p->block_utt.empty())
            std::memcpy(p->head.data() + p->o_blkutt, p->block_utt.data(), p->block_utt.size() * 4);

        // result blob layout
        int64_t r = 0;
        auto rreg = [&](int64_t bytes) { const int64_t at = r; r = align_up(r + bytes, 16); return at; };
        p->res.status = rreg((int64_t)n_utt * 4);
        p->res.n_seg = rreg((int64_t)n_utt * 4);
        p->res.end_state = rreg((int64_t)n_utt * 4);
        p->res.final_score = rreg((int64_t)n_utt * 4);
        p->res.total_conf = rreg((int64_t)n_utt * 4);
        p->res.ph_idx_seq = rreg(p->total_states * 4);
        p->res.ph_time_int = rreg(p->total_states * 4);
        p->res.intervals = rreg(p->total_states * 16);
        p->res.total_bytes = std::max<int64_t>(r, 16);
    } catch (const std::bad_alloc &) {
        delete p;
        return fail(HFA_ERR_NOMEM, "hfa_plan_create: out of host memory");
    }
    *out = p;
    return HFA_OK;
}

void hfa_plan_destroy(hfa_plan *plan) { delete plan; }

int64_t hfa_plan_workspace_bytes(const hfa_plan *p) { return p ? p->ws_bytes : 0; }
int64_t hfa_plan_total_frames(const hfa_plan *p) { return p ? p->total_frames : 0; }
int64_t hfa_plan_total_states(const hfa_plan *p) { return p ? p->total_states : 0; }
int64_t hfa_plan_total_cells(const hfa_plan *p) { return p ? p->total_cells : 0; }
const int64_t *hfa_plan_frame_offsets(const hfa_plan *p) { return p ? p->frame_off.data() : nullptr; }
const int64_t *hfa_plan_seg_offsets(const hfa_plan *p) { return p ? p->seg_off.data() : nullptr; }

int hfa_plan_result_layout(const hfa_plan *p, HfaResultLayout *out)
{
    if (!p || !out) return fail(HFA_ERR_ARG, "hfa_plan_result_layout: NULL argument");
    *out = p->res;
    return HFA_OK;
}

int hfa_plan_algorithmic_bytes(const hfa_plan *p, int32_t dtype, int64_t out[3])
{
    if (!p || !out) return fail(HFA_ERR_ARG, "hfa_plan_algorithmic_bytes: NULL argument");
    const int64_t in_b = (dtype == HFA_DTYPE_F32) ? 4 : 2;
    int64_t words = 0, kept_cells = 0, kept_frames = 0;
    for (const HfaUtt &m : p->utt)
        if (m.status == 0) {
            words += (int64_t)((m.T + 15) / 16) * m.S;
            if (m.dp_off >= 0) {
                kept_cells += (int64_t)m.T * m.S;
                kept_frames += m.T;
            }
        }
    // unpadded figures (SURVEY.md 8d): emission reads V logits + 1 edge logit per frame and writes
    // S emissions + {edge_log, not_edge_log, edge_pred}; the DP reads them back and writes 2 bits
    // per cell; the backtrace reads the path's backpointers and operands and writes the segments.
    out[0] = p->total_frames * ((int64_t)p->vocab * in_b + in_b) + p->total_cells * 4 +
             p->total_frames * 12;
    // banded routing: the forward pass also writes dp (4 B per cell) and the backtrace reads
    // dp[t, s_t] instead of the path's emissions and edge logs
    out[1] = p->total_cells * 4 + p->total_frames * 8 + words * 4 + kept_cells * 4;
    out[2] = (p->total_frames - kept_frames) * (8 + 8) + kept_frames * (8 + 4) + p->total_states * 24;
    return HFA_OK;
}

int hfa_plan_routing(const hfa_plan *p, int32_t out[8])
{
    if (!p || !out) return fail(HFA_ERR_ARG, "hfa_plan_routing: NULL argument");
    out[0] = p->warp_all_count;
    out[1] = p->band_count[0];
    out[2] = p->band_k[0];
    out[3] = p->band_count[1];
    out[4] = p->band_k[1];
    out[5] = p->class_count[HFA_NUM_CLASSES];
    out[6] = p->dp_store_elems > 0;
    out[7] = std::max(p->band_skew[0], p->band_skew[1]);
    return HFA_OK;
}

int32_t hfa_plan_pair_utterances(const hfa_plan *p) { return p ? p->pair_count : 0; }
int32_t hfa_plan_bt_walk_utterances(const hfa_plan *p) { return p ? p->n_walk : 0; }
int32_t hfa_plan_skew_ctas_per_sm(const hfa_plan *p, int32_t list)
{
    if (!p || list < 0 || list > 1) return 0;
    return (p->band_skew[list] > 0 && p->band_count[list] > 0) ? p->skew_ctas[list] : 0;
}
int64_t hfa_plan_stored_emission_bytes(const hfa_plan *p) { return p ? p->stored_emis * 4 : 0; }

int64_t hfa_plan_debug_region(const hfa_plan *p, int32_t which, int64_t *n_bytes)
{
    if (!p) return -1;
    int64_t off = -1, n = 0;
    switch (which) {
        case 0: off = p->o_emis; n = p->padded_cells * 4; break;
        case 1: off = p->o_edge2; n = p->total_edge * 8; break;
        case 2: off = p->o_edgep; n = p->total_edge * 4; break;
        case 3: off = p->o_bp; n = p->total_words * 4; break;
        case 4: off = p->o_band_xchg; n = p->band_xchg_elems * 16; break;
        default: break;
    }
    if (n_bytes) *n_bytes = n;
    return off;
}

int hfa_plan_upload(const hfa_plan *p, void *workspace, void *stream)
{
    if (!p || !workspace) return fail(HFA_ERR_ARG, "hfa_plan_upload: NULL argument");
    if (p->head_bytes == 0) return HFA_OK;
    cudaError_t e = cudaMemcpyAsync(workspace, p->head.data(), (size_t)p->head_bytes,
                                    cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return cuda_fail(e, "hfa_plan_upload");
    if (p->n_tmaps > 0 && p->use_tmaps) try {
        // TMA tensor maps over emis[t][s] of the banded utterances (they hold the workspace address, so
        // they are built here): rank 2, f32, dims {Sp, T}, row pitch Sp * 4 B, box {32 K, 16}
        std::vector<CUtensorMap> maps((size_t)p->n_tmaps);
        for (const HfaUtt &m : p->utt) {
            if (m.status != 0 || m.tmap < 0) continue;
            const cuuint64_t dims[2] = {(cuuint64_t)m.Sp, (cuuint64_t)m.T};
            const cuuint64_t pitch[1] = {(cuuint64_t)m.Sp * 4};
            const cuuint32_t box[2] = {(cuuint32_t)(m.skew_d > 0 ? HFA_SKEW_BOX : 32 * m.band_k),
                                       (cuuint32_t)(m.skew_d > 0 ? HFA_SKEW_BLK : HFA_TILE_T)};
            const cuuint32_t estr[2] = {1, 1};
            void *base = static_cast<unsigned char *>(workspace) + p->o_emis + m.emis_off * 4;
            const CUresult r = tensor_map_encoder()(&maps[(size_t)m.tmap], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base,
                                                    dims, pitch, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) return fail(HFA_ERR_CUDA, "hfa_plan_upload: cuTensorMapEncodeTiled failed (%d)", (int)r);
        }
        e = cudaMemcpyAsync(static_cast<unsigned char *>(workspace) + p->o_tmaps, maps.data(), maps.size() * 128,
                            cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream));
        if (e != cudaSuccess) return cuda_fail(e, "hfa_plan_upload: tensor maps");
    } catch (const std::bad_alloc &) {
        return fail(HFA_ERR_NOMEM, "hfa_plan_upload: out of host memory");
    }
    if (p->n_compact > 0) {        // no emissions yet: plain rows
        e = cudaMemsetAsync(static_cast<unsigned char *>(workspace) + p->o_emode, 0, (size_t)p->n_utt * 4,
                            static_cast<cudaStream_t>(stream));
        if (e != cudaSuccess) return cuda_fail(e, "hfa_plan_upload: emission mode reset");
    }
    if (p->band_bytes > 0) {       // band tickets + exchange slots start (and are left) all-zero
        e = cudaMemsetAsync(static_cast<unsigned char *>(workspace) + p->o_band_ticket, 0,
                            (size_t)p->band_bytes, static_cast<cudaStream_t>(stream));
        if (e != cudaSuccess) return cuda_fail(e, "hfa_plan_upload: band table reset");
    }
    return HFA_OK;
}

int hfa_set_inputs(const hfa_plan *p, void *workspace, const void *const *frame_ptrs,
                   const int64_t *frame_stride_t, const int64_t *frame_stride_v,
                   const void *const *edge_ptrs, const int64_t *edge_stride, void *stream)
{
    if (!p || !workspace) return fail(HFA_ERR_ARG, "hfa_set_inputs: NULL plan/workspace");
    if (p->n_utt == 0) return HFA_OK;
    if (!frame_ptrs || !frame_stride_t || !frame_stride_v || !edge_ptrs || !edge_stride)
        return fail(HFA_ERR_ARG, "hfa_set_inputs: NULL input table");
    try {
        std::vector<HfaInput> in((size_t)p->n_utt);
        int64_t row_stride = 0;
        bool contiguous = true;
        for (int32_t b = 0; b < p->n_utt; ++b) {
            if (p->utt[b].status == 0 && (!frame_ptrs[b] || !edge_ptrs[b]))
                return fail(HFA_ERR_ARG, "hfa_set_inputs: NULL logits pointer for utterance %d", b);
            if (p->utt[b].status == 0) {
                if (frame_stride_v[b] != 1 || frame_stride_t[b] < p->vocab ||
                    (reinterpret_cast<uintptr_t>(frame_ptrs[b]) & 3u))
                    contiguous = false;
                row_stride = std::max(row_stride, frame_stride_t[b]);
            }
            in[b].frame = frame_ptrs[b];
            in[b].edge = edge_ptrs[b];
            in[b].frame_st = frame_stride_t[b];
            in[b].frame_sv = frame_stride_v[b];
            in[b].edge_st = edge_stride[b];
        }
        HfaLaunchCtx c = make_ctx(p, workspace, stream);
        // pageable source: the runtime stages the table before returning, `in` may go out of scope
        cudaError_t e = cudaMemcpyAsync(c.ws.inputs, in.data(), in.size() * sizeof(HfaInput),
                                        cudaMemcpyHostToDevice, c.stream);
        if (e != cudaSuccess) return cuda_fail(e, "hfa_set_inputs: input table upload");
        p->set_row_stride(workspace, contiguous ? row_stride : 0);
    } catch (const std::bad_alloc &) {
        return fail(HFA_ERR_NOMEM, "hfa_set_inputs: out of host memory");
    }
    return HFA_OK;
}

static_assert(sizeof(HfaInputDesc) == sizeof(HfaInput), "the public descriptor is the kernels' own");

int hfa_set_inputs_device(const hfa_plan *p, void *workspace, const HfaInputDesc *table, int64_t max_row_stride,
                          void *stream)
{
    if (!p || !workspace) return fail(HFA_ERR_ARG, "hfa_set_inputs_device: NULL plan/workspace");
    if (p->n_utt == 0) return HFA_OK;
    if (!table) return fail(HFA_ERR_ARG, "hfa_set_inputs_device: NULL table");
    if (max_row_stride < 0) return fail(HFA_ERR_ARG, "hfa_set_inputs_device: negative row stride");
    HfaLaunchCtx c = make_ctx(p, workspace, stream);
    // device -> device: a plain copy node, so the whole step can be captured into a CUDA graph
    cudaError_t e = cudaMemcpyAsync(c.ws.inputs, table, (size_t)p->n_utt * sizeof(HfaInput),
                                    cudaMemcpyDeviceToDevice, c.stream);
    if (e != cudaSuccess) return cuda_fail(e, "hfa_set_inputs_device: table copy");
    try {
        p->set_row_stride(workspace, max_row_stride);
    } catch (const std::bad_alloc &) {
        return fail(HFA_ERR_NOMEM, "hfa_set_inputs_device: out of host memory");
    }
    return HFA_OK;
}

void hfa_release_thread_resources(void)
{
    for (HfaSideStreams *s : side_pool()) {
        for (int i = 0; i < HFA_NUM_CLASSES; ++i) {
            if (s->stream[i]) cudaStreamDestroy(s->stream[i]);
            if (s->join[i]) cudaEventDestroy(s->join[i]);
        }
        if (s->fork) cudaEventDestroy(s->fork);
        delete s;
    }
    side_pool().clear();
}

int hfa_emission(const hfa_plan *p, void *workspace, int32_t dtype, void *stream)
{
    if (!p || !workspace) return fail(HFA_ERR_ARG, "hfa_emission: NULL plan/workspace");
    if (p->n_utt == 0 || p->total_frames == 0) return HFA_OK;
    if (dtype < 0 || dtype > 2) return fail(HFA_ERR_ARG, "hfa_emission: bad dtype %d", dtype);
    HfaLaunchCtx c = make_ctx(p, workspace, stream);
    const int64_t row_stride = p->row_stride_of(workspace);
    // The persistent (TMA) emission kernel leaves the edge stream to its own small kernel, forked
    // onto a side stream so that the two overlap and joined before anything downstream.  The fork
    // point has to be recorded BEFORE the emission launch is queued.
    HfaSideStreams *ss = nullptr;
    cudaError_t e = cudaSuccess;
    if (row_stride > 0) {
        ss = side_streams();
        if (!ss) return fail(HFA_ERR_CUDA, "hfa_emission: cannot create side streams");
        e = cudaEventRecord(ss->fork, c.stream);
        if (e != cudaSuccess) return cuda_fail(e, "hfa_emission: fork");
    }
    int n_launched = 0;
    e = hfa_launch_emission(c, p->row_blocks[p->n_utt], p->max_sp, dtype, row_stride, &n_launched);
    if (e != cudaSuccess) return cuda_fail(e, "hfa_emission: launch");
    if (n_launched == 2) {
        HfaLaunchCtx cs = c;
        cs.stream = ss->stream[HFA_NUM_CLASSES - 1];
        e = cudaStreamWaitEvent(cs.stream, ss->fork, 0);
        if (e == cudaSuccess) e = hfa_launch_edge(cs, p->row_blocks[p->n_utt], dtype);
        if (e == cudaSuccess) e = cudaEventRecord(ss->join[HFA_NUM_CLASSES - 1], cs.stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(c.stream, ss->join[HFA_NUM_CLASSES - 1], 0);
        if (e != cudaSuccess) return cuda_fail(e, "hfa_emission: edge kernel");
    }
    g_launches += n_launched;
    return HFA_OK;
}

int hfa_pack_emissions(const hfa_plan *p, void *workspace, const float *prob_log,
                       const float *edge_log, const float *not_edge_log, const float *edge_pred,
                       void *stream)
{
    if (!p || !workspace) return fail(HFA_ERR_ARG, "hfa_pack_emissions: NULL plan/workspace");
    if (p->n_utt == 0 || p->total_frames == 0) return HFA_OK;
    if (!prob_log || !edge_log || !not_edge_log)
        return fail(HFA_ERR_ARG, "hfa_pack_emissions: NULL input");
    HfaLaunchCtx c = make_ctx(p, workspace, stream);
    cudaError_t e = hfa_launch_pack(c, p->row_blocks[p->n_utt], prob_log, edge_log, not_edge_log,
                                    edge_pred);
    if (e != cudaSuccess) return cuda_fail(e, "hfa_pack_emissions: launch");
    g_launches += 1;
    return HFA_OK;
}

// fused_row_stride > 0 (hfa_align_batch only): every utterance is in the banded kernel and the
// producer warps compute the emissions from the logits themselves
static int viterbi_forward_impl(const hfa_plan *p, void *workspace, float *dp_dump, void *stream,
                                int64_t fused_row_stride)
{
    if (!p || !workspace) return fail(HFA_ERR_ARG, "hfa_viterbi_forward: NULL plan/workspace");
    HfaLaunchCtx c = make_ctx(p, workspace, stream);
    const int n_cta = p->class_count[HFA_NUM_CLASSES];
    // launches of this call: the merged warp kernel (every state class in one launch), the strips / bands of the
    // two lists, the CTA-per-utterance kernel -- forked onto side streams when there is more than one
    struct Item { int k; const int32_t *order; int n; };
    Item items[4];
    int n_items = 0;
    if (p->warp_all_count > 0) items[n_items++] = {0, c.ws.order + p->warp_all_begin, p->warp_all_count};
    if (p->band_count[0] > 0) items[n_items++] = {-3, nullptr, 0};
    if (p->band_count[1] > 0) items[n_items++] = {-4, nullptr, 1};
    if (n_cta > 0) items[n_items++] = {-1, c.ws.order + p->class_begin[HFA_NUM_CLASSES], n_cta};
    if (n_items == 0) return HFA_OK;

    const bool fork = n_items > 1;
    HfaSideStreams *ss = nullptr;
    if (fork) {
        ss = side_streams();
        if (!ss) return fail(HFA_ERR_CUDA, "hfa_viterbi_forward: cannot create side streams");
        cudaError_t e = cudaEventRecord(ss->fork, c.stream);
        if (e != cudaSuccess) return cuda_fail(e, "hfa_viterbi_forward: fork record");
    }
    const cudaStream_t user = c.stream;
    for (int it = 0; it < n_items; ++it) {
        cudaError_t e;
        const bool side = fork && it > 0;
        c.stream = side ? ss->stream[it - 1] : user;
        if (side) {
            e = cudaStreamWaitEvent(c.stream, ss->fork, 0);
            if (e != cudaSuccess) return cuda_fail(e, "hfa_viterbi_forward: fork wait");
        }
        if (items[it].k == 0)
            e = hfa_launch_dp_warp_any(c, p->warp_max_k, p->warp_max_pair_k, items[it].order, items[it].n, dp_dump);
        else if (items[it].k == -3 || items[it].k == -4) {
            const int wh = items[it].k == -3 ? 0 : 1;
            if (p->band_skew[wh] > 0)
                e = hfa_launch_dp_skew(c, p->band_skew[wh], p->skew_ctas[wh], p->band_begin[wh], p->band_count[wh],
                                       c.ws.band_ticket + wh, p->dp_store_elems > 0, p->skew_slow, dp_dump);
            else
                e = hfa_launch_dp_band(c, p->band_k[wh], p->band_begin[wh], p->band_count[wh],
                                       c.ws.band_ticket + wh, p->dp_store_elems > 0, fused_row_stride, dp_dump);
        }
        else
            e = hfa_launch_dp_cta(c, items[it].order, items[it].n, p->cta_max_sp, dp_dump);
        if (e != cudaSuccess) return cuda_fail(e, "hfa_viterbi_forward: kernel launch");
        g_launches += 1;
        if (side) {
            e = cudaEventRecord(ss->join[it - 1], c.stream);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(user, ss->join[it - 1], 0);
            if (e != cudaSuccess) return cuda_fail(e, "hfa_viterbi_forward: join");
        }
    }
    return HFA_OK;
}

int hfa_viterbi_forward(const hfa_plan *p, void *workspace, float *dp_dump, void *stream)
{
    return viterbi_forward_impl(p, workspace, dp_dump, stream, 0);
}

int hfa_backtrace(const hfa_plan *p, void *workspace, void *result, float *frame_conf,
                  float *dp_path, void *stream)
{
    if (!p || !workspace || !result) return fail(HFA_ERR_ARG, "hfa_backtrace: NULL argument");
    if (p->n_utt == 0) return HFA_OK;
    HfaLaunchCtx c = make_ctx(p, workspace, stream);
    const HfaResultPtrs r = make_res(p, result);
    // utterances whose forward pass kept dp (latency plans): one CTA per utterance, the walk set straight from
    // its staged backpointers, the table set after the jump tables; the warp-per-utterance kernel below skips
    // them (and they skip the others)
    if (p->n_walk > 0) {
        cudaError_t ew = hfa_launch_backtrace_walk(c, c.ws.order + p->walk_begin, p->n_walk, p->walk_smem, r,
                                                   frame_conf, dp_path);
        if (ew != cudaSuccess) return cuda_fail(ew, "hfa_backtrace: walk kernel");
        g_launches += 1;
    }
    if (p->n_tab > 0) {
        cudaError_t ej = hfa_launch_jump_tables(c, (int)p->jblk_utt.size());
        if (ej == cudaSuccess)
            ej = hfa_launch_backtrace_tables(c, c.ws.order + p->tab_begin, p->n_tab, r, frame_conf, dp_path);
        if (ej != cudaSuccess) return cuda_fail(ej, "hfa_backtrace: table kernels");
        g_launches += 2;
    }
    if (p->n_kept > 0 && p->n_kept == p->n_utt) return HFA_OK;   // nothing left for the warp kernel
    cudaError_t e = hfa_launch_backtrace(c, c.ws.order + p->bt_begin, p->n_utt, r, frame_conf,
                                         dp_path);
    if (e != cudaSuccess) return cuda_fail(e, "hfa_backtrace: launch");
    g_launches += 1;
    return HFA_OK;
}

static bool fused_ok(const hfa_plan *p, const void *workspace, int32_t dtype)
{
    const int64_t max_row_stride = p->row_stride_of(workspace);
    const bool all_banded = p->warp_all_count == 0 &&
                            p->class_count[HFA_NUM_CLASSES] == 0 && !p->band_items.empty();
    const bool skewed = p->band_skew[0] > 0 || p->band_skew[1] > 0;   // no producer warp there to fuse into
    // max_sp: the fused band kernel is not shown to handle utterances beyond the CTA kernel's range
    return all_banded && !skewed && p->max_sp <= HFA_CTA_MAX_S && p->dp_store_elems > 0 && dtype == HFA_DTYPE_F32 &&
           max_row_stride > 0 &&
           p->vocab <= 256 && max_row_stride * 4 * HFA_TILE_T <= 48 * 1024;
}

int hfa_forward_fused(const hfa_plan *p, void *workspace, int32_t dtype, void *stream)
{
    if (!p || !workspace) return fail(HFA_ERR_ARG, "hfa_forward_fused: NULL plan/workspace");
    if (!fused_ok(p, workspace, dtype))
        return fail(HFA_ERR_UNSUPPORTED, "hfa_forward_fused: needs an all-banded plan that keeps dp, f32 logits "
                                         "with contiguous rows (set by hfa_set_inputs) and V <= 256");
    HfaLaunchCtx c = make_ctx(p, workspace, stream);
    cudaError_t e = hfa_launch_edge(c, p->row_blocks[p->n_utt], dtype);
    if (e != cudaSuccess) return cuda_fail(e, "hfa_forward_fused: edge kernel");
    g_launches += 1;
    return viterbi_forward_impl(p, workspace, nullptr, stream, p->row_stride_of(workspace));
}

int64_t hfa_plan_algorithmic_bytes_fused(const hfa_plan *p, int32_t dtype)
{
    if (!p) return 0;
    const int64_t in_b = (dtype == HFA_DTYPE_F32) ? 4 : 2;
    int64_t words = 0;
    for (const HfaUtt &m : p->utt)
        if (m.status == 0) words += (int64_t)((m.T + 15) / 16) * m.S;
    return p->total_frames * ((int64_t)p->vocab * in_b + in_b) + p->total_frames * 12 + words * 4 +
           p->total_cells * 4;
}

int hfa_align_batch(const hfa_plan *p, void *workspace, int32_t dtype, void *result,
                    float *frame_conf, void *stream)
{
    if (!p || !workspace) return fail(HFA_ERR_ARG, "hfa_align_batch: NULL plan/workspace");
    // Fused route (small batches): when every utterance is in the banded kernel, keeps its dp, and
    // the logits are f32 rows the TMA engine can fetch, the emission stage disappears -- only the
    // edge stream is computed up front, the emissions are produced inside the DP kernel's producer
    // warps and never written to HBM.
    // Measured (B200): the fused route wins when no utterance is split into several bands (config 1:
    // 0.137 vs 0.173 ms per decode) and loses otherwise -- every band of an utterance recomputes the
    // softmax normaliser of its frames, and a single producer warp then cannot keep up with its
    // compute warp (config 2: 0.29 vs 0.22 ms).
    int64_t n_valid = 0;
    for (const HfaUtt &m : p->utt) n_valid += (m.status == 0);
    const bool unsplit = (int64_t)p->band_items.size() == n_valid;
    int rc;
    if (unsplit && fused_ok(p, workspace, dtype)) {
        rc = hfa_forward_fused(p, workspace, dtype, stream);
    } else {
        rc = hfa_emission(p, workspace, dtype, stream);
        if (rc != HFA_OK) return rc;
        rc = viterbi_forward_impl(p, workspace, nullptr, stream, 0);
    }
    if (rc != HFA_OK) return rc;
    return hfa_backtrace(p, workspace, result, frame_conf, nullptr, stream);
}

int hfa_ctc_greedy(const void *logits, int32_t dtype, int64_t T, int64_t V, int64_t stride_t,
                   int64_t stride_v, int32_t *scratch, int32_t *out_ids, int32_t *out_len, void *stream)
{
    if (!logits || !scratch || !out_ids || !out_len) return fail(HFA_ERR_ARG, "hfa_ctc_greedy: NULL argument");
    if (T < 0 || V < 1 || T > INT32_MAX || V > INT32_MAX || dtype < 0 || dtype > 2)
        return fail(HFA_ERR_ARG, "hfa_ctc_greedy: bad shape / dtype (T=%lld, V=%lld)", (long long)T, (long long)V);
    cudaError_t e = hfa_launch_ctc_greedy(logits, dtype, (int)T, (int)V, stride_t, stride_v, scratch, out_ids,
                                          out_len, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return cuda_fail(e, "hfa_ctc_greedy: launch");
    g_launches += 1;
    return HFA_OK;
}

int hfa_ctc_greedy_batch(const hfa_plan *p, void *workspace, const HfaCtcDesc *table, int64_t V, int32_t dtype,
                         int32_t *scratch, int32_t *out_ids, int32_t *out_len, void *stream)
{
    if (!p || !workspace) return fail(HFA_ERR_ARG, "hfa_ctc_greedy_batch: NULL plan/workspace");
    if (V < 1 || V > INT32_MAX || dtype < 0 || dtype > 2)
        return fail(HFA_ERR_ARG, "hfa_ctc_greedy_batch: bad width / dtype (V=%lld, dtype=%d)", (long long)V, dtype);
    if (p->n_utt == 0) return HFA_OK;
    if (!table || !scratch || !out_ids || !out_len) return fail(HFA_ERR_ARG, "hfa_ctc_greedy_batch: NULL argument");
    HfaLaunchCtx c = make_ctx(p, workspace, stream);
    // out_len is the kernel's per-utterance count of finished frames before it holds the lengths
    cudaError_t e = cudaMemsetAsync(out_len, 0, (size_t)p->n_utt * sizeof(int32_t), c.stream);
    if (e != cudaSuccess) return cuda_fail(e, "hfa_ctc_greedy_batch: out_len reset");
    if (p->total_frames == 0) return HFA_OK;
    e = hfa_launch_ctc_batch(c, p->row_blocks[p->n_utt], table, (int)V, dtype, scratch, out_ids, out_len);
    if (e != cudaSuccess) return cuda_fail(e, "hfa_ctc_greedy_batch: launch");
    g_launches += 1;
    return HFA_OK;
}

int hfa_frame_states(const hfa_plan *p, void *workspace, const void *result, int32_t *out, void *stream)
{
    if (!p || !workspace) return fail(HFA_ERR_ARG, "hfa_frame_states: NULL plan/workspace");
    if (p->n_utt == 0 || p->total_frames == 0) return HFA_OK;
    if (!result || !out) return fail(HFA_ERR_ARG, "hfa_frame_states: NULL argument");
    HfaLaunchCtx c = make_ctx(p, workspace, stream);
    cudaError_t e = hfa_launch_frame_states(c, p->row_blocks[p->n_utt],
                                            make_res(p, const_cast<void *>(result)), out);
    if (e != cudaSuccess) return cuda_fail(e, "hfa_frame_states: launch");
    g_launches += 1;
    return HFA_OK;
}

int hfa_debug_unpack_backptr(const hfa_plan *p, const void *workspace, int32_t utt, int8_t *out,
                             void *stream)
{
    if (!p || !workspace || !out) return fail(HFA_ERR_ARG, "hfa_debug_unpack_backptr: NULL argument");
    if (utt < 0 || utt >= p->n_utt || p->utt[utt].status != 0)
        return fail(HFA_ERR_ARG, "hfa_debug_unpack_backptr: bad utterance %d", utt);
    HfaLaunchCtx c = make_ctx(p, const_cast<void *>(workspace), stream);
    cudaError_t e = hfa_launch_unpack_bp(c, utt, out);
    if (e != cudaSuccess) return cuda_fail(e, "hfa_debug_unpack_backptr: launch");
    g_launches += 1;
    return HFA_OK;
}

int hfa_debug_unpack_dp(const hfa_plan *p, const void *workspace, int32_t utt, float *out, void *stream)
{
    if (!p || !workspace || !out) return fail(HFA_ERR_ARG, "hfa_debug_unpack_dp: NULL argument");
    if (utt < 0 || utt >= p->n_utt || p->utt[utt].status != 0)
        return fail(HFA_ERR_ARG, "hfa_debug_unpack_dp: bad utterance %d", utt);
    if (p->utt[utt].dp_off < 0)
        return fail(HFA_ERR_UNSUPPORTED, "hfa_debug_unpack_dp: the forward pass keeps no dp for utterance %d", utt);
    HfaLaunchCtx c = make_ctx(p, const_cast<void *>(workspace), stream);
    cudaError_t e = hfa_launch_unpack_dp(c, utt, out);
    if (e != cudaSuccess) return cuda_fail(e, "hfa_debug_unpack_dp: launch");
    g_launches += 1;
    return HFA_OK;
}

int hfa_debug_unpack_emissions(const hfa_plan *p, const void *workspace, float *out, void *stream)
{
    if (!p || !workspace || !out) return fail(HFA_ERR_ARG, "hfa_debug_unpack_emissions: NULL argument");
    HfaLaunchCtx c = make_ctx(p, const_cast<void *>(workspace), stream);
    cudaError_t e = hfa_launch_unpack_emissions(c, p->n_utt > 0 ? p->row_blocks[p->n_utt] : 0, out);
    if (e != cudaSuccess) return cuda_fail(e, "hfa_debug_unpack_emissions: launch");
    g_launches += 1;
    return HFA_OK;
}

}  // extern "C"
