// hfa_dp_skew.cu -- the recurrence as a time-skewed wavefront: the latency-regime forward kernel.
//
// Reference semantics: tools/alignment_decoder.py:170-230 (forward_pass) and :245-257 (init); the
// arithmetic contract is the one spelled out at the top of hfa_dp.cu.
//
// Why a skew.  dp[t][i] depends on dp[t-1][i] through two f32 adds and a max ("stay", ~14 cycles of
// latency) and on dp[t-1][i-1], dp[t-1][i-2] through  FADD FADD F2F DADD F2F  + a lane exchange
// ("advance", ~80 cycles).  A kernel that walks all states of an utterance through frame t before
// frame t+1 pays the long chain on every frame: T x 85 cycles at best (the banded kernel: 154).  But a
// best path advances at most S times in T frames, so the critical path of the whole DAG is only
// ~ 80 S + 14 (T - S) cycles.  Here lane p (state c0 + p) works on frame  t = n - p D  at iteration n: its
// left neighbours finished that frame D and 2 D iterations EARLIER, so their advance scores are old
// values that arrive by warp shuffle long before they are needed, and the loop-carried chain of an
// iteration is just   dp -> FADD -> FADD -> FMNMX -> FMNMX.   The conversions, the f64 add and the
// shuffles are pipelined work, off the chain.  Cost: T + 31 D iterations per strip instead of T.
//
// Mapping.  One CTA per STRIP of 32 columns: a compute warp with one state per lane and a producer warp.
// The compute warp only runs the recurrence: wait for the block's stage (READY), run the block, arrive
// on DONE.  The producer does everything else off that serial chain -- TMA ring, exchange wait, ghost
// columns, publication, kept-dp bulk store -- and runs ahead of it.  Strip 0 owns states 0..31.
// Strip w > 0 starts at column 30 w: lanes 0 and 1 are GHOSTS of the left strip's last two
// states -- they inject the advance scores the left strip published -- and lanes 2..31 own 30 states.
// A strip publishes {adv[31](t), adv[30](t)} for every frame into a per-frame slot in HBM/L2: lanes 31 and
// 30 park them in shared memory each iteration, and once per block the producer writes two tagged 64-bit
// words {f32 bits | tag << 32}, tag = t + 1, per frame (hfa_st_xchg_word: single-copy atomic, so a word
// is valid iff its tag matches -- no flag, no fence); the reader zeroes the slot after use and the table
// is all-zero between calls.  The right strip fetches BLK frames of slots per block and simply runs that
// far behind.  Work items are claimed through an atomic ticket in (utterance, strip) order, so a strip's
// left neighbour has always started; strip 0 never waits.
//
// All shared-memory traffic uses 32-bit shared-window addresses derived from ONE base computed at kernel
// start (forming generic pointers costs an S2UR + ULEA per use on sm_100).
//
// Emissions: ONE TMA tensor-tile copy (cp.async.bulk.tensor.2d, 32 frames x 36 columns: the box must
// start at a 16-byte boundary, 30 w rounded down to a multiple of 4, so it is 4 columns wider than the
// strip) per block of BLK = 32 iterations into a ring of NSTG = 5 or 6 stages (the 32 lanes of a strip span
// 31 D frames = 2-3 tiles; the stage count sets how many CTAs share an SM), plus a bulk copy of the block's
// 256 bytes of edge pairs; stage 0 is copied twice, the second time behind the last stage, so a lane's 32
// rows of a block are always contiguous and every shared-memory load of the unrolled block is
// [per-lane base + constant].  Kept dp (for the table backtrace): each iteration's 32 values form one
// 128-byte row of a staging tile that leaves as one 4 KB bulk store per block (hfa_skew_dp_index) -- no halo columns, nothing stored twice.
//
// Three block bodies: the unrolled steady-state one (all 32 lanes inside frames 1 .. T-1 for all 32
// iterations), the same with a per-lane `live` predicate for the ramps at both ends (and for every block
// of a dp-dump run), and a rolled one for the single block that seeds frame 0.
#include <cstdlib>

#include "hfa_common.cuh"

namespace {

// One frame of one state with curr carried as P = f64(curr) * ratio (alignment_decoder.py:210-228).
// Value: max of the three candidates (up2 is already capped where a two-state jump is not allowed).
// Backpointer: strict '>' scanned in the order stay, +1, +2 (ties keep the earlier candidate); mr has the
// frame's bit set in both halves.  curr: moved ? e : max(curr, e), 0 for id-0 states (sp_hi == 0: a zero
// high word makes P a subnormal that adds to any f64(f32) exactly like +0.0).
__device__ __forceinline__ void sk_select(float up1, float stay, float up2, double pe, uint32_t sp_hi, uint32_t mr,
                                          float &dp, double &P, uint32_t &acc)
{
    asm("{\n\t"
        ".reg .pred q1, q2, q3;\n\t"
        ".reg .f32 m;\n\t"
        ".reg .f64 pn;\n\t"
        ".reg .b32 lo, hi;\n\t"
        "setp.gt.f32 q1, %3, %4;\n\t"
        "max.f32 m, %4, %3;\n\t"
        "setp.gt.f32 q2, %5, m;\n\t"
        "max.f32 %0, m, %5;\n\t"
        "@q1 lop3.b32 %2, %2, %8, 0x0000ffff, 0xf8;\n\t"
        "@q2 lop3.b32 %2, %2, %8, 0xffff0000, 0xf8;\n\t"
        "or.pred q3, q1, q2;\n\t"
        "setp.gt.or.f64 q3, %6, %1, q3;\n\t"
        "selp.f64 pn, %6, %1, q3;\n\t"
        "mov.b64 {lo, hi}, pn;\n\t"
        "and.b32 hi, hi, %7;\n\t"
        "mov.b64 %1, {lo, hi};\n\t"
        "}"
        : "=&f"(dp), "+d"(P), "+r"(acc)
        : "f"(up1), "f"(stay), "f"(up2), "d"(pe), "r"(sp_hi), "r"(mr));
}
// The same frame for a lane that may be outside its utterance's frames 1 .. T-1 (`live` false): nothing
// changes then -- dp, P and the backpointer bits keep their values.
__device__ __forceinline__ void sk_select_guarded(float up1, float stay, float up2, double pe, uint32_t sp_hi,
                                                  uint32_t mr, int live, float &dp, double &P, uint32_t &acc)
{
    asm("{\n\t"
        ".reg .pred pl, q1, q2, q3;\n\t"
        ".reg .f32 m, dn;\n\t"
        ".reg .f64 pn;\n\t"
        ".reg .b32 lo, hi, msk;\n\t"
        "setp.ne.b32 pl, %9, 0;\n\t"
        "setp.gt.and.f32 q1, %3, %4, pl;\n\t"
        "max.f32 m, %4, %3;\n\t"
        "setp.gt.and.f32 q2, %5, m, pl;\n\t"
        "max.f32 dn, m, %5;\n\t"
        "selp.f32 %0, dn, %0, pl;\n\t"
        "@q1 lop3.b32 %2, %2, %8, 0x0000ffff, 0xf8;\n\t"
        "@q2 lop3.b32 %2, %2, %8, 0xffff0000, 0xf8;\n\t"
        "or.pred q3, q1, q2;\n\t"
        "setp.gt.or.f64 q3, %6, %1, q3;\n\t"
        "and.pred q3, q3, pl;\n\t"
        "selp.f64 pn, %6, %1, q3;\n\t"
        "mov.b64 {lo, hi}, pn;\n\t"
        "selp.b32 msk, %7, 0xffffffff, pl;\n\t"
        "and.b32 hi, hi, msk;\n\t"
        "mov.b64 %1, {lo, hi};\n\t"
        "}"
        : "+f"(dp), "+d"(P), "+r"(acc)
        : "f"(up1), "f"(stay), "f"(up2), "d"(pe), "r"(sp_hi), "r"(mr), "r"(live));
}

constexpr int SK_BOXW = HFA_SKEW_BOX;                // columns of an emission tile in shared memory
constexpr int BLK = HFA_SKEW_BLK;                    // iterations (= frames per lane) per block: one TMA tile,
                                                     // one exchange batch, one dp staging tile, BLK / 16 backpointer words
constexpr uint32_t SK_ROW_B = SK_BOXW * 4u;          // 144-byte rows
constexpr uint32_t SK_STG_B = BLK * SK_ROW_B;        // bytes per stage (a multiple of 128)
constexpr uint32_t SK_EDGE_B = BLK * 8u;             // edge pairs of a stage
constexpr uint32_t SK_DPST_B = BLK * 128u;           // one dp staging tile
constexpr uint32_t SK_PUB_B = (2 * BLK + BLK + 32) * 4u;   // adv31 [BLK], adv30 [BLK], scratch [BLK + 32]
constexpr int SK_LOOK = 3;                           // operands are loaded this many iterations ahead
constexpr int SK_NBUF = 3;                           // dp and publication staging buffers: block j reuses block j - 3's

// shared-memory map (byte offsets from the 128-byte aligned base)
template <int NSTG> struct SkSmem {
    static constexpr uint32_t TILE = 0;                                   // [(NSTG + 1) x BLK][36] f32 (+1: mirror of stage 0)
    static constexpr uint32_t EDGE = TILE + (NSTG + 1) * SK_STG_B;        // [(NSTG + 1) x BLK] float2
    static constexpr uint32_t DPST = EDGE + (NSTG + 1) * SK_EDGE_B;       // SK_NBUF x [BLK][32] f32: kept-dp staging
    static constexpr uint32_t PUB = DPST + SK_NBUF * SK_DPST_B;           // SK_NBUF x publication staging
    static constexpr uint32_t FULL = PUB + SK_NBUF * SK_PUB_B;            // NSTG mbarriers: the tile has landed
    static constexpr uint32_t READY = FULL + NSTG * 8;                    // NSTG: ... and its ghost columns are in
    static constexpr uint32_t DONE = READY + NSTG * 8;                    // NSTG: the compute warp is done with a block
    static constexpr uint32_t SLOT = DONE + NSTG * 8;                     // work-item ticket, role swap
    static constexpr uint32_t BYTES = SLOT + 16;
};

template <int D, int NSTG, bool KEEP, bool DUMP>
__global__ void __launch_bounds__(64)
hfa_dp_skew_kernel(HfaWs ws, int item_begin, int32_t *ticket, float *__restrict__ dp_dump, int force_slow)
{
    using SM = SkSmem<NSTG>;
    constexpr int R = NSTG * BLK;                   // ring rows
    constexpr int Q = (31 * D + BLK - 1) / BLK;     // tiles behind the newest one that lanes still read
    constexpr int PF = NSTG - 1 - Q;                // tiles fetched ahead of the newest one in use
    static_assert(D >= 2, "advance scores must be at least two iterations old when they are consumed");
    static_assert(PF >= 1, "ring too small for this skew");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint32_t sm0;
    {   // computed ONCE: the volatile move keeps the compiler from re-deriving it (S2UR + ULEA) at every use
        const uint32_t a = hfa_smem_u32(smem_raw);
        asm volatile("mov.u32 %0, %1;" : "=r"(sm0) : "r"(a));
    }

    // Which of the two warps computes?  As in hfa_dp_band_kernel: the warps of a 2-warp CTA land on an
    // aligned pair of warp slots (slot % 4 = scheduler partition), so "warp 0 computes" would put every
    // compute warp of the SM on partitions 0 and 2; swapping the roles in every other pair spreads them.
    if (threadIdx.x == 0) {
        unsigned hw_slot;
        asm volatile("mov.u32 %0, %%warpid;" : "=r"(hw_slot));
        hfa_sts_s32(sm0 + SM::SLOT + 4u, (int)((hw_slot >> 2) & 1u));
        hfa_sts_s32(sm0 + SM::SLOT,
                    (int)atomicInc(reinterpret_cast<unsigned int *>(ticket), gridDim.x - 1));   // self-resetting
#pragma unroll
        for (int s = 0; s < NSTG; ++s) {
            hfa_mbar_init(sm0 + SM::FULL + 8u * s, 1);      // the copy issuer (+ the TMA bytes)
            hfa_mbar_init(sm0 + SM::READY + 8u * s, 32);    // every producer lane, after the ghost columns
            hfa_mbar_init(sm0 + SM::DONE + 8u * s, 32);     // every compute lane, after the block
        }
        hfa_fence_mbar_init();
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    // (broadcast from lane 0 so that the compiler knows the role is warp-uniform: without it, the compute
    // warp's shuffles are compiled for a possibly diverged warp)
    const bool producer =
        __shfl_sync(0xffffffffu, (threadIdx.x >> 5) ^ (unsigned)hfa_lds_s32(sm0 + SM::SLOT + 4u), 0) != 0;
    const int item = item_begin + hfa_lds_s32(sm0 + SM::SLOT);
    const HfaBandItem bi = ws.band_items[item];
    const int u = bi.utt, w = bi.band;
    const HfaUtt m = ws.utt[u];
    const int T = m.T, S = m.S, Sp = m.Sp;
    const bool has_left = w > 0, has_right = w + 1 < hfa_skew_strips(Sp);
    const int c0 = HFA_SKEW_OWN * w;
    const int NB = hfa_skew_blocks(D, T);

    if (producer) {
        // ---------------- producer: TMA ring, left exchange -> ghost columns, publication, dp store ----------------
        // Block a is PREPARED (tile landed, the left strip's advance scores stored over the ghost columns:
        // READY) and block b RETIRED (after DONE: its advance scores published, its dp rows stored, the
        // stage it read last refilled).  Retiring comes first -- the right strip waits for it -- and
        // neither step blocks the other: the loop polls both.  Preparing runs ahead as far as the left
        // strip, the ring (tile a is fetched when block a - PF - 1 retires) and the staging buffers (block
        // a writes the ones block a - SK_NBUF wrote: a <= b + SK_NBUF - 1) allow.
        const float2 *g_edge = ws.edge2 + m.edge_off;
        const unsigned char *tmap = static_cast<const unsigned char *>(ws.tmaps) + (size_t)m.tmap * 128;
        float *g_dp = (KEEP && m.dp_off >= 0) ? ws.dp_store + m.dp_off + (int64_t)w * NB * (BLK * 32) : nullptr;
        // tile i -> stage st (= i % NSTG, kept as a running counter); executed by ONE elected lane.  The edge
        // pairs of an utterance are padded to a multiple of 16 frames: the last copy of a 32-frame block may be short.
        const int edge_len = (T + 15) & ~15;
        auto issue = [&](int i, int st) {
            const int t0 = i * BLK;
            const uint32_t bar = sm0 + SM::FULL + 8u * (uint32_t)st;
            if (t0 >= T) {                                     // nothing to fetch: complete the phase
                hfa_mbar_arrive(bar);
                return;
            }
            const uint32_t ebytes = (uint32_t)min(BLK, edge_len - t0) * 8u;
            const uint32_t bytes = SK_STG_B + ebytes;
            hfa_mbar_expect_tx(bar, st == 0 ? 2u * bytes : bytes);
            hfa_tensor_load_2d(sm0 + SM::TILE + (uint32_t)st * SK_STG_B, tmap, c0 & ~3, t0, bar);
            hfa_bulk_load(sm0 + SM::EDGE + (uint32_t)st * SK_EDGE_B, g_edge + t0, ebytes, bar);
            if (st == 0) {                                     // the mirror behind the last stage
                hfa_tensor_load_2d(sm0 + SM::TILE + (uint32_t)NSTG * SK_STG_B, tmap, c0 & ~3, t0, bar);
                hfa_bulk_load(sm0 + SM::EDGE + (uint32_t)NSTG * SK_EDGE_B, g_edge + t0, ebytes, bar);
            }
        };
        static_assert(PF + 1 <= NSTG, "prologue fills distinct stages");
        if (hfa_elect_one())
            for (int i = 0; i <= PF && i < NB; ++i) issue(i, i);   // tiles 0 .. PF (tile b + PF + 1 follows block b)

        const ulonglong2 *left_x = reinterpret_cast<const ulonglong2 *>(ws.band_xchg) +
                                   (has_left ? ws.band_items[item - 1].xoff : 0);
        ulonglong2 *my_x = reinterpret_cast<ulonglong2 *>(ws.band_xchg) + bi.xoff;
        auto slot_needed = [&](int jj) { const int t = BLK * jj + lane; return has_left && lane < BLK && t >= 1 && t < T; };
        // exchange slots of the block being prepared, fetched one block early (the left strip is normally
        // that far ahead)
        ulonglong2 xv = make_ulonglong2(0ull, 0ull);
        if (slot_needed(0)) xv = hfa_ld_xchg(left_x + lane);

        int a = 0, st_a = 0, buf_b = 0;
        uint32_t par_a = 0;
        int b = 0, st_b = 0;
        uint32_t par_b = 0;
        int st_issue = (PF + 1) % NSTG;                        // stage of the next tile to fetch
        uint32_t spins = 0;
        while (b < NB) {
            if (b < a && __all_sync(0xffffffffu, hfa_mbar_test_wait(sm0 + SM::DONE + 8u * (uint32_t)st_b, par_b))) {
                if (has_right) {
                    // the advance scores lanes 31 and 30 have parked: published as tagged 64-bit words, adv31 of
                    // frame BLK b + i - 31 D into .x, adv30 of frame BLK b + i - 30 D into .y (frames 1 .. T-1 only)
#pragma unroll
                    for (int q = lane; q < 2 * BLK; q += 32) {
                        const int half = q / BLK, i = q % BLK;
                        const int t = BLK * b + i - (31 - half) * D;
                        if (t >= 1 && t < T) {
                            const float v = hfa_lds_f32(sm0 + SM::PUB + (uint32_t)buf_b * SK_PUB_B + 4u * (uint32_t)q);
                            hfa_st_xchg_word(reinterpret_cast<unsigned long long *>(my_x + t) + half,
                                             hfa_tagged(__float_as_uint(v), (uint32_t)t + 1u));
                        }
                    }
                }
                if (hfa_elect_one()) {
                    if (KEEP && g_dp != nullptr) {             // the block's rows of dp leave as one bulk store
                        hfa_bulk_store(g_dp + (int64_t)b * (BLK * 32), sm0 + SM::DPST + (uint32_t)buf_b * SK_DPST_B,
                                      SK_DPST_B);
                        hfa_bulk_commit();
                    }
                    if (b + PF + 1 < NB) issue(b + PF + 1, st_issue);   // into the stage block b read last
                }
                if (++st_issue == NSTG) st_issue = 0;
                if (++st_b == NSTG) {
                    st_b = 0;
                    par_b ^= 1u;
                }
                if (++buf_b == SK_NBUF) buf_b = 0;
                ++b;
                spins = 0;
                continue;
            }
            if (a < NB && a <= b + SK_NBUF - 1 &&
                __all_sync(0xffffffffu, hfa_mbar_test_wait(sm0 + SM::FULL + 8u * (uint32_t)st_a, par_a))) {
                bool go = true;
                if (has_left) {
                    // The left strip's advance scores for frames BLK a .. BLK a + BLK - 1 go where the ghost lanes
                    // look for their "emission": ghost lane 0 (the left strip's state 30) reads column c0 of row t
                    // of the tile, ghost lane 1 (state 31) column c0 + 1 -- the emissions TMA put there are of no
                    // use to anybody.
                    const int t = BLK * a + lane;
                    const bool need = slot_needed(a);
                    ulonglong2 *src = const_cast<ulonglong2 *>(left_x) + t;
                    const uint32_t tag = (uint32_t)t + 1u;
                    const bool ok = !need || ((uint32_t)(xv.x >> 32) == tag && (uint32_t)(xv.y >> 32) == tag);
                    go = __all_sync(0xffffffffu, ok);
                    if (!go) {
                        if (!ok) xv = hfa_ld_xchg(src);
                    } else {
                        const ulonglong2 v = xv;
                        xv = slot_needed(a + 1) ? hfa_ld_xchg(src + BLK) : make_ulonglong2(0ull, 0ull);
                        if (lane < BLK) {
                            const float a30 = need ? __uint_as_float((uint32_t)v.y) : 0.0f;
                            const float a31 = need ? __uint_as_float((uint32_t)v.x) : 0.0f;
                            const uint32_t row_sa = sm0 + SM::TILE + (uint32_t)st_a * SK_STG_B + (uint32_t)lane * SK_ROW_B +
                                                    4u * (uint32_t)(c0 & 3);
                            hfa_sts_f32(row_sa, a30);
                            hfa_sts_f32(row_sa + 4u, a31);
                            if (st_a == 0) {                                       // and its mirror
                                hfa_sts_f32(row_sa + (uint32_t)NSTG * SK_STG_B, a30);
                                hfa_sts_f32(row_sa + (uint32_t)NSTG * SK_STG_B + 4u, a31);
                            }
                            if (need) hfa_st_xchg(src, 0ull, 0ull);                 // leave the table clean
                        }
                        hfa_fence_async_smem();   // generic writes into a stage the TMA engine will refill later
                    }
                }
                if (go) {
                    // block a overwrites the dp staging of block a - SK_NBUF: that bulk store must have been read
                    // out (stores 0 .. b - 1 are in flight; a - SK_NBUF <= b - 2 unless a = b + SK_NBUF - 1)
                    if (KEEP && a >= SK_NBUF && hfa_elect_one()) {
                        if (a == b + SK_NBUF - 1) hfa_bulk_wait_read<0>();
                        else hfa_bulk_wait_read<1>();
                    }
                    hfa_mbar_arrive(sm0 + SM::READY + 8u * (uint32_t)st_a);
                    if (++st_a == NSTG) {
                        st_a = 0;
                        par_a ^= 1u;
                    }
                    ++a;
                    spins = 0;
                    continue;
                }
            }
            // neither step can go: the compute warp is inside its block, or the left strip is behind
            if (++spins > HFA_POLLS_EXCHANGE) __trap();
        }
        if (KEEP && hfa_elect_one()) hfa_bulk_wait_all();
        return;
    }

    // ---------------- compute warp: the recurrence, nothing else ----------------
    const int s = c0 + lane;                                   // this lane's state
    const bool ghost = has_left && lane < 2;
    const bool real = !ghost && s < Sp;                        // owns a column of the padded matrices
    const int n_rows = (T + 15) >> 4;
    uint32_t *g_bp = ws.bp + m.bp_off;
    const double ratio = __ddiv_rn((double)T, (double)S);      // T / S (:186)
    const float NEG = HFA_NEG_INF, POS = __uint_as_float(0x7f800000u);

    // per-state constants (:194, :227, :250-254)
    const int32_t *ids = ws.ids + m.seg_off;
    uint32_t sp_hi = 0xffffffffu;                              // 0 for id-0 (SP) states: curr is zeroed
    float jcap = NEG;                                          // +inf where a two-state jump may enter
    if (s < S) {
        if (ids[s] == 0) sp_hi = 0u;
        if (s >= 2 && ids[s - 1] == 0) jcap = POS;
    }
    const bool lead_sp = (ids[0] == 0) && (S > 1);
    const bool seeded = !ghost && (s == 0 || (s == 1 && lead_sp));
    const float cap1 = (s == 0) ? NEG : POS;                   // nothing to the left of state 0

    int st_wait = 0;                                           // stage and phase parity of the current block's tile
    uint32_t par_wait = 0;
    int buf = 0;                                               // staging buffer of the current block (j % SK_NBUF)

    // loop-carried state
    float dp = NEG;
    double P = __longlong_as_double(0xfff0000000000000ll);     // f64(curr) * ratio, curr = -inf
    uint32_t bits = 0;                                         // first part of the backpointer row in progress
    float q1[D], q2[2 * D];                                    // advance scores in flight: q1[0] / q2[0] are due now
#pragma unroll
    for (int i = 0; i < D; ++i) q1[i] = NEG;
#pragma unroll
    for (int i = 0; i < 2 * D; ++i) q2[i] = NEG;

    // per-lane ring position of the first row of the current block: (BLK j - lane D) mod R
    int u_row = ((-lane * D) % R + R) % R;
    // (a ghost lane's "emission" is the left strip's advance score: the producer writes it over its column)
    const uint32_t tile_sa = sm0 + SM::TILE + 4u * (uint32_t)(lane + (c0 & 3));
    const uint32_t edge_sa = sm0 + SM::EDGE;
    const uint32_t dpst_sa = sm0 + SM::DPST + 4u * (uint32_t)lane;
    // backpointer bookkeeping: the 16 frames of a half-block straddle two 16-frame rows
    const int o_res = (lane * D) & 15;
    const int q_rows = (lane * D + 15) >> 4;
    const uint32_t m16 = o_res ? ((0xffffu << (16 - o_res)) & 0xffffu) : 0xffffu;
    const uint32_t hi_mask = m16 | (m16 << 16);
    const uint32_t mrot0 = 0x00010001u << ((16 - o_res) & 15);
    // publication staging: every iteration each lane parks its advance score at [its base + 4 k]; only the
    // rows of lanes 31 and 30 are read back (the other lanes write to a scratch area, one column each)
    const uint32_t pub_sa = sm0 + SM::PUB +
                            ((has_right && lane == 31) ? 0u : (has_right && lane == 30) ? 4u * BLK
                                                                                        : 8u * BLK + 4u * (uint32_t)lane);
    // running pointer of this lane's backpointer word of row (16-frame half-block index) - q_rows
    uint32_t *bp_ptr = g_bp + (int64_t)(-q_rows) * Sp + s;
    int bp_row = -q_rows;

    // one 16-frame backpointer word: `bits` holds the first part of row bp_row (from the previous half-block),
    // its last part is acc[hi_mask]; the rest of acc opens the next row
    auto flush_bits = [&](uint32_t acc, bool all_valid) {
        if (real && (all_valid || (bp_row >= 0 && bp_row < n_rows))) *bp_ptr = bits | (acc & hi_mask);
        bits = acc & ~hi_mask;
        bp_ptr += Sp;
        ++bp_row;
    };

    for (int j = 0; j < NB; ++j) {
        // READY covers the producer's wait for the left strip as well as the copy: the exchange bound
        hfa_mbar_wait(sm0 + SM::READY + 8u * (uint32_t)st_wait, par_wait, HFA_POLLS_EXCHANGE);
        const int st_cur = st_wait;                            // stage that holds frames BLK j .. BLK j + BLK - 1
        if (++st_wait == NSTG) {
            st_wait = 0;
            par_wait ^= 1u;
        }

        const uint32_t e_sa = tile_sa + (uint32_t)u_row * SK_ROW_B;
        const uint32_t d_sa = edge_sa + (uint32_t)u_row * 8u;
        const uint32_t k_sa = dpst_sa + (uint32_t)buf * SK_DPST_B;
        const uint32_t p_sa = pub_sa + (uint32_t)buf * SK_PUB_B;
        // all 32 lanes inside frames 1 .. T-1 for all BLK iterations?
        const bool steady = (BLK * j - 31 * D >= 1) && (BLK * j + BLK - 1 <= T - 1);

        if ((j == 0 && !has_left) || force_slow) {
            // ---------------- the block that seeds frame 0 (:250-254): rolled, one frame at a time ----------------
            uint32_t acc = 0;
#pragma unroll 1
            for (int k = 0; k < BLK; ++k) {
                const int t = BLK * j + k - lane * D;
                const bool live = (t >= 1) && (t < T);
                const float e = hfa_lds_f32(e_sa + SK_ROW_B * k);
                const float2 ed = hfa_lds_f2(d_sa + 8u * k);
                const float base = __fadd_rn(dp, e);
                const float stay = __fadd_rn(base, ed.y);
                const float adv = __double2float_rn(__dadd_rn((double)__fadd_rn(base, ed.x), P));
                const float advx = ghost ? e : adv;
                const float n1 = fminf(__shfl_up_sync(0xffffffffu, advx, 1), cap1);
                const float n2 = fminf(__shfl_up_sync(0xffffffffu, advx, 2), jcap);
                const float up1 = q1[0], up2 = q2[0];
#pragma unroll
                for (int i = 0; i + 1 < D; ++i) q1[i] = q1[i + 1];
                q1[D - 1] = n1;
#pragma unroll
                for (int i = 0; i + 1 < 2 * D; ++i) q2[i] = q2[i + 1];
                q2[2 * D - 1] = n2;
                hfa_sts_f32(p_sa + 4u * k, advx);
                const float mm = fmaxf(stay, up1);
                const bool b1 = up1 > stay, b2 = up2 > mm;
                const double pe = __dmul_rn((double)e, ratio);
                if (live) {
                    dp = fmaxf(mm, up2);
                    if (b1) acc |= 1u << (t & 15);
                    if (b2) acc |= 0x10000u << (t & 15);
                    const double pn = (b1 || b2 || pe > P) ? pe : P;
                    P = __hiloint2double(__double2hiint(pn) & (int)sp_hi, __double2loint(pn));
                }
                if (t == 0 && seeded) {                        // curr keeps the emission even for an id-0 state
                    dp = e;                                    // until the first step has run
                    P = pe;
                }
                if (KEEP) hfa_sts_f32(k_sa + 128u * k, dp);
                if (DUMP) {
                    if (!ghost && s < S && t >= 0 && t < T) dp_dump[m.cell_off + (int64_t)t * S + s] = dp;
                }
                if ((k & 15) == 15) {
                    flush_bits(acc, false);
                    acc = 0;
                }
            }
        } else {
            // ---------------- BLK iterations unrolled; `steady`: no lane needs a guard ----------------
            // operands are fetched SK_LOOK iterations ahead, interleaved with the arithmetic
            float ev[BLK];
            float2 dv[BLK];
#pragma unroll
            for (int k = 0; k < SK_LOOK; ++k) {
                ev[k] = hfa_lds_f32(e_sa + SK_ROW_B * k);
                dv[k] = hfa_lds_f2(d_sa + 8u * k);
            }
            float r1[BLK + D], r2[BLK + 2 * D];
#pragma unroll
            for (int i = 0; i < D; ++i) r1[i] = q1[i];
#pragma unroll
            for (int i = 0; i < 2 * D; ++i) r2[i] = q2[i];
            uint32_t mr = mrot0, acc = 0;
            if (!DUMP && steady) {
#pragma unroll
                for (int k = 0; k < BLK; ++k) {
                    if (k + SK_LOOK < BLK) {
                        ev[k + SK_LOOK] = hfa_lds_f32(e_sa + SK_ROW_B * (k + SK_LOOK));
                        dv[k + SK_LOOK] = hfa_lds_f2(d_sa + 8u * (k + SK_LOOK));
                    }
                    const float e = ev[k];
                    const float base = __fadd_rn(dp, e);
                    const float stay = __fadd_rn(base, dv[k].y);
                    const float adv = __double2float_rn(__dadd_rn((double)__fadd_rn(base, dv[k].x), P));
                    const float advx = ghost ? e : adv;
                    r1[k + D] = fminf(__shfl_up_sync(0xffffffffu, advx, 1), cap1);
                    r2[k + 2 * D] = fminf(__shfl_up_sync(0xffffffffu, advx, 2), jcap);
                    hfa_sts_f32(p_sa + 4u * k, advx);
                    const double pe = __dmul_rn((double)e, ratio);
                    sk_select(r1[k], stay, r2[k], pe, sp_hi, mr, dp, P, acc);
                    mr = __funnelshift_l(mr, mr, 1);
                    if (KEEP) hfa_sts_f32(k_sa + 128u * k, dp);
                    if ((k & 15) == 15) {
                        flush_bits(acc, true);
                        acc = 0;
                    }
                }
            } else {
                const int tb = BLK * j - lane * D - 1;         // (frame of iteration 0) - 1
#pragma unroll
                for (int k = 0; k < BLK; ++k) {
                    if (k + SK_LOOK < BLK) {
                        ev[k + SK_LOOK] = hfa_lds_f32(e_sa + SK_ROW_B * (k + SK_LOOK));
                        dv[k + SK_LOOK] = hfa_lds_f2(d_sa + 8u * (k + SK_LOOK));
                    }
                    const int live = (unsigned)(tb + k) < (unsigned)(T - 1);     // 1 <= t <= T-1
                    const float e = ev[k];
                    const float base = __fadd_rn(dp, e);
                    const float stay = __fadd_rn(base, dv[k].y);
                    const float adv = __double2float_rn(__dadd_rn((double)__fadd_rn(base, dv[k].x), P));
                    const float advx = ghost ? e : adv;
                    r1[k + D] = fminf(__shfl_up_sync(0xffffffffu, advx, 1), cap1);
                    r2[k + 2 * D] = fminf(__shfl_up_sync(0xffffffffu, advx, 2), jcap);
                    hfa_sts_f32(p_sa + 4u * k, advx);
                    const double pe = __dmul_rn((double)e, ratio);
                    sk_select_guarded(r1[k], stay, r2[k], pe, sp_hi, mr, live, dp, P, acc);
                    mr = __funnelshift_l(mr, mr, 1);
                    if (KEEP) hfa_sts_f32(k_sa + 128u * k, dp);
                    if (DUMP) {
                        const int t = tb + 1 + k;
                        if (!ghost && s < S && t >= 0 && t < T) dp_dump[m.cell_off + (int64_t)t * S + s] = dp;
                    }
                    if ((k & 15) == 15) {
                        flush_bits(acc, false);
                        acc = 0;
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < D; ++i) q1[i] = r1[BLK + i];
#pragma unroll
            for (int i = 0; i < 2 * D; ++i) q2[i] = r2[BLK + i];
        }
        if (KEEP) hfa_fence_async_smem();                      // this block's dp rows -> visible to the bulk store
        hfa_mbar_arrive(sm0 + SM::DONE + 8u * (uint32_t)st_cur);   // the stage, the staging rows: the producer's now
        if (++buf == SK_NBUF) buf = 0;
        u_row += BLK;
        if (u_row >= R) u_row -= R;
    }
    // a lane whose frames end before the loop does carries the first part of one more row
    if (real && o_res != 0 && bp_row >= 0 && bp_row < n_rows) *bp_ptr = bits;
    // nothing touched dp after frame T-1: it is dp[T-1][s] (:269-272 needs the last two states)
    if (!ghost) {
        if (s == S - 1) ws.dp_last[2 * u] = dp;
        if (s == S - 2) ws.dp_last[2 * u + 1] = dp;
    }
}

template <int D, int NSTG, bool KEEP, bool DUMP>
cudaError_t launch_skew(const HfaLaunchCtx &c, int item_begin, int n_items, int32_t *ticket, float *dp_dump,
                        int force_slow)
{
    const size_t smem = SkSmem<NSTG>::BYTES;
    cudaError_t e = cudaFuncSetAttribute(hfa_dp_skew_kernel<D, NSTG, KEEP, DUMP>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    hfa_dp_skew_kernel<D, NSTG, KEEP, DUMP><<<n_items, 64, smem, c.stream>>>(c.ws, item_begin, ticket, dp_dump,
                                                                            force_slow);
    return cudaGetLastError();
}

template <int D, int NSTG>
cudaError_t launch_skew_d(const HfaLaunchCtx &c, int item_begin, int n_items, int32_t *ticket, bool keep_dp,
                          float *dp_dump, int force_slow)
{
    if (dp_dump != nullptr)
        return keep_dp ? launch_skew<D, NSTG, true, true>(c, item_begin, n_items, ticket, dp_dump, force_slow)
                       : launch_skew<D, NSTG, false, true>(c, item_begin, n_items, ticket, dp_dump, force_slow);
    return keep_dp ? launch_skew<D, NSTG, true, false>(c, item_begin, n_items, ticket, dp_dump, force_slow)
                   : launch_skew<D, NSTG, false, false>(c, item_begin, n_items, ticket, dp_dump, force_slow);
}

}  // namespace

// skewed kernel: items [item_begin, item_begin + n_items) of the plan's strip table, one 2-warp CTA each.
// d = frames of skew per state (2 or 3, fixed when the plan was made: the dp store layout depends on it).
// ctas_per_sm = strips resident per SM, the plan's choice: a ring of 5 stages (43 144 B of shared memory) lets
// 5 CTAs share an SM, 6 stages (48 032 B) only 4 -- one compute warp per scheduler partition, one more tile
// fetched ahead.
cudaError_t hfa_launch_dp_skew(const HfaLaunchCtx &c, int d, int ctas_per_sm, int item_begin, int n_items,
                               int32_t *ticket, bool keep_dp, float *dp_dump)
{
    if (n_items <= 0) return cudaSuccess;
    if (c.ws.tmaps == nullptr) return cudaErrorNotSupported;
    // HFA_SKEW_SLOW=1: every block through the guarded body (A/B against the unrolled steady state)
    const char *sl = getenv("HFA_SKEW_SLOW");
    const int force_slow = (sl && sl[0] == '1') ? 1 : 0;
    if (ctas_per_sm == 4) {
        if (d == 2) return launch_skew_d<2, 6>(c, item_begin, n_items, ticket, keep_dp, dp_dump, force_slow);
        if (d == 3) return launch_skew_d<3, 6>(c, item_begin, n_items, ticket, keep_dp, dp_dump, force_slow);
    } else if (ctas_per_sm == 5) {
        if (d == 2) return launch_skew_d<2, 5>(c, item_begin, n_items, ticket, keep_dp, dp_dump, force_slow);
        if (d == 3) return launch_skew_d<3, 5>(c, item_begin, n_items, ticket, keep_dp, dp_dump, force_slow);
    }
    return cudaErrorInvalidValue;
}
