/*
 * hfa_oracle_lowmem.c -- TEST INFRASTRUCTURE ONLY.  The DP of hfa_oracle_decode (hfa_oracle.c) in about
 * 0.25 B per DP cell instead of 5: two rolling dp rows and 2-bit backpointers, with the emission rows fed
 * in chunks so that the caller never holds the [T][S] matrix either.  Same arithmetic, operation for
 * operation (the arithmetic contract at the top of hfa_oracle.c holds here too: build with
 * -ffp-contract=off, no -ffast-math), so path, end state and dp are bit-identical to hfa_oracle_decode.
 *
 * dp along the path (the reference's dp_path, alignment_decoder.py:276) is not kept by the forward pass;
 * hfa_lowmem_path_rows recomputes it in a second pass over the same rows.  dp[t][s_t] is the candidate the
 * recorded backpointer chose: it needs dp[t-1][s_{t-1}] (the previous entry), e[t][s_{t-1}], the edge logs
 * of frame t and curr[s_{t-1}] -- which depends only on the backpointers of column s_{t-1} back to the frame
 * the path entered it, i.e. on the path itself.
 *
 * Use: create -> rows (frames 0 .. T-1 in order, any chunking) -> finish -> [path_rows (0 .. T-1)] -> destroy.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define HFA_NEG_INF (-INFINITY)

typedef struct {
    int32_t T, S, t_next, t_path, rc;
    int32_t *ids;
    double ratio;
    float *prev, *cur, *adv;
    double *curr;
    uint8_t *bt;          /* [T][ceil(S/4)], 2 bits per cell: 0 stay, 1 advance, 2 jump (row 0 unused) */
    int64_t row_bytes;
    int32_t *path;        /* [T] state of the best path at every frame (after finish)                 */
    float path_dp;        /* dp_path of the last frame path_rows handled                              */
    double path_curr;     /* curr of that frame's path state                                          */
} hfa_lowmem;

void hfa_lowmem_destroy(hfa_lowmem *h)
{
    if (!h) return;
    free(h->ids); free(h->prev); free(h->cur); free(h->adv); free(h->curr); free(h->bt); free(h->path);
    free(h);
}

hfa_lowmem *hfa_lowmem_create(int32_t T, int32_t S, const int32_t *ph_ids)
{
    if (T < 1 || S < 1) return 0;
    hfa_lowmem *h = (hfa_lowmem *)calloc(1, sizeof(hfa_lowmem));
    if (!h) return 0;
    h->T = T;
    h->S = S;
    h->row_bytes = ((int64_t)S + 3) / 4;
    h->ids = (int32_t *)malloc(sizeof(int32_t) * (size_t)S);
    h->prev = (float *)malloc(sizeof(float) * (size_t)S);
    h->cur = (float *)malloc(sizeof(float) * (size_t)S);
    h->adv = (float *)malloc(sizeof(float) * (size_t)S);
    h->curr = (double *)malloc(sizeof(double) * (size_t)S);
    h->bt = (uint8_t *)calloc((size_t)T * (size_t)h->row_bytes, 1);
    h->path = (int32_t *)malloc(sizeof(int32_t) * (size_t)T);
    if (!h->ids || !h->prev || !h->cur || !h->adv || !h->curr || !h->bt || !h->path) {
        hfa_lowmem_destroy(h);
        return 0;
    }
    memcpy(h->ids, ph_ids, sizeof(int32_t) * (size_t)S);
    h->ratio = (double)T / (double)S;                                /* :186,:201  T / S */
    return h;
}

/* frames t_next .. t_next + n - 1: prob_log [n][ld] (gathered emissions), edge_log / not_edge_log [n] */
int hfa_lowmem_rows(hfa_lowmem *h, int32_t n, const float *prob_log, int64_t ld, const float *edge_log,
                    const float *not_edge_log)
{
    if (!h || n < 0 || h->t_next + (int64_t)n > h->T) return -1;
    const int32_t S = h->S;
    const int32_t *ids = h->ids;
    for (int32_t r = 0; r < n; ++r) {
        const int32_t t = h->t_next++;
        const float *e = prob_log + (int64_t)r * ld;
        if (t == 0) {                                                /* :245-254 */
            for (int32_t i = 0; i < S; ++i) { h->prev[i] = HFA_NEG_INF; h->curr[i] = (double)HFA_NEG_INF; }
            h->prev[0] = e[0];
            h->curr[0] = (double)e[0];
            if (ids[0] == 0 && S > 1) {
                h->prev[1] = e[1];
                h->curr[1] = (double)e[1];
            }
            continue;
        }
        const float *prev = h->prev;
        float *cur = h->cur;
        uint8_t *btr = h->bt + (int64_t)t * h->row_bytes;
        const float el = edge_log[r], ne = not_edge_log[r];
        for (int32_t j = 0; j < S; ++j) {
            const float a = (prev[j] + e[j]) + el;
            h->adv[j] = (float)((double)a + h->curr[j] * h->ratio);
        }
        for (int32_t i = 0; i < S; ++i) {
            const float stay = (prev[i] + e[i]) + ne;
            const float one = (i >= 1) ? h->adv[i - 1] : HFA_NEG_INF;
            const float two = (i >= 2 && ids[i - 1] == 0) ? h->adv[i - 2] : HFA_NEG_INF;
            const int g1 = one > stay;
            const float m = g1 ? one : stay;
            const int g2 = two > m;
            cur[i] = g2 ? two : m;
            const int code = g2 ? 2 : g1;
            btr[i >> 2] |= (uint8_t)(code << (2 * (i & 3)));
            const double ei = (double)e[i];
            const double held = (ei > h->curr[i]) ? ei : h->curr[i];
            const double c = (code == 0) ? held : ei;
            h->curr[i] = (ids[i] == 0) ? 0.0 : c;
        }
        h->cur = h->prev;
        h->prev = cur;
    }
    return 0;
}

static int bt_code(const hfa_lowmem *h, int32_t t, int32_t s)
{
    return (h->bt[(int64_t)t * h->row_bytes + (s >> 2)] >> (2 * (s & 3))) & 3;
}

/* after all T rows: end state (:269-272), backtrace (:274-283), dp[T-1][end] */
int hfa_lowmem_finish(hfa_lowmem *h, int32_t *ph_idx_seq, int32_t *ph_time_int, int32_t *n_seg,
                      int32_t *end_state, float *final_score)
{
    if (!h || h->t_next != h->T) return -1;
    const int32_t S = h->S, T = h->T;
    const float *last = h->prev;
    int32_t s = S - 1;
    if (S >= 2 && last[S - 2] > last[S - 1] && h->ids[S - 1] == 0) s = S - 2;
    *end_state = s;
    *final_score = last[s];
    int32_t n = 0;
    for (int32_t t = T - 1; t >= 0; --t) {
        h->path[t] = s;
        const int code = (t == 0) ? -1 : bt_code(h, t, s);
        if (code != 0) {
            if (n < S) { ph_idx_seq[n] = s; ph_time_int[n] = t; }
            ++n;
            s -= code;
        }
    }
    if (n > S) return -3;
    for (int32_t a = 0, b = n - 1; a < b; ++a, --b) {
        int32_t tmp = ph_idx_seq[a]; ph_idx_seq[a] = ph_idx_seq[b]; ph_idx_seq[b] = tmp;
        tmp = ph_time_int[a]; ph_time_int[a] = ph_time_int[b]; ph_time_int[b] = tmp;
    }
    *n_seg = n;
    return 0;
}

/* second pass, frames t_path .. t_path + n - 1 in order: dp_path[r] = dp[t][s_t] (:276) */
int hfa_lowmem_path_rows(hfa_lowmem *h, int32_t n, const float *prob_log, int64_t ld, const float *edge_log,
                         const float *not_edge_log, float *dp_path)
{
    if (!h || h->t_next != h->T || n < 0 || h->t_path + (int64_t)n > h->T) return -1;
    for (int32_t r = 0; r < n; ++r) {
        const int32_t t = h->t_path++;
        const float *e = prob_log + (int64_t)r * ld;
        const int32_t s = h->path[t];
        if (t == 0) {
            const int seeded = s == 0 || (s == 1 && h->ids[0] == 0 && h->S > 1);
            h->path_dp = seeded ? e[s] : HFA_NEG_INF;
            h->path_curr = seeded ? (double)e[s] : (double)HFA_NEG_INF;
        } else {
            const int code = bt_code(h, t, s);
            const int32_t j = s - code;                              /* the path's state at t - 1 */
            float v;
            if (code == 0) {
                v = (h->path_dp + e[s]) + not_edge_log[r];
            } else {
                const float a = (h->path_dp + e[j]) + edge_log[r];
                v = (float)((double)a + h->path_curr * h->ratio);
            }
            const double ei = (double)e[s];
            const double held = (ei > h->path_curr) ? ei : h->path_curr;
            const double c = (code == 0) ? held : ei;
            h->path_curr = (h->ids[s] == 0) ? 0.0 : c;
            h->path_dp = v;
        }
        dp_path[r] = h->path_dp;
    }
    return 0;
}
