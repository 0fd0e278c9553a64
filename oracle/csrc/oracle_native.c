/*
 * Plain-C restatement of the sequential inner loops of the reference hot path.
 * TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Compile with
 *   gcc -O2 -ffp-contract=off -shared -fPIC   (no FMA contraction: numba/numpy do not fuse)
 *
 *  orc_local_score  : librosa.beat.__beat_local_score, static tempo  (SURVEY Appendix A.4; tempo.py:45,159)
 *  orc_beat_dp      : librosa.beat.__beat_track_dp                    (SURVEY Appendix A.4)
 *  orc_beat_dp_pen  : the same DP on a given penalty table, with per-frame predecessor margins
 *  orc_bootstrap    : numpy Generator(PCG64).choice(..., replace=True) + median, the loop of
 *                     consensus.py:259-262 / :304-307 / pitch.py:145-148 (SURVEY §4 RNG KATs)
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef unsigned __int128 u128;

void orc_local_score(const double *onset, int64_t N, const double *window, int64_t K, double *out) {
    for (int64_t i = 0; i < N; ++i) {
        double acc = 0.0;
        int64_t k0 = i + K / 2 - N + 1;
        if (k0 < 0) k0 = 0;
        int64_t k1 = i + K / 2;
        if (k1 > K) k1 = K;
        for (int64_t k = k0; k < k1; ++k) acc += window[k] * onset[i + K / 2 - k];
        out[i] = acc;
    }
}

/* pen == NULL: the transition penalty is tightness·(log(d) − log(fpb))², as librosa computes it; otherwise it is read
 * from the table pen[d − near], d = near .. far (a caller that wants another machine's log).  margin != NULL receives,
 * per frame, (best − second best) / max(|best|, |second best|) over its candidate predecessors (+inf with fewer than
 * two candidates, 0 on an exact tie). */
static void beat_dp(const double *ls, int64_t N, double fpb, double tightness, const double *pen, int64_t *backlink,
                    double *cumscore, double *margin) {
    double mx = ls[0];
    for (int64_t i = 1; i < N; ++i)
        if (ls[i] > mx) mx = ls[i];
    const double score_thresh = 0.01 * mx;
    int first_beat = 1;
    backlink[0] = -1;
    cumscore[0] = ls[0];
    const int64_t near = (int64_t)nearbyint(fpb / 2.0); /* np.round: half to even */
    const int64_t far = (int64_t)(2.0 * fpb);
    const double logf = log(fpb);
    for (int64_t i = 0; i < N; ++i) {
        double best = -INFINITY, second = -INFINITY;
        int64_t bl = -1;
        for (int64_t loc = i - near; loc > i - far - 1; --loc) {
            if (loc < 0) break;
            double score;
            if (pen) {
                score = cumscore[loc] - pen[i - loc - near];
            } else {
                double d = log((double)(i - loc)) - logf;
                score = cumscore[loc] - tightness * (d * d);
            }
            if (score > best) {
                second = best;
                best = score;
                bl = loc;
            } else if (score > second) {
                second = score;
            }
        }
        if (margin) {
            if (second == -INFINITY) {
                margin[i] = INFINITY;
            } else {
                double s = fabs(best) > fabs(second) ? fabs(best) : fabs(second);
                margin[i] = (best == second) ? 0.0 : (best - second) / s;
            }
        }
        cumscore[i] = (bl >= 0) ? ls[i] + best : ls[i];
        if (first_beat && ls[i] < score_thresh) {
            backlink[i] = -1;
        } else {
            backlink[i] = bl;
            first_beat = 0;
        }
    }
}

void orc_beat_dp(const double *ls, int64_t N, double fpb, double tightness, int64_t *backlink, double *cumscore) {
    beat_dp(ls, N, fpb, tightness, NULL, backlink, cumscore, NULL);
}

/* orc_beat_dp with the penalty table pen[d − near] (NULL: librosa's log form) and the optional per-frame margin */
void orc_beat_dp_pen(const double *ls, int64_t N, double fpb, double tightness, const double *pen, int64_t *backlink,
                     double *cumscore, double *margin) {
    beat_dp(ls, N, fpb, tightness, pen, backlink, cumscore, margin);
}

/* ---- PCG64 (numpy): 128-bit LCG step, then XSL-RR output of the new state ---- */
typedef struct {
    u128 state, inc;
    int has32;
    uint32_t buf32;
} pcg_t;

static const u128 PCG_MULT = (((u128)0x2360ED051FC65DA4ULL) << 64) | 0x4385DF649FCCF645ULL;

static inline uint64_t pcg_next64(pcg_t *g) {
    g->state = g->state * PCG_MULT + g->inc;
    uint64_t hi = (uint64_t)(g->state >> 64), lo = (uint64_t)g->state;
    uint64_t x = hi ^ lo;
    unsigned rot = (unsigned)(g->state >> 122);
    return (x >> rot) | (x << ((64 - rot) & 63));
}

static inline uint32_t pcg_next32(pcg_t *g) {
    if (g->has32) {
        g->has32 = 0;
        return g->buf32;
    }
    uint64_t v = pcg_next64(g);
    g->has32 = 1;
    g->buf32 = (uint32_t)(v >> 32);
    return (uint32_t)(v & 0xffffffffu);
}

/* numpy buffered_bounded_lemire_uint32, rng = n-1 */
static inline uint32_t bounded32(pcg_t *g, uint32_t n) {
    if (n == 1) return 0;
    uint64_t m = (uint64_t)pcg_next32(g) * n;
    uint32_t leftover = (uint32_t)m;
    if (leftover < n) {
        uint32_t threshold = (uint32_t)((0xffffffffu - (n - 1)) % n);
        while (leftover < threshold) {
            m = (uint64_t)pcg_next32(g) * n;
            leftover = (uint32_t)m;
        }
    }
    return (uint32_t)(m >> 32);
}

static int cmp_double(const void *a, const void *b) {
    double x = *(const double *)a, y = *(const double *)b;
    return (x > y) - (x < y);
}

static double median_inplace(double *v, int n) {
    qsort(v, n, sizeof(double), cmp_double);
    if (n & 1) return v[n / 2];
    return (v[n / 2 - 1] + v[n / 2]) / 2.0; /* np.median: mean of the two middle values */
}

/* a is drawn first, then b (b may be NULL / nb = 0 for the single-array pitch bootstrap).
 * boot[i] = median(a*) / median(b*)   (or median(a*) when nb == 0)
 * idx_out (optional): all bounded draws in order, n_boot*(na+nb) int32. */
void orc_bootstrap(const double *a, int na, const double *b, int nb, int n_boot, uint64_t st_hi, uint64_t st_lo,
                   uint64_t inc_hi, uint64_t inc_lo, double *boot, int32_t *idx_out) {
    pcg_t g;
    g.state = ((u128)st_hi << 64) | st_lo;
    g.inc = ((u128)inc_hi << 64) | inc_lo;
    g.has32 = 0;
    g.buf32 = 0;
    double *ta = (double *)malloc(sizeof(double) * (na > 0 ? na : 1));
    double *tb = (double *)malloc(sizeof(double) * (nb > 0 ? nb : 1));
    int64_t w = 0;
    for (int i = 0; i < n_boot; ++i) {
        for (int j = 0; j < na; ++j) {
            uint32_t r = bounded32(&g, (uint32_t)na);
            ta[j] = a[r];
            if (idx_out) idx_out[w++] = (int32_t)r;
        }
        for (int j = 0; j < nb; ++j) {
            uint32_t r = bounded32(&g, (uint32_t)nb);
            tb[j] = b[r];
            if (idx_out) idx_out[w++] = (int32_t)r;
        }
        double ma = median_inplace(ta, na);
        boot[i] = nb > 0 ? ma / median_inplace(tb, nb) : ma;
    }
    free(ta);
    free(tb);
}

/* raw stream access for the known-answer tests */
void orc_pcg64_raw(uint64_t st_hi, uint64_t st_lo, uint64_t inc_hi, uint64_t inc_lo, int n, uint64_t *out) {
    pcg_t g;
    g.state = ((u128)st_hi << 64) | st_lo;
    g.inc = ((u128)inc_hi << 64) | inc_lo;
    g.has32 = 0;
    for (int i = 0; i < n; ++i) out[i] = pcg_next64(&g);
}
