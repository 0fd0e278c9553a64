// Tempo from an onset envelope: mean inf-normalised Hann-windowed autocorrelation tempogram,
// log-normal prior, argmax lag.  Replaces librosa.feature.tempo as called at tempo.py:63-66 and
// inside librosa.beat.beat_track (tempo.py:45,159).  SURVEY.md Appendix A.3.
//
// librosa materialises an FFT autocorrelation for every frame (win_length × n_frames doubles).
// Here nothing is materialised: with w[j] = ½(1 − cos θj), θ = 2π/W, the lag-k autocorrelation
// of frame t is
//   R_t[k] = ¼[(1+½c_k)·S0 − (1+c_k)·Re S1 + s_k·Im S1 + ½c_k·Re S2 − ½s_k·Im S2],
//   S0 = Σ_j z_j,  S1 = Σ_j z_j e^{iθj},  S2 = Σ_j z_j e^{2iθj},  z_j = x[t+j]·x[t+j+k],  j < W−k,
// and all three sums slide from t to t+1 with one remove, one add and one rotation (float64).
// One thread owns one lag k and walks a chunk of frames; the per-frame normaliser R_t[0] is
// computed first by direct summation (exact, no cancellation).
//
// Only the argmax lag is observable, and every inf-normalised tempogram value is <= 1, so
// score_k = log1p(1e6·tg_k) + prior_k <= log1p(1e6) + prior_k.  The lags are therefore evaluated
// branch-and-bound: phase 1 covers the lag blocks within half an octave of the prior's centre and
// yields a best score s*; phase 2 evaluates only the remaining blocks that contain a lag with
// prior_k > s* − log1p(1e6) − 1e-6 (the prior is unimodal, so that set is one interval).  Lags outside
// cannot win, so the argmax is unchanged; typically ~80 % of the 2691 hop-64 lags are never touched.
#include "ncfa_common.cuh"

namespace ncfa {

constexpr int kLagThreads = 128;
constexpr double kReinitRatio = 1e-4;  // re-sum exactly when the frame energy collapses

// x[m], m in [0, n + 2p): envelope padded with np.pad(mode='linear_ramp', end_values=0)
__device__ __forceinline__ double padded_env(const float *__restrict__ on, int n, int p, int m) {
    if (m < p) return (double)(float)((double)m * ((double)on[0] / (double)p));
    if (m < n + p) return (double)on[m - p];
    int j = m - (n + p);
    return (double)(float)((double)(p - 1 - j) * ((double)on[n - 1] / (double)p));
}

// trig[j] = (cos θj, sin θj), w2[j] = w[j]^2
__global__ void tg_tables_kernel(int W, double2 *__restrict__ trig, double *__restrict__ w2) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= W) return;
    double s, c;
    sincospi(2.0 * (double)j / (double)W, &s, &c);
    trig[j] = make_double2(c, s);
    double w = 0.5 - 0.5 * c;
    w2[j] = w * w;
}

// pass 1: r0[seg][t] = Σ_j w[j]²·x[t+j]²  — the lag-0 autocorrelation every frame is normalised by.
// w² = 3/8 − ½cos θj + ⅛cos 2θj, so r0 = ⅜S0 − ½Re S1 + ⅛Re S2 with the same three running sums as the lags
// (L = W).  A thread owns kR0Block = 32 consecutive frames: it needs the exact sums at its first frame and slides from
// there.  The exact sums are assembled from per-block partials shared by the whole CTA — P[b] = Σ_{j<32} z[32b+j]·e^{iθj},
// S(32t) = Σ_m e^{iθ·32m}·P[t+m] + the W mod 32 tail — i.e. ~90 complex multiply-adds per thread instead of W = 2756
// terms.  Whenever the combination cancels (r0 below 1e-3 of its S0 part) the frame is re-summed directly with the w²
// table.
constexpr int kR0Block = 32;
constexpr int kR0Threads = 256;
__device__ __forceinline__ int r0_pad(int i) { return i + (i >> 5); }  // spreads the per-thread streams over banks

__global__ void __launch_bounds__(kR0Threads) tg_r0_kernel(const float *__restrict__ onset,
                                                           const int64_t *__restrict__ onset_off,
                                                           const int32_t *__restrict__ env_len, int env_stride, int W,
                                                           const double2 *__restrict__ trig,
                                                           const double *__restrict__ w2, double *__restrict__ r0,
                                                           double *__restrict__ r0inv, int frames_cap) {
    // frames_cap = frames per CTA (blockDim.x · kR0Block)
    extern __shared__ double zs[];  // r0_pad(frames_cap + W + 32) squared padded-envelope samples | block partials
    const int seg = blockIdx.y;
    const int n = env_len[seg];
    const int f0 = blockIdx.x * frames_cap;
    if (f0 >= n) return;
    const float *on = onset + onset_off[seg];
    const int p = W / 2;
    const int frames = min(frames_cap, n - f0);
    const int span = frames + W;
    const int span_cap = frames_cap + W;
    double *P = zs + r0_pad(span_cap + 32) + 1;  // [5][n_blocks]: S0, S1r, S1i, S2r, S2i of every 32-sample block
    const int n_blocks = (span_cap + 31) / 32;
    for (int i = threadIdx.x; i < n_blocks * 32; i += blockDim.x) {
        const int m = f0 + i;
        const double v = (i < span && m < n + 2 * p) ? padded_env(on, n, p, m) : 0.0;
        if (i < span_cap + 32) zs[r0_pad(i)] = v * v;
    }
    __syncthreads();
    for (int b = threadIdx.x; b < n_blocks; b += blockDim.x) {
        double S0 = 0, S1r = 0, S1i = 0, S2r = 0, S2i = 0;
        for (int j = 0; j < 32; ++j) {
            const double z = zs[r0_pad(32 * b + j)];
            const double2 a = trig[j % W];
            const double2 c = trig[(2 * j) % W];
            S0 += z;
            S1r = fma(z, a.x, S1r);
            S1i = fma(z, a.y, S1i);
            S2r = fma(z, c.x, S2r);
            S2i = fma(z, c.y, S2i);
        }
        P[b] = S0;
        P[n_blocks + b] = S1r;
        P[2 * n_blocks + b] = S1i;
        P[3 * n_blocks + b] = S2r;
        P[4 * n_blocks + b] = S2i;
    }
    __syncthreads();
    const int tb = f0 + threadIdx.x * kR0Block;
    if (tb >= n) return;
    const int te = min(n, tb + kR0Block);
    const int o0 = tb - f0;  // = 32·threadIdx.x
    double S0 = 0, S1r = 0, S1i = 0, S2r = 0, S2i = 0;
    const int M = W / 32;
    for (int m = 0; m < M; ++m) {
        const int b = threadIdx.x + m;
        const double2 a = trig[32 * m];               // e^{iθ·32m}
        const double2 c = trig[(64 * m) % W];         // e^{2iθ·32m}
        const double p1r = P[n_blocks + b], p1i = P[2 * n_blocks + b];
        const double p2r = P[3 * n_blocks + b], p2i = P[4 * n_blocks + b];
        S0 += P[b];
        S1r = fma(p1r, a.x, fma(-p1i, a.y, S1r));
        S1i = fma(p1r, a.y, fma(p1i, a.x, S1i));
        S2r = fma(p2r, c.x, fma(-p2i, c.y, S2r));
        S2i = fma(p2r, c.y, fma(p2i, c.x, S2i));
    }
    for (int j = 32 * M; j < W; ++j) {  // the W mod 32 tail
        const double z = zs[r0_pad(o0 + j)];
        const double2 a = trig[j];
        int j2 = 2 * j;
        if (j2 >= W) j2 -= W;
        const double2 c = trig[j2];
        S0 += z;
        S1r = fma(z, a.x, S1r);
        S1i = fma(z, a.y, S1i);
        S2r = fma(z, c.x, S2r);
        S2i = fma(z, c.y, S2i);
    }
    const double2 e1 = trig[1 % W], e2 = trig[2 % W];
    double *out = r0 + (size_t)seg * env_stride;
    double *out_inv = r0inv + (size_t)seg * env_stride;
    for (int t = tb; t < te; ++t) {
        const int o = t - f0;
        double r = 0.375 * S0 - 0.5 * S1r + 0.125 * S2r;
        if (!(r >= 1e-3 * (0.375 * S0))) {  // cancellation (or NaN): exact direct sum for this frame
            r = 0.0;
            for (int j = 0; j < W; ++j) r = fma(__ldg(w2 + j), zs[r0_pad(o + j)], r);
        }
        out[t] = r;
        // librosa.util.normalize(norm=inf): frames whose max (= R_t[0]) is below tiny stay unscaled.  The reciprocal is
        // the same for every lag, so it is taken once here instead of once per (lag, frame) in tg_lag_kernel.
        out_inv[t] = (r < 2.2250738585072014e-308) ? 1.0 : 1.0 / r;
        if (t + 1 < te) {
            const double d = zs[r0_pad(o + W)] - zs[r0_pad(o)];  // e^{iθW} = 1: the entering sample has phase 0 after the shift
            S0 += d;
            const double a1 = S1r + d, a2 = S2r + d;
            S1r = a1 * e1.x + S1i * e1.y;
            S1i = S1i * e1.x - a1 * e1.y;
            S2r = a2 * e2.x + S2i * e2.y;
            S2i = S2i * e2.x - a2 * e2.y;
        }
    }
}

// pass 1b: which frames must rebuild the running sums from scratch?  The first frame of every chunk, and every frame
// whose energy R_t[0] collapses below kReinitRatio of the largest energy since the last rebuild (the sliding update
// would otherwise carry the rounding error of sums 10^4 times larger).  The decision depends on the frame only, so it
// is taken once here — one warp per (segment, chunk), lanes load 32 frames at a time and replay them in order — and
// stored in the SIGN of r0inv (1/R_t[0] > 0): tg_lag_kernel then needs a single uniform load per frame.
__global__ void __launch_bounds__(128) tg_flags_kernel(const int32_t *__restrict__ env_len, int env_stride, int chunk,
                                                       int n_chunks, int n_seg, const double *__restrict__ r0,
                                                       double *__restrict__ r0inv) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n_seg * n_chunks) return;
    const int seg = w / n_chunks, c = w - seg * n_chunks;
    const int n = env_len[seg];
    const int t0 = c * chunk;
    if (t0 >= n) return;
    const int t1 = min(n, t0 + chunk);
    const double *e = r0 + (size_t)seg * env_stride;
    double *inv = r0inv + (size_t)seg * env_stride;
    double runmax = 0.0;
    bool first = true;
    for (int tb = t0; tb < t1; tb += 32) {
        const int t = tb + lane;
        const double mine = (t < t1) ? e[t] : 0.0;
        bool flag = false;
        const int cnt = min(32, t1 - tb);
        for (int l = 0; l < cnt; ++l) {
            const double e0 = __shfl_sync(0xffffffffu, mine, l);
            const bool f = first || (e0 < kReinitRatio * runmax);
            if (f) runmax = e0;
            runmax = fmax(runmax, e0);
            first = false;
            if (l == lane) flag = f;
        }
        if (t < t1 && flag) inv[t] = -inv[t];
    }
}

// pass 2: partial[seg][chunk][k] = Σ_{t in chunk} R_t[k] / R_t[0] for the lags k in todo[seg] \ done[seg] (exact
// intervals; CTA b covers todo.x + 128·b …, warps without a live lag leave at once).  One thread = one lag.
__global__ void __launch_bounds__(kLagThreads, 7) tg_lag_kernel(const float *__restrict__ onset,
                                                             const int64_t *__restrict__ onset_off,
                                                             const int32_t *__restrict__ env_len, int env_stride,
                                                             int W, int chunk, int n_chunks,
                                                             const double2 *__restrict__ trig,
                                                             const double *__restrict__ r0inv,
                                                             const int2 *__restrict__ todo,
                                                             const int2 *__restrict__ done,
                                                             double *__restrict__ partial) {
    // chunk + W padded-envelope samples.  They are float32 values (the onset envelope and the linear-ramp padding, which
    // numpy computes in the envelope's dtype), so staging them as float loses nothing and halves the shared memory of a
    // CTA: 7 instead of 4 CTAs per SM hide the FP64 latencies of the sliding update.
    extern __shared__ float xs[];
    const int seg = blockIdx.z;
    const int n = env_len[seg];
    const int t0 = blockIdx.y * chunk;
    if (t0 >= n) return;
    // A CTA serves the lag blocks blockIdx.x, blockIdx.x + gridDim.x, … of its (chunk, segment): the live lag range is
    // data dependent — 1-2 blocks of the 22 in phase 1, usually none in phase 2 — and a grid with one CTA per possible
    // block spent ~1 ms per launch scheduling CTAs that return at once (88 000 CTAs per 250 tracks, ncu r3e).
    const int2 td = todo[seg];
    int2 dn = make_int2(0, 0);
    if (done != nullptr) dn = done[seg];
    auto block_live = [&](int kb) { return !(done != nullptr && kb >= dn.x && min(kb + kLagThreads, td.y) <= dn.y); };
    bool any = false;
    for (int kb = td.x + (int)blockIdx.x * kLagThreads; kb < td.y && kb < W; kb += (int)gridDim.x * kLagThreads)
        if (block_live(kb)) {
            any = true;
            break;
        }
    if (!any) return;  // CTA-uniform
    const int t1 = min(n, t0 + chunk);
    const float *on = onset + onset_off[seg];
    const int p = W / 2;
    const int span = (t1 - t0) + W;  // x[t0 .. t1-1+W]
    for (int i = threadIdx.x; i < span; i += kLagThreads) {
        int m = t0 + i;
        xs[i] = (m < n + 2 * p) ? (float)padded_env(on, n, p, m) : 0.0f;
    }
    __syncthreads();
    const double *ri = r0inv + (size_t)seg * env_stride;
    const double2 e1 = trig[1 % W], e2 = trig[2 % W];
    for (int kb = td.x + (int)blockIdx.x * kLagThreads; kb < td.y && kb < W; kb += (int)gridDim.x * kLagThreads) {
    if (!block_live(kb)) continue;
    const int k = kb + threadIdx.x;
    const bool active = k < td.y && k < W && !(k >= dn.x && k < dn.y);
    if (!__any_sync(0xffffffffu, active)) continue;  // no barrier below: warps of a CTA are independent from here on
    // lanes without a live lag shadow the warp's first lag (live warps have kw < W): same trip counts, in-bounds reads
    const int kk = active ? k : kb + (int)(threadIdx.x & ~31u);
    const int L = W - kk;
    const double2 ek = trig[kk];
    const double2 eL = trig[L % W], e2L = trig[(2 * L) % W];
    const double q0 = 0.25 * (1.0 + 0.5 * ek.x), q1r = -0.25 * (1.0 + ek.x), q1i = 0.25 * ek.y,
                 q2r = 0.125 * ek.x, q2i = -0.125 * ek.y;
    // the warp's longest window (smallest k) bounds the uniform rebuild loop
    const int Lmax = W - min(W - 1, kb + (int)(threadIdx.x & ~31u));
    double acc = 0.0;
    int t = t0;
    while (t < t1) {
        // ---- rebuild the three running sums at frame t
        const float *xa = xs + (t - t0);
        double S0 = 0, S1r = 0, S1i = 0, S2r = 0, S2i = 0;
        auto term = [&](int j) {
            const double z = (double)xa[j] * (double)xa[j + kk];
            const double2 a = trig[j];
            int j2 = 2 * j;
            if (j2 >= W) j2 -= W;
            const double2 b = trig[j2];
            S0 += z;
            S1r = fma(z, a.x, S1r);
            S1i = fma(z, a.y, S1i);
            S2r = fma(z, b.x, S2r);
            S2i = fma(z, b.y, S2i);
        };
        // every lane of the warp has L >= Lmax - 31: that part needs no predicate, so its table loads can be batched
        const int Lcommon = Lmax > 31 ? Lmax - 31 : 0;
        int j = 0;
#pragma unroll 4
        for (; j < Lcommon; ++j) term(j);
        for (; j < Lmax; ++j)
            if (j < L) term(j);
        double inv = fabs(ri[t]);
        const float *xk = xa + kk, *xl = xa + L, *xw = xa + W;
        const double *rn = ri + t + 1;
        double nx = *rn;  // one frame ahead (the entry after the last frame is never used, but it is inside the workspace)
        // ---- slide until the chunk ends or the next frame asks for a rebuild
        for (;;) {
            const double R = q0 * S0 + q1r * S1r + q1i * S1i + q2r * S2r + q2i * S2i;
            acc = fma(R, inv, acc);
            if (++t >= t1) break;
            const double cur = nx;
            nx = *++rn;
            if (__double2hiint(cur) < 0) break;  // sign set (or a NaN with it): rebuild at t
            inv = cur;
            const double zr = (double)(*xa++) * (double)(*xk++);
            const double za = (double)(*xl++) * (double)(*xw++);
            S0 = S0 - zr + za;
            const double a1 = fma(za, eL.x, S1r - zr), b1 = fma(za, eL.y, S1i);
            S1r = a1 * e1.x + b1 * e1.y;
            S1i = b1 * e1.x - a1 * e1.y;
            const double a2 = fma(za, e2L.x, S2r - zr), b2 = fma(za, e2L.y, S2i);
            S2r = a2 * e2.x + b2 * e2.y;
            S2i = b2 * e2.x - a2 * e2.y;
        }
    }
    if (active) partial[((size_t)seg * n_chunks + blockIdx.y) * W + k] = acc;
    }  // lag blocks of this CTA
}

__device__ __forceinline__ double tg_score(const double *__restrict__ partial, int seg, int n_chunks, int used_chunks,
                                           int W, int k, int n, int hop, int sr, double l2s) {
    double s = 0.0;
    for (int c = 0; c < used_chunks; ++c) s += partial[((size_t)seg * n_chunks + c) * W + k];
    const double tg = s / (double)n;
    const double bpm = (60.0 * (double)sr) / ((double)hop * (double)k);
    const double d = log2(bpm) - l2s;
    return log1p(1e6 * tg) + (-0.5 * (d * d));
}

// phase-1 range: the lags within ±half an octave of the prior centre, [x, y) (one thread per segment)
__global__ void tg_range_kernel(int n_seg, int W, int k_min, int hop, int sr, const double *__restrict__ start_bpm,
                                int2 *__restrict__ range1) {
    const int seg = blockIdx.x * blockDim.x + threadIdx.x;
    if (seg >= n_seg) return;
    const double k0 = (60.0 * (double)sr) / ((double)hop * start_bpm[seg]);
    int klo = (int)floor(k0 / 1.4142135623730951), khi = (int)ceil(k0 * 1.4142135623730951);
    if (!(k0 == k0) || k0 <= 0.0) klo = khi = k_min;
    klo = klo < k_min ? k_min : (klo > W - 1 ? W - 1 : klo);
    khi = khi < klo ? klo : (khi > W - 1 ? W - 1 : khi);
    range1[seg] = make_int2(klo, khi + 1);
}

// after phase 1: s* = best score so far; phase-2 range = hull of lags whose prior alone could still beat it
__global__ void __launch_bounds__(256) tg_bound_kernel(const int32_t *__restrict__ env_len, int W, int n_chunks, int chunk,
                                                       int k_min, int hop, int sr, const double *__restrict__ start_bpm,
                                                       const double *__restrict__ partial, const int2 *__restrict__ range1,
                                                       int2 *__restrict__ range2, int2 *__restrict__ hull) {
    __shared__ double s_best[256];
    __shared__ int s_lo[256], s_hi[256];
    const int seg = blockIdx.x;
    const int n = env_len[seg];
    const int used_chunks = (n + chunk - 1) / chunk;
    const double l2s = log2(start_bpm[seg]);
    const int2 r1 = range1[seg];
    double best = -INFINITY;
    for (int k = r1.x + threadIdx.x; k < r1.y && k < W; k += 256)
        best = fmax(best, tg_score(partial, seg, n_chunks, used_chunks, W, k, n, hop, sr, l2s));
    s_best[threadIdx.x] = best;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) s_best[threadIdx.x] = fmax(s_best[threadIdx.x], s_best[threadIdx.x + o]);
        __syncthreads();
    }
    best = s_best[0];
    // a NaN score (degenerate envelope) disables pruning: evaluate everything
    const double cut = (best == best) ? best - 13.815511557963774 - 1e-6 : -INFINITY;  // log1p(1e6)
    int lo = 0x7fffffff, hi = -1;
    for (int k = k_min + threadIdx.x; k < W; k += 256) {
        const double bpm = (60.0 * (double)sr) / ((double)hop * (double)k);
        const double d = log2(bpm) - l2s;
        if (!(-0.5 * (d * d) <= cut)) {
            lo = k < lo ? k : lo;
            hi = k > hi ? k : hi;
        }
    }
    s_lo[threadIdx.x] = lo;
    s_hi[threadIdx.x] = hi;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            s_lo[threadIdx.x] = min(s_lo[threadIdx.x], s_lo[threadIdx.x + o]);
            s_hi[threadIdx.x] = max(s_hi[threadIdx.x], s_hi[threadIdx.x + o]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        int2 r2 = r1;
        if (s_hi[0] >= 0) r2 = make_int2(s_lo[0], s_hi[0] + 1);
        range2[seg] = r2;
        hull[seg] = make_int2(min(r1.x, r2.x), max(r1.y, r2.y));
        // lags between r1 and r2 (if disjoint) must be evaluated too so that the hull holds no garbage
        range2[seg] = hull[seg];
    }
}

// pass 3: tg[k] = Σ_chunks partial / n;  lag = argmax_k log1p(1e6·tg[k]) − ½(log2(bpm_k) − log2(start_bpm))²
__global__ void __launch_bounds__(256) tg_argmax_kernel(const float *__restrict__ onset,
                                                        const int64_t *__restrict__ onset_off,
                                                        const int32_t *__restrict__ env_len, int W, int n_chunks,
                                                        int chunk, int k_min, int hop, int sr,
                                                        const double *__restrict__ start_bpm,
                                                        const double *__restrict__ partial,
                                                        const int2 *__restrict__ hull, int32_t *__restrict__ lag_out) {
    __shared__ double s_best[256];
    __shared__ int s_idx[256];
    __shared__ int s_any;
    const int seg = blockIdx.x;
    const int n = env_len[seg];
    const float *on = onset + onset_off[seg];
    if (threadIdx.x == 0) s_any = 0;
    __syncthreads();
    int any = 0;
    for (int i = threadIdx.x; i < n; i += 256) any |= (on[i] != 0.0f);
    if (any) s_any = 1;
    __syncthreads();
    if (!s_any) {
        if (threadIdx.x == 0) lag_out[seg] = 0;
        return;
    }
    const int used_chunks = (n + chunk - 1) / chunk;
    const double l2s = log2(start_bpm[seg]);
    double best = -INFINITY;
    int bidx = 0x7fffffff;
    const int2 hl = hull[seg];
    for (int k = hl.x + threadIdx.x; k < hl.y && k < W; k += 256) {
        const double score = tg_score(partial, seg, n_chunks, used_chunks, W, k, n, hop, sr, l2s);
        if (score > best) {  // ascending k: strict > keeps the first maximum
            best = score;
            bidx = k;
        }
    }
    s_best[threadIdx.x] = best;
    s_idx[threadIdx.x] = bidx;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            double b2 = s_best[threadIdx.x + o];
            int i2 = s_idx[threadIdx.x + o];
            if (b2 > s_best[threadIdx.x] || (b2 == s_best[threadIdx.x] && i2 < s_idx[threadIdx.x])) {
                s_best[threadIdx.x] = b2;
                s_idx[threadIdx.x] = i2;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) lag_out[seg] = (s_idx[0] == 0x7fffffff) ? k_min : s_idx[0];
}

// frames per chunk of pass 2: short envelopes in one chunk, long ones in chunks of 4096 frames
static int tempo_chunk(int max_env_len) {
    if (max_env_len <= 1024) return max_env_len < 1 ? 1 : max_env_len;
    return 4096;
}

struct TempoWs {
    double2 *trig;
    double *w2, *r0, *r0inv, *partial;
    int2 *range1, *range2, *hull;
    size_t bytes;
};

static TempoWs tempo_ws(int n_seg, int max_env_len, int W, void *base) {
    const int chunk = tempo_chunk(max_env_len);
    const size_t n_chunks = (max_env_len + chunk - 1) / chunk;
    Carve c(base);
    TempoWs w;
    w.trig = c.take<double2>(W);
    w.w2 = c.take<double>(W);
    w.r0 = c.take<double>((size_t)n_seg * max_env_len);
    w.r0inv = c.take<double>((size_t)n_seg * max_env_len);
    w.partial = c.take<double>((size_t)n_seg * n_chunks * W);
    w.range1 = c.take<int2>(n_seg);
    w.range2 = c.take<int2>(n_seg);
    w.hull = c.take<int2>(n_seg);
    w.bytes = c.used;
    return w;
}

}  // namespace ncfa

using namespace ncfa;

extern "C" size_t ncfa_tempo_workspace_bytes(int n_seg, int max_env_len, int win_length) {
    if (n_seg <= 0 || max_env_len <= 0 || win_length <= 0) return 0;
    return tempo_ws(n_seg, max_env_len, win_length, nullptr).bytes;
}

extern "C" int ncfa_tempo_lag_batched(const float *d_onset, const int64_t *d_onset_off, const int32_t *d_env_len,
                                      int n_seg, int max_env_len, int hop, int sr, const double *d_start_bpm,
                                      int32_t *d_lag, void *d_workspace, size_t workspace_bytes, void *stream) {
    NCFA_REQUIRE(n_seg >= 0 && n_seg <= 65535, "n_seg must be in [0, 65535] per call");
    if (n_seg == 0) return NCFA_OK;
    NCFA_REQUIRE(d_onset && d_onset_off && d_env_len && d_start_bpm && d_lag && d_workspace, "null pointer");
    NCFA_REQUIRE(hop > 0 && sr > 0 && max_env_len > 0, "hop/sr/max_env_len");
    const int W = (int)floor(8.0 * (double)sr / (double)hop);  // time_to_frames(ac_size=8.0)
    NCFA_REQUIRE(W >= 4 && W <= 5000, "win_length out of the supported range [4, 5000]");
    const TempoWs w = tempo_ws(n_seg, max_env_len, W, d_workspace);
    int rc = check_workspace("tempo", workspace_bytes, w.bytes);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int chunk = tempo_chunk(max_env_len);
    const int n_chunks = (max_env_len + chunk - 1) / chunk;

    // first lag whose bpm is below max_tempo = 320 (logprior[:max_idx] = -inf)
    int k_min = 1;
    while (k_min < W && !((60.0 * (double)sr) / ((double)hop * (double)k_min) < 320.0)) ++k_min;
    NCFA_REQUIRE(k_min < W, "no admissible lag");

    if ((rc = launch("tg_tables_kernel", tg_tables_kernel, (W + 255) / 256, 256, 0, st, W, w.trig, w.w2))) return rc;
    {
        // frames per CTA: 8192 for whole tracks, one warp's worth of 32-frame blocks for short envelopes
        int threads = ((max_env_len + kR0Block - 1) / kR0Block + 31) / 32 * 32;
        threads = threads < 32 ? 32 : (threads > kR0Threads ? kR0Threads : threads);
        const int per_cta = threads * kR0Block;
        dim3 g((max_env_len + per_cta - 1) / per_cta, n_seg);
        const int span_cap = per_cta + W;
        const int n_blocks = (span_cap + 31) / 32;
        size_t sh = (size_t)(span_cap + 32 + ((span_cap + 32) >> 5) + 2 + 5 * n_blocks) * 8;
        if ((rc = launch("tg_r0_kernel", tg_r0_kernel, g, threads, sh, st, d_onset, d_onset_off, d_env_len, max_env_len,
                         W, w.trig, w.w2, w.r0, w.r0inv, per_cta)))
            return rc;
    }
    if ((rc = launch("tg_range_kernel", tg_range_kernel, (n_seg + 127) / 128, 128, 0, st, n_seg, W, k_min, hop, sr,
                     d_start_bpm, w.range1)))
        return rc;
    const int warps = n_seg * n_chunks;
    if ((rc = launch("tg_flags_kernel", tg_flags_kernel, (warps + 3) / 4, 128, 0, st, d_env_len, max_env_len, chunk,
                     n_chunks, n_seg, w.r0, w.r0inv)))
        return rc;
    const char *lag_name = n_chunks > 1 ? "tg_lag_kernel[long]" : "tg_lag_kernel";
    const int lag_blocks = (W - k_min + kLagThreads - 1) / kLagThreads;
    const dim3 g(lag_blocks < 2 ? lag_blocks : 2, n_chunks, n_seg);  // a CTA strides over the lag blocks (the kernel)
    const size_t sh = (size_t)(chunk + W) * 4;
    if ((rc = launch(lag_name, tg_lag_kernel, g, kLagThreads, sh, st, d_onset, d_onset_off, d_env_len, max_env_len, W,
                     chunk, n_chunks, w.trig, w.r0inv, w.range1, nullptr, w.partial)))
        return rc;
    if ((rc = launch("tg_bound_kernel", tg_bound_kernel, n_seg, 256, 0, st, d_env_len, W, n_chunks, chunk, k_min, hop,
                     sr, d_start_bpm, w.partial, w.range1, w.range2, w.hull)))
        return rc;
    if ((rc = launch(lag_name, tg_lag_kernel, g, kLagThreads, sh, st, d_onset, d_onset_off, d_env_len, max_env_len, W,
                     chunk, n_chunks, w.trig, w.r0inv, w.range2, w.range1, w.partial)))
        return rc;
    return launch("tg_argmax_kernel", tg_argmax_kernel, n_seg, 256, 0, st, d_onset, d_onset_off, d_env_len, W, n_chunks,
                  chunk, k_min, hop, sr, d_start_bpm, w.partial, w.hull, d_lag);
}
