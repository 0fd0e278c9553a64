// Dynamic-programming beat tracker.  Replaces librosa.beat.beat_track(onset_envelope, sr,
// hop_length, start_bpm) as called at tempo.py:45-49 and tempo.py:159-164 (the tempo itself comes
// from tempo.cu; frames-per-beat = round(60·(sr/hop)/bpm) = the tempogram lag).  SURVEY Appendix A.4.
//
// One CTA per envelope.  All arithmetic is float64 and this file is compiled with -fmad=false so
// that sums and products round exactly like the CPU restatement (oracle/csrc/oracle_native.c).
// The DP is sequential in time, but frame i only looks back to [i-2·fpb, i-round(fpb/2)], so
// round(fpb/2) consecutive frames are independent: they form one wavefront, computed in parallel.
#include "ncfa_common.cuh"

namespace ncfa {

struct BeatWs {
    double *onorm, *ls, *cum, *window, *pen;
    int32_t *backlink, *tmp;
};

__device__ __forceinline__ unsigned long long f64_to_ordered(double d) {
    unsigned long long u = (unsigned long long)__double_as_longlong(d);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double ordered_to_f64(unsigned long long u) {
    return __longlong_as_double((long long)((u >> 63) ? (u & 0x7fffffffffffffffull) : ~u));
}

__device__ __forceinline__ bool is_localmax(const double *c, int i, int n) {
    if (i < 1) return false;
    const double r = c[i + 1 < n ? i + 1 : n - 1];
    return c[i] > c[i - 1] && c[i] >= r;
}

// block-wide sum / max / min helpers (deterministic tree)
template <typename T, typename Op>
__device__ T block_reduce(T v, T *sh, Op op) {
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = blockDim.x >> 1; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] = op(sh[threadIdx.x], sh[threadIdx.x + o]);
        __syncthreads();
    }
    T r = sh[0];
    __syncthreads();
    return r;
}

// rank-th smallest (0-based) of {cum[i] : localmax(i)} by 8-bit radix select on ordered keys
__device__ double select_localmax(const double *cum, int n, int rank, int *hist, unsigned long long *s_prefix,
                                  int *s_rank) {
    if (threadIdx.x == 0) {
        *s_prefix = 0ull;
        *s_rank = rank;
    }
    __syncthreads();
    for (int shift = 56; shift >= 0; shift -= 8) {
        for (int b = threadIdx.x; b < 256; b += blockDim.x) hist[b] = 0;
        __syncthreads();
        const unsigned long long prefix = *s_prefix;
        const unsigned long long himask = (shift == 56) ? 0ull : (~0ull << (shift + 8));
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            if (is_localmax(cum, i, n)) {
                unsigned long long key = f64_to_ordered(cum[i]);
                if ((key & himask) == prefix) atomicAdd(&hist[(int)((key >> shift) & 0xff)], 1);
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int r = *s_rank, b = 0;
            while (b < 255 && r >= hist[b]) {
                r -= hist[b];
                ++b;
            }
            *s_rank = r;
            *s_prefix = prefix | ((unsigned long long)b << shift);
        }
        __syncthreads();
    }
    return ordered_to_f64(*s_prefix);
}

// Workspace of one segment (doubles): onorm[env_stride] | ls[env_stride] | cum[env_stride] | window[2·max_fpb+1] |
// (2·max_fpb+1 unused) | 8 spare — spare[0] holds max(ls) as an order-preserving 64-bit key.
__device__ __forceinline__ double *beat_seg_base(double *ws_f64, int seg, int env_stride, int max_fpb) {
    const size_t K = 2 * (size_t)max_fpb + 1;
    return ws_f64 + (size_t)seg * (3 * (size_t)env_stride + 2 * K + 8);
}

// pass 1 (one CTA per envelope): onsets / (std(ddof=1) + tiny) and the Gaussian window exp(-½((k-fpb)·32/fpb)²)
__global__ void __launch_bounds__(256) beat_prep_kernel(const float *__restrict__ onset,
                                                        const int64_t *__restrict__ onset_off,
                                                        const int32_t *__restrict__ env_len, int env_stride,
                                                        const int32_t *__restrict__ lag, double *__restrict__ ws_f64,
                                                        int max_fpb) {
    __shared__ double sh_d[256];
    const int seg = blockIdx.x;
    const int N = env_len[seg];
    const int fpb = lag[seg];
    if (fpb < 2 || fpb > max_fpb || N < 2) return;
    const float *on = onset + onset_off[seg];
    const int tid = threadIdx.x, nt = blockDim.x;
    const size_t K = 2 * (size_t)max_fpb + 1;
    double *base = beat_seg_base(ws_f64, seg, env_stride, max_fpb);
    double *onorm = base, *window = base + 3 * (size_t)env_stride;
    if (tid == 0) *reinterpret_cast<unsigned long long *>(window + 2 * K) = f64_to_ordered(-INFINITY);
    // ---- onsets / (std(ddof=1) + tiny)
    double s = 0.0;
    for (int i = tid; i < N; i += nt) s += (double)on[i];
    const double mean = block_reduce(s, sh_d, [](double a, double b) { return a + b; }) / (double)N;
    s = 0.0;
    for (int i = tid; i < N; i += nt) {
        double d = (double)on[i] - mean;
        s += d * d;
    }
    const double var = block_reduce(s, sh_d, [](double a, double b) { return a + b; }) / (double)(N - 1);
    const double denom = sqrt(var) + 2.2250738585072014e-308;
    for (int i = tid; i < N; i += nt) onorm[i] = (double)on[i] / denom;

    const int Kw = 2 * fpb + 1;
    const double dfpb = (double)fpb;
    for (int k = tid; k < Kw; k += nt) {
        double a = ((double)(k - fpb) * 32.0) / dfpb;
        window[k] = exp(-0.5 * (a * a));
    }
}

// pass 2 (all frames of all envelopes in parallel): local score = 'same' convolution of the normalised onsets with
// the window, restated with librosa's loop bounds (ascending k, unfused multiply-add), and its maximum per envelope
constexpr int kScoreFramesPerThread = 4;  // the sliding window below is written for 4
__global__ void __launch_bounds__(256) beat_score_kernel(const int32_t *__restrict__ env_len, int env_stride,
                                                         const int32_t *__restrict__ lag, double *__restrict__ ws_f64,
                                                         int max_fpb) {
    __shared__ double sh_d[256];
    const int seg = blockIdx.x;
    const int N = env_len[seg];
    const int fpb = lag[seg];
    if (fpb < 2 || fpb > max_fpb || N < 2) return;
    const int i0 = blockIdx.y * (256 * kScoreFramesPerThread);
    if (i0 >= N) return;
    const size_t K = 2 * (size_t)max_fpb + 1;
    double *base = beat_seg_base(ws_f64, seg, env_stride, max_fpb);
    const double *onorm = base, *window = base + 3 * (size_t)env_stride;
    double *ls = base + env_stride;
    const int Kw = 2 * fpb + 1;
    // the CTA's slice of the normalised onsets, onorm[i0 − fpb … i0 + 1023 + fpb], staged in shared memory with a skewed
    // index (e + e/16): lanes read elements 4 apart, which would otherwise be a 4-way bank conflict — and, from global
    // memory, 32 sectors per load instruction (the LSU queue was the top stall of this kernel, profiles r1bl)
    extern __shared__ double tile[];
    const int lo_idx = i0 - fpb;
    const int span = min(256 * kScoreFramesPerThread, N - i0) + 2 * fpb + 1;
    for (int e = threadIdx.x; e < span; e += 256) {
        const int idx = lo_idx + e;
        tile[e + (e >> 4)] = (idx >= 0 && idx < N) ? onorm[idx] : 0.0;
    }
    __syncthreads();
    double lmax = -INFINITY;
    // a thread owns kScoreFramesPerThread CONSECUTIVE frames: away from the envelope's ends all of them run over the
    // full window, so one window load and one new onset load feed four multiply-adds (register sliding window); every
    // frame still adds its products in ascending k, exactly like the one-frame loop used at the ends
    const int ib = i0 + (int)threadIdx.x * kScoreFramesPerThread;
    if (ib < N) {
        if (ib + fpb >= Kw && ib + kScoreFramesPerThread - 1 + fpb - N + 1 <= 0) {
            // acc_r = Σ_k window[k]·onorm[ib + r + fpb − k]: with x_j = onorm[ib + fpb − k + j], step k → k+1 shifts x down
            const int e0 = (ib - i0) + 2 * fpb;  // tile index of onorm[ib + fpb]
            auto T = [&](int e) { return tile[e + (e >> 4)]; };
            double x0 = T(e0), x1 = T(e0 + 1), x2 = T(e0 + 2), x3 = T(e0 + 3);
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
            for (int k = 0; k < Kw; ++k) {
                const double w = window[k];
                a0 = a0 + w * x0;
                a1 = a1 + w * x1;
                a2 = a2 + w * x2;
                a3 = a3 + w * x3;
                x3 = x2;
                x2 = x1;
                x1 = x0;
                const int en = e0 - (k + 1);  // −1 after the last tap of the tile's first frame: that value is never used
                x0 = T(en < 0 ? 0 : en);
            }
            ls[ib] = a0;
            ls[ib + 1] = a1;
            ls[ib + 2] = a2;
            ls[ib + 3] = a3;
            lmax = fmax(fmax(a0, a1), fmax(a2, a3));
        } else {
            for (int r = 0; r < kScoreFramesPerThread; ++r) {
                const int i = ib + r;
                if (i >= N) break;
                int k0 = i + fpb - N + 1;
                if (k0 < 0) k0 = 0;
                int k1 = i + fpb;
                if (k1 > Kw) k1 = Kw;
                double acc = 0.0;
                for (int k = k0; k < k1; ++k) acc = acc + window[k] * onorm[i + fpb - k];
                ls[i] = acc;
                lmax = fmax(lmax, acc);
            }
        }
    }
    lmax = block_reduce(lmax, sh_d, [](double a, double b) { return fmax(a, b); });
    if (threadIdx.x == 0)
        atomicMax(reinterpret_cast<unsigned long long *>(base + 3 * (size_t)env_stride + 2 * K), f64_to_ordered(lmax));
}

// The DP exploits that the best predecessor moves monotonically with the frame — see the comment at the wavefront loop.
__global__ void beat_track_kernel(const float *__restrict__ onset, const int64_t *__restrict__ onset_off,
                                  const int32_t *__restrict__ env_len, int env_stride, const int32_t *__restrict__ lag,
                                  double *__restrict__ ws_f64, int32_t *__restrict__ ws_i32, int max_fpb,
                                  int32_t *__restrict__ beats_out, int max_beats, int32_t *__restrict__ n_beats,
                                  int ring) {
    // blockDim doubles (reductions) | ring doubles: cumulative scores of the last `ring` frames (power of two >=
    // far + near for every admissible fpb) | transition penalties for d = near .. far
    extern __shared__ double sh_d[];
    double *cring = sh_d + blockDim.x;
    double *pen = cring + ring;
    const int rmask = ring - 1;
    __shared__ int hist[256];
    __shared__ unsigned long long s_prefix;
    __shared__ int s_rank, s_cnt;
    __shared__ double s_thr;
    const int seg = blockIdx.x;
    const int N = env_len[seg];
    const int fpb = lag[seg];
    const int tid = threadIdx.x, nt = blockDim.x;
    if (fpb < 2 || fpb > max_fpb || N < 2) {
        if (tid == 0) n_beats[seg] = 0;
        return;
    }
    // workspace carve-up (per segment)
    const size_t K = 2 * (size_t)max_fpb + 1;
    double *base = ws_f64 + (size_t)seg * (3 * (size_t)env_stride + 2 * K + 8);
    double *ls = base + env_stride, *cum = base + 2 * (size_t)env_stride;
    double *window = base + 3 * (size_t)env_stride;
    int32_t *backlink = ws_i32 + (size_t)seg * 2 * env_stride, *tmp = backlink + env_stride;

    // (onset normalisation, the Gaussian window and the local score come from beat_prep_kernel / beat_score_kernel)
    const double dfpb = (double)fpb;
    const int near = (int)rint(dfpb / 2.0);  // np.round: half to even
    const int far = 2 * fpb;
    const double logf = log(dfpb);
    for (int d = near + tid; d <= far; d += nt) {
        double x = log((double)d) - logf;
        pen[d - near] = 100.0 * (x * x);
    }
    __syncthreads();

    const double lmax = ordered_to_f64(*reinterpret_cast<const unsigned long long *>(window + 2 * K));
    const double score_thresh = 0.01 * lmax;
    // first frame whose local score reaches the threshold: before it backlink = -1
    int first = N;
    for (int i = tid; i < N; i += nt)
        if (!(ls[i] < score_thresh)) {
            first = i;
            break;
        }
    {
        int *sh_i = reinterpret_cast<int *>(sh_d);
        first = block_reduce(first, sh_i, [](int a, int b) { return a < b ? a : b; });
    }

    // ---- DP over wavefronts of `near` independent frames, with a MONOTONE ARGMAX search.
    // score(i, loc) = cum[loc] − pen[i − loc], pen(d) = 100·ln²(d / fpb) is strictly convex for d < e·fpb, and the
    // search window ends at d = 2·fpb.  For loc2 < loc1 the exact scores satisfy
    //     score(i, loc2) + score(i+1, loc1) − score(i, loc1) − score(i+1, loc2) = Σ_{d} pen''(d) >= 15 / fpb² (> 3e-5 here),
    // an inverse-Monge gap that is five orders of magnitude above the rounding of the float64 scores (half an ulp of
    // cum, < 1e-10 for any envelope length that fits the workspace) — so the winning predecessor (maximum score, ties
    // to the nearest = largest loc, librosa's rule) of frame i+1 is never farther back than the one of frame i, for
    // the COMPUTED values too.  Hence: every S-th frame of the wavefront (and its last frame) is an anchor and gets
    // the full scan, one warp each; a frame between two anchors only scans [best(anchor before), best(anchor after)]
    // — typically a handful of candidates instead of 1.5·fpb.  Same maxima, same tie rule, same float64 values as
    // the full scan; ~5x fewer evaluations.
    constexpr int S = 8;
    int *wloc = reinterpret_cast<int *>(pen + (far - near + 1) + 1);  // best predecessor of every frame of the wavefront
    const int lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
    constexpr int L = 4;
    const int ngroups = nt / L, grp = tid / L, sub = tid % L;
    for (int basei = 0; basei < N; basei += near) {
        const int nf = min(near, N - basei);
        const int na = (nf - 1) / S + 1 + (((nf - 1) % S) ? 1 : 0);
        // phase A: anchors, one warp per anchor
        for (int a = warp; a < na; a += nwarps) {
            const int j = min(a * S, nf - 1);
            const int i = basei + j;
            const double lsi = (lane == 0) ? ls[i] : 0.0;
            double best = -INFINITY;
            int bl = -1;
            const int lo = max(0, i - far);
            for (int loc = i - near - lane; loc >= lo; loc -= 32) {  // nearest first: strict > keeps the lane's nearest maximum
                const double sc = cring[loc & rmask] - pen[i - loc - near];
                if (sc > best) {
                    best = sc;
                    bl = loc;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                const int ol = __shfl_xor_sync(0xffffffffu, bl, o);
                if (ol >= 0 && (bl < 0 || ob > best || (ob == best && ol > bl))) {
                    best = ob;
                    bl = ol;
                }
            }
            if (lane == 0) {
                const double c = (bl >= 0) ? lsi + best : lsi;
                cum[i] = c;
                cring[i & rmask] = c;  // frames of this wavefront never alias the ones being read: ring >= far + near
                backlink[i] = (i < first) ? -1 : bl;
                wloc[j] = bl;
            }
        }
        __syncthreads();
        // phase B: the frames between anchors, a group of L lanes each, over the interval the anchors leave
        const int n_between = (nf - 1) - ((nf - 1 + S - 1) / S);  // j in (0, nf−1) with j % S != 0
        const int rounds = (n_between + ngroups - 1) / ngroups;
        for (int r = 0; r < rounds; ++r) {  // warp-uniform trip count: every lane takes part in the shuffles
            const int g = r * ngroups + grp;
            const int j = (g / (S - 1)) * S + 1 + g % (S - 1);
            const bool active = g < n_between && j < nf - 1;
            const int i = basei + j;
            double best = -INFINITY;
            int bl = -1;
            const double lsi = (active && sub == 0) ? ls[i] : 0.0;
            if (active) {
                const int ja = (j / S) * S, jb = min(ja + S, nf - 1);
                const int A = wloc[ja], B = wloc[jb];
                int lo = max(0, i - far), hi = i - near;
                if (A >= 0) lo = max(lo, A);
                if (B >= 0) hi = min(hi, B);  // B < 0: the later anchor has no predecessor at all, then neither has i (hi < 0)
                for (int loc = hi - sub; loc >= lo; loc -= L) {
                    const double sc = cring[loc & rmask] - pen[i - loc - near];
                    if (sc > best) {
                        best = sc;
                        bl = loc;
                    }
                }
            }
#pragma unroll
            for (int o = L >> 1; o > 0; o >>= 1) {
                const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                const int ol = __shfl_xor_sync(0xffffffffu, bl, o);
                if (ol >= 0 && (bl < 0 || ob > best || (ob == best && ol > bl))) {
                    best = ob;
                    bl = ol;
                }
            }
            if (active && sub == 0) {
                const double c = (bl >= 0) ? lsi + best : lsi;
                cum[i] = c;
                cring[i & rmask] = c;
                backlink[i] = (i < first) ? -1 : bl;
            }
        }
        __syncthreads();
    }

    // ---- last beat: last local max of cumscore with cumscore >= ½·median(local-max scores)
    int cnt = 0;
    for (int i = tid; i < N; i += nt) cnt += is_localmax(cum, i, N) ? 1 : 0;
    {
        int *sh_i = reinterpret_cast<int *>(sh_d);
        cnt = block_reduce(cnt, sh_i, [](int a, int b) { return a + b; });
    }
    int tail = N - 1;
    if (cnt > 0) {
        const double a = select_localmax(cum, N, (cnt - 1) / 2, hist, &s_prefix, &s_rank);
        __syncthreads();
        const double b = select_localmax(cum, N, cnt / 2, hist, &s_prefix, &s_rank);
        __syncthreads();
        const double thr = 0.5 * ((a + b) / 2.0);
        int t = -1;
        for (int i = tid; i < N; i += nt)
            if (is_localmax(cum, i, N) && cum[i] >= thr) t = i;  // ascending per thread: keeps the largest
        int *sh_i = reinterpret_cast<int *>(sh_d);
        t = block_reduce(t, sh_i, [](int a, int b) { return a > b ? a : b; });
        if (t >= 0) tail = t;
    }

    // ---- backtrack (sequential pointer chase) and trim threshold
    if (tid == 0) {
        int c = 0;
        for (int n = tail; n >= 0; n = backlink[n]) tmp[c++] = n;
        s_cnt = c;
        // smooth = np.convolve(ls[beats], hanning(5))[2 : N+2];  threshold = ½·sqrt(mean(smooth²))
        const int nb = c;
        const int jend = (nb + 4 < N + 2) ? nb + 4 : N + 2;
        double ss = 0.0;
        for (int j = 2; j < jend; ++j) {
            auto x = [&](int q) -> double { return (q >= 0 && q < nb) ? ls[tmp[nb - 1 - q]] : 0.0; };
            double v = 0.5 * x(j - 1) + 1.0 * x(j - 2) + 0.5 * x(j - 3);
            ss += v * v;
        }
        const int m = jend - 2;
        s_thr = (m > 0) ? 0.5 * sqrt(ss / (double)m) : 0.0;
    }
    __syncthreads();
    const double thr = s_thr;
    int n0 = N, n1 = -1;
    for (int i = tid; i < N; i += nt)
        if (ls[i] > thr) {
            if (i < n0) n0 = i;
            n1 = i;
        }
    {
        int *sh_i = reinterpret_cast<int *>(sh_d);
        n0 = block_reduce(n0, sh_i, [](int a, int b) { return a < b ? a : b; });
        n1 = block_reduce(n1, sh_i, [](int a, int b) { return a > b ? a : b; });
    }
    if (tid == 0) {
        const int nb = s_cnt;
        int w = 0;
        bool overflow = false;
        for (int q = 0; q < nb; ++q) {
            int b = tmp[nb - 1 - q];
            if (b >= n0 && b <= n1) {
                if (w < max_beats)
                    beats_out[(size_t)seg * max_beats + w] = b;
                else
                    overflow = true;
                ++w;
            }
        }
        n_beats[seg] = overflow ? -1 : w;
    }
}

// shared-memory ring for the DP: power of two >= far + near = 2·fpb + round(fpb/2) at fpb = max_fpb
static int beat_ring(int max_fpb) {
    int r = 64;
    while (r < 2 * max_fpb + max_fpb / 2 + 2) r *= 2;
    return r;
}

static size_t beat_f64_per_seg(int max_env_len, int max_fpb) {
    return 3 * (size_t)max_env_len + 2 * (2 * (size_t)max_fpb + 1) + 8;
}

// the per-segment BeatWs regions: float64 ones of all segments, then int32 ones
struct BeatWorkspace {
    double *f64;
    int32_t *i32;
    size_t bytes;
};

static BeatWorkspace beat_ws(int n_seg, int max_env_len, int max_lag, void *base) {
    Carve c(base);
    BeatWorkspace w;
    w.f64 = c.take<double>((size_t)n_seg * beat_f64_per_seg(max_env_len, max_lag));
    w.i32 = c.take<int32_t>((size_t)n_seg * 2 * max_env_len);
    w.bytes = c.used;
    return w;
}

}  // namespace ncfa

using namespace ncfa;

extern "C" size_t ncfa_beat_workspace_bytes(int n_seg, int max_env_len, int max_lag) {
    if (n_seg <= 0 || max_env_len <= 0 || max_lag <= 0) return 0;
    return beat_ws(n_seg, max_env_len, max_lag, nullptr).bytes;
}

extern "C" int ncfa_beat_track_batched(const float *d_onset, const int64_t *d_onset_off, const int32_t *d_env_len,
                                       int n_seg, int max_env_len, const int32_t *d_lag, int max_lag,
                                       int32_t *d_beats, int max_beats, int32_t *d_n_beats, void *d_workspace,
                                       size_t workspace_bytes, void *stream) {
    NCFA_REQUIRE(n_seg >= 0, "n_seg");
    if (n_seg == 0) return NCFA_OK;
    NCFA_REQUIRE(d_onset && d_onset_off && d_env_len && d_lag && d_beats && d_n_beats && d_workspace, "null pointer");
    NCFA_REQUIRE(max_env_len > 0 && max_beats > 0 && max_lag > 0, "max_env_len/max_beats/max_lag");
    const BeatWorkspace w = beat_ws(n_seg, max_env_len, max_lag, d_workspace);
    if (int rc = check_workspace("beat", workspace_bytes, w.bytes)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    // long envelopes: measured on B200, 9.9 ms (512 threads) vs 11.1 (1024) vs 12.5 (256) per 250 pairs
    const int threads = max_env_len <= 2048 ? 64 : 512;
    const int ring = beat_ring(max_lag);
    // reduction scratch | score ring | transition penalties | best predecessor per frame of a wavefront (ints)
    const size_t smem = ((size_t)threads + ring + (3 * (size_t)max_lag / 2 + 4) + ((size_t)max_lag / 4 + 4)) * sizeof(double);
    const dim3 gs(n_seg, (max_env_len + 256 * kScoreFramesPerThread - 1) / (256 * kScoreFramesPerThread));
    NCFA_REQUIRE(gs.y <= 65535, "envelope too long for one call");
    const size_t tile_elems = (size_t)256 * kScoreFramesPerThread + 2 * (size_t)max_lag + 1;
    const size_t smem_score = (tile_elems + tile_elems / 16 + 2) * sizeof(double);
    int rc;
    if ((rc = launch("beat_prep_kernel", beat_prep_kernel, n_seg, 256, 0, st, d_onset, d_onset_off, d_env_len,
                     max_env_len, d_lag, w.f64, max_lag)))
        return rc;
    if ((rc = launch("beat_score_kernel", beat_score_kernel, gs, 256, smem_score, st, d_env_len, max_env_len, d_lag,
                     w.f64, max_lag)))
        return rc;
    return launch(max_env_len <= 2048 ? "beat_track_kernel" : "beat_track_kernel[long]", beat_track_kernel, n_seg,
                  threads, smem, st, d_onset, d_onset_off, d_env_len, max_env_len, d_lag, w.f64, w.i32, max_lag,
                  d_beats, max_beats, d_n_beats, ring);
}
