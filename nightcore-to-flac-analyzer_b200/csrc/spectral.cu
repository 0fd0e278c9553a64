// Whole-file STFT statistics.  Replaces the librosa calls of spectral.analyze (spectral.py:54-96):
// spectral_centroid, spectral_rolloff(roll_percent=0.85), the five band means of |STFT| and the per-bin mean of
// amplitude_to_db(|STFT|, ref=np.max) (top_db = 80) that the effective-bandwidth estimate is read from.
// SURVEY.md §8(f) row 3: the un-reduced STFT kernel (stft_core.cuh) with different epilogues.
//
//   spectral_pass1_kernel  grid (ctas_per_seg, n_seg), 16 warps, one warp = one frame (frames straight from global
//                          memory): |X[k]| → Σ|X|, Σ k·|X| (centroid), 85 % roll-off bin (warp scan), 5 band sums, max
//   spectral_pass2_kernel  the same transform again (cheaper than storing 4 KB per frame) → dB relative to the file
//                          maximum, clamped at −80 → per-bin sums (shared-memory float64 accumulators per CTA)
//   spectral_finish_kernel fixed-order reduction of the per-CTA partials
#include "stft_core.cuh"

namespace ncfa {

constexpr int kSpWarps = 16;
constexpr int kSpThreads = kSpWarps * 32;
constexpr int kSpSlots = 16;   // per-CTA partial record: 0 Σcentroid, 1 Σrolloff bin·hz, 2..6 band sums, 7 frames, 8 max
constexpr int kSpBins = 1025;

struct SpectralBands {
    int lo[5], hi[5];  // FFT bin ranges [lo, hi) of sub-bass, bass, midrange, presence, brilliance
};

struct SpectralSmem {
    float hann[2048];
    float2 tw[1024];
    float2 scr[kSpWarps][32 * kScrStride];
    double red[kSpWarps][kSpSlots];
    double bin_acc[kSpBins];
};

__device__ __forceinline__ void sp_stage_tables(SpectralSmem &sm, const Tables &tb, int tid) {
    for (int i = tid; i < 2048; i += kSpThreads) sm.hann[i] = tb.hann[i];
    for (int i = tid; i < 1024; i += kSpThreads) sm.tw[i] = tb.tw1024[i];
}

__global__ void __launch_bounds__(kSpThreads, 1) spectral_pass1_kernel(const float *__restrict__ audio,
                                                                       const int64_t *__restrict__ seg_off,
                                                                       const int32_t *__restrict__ seg_len,
                                                                       double hz_per_bin, SpectralBands bands, Tables tb,
                                                                       double *__restrict__ partial) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SpectralSmem &sm = *reinterpret_cast<SpectralSmem *>(smem_raw);
    const int seg = blockIdx.y;
    const int len = seg_len[seg];
    const int n_frames = 1 + len / 512;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    sp_stage_tables(sm, tb, tid);
    __syncthreads();
    const cf twl = cf{tb.tw2048[lane].x, tb.tw2048[lane].y};
    float2 *scr = sm.scr[warp];
    float *S = reinterpret_cast<float *>(scr);
    const float *src = audio + seg_off[seg];
    double a_cent = 0.0, a_roll = 0.0, a_band[5] = {0, 0, 0, 0, 0};
    float a_max = 0.0f;
    int a_frames = 0;
    for (int frame = blockIdx.x * kSpWarps + warp; frame < n_frames; frame += gridDim.x * kSpWarps) {
        warp_power_spectrum_global(src, (int64_t)frame * 512 - 1024, len, sm.hann, sm.tw, scr, twl, lane);
        // lane owns the contiguous bins [33·lane, 33·lane + 33) ∩ [0, 1025): a contiguous split makes the cumulative
        // sum of the roll-off a per-lane run plus one warp scan
        const int k0 = 33 * lane, k1 = min(kSpBins, k0 + 33);
        double s0 = 0.0, s1 = 0.0;
        float run = 0.0f, mx = 0.0f;
        for (int k = k0; k < k1; ++k) {
            const float m = sqrtf(S[k]);
            S[k] = m;
            s0 += (double)m;
            s1 += (double)k * (double)m;
            run += m;
            mx = fmaxf(mx, m);
        }
        __syncwarp();
        const double tot = warp_sum(s0), mom = warp_sum(s1);
        a_max = fmaxf(a_max, warp_max(mx));
        // librosa.util.normalize(norm=1): frames whose sum is below tiny stay unscaled → centroid Σ f·S (≈ 0)
        const double denom = (tot < 1.1754943508222875e-38) ? 1.0 : tot;
        a_cent += mom * hz_per_bin / denom;
        // roll-off: first bin whose float32 cumulative sum reaches float32(0.85·total)
        float excl = run;  // inclusive scan of the per-lane runs
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float up = __shfl_up_sync(0xffffffffu, excl, o);
            if (lane >= o) excl += up;
        }
        const float total32 = __shfl_sync(0xffffffffu, excl, 31);
        const float thr = 0.85f * total32;
        float cum = excl - run;  // sum of all bins before this lane's run
        int first = 0x7fffffff;
        for (int k = k0; k < k1; ++k) {
            cum += S[k];
            if (first == 0x7fffffff && !(cum < thr)) first = k;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
        a_roll += (double)(first == 0x7fffffff ? kSpBins - 1 : first) * hz_per_bin;
#pragma unroll
        for (int b = 0; b < 5; ++b) {
            double s = 0.0;
            for (int k = bands.lo[b] + lane; k < bands.hi[b]; k += 32) s += (double)S[k];
            a_band[b] += warp_sum(s);
        }
        ++a_frames;
        __syncwarp();
    }
    if (lane == 0) {
        sm.red[warp][0] = a_cent;
        sm.red[warp][1] = a_roll;
        for (int b = 0; b < 5; ++b) sm.red[warp][2 + b] = a_band[b];
        sm.red[warp][7] = (double)a_frames;
        sm.red[warp][8] = (double)a_max;
    }
    __syncthreads();
    if (tid < 9) {
        double v = 0.0;
        for (int w = 0; w < kSpWarps; ++w) v = (tid == 8) ? fmax(v, sm.red[w][8]) : v + sm.red[w][tid];
        partial[((size_t)seg * gridDim.x + blockIdx.x) * kSpSlots + tid] = v;
    }
}

__global__ void __launch_bounds__(kSpThreads, 1) spectral_pass2_kernel(const float *__restrict__ audio,
                                                                       const int64_t *__restrict__ seg_off,
                                                                       const int32_t *__restrict__ seg_len, Tables tb,
                                                                       const double *__restrict__ stats,
                                                                       double *__restrict__ bin_partial) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SpectralSmem &sm = *reinterpret_cast<SpectralSmem *>(smem_raw);
    const int seg = blockIdx.y;
    const int len = seg_len[seg];
    const int n_frames = 1 + len / 512;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    sp_stage_tables(sm, tb, tid);
    for (int i = tid; i < kSpBins; i += kSpThreads) sm.bin_acc[i] = 0.0;
    __syncthreads();
    const cf twl = cf{tb.tw2048[lane].x, tb.tw2048[lane].y};
    float2 *scr = sm.scr[warp];
    const float *P = reinterpret_cast<const float *>(scr);
    const float *src = audio + seg_off[seg];
    // amplitude_to_db(ref=np.max, amin=1e-5, top_db=80) in float32: 10·log10(max(amin², S²)) − 10·log10(max(amin², ref²)),
    // then max(·, max − 80); the maximum of the whole array is 0 by construction
    const float ref = (float)stats[(size_t)seg * kSpSlots + 8];
    const float ref_db = 10.0f * log10f(fmaxf(1e-10f, ref * ref));
    for (int frame = blockIdx.x * kSpWarps + warp; frame < n_frames; frame += gridDim.x * kSpWarps) {
        warp_power_spectrum_global(src, (int64_t)frame * 512 - 1024, len, sm.hann, sm.tw, scr, twl, lane);
        for (int k = lane; k < kSpBins; k += 32) {
            const float m = sqrtf(P[k]);
            const float db = fmaxf(10.0f * log10f(fmaxf(1e-10f, m * m)) - ref_db, -80.0f);
            atomicAdd(&sm.bin_acc[k], (double)db);
        }
        __syncwarp();
    }
    __syncthreads();
    for (int i = tid; i < kSpBins; i += kSpThreads)
        bin_partial[((size_t)seg * gridDim.x + blockIdx.x) * kSpBins + i] = sm.bin_acc[i];
}

// stats[seg][0..8]: Σcentroid, Σrolloff, 5 band sums, frames, max  (fixed CTA order)
__global__ void spectral_reduce1_kernel(const double *__restrict__ partial, int ctas, double *__restrict__ stats) {
    const int seg = blockIdx.x, s = threadIdx.x;
    if (s >= 9) return;
    double v = 0.0;
    for (int c = 0; c < ctas; ++c) {
        const double p = partial[((size_t)seg * ctas + c) * kSpSlots + s];
        v = (s == 8) ? fmax(v, p) : v + p;
    }
    stats[(size_t)seg * kSpSlots + s] = v;
}

__global__ void spectral_reduce2_kernel(const double *__restrict__ bin_partial, int ctas,
                                        const int32_t *__restrict__ seg_len, float *__restrict__ bin_db_mean) {
    const int seg = blockIdx.y;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= kSpBins) return;
    double v = 0.0;
    for (int c = 0; c < ctas; ++c) v += bin_partial[((size_t)seg * ctas + c) * kSpBins + k];
    bin_db_mean[(size_t)seg * kSpBins + k] = (float)(v / (double)(1 + seg_len[seg] / 512));
}

}  // namespace ncfa

using namespace ncfa;

static int spectral_ctas(int n_seg) {
    int n_sm = 148;
    (void)sm_count(&n_sm);
    int c = (n_sm + n_seg - 1) / n_seg;
    return c < 1 ? 1 : c;
}

// per segment `ctas` CTAs, each with kSpSlots pass-1 partial sums and kSpBins pass-2 per-bin partial sums
struct SpectralWs {
    int ctas;
    double *partial, *bin_partial;
    size_t bytes;
};

static SpectralWs spectral_ws(int n_seg, void *base) {
    Carve c(base);
    SpectralWs w;
    w.ctas = spectral_ctas(n_seg);
    w.partial = c.take<double>((size_t)n_seg * w.ctas * kSpSlots);
    w.bin_partial = c.take<double>((size_t)n_seg * w.ctas * kSpBins);
    w.bytes = c.used;
    return w;
}

extern "C" size_t ncfa_spectral_workspace_bytes(int n_seg) {
    if (n_seg <= 0) return 0;
    return spectral_ws(n_seg, nullptr).bytes;
}

extern "C" int ncfa_spectral_stats_batched(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len,
                                           int n_seg, int sr, double *d_stats, float *d_bin_db_mean, void *d_workspace,
                                           size_t workspace_bytes, void *stream) {
    NCFA_REQUIRE(n_seg >= 0 && n_seg <= 65535, "n_seg must be in [0, 65535] per call");
    if (n_seg == 0) return NCFA_OK;
    NCFA_REQUIRE(d_audio && d_seg_off && d_seg_len && d_stats && d_bin_db_mean && d_workspace, "null pointer");
    NCFA_REQUIRE(sr > 0, "sr");
    const SpectralWs w = spectral_ws(n_seg, d_workspace);
    int rc = check_workspace("spectral", workspace_bytes, w.bytes);
    if (rc) return rc;
    Tables tb;
    if ((rc = get_tables(sr, &tb))) return rc;
    // band masks of spectral.py:70-78: (freqs >= lo) & (freqs < hi) with freqs = k · (1 / (n_fft · (1/sr)))
    const double val = 1.0 / (2048.0 * (1.0 / (double)sr));
    const double edges[5][2] = {{20, 80}, {80, 250}, {250, 2000}, {2000, 6000}, {6000, 20000}};
    SpectralBands bands;
    for (int b = 0; b < 5; ++b) {
        int lo = 0, hi = 0;
        while (lo < kSpBins && !((double)lo * val >= edges[b][0])) ++lo;
        hi = lo;
        while (hi < kSpBins && (double)hi * val < edges[b][1]) ++hi;
        bands.lo[b] = lo;
        bands.hi[b] = hi;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 g(w.ctas, n_seg);
    if ((rc = launch("spectral_pass1_kernel", spectral_pass1_kernel, g, kSpThreads, sizeof(SpectralSmem), st, d_audio,
                     d_seg_off, d_seg_len, (double)sr / 2048.0, bands, tb, w.partial)))
        return rc;
    if ((rc = launch("spectral_reduce1_kernel", spectral_reduce1_kernel, n_seg, 32, 0, st, w.partial, w.ctas, d_stats)))
        return rc;
    if ((rc = launch("spectral_pass2_kernel", spectral_pass2_kernel, g, kSpThreads, sizeof(SpectralSmem), st, d_audio,
                     d_seg_off, d_seg_len, tb, d_stats, w.bin_partial)))
        return rc;
    return launch("spectral_reduce2_kernel", spectral_reduce2_kernel, dim3((kSpBins + 255) / 256, n_seg), 256, 0, st,
                  w.bin_partial, w.ctas, d_seg_len, d_bin_db_mean);
}
