// CQT chroma family.  Replaces librosa.feature.chroma_cqt(y, sr, bins_per_octave=36, hop_length=512)
// followed by .mean(axis=1) as called by pitch._mean_chroma (pitch.py:55-64), and the 12-lag cyclic
// cross-correlation of pitch._cyclic_xcorr_peak (pitch.py:67-85).  SURVEY.md §3.4, Appendix A.8.
//
//   tuning_peaks_kernel   STFT(2048, 512, Hann) magnitude → piptrack peaks (parabolic interpolation)
//                         in 150..4000 Hz → (magnitude, 1/36-octave residual histogram bin) per peak
//   tuning_pick_kernel    median magnitude over the segment (radix select) → histogram of the peaks at
//                         or above it → first fullest bin = tuning index j, tuning = −0.5 + j/100
//   decimate2_kernel      2:1 decimation ×√2 between octaves (127-tap Kaiser half-band, float64 sums)
//   cqt_tc_kernel         per octave: the 36 CQT responses of every frame as ONE real contraction on the tensor
//                         cores, C[72 × frames] = K[72 × 1024] · X[1024 × frames],  X[n][t] = y_oct[t·hop_oct + n − 512]
//                         (K = sparsified FFT-domain basis ∘ DFT, folded on the host in float64 — the same
//                         linear map as rectangular-window STFT followed by the sparse basis product),
//                         then |·|, fold 252 → 12 chroma, inf-norm per frame, partial sums over frames
//   chroma_mean_kernel    partial sums → mean chroma float64[12] per segment
//   cyclic_xcorr_kernel   argmax_k dot(src, roll(nc, −k)) wrapped to (−n/2, n/2]
#include <cmath>
#include <cstring>
#include <algorithm>
#include <complex>
#include <map>
#include <mutex>
#include <vector>
#include "stft_core.cuh"
#include "tc05.cuh"

namespace ncfa {

constexpr int kNTunings = 100;
constexpr int kCqtBins = 36;          // bins per octave
constexpr int kCqtRows = 2 * kCqtBins;  // real + imaginary rows of K
constexpr int kCqtNfft = 1024;
constexpr int kOctaves = 7;
constexpr int kChroma = 12;
constexpr int kHbTaps = 127;
constexpr int kPeakStride = 180;  // ≥ max local maxima among the 358 candidate bins (179)

struct ChromaTables {
    const double *hb;   // [127] half-band taps
    // [100][32 k-tiles][hi, lo][80 rows × 32 k] tf32 split of K as swizzle-128B shared-memory images, where
    // K[j][n][r] (tuning j, [100][1024][72]): r < 36 real part of bin r, r ≥ 36 imaginary part of bin r−36
    const float *Bimg;
};

constexpr int kTcN = 80;                          // MMA N: 72 rows of K + 8 zero rows (N % 16 == 0 for M = 128)
constexpr int kTcKT = 32;                         // k (time-sample) tile = one 128-byte swizzle row of tf32
constexpr int kTcBTileBytes = kTcN * kTcKT * 4;   // 10240: one of {hi, lo}
constexpr int kTcBStageBytes = 2 * kTcBTileBytes; // hi then lo

static float host_tf32_rna(float x) {  // cvt.rna.tf32.f32: nearest, ties away from zero, low 13 mantissa bits cleared
    uint32_t u;
    memcpy(&u, &x, 4);
    u = (u + 0x1000u) & ~0x1FFFu;
    float r;
    memcpy(&r, &u, 4);
    return r;
}

// K[1024][72] of one tuning → 32 stage images; element (row r, k c) of a tile lives at
// (r/8)·1024 + (r%8)·128 + ((c/4) ^ (r%8))·16 + (c%4)·4   (Swizzle<3,4,3> on a 1024-byte aligned tile)
static void build_b_image(const float *K, float *img /* [32][2][80*32] */) {
    for (int kt = 0; kt < kCqtNfft / kTcKT; ++kt)
        for (int r = 0; r < kTcN; ++r)
            for (int c = 0; c < kTcKT; ++c) {
                const float x = r < kCqtRows ? K[(size_t)(kt * kTcKT + c) * kCqtRows + r] : 0.0f;
                const float hi = host_tf32_rna(x), lo = x - hi;
                const size_t off = ((size_t)(r >> 3) * 1024 + (size_t)(r & 7) * 128 + (size_t)(((c >> 2) ^ (r & 7)) * 16) +
                                    (size_t)(c & 3) * 4) / 4;
                img[((size_t)kt * 2 + 0) * (kTcN * kTcKT) + off] = hi;
                img[((size_t)kt * 2 + 1) * (kTcN * kTcKT) + off] = lo;
            }
}

// ------------------------------------------------------------------------------------------------ host tables
static void fft_inplace(std::vector<std::complex<double>> &a) {
    const size_t n = a.size();
    for (size_t i = 1, j = 0; i < n; ++i) {
        size_t bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) std::swap(a[i], a[j]);
    }
    const double PI = 3.14159265358979323846;
    for (size_t len = 2; len <= n; len <<= 1) {
        const double ang = -2.0 * PI / (double)len;
        for (size_t i = 0; i < n; i += len)
            for (size_t k = 0; k < len / 2; ++k) {
                const std::complex<double> w(cos(ang * (double)k), sin(ang * (double)k));
                const std::complex<double> u = a[i + k], v = a[i + k + len / 2] * w;
                a[i + k] = u + v;
                a[i + k + len / 2] = u - v;
            }
    }
}

// librosa.filters.wavelet + __vqt_filter_fft + util.sparsify_rows for the top octave at the full rate
// (Appendix A.8), then folded with the DFT and the final 1/sqrt(length) scale:  K[n][r]
static int build_cqt_matrix(int sr, double tuning, std::vector<float> &K /* [1024][72] */) {
    const double PI = 3.14159265358979323846;
    const double c1 = 440.0 * pow(2.0, (12.0 * 2.0 + 0.0 - 69.0) / 12.0);
    const double fmin = c1 * pow(2.0, tuning / 36.0);
    const double r = pow(2.0, 1.0 / 36.0);
    const double alpha = (r * r - 1.0) / (r * r + 1.0);
    const double Q = 1.0 / alpha;
    const int n_bins = kOctaves * kCqtBins;
    std::vector<std::complex<double>> tw(kCqtNfft);
    for (int i = 0; i < kCqtNfft; ++i) tw[i] = std::complex<double>(cos(-2.0 * PI * i / kCqtNfft), sin(-2.0 * PI * i / kCqtNfft));
    K.assign((size_t)kCqtNfft * kCqtRows, 0.0f);
    for (int b = 0; b < kCqtBins; ++b) {
        const int k = n_bins - kCqtBins + b;
        const double freq = fmin * pow(2.0, (double)k / 36.0);
        const double ilen = Q * (double)sr / freq;
        const long t0 = (long)floor(-ilen / 2.0), t1 = (long)floor(ilen / 2.0);
        const int N = (int)(t1 - t0);
        if (N < 2 || N > kCqtNfft) {
            set_error("CQT filter length %d does not fit n_fft=1024 at sr=%d", N, sr);
            return NCFA_E_INVALID;
        }
        std::vector<std::complex<double>> sig(N);
        double l1 = 0.0;
        for (int i = 0; i < N; ++i) {
            const double t = (double)(t0 + i);
            const double ph = t * 2.0 * PI * freq / (double)sr;
            const double w = 0.5 - 0.5 * cos(2.0 * PI * (double)i / (double)N);
            sig[i] = std::complex<double>(cos(ph), sin(ph)) * w;
            l1 += std::abs(sig[i]);
        }
        std::vector<std::complex<double>> buf(kCqtNfft, std::complex<double>(0.0, 0.0));
        const int lpad = (kCqtNfft - N) / 2;
        for (int i = 0; i < N; ++i) buf[lpad + i] = sig[i] / l1 * (ilen / (double)kCqtNfft);
        fft_inplace(buf);
        // sparsify_rows(quantile=0.01) over the 513 kept bins
        const int nb = kCqtNfft / 2 + 1;
        std::vector<double> mags(nb), sorted;
        double norm = 0.0;
        for (int i = 0; i < nb; ++i) {
            mags[i] = std::abs(buf[i]);
            norm += mags[i];
        }
        sorted = mags;
        std::sort(sorted.begin(), sorted.end());
        double cum = 0.0, thr = sorted[0];
        for (int i = 0; i < nb; ++i) {
            cum += sorted[i] / norm;
            if (!(cum < 0.01)) {
                thr = sorted[i];
                break;
            }
        }
        const double scale = 1.0 / sqrt(ilen);  // V /= sqrt(lengths): identical in every octave (length·2^oct vs sqrt(2^oct)·√2 chain)
        std::vector<double> kre(kCqtNfft, 0.0), kim(kCqtNfft, 0.0);
        for (int i = 0; i < nb; ++i) {
            if (!(mags[i] >= thr)) continue;
            const std::complex<double> c((double)(float)buf[i].real(), (double)(float)buf[i].imag());  // complex64 basis
            for (int n = 0; n < kCqtNfft; ++n) {
                const std::complex<double> v = c * tw[(i * n) & (kCqtNfft - 1)];
                kre[n] += v.real();
                kim[n] += v.imag();
            }
        }
        for (int n = 0; n < kCqtNfft; ++n) {
            K[(size_t)n * kCqtRows + b] = (float)(kre[n] * scale);
            K[(size_t)n * kCqtRows + kCqtBins + b] = (float)(kim[n] * scale);
        }
    }
    return NCFA_OK;
}

static double bessel_i0(double x) {  // power series, converges fast for x ≤ ~20
    const double q = x * x / 4.0;
    double term = 1.0, sum = 1.0;
    for (int k = 1; k < 200; ++k) {
        term *= q / ((double)k * (double)k);
        sum += term;
        if (term < 1e-18 * sum) break;
    }
    return sum;
}

static void build_halfband(std::vector<double> &h) {
    // Kaiser(127, β=10)-windowed sinc half-band, DC gain 1 (the 2:1 decimator between CQT octaves; librosa
    // uses soxr_hq there, which is not reproducible — documented deviation, DESIGN.md)
    const double PI = 3.14159265358979323846;
    h.assign(kHbTaps, 0.0);
    double hs = 0.0;
    const double al = (kHbTaps - 1) / 2.0, i0b = bessel_i0(10.0);
    for (int i = 0; i < kHbTaps; ++i) {
        const double n = (double)i - al;
        double x = 0.5 * n;
        if (x == 0.0) x = 1e-20;
        const double sinc = sin(PI * x) / (PI * x);
        const double rr = n / al;
        const double kw = bessel_i0(10.0 * sqrt(fmax(0.0, 1.0 - rr * rr))) / i0b;
        h[i] = 0.5 * sinc * kw;
        hs += h[i];
    }
    for (auto &v : h) v /= hs;
}

// the 64 even taps and the centre tap of the half-band filter also live in constant memory: the decimator's FMAs take
// them as constant-bank operands (no shared-memory load per tap)
__constant__ double c_hb_even[64];
__constant__ double c_hb_mid;

static std::mutex g_hb_mu;
static std::map<int, const double *> g_hb;
int get_halfband_device(const double **out) {
    int dev = 0;
    NCFA_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_hb_mu);
    auto it = g_hb.find(dev);
    if (it != g_hb.end()) {
        *out = it->second;
        return NCFA_OK;
    }
    std::vector<double> h;
    build_halfband(h);
    double *dh = nullptr;
    NCFA_CUDA_OK(cudaMalloc(&dh, h.size() * sizeof(double)));
    NCFA_CUDA_OK(cudaMemcpy(dh, h.data(), h.size() * sizeof(double), cudaMemcpyHostToDevice));
    {
        double ev[64];
        for (int m = 0; m < 64; ++m) ev[m] = h[2 * m];
        const double mid = h[(kHbTaps - 1) / 2];
        NCFA_CUDA_OK(cudaMemcpyToSymbol(c_hb_even, ev, sizeof(ev)));
        NCFA_CUDA_OK(cudaMemcpyToSymbol(c_hb_mid, &mid, sizeof(mid)));
    }
    g_hb[dev] = dh;
    *out = dh;
    return NCFA_OK;
}

static std::mutex g_chroma_mu;
static std::map<std::pair<int, int>, ChromaTables> g_chroma_tables;

static int get_chroma_tables(int sr, ChromaTables *out) {
    int dev = 0;
    NCFA_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_chroma_mu);
    auto key = std::make_pair(dev, sr);
    auto it = g_chroma_tables.find(key);
    if (it != g_chroma_tables.end()) {
        *out = it->second;
        return NCFA_OK;
    }
    std::vector<float> all((size_t)kNTunings * kCqtNfft * kCqtRows), one;
    for (int j = 0; j < kNTunings; ++j) {
        const double tuning = (double)j * 0.01 + (-0.5);  // np.linspace(-0.5, 0.5, 101)[j]
        int rc = build_cqt_matrix(sr, tuning, one);
        if (rc) return rc;
        memcpy(all.data() + (size_t)j * kCqtNfft * kCqtRows, one.data(), one.size() * sizeof(float));
    }
    ChromaTables t;
    {
        int rc = get_halfband_device(&t.hb);
        if (rc) return rc;
    }
    {
        const size_t per = (size_t)(kCqtNfft / kTcKT) * 2 * kTcN * kTcKT;
        std::vector<float> img((size_t)kNTunings * per);
        for (int j = 0; j < kNTunings; ++j)
            build_b_image(all.data() + (size_t)j * kCqtNfft * kCqtRows, img.data() + (size_t)j * per);
        float *dB = nullptr;
        NCFA_CUDA_OK(cudaMalloc(&dB, img.size() * sizeof(float)));
        NCFA_CUDA_OK(cudaMemcpy(dB, img.data(), img.size() * sizeof(float), cudaMemcpyHostToDevice));
        t.Bimg = dB;
    }
    g_chroma_tables[key] = t;
    *out = t;
    return NCFA_OK;
}

// ------------------------------------------------------------------------------------------------ geometry
// octave o works on level o of the decimation pyramid: len_0 = n, len_o = ceil(len_{o-1}/2), hop_o = 512 >> o
__host__ __device__ inline int level_len(int n, int o) {
    for (int i = 0; i < o; ++i) n = (n + 1) >> 1;
    return n;
}
__host__ __device__ inline int cqt_frames(int n) {  // cqt trims every octave to the shortest (max_col)
    int f = 0x7fffffff;
    for (int o = 0; o < kOctaves; ++o) {
        const int fo = 1 + level_len(n, o) / (512 >> o);
        f = fo < f ? fo : f;
    }
    return f;
}
// float offsets of pyramid levels 1..6 of one segment (each 4-aligned), total in off[7]
__host__ __device__ inline void pyramid_layout(int max_len, size_t off[kOctaves + 1]) {
    size_t p = 0;
    off[0] = 0;
    for (int o = 1; o < kOctaves; ++o) {
        off[o] = p;
        p += ((size_t)level_len(max_len, o) + 3) / 4 * 4;
    }
    off[kOctaves] = p;
}

// ------------------------------------------------------------------------------------------------ tuning
constexpr int kTunWarps = 20;
constexpr int kTunThreads = kTunWarps * 32;

struct TuningSmem {
    float hann[2048];
    float2 tw[1024];
    float2 scr[kTunWarps][32 * kScrStride];
};

// persistent CTAs (one per SM), one warp per frame, frames read straight from global memory (see stft_onset.cu)
__global__ void __launch_bounds__(kTunThreads, 1) tuning_peaks_kernel(const float *__restrict__ audio,
                                                                      const int64_t *__restrict__ seg_off,
                                                                      const int32_t *__restrict__ seg_len, int n_seg,
                                                                      int frame_stride, int kmin, int kmax,
                                                                      double hz_per_bin, Tables tb,
                                                                      float *__restrict__ pk_mag,
                                                                      uint8_t *__restrict__ pk_bin,
                                                                      int32_t *__restrict__ pk_cnt) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    TuningSmem &sm = *reinterpret_cast<TuningSmem *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < 2048; i += kTunThreads) sm.hann[i] = tb.hann[i];
    for (int i = tid; i < 1024; i += kTunThreads) sm.tw[i] = tb.tw1024[i];
    __syncthreads();
    const cf twl = cf{tb.tw2048[lane].x, tb.tw2048[lane].y};
    float2 *scr = sm.scr[warp];
    float *S = reinterpret_cast<float *>(scr);
    const int64_t total = (int64_t)n_seg * frame_stride;
    for (int64_t item = (int64_t)blockIdx.x * kTunWarps + warp; item < total; item += (int64_t)gridDim.x * kTunWarps) {
        const int seg = (int)(item / frame_stride);
        const int frame = (int)(item - (int64_t)seg * frame_stride);
        const int len = seg_len[seg];
        if (frame >= 1 + len / 512) continue;
        warp_power_spectrum_global(audio + seg_off[seg], (int64_t)frame * 512 - 1024, len, sm.hann, sm.tw, scr, twl, lane);
        float mx = 0.0f;
        for (int k = lane; k < 1025; k += 32) {
            const float m = sqrtf(S[k]);
            S[k] = m;
            mx = fmaxf(mx, m);
        }
        mx = warp_max(mx);
        __syncwarp();
        const float ref = 0.1f * mx;  // threshold · max over the frame
        const size_t slot0 = ((size_t)seg * frame_stride + frame) * kPeakStride;
        int count = 0;
        for (int kb = kmin; kb <= kmax; kb += 32) {
            const int k = kb + lane;
            bool peak = false;
            float mag = 0.0f;
            int hbin = 0;
            if (k <= kmax) {
                const float sl = S[k - 1], sc = S[k], sr_ = S[k + 1];
                const float ml = sl > ref ? sl : 0.0f, mc = sc > ref ? sc : 0.0f, mr = sr_ > ref ? sr_ : 0.0f;
                peak = (mc > ml) && (mc >= mr);
                if (peak) {
                    const float a = __fsub_rn(__fadd_rn(sr_, sl), __fmul_rn(2.0f, sc));
                    const float b = __fmul_rn(__fsub_rn(sr_, sl), 0.5f);
                    const float shift = (fabsf(b) >= fabsf(a)) ? 0.0f : __fdiv_rn(-b, a);
                    mag = __fadd_rn(sc, __fmul_rn(__fmul_rn(0.5f, b), shift));
                    // residual of 36·log2(f/27.5) mod 1 → one of 100 histogram bins.  Fast path in float32 (position error
                    // < 4e-3 of a bin); anything within 2 % of a bin edge takes the exact float64 path below.
                    const float r32 = 36.0f * __log2f(((float)k + shift) * (float)(hz_per_bin / 27.5));
                    const float fr = r32 - floorf(r32);
                    const float pos = (fr < 0.5f ? fr + 0.5f : fr - 0.5f) * 100.0f;
                    int i0 = (int)pos;
                    const float dpos = pos - (float)i0;
                    if (!(dpos > 0.02f && dpos < 0.98f && i0 >= 0 && i0 <= 99)) {
                        const double pitch = __dmul_rn(__dadd_rn((double)k, (double)shift), hz_per_bin);
                        double res = fmod(__dmul_rn(36.0, log2(pitch / 27.5)), 1.0);
                        if (res >= 0.5) res = __dadd_rn(res, -1.0);
                        i0 = (int)floor((res + 0.5) * 100.0);
                        i0 = i0 < 0 ? 0 : (i0 > 99 ? 99 : i0);
                        // bin i holds edge(i) <= x < edge(i+1), edge(i) = i·0.01 − 0.5 as np.linspace computes it
                        while (i0 > 0 && res < __dadd_rn(__dmul_rn((double)i0, 0.01), -0.5)) --i0;
                        while (i0 < 99 && res >= __dadd_rn(__dmul_rn((double)(i0 + 1), 0.01), -0.5)) ++i0;
                    }
                    hbin = i0;
                }
            }
            const unsigned m = __ballot_sync(0xffffffffu, peak);
            if (peak) {
                const int slot = count + __popc(m & ((1u << lane) - 1u));
                pk_mag[slot0 + slot] = mag;
                pk_bin[slot0 + slot] = (uint8_t)hbin;
            }
            count += __popc(m);
        }
        if (lane == 0) pk_cnt[(size_t)seg * frame_stride + frame] = count;
        __syncwarp();
    }
}

// median(mag) over all peaks of the segment, histogram of residual bins of peaks with mag >= median
__global__ void __launch_bounds__(256) tuning_pick_kernel(const int32_t *__restrict__ seg_len, int frame_stride,
                                                          const float *__restrict__ pk_mag,
                                                          const uint8_t *__restrict__ pk_bin,
                                                          const int32_t *__restrict__ pk_cnt,
                                                          int32_t *__restrict__ tuning_idx) {
    __shared__ int hist[256];
    __shared__ unsigned s_prefix;
    __shared__ int s_rank, s_total;
    __shared__ float s_sel[2];
    const int seg = blockIdx.x;
    const int n_frames = 1 + seg_len[seg] / 512;
    const int tid = threadIdx.x;
    const int32_t *cnt = pk_cnt + (size_t)seg * frame_stride;
    const float *mags = pk_mag + (size_t)seg * frame_stride * kPeakStride;
    const uint8_t *bins = pk_bin + (size_t)seg * frame_stride * kPeakStride;
    if (tid == 0) s_total = 0;
    __syncthreads();
    int local = 0;
    for (int f = tid; f < n_frames; f += 256) local += cnt[f];
    atomicAdd(&s_total, local);
    __syncthreads();
    const int total = s_total;
    if (total == 0) {
        if (tid == 0) tuning_idx[seg] = 50;  // pitch_tuning: no pitches → 0.0 = edge 50
        return;
    }
    // one warp walks one frame's slots at a time
    const int warp = tid >> 5, lane = tid & 31;
    for (int which = 0; which < 2; ++which) {
        if (tid == 0) {
            s_prefix = 0u;
            s_rank = which == 0 ? (total - 1) / 2 : total / 2;
        }
        __syncthreads();
        for (int shift = 24; shift >= 0; shift -= 8) {
            hist[tid] = 0;
            __syncthreads();
            const unsigned prefix = s_prefix;
            const unsigned himask = (shift == 24) ? 0u : (~0u << (shift + 8));
            for (int f = warp; f < n_frames; f += 8) {
                const int c = cnt[f];
                for (int e = lane; e < c; e += 32) {
                    const unsigned key = float_to_ordered(mags[(size_t)f * kPeakStride + e]);
                    if ((key & himask) == prefix) atomicAdd(&hist[(key >> shift) & 0xff], 1);
                }
            }
            __syncthreads();
            if (tid == 0) {
                int r = s_rank, b = 0;
                while (b < 255 && r >= hist[b]) {
                    r -= hist[b];
                    ++b;
                }
                s_rank = r;
                s_prefix = prefix | ((unsigned)b << shift);
            }
            __syncthreads();
        }
        if (tid == 0) s_sel[which] = ordered_to_float(s_prefix);
        __syncthreads();
    }
    const float thr = __fmul_rn(__fadd_rn(s_sel[0], s_sel[1]), 0.5f);  // np.median of float32
    hist[tid] = 0;
    __syncthreads();
    for (int f = warp; f < n_frames; f += 8) {
        const int c = cnt[f];
        for (int e = lane; e < c; e += 32)
            if (mags[(size_t)f * kPeakStride + e] >= thr) atomicAdd(&hist[bins[(size_t)f * kPeakStride + e]], 1);
    }
    __syncthreads();
    if (tid == 0) {
        int best = 0;
        for (int i = 1; i < kNTunings; ++i)
            if (hist[i] > hist[best]) best = i;  // np.argmax: first maximum
        tuning_idx[seg] = best;
    }
}

// ------------------------------------------------------------------------------------------------ decimation
// out[t] = float32( √2 · Σ_k h[k]·in[2t + k − 63] ),  n_out = ceil(n_in / 2).
// Half-band structure: besides the centre tap only the even-indexed taps are non-zero (the others are sin(mπ)
// rounding residue below 1e-17 and are skipped), and they all hit ODD input samples:
//     out[t] = h[63]·xe[t] + Σ_{m<64} h[2m]·xo[t + m − 32],   xe[j] = in[2j], xo[j] = in[2j+1].
// A CTA de-interleaves its input span into xe / xo in shared memory; each thread produces 4 consecutive outputs
// from a 67-sample register window (17 conflict-free LDS.128), float64 accumulation.
// Accumulation type: float64 like the oracle.  A float32 variant was measured: 10.6 -> 8.3 ms per
// 250 pairs only — the kernel is paced by its strided staging loads, not by the FP64 pipe — so the exact sums stay.
// ncu (profiles/r2f_ncu_summary.md, 4 outputs per thread): XU pipe 61 % — the float → double conversions of the register
// window, 17.75 per output — next to FP64 54 %.  Eight outputs per thread share a 71-sample window: 9.9 conversions per
// output, and the kernel is left with its 64 float64 FMAs per output.
constexpr int kDecPerThread = 8;
constexpr int kDecOutPerCta = 256 * kDecPerThread;
__global__ void __launch_bounds__(256) decimate2_kernel(const float *__restrict__ audio,
                                                        const int64_t *__restrict__ seg_off,
                                                        const int32_t *__restrict__ seg_len, int level,
                                                        float *__restrict__ pyr, size_t pyr_stride, size_t in_off,
                                                        size_t out_off, const double *__restrict__ hb) {
    __shared__ __align__(16) float xo[kDecOutPerCta + 64 + 8];
    __shared__ __align__(16) float xe[kDecOutPerCta];
    const int seg = blockIdx.y;
    const int n0 = seg_len[seg];
    const int n_in = level_len(n0, level - 1), n_out = (n_in + 1) >> 1;
    const int o0 = blockIdx.x * kDecOutPerCta;
    if (o0 >= n_out) return;
    const float *in = (level == 1) ? audio + seg_off[seg] : pyr + (size_t)seg * pyr_stride + in_off;
    float *out = pyr + (size_t)seg * pyr_stride + out_off;
    // xo[i] = in[2(o0 − 32 + i) + 1], i < kDecOutPerCta + 64 + 8;  xe[i] = in[2(o0 + i)], i < kDecOutPerCta: one coalesced
    // float2 load (even sample, odd sample) feeds both arrays when the level's base is 8-byte aligned
    if ((reinterpret_cast<uintptr_t>(in) & 7u) == 0) {
        for (int i = threadIdx.x; i < kDecOutPerCta + 64 + 8; i += 256) {
            const int64_t p = 2 * ((int64_t)o0 - 32 + i);
            float2 v = make_float2(0.0f, 0.0f);
            if (p >= 0 && p + 1 < n_in) v = __ldg(reinterpret_cast<const float2 *>(in + p));
            else if (p >= 0 && p < n_in) v.x = __ldg(in + p);
            xo[i] = v.y;
            if (i >= 32 && i < 32 + kDecOutPerCta) xe[i - 32] = v.x;
        }
    } else {
        for (int i = threadIdx.x; i < kDecOutPerCta + 64 + 8; i += 256) {
            const int64_t p = 2 * ((int64_t)o0 - 32 + i) + 1;
            xo[i] = (p >= 0 && p < n_in) ? __ldg(in + p) : 0.0f;
        }
        for (int i = threadIdx.x; i < kDecOutPerCta; i += 256) {
            const int64_t p = 2 * ((int64_t)o0 + i);
            xe[i] = (p < n_in) ? __ldg(in + p) : 0.0f;
        }
    }
    __syncthreads();
    const int t = kDecPerThread * threadIdx.x;  // outputs o0 + t .. o0 + t + 7 use xo[t .. t + 70]
    double w[72];
#pragma unroll
    for (int j = 0; j < 18; ++j) {
        const float4 v = *reinterpret_cast<const float4 *>(xo + t + 4 * j);
        w[4 * j] = (double)v.x;
        w[4 * j + 1] = (double)v.y;
        w[4 * j + 2] = (double)v.z;
        w[4 * j + 3] = (double)v.w;
    }
    double a[kDecPerThread];
    {
        const float4 e0 = *reinterpret_cast<const float4 *>(xe + t);
        const float4 e1 = *reinterpret_cast<const float4 *>(xe + t + 4);
        const double hm = c_hb_mid;
        a[0] = hm * (double)e0.x, a[1] = hm * (double)e0.y, a[2] = hm * (double)e0.z, a[3] = hm * (double)e0.w;
        a[4] = hm * (double)e1.x, a[5] = hm * (double)e1.y, a[6] = hm * (double)e1.z, a[7] = hm * (double)e1.w;
    }
#pragma unroll
    for (int m = 0; m < 64; ++m) {  // ascending m per output, as before: the sums round identically
        const double hm = c_hb_even[m];  // compile-time index: a constant-bank operand of the FMAs
#pragma unroll
        for (int u = 0; u < kDecPerThread; ++u) a[u] = fma(hm, w[m + u], a[u]);
    }
    const double r2 = 1.4142135623730951;
    const int o = o0 + t;
    if (o + kDecPerThread - 1 < n_out && (reinterpret_cast<uintptr_t>(out + o) & 15u) == 0) {  // level offsets: multiples of 4 floats
        *reinterpret_cast<float4 *>(out + o) =
            make_float4((float)(a[0] * r2), (float)(a[1] * r2), (float)(a[2] * r2), (float)(a[3] * r2));
        *reinterpret_cast<float4 *>(out + o + 4) =
            make_float4((float)(a[4] * r2), (float)(a[5] * r2), (float)(a[6] * r2), (float)(a[7] * r2));
    } else {
#pragma unroll
        for (int u = 0; u < kDecPerThread; ++u)
            if (o + u < n_out) out[o + u] = (float)(a[u] * r2);
    }
}

// ------------------------------------------------------------------------------------------------ CQT → chroma
constexpr int kPartialTF = 32;  // frames per tile of the partial[] stride (the workspace is sized in 32-frame tiles)

// |re + i·im| as np.abs(complex64) gives it (hypot): re² + im² underflows in float32 below ~1e-19, and a frame whose only
// content is that small (the tail of a decayed note reaching the lowest octave of an otherwise digitally silent stretch)
// is scaled up to 1 by the per-frame inf-norm — so tiny responses are squared after an exact rescale by 2^96.
__device__ __forceinline__ float cabs_f32(float re, float im) {
    const float a = fabsf(re), b = fabsf(im);
    if (fmaxf(a, b) >= 0x1p-60f) return sqrtf(a * a + b * b);
    const float as = a * 0x1p96f, bs = b * 0x1p96f;
    return sqrtf(as * as + bs * bs) * 0x1p-96f;
}

struct PyrOffsets {
    size_t off[kOctaves + 1];  // float offset of level o (1..6) inside a segment's pyramid; off[7] = stride
};

// ------------------------------------------------------------------------------------------------ CQT on tcgen05
// The contraction on the 5th-generation tensor cores:  D[128 frames × 80] (+)= A[128 × 8]·B[80 × 8]^T, kind::tf32,
// with the 3×TF32 split  x = hi + lo  (hi = x truncated to tf32, lo = x − hi exactly):  A·B ≈ Ah·Bh + Al·Bh + Ah·Bl.
//   A (the Hankel matrix of frames) is never materialised in memory: the frame warps stage the rows of a k-tile in shared
//     memory with coalesced cp.async copies (64 contiguous bytes of eight rows per instruction; L1/L2 serve the overlap
//     between frames), every frame thread then reads its own row piece, splits it in registers and writes hi / lo into
//     TENSOR MEMORY with tcgen05.st; the MMA reads A from TMEM (TS form).
//   B (the folded CQT matrix) is pre-split and pre-swizzled on the host as shared-memory images, so a k-tile is ONE
//     20 KB 1-D bulk async copy (cp.async.bulk + mbarrier complete_tx) — no tensor map needed.
//   D lives in TMEM; the epilogue is tcgen05.ld → |re + i·im| → fold to 12 chroma.
// Warp roles (320 threads): warps 0-7 frame warps (A producer + epilogue; warp w serves rows 32·(w & 3) … +31 — its TMEM
// lane quarter — and column half q = w >> 2 of every k-tile), warp 8 MMA issuer and TMEM allocator, warp 9 B loader.
// Pipeline shape: TWO CTAs per SM, each with a shallow pipeline (2 A stages in TMEM, 2 B images in shared memory, one
// accumulator, 256 TMEM columns, 100 KB of shared memory).  Timing experiments (profiles/r2l_cqt_debug.log) showed that
// with A traffic, B traffic AND the MMAs all switched off, a deep one-CTA-per-SM pipeline (5 stages, two accumulators,
// 512 TMEM columns) still took 12.3 of its 13.4 ms: what paces the kernel is the latency of one CTA's serial producer →
// MMA → release chain, with two or three warps per scheduler to hide it.  A second resident CTA overlaps two such chains
// on the same tensor pipe: 13.4 -> 9.8 ms per 1750 chunks on B200 (profiles/r2m).  (A k-tile-major variant that fetched
// every B image once per four octaves — 3.5x less bulk-copy traffic — measured exactly the same 13.4 ms as the
// octave-major order and was dropped: B traffic is not the limiter either.)
constexpr int kTcFrames = 128;
constexpr int kTcQ = 2;                                  // column splits of a k-tile row (threads per frame row)
constexpr int kTcVals = kTcKT / kTcQ;                    // samples per thread per k-tile (16)
constexpr int kTcFrameWarps = 4 * kTcQ;
constexpr int kTcThreads = (kTcFrameWarps + 2) * 32;     // 320
constexpr int kTcMinBlocks = 2;                          // resident CTAs per SM
constexpr int kTcStages = 2;                             // A stages (TMEM) = B stages (shared memory): A and B share the
                                                         // stage index and ONE release barrier per stage
constexpr int kTcACols = 2 * kTcKT;                      // hi + lo columns of one A stage
constexpr int kTcAccN = kTcN;                            // accumulator columns (80: 36 real, 36 imaginary, 8 pad)
constexpr int kTcTmemCols = 256;                         // half of the SM's TMEM per CTA
constexpr int kTcAPre = 3;                               // k-tiles of A rows in flight (cp.async ring in shared memory)
constexpr int kTcAPlane = kTcFrames + 1;                 // float4 per chunk plane of the A staging ring

struct TcSmem {
    alignas(1024) unsigned char b[kTcStages][kTcBStageBytes];
    float4 arow[kTcAPre][8 * kTcAPlane];  // [slot][16-byte chunk · kTcAPlane + frame]: the odd plane stride keeps both the
                                          // (8 rows × 4 chunks) cp.async writes and the per-row LDS.128 reads conflict free
    float chroma_part[kTcFrames][16];    // [frame][4·q + j]: partial chroma (3q + j) mod 12 of column quarter q
    alignas(8) uint64_t full_a[kTcStages], empty_a[kTcStages], full_b[kTcStages], empty_b[kTcStages];
    uint64_t acc_full, acc_empty;
    uint32_t tmem_base;
    double red[4][kChroma];
};

// Epilogue share of column quarter Q: CQT bins b = 9Q … 9Q+8 of this thread's frame.  Accumulator columns: b (real part)
// and 36+b (imaginary part).  Bin b feeds chroma ((b + 1) mod 36) / 3, i.e.
// acc[j] collects chroma (3Q + j) mod 12, j = 0..3.
template <int Q>
__device__ __forceinline__ void tc_epilogue_quarter(uint32_t acc_addr, float (&part)[4]) {
    using namespace tc05;
    float re[9], im[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) re[i] = im[i] = 0.0f;
    uint32_t v[16];
#pragma unroll
    for (int piece = 0; piece < 2; ++piece) {
        constexpr int kBase[2] = {0, kCqtBins};
        const int c0 = kBase[piece] + 9 * Q;
        const int start = c0 & ~7;  // 8-column aligned 16-column load covers c0 … c0+8
        tmem_ld16(acc_addr + (uint32_t)start, v);
        wait_ld();
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            const float val = __uint_as_float(v[c0 - start + i]);
            if (piece & 1) im[i] += val; else re[i] += val;
        }
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        const int b = 9 * Q + i;
        const int ch = ((b + 1) % kCqtBins) / 3;
        const int j = (ch - 3 * Q + kChroma) % kChroma;  // 0..3
        part[j] += cabs_f32(re[i], im[i]);
    }
}

__global__ void __launch_bounds__(kTcThreads, kTcMinBlocks) cqt_tc_kernel(const float *__restrict__ audio,
                                                                         const int64_t *__restrict__ seg_off,
                                                                         const int32_t *__restrict__ seg_len,
                                                                         const float *__restrict__ pyr, PyrOffsets po,
                                                                         const int32_t *__restrict__ tuning_idx,
                                                                         const float *__restrict__ Bimg, int tile_stride,
                                                                         double *__restrict__ partial) {
    using namespace tc05;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    TcSmem &sm = *reinterpret_cast<TcSmem *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    constexpr int kPre = kTcAPre;
    constexpr int kAS = kTcStages, kBS = kTcStages;  // A stages (TMEM), B stages (shared memory)
    constexpr int kAccCol0 = kAS * kTcACols;
    static_assert(kAccCol0 + kTcAccN <= kTcTmemCols, "TMEM budget");
    const int seg = blockIdx.y;
    const int n = seg_len[seg];
    const int n_frames = cqt_frames(n);
    const int t0 = blockIdx.x * kTcFrames;
    if (t0 >= n_frames) return;  // whole CTA leaves before any barrier / TMEM state exists
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        for (int i = 0; i < kAS; ++i) {
            mbar_init(&sm.full_a[i], kTcFrameWarps);  // one arrival per frame warp
            mbar_init(&sm.empty_a[i], 1);
        }
        for (int i = 0; i < kBS; ++i) {
            mbar_init(&sm.full_b[i], 1);
            mbar_init(&sm.empty_b[i], 1);
        }
        mbar_init(&sm.acc_full, 1);
        mbar_init(&sm.acc_empty, kTcFrameWarps);
        fence_mbar_init();
    }
    if (warp == kTcFrameWarps) tmem_alloc(&sm.tmem_base, kTcTmemCols);
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = sm.tmem_base;

    int tj = tuning_idx[seg];
    tj = tj < 0 ? 0 : (tj >= kNTunings ? kNTunings - 1 : tj);
    constexpr int kKTiles = kCqtNfft / kTcKT;  // 32
    constexpr int kIters = kOctaves * kKTiles;
    // Every CTA walks the 32 k-tiles of the contraction from a different starting tile: all CTAs of a launch read the
    // same few B images, and in lock step they would all hit the same L2 lines at the same time.
    const int kshift = (int)((blockIdx.x * 5u + blockIdx.y * 11u) & (kKTiles - 1));

    if (warp < kTcFrameWarps) {
        // ===================== frame warps: A producer + epilogue =====================
        const int rg = warp & 3, q = warp >> 2;   // TMEM lane quarter, column split
        const int f = 32 * rg + lane;  // row of the tile = TMEM lane
        const uint32_t lane_base = (uint32_t)(32 * rg) << 16;
        const float *pseg = pyr + (size_t)seg * po.off[kOctaves];
        constexpr int kQPer = 4 / kTcQ;  // epilogue quarters (9 CQT bins each) per thread
        float part[kQPer][4];
#pragma unroll
        for (int a = 0; a < kQPer; ++a)
#pragma unroll
            for (int j = 0; j < 4; ++j) part[a][j] = 0.0f;

        auto epilogue = [&](int o) {
            mbar_wait_warp(&sm.acc_full, (uint32_t)(o & 1), 100);
            fence_after_sync();
            const uint32_t acc = tmem + lane_base + (uint32_t)kAccCol0;
#pragma unroll
            for (int a = 0; a < kQPer; ++a) {
                switch (q * kQPer + a) {  // warp-uniform
                    case 0: tc_epilogue_quarter<0>(acc, part[a]); break;
                    case 1: tc_epilogue_quarter<1>(acc, part[a]); break;
                    case 2: tc_epilogue_quarter<2>(acc, part[a]); break;
                    default: tc_epilogue_quarter<3>(acc, part[a]); break;
                }
            }
            fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.acc_empty);
        };

        // A rows stream through a cp.async ring (kPre k-tiles ahead, flat over octaves × k-tiles): thread (f, q) owns
        // kTcVals consecutive samples (kTcVals/4 16-byte chunks) of row f in every k-tile.  Zero padding outside [0, len)
        // comes from the src-size (zfill) form — row starts are multiples of 4 samples, so a chunk never straddles 0.
        // The per-tile address arithmetic is kept to a handful of 32-bit operations: this instruction stream, not the
        // MMAs or the memory system, is what paces the kernel (timing experiments, profiles/r2l_cqt_debug.log).
        // The global side of the copies is coalesced: per cp.async instruction the warp's lanes (r8 = lane >> 2, c = lane & 3)
        // fetch the four 16-byte chunks (column half q) of EIGHT rows — 64 contiguous bytes per row — instead of one
        // chunk of 32 different rows (32 different cache lines per instruction at the upper octaves: the L1 tag stage,
        // not the tensor pipe, paced the kernel — profiles/r2f_ncu_summary.md, l1tex 65 % busy).  Four instructions
        // j = 0..3 cover the warp's 32 rows (row 8j + r8).
        constexpr int kChunks = kTcVals / 4;
        static_assert(kChunks == 4, "lane mapping below assumes 4 chunks per row half");
        const float *y0 = audio + seg_off[seg];
        const bool y0_aligned = (reinterpret_cast<uintptr_t>(y0) & 15u) == 0;
        const float *y0_down = reinterpret_cast<const float *>(reinterpret_cast<uintptr_t>(y0) & ~uintptr_t(15));
        const int r8 = lane >> 2, cc = lane & 3;
        const float *ylev = nullptr;  // level base of the octave being issued
        int row0 = 0, row_step = 0, len_o = 0;  // sample offset of (row 32rg + r8, chunk 4q + cc) at k-tile 0; 8·hop; level length
        bool oct_async = true;
        // `oct_fast` (warp-uniform, per octave): every 16-byte piece this warp fetches in the octave lies inside [0, len) and
        // the level is 16-byte aligned — then a copy is one pointer add and one cp.async, with no clamping arithmetic.  The
        // frame warps' instruction count per k-tile, not the tensor pipe, paces this kernel.
        bool oct_fast = false;
        const float *ybase = nullptr;  // ylev + row0 (fast path)
        const uint32_t arow_u32 = smem_u32(&sm.arow[0][0]);
        const uint32_t slot_off = (uint32_t)(((kChunks * q + cc) * kTcAPlane + 32 * rg + r8) * sizeof(float4));
        constexpr uint32_t kSlotBytes = 8 * kTcAPlane * sizeof(float4);
        auto issue = [&](int it) {
            const int kt = ((it & 31) + kshift) & 31;
            if ((it & 31) == 0) {  // new octave: row geometry
                const int o = it >> 5;
                const int hop = 512 >> o;
                ylev = (o == 0) ? y0 : pseg + po.off[o];
                len_o = level_len(n, o);
                row0 = (t0 + 32 * rg + r8) * hop - kCqtNfft / 2 + kTcVals * q + 4 * cc;
                row_step = 8 * hop;
                oct_async = (o > 0) || y0_aligned;
                const bool inside = row0 >= 0 && row0 + 3 * row_step + (kCqtNfft - kTcKT) + 4 <= len_o;
                oct_fast = oct_async && __all_sync(0xffffffffu, inside);
                ybase = ylev + row0;
            }
            const uint32_t slot_u32 = arow_u32 + (uint32_t)(it % kPre) * kSlotBytes + slot_off;
            if (oct_fast) {
                const float *src = ybase + kt * kTcKT;
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(slot_u32 + (uint32_t)(8 * j * sizeof(float4))),
                                 "l"(src + j * row_step)
                                 : "memory");
            } else if (oct_async) {
                const int p0 = row0 + kt * kTcKT;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int p = p0 + j * row_step;  // first sample of this 16-byte piece (multiple of 4: never straddles 0)
                    const int rem = (len_o - p) * 4;
                    const uint32_t bytes = (p < 0 || rem <= 0) ? 0u : (uint32_t)(rem > 16 ? 16 : rem);
                    const float *src = bytes ? ylev + p : y0_down;  // src-size 0: nothing is read, but the address stays aligned
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(slot_u32 + (uint32_t)(8 * j * sizeof(float4))),
                                 "l"(src), "r"(bytes)
                                 : "memory");
                }
            } else {  // unaligned first level (arbitrary caller offset): plain loads into the same slots
                const int p0 = row0 + kt * kTcKT;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float xr[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int p = p0 + j * row_step + i;
                        xr[i] = (p >= 0 && p < len_o) ? __ldg(ylev + p) : 0.0f;
                    }
                    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(slot_u32 + (uint32_t)(8 * j * sizeof(float4))),
                                 "f"(xr[0]), "f"(xr[1]), "f"(xr[2]), "f"(xr[3])
                                 : "memory");
                }
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        for (int it = 0; it < kPre - 1; ++it) issue(it);
        bool pending = false;
        for (int it = 0; it < kIters; ++it) {
            if (it + kPre - 1 < kIters) issue(it + kPre - 1);
            else asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group %0;" ::"n"(kPre - 1) : "memory");
            __syncwarp();  // the row this thread reads was fetched by other lanes of its warp
            const int o = it >> 5, kt = it & 31;
            const int st = it % kAS;
            uint32_t h[kTcVals], l[kTcVals];
            {
                // x = hi + lo with hi = x truncated to tf32 (one LOP3; cvt.rna.tf32 is a five-instruction sequence here) and
                // lo = x − hi exactly; |lo| < 2^-10·|x|, and the tensor core reads lo's leading 11 bits: the split is good to
                // 2^-20·|x|, on a 1e-4 tolerance (measured worst chroma error 5e-7 of the maximum, tests/test_gpu_pitch.py)
                const uint32_t rd = arow_u32 + (uint32_t)(it % kPre) * kSlotBytes +
                                    (uint32_t)(((kChunks * q) * kTcAPlane + f) * sizeof(float4));
#pragma unroll
                for (int c = 0; c < kChunks; ++c) {
                    float x[4];
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                                 : "=f"(x[0]), "=f"(x[1]), "=f"(x[2]), "=f"(x[3])
                                 : "r"(rd + (uint32_t)(c * kTcAPlane * sizeof(float4)))
                                 : "memory");
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const uint32_t hb = __float_as_uint(x[i]) & 0xffffe000u;
                        h[4 * c + i] = hb;
                        l[4 * c + i] = __float_as_uint(x[i] - __uint_as_float(hb));
                    }
                }
            }
            __syncwarp();  // all lanes have read the slot before other lanes re-fill it (issue() of the next iteration)
            if (pending) {  // publish the PREVIOUS tile: its tcgen05.st had a whole iteration to land
                wait_st();
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.full_a[(it - 1) % kAS]);
            }
            mbar_wait_warp(&sm.empty_a[st], (uint32_t)(((it / kAS) & 1) ^ 1), 40);
            fence_after_sync();
            const uint32_t a0 = tmem + lane_base + (uint32_t)(st * kTcACols + kTcVals * q);
            tmem_st_vals(a0, h);
            tmem_st_vals(a0 + kTcKT, l);
            pending = true;
            if (kt == kKTiles - 1) {  // octave boundary (and the very last tile): publish before the epilogue
                wait_st();
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.full_a[st]);
                pending = false;
                epilogue(o);  // one accumulator: the MMAs of the next octave wait for this read
            }
        }

        // ---- combine the four column quarters of every frame, librosa.util.normalize(norm=inf) per frame, then the
        // tile's sum over frames (float64)
#pragma unroll
        for (int a = 0; a < kQPer; ++a)
#pragma unroll
            for (int j = 0; j < 4; ++j) sm.chroma_part[f][4 * (q * kQPer + a) + j] = part[a][j];
        asm volatile("bar.sync 1, %0;" ::"n"(kTcFrameWarps * 32) : "memory");  // the frame warps only
        if (q == 0) {
            float chroma[kChroma];
#pragma unroll
            for (int c = 0; c < kChroma; ++c) {
                // chroma c = slot j = c % 3 of quarter c / 3, plus slot 3 of the previous quarter when c % 3 == 0
                float v = sm.chroma_part[f][4 * (c / 3) + (c % 3)];
                if (c % 3 == 0) v += sm.chroma_part[f][4 * ((c / 3 + 3) % 4) + 3];
                chroma[c] = v;
            }
            const bool valid = (t0 + f) < n_frames;
            float mx = 0.0f;
#pragma unroll
            for (int c = 0; c < kChroma; ++c) mx = fmaxf(mx, chroma[c]);
            const double len_ = (mx < 1.17549435e-38f) ? 1.0 : (double)mx;
#pragma unroll
            for (int c = 0; c < kChroma; ++c) {
                double v = valid ? (double)chroma[c] / len_ : 0.0;
                v = warp_sum(v);
                if (lane == 0) sm.red[rg][c] = v;
            }
            asm volatile("bar.sync 2, 128;" ::: "memory");  // warps 0-3
            if (tid < kChroma)
                partial[((size_t)seg * tile_stride + blockIdx.x) * kChroma + tid] =
                    ((sm.red[0][tid] + sm.red[1][tid]) + sm.red[2][tid]) + sm.red[3][tid];
        }
    } else if (warp == kTcFrameWarps) {
        // ===================== MMA issuer (warp-uniform control flow, one elected lane issues) =====================
        constexpr uint32_t idesc = idesc_tf32(kTcFrames, kTcN);  // M 128 × N 80 × K 8
        for (int o = 0; o < kOctaves; ++o) {
            mbar_wait_warp(&sm.acc_empty, (uint32_t)((o & 1) ^ 1));
            fence_after_sync();
            const uint32_t d = tmem + (uint32_t)kAccCol0;
            for (int kt = 0; kt < kKTiles; ++kt) {
                const int it = o * kKTiles + kt;
                const int sa = it % kAS, sb = it % kBS;
                mbar_wait_warp(&sm.full_a[sa], (uint32_t)((it / kAS) & 1));
                mbar_wait_warp(&sm.full_b[sb], (uint32_t)((it / kBS) & 1));
                fence_after_sync();
                const uint64_t bh = smem_desc_k128(sm.b[sb]);                  // hi image of the K tile
                const uint64_t bl = smem_desc_k128(sm.b[sb] + kTcBTileBytes);  // lo image
                const uint32_t ah = tmem + (uint32_t)(sa * kTcACols), al = ah + kTcKT;
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < kTcKT / 8; ++k) {
                        const uint64_t adv = (uint64_t)((k * 8 * 4) >> 4);  // 32 bytes per K = 8 step inside the swizzle row
                        mma_tf32_ts(d, ah + 8 * k, bh + adv, idesc, (kt | k) != 0);  // 3×TF32: Ah·Bh + Al·Bh + Ah·Bl
                        mma_tf32_ts(d, al + 8 * k, bh + adv, idesc, 1);
                        mma_tf32_ts(d, ah + 8 * k, bl + adv, idesc, 1);
                    }
                    commit(&sm.empty_a[sa]);  // frees the A stage (TMEM) and the B stage (shared memory) of this tile together:
                                              // tcgen05.commit is the scarce operation of this pipeline, one per tile
                    if (kt == kKTiles - 1) commit(&sm.acc_full);
                }
                __syncwarp();
            }
        }
    } else {
        // ===================== B loader (warp-uniform, one elected lane issues the bulk copy) =====================
        const unsigned char *src = reinterpret_cast<const unsigned char *>(Bimg) + (size_t)tj * kKTiles * kTcBStageBytes;
        for (int it = 0; it < kIters; ++it) {
            const int sb = it % kBS, kt = ((it % kKTiles) + kshift) & (kKTiles - 1);
            mbar_wait_warp(&sm.empty_a[sb], (uint32_t)(((it / kBS) & 1) ^ 1), 100);
            if (elect_one()) {
                mbar_arrive_expect_tx(&sm.full_b[sb], kTcBStageBytes);
                bulk_g2s(sm.b[sb], src + (size_t)kt * kTcBStageBytes, kTcBStageBytes, &sm.full_b[sb]);
            }
            __syncwarp();
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == kTcFrameWarps) {
        fence_after_sync();
        tmem_dealloc(tmem, kTcTmemCols);
    }
}

// mean over frames: one warp per segment sums the tile partials in tile order
__global__ void __launch_bounds__(32) chroma_mean_kernel(const int32_t *__restrict__ seg_len, int tile_stride,
                                                         int frames_per_tile, const double *__restrict__ partial,
                                                         double *__restrict__ chroma) {
    const int seg = blockIdx.x;
    const int n_frames = cqt_frames(seg_len[seg]);
    const int n_tiles = (n_frames + frames_per_tile - 1) / frames_per_tile;
    const int ch = threadIdx.x;
    if (ch >= kChroma) return;
    double s = 0.0;
    for (int t = 0; t < n_tiles; ++t) s += partial[((size_t)seg * tile_stride + t) * kChroma + ch];
    chroma[(size_t)seg * kChroma + ch] = s / (double)n_frames;
}

// pitch._cyclic_xcorr_peak: xcorr[k] = dot(src, roll(nc, -k)); first maximum; wrap lags > n/2
__global__ void __launch_bounds__(64) cyclic_xcorr_kernel(const double *__restrict__ src, const double *__restrict__ nc,
                                                          int n_pairs, int n_bins, int32_t *__restrict__ lag) {
    const int p = blockIdx.x * 64 + threadIdx.x;
    if (p >= n_pairs) return;
    const double *a = src + (size_t)p * n_bins, *b = nc + (size_t)p * n_bins;
    double best = -INFINITY;
    int bk = 0;
    for (int k = 0; k < n_bins; ++k) {
        double s = 0.0;
        for (int i = 0; i < n_bins; ++i) {
            int j = i + k;
            if (j >= n_bins) j -= n_bins;  // roll(nc, -k)[i] = nc[(i + k) mod n]
            s = fma(a[i], b[j], s);
        }
        if (s > best) {
            best = s;
            bk = k;
        }
    }
    if (bk > n_bins / 2) bk -= n_bins;
    lag[p] = bk;
}

}  // namespace ncfa

using namespace ncfa;

static size_t tuning_frames(int max_seg_len) { return 1 + (size_t)max_seg_len / 512; }

// per frame kPeakStride candidate peaks (magnitude, bin) and their count
struct TuningWs {
    float *pk_mag;
    uint8_t *pk_bin;
    int32_t *pk_cnt;
    size_t bytes;
};

static TuningWs tuning_ws(int n_seg, int max_seg_len, void *base) {
    const size_t frames = (size_t)n_seg * tuning_frames(max_seg_len);
    Carve c(base);
    TuningWs w;
    w.pk_mag = c.take<float>(frames * kPeakStride);
    w.pk_bin = c.take<uint8_t>(frames * kPeakStride);
    w.pk_cnt = c.take<int32_t>(frames);
    w.bytes = c.used;
    return w;
}

extern "C" size_t ncfa_tuning_workspace_bytes(int n_seg, int max_seg_len) {
    if (n_seg <= 0 || max_seg_len < 0) return 0;
    return tuning_ws(n_seg, max_seg_len, nullptr).bytes;
}

extern "C" int ncfa_tuning_estimate_batched(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len,
                                            int n_seg, int max_seg_len, int sr, int32_t *d_tuning_idx,
                                            void *d_workspace, size_t workspace_bytes, void *stream) {
    NCFA_REQUIRE(n_seg >= 0 && n_seg <= 65535, "n_seg must be in [0, 65535] per call");
    if (n_seg == 0) return NCFA_OK;
    NCFA_REQUIRE(d_audio && d_seg_off && d_seg_len && d_tuning_idx && d_workspace, "null pointer");
    NCFA_REQUIRE(max_seg_len >= 0 && sr > 0, "max_seg_len/sr");
    const TuningWs w = tuning_ws(n_seg, max_seg_len, d_workspace);
    int rc = check_workspace("tuning", workspace_bytes, w.bytes);
    if (rc) return rc;
    Tables tb;
    if ((rc = get_tables(sr, &tb))) return rc;
    // piptrack frequency mask: fmin=150 <= fft_freq < min(4000, sr/2), fft_freq[k] = k · (1 / (n_fft · (1/sr)))
    const double val = 1.0 / (2048.0 * (1.0 / (double)sr));
    const double fmax = fmin(4000.0, (double)sr / 2.0);
    int kmin = 1, kmax = 1023;
    while (kmin < 1024 && !((double)kmin * val >= 150.0)) ++kmin;
    while (kmax > 0 && !((double)kmax * val < fmax)) --kmax;
    NCFA_REQUIRE(kmin <= kmax && (kmax - kmin + 2) / 2 <= kPeakStride, "piptrack band does not fit the peak buffer");
    cudaStream_t st = (cudaStream_t)stream;
    const int frames = (int)tuning_frames(max_seg_len);
    int n_sm = 0;
    if ((rc = sm_count(&n_sm))) return rc;
    const int64_t groups = ((int64_t)n_seg * frames + kTunWarps - 1) / kTunWarps;
    const int grid = (int)(groups < n_sm ? groups : n_sm);
    if ((rc = launch("tuning_peaks_kernel", tuning_peaks_kernel, grid, kTunThreads, sizeof(TuningSmem), st, d_audio,
                     d_seg_off, d_seg_len, n_seg, frames, kmin, kmax, (double)sr / 2048.0, tb, w.pk_mag, w.pk_bin,
                     w.pk_cnt)))
        return rc;
    return launch("tuning_pick_kernel", tuning_pick_kernel, n_seg, 256, 0, st, d_seg_len, frames, w.pk_mag, w.pk_bin,
                  w.pk_cnt, d_tuning_idx);
}

static int chroma_tiles(int max_seg_len) { return (cqt_frames(max_seg_len) + kPartialTF - 1) / kPartialTF; }

// the decimated pyramid of every segment (plus 16 bytes), then kChroma float64 partial sums per tile of frames
struct ChromaWs {
    float *pyr;
    double *partial;
    size_t bytes;
};

static ChromaWs chroma_ws(int n_seg, int max_seg_len, const PyrOffsets &po, void *base) {
    Carve c(base);
    ChromaWs w;
    w.pyr = c.take<float>((size_t)n_seg * po.off[kOctaves] + 4);
    w.partial = c.take<double>((size_t)n_seg * chroma_tiles(max_seg_len) * kChroma);
    w.bytes = c.used;
    return w;
}

extern "C" size_t ncfa_chroma_workspace_bytes(int n_seg, int max_seg_len) {
    if (n_seg <= 0 || max_seg_len < 0) return 0;
    PyrOffsets po;
    pyramid_layout(max_seg_len, po.off);
    return chroma_ws(n_seg, max_seg_len, po, nullptr).bytes;
}

extern "C" int ncfa_chroma_mean_batched(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len,
                                        int n_seg, int max_seg_len, int sr, const int32_t *d_tuning_idx,
                                        double *d_chroma, void *d_workspace, size_t workspace_bytes, void *stream) {
    NCFA_REQUIRE(n_seg >= 0 && n_seg <= 65535, "n_seg must be in [0, 65535] per call");
    if (n_seg == 0) return NCFA_OK;
    NCFA_REQUIRE(d_audio && d_seg_off && d_seg_len && d_tuning_idx && d_chroma && d_workspace, "null pointer");
    NCFA_REQUIRE(max_seg_len >= 0, "max_seg_len");
    NCFA_REQUIRE(sr == 22050, "the CQT path is laid out for sr = 22050 (7 octaves from C1, n_fft 1024, no early downsampling)");
    PyrOffsets po;
    pyramid_layout(max_seg_len, po.off);
    const ChromaWs w = chroma_ws(n_seg, max_seg_len, po, d_workspace);
    int rc = check_workspace("chroma", workspace_bytes, w.bytes);
    if (rc) return rc;
    ChromaTables ct;
    if ((rc = get_chroma_tables(sr, &ct))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t stride = po.off[kOctaves];
    for (int level = 1; level < kOctaves; ++level) {
        const int n_out = level_len(max_seg_len, level);
        if (n_out <= 0) continue;
        if ((rc = launch("decimate2_kernel", decimate2_kernel, dim3((n_out + kDecOutPerCta - 1) / kDecOutPerCta, n_seg),
                         256, 0, st, d_audio, d_seg_off, d_seg_len, level, w.pyr, stride,
                         level >= 2 ? po.off[level - 1] : 0, po.off[level], ct.hb)))
            return rc;
    }
    const int tiles = chroma_tiles(max_seg_len);  // partial[] stride
    if ((rc = launch("cqt_tc_kernel", cqt_tc_kernel, dim3((cqt_frames(max_seg_len) + kTcFrames - 1) / kTcFrames, n_seg),
                     kTcThreads, sizeof(TcSmem) + 1024, st, d_audio, d_seg_off, d_seg_len, w.pyr, po, d_tuning_idx,
                     ct.Bimg, tiles, w.partial)))
        return rc;
    return launch("chroma_mean_kernel", chroma_mean_kernel, n_seg, 32, 0, st, d_seg_len, tiles, kTcFrames, w.partial,
                  d_chroma);
}

extern "C" int ncfa_cyclic_xcorr_batched(const double *d_src, const double *d_nc, int n_pairs, int n_bins,
                                         int32_t *d_lag, void *stream) {
    NCFA_REQUIRE(n_pairs >= 0 && n_bins > 0, "n_pairs/n_bins");
    if (n_pairs == 0) return NCFA_OK;
    NCFA_REQUIRE(d_src && d_nc && d_lag, "null pointer");
    return launch("cyclic_xcorr_kernel", cyclic_xcorr_kernel, (n_pairs + 63) / 64, 64, 0, (cudaStream_t)stream, d_src,
                  d_nc, n_pairs, n_bins, d_lag);
}

// Host-side table builders, exported so that the CPU test-suite can check them without a GPU.
extern "C" int ncfa_host_cqt_matrix(int sr, int tuning_index, float *h_K /* [1024][72] */) {
    NCFA_REQUIRE(h_K && tuning_index >= 0 && tuning_index < kNTunings, "h_K/tuning_index");
    std::vector<float> K;
    int rc = build_cqt_matrix(sr, (double)tuning_index * 0.01 + (-0.5), K);
    if (rc) return rc;
    memcpy(h_K, K.data(), K.size() * sizeof(float));
    return NCFA_OK;
}

extern "C" int ncfa_host_halfband_taps(double *h_taps /* [127] */) {
    NCFA_REQUIRE(h_taps, "h_taps");
    std::vector<double> h;
    build_halfband(h);
    memcpy(h_taps, h.data(), h.size() * sizeof(double));
    return NCFA_OK;
}
