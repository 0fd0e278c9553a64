// Band-limited speed change (sox `speed X`, workflow.py:117): output sample m of a segment is the source evaluated at
// input time t = m·R through a Kaiser-windowed sinc read from a table with linear interpolation, low-passed at the new
// Nyquist frequency when R > 1.  Every float64 operation and the order of the tap sum are fixed (include/ncfa.h), and one
// thread owns each output, so with -fmad=false the result is bit-for-bit that of oracle/render_restated.py.
#include <math.h>
#include <map>
#include <mutex>
#include <vector>
#include "ncfa_common.cuh"

namespace ncfa {

constexpr int RENDER_ZL = NCFA_RENDER_ZEROS * NCFA_RENDER_PHASES;  // table entries up to the last zero crossing
constexpr int RENDER_TILE = 256;                                   // consecutive outputs per CTA, one per thread
// Input span of one tile at the largest ratio: (TILE − 1)·R_max + 2 for the two floors, plus the taps ceil(2·half) + 1
// of half = Z·R_max/ρ (= 271 at R = 4), rounded up.
constexpr int RENDER_SPAN_MAX = (RENDER_TILE - 1) * 4 + 2 + 272 + 8;

__host__ __device__ inline int64_t render_out_len(int32_t len, double ratio) {
    return len > 0 ? (int64_t)floor((double)(len - 1) / ratio) + 1 : 0;
}

// I0 by the Chebyshev expansions of Clenshaw (1962) on [0, 8] and (8, ∞), with Cephes' coefficients and the same
// operations as numpy.i0, so the table agrees with numpy's statement of the formula to a float64 ulp or so.
static const double I0_A[30] = {
    -4.4153416464793395e-18, 3.3307945188222384e-17, -2.431279846547955e-16,
    1.715391285555133e-15, -1.1685332877993451e-14, 7.676185498604936e-14,
    -4.856446783111929e-13, 2.95505266312964e-12, -1.726826291441556e-11,
    9.675809035373237e-11, -5.189795601635263e-10, 2.6598237246823866e-09,
    -1.300025009986248e-08, 6.046995022541919e-08, -2.670793853940612e-07,
    1.1173875391201037e-06, -4.4167383584587505e-06, 1.6448448070728896e-05,
    -5.754195010082104e-05, 0.00018850288509584165, -0.0005763755745385824,
    0.0016394756169413357, -0.004324309995050576, 0.010546460394594998,
    -0.02373741480589947, 0.04930528423967071, -0.09490109704804764,
    0.17162090152220877, -0.3046826723431984, 0.6767952744094761};
static const double I0_B[25] = {
    -7.233180487874754e-18, -4.830504485944182e-18, 4.46562142029676e-17,
    3.461222867697461e-17, -2.8276239805165836e-16, -3.425485619677219e-16,
    1.7725601330565263e-15, 3.8116806693526224e-15, -9.554846698828307e-15,
    -4.150569347287222e-14, 1.54008621752141e-14, 3.8527783827421426e-13,
    7.180124451383666e-13, -1.7941785315068062e-12, -1.3215811840447713e-11,
    -3.1499165279632416e-11, 1.1889147107846439e-11, 4.94060238822497e-10,
    3.3962320257083865e-09, 2.266668990498178e-08, 2.0489185894690638e-07,
    2.8913705208347567e-06, 6.889758346916825e-05, 0.0033691164782556943,
    0.8044904110141088};
template <int N>
static double chbevl(double x, const double (&v)[N]) {
    double b0 = v[0], b1 = 0.0, b2 = 0.0;
    for (int i = 1; i < N; ++i) {
        b2 = b1;
        b1 = b0;
        b0 = x * b1 - b2 + v[i];
    }
    return 0.5 * (b0 - b2);
}
static double bessel_i0(double x) {
    x = fabs(x);
    return x <= 8.0 ? exp(x) * chbevl(x / 2.0 - 2.0, I0_A) : exp(x) * chbevl(32.0 / x - 2.0, I0_B) / sqrt(x);
}

static void build_render_table(std::vector<double> &t) {
    const double PI = 3.14159265358979323846, L = NCFA_RENDER_PHASES, ZL = RENDER_ZL, beta = NCFA_RENDER_BETA;
    const double i0b = bessel_i0(beta);
    t.assign(RENDER_ZL + 1, 0.0);  // t[ZL] = 0: the interpolation partner of the last entry
    for (int j = 0; j < RENDER_ZL; ++j) {
        const double x = j / L, r = j / ZL;
        const double sinc = j == 0 ? 1.0 : sin(PI * x) / (PI * x);
        t[j] = sinc * bessel_i0(beta * sqrt(1.0 - r * r)) / i0b;
    }
}

static std::mutex g_rt_mu;
static std::map<int, const double *> g_rt;
static int get_render_table_device(const double **out) {
    int dev = 0;
    NCFA_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_rt_mu);
    auto it = g_rt.find(dev);
    if (it != g_rt.end()) {
        *out = it->second;
        return NCFA_OK;
    }
    std::vector<double> h;
    build_render_table(h);
    double *d = nullptr;
    NCFA_CUDA_OK(cudaMalloc(&d, h.size() * sizeof(double)));
    NCFA_CUDA_OK(cudaMemcpy(d, h.data(), h.size() * sizeof(double), cudaMemcpyHostToDevice));
    g_rt[dev] = d;
    *out = d;
    return NCFA_OK;
}

// CTA (x, seg) renders outputs [256·x, 256·x + 256) of segment seg.  It first stages its whole input span in shared
// memory as float64, zero outside the segment, so the edges and every sample alignment are handled in one place and the
// tap loop has no bounds test.  A staged zero adds ±0 to an accumulator that is never −0, exactly like the skipped tap
// of the specification.  The table is read through L1.
__global__ void __launch_bounds__(RENDER_TILE) render_kernel(const float *__restrict__ audio,
                                                             const int64_t *__restrict__ seg_off,
                                                             const int32_t *__restrict__ seg_len,
                                                             const double *__restrict__ ratio,
                                                             const int64_t *__restrict__ out_off,
                                                             const double *__restrict__ table, float *__restrict__ out) {
    __shared__ double xs[RENDER_SPAN_MAX];
    const int seg = blockIdx.y;
    const int len = seg_len[seg];
    const double R = ratio[seg];
    const int64_t n_out = render_out_len(len, R);
    const int64_t m0 = (int64_t)blockIdx.x * RENDER_TILE;
    if (m0 >= n_out) return;
    const double c = NCFA_RENDER_ROLLOFF / fmax(1.0, R);
    const double half = NCFA_RENDER_ZEROS / c;
    const int taps = (int)ceil(2.0 * half) + 1;
    const float *x = audio + seg_off[seg];
    // n0 = floor(m·R − half) + 1 is non-decreasing in m, so the tile reads [n0(m0), n0(m_last) + taps)
    const int64_t m_last = min(m0 + RENDER_TILE, n_out) - 1;
    const int64_t lo = (int64_t)floor((double)m0 * R - half) + 1;
    const int span = (int)((int64_t)floor((double)m_last * R - half) + 1 + taps - lo);
    if (span > RENDER_SPAN_MAX) return;  // only a d_ratio outside [0.25, 4] (the host checked h_ratio) gets here
    for (int j = threadIdx.x; j < span; j += RENDER_TILE) {
        const int64_t p = lo + j;
        xs[j] = (p >= 0 && p < len) ? (double)__ldg(x + p) : 0.0;
    }
    __syncthreads();
    const int64_t m = m0 + threadIdx.x;
    if (m > m_last) return;
    const double t = (double)m * R;
    const double n0 = floor(t - half) + 1.0;
    const double *xp = xs + ((int64_t)n0 - lo);
    double acc = 0.0;
    for (int k = 0; k < taps; ++k) {
        const double d = (fabs(t - (n0 + (double)k)) * c) * (double)NCFA_RENDER_PHASES;
        const int i = (int)d;  // d >= 0: truncation is floor
        const double f = d - (double)i;
        if (i < RENDER_ZL) {
            const double t0 = __ldg(table + i), t1 = __ldg(table + i + 1);
            acc += (t0 + f * (t1 - t0)) * xp[k];
        }
    }
    out[out_off[seg] + m] = (float)(acc * c);
}

}  // namespace ncfa

using namespace ncfa;

extern "C" int64_t ncfa_render_out_len(int32_t len, double ratio) { return render_out_len(len, ratio); }

extern "C" int ncfa_host_render_table(double *h_table) {
    NCFA_REQUIRE(h_table, "h_table");
    std::vector<double> t;
    build_render_table(t);
    memcpy(h_table, t.data(), t.size() * sizeof(double));
    return NCFA_OK;
}

extern "C" int ncfa_render_batched(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len,
                                   const double *d_ratio, const double *h_ratio, int n_seg, int max_seg_len,
                                   const int64_t *d_out_off, float *d_out, void *stream) {
    NCFA_REQUIRE(n_seg >= 0 && n_seg <= 65535, "n_seg must be in [0, 65535] per call");
    if (n_seg == 0) return NCFA_OK;
    NCFA_REQUIRE(d_audio && d_seg_off && d_seg_len && d_ratio && h_ratio && d_out_off && d_out, "null pointer");
    NCFA_REQUIRE(max_seg_len >= 0, "max_seg_len");
    double r_min = 4.0;
    for (int i = 0; i < n_seg; ++i) {
        NCFA_REQUIRE(isfinite(h_ratio[i]) && h_ratio[i] >= 0.25 && h_ratio[i] <= 4.0, "ratio must be finite and in [0.25, 4]");
        r_min = fmin(r_min, h_ratio[i]);
    }
    const double *table = nullptr;
    if (int rc = get_render_table_device(&table)) return rc;
    // at least one CTA per segment, so a batch of empty segments is still one launch
    const int64_t tiles = (render_out_len(max_seg_len, r_min) + RENDER_TILE - 1) / RENDER_TILE;
    return launch("render_kernel", render_kernel, dim3((unsigned)(tiles > 0 ? tiles : 1), n_seg), RENDER_TILE, 0,
                  (cudaStream_t)stream, d_audio, d_seg_off, d_seg_len, d_ratio, d_out_off, table, d_out);
}
