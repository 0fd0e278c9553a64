// Energy reductions: per-window mean square in float64 (io.py:38-40 _rms_db, used by
// slice_windows io.py:94-110 and energy_gate io.py:115-126) and framed RMS
// (librosa.feature.rms / effects.trim: io.py:76, xcorr.py:210-211; SURVEY Appendix A.6/A.7).
#include "ncfa_common.cuh"

namespace ncfa {

__global__ void __launch_bounds__(256) window_energy_kernel(const float *__restrict__ audio,
                                                            const int64_t *__restrict__ seg_off,
                                                            const int32_t *__restrict__ seg_len,
                                                            double *__restrict__ meansq) {
    __shared__ double sh[8];
    const int seg = blockIdx.x;
    const int n = seg_len[seg];
    const float *x = audio + seg_off[seg];
    double acc = 0.0;
    // 4 independent accumulators per thread keep the FP64 pipe busy behind the loads
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    int i = threadIdx.x;
    for (; i + 768 < n; i += 1024) {
        double v0 = (double)__ldg(x + i), v1 = (double)__ldg(x + i + 256), v2 = (double)__ldg(x + i + 512),
               v3 = (double)__ldg(x + i + 768);
        a0 = fma(v0, v0, a0);
        a1 = fma(v1, v1, a1);
        a2 = fma(v2, v2, a2);
        a3 = fma(v3, v3, a3);
    }
    for (; i < n; i += 256) {
        double v = (double)__ldg(x + i);
        a0 = fma(v, v, a0);
    }
    acc = (a0 + a1) + (a2 + a3);
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s += sh[w];
        meansq[seg] = n > 0 ? s / (double)n : 0.0;
    }
}

// one warp per frame; frame f covers samples [f·hop − L/2, f·hop + L/2), zeros outside [0, n)
__global__ void __launch_bounds__(256) rms_frames_kernel(const float *__restrict__ x, int64_t n, int frame_length,
                                                         int hop, int64_t n_frames, float *__restrict__ out) {
    const int64_t f = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (f >= n_frames) return;
    const int lane = threadIdx.x & 31;
    const int64_t s0 = f * hop - frame_length / 2;
    double acc = 0.0;
    for (int j = lane; j < frame_length; j += 32) {
        int64_t p = s0 + j;
        if (p >= 0 && p < n) {
            double v = (double)__ldg(x + p);
            acc = fma(v, v, acc);
        }
    }
    acc = warp_sum(acc);
    if (lane == 0) out[f] = (float)sqrt(acc / (double)frame_length);
}


// ---- batched librosa.effects.trim bounds (io.py:58-79 for every track of a batch, no host round trip per track)
// Frame f (2048 samples centred on f·512, zero padded) is the union of four 512-sample blocks, so every sample is
// read once: pass 1 writes float64 block sums, pass 2 forms rms[f] = float32(sqrt(Σ4 blocks / 2048)), the track
// maximum, db = 10·log10(max(1e-10, rms²)) − 10·log10(max(1e-10, max²)) in float32 like numpy on float32 input, and
// the first / last frame with db > −top_db → start = 512·first, end = min(n, 512·(last + 1)); none → (0, 0).
__global__ void __launch_bounds__(256) trim_blocksum_kernel(const float *__restrict__ audio,
                                                            const int64_t *__restrict__ seg_off,
                                                            const int32_t *__restrict__ seg_len, int block_stride,
                                                            double *__restrict__ bsum) {
    const int seg = blockIdx.y;
    const int n = seg_len[seg];
    const int n_blocks = n / 512 + 4;  // blocks j = 0 .. n_frames + 2, block j = samples [(j−2)·512, (j−1)·512)
    const int j = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (j >= n_blocks) return;
    const int lane = threadIdx.x & 31;
    const float *x = audio + seg_off[seg];
    const int64_t s0 = ((int64_t)j - 2) * 512;
    double acc = 0.0;
#pragma unroll 4
    for (int i = lane; i < 512; i += 32) {
        const int64_t p = s0 + i;
        if (p >= 0 && p < n) {
            const double v = (double)__ldg(x + p);
            acc = fma(v, v, acc);
        }
    }
    acc = warp_sum(acc);
    if (lane == 0) bsum[(size_t)seg * block_stride + j] = acc;
}

__global__ void __launch_bounds__(256) trim_bounds_kernel(const int32_t *__restrict__ seg_len, int block_stride,
                                                          const double *__restrict__ bsum, float top_db,
                                                          int64_t *__restrict__ bounds) {
    __shared__ float s_max[256];
    __shared__ int s_lo[256], s_hi[256];
    const int seg = blockIdx.x;
    const int n = seg_len[seg];
    const int n_frames = 1 + n / 512;
    const double *b = bsum + (size_t)seg * block_stride;
    auto rms_of = [&](int f) { return (float)sqrt((((b[f] + b[f + 1]) + b[f + 2]) + b[f + 3]) / 2048.0); };
    float mx = 0.0f;
    for (int f = threadIdx.x; f < n_frames; f += 256) mx = fmaxf(mx, rms_of(f));
    s_max[threadIdx.x] = mx;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) s_max[threadIdx.x] = fmaxf(s_max[threadIdx.x], s_max[threadIdx.x + o]);
        __syncthreads();
    }
    mx = s_max[0];
    const float ref_db = __fmul_rn(10.0f, log10f(fmaxf(1e-10f, __fmul_rn(mx, mx))));
    int lo = 0x7fffffff, hi = -1;
    for (int f = threadIdx.x; f < n_frames; f += 256) {
        const float m = rms_of(f);
        const float db = __fsub_rn(__fmul_rn(10.0f, log10f(fmaxf(1e-10f, __fmul_rn(m, m)))), ref_db);
        if (db > -top_db) {
            lo = f < lo ? f : lo;
            hi = f > hi ? f : hi;
        }
    }
    s_lo[threadIdx.x] = lo;
    s_hi[threadIdx.x] = hi;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            s_lo[threadIdx.x] = min(s_lo[threadIdx.x], s_lo[threadIdx.x + o]);
            s_hi[threadIdx.x] = max(s_hi[threadIdx.x], s_hi[threadIdx.x + o]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        int64_t start = 0, end = 0;
        if (s_hi[0] >= 0) {
            start = (int64_t)s_lo[0] * 512;
            end = (int64_t)(s_hi[0] + 1) * 512;
            if (end > n) end = n;
        }
        bounds[2 * seg] = start;
        bounds[2 * seg + 1] = end;
    }
}

// one float64 sum per 512-sample block, `stride` blocks (3 spare) per segment
struct TrimWs {
    int stride;
    double *bsum;
    size_t bytes;
};

static TrimWs trim_ws(int n_seg, int max_seg_len, void *base) {
    Carve c(base);
    TrimWs w;
    w.stride = max_seg_len / 512 + 4;
    w.bsum = c.take<double>((size_t)n_seg * w.stride);
    w.bytes = c.used;
    return w;
}

}  // namespace ncfa

using namespace ncfa;

extern "C" int ncfa_window_energy(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len, int n_seg,
                                  double *d_meansq, void *stream) {
    NCFA_REQUIRE(n_seg >= 0, "n_seg");
    if (n_seg == 0) return NCFA_OK;
    NCFA_REQUIRE(d_audio && d_seg_off && d_seg_len && d_meansq, "null pointer");
    return launch("window_energy_kernel", window_energy_kernel, n_seg, 256, 0, (cudaStream_t)stream, d_audio, d_seg_off,
                  d_seg_len, d_meansq);
}

extern "C" int ncfa_rms_frames(const float *d_audio, int64_t n, int frame_length, int hop, float *d_rms, void *stream) {
    NCFA_REQUIRE(d_audio && d_rms, "null pointer");
    NCFA_REQUIRE(n >= 0 && frame_length > 0 && hop > 0, "n/frame_length/hop");
    const int64_t n_frames = 1 + n / hop;
    NCFA_REQUIRE((n_frames + 7) / 8 < 2147483647LL, "too many frames");
    return launch("rms_frames_kernel", rms_frames_kernel, (unsigned)((n_frames + 7) / 8), 256, 0, (cudaStream_t)stream,
                  d_audio, n, frame_length, hop, n_frames, d_rms);
}

extern "C" size_t ncfa_trim_workspace_bytes(int n_seg, int max_seg_len) {
    if (n_seg <= 0 || max_seg_len < 0) return 0;
    return trim_ws(n_seg, max_seg_len, nullptr).bytes;
}

extern "C" int ncfa_trim_bounds_batched(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len,
                                        int n_seg, int max_seg_len, double top_db, int64_t *d_bounds, void *d_workspace,
                                        size_t workspace_bytes, void *stream) {
    NCFA_REQUIRE(n_seg >= 0 && n_seg <= 65535, "n_seg must be in [0, 65535] per call");
    if (n_seg == 0) return NCFA_OK;
    NCFA_REQUIRE(d_audio && d_seg_off && d_seg_len && d_bounds && d_workspace, "null pointer");
    NCFA_REQUIRE(max_seg_len >= 0, "max_seg_len");
    const TrimWs w = trim_ws(n_seg, max_seg_len, d_workspace);
    if (int rc = check_workspace("trim", workspace_bytes, w.bytes)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = launch("trim_blocksum_kernel", trim_blocksum_kernel, dim3((w.stride + 7) / 8, n_seg), 256, 0, st,
                        d_audio, d_seg_off, d_seg_len, w.stride, w.bsum))
        return rc;
    return launch("trim_bounds_kernel", trim_bounds_kernel, n_seg, 256, 0, st, d_seg_len, w.stride, w.bsum,
                  (float)top_db, d_bounds);
}
