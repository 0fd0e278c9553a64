// Waveform cross-correlation speed search.  Replaces the candidate loop of
// xcorr.estimate_speed_xcorr (xcorr.py:113-148): for every reference window wa of track A and every
// candidate position pb = lo_b + j·stride of track B,
//     c = dot(wa, wb) / (‖wa‖·‖wb‖),
// the first strict maximum over j is kept (xcorr.py:142-144) when it is > 0 (xcorr.py:146).
// The reference is NOT FFT based (SURVEY.md §0.3): the observable result is the argmax on the
// strided candidate grid, so that grid is what is evaluated here.
//
// This family is memory bound (0.5 flop/B).  The reference's stride is win // 4 (xcorr.py:104), so
// the search span of a window is a run of stride-long BLOCKS of B and candidate j is blocks
// j .. j+3 (plus a tail of win − 4·stride <= 3 samples): with D[q][m] = <A block q, B block m> and
// S[m] = ‖B block m‖²,
//     dot(wa, wb_j) = D[0][j] + D[1][j+1] + D[2][j+2] + D[3][j+3] (+ tail),   ‖wb_j‖² = S[j] + ... + S[j+3] (+ tail).
// xcorr_blocks_ring_kernel gives a CTA one window and G = 8 consecutive B blocks; a consumer thread walks the
// sample index i, keeps the 8 x 5 partial sums of its blocks in registers and reads the four A samples of
// index i once for all of them — every B sample is read from HBM ONCE and used in five float64 FMAs,
// every A sample once per CTA of its window (L2).  The tiles reach shared memory through a ring of 1-D TMA
// bulk copies issued by a producer warp (see the kernel).  xcorr_pick_blocks_kernel adds the partials in
// a fixed order (deterministic) and scans the candidates.  Sums are float64 (the float32 inputs are
// exact in float64; the reference's float32 BLAS sums differ from these by rounding only).
// The general (win, stride) case of the C ABI — more than 4 blocks per window — keeps the direct
// kernel (one CTA per (window, candidate)).
#include "ncfa_common.cuh"
#include "tc05.cuh"

namespace ncfa {

constexpr int kXcThreads = 256;

__device__ __forceinline__ double block_sum_256(double v, double *sh) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0) {
        for (int w = 0; w < kXcThreads / 32; ++w) s += sh[w];
        sh[0] = s;
    }
    __syncthreads();
    s = sh[0];
    __syncthreads();
    return s;
}

// grid (max_cand + 1, n_windows): blockIdx.x == max_cand computes ‖wa‖² (and the RMS gate input)
__global__ void __launch_bounds__(kXcThreads) xcorr_dots_kernel(const float *__restrict__ a, const float *__restrict__ b,
                                                                 const int64_t *__restrict__ a_pos,
                                                                 const int64_t *__restrict__ b_lo,
                                                                 const int32_t *__restrict__ n_cand, int max_cand,
                                                                 int win, int stride, double *__restrict__ dots,
                                                                 double *__restrict__ nb2, double *__restrict__ na2) {
    __shared__ double sh[kXcThreads / 32];
    const int w = blockIdx.y;
    const int j = blockIdx.x;
    const float *wa = a + a_pos[w];
    if (j == max_cand) {
        double acc = 0.0;
        for (int i = threadIdx.x; i < win; i += kXcThreads) {
            const double x = (double)__ldg(wa + i);
            acc = fma(x, x, acc);
        }
        acc = block_sum_256(acc, sh);
        if (threadIdx.x == 0) na2[w] = acc;
        return;
    }
    if (j >= n_cand[w]) return;
    const float *wb = b + b_lo[w] + (int64_t)j * stride;
    double d0 = 0.0, d1 = 0.0, q0 = 0.0, q1 = 0.0;
    int i = threadIdx.x;
    for (; i + kXcThreads < win; i += 2 * kXcThreads) {
        const double x0 = (double)__ldg(wa + i), y0 = (double)__ldg(wb + i);
        const double x1 = (double)__ldg(wa + i + kXcThreads), y1 = (double)__ldg(wb + i + kXcThreads);
        d0 = fma(x0, y0, d0);
        q0 = fma(y0, y0, q0);
        d1 = fma(x1, y1, d1);
        q1 = fma(y1, y1, q1);
    }
    if (i < win) {
        const double x0 = (double)__ldg(wa + i), y0 = (double)__ldg(wb + i);
        d0 = fma(x0, y0, d0);
        q0 = fma(y0, y0, q0);
    }
    const double d = block_sum_256(d0 + d1, sh);
    const double q = block_sum_256(q0 + q1, sh);
    if (threadIdx.x == 0) {
        dots[(size_t)w * max_cand + j] = d;
        nb2[(size_t)w * max_cand + j] = q;
    }
}

// ---- block form: stride-long blocks of B, nq = win / stride <= 4 of them per candidate ----------------------------------
constexpr int kMaxPieces = 4;      // A blocks per window (win / stride)

// ---- ring form: the tiles of a CTA stream through a ring with full / empty mbarriers and a producer warp ---------------
// History of this kernel on B200 (config 4, 16 pairs, algorithmic bytes per second; profiles/README.md has the files):
//   one CTA per (window, candidate), scalar loads (round 1)                                             0.35 TB/s
//   block form, register loads (8 in flight per thread: long-scoreboard bound)                          1.1
//   block form, 3-stage TMA ring, one lane computes byte counts and issues all copies, __syncthreads    2.6
//     (ncu r2f: a third of all stall samples behind that barrier — the issuing lane's serial path)
//   producer warp (lane t owns tile t), full / empty mbarriers, 512-sample chunks = 2 KB copies         1.5
//     (the SM's copy engine has a fixed cost per bulk copy: 2 KB copies sustain 16 B/clk/SM, 4 KB 25 —
//      profiles/r2k_tma_bulk_copy_bandwidth.log)
//   same with 8 KB copies, 4 B blocks per CTA                                                           2.6
//   8 B blocks per CTA (the A re-reads drop from 1/2 to 1/3 of the bytes), 4 KB copies, 4 stages        2.7
//   + the CTA's 41 sums reduced through the idle ring memory with two barriers instead of 123           3.0
// Not kept: A blocks through registers with only B in the ring (2.45), two CTAs per SM at 112 registers (1.95).
// Nothing is CTA-wide inside the loop: the last warp only produces (eight..twelve lanes issue the bulk copies of a stage
// in parallel, from pointers computed once), the other warps only consume (wait full → shared loads + float64 FMAs → one
// arrive per warp on the stage's empty barrier).
// G = B blocks per CTA.  The A blocks are re-read by every CTA of a window, so the bytes a CTA pulls through the copy
// engine are (NQ + G) / G times its algorithmic share: 2x at G = 4, 1.5x at G = 8 (40 float64 accumulators per thread).
template <int NQ, int G, int CHUNK, int STAGES, int CONSUMERS>
struct XrSmem {
    float tile[STAGES][NQ + G][CHUNK + 8];
    uint64_t full[STAGES], empty[STAGES];
};

template <int NQ, int G, int CHUNK, int STAGES, int CONSUMERS>
__global__ void __launch_bounds__(CONSUMERS + 32, 1) xcorr_blocks_ring_kernel(const float *__restrict__ a,
                                                                       const float *__restrict__ b,
                                                                       const int64_t *__restrict__ a_pos,
                                                                       const int64_t *__restrict__ b_lo,
                                                                       const int32_t *__restrict__ n_cand, int max_blocks,
                                                                       int win, int stride, double *__restrict__ part,
                                                                       double *__restrict__ na2) {
    using namespace tc05;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    XrSmem<NQ, G, CHUNK, STAGES, CONSUMERS> &sm = *reinterpret_cast<XrSmem<NQ, G, CHUNK, STAGES, CONSUMERS> *>(smem_raw);
    const int w = blockIdx.y;
    const int nc = n_cand[w];
    if (nc <= 0 && blockIdx.x != 0) return;
    const int n_blocks = nc > 0 ? nc + NQ - 1 : 0;
    const int m0 = blockIdx.x * G;
    if (m0 >= n_blocks && blockIdx.x != 0) return;
    const float *wa = a + a_pos[w];
    const float *wb = b + b_lo[w] + (int64_t)m0 * stride;
    const int live = max(0, min(G, n_blocks - m0));
    const int n_tiles = NQ + live;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&sm.full[s], 1);
            mbar_init(&sm.empty[s], CONSUMERS / 32);
        }
        fence_mbar_init();
    }
    __syncthreads();
    const int n_chunks = (stride + CHUNK - 1) / CHUNK;

    if (warp == CONSUMERS / 32) {
        // ===================== producer warp: lane t streams tile t (A blocks 0..NQ-1, then the CTA's B blocks) =====================
        const float *base = lane < NQ ? wa + (int64_t)lane * stride : wb + (int64_t)(lane - NQ) * stride;
        const int o = (int)((reinterpret_cast<uintptr_t>(base) & 15u) >> 2);   // offset inside the 16-byte aligned superset
        for (int c = 0; c < n_chunks; ++c) {
            const int st = c % STAGES;
            if (c >= STAGES) mbar_wait_warp(&sm.empty[st], (uint32_t)((c / STAGES - 1) & 1), 20);
            const int i0 = c * CHUNK;
            const int len = min(CHUNK, stride - i0);
            const uint32_t bytes = lane < n_tiles ? (uint32_t)((o + len + 3) & ~3) * 4u : 0u;
            uint32_t total = bytes;
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) total += __shfl_xor_sync(0xffffffffu, total, d);
            if (lane == 0) mbar_arrive_expect_tx(&sm.full[st], total);
            __syncwarp();
            if (lane < n_tiles) bulk_g2s(&sm.tile[st][lane][0], base + i0 - o, bytes, &sm.full[st]);
        }
        return;
    }

    // ===================== consumer warps =====================
    int off[NQ + G];
#pragma unroll
    for (int t = 0; t < NQ + G; ++t) {
        const float *base = t < NQ ? wa + (int64_t)t * stride : wb + (int64_t)(t - NQ) * stride;
        off[t] = (int)((reinterpret_cast<uintptr_t>(base) & 15u) >> 2);
    }
    double d[G][NQ], s2[G], sa = 0.0;
#pragma unroll
    for (int g = 0; g < G; ++g) {
        s2[g] = 0.0;
#pragma unroll
        for (int q = 0; q < NQ; ++q) d[g][q] = 0.0;
    }
    for (int c = 0; c < n_chunks; ++c) {
        const int st = c % STAGES;
        mbar_wait_warp(&sm.full[st], (uint32_t)(c / STAGES) & 1u);
        const int len = min(CHUNK, stride - c * CHUNK);
        if (live == G) {
#pragma unroll
            for (int k = 0; k < CHUNK / CONSUMERS; ++k) {
                const int i = tid + k * CONSUMERS;
                if (i < len) {
                    double x[NQ], y[G];
#pragma unroll
                    for (int q = 0; q < NQ; ++q) x[q] = (double)sm.tile[st][q][off[q] + i];
#pragma unroll
                    for (int g = 0; g < G; ++g) y[g] = (double)sm.tile[st][NQ + g][off[NQ + g] + i];
#pragma unroll
                    for (int g = 0; g < G; ++g) {
                        s2[g] = fma(y[g], y[g], s2[g]);
#pragma unroll
                        for (int q = 0; q < NQ; ++q) d[g][q] = fma(x[q], y[g], d[g][q]);
                    }
                    if (blockIdx.x == 0) {
#pragma unroll
                        for (int q = 0; q < NQ; ++q) sa = fma(x[q], x[q], sa);
                    }
                }
            }
        } else {
#pragma unroll
            for (int k = 0; k < CHUNK / CONSUMERS; ++k) {
                const int i = tid + k * CONSUMERS;
                if (i < len) {
                    double x[NQ];
#pragma unroll
                    for (int q = 0; q < NQ; ++q) x[q] = (double)sm.tile[st][q][off[q] + i];
#pragma unroll
                    for (int g = 0; g < G; ++g) {
                        if (g < live) {
                            const double y = (double)sm.tile[st][NQ + g][off[NQ + g] + i];
                            s2[g] = fma(y, y, s2[g]);
#pragma unroll
                            for (int q = 0; q < NQ; ++q) d[g][q] = fma(x[q], y, d[g][q]);
                        }
                    }
                    if (blockIdx.x == 0) {
#pragma unroll
                        for (int q = 0; q < NQ; ++q) sa = fma(x[q], x[q], sa);
                    }
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.empty[st]);   // this warp is done reading the stage
    }
    // ---- the CTA's (G·(NQ+1) + 1) sums: per-thread partials go through the (now idle) ring memory, then warp v sums
    // column v in a fixed order — two barriers instead of three per value (the per-value block reductions were 10 % of
    // the kernel's stall samples, with the copy pipeline drained)
    constexpr int NV = G * (NQ + 1) + 1;
    static_assert((size_t)NV * CONSUMERS * sizeof(double) <= sizeof(sm.tile), "reduction scratch must fit in the ring");
    double *red = reinterpret_cast<double *>(&sm.tile[0][0][0]);
    asm volatile("bar.sync 1, %0;" ::"n"(CONSUMERS) : "memory");  // every consumer is through with the ring
#pragma unroll
    for (int g = 0; g < G; ++g) {
#pragma unroll
        for (int q = 0; q < NQ; ++q) red[(size_t)(g * (NQ + 1) + q) * CONSUMERS + tid] = d[g][q];
        red[(size_t)(g * (NQ + 1) + NQ) * CONSUMERS + tid] = s2[g];
    }
    if (blockIdx.x == 0) {
        // the tail samples [NQ·stride, win) of wa belong to ‖wa‖² too
        for (int i = NQ * stride + tid; i < win; i += CONSUMERS) {
            const double x = (double)__ldg(wa + i);
            sa = fma(x, x, sa);
        }
    }
    red[(size_t)(NV - 1) * CONSUMERS + tid] = sa;
    asm volatile("bar.sync 1, %0;" ::"n"(CONSUMERS) : "memory");
    double *pw = part + (size_t)w * (kMaxPieces + 1) * max_blocks;
    for (int v = warp; v < NV; v += CONSUMERS / 32) {
        double acc = 0.0;
        for (int t = lane; t < CONSUMERS; t += 32) acc += red[(size_t)v * CONSUMERS + t];
        acc = warp_sum(acc);
        if (lane == 0) {
            if (v == NV - 1) {
                if (blockIdx.x == 0) na2[w] = acc;
            } else {
                const int g = v / (NQ + 1), q = v - g * (NQ + 1);
                if (g < live) pw[(size_t)(q == NQ ? kMaxPieces : q) * max_blocks + m0 + g] = acc;
            }
        }
    }
}

// one warp per window: candidate sums from the block partials (fixed order), then the same gates and scan as below
__global__ void __launch_bounds__(32) xcorr_pick_blocks_kernel(const float *__restrict__ a, const float *__restrict__ b,
                                                               const int64_t *__restrict__ a_pos,
                                                               const int64_t *__restrict__ b_lo,
                                                               const int32_t *__restrict__ n_cand, int max_blocks, int nq,
                                                               int win, int stride, double rms_gate,
                                                               const double *__restrict__ part,
                                                               const double *__restrict__ na2,
                                                               int32_t *__restrict__ best_j, double *__restrict__ best_c) {
    const int w = blockIdx.x;
    const int lane = threadIdx.x;
    const int nc = n_cand[w];
    const double *pw = part + (size_t)w * (kMaxPieces + 1) * max_blocks;
    const float *wa = a + a_pos[w];
    const float *wb = b + b_lo[w];
    const float rms_a = (float)sqrt(na2[w] / (double)win);
    const float norm_a32 = (float)sqrt(na2[w]);
    const double norm_a = (double)norm_a32;
    int bj = -1;
    double bc = -1.0;  // best_corr starts at -1.0 (xcorr.py:130)
    if (!((double)rms_a < rms_gate) && !(norm_a < 1e-10)) {
        for (int j = lane; j < nc; j += 32) {
            double dot = 0.0, nb2 = 0.0;
            for (int q = 0; q < nq; ++q) {
                dot += pw[(size_t)q * max_blocks + j + q];
                nb2 += pw[(size_t)kMaxPieces * max_blocks + j + q];
            }
            for (int i = nq * stride; i < win; ++i) {  // win − nq·stride < stride tail samples (<= 3 on the reference's grid)
                const double x = (double)__ldg(wa + i), y = (double)__ldg(wb + (int64_t)j * stride + i);
                dot = fma(x, y, dot);
                nb2 = fma(y, y, nb2);
            }
            const double norm_b = (double)(float)sqrt(nb2);
            if (norm_b < 1e-10) continue;
            const double c = (double)(float)dot / (norm_a * norm_b);  // np.dot is float32; float32 / float64 → float64
            if (c > bc) {
                bc = c;
                bj = j;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double oc = __shfl_xor_sync(0xffffffffu, bc, o);
        const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
        if (oj >= 0 && (bj < 0 || oc > bc || (oc == bc && oj < bj))) {
            bc = oc;
            bj = oj;
        }
    }
    if (lane == 0) {
        const bool keep = bj >= 0 && bc > 0.0;  // xcorr.py:146
        best_j[w] = keep ? bj : -1;
        best_c[w] = keep ? bc : 0.0;
    }
}

// one warp per window: the gates of xcorr.py:118-131 and the first-maximum scan of :133-148
__global__ void __launch_bounds__(32) xcorr_pick_kernel(const int32_t *__restrict__ n_cand, int max_cand, int win,
                                                        double rms_gate, const double *__restrict__ dots,
                                                        const double *__restrict__ nb2, const double *__restrict__ na2,
                                                        int32_t *__restrict__ best_j, double *__restrict__ best_c) {
    const int w = blockIdx.x;
    const int lane = threadIdx.x;
    const int nc = n_cand[w];
    // xcorr.py:118 computes sqrt(mean(wa²)) and :127 ‖wa‖ in float32; compare the float32-rounded values
    const float rms_a = (float)sqrt(na2[w] / (double)win);
    const float norm_a32 = (float)sqrt(na2[w]);
    const double norm_a = (double)norm_a32;
    int bj = -1;
    double bc = -1.0;  // best_corr starts at -1.0 (xcorr.py:130)
    if (!((double)rms_a < rms_gate) && !(norm_a < 1e-10)) {
        for (int j = lane; j < nc; j += 32) {
            const double norm_b = (double)(float)sqrt(nb2[(size_t)w * max_cand + j]);
            if (norm_b < 1e-10) continue;
            // np.dot(wa, wb) is float32; float32 / float64 → float64
            const double c = (double)(float)dots[(size_t)w * max_cand + j] / (norm_a * norm_b);
            if (c > bc) {  // ascending j per lane: strict > keeps the lane's first maximum
                bc = c;
                bj = j;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double oc = __shfl_xor_sync(0xffffffffu, bc, o);
        const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
        if (oj >= 0 && (bj < 0 || oc > bc || (oc == bc && oj < bj))) {
            bc = oc;
            bj = oj;
        }
    }
    if (lane == 0) {
        const bool keep = bj >= 0 && bc > 0.0;  // xcorr.py:146
        best_j[w] = keep ? bj : -1;
        best_c[w] = keep ? bc : 0.0;
    }
}


// ---------------------------------------------------------------------------------------------------------------
// Intro alignment (xcorr.find_content_offset, xcorr.py:165-259): for each candidate speed the nightcore RMS
// envelope is stretched by linear interpolation (np.interp over two np.linspace grids), correlated against
// the source envelope over the first n_lag lags (np.correlate 'valid'), and the peak is cosine-normalised.

// plain 2:1 decimation (librosa.resample(orig_sr = 2·target_sr) stand-in; same half-band FIR as the CQT path,
// no √2 scale): out[i] = float32(Σ_k h[k]·in[2i + k − 63]), n_out = ceil(n/2)
__global__ void __launch_bounds__(256) align_decimate2_kernel(const float *__restrict__ in, int64_t n_in,
                                                              float *__restrict__ out, int64_t n_out,
                                                              const double *__restrict__ hb) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n_out) return;
    double acc = 0.0;
    for (int k = 0; k < 127; ++k) {
        const int64_t p = 2 * i + k - 63;
        if (p >= 0 && p < n_in) acc = fma(__ldg(hb + k), (double)__ldg(in + p), acc);
    }
    out[i] = (float)acc;
}

__global__ void __launch_bounds__(256) f32_to_f64_kernel(const float *__restrict__ in, int64_t n, double *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i < n) out[i] = (double)in[i];
}

// np.linspace(0, 1, n)[i]
__device__ __forceinline__ double lin01(int i, int n, double step) { return (i == n - 1) ? 1.0 : __dmul_rn((double)i, step); }

// stretched[s][i] = np.interp(linspace(0,1,ns)[i], linspace(0,1,n_nc), nc_env)
__global__ void __launch_bounds__(256) align_stretch_kernel(const double *__restrict__ nc_env, int n_nc,
                                                            const int32_t *__restrict__ n_str, int str_stride,
                                                            double *__restrict__ stretched) {
    const int sp = blockIdx.y;
    const int ns = n_str[sp];
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= ns) return;
    const double step_o = __ddiv_rn(1.0, (double)(n_nc - 1)), step_n = __ddiv_rn(1.0, (double)(ns - 1));
    const double x = lin01(i, ns, step_n);
    // largest j with xp[j] <= x
    int lo = 0, hi = n_nc - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (lin01(mid, n_nc, step_o) <= x) lo = mid; else hi = mid - 1;
    }
    const int j = lo;
    double r;
    const double xj = lin01(j, n_nc, step_o);
    if (j >= n_nc - 1 || xj == x) {
        r = nc_env[j >= n_nc - 1 ? n_nc - 1 : j];
    } else {
        const double slope = __ddiv_rn(__dsub_rn(nc_env[j + 1], nc_env[j]), __dsub_rn(lin01(j + 1, n_nc, step_o), xj));
        r = __dadd_rn(__dmul_rn(slope, __dsub_rn(x, xj)), nc_env[j]);
    }
    stretched[(size_t)sp * str_stride + i] = r;
}

// corr[s][l] = Σ_j src[l + j]·stretched[s][j]   (one CTA per (lag, speed))
__global__ void __launch_bounds__(kXcThreads) align_corr_kernel(const double *__restrict__ src_env,
                                                                const double *__restrict__ stretched, int str_stride,
                                                                const int32_t *__restrict__ n_str,
                                                                const int32_t *__restrict__ n_lag, int lag_stride,
                                                                double *__restrict__ corr) {
    __shared__ double sh[kXcThreads / 32];
    const int sp = blockIdx.y, l = blockIdx.x;
    if (l >= n_lag[sp]) return;
    const int ns = n_str[sp];
    const double *q = stretched + (size_t)sp * str_stride;
    double acc = 0.0;
    for (int j = threadIdx.x; j < ns; j += kXcThreads) acc = fma(src_env[l + j], q[j], acc);
    acc = block_sum_256(acc, sh);
    if (threadIdx.x == 0) corr[(size_t)sp * lag_stride + l] = acc;
}

// per speed: first argmax, window / query energies, cosine score (xcorr.py:242-252)
__global__ void __launch_bounds__(kXcThreads) align_pick_kernel(const double *__restrict__ src_env,
                                                                const double *__restrict__ stretched, int str_stride,
                                                                const int32_t *__restrict__ n_str,
                                                                const int32_t *__restrict__ n_lag, int lag_stride,
                                                                const double *__restrict__ corr,
                                                                int32_t *__restrict__ peak_idx, double *__restrict__ score) {
    __shared__ double sh[kXcThreads / 32];
    __shared__ double s_val[kXcThreads];
    __shared__ int s_idx[kXcThreads];
    const int sp = blockIdx.x;
    const int L = n_lag[sp], ns = n_str[sp];
    if (L <= 0) {
        if (threadIdx.x == 0) {
            peak_idx[sp] = -1;
            score[sp] = 0.0;
        }
        return;
    }
    double bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int l = threadIdx.x; l < L; l += kXcThreads) {
        const double v = corr[(size_t)sp * lag_stride + l];
        if (v > bv) {
            bv = v;
            bi = l;
        }
    }
    s_val[threadIdx.x] = bv;
    s_idx[threadIdx.x] = bi;
    __syncthreads();
    for (int o = kXcThreads / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            const double v2 = s_val[threadIdx.x + o];
            const int i2 = s_idx[threadIdx.x + o];
            if (v2 > s_val[threadIdx.x] || (v2 == s_val[threadIdx.x] && i2 < s_idx[threadIdx.x])) {
                s_val[threadIdx.x] = v2;
                s_idx[threadIdx.x] = i2;
            }
        }
        __syncthreads();
    }
    const int pk = s_idx[0] == 0x7fffffff ? 0 : s_idx[0];
    const double pv = s_val[0];
    __syncthreads();
    double we = 0.0, qe = 0.0;
    const double *q = stretched + (size_t)sp * str_stride;
    for (int j = threadIdx.x; j < ns; j += kXcThreads) {
        const double a = src_env[pk + j], b = q[j];
        we = fma(a, a, we);
        qe = fma(b, b, qe);
    }
    we = block_sum_256(we, sh);
    qe = block_sum_256(qe, sh);
    if (threadIdx.x == 0) {
        const double denom = sqrt(we * qe);
        peak_idx[sp] = pk;
        score[sp] = denom > 1e-12 ? pv / denom : 0.0;
    }
}

// launch shape of the block form (the last line of the table above): G = 8 B blocks per CTA, 1024-sample chunks (4 KB
// copies), 4 stages, 8 consumer warps
constexpr int kXrG = 8, kXrChunk = 1024, kXrStages = 4, kXrConsumers = 256;
template <int NQ>
using XrSmemT = XrSmem<NQ, kXrG, kXrChunk, kXrStages, kXrConsumers>;
template <int NQ>
static void xr_kernel_for(decltype(&xcorr_blocks_ring_kernel<1, kXrG, kXrChunk, kXrStages, kXrConsumers>) *kfn,
                          size_t *smem) {
    *kfn = xcorr_blocks_ring_kernel<NQ, kXrG, kXrChunk, kXrStages, kXrConsumers>;
    *smem = sizeof(XrSmemT<NQ>);
}

// block form: (kMaxPieces + 1) partial tables of max_cand + kMaxPieces − 1 blocks per window, then ‖a‖² per window
struct XcorrBlockWs {
    double *part, *na2;
    size_t bytes;
};

static XcorrBlockWs xcorr_block_ws(int n_windows, int max_cand, void *base) {
    Carve c(base);
    XcorrBlockWs w;
    w.part = c.take<double>((size_t)n_windows * (kMaxPieces + 1) * (max_cand + kMaxPieces - 1));
    w.na2 = c.take<double>(n_windows);
    w.bytes = c.used;
    return w;
}

// direct form: dot product and ‖b‖² per candidate, then ‖a‖² per window
struct XcorrDirectWs {
    double *dots, *nb2, *na2;
    size_t bytes;
};

static XcorrDirectWs xcorr_direct_ws(int n_windows, int max_cand, void *base) {
    Carve c(base);
    XcorrDirectWs w;
    w.dots = c.take<double>((size_t)n_windows * max_cand);
    w.nb2 = c.take<double>((size_t)n_windows * max_cand);
    w.na2 = c.take<double>(n_windows);
    w.bytes = c.used;
    return w;
}

}  // namespace ncfa

using namespace ncfa;

extern "C" size_t ncfa_xcorr_workspace_bytes(int n_windows, int max_cand) {
    if (n_windows <= 0 || max_cand <= 0) return 0;
    const size_t block = xcorr_block_ws(n_windows, max_cand, nullptr).bytes;
    const size_t direct = xcorr_direct_ws(n_windows, max_cand, nullptr).bytes;
    return block > direct ? block : direct;
}

extern "C" int ncfa_xcorr_search_batched(const float *d_a, const float *d_b, const int64_t *d_a_pos,
                                         const int64_t *d_b_lo, const int32_t *d_n_cand, int n_windows, int max_cand,
                                         int win, int stride, double rms_gate, int32_t *d_best_j, double *d_best_c,
                                         void *d_workspace, size_t workspace_bytes, void *stream) {
    NCFA_REQUIRE(n_windows >= 0 && n_windows <= 65535, "n_windows must be in [0, 65535] per call");
    if (n_windows == 0) return NCFA_OK;
    NCFA_REQUIRE(d_a && d_b && d_a_pos && d_b_lo && d_n_cand && d_best_j && d_best_c && d_workspace, "null pointer");
    NCFA_REQUIRE(win > 0 && stride > 0 && max_cand > 0, "win/stride/max_cand");
    int rc = check_workspace("xcorr", workspace_bytes, ncfa_xcorr_workspace_bytes(n_windows, max_cand));
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int nq = win / stride;
    // the tail (win − nq·stride samples per candidate) is summed by one lane in the pick kernel: keep it short
    if (nq >= 1 && nq <= kMaxPieces && win - nq * stride <= 16) {
        const XcorrBlockWs w = xcorr_block_ws(n_windows, max_cand, d_workspace);
        const int max_blocks = max_cand + kMaxPieces - 1;
        decltype(&xcorr_blocks_ring_kernel<1, kXrG, kXrChunk, kXrStages, kXrConsumers>) kfn;
        size_t smem;
        switch (nq) {
            case 1: xr_kernel_for<1>(&kfn, &smem); break;
            case 2: xr_kernel_for<2>(&kfn, &smem); break;
            case 3: xr_kernel_for<3>(&kfn, &smem); break;
            default: xr_kernel_for<4>(&kfn, &smem); break;
        }
        if ((rc = launch("xcorr_blocks_kernel", kfn, dim3((max_cand + nq - 1 + kXrG - 1) / kXrG, n_windows),
                         kXrConsumers + 32, smem, st, d_a, d_b, d_a_pos, d_b_lo, d_n_cand, max_blocks, win, stride,
                         w.part, w.na2)))
            return rc;
        return launch("xcorr_pick_kernel", xcorr_pick_blocks_kernel, n_windows, 32, 0, st, d_a, d_b, d_a_pos, d_b_lo,
                      d_n_cand, max_blocks, nq, win, stride, rms_gate, w.part, w.na2, d_best_j, d_best_c);
    }
    const XcorrDirectWs w = xcorr_direct_ws(n_windows, max_cand, d_workspace);
    if ((rc = launch("xcorr_dots_kernel", xcorr_dots_kernel, dim3(max_cand + 1, n_windows), kXcThreads, 0, st, d_a, d_b,
                     d_a_pos, d_b_lo, d_n_cand, max_cand, win, stride, w.dots, w.nb2, w.na2)))
        return rc;
    return launch("xcorr_pick_kernel", xcorr_pick_kernel, n_windows, 32, 0, st, d_n_cand, max_cand, win, rms_gate,
                  w.dots, w.nb2, w.na2, d_best_j, d_best_c);
}

extern "C" int ncfa_decimate2(const float *d_in, int64_t n_in, float *d_out, void *stream) {
    NCFA_REQUIRE(d_in && d_out && n_in >= 0, "d_in/d_out/n_in");
    const int64_t n_out = (n_in + 1) / 2;
    if (n_out == 0) return NCFA_OK;
    const double *hb = nullptr;
    int rc = ncfa::get_halfband_device(&hb);
    if (rc) return rc;
    return launch("align_decimate2_kernel", align_decimate2_kernel, (unsigned)((n_out + 255) / 256), 256, 0,
                  (cudaStream_t)stream, d_in, n_in, d_out, n_out, hb);
}

extern "C" int ncfa_f32_to_f64(const float *d_in, int64_t n, double *d_out, void *stream) {
    NCFA_REQUIRE(d_in && d_out && n >= 0, "d_in/d_out/n");
    if (n == 0) return NCFA_OK;
    return launch("f32_to_f64_kernel", f32_to_f64_kernel, (unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream,
                  d_in, n, d_out);
}

// the stretched nc envelope of every speed, then its correlation at every lag
struct AlignWs {
    double *stretched, *corr;
    size_t bytes;
};

static AlignWs align_ws(int n_speeds, int max_stretched, int max_lags, void *base) {
    Carve c(base);
    AlignWs w;
    w.stretched = c.take<double>((size_t)n_speeds * max_stretched);
    w.corr = c.take<double>((size_t)n_speeds * max_lags);
    w.bytes = c.used;
    return w;
}

extern "C" size_t ncfa_align_workspace_bytes(int n_speeds, int max_stretched, int max_lags) {
    if (n_speeds <= 0 || max_stretched <= 0 || max_lags <= 0) return 0;
    return align_ws(n_speeds, max_stretched, max_lags, nullptr).bytes;
}

extern "C" int ncfa_align_search(const double *d_src_env, int n_src, const double *d_nc_env, int n_nc,
                                 const int32_t *d_n_stretched, const int32_t *d_n_lags, int n_speeds, int max_stretched,
                                 int max_lags, int32_t *d_peak_idx, double *d_score, void *d_workspace,
                                 size_t workspace_bytes, void *stream) {
    NCFA_REQUIRE(n_speeds >= 0 && n_speeds <= 65535, "n_speeds");
    if (n_speeds == 0) return NCFA_OK;
    NCFA_REQUIRE(d_src_env && d_nc_env && d_n_stretched && d_n_lags && d_peak_idx && d_score && d_workspace, "null pointer");
    NCFA_REQUIRE(n_src > 0 && n_nc > 1 && max_stretched >= 2 && max_lags > 0, "n_src/n_nc/max_stretched/max_lags");
    // per speed n_stretched[s] + n_lags[s] − 1 <= n_src by construction (xcorr.py:232: search_len <= n_src − n_stretched)
    const AlignWs w = align_ws(n_speeds, max_stretched, max_lags, d_workspace);
    int rc = check_workspace("align", workspace_bytes, w.bytes);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = launch("align_stretch_kernel", align_stretch_kernel, dim3((max_stretched + 255) / 256, n_speeds), 256, 0,
                     st, d_nc_env, n_nc, d_n_stretched, max_stretched, w.stretched)))
        return rc;
    if ((rc = launch("align_corr_kernel", align_corr_kernel, dim3(max_lags, n_speeds), kXcThreads, 0, st, d_src_env,
                     w.stretched, max_stretched, d_n_stretched, d_n_lags, max_lags, w.corr)))
        return rc;
    return launch("align_pick_kernel", align_pick_kernel, n_speeds, kXcThreads, 0, st, d_src_env, w.stretched,
                  max_stretched, d_n_stretched, d_n_lags, max_lags, w.corr, d_peak_idx, d_score);
}
