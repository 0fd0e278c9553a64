// Framing → Hann → real FFT-2048 → |.|^2 → Slaney mel(128) → dB  (kernel 1)
// and top_db clamp → positive flux → mean over mels → onset envelope (kernel 2).
//
// Replaces librosa.onset.onset_strength as called at tempo.py:44 (hop 512, one 10 s window per
// segment) and tempo.py:158 (hop 64, whole track per segment).  SURVEY.md Appendix A.1/A.2.
//
// Kernel 1 layout: persistent CTAs, one per SM; the constant tables (Hann, W_1024 twiddles, lane-transposed mel bank)
// are staged in shared memory once per CTA.  **One warp = one pair of frames** (2p, 2p+1) of a segment: the warp loads
// their samples straight from global memory (coalesced float2; consecutive pairs are handled by the warps of one SM at
// the same time, so L1 serves the 97 % overlap at hop 64), packs each frame as 1024 complex values (lane n2 holds
// z[32·n1+n2] in registers), runs a 32-point FFT over n1, multiplies by W_1024^(n2·k1), transposes through a padded
// per-warp shared tile, runs the second 32-point FFT and un-packs the real spectrum with one shuffle per complex value
// (stft_core.cuh: warp_power_spectrum_global2).  Both frames go through one instruction stream: the Hann window, the
// W_1024 twiddles, W_2048^k and the mel weights are read from shared memory once per pair, and at hop 64 the two frames
// share 31 of their 32 register loads.  The power spectra go through the same per-warp tiles into the sparse mel
// projection (lane owns bands l, 63−l, 64+l, 127−l; weights are stored lane-transposed so the reads are bank-conflict
// free).  No block-level synchronisation in the loop.  Measured on B200 (round 1/2, profiles/): the pair form needs ~340
// shared-memory/L1 wavefronts per frame against 510 for one frame per warp, and its wider register budget removes the
// spills of that form; a CTA-wide tile form (lane = frame in the mel phase) was 7–19 % slower and latency bound.
#include "stft_core.cuh"

namespace ncfa {

constexpr int kWarps2Max = 12;  // 168 registers per thread × 384 threads fill the register file
constexpr size_t kScrBytes2 = 2 * 32 * kScrStride * sizeof(float2);  // two transpose tiles per warp

// dynamic shared memory: [hann 8 KB][tw 8 KB][lane_bin0 512 B][mel weights rows·128 B][scr: warps × 16.5 KB]
__host__ __device__ inline size_t onset2_fixed_bytes(int mel_rows) { return 8192 + 8192 + 512 + (size_t)mel_rows * 128; }

template <int SHIFT>
__global__ void __launch_bounds__(kWarps2Max * 32, 1) stft_logmel2_kernel(const float *__restrict__ audio,
                                                                    const int64_t *__restrict__ seg_off,
                                                                    const int32_t *__restrict__ seg_len, int n_seg,
                                                                    int hop, int frame_stride, Tables tb,
                                                                    float *__restrict__ S, unsigned *__restrict__ seg_max) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    struct {
        float *hann;
        float2 *tw;
        int *lane_bin0;
        float *melwt;
    } sm;
    sm.hann = reinterpret_cast<float *>(smem_raw);
    sm.tw = reinterpret_cast<float2 *>(smem_raw + 8192);
    sm.lane_bin0 = reinterpret_cast<int *>(smem_raw + 16384);
    sm.melwt = reinterpret_cast<float *>(smem_raw + 16896);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int kThreads2 = blockDim.x, kWarps2 = blockDim.x >> 5;
    for (int i = tid; i < 2048; i += kThreads2) sm.hann[i] = tb.hann[i];
    for (int i = tid; i < 1024; i += kThreads2) sm.tw[i] = tb.tw1024[i];
    for (int i = tid; i < tb.mel_wt_rows * 32; i += kThreads2) sm.melwt[i] = tb.mel_wt[i];
    for (int i = tid; i < 4 * 32; i += kThreads2) sm.lane_bin0[i] = tb.mel_lane_bin0[i];
    __syncthreads();

    const cf twl = cf{tb.tw2048[lane].x, tb.tw2048[lane].y};
    float2 *scra = reinterpret_cast<float2 *>(smem_raw + onset2_fixed_bytes(tb.mel_wt_rows) + (size_t)warp * kScrBytes2);
    float2 *scrb = scra + 32 * kScrStride;
    const float *pa = reinterpret_cast<const float *>(scra), *pb = reinterpret_cast<const float *>(scrb);
    int b0[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) b0[q] = sm.lane_bin0[q * 32 + lane];
    const int pair_stride = (frame_stride + 1) >> 1;
    const int64_t total = (int64_t)n_seg * pair_stride;
    int cur_seg = -1;
    float cur_max = -INFINITY;
    // items (seg, frame pair) are dealt in groups of kWarps2 consecutive pairs per CTA (2·kWarps2 consecutive frames:
    // L1 serves the overlap between them)
    for (int64_t item = (int64_t)blockIdx.x * kWarps2 + warp; item < total; item += (int64_t)gridDim.x * kWarps2) {
        const int seg = (int)(item / pair_stride);
        const int fa = 2 * (int)(item - (int64_t)seg * pair_stride);
        const int len = seg_len[seg];
        const int n_frames = 1 + len / hop;
        if (fa >= n_frames) continue;
        const bool b_valid = fa + 1 < n_frames;
        if (seg != cur_seg) {
            if (cur_seg >= 0 && lane == 0) atomicMax(seg_max + cur_seg, float_to_ordered(cur_max));
            cur_seg = seg;
            cur_max = -INFINITY;
        }
        warp_power_spectrum_global2<SHIFT>(audio + seg_off[seg], (int64_t)fa * hop - 1024, hop, len, b_valid, sm.hann,
                                           sm.tw, scra, scrb, twl, lane);
        float *Sa = S + ((size_t)seg * frame_stride + fa) * NCFA_N_MELS;
        float vmax = -INFINITY;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float *wt = sm.melwt + (size_t)tb.mel_qoff[q] * 32 + lane;
            const float *ka = pa + b0[q], *kb = pb + b0[q];
            const int nw = tb.mel_qw[q];
            float acca = 0.0f, accb = 0.0f;
            for (int i = 0; i < nw; ++i) {  // zero weights beyond the band's support
                const float w = wt[i * 32];
                acca = fmaf(w, ka[i], acca);
                accb = fmaf(w, kb[i], accb);
            }
            // the pair form stores 4·|X|² (stft_core.cuh PostStage2): exact ¼ here
            const float dba = 10.0f * log10f(fmaxf(1e-10f, 0.25f * acca));
            const float dbb = 10.0f * log10f(fmaxf(1e-10f, 0.25f * accb));
            const int band = mel_band_of(q, lane);
            Sa[band] = dba;
            vmax = fmaxf(vmax, dba);
            if (b_valid) {
                Sa[NCFA_N_MELS + band] = dbb;
                vmax = fmaxf(vmax, dbb);
            }
        }
        cur_max = fmaxf(cur_max, warp_max(vmax));
        __syncwarp();
    }
    if (cur_seg >= 0 && lane == 0) atomicMax(seg_max + cur_seg, float_to_ordered(cur_max));
}

// onset[j] = 0 for j < pad;  else mean_m relu(clamp(S[j-pad+1][m]) - clamp(S[j-pad][m]))
// A warp walks kFluxRun consecutive frames and keeps the previous log-mel row in registers, so every row is read from
// L2 once (the kernel is L2-bandwidth bound: 512 B per frame).  Per frame: 4 bands per lane, then the xor tree.
constexpr int kFluxRun = 8;
__global__ void __launch_bounds__(256) flux_kernel(const float *__restrict__ S, const unsigned *__restrict__ seg_max,
                                                   const int32_t *__restrict__ seg_len, int hop, int frame_stride,
                                                   int pad, float *__restrict__ onset,
                                                   const int64_t *__restrict__ onset_off) {
    const int seg = blockIdx.y;
    const int n_frames = 1 + seg_len[seg] / hop;
    const int lane = threadIdx.x & 31;
    const int j0 = (blockIdx.x * 8 + (threadIdx.x >> 5)) * kFluxRun;
    if (j0 >= n_frames) return;
    float *out = onset + onset_off[seg];
    const float floor_db = ordered_to_float(seg_max[seg]) - 80.0f;
    const float4 *rows = reinterpret_cast<const float4 *>(S + (size_t)seg * frame_stride * NCFA_N_MELS);
    const int j1 = min(n_frames, j0 + kFluxRun);
    int j = j0;
    for (; j < j1 && j < pad; ++j)
        if (lane == 0) out[j] = 0.0f;
    if (j >= j1) return;
    float4 a = rows[(size_t)(j - pad) * (NCFA_N_MELS / 4) + lane];
    a.x = fmaxf(a.x, floor_db);
    a.y = fmaxf(a.y, floor_db);
    a.z = fmaxf(a.z, floor_db);
    a.w = fmaxf(a.w, floor_db);
    for (; j < j1; ++j) {
        float4 b = rows[(size_t)(j - pad + 1) * (NCFA_N_MELS / 4) + lane];
        b.x = fmaxf(b.x, floor_db);
        b.y = fmaxf(b.y, floor_db);
        b.z = fmaxf(b.z, floor_db);
        b.w = fmaxf(b.w, floor_db);
        float s = fmaxf(0.0f, b.x - a.x);
        s += fmaxf(0.0f, b.y - a.y);
        s += fmaxf(0.0f, b.z - a.z);
        s += fmaxf(0.0f, b.w - a.w);
        s = warp_sum(s);
        if (lane == 0) out[j] = s * (1.0f / NCFA_N_MELS);
        a = b;
    }
}

// log-mel spectrogram S in whole tiles of 32 frames per segment, then one ordered-uint maximum per segment
struct OnsetWs {
    float *S;
    unsigned *seg_max;
    size_t bytes;
};

static OnsetWs onset_ws(int n_seg, int max_seg_len, int hop, void *base) {
    Carve c(base);
    OnsetWs w;
    const size_t frames = (1 + (size_t)max_seg_len / hop + 31) / 32 * 32;
    w.S = c.take<float>((size_t)n_seg * frames * NCFA_N_MELS);
    w.seg_max = c.take<unsigned>(n_seg);
    w.bytes = c.used;
    return w;
}

}  // namespace ncfa

using namespace ncfa;

extern "C" size_t ncfa_onset_workspace_bytes(int n_seg, int max_seg_len, int hop) {
    if (n_seg <= 0 || hop <= 0 || max_seg_len < 0) return 0;
    return onset_ws(n_seg, max_seg_len, hop, nullptr).bytes;
}

extern "C" int ncfa_onset_strength_batched(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len,
                                           int n_seg, int max_seg_len, int hop, int sr, float *d_onset,
                                           const int64_t *d_onset_off, void *d_workspace, size_t workspace_bytes,
                                           void *stream) {
    NCFA_REQUIRE(n_seg >= 0 && n_seg <= 65535, "n_seg must be in [0, 65535] per call");
    if (n_seg == 0) return NCFA_OK;
    NCFA_REQUIRE(d_audio && d_seg_off && d_seg_len && d_onset && d_onset_off && d_workspace, "null pointer");
    NCFA_REQUIRE(hop >= 16 && hop <= 1024 && (hop % 2) == 0, "hop must be even and in [16, 1024]");
    NCFA_REQUIRE(max_seg_len >= 0, "max_seg_len");
    const OnsetWs w = onset_ws(n_seg, max_seg_len, hop, d_workspace);
    int rc = check_workspace("onset", workspace_bytes, w.bytes);
    if (rc) return rc;
    Tables tb;
    if ((rc = get_tables(sr, &tb))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int frames = 1 + max_seg_len / hop;
    NCFA_CUDA_OK(cudaMemsetAsync(w.seg_max, 0, (size_t)n_seg * 4, st));
    int n_sm = 0;
    if ((rc = sm_count(&n_sm))) return rc;
    // as many warps as the 227 KB of shared memory hold (12 at 22 050 Hz: 95 mel-weight rows)
    const size_t fixed = onset2_fixed_bytes(tb.mel_wt_rows);
    int warps = (int)((232448 - fixed) / kScrBytes2);
    if (warps > kWarps2Max) warps = kWarps2Max;
    NCFA_REQUIRE(warps >= 1, "mel table too large for shared memory");
    const size_t smem = fixed + (size_t)warps * kScrBytes2;
    const int64_t groups = ((int64_t)n_seg * ((frames + 1) / 2) + warps - 1) / warps;
    const int grid = (int)(groups < n_sm ? groups : n_sm);  // persistent: one CTA per SM
    auto logmel = hop == 64 ? stft_logmel2_kernel<1> : (hop == 512 ? stft_logmel2_kernel<8> : stft_logmel2_kernel<0>);
    if ((rc = launch(hop <= 128 ? "stft_logmel_kernel[hop<=128]" : "stft_logmel_kernel[hop>128]", logmel, grid,
                     warps * 32, smem, st, d_audio, d_seg_off, d_seg_len, n_seg, hop, frames, tb, w.S, w.seg_max)))
        return rc;
    const int pad = 1 + NCFA_N_FFT / (2 * hop);
    return launch("flux_kernel", flux_kernel, dim3((frames + 8 * kFluxRun - 1) / (8 * kFluxRun), n_seg), 256, 0, st,
                  w.S, w.seg_max, d_seg_len, hop, frames, pad, d_onset, d_onset_off);
}
