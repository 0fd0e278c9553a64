// Shared STFT core: one warp turns one 2048-sample frame (already in shared memory) into its
// 1025-bin power spectrum (periodic Hann, real FFT as a packed 1024-point complex FFT).
// Used by the onset front-end (stft_onset.cu) and the tuning estimator (chroma.cu).
#pragma once
#include "ncfa_common.cuh"
#include "fft_core.cuh"

namespace ncfa {

constexpr int kScrStride = 33;  // complex elements per row of the per-warp transpose tile

// a · W_64^K2,  W_64 = exp(-2πi/64), K2 < 32
template <int K2>
__device__ __forceinline__ cf mul_w64(cf a) {
    constexpr float C[32] = {
        1.00000000000000000000f,  0.99518472667219692873f,  0.98078528040323043058f,  0.95694033573220882438f,
        0.92387953251128673848f,  0.88192126434835504956f,  0.83146961230254523567f,  0.77301045336273699338f,
        0.70710678118654757274f,  0.63439328416364548779f,  0.55557023301960228867f,  0.47139673682599780857f,
        0.38268343236508983729f,  0.29028467725446233105f,  0.19509032201612833135f,  0.09801714032956077016f,
        0.0f,                     -0.09801714032956064526f, -0.19509032201612819257f, -0.29028467725446216452f,
        -0.38268343236508972627f, -0.47139673682599769755f, -0.55557023301960195560f, -0.63439328416364537677f,
        -0.70710678118654746172f, -0.77301045336273699338f, -0.83146961230254534669f, -0.88192126434835493853f,
        -0.92387953251128673848f, -0.95694033573220882438f, -0.98078528040323043058f, -0.99518472667219681771f};
    constexpr float S[32] = {
        0.0f,                    0.09801714032956060363f, 0.19509032201612824808f, 0.29028467725446233105f,
        0.38268343236508978178f, 0.47139673682599764204f, 0.55557023301960217765f, 0.63439328416364548779f,
        0.70710678118654746172f, 0.77301045336273699338f, 0.83146961230254523567f, 0.88192126434835493853f,
        0.92387953251128673848f, 0.95694033573220893540f, 0.98078528040323043058f, 0.99518472667219681771f,
        1.0f,                    0.99518472667219692873f, 0.98078528040323043058f, 0.95694033573220893540f,
        0.92387953251128673848f, 0.88192126434835504956f, 0.83146961230254545772f, 0.77301045336273710440f,
        0.70710678118654757274f, 0.63439328416364548779f, 0.55557023301960217765f, 0.47139673682599786408f,
        0.38268343236508989280f, 0.29028467725446238656f, 0.19509032201612860891f, 0.09801714032956082567f};
    if constexpr (K2 == 0) {
        return a;
    } else {
        return cmul_cs(a, C[K2], S[K2]);  // a · (c - i s)
    }
}

template <int K2>
struct PostStage {
    // Un-pack the real FFT from the packed complex one and store powers.  With E = ½(Z[k] + conj Z[N−k]),
    // O = (Z[k] − conj Z[N−k])/(2i), W = W_2048^k:  X[k] = E + W·O and X[1024−k] = conj(E − W·O), so one (E, W·O)
    // pair yields both bins: K2 runs over 0..15 only (k = lane + 32·K2 < 512), bin 512 is |Z[512]|².
    static __device__ __forceinline__ void run(const cf (&v)[32], int lane, cf twl, float *pw) {
        cf zk = v[br5(K2)];
        cf own = v[br5((32 - K2) & 31)];
        cf snd = v[br5(31 - K2)];
        int src = (32 - lane) & 31;
        cf p;
        p.x = __shfl_sync(0xffffffffu, snd.x, src);
        p.y = __shfl_sync(0xffffffffu, snd.y, src);
        if (lane == 0) p = own;
        cf e = cscale(cadd_conj(zk, p), 0.5f);            // ½(Z[k] + conj Z[N−k])
        cf o = cscale(cmul_mi(csub_conj(zk, p)), 0.5f);   // (Z[k] − conj Z[N−k]) / (2i)
        cf w = mul_w64<K2>(twl);  // W_2048^(lane + 32·K2)
        cf wo = cmul(o, w);
        cf x = cadd(e, wo);
        cf y = csub(e, wo);
        pw[lane + 32 * K2] = x.x * x.x + x.y * x.y;
        pw[1024 - lane - 32 * K2] = y.x * y.x + y.y * y.y;
        if constexpr (K2 + 1 < 16) PostStage<K2 + 1>::run(v, lane, twl, pw);
        if constexpr (K2 == 0) {
            if (lane == 0) {
                cf z = v[br5(16)];
                pw[512] = z.x * z.x + z.y * z.y;
            }
        }
    }
};


// v[n1] = windowed (x[64·n1 + 2·lane], x[64·n1 + 2·lane + 1]) on entry; on return the first 1025 floats of scr
// hold |X[k]|^2.  tw: [32][32] W_1024 twiddles (shared), scr: per-warp scratch of 32*kScrStride float2.
__device__ __forceinline__ void warp_power_spectrum_regs(cf (&v)[32], const float2 *tw, float2 *scr, cf twl, int lane) {
    fft32_dif(v);
#pragma unroll
    for (int k1 = 0; k1 < 32; ++k1) {
        float2 t = tw[k1 * 32 + lane];
        cf y = cmul(v[br5(k1)], cf{t.x, t.y});
        scr[k1 * kScrStride + lane] = make_float2(y.x, y.y);
    }
    __syncwarp();
#pragma unroll
    for (int n2 = 0; n2 < 32; ++n2) {
        float2 t = scr[lane * kScrStride + n2];
        v[n2] = cf{t.x, t.y};
    }
    __syncwarp();
    fft32_dif(v);
    PostStage<0>::run(v, lane, twl, reinterpret_cast<float *>(scr));
    __syncwarp();
}

// Frame straight from global memory (L1/L2 serve the overlap between frames): samples x[pos .. pos+2048) of a
// segment of `len` samples starting at `src`, zeros outside [0, len); hann: 2048 floats (shared).
__device__ __forceinline__ void warp_power_spectrum_global(const float *__restrict__ src, int64_t pos, int len,
                                                           const float *hann, const float2 *tw, float2 *scr, cf twl,
                                                           int lane) {
    cf v[32];
    const bool inside = pos >= 0 && pos + 2048 <= (int64_t)len;
    const float *fr = src + pos;
    if (inside && ((reinterpret_cast<uintptr_t>(fr) & 7u) == 0)) {
#pragma unroll
        for (int n1 = 0; n1 < 32; ++n1) {
            const float2 xs = __ldg(reinterpret_cast<const float2 *>(fr + 64 * n1 + 2 * lane));
            const float2 ws = *reinterpret_cast<const float2 *>(hann + 64 * n1 + 2 * lane);
            v[n1] = cmul_elem(cf{xs.x, xs.y}, cf{ws.x, ws.y});
        }
    } else {
#pragma unroll
        for (int n1 = 0; n1 < 32; ++n1) {
            const int64_t p = pos + 64 * n1 + 2 * lane;
            const float x0 = (p >= 0 && p < len) ? __ldg(src + p) : 0.0f;
            const float x1 = (p + 1 >= 0 && p + 1 < len) ? __ldg(src + p + 1) : 0.0f;
            const float2 ws = *reinterpret_cast<const float2 *>(hann + 64 * n1 + 2 * lane);
            v[n1] = cmul_elem(cf{x0, x1}, cf{ws.x, ws.y});
        }
    }
    warp_power_spectrum_regs(v, tw, scr, twl, lane);
}

// ---- two frames per warp ------------------------------------------------------------------------------------------------
// The warp transforms frames A and B in ONE instruction stream: every constant it needs from shared memory — the Hann
// window, the W_1024 twiddles, W_2048^k of the un-pack and (in the caller) the mel weights — is loaded once and used
// twice, and the two independent FFTs interleave in the pipeline.  The arithmetic of each frame is exactly that of
// warp_power_spectrum_regs (same products, same order), so the spectra are bit-identical.
template <int K2>
struct PostStage2 {
    // Stores 4·|X[k]|²: the two halvings of the un-pack (E = ½(..), O = ½(..)) are exact scalings by a power of two, so
    // they commute with every rounding below — the caller multiplies the mel sums by ¼ instead (two FMUL2 fewer per
    // bin pair, bit-identical log-mel values).
    static __device__ __forceinline__ void one(const cf (&v)[32], int lane, cf w, float *pw) {
        cf zk = v[br5(K2)];
        cf own = v[br5((32 - K2) & 31)];
        cf snd = v[br5(31 - K2)];
        int src = (32 - lane) & 31;
        cf p;
        p.x = __shfl_sync(0xffffffffu, snd.x, src);
        p.y = __shfl_sync(0xffffffffu, snd.y, src);
        if (lane == 0) p = own;
        cf e = cadd_conj(zk, p);            // 2E = Z[k] + conj Z[N−k]
        cf o = cmul_mi(csub_conj(zk, p));   // 2O = (Z[k] − conj Z[N−k]) / i
        cf wo = cmul(o, w);
        cf x = cadd(e, wo);
        cf y = csub(e, wo);
        pw[lane + 32 * K2] = x.x * x.x + x.y * x.y;
        pw[1024 - lane - 32 * K2] = y.x * y.x + y.y * y.y;
    }
    static __device__ __forceinline__ void run(const cf (&a)[32], const cf (&b)[32], int lane, cf twl, float *pa, float *pb) {
        const cf w = mul_w64<K2>(twl);  // W_2048^(lane + 32·K2), shared by both frames
        one(a, lane, w, pa);
        one(b, lane, w, pb);
        if constexpr (K2 + 1 < 16) PostStage2<K2 + 1>::run(a, b, lane, twl, pa, pb);
        if constexpr (K2 == 0) {
            if (lane == 0) {
                cf z = a[br5(16)];
                pa[512] = 4.0f * (z.x * z.x + z.y * z.y);
                z = b[br5(16)];
                pb[512] = 4.0f * (z.x * z.x + z.y * z.y);
            }
        }
    }
};

// a, b: windowed packed frames (as warp_power_spectrum_regs); scra / scrb: two per-warp scratch tiles; on return
// their first 1025 floats hold the two power spectra.
__device__ __forceinline__ void warp_power_spectrum_regs2(cf (&a)[32], cf (&b)[32], const float2 *tw, float2 *scra,
                                                          float2 *scrb, cf twl, int lane) {
    fft32_dif(a);
    fft32_dif(b);
#pragma unroll
    for (int k1 = 0; k1 < 32; ++k1) {
        const float2 t = tw[k1 * 32 + lane];
        const cf ya = cmul(a[br5(k1)], cf{t.x, t.y});
        const cf yb = cmul(b[br5(k1)], cf{t.x, t.y});
        scra[k1 * kScrStride + lane] = make_float2(ya.x, ya.y);
        scrb[k1 * kScrStride + lane] = make_float2(yb.x, yb.y);
    }
    __syncwarp();
#pragma unroll
    for (int n2 = 0; n2 < 32; ++n2) {
        const float2 ta = scra[lane * kScrStride + n2];
        const float2 tb = scrb[lane * kScrStride + n2];
        a[n2] = cf{ta.x, ta.y};
        b[n2] = cf{tb.x, tb.y};
    }
    __syncwarp();
    fft32_dif(a);
    fft32_dif(b);
    PostStage2<0>::run(a, b, lane, twl, reinterpret_cast<float *>(scra), reinterpret_cast<float *>(scrb));
    __syncwarp();
}

// one frame's raw packed samples, zeros outside [0, len) (slow path: frames that touch a segment edge)
__device__ __forceinline__ void load_frame_guarded(const float *__restrict__ src, int64_t pos, int len, int lane,
                                                   cf (&raw)[32]) {
#pragma unroll
    for (int n1 = 0; n1 < 32; ++n1) {
        const int64_t p = pos + 64 * n1 + 2 * lane;
        raw[n1].x = (p >= 0 && p < len) ? __ldg(src + p) : 0.0f;
        raw[n1].y = (p + 1 >= 0 && p + 1 < len) ? __ldg(src + p + 1) : 0.0f;
    }
}

// Frames A (at pos) and B (at pos + hop) of one segment straight from global memory.  SHIFT = hop / 64 when the hop is
// a multiple of 64 samples (then B's register n1 holds the samples of A's register n1 + SHIFT: hop 64 loads 33
// float2 per lane for the two frames instead of 64), 0 otherwise.  b_valid = false: B is not a frame of the segment
// (odd frame count); its spectrum is computed on zeros and the caller discards it.
template <int SHIFT>
__device__ __forceinline__ void warp_power_spectrum_global2(const float *__restrict__ src, int64_t pos, int hop, int len,
                                                            bool b_valid, const float *hann, const float2 *tw,
                                                            float2 *scra, float2 *scrb, cf twl, int lane) {
    cf a[32], b[32];
    const float *fr = src + pos;
    const bool inside = b_valid && pos >= 0 && pos + hop + 2048 <= (int64_t)len &&
                        ((reinterpret_cast<uintptr_t>(fr) & 7u) == 0) && ((hop & 1) == 0);
    if (inside) {
        if constexpr (SHIFT > 0 && SHIFT < 32) {
            // raw[n1] = x[pos + 64·n1 + 2·lane ..+1], n1 < 32 + SHIFT; A uses raw[n1], B uses raw[n1 + SHIFT]
            cf raw[32 + SHIFT];
#pragma unroll
            for (int n1 = 0; n1 < 32 + SHIFT; ++n1) {
                const float2 xs = __ldg(reinterpret_cast<const float2 *>(fr + 64 * n1 + 2 * lane));
                raw[n1] = cf{xs.x, xs.y};
            }
#pragma unroll
            for (int n1 = 0; n1 < 32; ++n1) {
                const float2 ws = *reinterpret_cast<const float2 *>(hann + 64 * n1 + 2 * lane);
                a[n1] = cmul_elem(raw[n1], cf{ws.x, ws.y});
                b[n1] = cmul_elem(raw[n1 + SHIFT], cf{ws.x, ws.y});
            }
        } else {
#pragma unroll
            for (int n1 = 0; n1 < 32; ++n1) {
                const float2 xa = __ldg(reinterpret_cast<const float2 *>(fr + 64 * n1 + 2 * lane));
                const float2 xb = __ldg(reinterpret_cast<const float2 *>(fr + hop + 64 * n1 + 2 * lane));
                const float2 ws = *reinterpret_cast<const float2 *>(hann + 64 * n1 + 2 * lane);
                a[n1] = cmul_elem(cf{xa.x, xa.y}, cf{ws.x, ws.y});
                b[n1] = cmul_elem(cf{xb.x, xb.y}, cf{ws.x, ws.y});
            }
        }
    } else {
        load_frame_guarded(src, pos, len, lane, a);
        if (b_valid) {
            load_frame_guarded(src, pos + hop, len, lane, b);
        } else {
#pragma unroll
            for (int n1 = 0; n1 < 32; ++n1) b[n1] = cf{0.0f, 0.0f};
        }
#pragma unroll
        for (int n1 = 0; n1 < 32; ++n1) {
            const float2 ws = *reinterpret_cast<const float2 *>(hann + 64 * n1 + 2 * lane);
            a[n1] = cmul_elem(a[n1], cf{ws.x, ws.y});
            b[n1] = cmul_elem(b[n1], cf{ws.x, ws.y});
        }
    }
    warp_power_spectrum_regs2(a, b, tw, scra, scrb, twl, lane);
}

}  // namespace ncfa
