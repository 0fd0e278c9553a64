// Shared helpers for libncfa (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "../../include/ncfa.h"

namespace ncfa {

void set_error(const char *fmt, ...);

#define NCFA_CUDA_OK(expr)                                                                          \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            ncfa::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return NCFA_E_CUDA;                                                                     \
        }                                                                                           \
    } while (0)

#define NCFA_REQUIRE(cond, msg)                                                                     \
    do {                                                                                            \
        if (!(cond)) {                                                                              \
            ncfa::set_error("invalid argument: %s", msg);                                           \
            return NCFA_E_INVALID;                                                                  \
        }                                                                                           \
    } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over a workspace: every region starts on a 256-byte boundary.  With base == nullptr it only measures,
// so one layout function per family serves both its ncfa_*_workspace_bytes query and its entry point.
struct Carve {
    char *base;
    size_t used = 0;
    explicit Carve(void *b) : base((char *)b) {}
    template <class T>
    T *take(size_t n) {
        T *p = base ? (T *)(base + used) : nullptr;
        used += align_up(n * sizeof(T), 256);
        return p;
    }
};

inline int check_workspace(const char *family, size_t have, size_t need) {
    if (have >= need) return NCFA_OK;
    set_error("%s workspace too small: %zu < %zu", family, have, need);
    return NCFA_E_WORKSPACE;
}

// Thread-safe, monotonic cudaFuncAttributeMaxDynamicSharedMemorySize (host threads on different streams share kernels).
int ensure_dynamic_smem(const void *func, size_t bytes);
// SM count of the current device (cached)
int sm_count(int *out);

// Every launch goes through launch() below, so it sits in a ProfScope.  A ProfScope always opens an NVTX range named
// after the kernel family (header-only NVTX3: a no-op costing one predicted branch unless a tool such as ncu / nsys
// injected itself), and — optional per-kernel timing (ncfa_profile_enable) — records two CUDA events on the launch
// stream (it owns both, so scopes of concurrent host threads never pair up with each other) and hands them to the
// registry when it closes; ncfa_profile_report() synchronises them and sums per kernel name.
bool prof_enabled();
void prof_commit(const char *name, cudaEvent_t e0, cudaEvent_t e1, cudaStream_t st);
struct ProfScope {
    const char *name;
    cudaStream_t st;
    bool on;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    ProfScope(const char *n, cudaStream_t s) : name(n), st(s), on(prof_enabled()) {
        nvtxRangePushA(n);
        if (on) {
            on = cudaEventCreate(&e0) == cudaSuccess && cudaEventCreate(&e1) == cudaSuccess &&
                 cudaEventRecord(e0, st) == cudaSuccess;
        }
    }
    ~ProfScope() {
        if (on && cudaEventRecord(e1, st) == cudaSuccess) prof_commit(name, e0, e1, st);
        nvtxRangePop();
    }
};

// Launches k<<<grid, block, smem, st>>>(args...) under ProfScope(name).  Any dynamic shared memory first raises the
// kernel's limit to smem: the default limit is 48 KB less the kernel's static shared memory, so smem just under 48 KB
// can need it too.  Returns NCFA_E_CUDA (the message names `name`) if the launch was rejected.
template <class... P, class... A>
int launch(const char *name, void (*k)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A &&...args) {
    if (smem > 0) {
        if (int rc = ensure_dynamic_smem((const void *)k, smem)) return rc;
    }
    {
        ProfScope _p(name, st);
        k<<<grid, block, smem, st>>>(static_cast<A &&>(args)...);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("launch of %s failed: %s", name, cudaGetErrorString(e));
        return NCFA_E_CUDA;
    }
    return NCFA_OK;
}

// Constant tables that live in device global memory, one set per device (see ncfa_api.cu).
struct Tables {
    const float *hann;        // [2048] periodic Hann, float32(float64 value)
    const float2 *tw1024;     // [32][32]: tw[k1*32 + n2] = exp(-2πi·k1·n2/1024)
    const float2 *tw2048;     // [32]: exp(-2πi·l/2048), l = lane
    int sr;
    // lane-transposed mel bank of the onset kernel: lane l owns bands l, 63−l, 64+l, 127−l (group q = 0..3);
    // mel_wt[(mel_qoff[q] + i)·32 + l] = i-th weight of that band (0 beyond its support), i < mel_qw[q]
    const float *mel_wt;
    const int *mel_lane_bin0;  // [4][32] first FFT bin of the band of (q, lane)
    int mel_qoff[4], mel_qw[4], mel_wt_rows;
};
__host__ __device__ inline int mel_band_of(int q, int lane) {
    return q == 0 ? lane : (q == 1 ? 63 - lane : (q == 2 ? 64 + lane : 127 - lane));
}
int get_tables(int sr, Tables *out);
// 127-tap half-band FIR (float64) on the current device (chroma.cu)
int get_halfband_device(const double **out);

// order-preserving float <-> uint encoding for atomicMax on floats
__device__ __forceinline__ unsigned float_to_ordered(float f) {
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ordered_to_float(unsigned u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace ncfa
