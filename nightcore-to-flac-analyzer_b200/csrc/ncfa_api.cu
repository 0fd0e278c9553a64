// Library plumbing: error string, version, constant tables (Hann, twiddles, Slaney mel bank).
#include <math.h>
#include <stdarg.h>
#include <algorithm>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>
#include "ncfa_common.cuh"

namespace ncfa {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static std::mutex g_attr_mu;
static std::map<std::pair<int, const void *>, size_t> g_dyn_smem;
static std::map<int, int> g_sm_count;

int ensure_dynamic_smem(const void *func, size_t bytes) {
    int dev = 0;
    NCFA_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_attr_mu);
    size_t &cur = g_dyn_smem[std::make_pair(dev, func)];
    if (bytes > cur) {
        NCFA_CUDA_OK(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        cur = bytes;
    }
    return NCFA_OK;
}

int sm_count(int *out) {
    int dev = 0;
    NCFA_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_attr_mu);
    auto it = g_sm_count.find(dev);
    if (it == g_sm_count.end()) {
        int n = 0;
        NCFA_CUDA_OK(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
        it = g_sm_count.emplace(dev, n).first;
    }
    *out = it->second;
    return NCFA_OK;
}

// ---- per-kernel event profiler
struct ProfEntry {
    const char *name;
    cudaEvent_t e0, e1;
    cudaStream_t st;
};
static std::mutex g_prof_mu;
static bool g_prof_on = false;
static std::vector<ProfEntry> g_prof;

bool prof_enabled() { return g_prof_on; }
void prof_commit(const char *name, cudaEvent_t e0, cudaEvent_t e1, cudaStream_t st) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof.push_back(ProfEntry{name, e0, e1, st});
}

// ---- Slaney mel scale (librosa.filters.mel(htk=False, norm='slaney'), SURVEY Appendix A.2)
static double hz_to_mel(double f) {
    const double f_sp = 200.0 / 3, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp, logstep = log(6.4) / 27.0;
    return f >= min_log_hz ? min_log_mel + log(f / min_log_hz) / logstep : f / f_sp;
}
static double mel_to_hz(double m) {
    const double f_sp = 200.0 / 3, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp, logstep = log(6.4) / 27.0;
    return m >= min_log_mel ? min_log_hz * exp(logstep * (m - min_log_mel)) : f_sp * m;
}

struct DeviceTables {
    Tables t;
};
static std::mutex g_mu;
static std::map<std::pair<int, int>, DeviceTables> g_tables;

template <typename T>
static int upload(const std::vector<T> &h, const T **d) {
    T *p = nullptr;
    NCFA_CUDA_OK(cudaMalloc(&p, h.size() * sizeof(T)));
    NCFA_CUDA_OK(cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    *d = p;
    return NCFA_OK;
}

// Host side of the Slaney mel bank (librosa.filters.mel(htk=False, norm='slaney'), SURVEY Appendix A.2): packed
// band-major weights, and from them the lane-transposed, bank-conflict-free copy the onset kernel reads.
struct MelHost {
    std::vector<float> w;          // packed non-zero weights, band-major
    std::vector<int> start, bin0;  // [129], [128]
    std::vector<float> wt;         // [rows][32] lane-transposed weights
    std::vector<int> lb;           // [4][32] first bin read by (q, lane)
    int qoff[4], qw[4], rows;
};

static int build_mel_host(int sr, MelHost *mh) {
    const int n_fft = NCFA_N_FFT, n_mels = NCFA_N_MELS, n_bins = n_fft / 2 + 1;
    std::vector<float> &w = mh->w;
    std::vector<int> &start = mh->start, &bin0 = mh->bin0;
    // mel bank
    std::vector<double> mel_f(n_mels + 2);
    {
        double lo = hz_to_mel(0.0), hi = hz_to_mel(sr / 2.0);
        double step = (hi - lo) / (n_mels + 1);
        for (int i = 0; i < n_mels + 2; ++i) mel_f[i] = mel_to_hz(i * step + lo);
        mel_f[n_mels + 1] = mel_to_hz(hi);
    }
    const double d = 1.0 / sr, val = 1.0 / (n_fft * d);
    w.clear();
    start.assign(n_mels + 1, 0);
    bin0.assign(n_mels, 0);
    for (int m = 0; m < n_mels; ++m) {
        const double fd0 = mel_f[m + 1] - mel_f[m], fd1 = mel_f[m + 2] - mel_f[m + 1];
        const double enorm = 2.0 / (mel_f[m + 2] - mel_f[m]);
        int first = -1, last = -1;
        std::vector<float> row(n_bins);
        for (int k = 0; k < n_bins; ++k) {
            const double f = k * val;
            const double lower = -(mel_f[m] - f) / fd0, upper = (mel_f[m + 2] - f) / fd1;
            const double tri = fmax(0.0, fmin(lower, upper));
            const float w32 = (float)tri;                       // weights[i] assigned into a float32 array
            row[k] = (float)((double)w32 * enorm);              // weights *= enorm[:, None]
            if (row[k] != 0.0f) {
                if (first < 0) first = k;
                last = k;
            }
        }
        start[m] = (int)w.size();
        bin0[m] = first < 0 ? 0 : first;
        if (first >= 0)
            for (int k = first; k <= last; ++k) w.push_back(row[k]);
    }
    start[n_mels] = (int)w.size();
    if ((int)w.size() > 2048) {
        set_error("mel bank has %zu non-zeros (> 2048) at sr=%d", w.size(), sr);
        return NCFA_E_OVERFLOW;
    }
    // lane-transposed copy (see Tables).  Lane l of group q reads the power spectrum at lane_bin0 + i, i < mel_qw[q]:
    // if two lanes start at bins that are congruent mod 32 every one of those reads is a shared-memory bank conflict
    // (measured 3-way on average with the natural starts).  A lane may start up to (rows − width) bins EARLY at no
    // cost but zero weights, so the starts are chosen by bipartite matching (lanes → residues mod 32) with the
    // smallest row count that admits a conflict-free assignment (95 rows instead of 91 at 22 050 Hz).
    {
        int rows = 0;
        std::vector<int> shift(4 * 32, 0);
        for (int q = 0; q < 4; ++q) {
            int mw = 0;
            for (int l = 0; l < 32; ++l) {
                const int m = mel_band_of(q, l);
                mw = std::max(mw, start[m + 1] - start[m]);
            }
            int nw = mw;
            for (;; ++nw) {
                // Kuhn's augmenting paths: owner[r] = lane that starts at residue r
                int owner[32], owner_d[32];
                for (int r = 0; r < 32; ++r) owner[r] = -1;
                std::function<bool(int, unsigned &)> assign = [&](int l, unsigned &seen) -> bool {
                    const int m = mel_band_of(q, l);
                    const int wdt = start[m + 1] - start[m];
                    for (int d = 0; d <= nw - wdt && bin0[m] - d >= 0; ++d) {
                        const int r = (bin0[m] - d) & 31;
                        if (seen & (1u << r)) continue;
                        seen |= 1u << r;
                        if (owner[r] < 0 || assign(owner[r], seen)) {
                            owner[r] = l;
                            owner_d[r] = d;
                            return true;
                        }
                    }
                    return false;
                };
                bool ok = true;
                for (int l = 0; l < 32 && ok; ++l) {
                    unsigned seen = 0;
                    ok = assign(l, seen);
                }
                if (ok) {
                    for (int r = 0; r < 32; ++r) shift[q * 32 + owner[r]] = owner_d[r];
                    break;
                }
                if (nw > mw + 64) {  // cannot happen (32 free residues within 32 extra rows); keep the natural starts
                    nw = mw;
                    for (int l = 0; l < 32; ++l) shift[q * 32 + l] = 0;
                    break;
                }
            }
            mh->qoff[q] = rows;
            mh->qw[q] = nw;
            rows += nw;
        }
        mh->rows = rows;
        if (rows > 128) {
            set_error("transposed mel bank has %d rows (> 128) at sr=%d", rows, sr);
            return NCFA_E_OVERFLOW;
        }
        std::vector<float> &wt = mh->wt;
        std::vector<int> &lb = mh->lb;
        wt.assign((size_t)rows * 32, 0.0f);
        lb.assign(4 * 32, 0);
        for (int q = 0; q < 4; ++q)
            for (int l = 0; l < 32; ++l) {
                const int m = mel_band_of(q, l);
                const int d = shift[q * 32 + l];
                lb[q * 32 + l] = bin0[m] - d;
                for (int i = start[m]; i < start[m + 1]; ++i)
                    wt[(size_t)(mh->qoff[q] + d + i - start[m]) * 32 + l] = w[i];
            }
    }
    return NCFA_OK;
}

int get_tables(int sr, Tables *out) {
    int dev = 0;
    NCFA_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_mu);
    auto key = std::make_pair(dev, sr);
    auto it = g_tables.find(key);
    if (it != g_tables.end()) {
        *out = it->second.t;
        return NCFA_OK;
    }
    NCFA_REQUIRE(sr >= 2000 && sr <= 768000, "sample rate out of range");
    const int n_fft = NCFA_N_FFT;
    const double PI = 3.14159265358979323846;
    std::vector<float> hann(n_fft);
    for (int i = 0; i < n_fft; ++i) hann[i] = (float)(0.5 - 0.5 * cos(2.0 * PI * i / n_fft));
    std::vector<float2> tw1024(1024), tw2048(32);
    for (int k1 = 0; k1 < 32; ++k1)
        for (int n2 = 0; n2 < 32; ++n2) {
            double a = -2.0 * PI * (double)(k1 * n2) / 1024.0;
            tw1024[k1 * 32 + n2] = make_float2((float)cos(a), (float)sin(a));
        }
    for (int l = 0; l < 32; ++l) {
        double a = -2.0 * PI * l / 2048.0;
        tw2048[l] = make_float2((float)cos(a), (float)sin(a));
    }
    MelHost mh;
    {
        const int mrc = build_mel_host(sr, &mh);
        if (mrc) return mrc;
    }
    DeviceTables dt;
    int rc;
    for (int q = 0; q < 4; ++q) {
        dt.t.mel_qoff[q] = mh.qoff[q];
        dt.t.mel_qw[q] = mh.qw[q];
    }
    dt.t.mel_wt_rows = mh.rows;
    if ((rc = upload(mh.wt, &dt.t.mel_wt))) return rc;
    if ((rc = upload(mh.lb, &dt.t.mel_lane_bin0))) return rc;
    if ((rc = upload(hann, &dt.t.hann))) return rc;
    if ((rc = upload(tw1024, &dt.t.tw1024))) return rc;
    if ((rc = upload(tw2048, &dt.t.tw2048))) return rc;
    dt.t.sr = sr;
    g_tables[key] = dt;
    *out = dt.t;
    return NCFA_OK;
}

}  // namespace ncfa

extern "C" int ncfa_version(void) { return 100; }
extern "C" void ncfa_profile_enable(int on) {
    std::lock_guard<std::mutex> lk(ncfa::g_prof_mu);
    ncfa::g_prof_on = on != 0;
}
// "name,launches,total_ms\n" per kernel, written into buf (NUL-terminated); clears the records.
extern "C" int ncfa_profile_report(char *buf, size_t cap) {
    using namespace ncfa;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    std::map<std::string, std::pair<int, double>> acc;
    for (auto &e : g_prof) {
        float ms = 0.f;
        if (cudaEventSynchronize(e.e1) == cudaSuccess && cudaEventElapsedTime(&ms, e.e0, e.e1) == cudaSuccess) {
            auto &a = acc[e.name];
            a.first += 1;
            a.second += ms;
        } else {
            (void)cudaGetLastError();  // never leave a stale error behind for the caller's next CUDA check
        }
        cudaEventDestroy(e.e0);
        cudaEventDestroy(e.e1);
    }
    g_prof.clear();
    std::string out;
    char line[256];
    for (auto &kv : acc) {
        snprintf(line, sizeof(line), "%s,%d,%.6f\n", kv.first.c_str(), kv.second.first, kv.second.second);
        out += line;
    }
    if (cap == 0) return NCFA_E_INVALID;
    size_t n = out.size() < cap - 1 ? out.size() : cap - 1;
    memcpy(buf, out.data(), n);
    buf[n] = 0;
    return NCFA_OK;
}
// "name,stream,t0_ms,t1_ms\n" per recorded launch (times relative to the first record's start), written into buf;
// clears the records.  Diagnostic companion of ncfa_profile_report: shows where the streams of concurrent host workers
// leave the device idle.
extern "C" int ncfa_profile_timeline(char *buf, size_t cap) {
    using namespace ncfa;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (cap == 0) return NCFA_E_INVALID;
    std::string out;
    char line[256];
    cudaEvent_t base = g_prof.empty() ? nullptr : g_prof[0].e0;
    if (base) cudaEventSynchronize(base);
    for (auto &e : g_prof) {
        float t0 = 0.f, t1 = 0.f;
        if (cudaEventSynchronize(e.e1) == cudaSuccess && cudaEventElapsedTime(&t0, base, e.e0) == cudaSuccess &&
            cudaEventElapsedTime(&t1, base, e.e1) == cudaSuccess) {
            snprintf(line, sizeof(line), "%s,%p,%.4f,%.4f\n", e.name, (void *)e.st, t0, t1);
            if (out.size() + strlen(line) + 1 < cap) out += line;
        } else {
            (void)cudaGetLastError();
        }
    }
    for (auto &e : g_prof) {
        cudaEventDestroy(e.e0);
        cudaEventDestroy(e.e1);
    }
    g_prof.clear();
    memcpy(buf, out.data(), out.size());
    buf[out.size()] = 0;
    return NCFA_OK;
}
extern "C" const char *ncfa_last_error(void) { return ncfa::g_err; }
namespace ncfa {
__global__ void __launch_bounds__(256) param_upload_kernel(unsigned char *__restrict__ dst,
                                                           const unsigned char *__restrict__ src, size_t nbytes) {
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (size_t)gridDim.x * blockDim.x;
    if ((((uintptr_t)dst | (uintptr_t)src) & 15u) == 0) {
        const size_t n16 = nbytes / 16;
        for (size_t i = tid; i < n16; i += nt) reinterpret_cast<uint4 *>(dst)[i] = reinterpret_cast<const uint4 *>(src)[i];
        for (size_t i = n16 * 16 + tid; i < nbytes; i += nt) dst[i] = src[i];
    } else {
        for (size_t i = tid; i < nbytes; i += nt) dst[i] = src[i];
    }
}
}  // namespace ncfa

extern "C" int ncfa_param_upload(void *d_dst, const void *h_pinned_src, size_t nbytes, void *stream) {
    using namespace ncfa;
    if (nbytes == 0) return NCFA_OK;
    NCFA_REQUIRE(d_dst && h_pinned_src, "null pointer");
    void *dsrc = nullptr;
    if (cudaHostGetDevicePointer(&dsrc, const_cast<void *>(h_pinned_src), 0) != cudaSuccess) {
        (void)cudaGetLastError();
        set_error("ncfa_param_upload: source is not pinned, device-mapped host memory");
        return NCFA_E_INVALID;
    }
    const size_t vecs = (nbytes + 15) / 16;
    const int grid = (int)std::min<size_t>(64, (vecs + 255) / 256);
    return launch("param_upload_kernel", param_upload_kernel, grid, 256, 0, (cudaStream_t)stream,
                  (unsigned char *)d_dst, (const unsigned char *)dsrc, nbytes);
}

// Host-only view of the lane-transposed mel bank (tests/test_host_tables.py): h_lane_bin0 int32[128] ((q, lane) order),
// h_qw int32[4] rows per group, h_wt float32[128][32] (rows beyond the used ones stay zero).  No device needed.
extern "C" int ncfa_host_mel_lanes(int sr, int32_t *h_lane_bin0, int32_t *h_qw, float *h_wt) {
    using namespace ncfa;
    NCFA_REQUIRE(h_lane_bin0 && h_qw && h_wt, "null pointer");
    NCFA_REQUIRE(sr >= 2000 && sr <= 768000, "sample rate out of range");
    MelHost mh;
    const int rc = build_mel_host(sr, &mh);
    if (rc) return rc;
    for (int i = 0; i < 128; ++i) h_lane_bin0[i] = mh.lb[i];
    for (int q = 0; q < 4; ++q) h_qw[q] = mh.qw[q];
    for (int i = 0; i < 128 * 32; ++i) h_wt[i] = i < mh.rows * 32 ? mh.wt[i] : 0.0f;
    return NCFA_OK;
}

extern "C" int ncfa_init_tables(int sr) {
    ncfa::Tables t;
    return ncfa::get_tables(sr, &t);
}
