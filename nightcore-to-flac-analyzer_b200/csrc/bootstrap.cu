// Bootstrap medians / confidence intervals, bit-exact with numpy's Generator(PCG64).choice.
// Replaces the Python loops of consensus.py:255-266 (_bootstrap_ratio), consensus.py:300-311
// (compute_ibi_ratio) and pitch.py:143-150 (chunk-shift bootstrap).  SURVEY.md §4 (RNG KATs), A.10.
//
// The reference draws serially from ONE PCG64 stream: iteration i resamples array a (n_a bounded
// 32-bit Lemire draws) and then array b.  PCG64 is a 128-bit LCG, so the state before any draw is
// reachable in O(log k) (jump-ahead); the only serial coupling is the number of Lemire rejections
// before iteration i, which shifts its start in the stream.  Pipeline (one launch each):
//   boot_tables   jump tables A^(2^b), C_(2^b) and the per-lane / stride-32 steps
//   boot_rank     rank transform of a and b (so medians become order statistics of integer ranks)
//   boot_offsets  per job: iterate "count rejections per iteration → prefix sum" to its fixed point
//   boot_median   one warp per (job, iteration): lanes draw in parallel (stride-32 LCG steps),
//                 histogram the ranks in shared memory, pick the middle order statistic(s)
//   boot_finish   point estimate and np.percentile(boot, q, method='linear') by rank selection
// float64 arithmetic is compiled with -fmad=false: every +,−,×,÷ rounds like numpy's.
#include "ncfa_common.cuh"

namespace ncfa {

constexpr int kBootFinishMaxStaged = 5000;  // bootstrap values of one job staged in shared memory (40 KB)

typedef unsigned __int128 u128;

struct LcgStep {
    u128 a, c;  // x -> a·x + c
};

struct BootTables {
    LcgStep pow2[64];  // 2^b steps
    LcgStep lane[32];  // l steps
    LcgStep stride32;  // 32 steps
};

__host__ __device__ inline u128 pcg_mult() {
    return (((u128)0x2360ED051FC65DA4ULL) << 64) | (u128)0x4385DF649FCCF645ULL;
}

__device__ __forceinline__ uint64_t pcg_output(u128 s) {
    const uint64_t hi = (uint64_t)(s >> 64), lo = (uint64_t)s;
    const uint64_t x = hi ^ lo;
    const unsigned rot = (unsigned)(hi >> 58);
    return (x >> rot) | (x << ((64u - rot) & 63u));
}

__global__ void boot_tables_kernel(u128 inc, BootTables *t) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    LcgStep s{pcg_mult(), inc};
    for (int b = 0; b < 64; ++b) {
        t->pow2[b] = s;
        LcgStep n;
        n.a = s.a * s.a;
        n.c = s.c * (s.a + 1);
        s = n;
    }
    LcgStep l{(u128)1, (u128)0};
    for (int i = 0; i < 32; ++i) {
        t->lane[i] = l;
        l.a = l.a * pcg_mult();
        l.c = l.c * pcg_mult() + inc;
    }
    t->stride32 = l;
}

// state after k steps from s
__device__ __forceinline__ u128 pcg_jump(u128 s, uint64_t k, const BootTables *__restrict__ t) {
    for (int b = 0; k; ++b, k >>= 1)
        if (k & 1) s = t->pow2[b].a * s + t->pow2[b].c;
    return s;
}

// Sequential reader of the 32-bit draw stream starting at raw position `pos`
// (pos/2 = index of the 64-bit output, pos&1 = half; numpy hands out the low half first).
struct Stream32 {
    u128 s, inc;
    uint32_t buf;
    bool has;
    __device__ void seek(u128 state0, u128 inc_, uint64_t pos, const BootTables *__restrict__ t) {
        inc = inc_;
        s = pcg_jump(state0, pos >> 1, t);
        has = false;
        if (pos & 1) {
            s = s * pcg_mult() + inc;
            buf = (uint32_t)(pcg_output(s) >> 32);
            has = true;
        }
    }
    __device__ __forceinline__ uint32_t next() {
        if (has) {
            has = false;
            return buf;
        }
        s = s * pcg_mult() + inc;
        const uint64_t v = pcg_output(s);
        buf = (uint32_t)(v >> 32);
        has = true;
        return (uint32_t)v;
    }
};

// numpy buffered_bounded_lemire_uint32 with rng = n-1 (n >= 2); *extra counts the redraws
__device__ __forceinline__ uint32_t bounded_draw(Stream32 &g, uint32_t n, int &extra) {
    uint64_t m = (uint64_t)g.next() * n;
    uint32_t leftover = (uint32_t)m;
    if (leftover < n) {
        const uint32_t threshold = (uint32_t)((0xffffffffu - (n - 1u)) % n);
        while (leftover < threshold) {
            m = (uint64_t)g.next() * n;
            leftover = (uint32_t)m;
            ++extra;
        }
    }
    return (uint32_t)(m >> 32);
}

// ---- rank transform: rank[i] = #{j : v[j] < v[i] or (v[j] == v[i] and j < i)};  sorted[rank[i]] = v[i]
__global__ void __launch_bounds__(256) boot_rank_kernel(const double *__restrict__ a, const int64_t *__restrict__ a_off,
                                                        const int32_t *__restrict__ a_len, const double *__restrict__ b,
                                                        const int64_t *__restrict__ b_off,
                                                        const int32_t *__restrict__ b_len, int max_a, int max_b,
                                                        int32_t *__restrict__ rank_a, int32_t *__restrict__ rank_b,
                                                        double *__restrict__ sorted_a, double *__restrict__ sorted_b) {
    __shared__ double tile[1024];
    const int job = blockIdx.x;
    const bool second = blockIdx.y == 1;
    const int n = second ? (b_len ? b_len[job] : 0) : a_len[job];
    if (n <= 0) return;
    const double *v = second ? b + b_off[job] : a + a_off[job];
    int32_t *rk = second ? rank_b + (size_t)job * max_b : rank_a + (size_t)job * max_a;
    double *so = second ? sorted_b + (size_t)job * max_b : sorted_a + (size_t)job * max_a;
    for (int base = 0; base < n; base += 256) {
        const int i = base + threadIdx.x;
        const double x = i < n ? v[i] : 0.0;
        int r = 0;
        for (int t0 = 0; t0 < n; t0 += 1024) {
            const int tn = min(1024, n - t0);
            __syncthreads();
            for (int j = threadIdx.x; j < tn; j += 256) tile[j] = v[t0 + j];
            __syncthreads();
            if (i < n) {
                for (int j = 0; j < tn; ++j) {
                    const double y = tile[j];
                    r += (y < x || (y == x && (t0 + j) < i)) ? 1 : 0;
                }
            }
        }
        if (i < n) {
            rk[i] = r;
            so[r] = x;
        }
    }
}

// ---- fixed point of the rejection prefix:  start[i] = i·per_iter + Σ_{j<i} extra[j]
__global__ void __launch_bounds__(1024) boot_offsets_kernel(const int32_t *__restrict__ a_len,
                                                            const int32_t *__restrict__ b_len, int n_boot, u128 state0,
                                                            u128 inc, const BootTables *__restrict__ tb,
                                                            int64_t *__restrict__ start, int32_t *__restrict__ extra) {
    __shared__ int s_warp[32];
    __shared__ int s_changed;
    __shared__ int s_carry;
    const int job = blockIdx.x;
    const uint32_t na = (uint32_t)a_len[job], nb = b_len ? (uint32_t)b_len[job] : 0u;
    const uint32_t ca = na > 1 ? na : 0u, cb = nb > 1 ? nb : 0u;  // n == 1 consumes nothing
    const int64_t per_iter = (int64_t)ca + cb;
    int64_t *st = start + (size_t)job * n_boot;
    int32_t *ex = extra + (size_t)job * n_boot;
    for (int i = threadIdx.x; i < n_boot; i += blockDim.x) {
        st[i] = (int64_t)i * per_iter;
        ex[i] = -1;  // not evaluated yet
    }
    __syncthreads();
    for (int round = 0; round <= n_boot; ++round) {
        if (threadIdx.x == 0) {
            s_changed = 0;
            s_carry = 0;
        }
        // (1) evaluate iterations whose start moved (or never ran)
        for (int i = threadIdx.x; i < n_boot; i += blockDim.x) {
            if (ex[i] < 0) {
                Stream32 g;
                g.seek(state0, inc, (uint64_t)st[i], tb);
                int e = 0;
                for (uint32_t l = 0; l < ca; ++l) (void)bounded_draw(g, na, e);
                for (uint32_t l = 0; l < cb; ++l) (void)bounded_draw(g, nb, e);
                ex[i] = e;
            }
        }
        __syncthreads();
        // (2) exclusive prefix sum of extra[] in index order (block scan over chunks of blockDim)
        for (int base = 0; base < n_boot; base += blockDim.x) {
            const int i = base + threadIdx.x;
            const int v = i < n_boot ? ex[i] : 0;
            int incl = v;
            const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            if (lane == 31) s_warp[warp] = incl;
            __syncthreads();
            if (warp == 0) {
                int w = lane < (int)(blockDim.x >> 5) ? s_warp[lane] : 0;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    int t = __shfl_up_sync(0xffffffffu, w, o);
                    if (lane >= o) w += t;
                }
                s_warp[lane] = w;
            }
            __syncthreads();
            const int carry = s_carry;
            const int excl = carry + (warp > 0 ? s_warp[warp - 1] : 0) + incl - v;
            if (i < n_boot) {
                const int64_t ns = (int64_t)i * per_iter + excl;
                if (ns != st[i]) {
                    st[i] = ns;
                    ex[i] = -1;
                    s_changed = 1;
                }
            }
            __syncthreads();
            if (threadIdx.x == 0) s_carry = carry + s_warp[(blockDim.x >> 5) - 1];
            __syncthreads();
        }
        if (!s_changed) break;
        __syncthreads();
    }
}

// k-th smallest rank present in hist[0..n) (warp-cooperative); returns the rank
__device__ __forceinline__ int warp_kth(const int *hist, int n, int k, int lane) {
    const int per = (n + 31) >> 5;
    const int lo = lane * per, hi = min(n, lo + per);
    int s = 0;
    for (int j = lo; j < hi; ++j) s += hist[j];
    int incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    const int excl = incl - s;
    const bool mine = (k >= excl) && (k < incl);
    int found = -1;
    if (mine) {
        int c = excl;
        for (int j = lo; j < hi; ++j) {
            c += hist[j];
            if (k < c) {
                found = j;
                break;
            }
        }
    }
    const unsigned m = __ballot_sync(0xffffffffu, mine);
    const int src = __ffs(m) - 1;
    return __shfl_sync(0xffffffffu, found, src < 0 ? 0 : src);
}

__global__ void __launch_bounds__(256) boot_median_kernel(
    const int32_t *__restrict__ a_len, const int32_t *__restrict__ b_len, int max_a, int max_b, int n_boot,
    int n_jobs, u128 state0, u128 inc, const BootTables *__restrict__ tb, const int64_t *__restrict__ start,
    const int32_t *__restrict__ extra, const int32_t *__restrict__ rank_a, const int32_t *__restrict__ rank_b,
    const double *__restrict__ sorted_a, const double *__restrict__ sorted_b, double *__restrict__ boot,
    int32_t *__restrict__ idx_out, int hist_stride) {
    extern __shared__ int s_hist[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int warps = blockDim.x >> 5;
    const long long total = (long long)n_jobs * n_boot;
    int *hist = s_hist + (size_t)warp * hist_stride;
    for (long long w = (long long)blockIdx.x * warps + warp; w < total; w += (long long)gridDim.x * warps) {
        const int job = (int)(w / n_boot), it = (int)(w % n_boot);
        const uint32_t na = (uint32_t)a_len[job], nb = b_len ? (uint32_t)b_len[job] : 0u;
        const uint32_t ca = na > 1 ? na : 0u, cb = nb > 1 ? nb : 0u;
        const uint32_t per = ca + cb;
        int *ha = hist, *hb = hist + na;
        for (uint32_t j = lane; j < na + nb; j += 32) hist[j] = 0;
        __syncwarp();
        const int32_t *ra = rank_a + (size_t)job * max_a;
        const int32_t *rb = rank_b + (size_t)job * max_b;
        const uint64_t p0 = (uint64_t)start[(size_t)job * n_boot + it];
        int32_t *io = idx_out ? idx_out + (size_t)it * (na + nb) : nullptr;  // n_jobs == 1 only
        if (na == 1 && lane == 0) {
            ha[0] = 1;
            if (io) io[0] = 0;
        }
        if (nb == 1 && lane == 0) {
            hb[0] = 1;
            if (io) io[na] = 0;
        }
        if (extra[(size_t)job * n_boot + it] == 0) {
            // no redraws: logical draw l sits at raw position p0 + l; lanes take 64-bit outputs round-robin
            const uint64_t q0 = p0 >> 1;
            const uint64_t q1 = (p0 + per + 1) >> 1;  // exclusive
            u128 s = pcg_jump(state0, q0, tb);
            s = tb->lane[lane].a * s + tb->lane[lane].c;
            const u128 a32 = tb->stride32.a, c32 = tb->stride32.c;
            for (uint64_t q = q0 + lane; q < q1; q += 32) {
                const u128 s1 = s * pcg_mult() + inc;  // state that produces output q
                const uint64_t v = pcg_output(s1);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const long long l = (long long)(2 * q + h) - (long long)p0;
                    if (l >= 0 && l < (long long)per) {
                        const uint32_t u = h ? (uint32_t)(v >> 32) : (uint32_t)v;
                        if (l < (long long)ca) {
                            const uint32_t r = (uint32_t)(((uint64_t)u * na) >> 32);
                            atomicAdd(&ha[ra[r]], 1);
                            if (io) io[l] = (int32_t)r;
                        } else {
                            const uint32_t r = (uint32_t)(((uint64_t)u * nb) >> 32);
                            atomicAdd(&hb[rb[r]], 1);
                            if (io) io[(l - ca) + na] = (int32_t)r;
                        }
                    }
                }
                s = a32 * s + c32;
            }
        } else if (lane == 0) {
            // rare: this iteration contains Lemire redraws — replay it serially
            Stream32 g;
            g.seek(state0, inc, p0, tb);
            int e = 0;
            for (uint32_t l = 0; l < ca; ++l) {
                const uint32_t r = bounded_draw(g, na, e);
                ha[ra[r]] += 1;
                if (io) io[l] = (int32_t)r;
            }
            for (uint32_t l = 0; l < cb; ++l) {
                const uint32_t r = bounded_draw(g, nb, e);
                hb[rb[r]] += 1;
                if (io) io[na + l] = (int32_t)r;
            }
        }
        __syncwarp();
        // np.median: middle order statistic, or the mean of the two middle ones
        const double *sa = sorted_a + (size_t)job * max_a;
        const int ka0 = warp_kth(ha, (int)na, ((int)na - 1) >> 1, lane);
        const int ka1 = warp_kth(ha, (int)na, (int)na >> 1, lane);
        double med = (na & 1u) ? sa[ka1] : (sa[ka0] + sa[ka1]) / 2.0;
        if (nb > 0) {
            const double *sb = sorted_b + (size_t)job * max_b;
            const int kb0 = warp_kth(hb, (int)nb, ((int)nb - 1) >> 1, lane);
            const int kb1 = warp_kth(hb, (int)nb, (int)nb >> 1, lane);
            const double mb = (nb & 1u) ? sb[kb1] : (sb[kb0] + sb[kb1]) / 2.0;
            med = med / mb;
        }
        if (lane == 0) boot[(size_t)job * n_boot + it] = med;
        __syncwarp();
    }
}

// np.percentile(method='linear') index arithmetic: q/100, virtual index (n-1)·quantile → (prev, next, gamma)
__device__ __forceinline__ void percentile_indices(int n, double q, int *prev, int *next, double *gamma) {
    const double quant = q / 100.0;
    const double virt = (double)(n - 1) * quant;
    int p = (int)floor(virt), nx = p + 1;
    if (virt >= (double)(n - 1)) p = nx = n - 1;
    if (virt < 0.0) p = nx = 0;
    *prev = p;
    *next = nx;
    *gamma = virt - floor(virt);
}
__device__ __forceinline__ double percentile_lerp(double a, double b, double gamma) {  // numpy's _lerp
    const double d = b - a;
    double r = a + d * gamma;
    if (gamma >= 0.5) r = b - d * (1.0 - gamma);
    return r;
}

// One CTA per job: ONE rank pass over the n_boot bootstrap values (staged in shared memory; rank of element i =
// #{k : v[k] < v[i] or (v[k] == v[i] and k < i)}, O(n²/threads)) picks the four order statistics that the two
// percentiles interpolate between.
__global__ void __launch_bounds__(256) boot_finish_kernel(const int32_t *__restrict__ a_len,
                                                          const int32_t *__restrict__ b_len, int max_a, int max_b,
                                                          int n_boot, const double *__restrict__ sorted_a,
                                                          const double *__restrict__ sorted_b,
                                                          const double *__restrict__ boot, double q_lo, double q_hi,
                                                          double *__restrict__ out) {
    extern __shared__ double sv[];  // n_boot values (global memory is read directly when they do not fit)
    __shared__ double s_stat[4];
    const int job = blockIdx.x;
    const int na = a_len[job], nb = b_len ? b_len[job] : 0;
    const double *vg = boot + (size_t)job * n_boot;
    const bool staged = n_boot <= kBootFinishMaxStaged;
    if (staged)
        for (int i = threadIdx.x; i < n_boot; i += blockDim.x) sv[i] = vg[i];
    __syncthreads();
    const double *v = staged ? sv : vg;
    int j[4];
    double g_lo, g_hi;
    percentile_indices(n_boot, q_lo, &j[0], &j[1], &g_lo);
    percentile_indices(n_boot, q_hi, &j[2], &j[3], &g_hi);
    for (int i = threadIdx.x; i < n_boot; i += blockDim.x) {
        const double x = v[i];
        int r = 0;
        for (int k = 0; k < i; ++k) r += (v[k] <= x) ? 1 : 0;           // y < x or (y == x and k < i)
        for (int k = i + 1; k < n_boot; ++k) r += (v[k] < x) ? 1 : 0;
#pragma unroll
        for (int m = 0; m < 4; ++m)
            if (r == j[m]) s_stat[m] = x;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const double lo = percentile_lerp(s_stat[0], s_stat[1], g_lo);
        const double hi = percentile_lerp(s_stat[2], s_stat[3], g_hi);
        const double *sa = sorted_a + (size_t)job * max_a;
        double point = (na & 1) ? sa[na >> 1] : (sa[(na - 1) >> 1] + sa[na >> 1]) / 2.0;
        if (nb > 0) {
            const double *sb = sorted_b + (size_t)job * max_b;
            const double mb = (nb & 1) ? sb[nb >> 1] : (sb[(nb - 1) >> 1] + sb[nb >> 1]) / 2.0;
            point = point / mb;
        }
        out[3 * job + 0] = point;
        out[3 * job + 1] = lo;
        out[3 * job + 2] = hi;
    }
}

struct BootWs {
    BootTables *tables;
    int32_t *rank_a, *rank_b;
    double *sorted_a, *sorted_b;
    int64_t *start;
    int32_t *extra;
    double *boot;
    size_t bytes;
};

static BootWs boot_ws(int n_jobs, int max_a, int max_b, int n_boot, void *base) {
    Carve c(base);
    BootWs w;
    const size_t mb = max_b > 0 ? max_b : 1;
    w.tables = c.take<BootTables>(1);
    w.rank_a = c.take<int32_t>((size_t)n_jobs * max_a);
    w.rank_b = c.take<int32_t>((size_t)n_jobs * mb);
    w.sorted_a = c.take<double>((size_t)n_jobs * max_a);
    w.sorted_b = c.take<double>((size_t)n_jobs * mb);
    w.start = c.take<int64_t>((size_t)n_jobs * n_boot);
    w.extra = c.take<int32_t>((size_t)n_jobs * n_boot);
    w.boot = c.take<double>((size_t)n_jobs * n_boot);
    w.bytes = c.used;
    return w;
}

}  // namespace ncfa

using namespace ncfa;

extern "C" size_t ncfa_bootstrap_workspace_bytes(int n_jobs, int max_a, int max_b, int n_boot) {
    if (n_jobs <= 0 || max_a <= 0 || max_b < 0 || n_boot <= 0) return 0;
    return boot_ws(n_jobs, max_a, max_b, n_boot, nullptr).bytes;
}

extern "C" int ncfa_bootstrap_ratio_batched(const double *d_a, const int64_t *d_a_off, const int32_t *d_a_len,
                                            const double *d_b, const int64_t *d_b_off, const int32_t *d_b_len,
                                            int n_jobs, int max_a, int max_b, int n_boot,
                                            const uint64_t h_pcg_state[4], double q_lo, double q_hi, double *d_out,
                                            double *d_boot, int32_t *d_idx, void *d_workspace, size_t workspace_bytes,
                                            void *stream) {
    NCFA_REQUIRE(n_jobs >= 0, "n_jobs");
    if (n_jobs == 0) return NCFA_OK;
    NCFA_REQUIRE(d_a && d_a_off && d_a_len && d_out && d_workspace && h_pcg_state, "null pointer");
    NCFA_REQUIRE(max_a >= 1 && max_b >= 0 && n_boot >= 1, "max_a/max_b/n_boot");
    NCFA_REQUIRE((max_b == 0) == (d_b == nullptr), "d_b must be given exactly when max_b > 0");
    NCFA_REQUIRE(d_b == nullptr || (d_b_off && d_b_len), "d_b_off/d_b_len");
    NCFA_REQUIRE(d_idx == nullptr || n_jobs == 1, "d_idx is only supported for n_jobs == 1");
    NCFA_REQUIRE(n_jobs <= 65535 * 32, "n_jobs too large for one call");
    const size_t hist_ints = (size_t)max_a + (size_t)max_b;
    if (hist_ints * 4 > 200 * 1024) {
        set_error("bootstrap arrays too long: %zu + %zu values exceed the 51200-entry shared-memory histogram",
                  (size_t)max_a, (size_t)max_b);
        return NCFA_E_OVERFLOW;
    }
    const BootWs w = boot_ws(n_jobs, max_a, max_b, n_boot, d_workspace);
    if (int rc = check_workspace("bootstrap", workspace_bytes, w.bytes)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    double *boot = d_boot ? d_boot : w.boot;
    const u128 state0 = ((u128)h_pcg_state[0] << 64) | h_pcg_state[1];
    const u128 inc = ((u128)h_pcg_state[2] << 64) | h_pcg_state[3];
    const int mb = max_b > 0 ? max_b : 1;
    const int32_t *b_len = d_b ? d_b_len : nullptr;
    int rc;
    if ((rc = launch("boot_tables_kernel", boot_tables_kernel, 1, 32, 0, st, inc, w.tables))) return rc;
    if ((rc = launch("boot_rank_kernel", boot_rank_kernel, dim3(n_jobs, d_b ? 2 : 1), 256, 0, st, d_a, d_a_off, d_a_len,
                     d_b, d_b_off, d_b_len, max_a, mb, w.rank_a, w.rank_b, w.sorted_a, w.sorted_b)))
        return rc;
    const int threads = n_boot >= 1024 ? 1024 : ((n_boot + 31) / 32) * 32;
    if ((rc = launch("boot_offsets_kernel", boot_offsets_kernel, n_jobs, threads, 0, st, d_a_len, b_len, n_boot,
                     state0, inc, w.tables, w.start, w.extra)))
        return rc;
    // warps per CTA bounded by the shared-memory histogram; stride padded to avoid lock-step banks
    const int hist_stride = (int)((hist_ints + 1) | 1);
    int warps = (int)((200 * 1024) / ((size_t)hist_stride * 4));
    warps = warps > 8 ? 8 : (warps < 1 ? 1 : warps);
    const long long total = (long long)n_jobs * n_boot;
    long long blocks = (total + warps - 1) / warps;
    if (blocks > 148LL * 64) blocks = 148LL * 64;
    if ((rc = launch("boot_median_kernel", boot_median_kernel, (unsigned)blocks, warps * 32,
                     (size_t)warps * hist_stride * 4, st, d_a_len, b_len, max_a, mb, n_boot, n_jobs, state0, inc,
                     w.tables, w.start, w.extra, w.rank_a, w.rank_b, w.sorted_a, w.sorted_b, boot, d_idx, hist_stride)))
        return rc;
    return launch("boot_finish_kernel", boot_finish_kernel, n_jobs, 256,
                  n_boot <= kBootFinishMaxStaged ? (size_t)n_boot * 8 : 0, st, d_a_len, b_len, max_a, mb, n_boot,
                  w.sorted_a, w.sorted_b, boot, q_lo, q_hi, d_out);
}
