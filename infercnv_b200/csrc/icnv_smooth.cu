// icnv_smooth.cu - the smooth block of infercnv::run() as sm_100a kernels.
//
//   K1  group_partial_sums / combine_partials / bounds_from_means
//         .get_normal_gene_mean_bounds (R/inferCNV_ops.R:1708-1735): per-gene mean over each
//         reference group, summed in a fixed chunk order so the result does not depend on how
//         the cells are spread over GPUs.
//   K2  cell_pipeline_kernel: one CTA per cell, the cell's whole gene vector resident in shared
//         memory, all of [log2(x+1)] -> .subtract_expr (ops.R:1742-1786) -> clamp (ops.R:2970-2983)
//         -> .smooth_helper pyramid (ops.R:2483-2532, 2640-2661) -> .center_columns median
//         (ops.R:2094-2109) -> .subtract_expr again -> 2^x (ops.R:2814-2826) between ONE read and
//         ONE write of the column.
//
// Data layout: X[g + ld*c], a cell's genes contiguous (R column-major).  HBM-bound integer-free
// streaming work: no tensor cores; what matters is coalesced 8/16-byte accesses, the column kept
// on chip between the stages, and a grid that fills 148 SMs x resident CTAs.
#include <cfloat>
#include <cmath>
#include <cstring>
#include <cstdlib>
#include <algorithm>

#include "icnv_common.cuh"

namespace icnv {

// =================================================================================================
// K1: group means
// =================================================================================================

// grid: (ceil(G/256), n_chunks); thread = gene, block row = chunk of list entries.
// Adjacent threads read adjacent genes of the same cell: fully coalesced.  The sum over the
// chunk's cells runs in list order in every configuration (determinism across GPU counts).
__global__ void __launch_bounds__(256) group_partial_sums_kernel(const double *__restrict__ X, int64_t G, int64_t ldx,
                                                                 const int32_t *__restrict__ cells, int64_t n_cells,
                                                                 int chunk, int apply_log,
                                                                 double *__restrict__ partial) {
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    int64_t q = blockIdx.y;
    int64_t i0 = q * chunk;
    int64_t i1 = i0 + chunk < n_cells ? i0 + chunk : n_cells;
    double s = 0.0;
    int64_t i = i0;
    // 4 independent loads in flight per thread, added in list order
    for (; i + 4 <= i1; i += 4) {
        double v0 = X[g + ldx * (int64_t)cells[i]];
        double v1 = X[g + ldx * (int64_t)cells[i + 1]];
        double v2 = X[g + ldx * (int64_t)cells[i + 2]];
        double v3 = X[g + ldx * (int64_t)cells[i + 3]];
        if (apply_log) {
            v0 = log2(v0 + 1.0);
            v1 = log2(v1 + 1.0);
            v2 = log2(v2 + 1.0);
            v3 = log2(v3 + 1.0);
        }
        s += v0;
        s += v1;
        s += v2;
        s += v3;
    }
    for (; i < i1; ++i) {
        double v = X[g + ldx * (int64_t)cells[i]];
        if (apply_log) v = log2(v + 1.0);
        s += v;
    }
    partial[g + G * q] = s;
}

__global__ void __launch_bounds__(256) combine_partials_kernel(const double *__restrict__ partial, int64_t G,
                                                               int64_t n_chunks, double inv_count_num,
                                                               double *__restrict__ means) {
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    double s = 0.0;
    for (int64_t q = 0; q < n_chunks; ++q) s += partial[g + G * q];
    means[g] = s / inv_count_num;  // a true division by the count, as mean() does
}

__global__ void __launch_bounds__(256) bounds_from_means_kernel(const double *__restrict__ means, int64_t G, int n_grp,
                                                                double *__restrict__ lo, double *__restrict__ hi,
                                                                double *__restrict__ mid) {
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    double mn = means[g], mx = means[g], s = 0.0;
    for (int k = 0; k < n_grp; ++k) {
        double m = means[g + G * k];
        mn = fmin(mn, m);
        mx = fmax(mx, m);
        s += m;
    }
    lo[g] = mn;
    hi[g] = mx;
    if (mid) mid[g] = s / (double)n_grp;
}

// Reference bounds straight from the (all-gathered) chunk sums: per gene and group the chunk rows of every rank are added
// in rank-major, then chunk order - the global list order, whatever the rank count - divided by the group size, and the
// min / max / mean over the groups written (ops.R:1708-1735).  One launch instead of a combine per group, a stack and
// bounds_from_means; zero rows (a rank's padding up to the longest rank) do not change a sum.
struct PartialBoundsParams {
    const double *part;   // [world][tot_rows][G]
    int64_t G, tot_rows;
    int world, n_grp;
    int row_off[33];      // rows of group k inside a rank's block: row_off[k] .. row_off[k + 1]
    double count[32];     // global group sizes
    double *lo, *hi, *mid;
    double *means;        // optional: the group means themselves, [n_grp][G]
};

__global__ void __launch_bounds__(256) bounds_from_partials_kernel(const PartialBoundsParams p) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= p.G) return;
    double mn = 0.0, mx = 0.0, sm = 0.0;
    for (int k = 0; k < p.n_grp; ++k) {
        double s = 0.0;
        const int r0 = p.row_off[k], r1 = p.row_off[k + 1];
        for (int w = 0; w < p.world; ++w) {
            const double *__restrict__ base = p.part + p.G * ((int64_t)w * p.tot_rows);
            for (int q = r0; q < r1; ++q) s += base[g + p.G * q];
        }
        const double m = s / p.count[k];  // a true division by the count, as mean() does
        if (p.means) p.means[g + p.G * k] = m;
        if (k == 0) {
            mn = m;
            mx = m;
        }
        mn = fmin(mn, m);
        mx = fmax(mx, m);
        sm += m;
    }
    if (p.lo) {
        p.lo[g] = mn;
        p.hi[g] = mx;
    }
    if (p.mid) p.mid[g] = sm / (double)p.n_grp;
}

// inv_log variant of the group mean: log2(mean(2^x - 1) + 1) (ops.R:1714-1717)
__global__ void __launch_bounds__(256) group_partial_sums_invlog_kernel(const double *__restrict__ X, int64_t G,
                                                                        int64_t ldx, const int32_t *__restrict__ cells,
                                                                        int64_t n_cells, int chunk,
                                                                        double *__restrict__ partial) {
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    int64_t q = blockIdx.y;
    int64_t i0 = q * chunk;
    int64_t i1 = i0 + chunk < n_cells ? i0 + chunk : n_cells;
    double s = 0.0;
    for (int64_t i = i0; i < i1; ++i) s += exp2(X[g + ldx * (int64_t)cells[i]]) - 1.0;
    partial[g + G * q] = s;
}

__global__ void __launch_bounds__(256) invlog_finish_kernel(double *__restrict__ means, int64_t n) {
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g < n) means[g] = log2(means[g] + 1.0);
}

// =================================================================================================
// K2: fused per-cell pipeline
// =================================================================================================

struct Seg {
    int start;   // first gene of the segment
    int len;     // number of genes (0 = idle thread)
    int cs;      // chromosome start
    int ce;      // chromosome end (exclusive)
    int tfirst;  // first thread of this chromosome (== own index for idle threads)
    int chr;     // chromosome index
};

struct CellParams {
    const double *X;
    int64_t G, ldx;
    const int32_t *cols;
    int64_t n_cols;
    double *Y;
    int64_t ldy;
    const Seg *segs;
    int apply_log;
    const double *lo1, *hi1, *mid1;
    double threshold;
    int window, h;
    int center;  // 0 none, 1 median, 2 mean
    const double *lo2, *hi2, *mid2;
    int apply_exp2;
    int *err_flag;
    int s_elems;  // doubles reserved per column buffer (G rounded up to even)
    int K;
    int q_elems;  // cell_pipeline3_kernel<NT, true>: doubles of the landing / padded-Q buffer (G + K (2h + 2), even)
    int ipad;     // cell_pipeline3_kernel<NT, true>: entries in front of the reciprocal-denominator table (>= longest slice, even)
};

constexpr int CAND_MAX = 64;   // candidates ranked directly at the end of the selection

__device__ unsigned long long g_stats[16];  // [0] median rounds, [1] medians, [2] split exits, [3] gather exits,
                                            // [4..9] cycles spent by CTA 0 in: wait, A, B scans, B outputs, C median, D

// ---- block-wide reductions with one __syncthreads each (double-buffered scratch) ----------------
template <int NW>
struct Red {
    double d[2][2][NW];
    int i[2][2][NW];
};

template <int NW>
__device__ __forceinline__ void block_sum2i(Red<NW> &r, int &phase, int a, int b, int &A, int &B) {
    a = __reduce_add_sync(0xffffffffu, a);
    b = __reduce_add_sync(0xffffffffu, b);
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) {
        r.i[phase][0][w] = a;
        r.i[phase][1][w] = b;
    }
    __syncthreads();
    // second level: every warp folds the NW partials with one redux each (no serial loop over warps)
    const int pa = (lane < NW) ? r.i[phase][0][lane] : 0;
    const int pb = (lane < NW) ? r.i[phase][1][lane] : 0;
    A = __reduce_add_sync(0xffffffffu, pa);
    B = __reduce_add_sync(0xffffffffu, pb);
    phase ^= 1;
}

// op: 0 = (min, max), 1 = (sum, sum), 2 = (max, min)
template <int NW, int OP>
__device__ __forceinline__ void block_red2d(Red<NW> &r, int &phase, double a, double b, double &A, double &B) {
    const double ida = (OP == 0) ? DBL_MAX : ((OP == 1) ? 0.0 : -DBL_MAX);
    const double idb = (OP == 0) ? -DBL_MAX : ((OP == 1) ? 0.0 : DBL_MAX);
    auto fold = [&](double &u, double &v) {
        if (OP == 0) {
            u = warp_min_d(u);
            v = warp_max_d(v);
        } else if (OP == 1) {
            u = warp_sum_d(u);
            v = warp_sum_d(v);
        } else {
            u = warp_max_d(u);
            v = warp_min_d(v);
        }
    };
    fold(a, b);
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) {
        r.d[phase][0][w] = a;
        r.d[phase][1][w] = b;
    }
    __syncthreads();
    double pa = (lane < NW) ? r.d[phase][0][lane] : ida;
    double pb = (lane < NW) ? r.d[phase][1][lane] : idb;
    fold(pa, pb);
    A = pa;
    B = pb;
    phase ^= 1;
}

#include "icnv_math_tables.inc"
__device__ double g_log_tab[128][2];
__device__ double g_exp_tab[128];

// log2(x + 1) as the reference computes it (add, then log2; ops.R:2760), table + degree-6 polynomial:
// v = 2^e * m, m in [1,2); c_i = 1/inv_c[i] is the table point next to m, r = m*inv_c - 1 (|r| < 2^-8),
// log2 v = e + log2 c_i + log2(1 + r).  Error <= 3e-16 (relative, absolute below 1).  ~25 instructions
// against ~90 for the library log2.
__constant__ double k_logc[6] = {ICNV_LOGC0, ICNV_LOGC1, ICNV_LOGC2, ICNV_LOGC3, ICNV_LOGC4, ICNV_LOGC5};
__constant__ double k_expc[5] = {ICNV_EXPC0, ICNV_EXPC1, ICNV_EXPC2, ICNV_EXPC3, ICNV_EXPC4};
__device__ __noinline__ double slow_log2(double v) { return log2(v); }
__device__ __noinline__ double slow_exp2(double x) { return exp2(x); }

__device__ __forceinline__ double fast_log2_1p(double x, const double2 *__restrict__ ltab) {
    const double v = x + 1.0;
    const int hi = __double2hiint(v);
    if ((unsigned)(hi - 0x00100000) >= 0x7fe00000u) return slow_log2(v);  // zero, negative, denormal, inf, nan
    const int e = (hi >> 20) - 1023;
    const double m = __hiloint2double((hi & 0x000fffff) | 0x3ff00000, __double2loint(v));
    const double2 t = ltab[(hi >> 13) & 127];
    const double r = fma(m, t.x, -1.0);
    double q = fma(r, k_logc[5], k_logc[4]);   // constant-bank operands: no immediates to materialise
    q = fma(r, q, k_logc[3]);
    q = fma(r, q, k_logc[2]);
    q = fma(r, q, k_logc[1]);
    q = fma(r, q, k_logc[0]);
    return (double)e + fma(r, q, t.y);
}

// The same without the range branch: `slow` is raised instead when the argument is outside the fast path's domain (the
// value returned is then meaningless and the caller re-evaluates with fast_log2_1p).  Lets several evaluations run as one
// straight-line block - the per-value branch with its convergence barrier costs ~8 issue slots of ~35.
__device__ __forceinline__ double fast_log2_1p_nc(double x, const double2 *__restrict__ ltab, bool &slow) {
    const double v = x + 1.0;
    const int hi = __double2hiint(v);
    slow |= (unsigned)(hi - 0x00100000) >= 0x7fe00000u;
    const int e = (hi >> 20) - 1023;
    const double m = __hiloint2double((hi & 0x000fffff) | 0x3ff00000, __double2loint(v));
    const double2 t = ltab[(hi >> 13) & 127];
    const double r = fma(m, t.x, -1.0);
    double q = fma(r, k_logc[5], k_logc[4]);
    q = fma(r, q, k_logc[3]);
    q = fma(r, q, k_logc[2]);
    q = fma(r, q, k_logc[1]);
    q = fma(r, q, k_logc[0]);
    return (double)e + fma(r, q, t.y);
}

// 2^x (invert_log2, ops.R:2818): x = k/128 + r, 2^x = 2^(k>>7) * T[k & 127] * 2^r, degree-5 polynomial.
__device__ __forceinline__ double fast_exp2(double x, const double *__restrict__ etab) {
    if (!(fabs(x) < 1000.0)) return slow_exp2(x);
    const double MAGIC = 6755399441055744.0;  // 1.5 * 2^52
    const double kk = fma(x, 128.0, MAGIC);
    const int ki = __double2loint(kk);
    const double r = fma(kk - MAGIC, -0.0078125, x);  // exact
    double q = fma(r, k_expc[4], k_expc[3]);
    q = fma(r, q, k_expc[2]);
    q = fma(r, q, k_expc[1]);
    q = fma(r, q, k_expc[0]);
    const double t = etab[ki & 127];
    const double res = fma(t * r, q, t);
    return __hiloint2double(__double2hiint(res) + ((ki >> 7) << 20), __double2loint(res));
}

__device__ __forceinline__ double fast_exp2_nc(double x, const double *__restrict__ etab, bool &slow) {
    slow |= !(fabs(x) < 1000.0);
    const double MAGIC = 6755399441055744.0;  // 1.5 * 2^52
    const double kk = fma(x, 128.0, MAGIC);
    const int ki = __double2loint(kk);
    const double r = fma(kk - MAGIC, -0.0078125, x);  // exact
    double q = fma(r, k_expc[4], k_expc[3]);
    q = fma(r, q, k_expc[2]);
    q = fma(r, q, k_expc[1]);
    q = fma(r, q, k_expc[0]);
    const double t = etab[ki & 127];
    const double res = fma(t * r, q, t);
    return __hiloint2double(__double2hiint(res) + ((ki >> 7) << 20), __double2loint(res));
}

// dead-band subtraction, .subtract_expr (ops.R:1764-1769): strict inequalities
__device__ __forceinline__ double sub_bounds(double x, double lo, double hi) {
    // x-hi above the band, x-lo below it, exactly 0 inside (lo <= hi always).  Written with compares and selects:
    // double-precision fmin / fmax expand to ~17 instructions each on sm_100, this form is 8 in total.
    const double above = x - hi, below = x - lo;
    return (x > hi) ? above : ((x < lo) ? below : 0.0);
}

// apply_max_threshold_bounds (ops.R:2970-2983): clamp to [-thr, thr]
__device__ __forceinline__ double clamp_sym(double x, double thr) { return (fabs(x) > thr) ? copysign(thr, x) : x; }

// Stage A / D of the fused-block configuration for U genes STRIDE apart, as one straight-line block: no bounds tests, and no
// range branch per value - fast_log2_1p_nc / fast_exp2_nc only raise `slow`, and the group is then re-evaluated through the
// library path (zero / negative / denormal / non-finite x + 1; |x| >= 1000 or NaN).
template <int U, int STRIDE>
__device__ __forceinline__ void stage_a_group(const double *__restrict__ src, double *__restrict__ dstv,
                                              const double *__restrict__ lo1, const double *__restrict__ hi1, int g0, double thr,
                                              const double2 *__restrict__ ltab, bool &bad) {
    double v[U], lo[U], hi[U], x[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        v[u] = src[g0 + u * STRIDE];
        lo[u] = lo1[g0 + u * STRIDE];
        hi[u] = hi1[g0 + u * STRIDE];
    }
    bool slow = false;
#pragma unroll
    for (int u = 0; u < U; ++u) x[u] = fast_log2_1p_nc(v[u], ltab, slow);
    if (slow) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (!is_finite_d(v[u])) bad = true;
            x[u] = fast_log2_1p(v[u], ltab);
        }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) dstv[g0 + u * STRIDE] = clamp_sym(sub_bounds(x[u], lo[u], hi[u]), thr);
}

template <int U, int STRIDE>
__device__ __forceinline__ void stage_d_group(const double *__restrict__ src, double *__restrict__ dst,
                                              const double *__restrict__ lo2, const double *__restrict__ hi2, int g0, double centre,
                                              const double *__restrict__ etab) {
    double v[U], lo[U], hi[U], x[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        v[u] = src[g0 + u * STRIDE];
        lo[u] = lo2[g0 + u * STRIDE];
        hi[u] = hi2[g0 + u * STRIDE];
    }
    bool slow = false;
#pragma unroll
    for (int u = 0; u < U; ++u) {
        v[u] = sub_bounds(v[u] - centre, lo[u], hi[u]);
        x[u] = fast_exp2_nc(v[u], etab, slow);
    }
    if (slow) {
#pragma unroll
        for (int u = 0; u < U; ++u) x[u] = fast_exp2(v[u], etab);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) dst[g0 + u * STRIDE] = x[u];
}

// ---- mbarrier / bulk-copy (TMA) helpers: the next cell's column is fetched by the copy engine
//      into shared memory while the CTA works on the current one --------------------------------
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(void *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, void *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(void *bar, unsigned parity) {
    unsigned ok = 0;
    const unsigned a = smem_u32(bar);
    while (!ok) {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(ok)
            : "r"(a), "r"(parity)
            : "memory");
    }
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

// =================================================================================================
// K2 v3: same pipeline, values never leave shared memory
// =================================================================================================
//
// v2 above keeps every thread's smoothed values in a register array across the median, which forces all
// per-gene loops to be fully unrolled with length predicates (~430 instructions per gene, 170 KB of code).
// v3 ping-pongs between the two shared-memory buffers instead: the raw column lands in buffer `in`, the
// element-wise steps write x' to `oth`, the prefix sums run in place there, the smoothed values go back to
// `in`, and the next cell's bulk copy is issued into `oth` as soon as Q is no longer needed.  All per-gene
// loops are short rolled loops over the thread's own slice; the median counts straight from shared memory.

// median of the n values vals[a0 .. a0+len) of all threads (same selection as block_median)
// median of the n values vals[a0 .. a0+len) of all threads (same selection as block_median).  s1 / s2 are this
// thread's sum and sum of squares of its values (accumulated while they were produced): they only place the
// first two pivots.  Min / max are not needed: the bracket starts at (-DBL_MAX, DBL_MAX].
template <int NT>
__device__ __forceinline__ double block_median_smem(const double *__restrict__ vals, int a0, int len, int n, double s1,
                                                    double s2, Red<NT / 32> &red, int &phase, double *cand, int *cand_n) {
    constexpr int NW = NT / 32;
    const int kA = (n - 1) >> 1, kB = n >> 1;
    const double *v0 = vals + a0;
    if (threadIdx.x == 0) *cand_n = 0;   // made visible by the reductions' barriers long before the gather
    double S1, S2;
    block_red2d<NW, 1>(red, phase, s1, s2, S1, S2);
    const double mean = S1 / (double)n;
    const double var = S2 / (double)n - mean * mean;
    const double sd = var > 0.0 ? sqrt(var) : 0.0;
    // invariant: #(x <= lo) <= kA and #(x <= hi) >= kB + 1
    double lo = -DBL_MAX, hi = DBL_MAX;
    int Flo = 0, Fhi = n;
    // first bracket: mean +- 0.35 sd holds the median of anything roughly unimodal and has near-uniform density
    // inside, which is what the interpolation rounds assume; a miss is repaired by the min / max pass below
    double p1 = mean - 0.35 * sd, p2 = mean + 0.35 * sd;
    bool force_bisect = false;
    double a_res = 0.0, b_res = 0.0;
    bool done = false;
    for (int round = 0; round < 200 && !done; ++round) {
        const int m = Fhi - Flo;
        if (m <= CAND_MAX) break;
        if (threadIdx.x == 0) atomicAdd(&g_stats[0], 1ull);
        if (round > 0 && (lo == -DBL_MAX || hi == DBL_MAX)) {
            // rare (zero variance, or a variance lost to cancellation): bound the bracket by the true extremes
            double mn = DBL_MAX, mx = -DBL_MAX;
            for (int t = 0; t < len; ++t) {
                mn = fmin(mn, v0[t]);
                mx = fmax(mx, v0[t]);
            }
            double MN, MX;
            block_red2d<NW, 0>(red, phase, mn, mx, MN, MX);
            if (!(MN < MX)) {   // all values equal
                a_res = b_res = MN;
                done = true;
                break;
            }
            double below = double_of_key(key_of(MN) - 1ull);
            if (!(below < MN)) below = double_of_key(key_of(MN) - 2ull);   // MN == +0.0: one key below is -0.0
            lo = fmax(lo, below);
            hi = fmin(hi, MX);
        }
        if (round > 0) {
            if (force_bisect) {   // rare: interpolation failed to halve the bracket -> bisect in key space
                const unsigned long long klo = key_of(lo), khi = key_of(hi);
                if (khi - klo < 2ull) {   // no double strictly between: every candidate equals hi
                    a_res = b_res = hi;
                    done = true;
                    break;
                }
                p1 = p2 = double_of_key(klo + ((khi - klo) >> 1));
            } else {
                // pivot placement only has to be identical in every thread, not accurate: cheap float math
                const float mf = (float)m;
                const float inv_m = __frcp_rn(mf);
                const float f = ((float)(kA - Flo) + 0.5f * (float)(kB - kA) + 0.5f) * inv_m;
                float wfrac = (3.0f * sqrtf(mf) + 8.0f) * inv_m;
                wfrac = fminf(wfrac, 0.5f);
                const double span = hi - lo;   // finite after the first round unless the data are degenerate
                const double pc = lo + span * (double)f;
                p1 = pc - span * (double)(0.5f * wfrac);
                p2 = pc + span * (double)(0.5f * wfrac);
            }
        }
        if (!(p1 > lo && p1 < hi) || !(p2 > lo && p2 < hi) || !(p1 <= p2)) {
            // degenerate placement (infinite span, rounding onto a bound, all-equal data ...): key-space midpoint
            const unsigned long long klo = key_of(lo), khi = key_of(hi);
            if (khi - klo < 2ull) {
                a_res = b_res = hi;
                done = true;
                break;
            }
            p1 = p2 = double_of_key(klo + ((khi - klo) >> 1));
        }
        int c1 = 0, c2 = 0;
#pragma unroll 4
        for (int t = 0; t < len; ++t) {
            const double v = v0[t];
            c1 += (v <= p1) ? 1 : 0;
            c2 += (v <= p2) ? 1 : 0;
        }
        int C1, C2;
        block_sum2i<NW>(red, phase, c1, c2, C1, C2);
        double split = 0.0;
        bool do_split = false;
        if (C1 >= kB + 1) {
            hi = p1;
            Fhi = C1;
        } else if (C1 > kA) {
            split = p1;
            do_split = true;
        } else if (C2 >= kB + 1) {
            lo = p1;
            Flo = C1;
            hi = p2;
            Fhi = C2;
        } else if (C2 > kA) {
            split = p2;
            do_split = true;
        } else {
            lo = p2;
            Flo = C2;
        }
        if (do_split) {   // s_kA <= split < s_kB: neighbours of the split point
            double below = -DBL_MAX, above = DBL_MAX;
            for (int t = 0; t < len; ++t) {
                const double v = v0[t];
                if (v <= split) below = fmax(below, v);
                else above = fmin(above, v);
            }
            block_red2d<NW, 2>(red, phase, below, above, a_res, b_res);
            done = true;
            break;
        }
        const int m_new = Fhi - Flo;
        force_bisect = (2 * m_new > m) && !force_bisect;
    }
    if (done) {
        if (threadIdx.x == 0) atomicAdd(&g_stats[2], 1ull);
        return (a_res + b_res) * 0.5;
    }
    if (threadIdx.x == 0) atomicAdd(&g_stats[3], 1ull);
    // ---- gather the <= CAND_MAX candidates in (lo, hi] and rank them --------------------------------
    for (int t = 0; t < len; ++t) {
        const double v = v0[t];
        if (v > lo && v <= hi) {
            const int slot = atomicAdd(cand_n, 1);
            if (slot < CAND_MAX) cand[slot] = v;
        }
    }
    __syncthreads();
    int m = *cand_n;
    if (m > CAND_MAX) m = CAND_MAX;   // cannot happen (m == Fhi - Flo); keeps the loop bounded
    const int ra = kA - Flo, rb = kB - Flo;
    {   // one warp per candidate: its 32 lanes compare it with all (<= 64) candidates, one redux gives the rank
        const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
        const double u1 = (lane < m) ? cand[lane] : INFINITY;
        const double u2 = (lane + 32 < m) ? cand[lane + 32] : INFINITY;
        for (int i = w; i < m; i += NW) {
            const double v = cand[i];
            int cnt = ((u1 < v) || (u1 == v && lane < i)) ? 1 : 0;
            cnt += ((u2 < v) || (u2 == v && lane + 32 < i)) ? 1 : 0;
            const int rank = __reduce_add_sync(0xffffffffu, cnt);
            if (lane == 0) {
                if (rank == ra) cand[CAND_MAX] = v;
                if (rank == rb) cand[CAND_MAX + 1] = v;
            }
        }
    }
    __syncthreads();
    return (cand[CAND_MAX] + cand[CAND_MAX + 1]) * 0.5;   // cand is next touched a whole cell (many barriers) later
}

// ---- median by one histogram pass ----------------------------------------------------------------
// |mean - median| <= sd for any distribution, so the HIST_NB equal-width bins spanning mean +- sd hold both middle
// order statistics.  bin(v) = low word of fma(v, scale, C) with C = 1.5*2^52 - (mean - sd)*scale is a monotone
// function of v evaluated by the same instruction in both passes, so "values in lower bins" are exactly the values
// ranked below the bin: pass 1 counts (shared-memory atomics for the inner bins, a register for "below"), a
// block-wide scan finds the bin(s) holding ranks kA and kB, pass 2 gathers those bins' values (<= CAND_MAX,
// otherwise the bracketing selection above takes over) and they are ranked directly.  Two passes over the
// values, any thread reads any value: both passes use the coalesced 16-byte mapping.
constexpr int HIST_NB = 2048;

// n = number of (finite) values, n_slots = slots of `vals` to walk (>= n; the extra slots hold +inf and are neither
// counted nor gathered).
template <int NT, int NB = HIST_NB>
__device__ __forceinline__ bool block_median_hist(const double *__restrict__ vals, int n, double inv_n, double S1, double S2, int *hist, int dump_off,
                                                  int *hres, int *wcnt, double *cand, int *cand_n, double &result, int n_slots = 0) {
    constexpr int NW = NT / 32;
    constexpr int BPT = NB / NT;   // bins scanned per thread
    static_assert(NB % NT == 0 && BPT >= 1 && BPT <= 8, "the bin count must be a small multiple of NT");
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned dump = (unsigned)(dump_off + lane);   // index (relative to hist) of this lane's spare word
    const int kA = (n - 1) >> 1, kB = n >> 1;
    // Bin geometry in cheap arithmetic: every thread evaluates the same instruction sequence, so all of them and both
    // passes bin with identical scale / C, and the median itself never depends on them (the candidates are ranked exactly) -
    // a single-precision reciprocal square root is enough for "about mean +- sd".  ~25 instead of ~100 instructions per
    // thread and cell (two divisions, a square root and a third division in double precision before).
    const double mean = S1 * inv_n;
    const double var = fma(S2, inv_n, -mean * mean);
    if (!(var > 0.0) || n <= 4 * CAND_MAX) return false;
    const float rs = rsqrtf((float)var);
    const double sd = var * (double)rs;
    const double scale = (double)(rs * (0.5f * NB));
    if (!(scale < 1e290) || !(scale > 0.0)) return false;   // var outside the single-precision range: bracketing selection
    const double MAGIC = 6755399441055744.0;   // 1.5 * 2^52: integers 0 .. 2^32-1 land in the low word, high word HI0
    constexpr int HI0 = 0x43380000;
    const double C = fma(sd - mean, scale, MAGIC);
    if (tid == 0) {
        hres[0] = -1;
        hres[2] = -1;
        *cand_n = 0;
    }
    const double2 *v2 = reinterpret_cast<const double2 *>(vals);
    const int n2 = ((n_slots > 0 ? n_slots : n) + 1) >> 1;   // an odd n is padded with +inf (never counted, never gathered)
    int cb = 0;
#pragma unroll 2
    for (int i = tid; i < n2; i += NT) {
        const double2 v = v2[i];
        const double tx = fma(v.x, scale, C), ty = fma(v.y, scale, C);
        const int hx = __double2hiint(tx), hy = __double2hiint(ty);
        const unsigned lx = (unsigned)__double2loint(tx), ly = (unsigned)__double2loint(ty);
        // values outside mean +- sd count into this lane's own spare word behind the tables (never read; per lane, so that
        // a third of the warp does not pile onto one address): one unconditional atomic per value instead of a branch around it
        atomicAdd(&hist[(hx == HI0 && lx < (unsigned)NB) ? lx : dump], 1);
        atomicAdd(&hist[(hy == HI0 && ly < (unsigned)NB) ? ly : dump], 1);
        cb += (hx < HI0) ? 1 : 0;
        cb += (hy < HI0) ? 1 : 0;
    }
    cb = __reduce_add_sync(0xffffffffu, cb);
    if (lane == 0) wcnt[warp] = cb;
    __syncthreads();   // histogram complete
    int cnt[BPT];
    int s = 0;
#pragma unroll
    for (int k = 0; k < BPT; ++k) {
        cnt[k] = hist[tid * BPT + k];
        hist[tid * BPT + k] = 0;   // left clean for the next cell
        s += cnt[k];
    }
    int inc = s;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) wcnt[NW + warp] = inc;
    __syncthreads();
    {
        const int below = __reduce_add_sync(0xffffffffu, (lane < NW) ? wcnt[lane] : 0);
        const int prev = __reduce_add_sync(0xffffffffu, (lane < warp) ? wcnt[NW + lane] : 0);
        int o = below + prev + inc - s;
#pragma unroll
        for (int k = 0; k < BPT; ++k) {
            const int c = cnt[k];
            if (c > 0) {
                if (o <= kA && kA < o + c) {
                    hres[0] = tid * BPT + k;
                    hres[1] = o;
                }
                if (o <= kB && kB < o + c) {
                    hres[2] = tid * BPT + k;
                    hres[3] = o + c;
                }
            }
            o += c;
        }
    }
    __syncthreads();
    const int bA = hres[0], offA = hres[1], bB = hres[2], endB = hres[3];
    if (bA < 0 || bB < 0 || endB - offA > CAND_MAX) return false;   // histogram already zeroed
    const int m = endB - offA;
#pragma unroll 2
    for (int i = tid; i < n2; i += NT) {
        const double2 v = v2[i];
        const double tx = fma(v.x, scale, C), ty = fma(v.y, scale, C);
        const int hx = __double2hiint(tx), hy = __double2hiint(ty);
        const unsigned lx = (unsigned)__double2loint(tx), ly = (unsigned)__double2loint(ty);
        const bool gx = hx == HI0 && (lx - (unsigned)bA) <= (unsigned)(bB - bA);
        const bool gy = hy == HI0 && (ly - (unsigned)bA) <= (unsigned)(bB - bA);
        if (gx | gy) {   // at most CAND_MAX of the n values: one branch per pair
            if (gx) cand[atomicAdd(cand_n, 1)] = v.x;
            if (gy) cand[atomicAdd(cand_n, 1)] = v.y;
        }
    }
    __syncthreads();
    const int ra = kA - offA, rb = kB - offA;
    {   // one warp per candidate: its 32 lanes compare it with all (<= 64) candidates, one redux gives the rank
        const double u1 = (lane < m) ? cand[lane] : INFINITY;
        const double u2 = (lane + 32 < m) ? cand[lane + 32] : INFINITY;
        for (int i = warp; i < m; i += NW) {
            const double v = cand[i];
            int c = ((u1 < v) || (u1 == v && lane < i)) ? 1 : 0;
            c += ((u2 < v) || (u2 == v && lane + 32 < i)) ? 1 : 0;
            const int rank = __reduce_add_sync(0xffffffffu, c);
            if (lane == 0) {
                if (rank == ra) cand[CAND_MAX] = v;
                if (rank == rb) cand[CAND_MAX + 1] = v;
            }
        }
    }
    __syncthreads();
    result = (cand[CAND_MAX] + cand[CAND_MAX + 1]) * 0.5;
    return true;
}

// PADQ = true (default when it fits): the prefix sums Q are written to a padded copy of the column - per chromosome h + 2
// zeros in front (Q(-1) .. Q(-h-2)) and the h values of the linear continuation behind - so the smoothing outputs read
// Q(j+h), Q(j-1), Q(j-h-2) at fixed offsets from one running pointer instead of selecting among the Q array, the
// continuation table and a zero slot per load (53 -> ~20 instructions per gene in that loop; results bit-identical).
// Buffer roles are then fixed instead of ping-pong: buf0 = landing buffer of the bulk copy, later the padded Q;
// buf1 = x', later the smoothed values that stages C and D read.
// LFIX > 0: every busy thread's slice has at most LFIX genes (the launcher's segment length): the three scan passes are then
// fully unrolled with a per-gene predicate instead of counted loops with remainders (21 -> 12.5 instructions per gene over
// the three passes); LFIX = 0 is the generic form.
template <int NT, bool PADQ, int LFIX>
__global__ void __launch_bounds__(NT, 1) cell_pipeline3_kernel(const CellParams p) {
    constexpr bool FIX = LFIX > 0;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NW = NT / 32;
    double2 *ltab = reinterpret_cast<double2 *>(smem_raw);
    double *etab = reinterpret_cast<double *>(ltab + 128);
    double *buf0 = etab + 128;
    double *buf1 = buf0 + (PADQ ? p.q_elems : p.s_elems);
    double *invD = buf1 + p.s_elems + (PADQ ? p.ipad : 0);   // PADQ: p.ipad (even) copies of invD[0] in front, indices -ipad .. -1
    double *ptot = invD + (p.h + 2);
    double *qtot = ptot + p.K;
    double *tails = qtot + p.K;                              // [2][NW]
    double *cand = tails + 2 * NW;
    Red<NW> &red = *reinterpret_cast<Red<NW> *>(cand + CAND_MAX + 2);
    double *rext = reinterpret_cast<double *>(&red + 1);     // [K][h] linear continuation of Q past each chromosome end
    double *zslot = rext + (PADQ ? 0 : p.K * p.h);           // a 0.0 the edge loads can point at (Q before the start)
    unsigned long long *bar = reinterpret_cast<unsigned long long *>(zslot + 2);
    int *hist = reinterpret_cast<int *>(bar + 2);            // HIST_NB bins, zero between cells
    int *hres = hist + HIST_NB;                              // 4 results of the bin search (+4 spare)
    int *wcnt = hres + 8;                                    // [2][NW]
    int *cand_n = wcnt + 2 * NW;
    int *chr_cs = cand_n + 2;                                // PADQ: [K] chromosome start, [K] chromosome length
    int *chr_n = chr_cs + p.K;
    int *hdump = chr_n + p.K;                                // [32] per-lane spare words of the histogram pass
    double *const sm = reinterpret_cast<double *>(smem_raw); // everything below is indexed relative to this

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = (int)p.G;
    const int h = p.h;
    const bool do_smooth = p.window >= 2;
    const double inv_G = 1.0 / (double)G;   // histogram-median bin geometry only
    int phase = 0;
    unsigned parity = 0;
    if (do_smooth) {
        const double full = (double)(h + 1) * (double)(h + 1);
        for (int r = tid; r <= h; r += NT) invD[r] = 1.0 / (full - 0.5 * (double)r * (double)(r + 1));
        if (PADQ)   // PADQ: IPAD copies of entry 0 in front of the table (see the output loop)
            for (int r = tid; r < p.ipad; r += NT) invD[-1 - r] = 1.0 / full;
    }
    if (tid == 0) {
        mbar_init(bar, 1);
        zslot[0] = 0.0;
        buf0[p.s_elems - 1] = INFINITY;   // pad of an odd G: never counted by the median (overwritten when G is even)
        buf1[p.s_elems - 1] = INFINITY;
    }
    for (int i = tid; i < HIST_NB; i += NT) hist[i] = 0;
    for (int i = tid; i < 128; i += NT) {
        ltab[i] = make_double2(g_log_tab[i][0], g_log_tab[i][1]);
        etab[i] = g_exp_tab[i];
    }
    const Seg seg = p.segs[tid];
    const int len = seg.len, a0 = seg.start, cs = seg.cs, ce = seg.ce, n = ce - cs;
    if (PADQ) {   // chromosome geometry for the pad loop: empty chromosomes own no thread and keep length 0
        for (int i = tid; i < p.K; i += NT) chr_n[i] = 0;
        __syncthreads();
        if (len > 0 && a0 == cs) {
            chr_cs[seg.chr] = cs;
            chr_n[seg.chr] = n;
        }
    }
    const int lane_first = max(seg.tfirst - (tid - lane), 0);
    const int wfirst = seg.tfirst >> 5;
    // PADQ output loop: index of the slice's first reciprocal denominator and its step per gene.  Inside a chromosome of at
    // least 2h + 1 genes only one end can be within h genes: rl = max(h - j, 0) falls by one per gene (step -1), rr =
    // max(j - (n - 1 - h), 0) rises (step +1); negative indices are the table's front pad = entry 0, so no clamp is needed
    // as long as the start index is >= -ipad.  Slices that see both ends (2h + 1 <= n < 2h + 1 + len) take the general loop.
    int r0I = 0, dI = 0;
    bool pad_fast = n >= 2 * h + 1;
    if (PADQ && pad_fast) {
        const int j0 = a0 - cs, hl = h - j0, hr = j0 - (n - 1 - h);
        if (hl > 0 && hr + len - 1 > 0) pad_fast = false;
        else if (hl > 0) { r0I = hl; dI = -1; }
        else if (hr + len - 1 > 0) { r0I = max(hr, -p.ipad); dI = 1; }
    }
    bool bad = false;
    const unsigned col_bytes = (unsigned)(p.G * sizeof(double));
    auto tma_ok = [&](int64_t col) {
        return ((col_bytes & 15u) == 0) && ((reinterpret_cast<uintptr_t>(p.X + p.ldx * col) & 15u) == 0);
    };
    double *in = buf0, *oth = buf1;
#ifdef ICNV_STAGE_TIMERS
    long long tstamp = clock64();
    unsigned long long tacc[6] = {0, 0, 0, 0, 0, 0};
    auto lap = [&](int slot) {   // stage timing by one thread of CTA 0 (diagnostic build, see icnv_debug_stats)
        if (tid == 0 && blockIdx.x == 0) {
            const long long now = clock64();
            tacc[slot] += (unsigned long long)(now - tstamp);
            tstamp = now;
        }
    };
#else
    auto lap = [](int) {};
#endif
    __syncthreads();
    if (tid == 0 && (int64_t)blockIdx.x < p.n_cols) {
        const int64_t col0 = p.cols ? (int64_t)p.cols[blockIdx.x] : (int64_t)blockIdx.x;
        if (tma_ok(col0)) {
            fence_proxy_async();
            mbar_expect_tx(bar, col_bytes);
            bulk_g2s(in, p.X + p.ldx * col0, col_bytes, bar);
        }
    }

    for (int64_t ci = blockIdx.x; ci < p.n_cols; ci += gridDim.x) {
        const int64_t col = p.cols ? (int64_t)p.cols[ci] : ci;
        double *__restrict__ dst = p.Y + p.ldy * ci;
        // ---- A: raw column (in) -> x' (oth) -------------------------------------------------------------
        if (tma_ok(col)) {
            mbar_wait(bar, parity);
            parity ^= 1u;
        } else {
            const double *__restrict__ src = p.X + p.ldx * col;
            for (int g = tid; g < G; g += NT) in[g] = src[g];
            __syncthreads();
        }
        lap(0);
        if (p.apply_log && p.lo1 && p.threshold > 0.0) {
            // groups of four genes NT apart as one straight-line block (no bounds tests, no per-value range branch), then
            // two, then one: at 10 000 genes and 1024 threads every thread runs 4 + 4 + (2 or 1)
            const double thr = p.threshold;
            int g0 = tid;
            for (; g0 + 3 * NT < G; g0 += 4 * NT) stage_a_group<4, NT>(in, oth, p.lo1, p.hi1, g0, thr, ltab, bad);
            if (g0 + NT < G) {
                stage_a_group<2, NT>(in, oth, p.lo1, p.hi1, g0, thr, ltab, bad);
                g0 += 2 * NT;
            }
            if (g0 < G) stage_a_group<1, NT>(in, oth, p.lo1, p.hi1, g0, thr, ltab, bad);
        } else {
            for (int g = tid; g < G; g += NT) {
                double x = in[g];
                if (!is_finite_d(x)) bad = true;
                if (p.apply_log) x = fast_log2_1p(x, ltab);
                if (p.lo1) x = sub_bounds(x, p.lo1[g], p.hi1[g]);
                else if (p.mid1) x = x - p.mid1[g];
                if (p.threshold > 0.0) x = clamp_sym(x, p.threshold);
                oth[g] = x;
            }
        }
        __syncthreads();   // `in` is free, x' complete in `oth`
        lap(1);

        // ---- B: pyramid smooth oth (x') -> in (smoothed) -------------------------------------------------
        const double *xs = oth + a0;
        double ys1 = 0.0, ys2 = 0.0;   // sum / sum of squares of this thread's outputs (first median pivots)
        if (!do_smooth) {
            for (int q = 0; q < len; ++q) {
                const double out = xs[q];
                if (!PADQ) in[a0 + q] = out;
                ys1 += out;
                ys2 = fma(out, out, ys2);
            }
        } else {
            // pass 1: segment total of x
            double tot = 0.0;
#pragma unroll(FIX ? LFIX : 4)
            for (int q = 0; q < (FIX ? LFIX : len); ++q)
                if (!FIX || q < len) tot += xs[q];
            double inc = tot;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double t = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane - d >= lane_first) inc += t;
            }
            double exc = __shfl_up_sync(0xffffffffu, inc, 1);
            if (lane <= lane_first) exc = 0.0;
            if (lane == 31) tails[warp] = inc;
            __syncthreads();
            double carry = 0.0;
            for (int u = wfirst; u < warp; ++u) carry += tails[u];
            const double offP = exc + carry;   // P just before this segment
            // pass 2: segment total of P (P = prefix of x inside the chromosome)
            double pr = offP, qsum = 0.0;
#pragma unroll(FIX ? LFIX : 4)
            for (int q = 0; q < (FIX ? LFIX : len); ++q)
                if (!FIX || q < len) {
                    pr += xs[q];
                    qsum += pr;
                }
            const double plast = pr;
            inc = qsum;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double t = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane - d >= lane_first) inc += t;
            }
            exc = __shfl_up_sync(0xffffffffu, inc, 1);
            if (lane <= lane_first) exc = 0.0;
            if (lane == 31) tails[NW + warp] = inc;
            __syncthreads();
            carry = 0.0;
            for (int u = wfirst; u < warp; ++u) carry += tails[NW + u];
            const double offQ = exc + carry;   // Q just before this segment
            // pass 3: Q in place (each thread touches only its own slice); PADQ: into the padded layout in `in`, where
            // Q(0) of chromosome c sits at cs + c (2h + 2) + (h + 2)
            const int pbase = cs + seg.chr * (2 * h + 2) + (h + 2);
            double *qdst = PADQ ? (in + pbase + (a0 - cs)) : (oth + a0);   // aliases xs in the ping-pong layout
            pr = offP;
            double qv = offQ;
#pragma unroll(FIX ? LFIX : 4)
            for (int q = 0; q < (FIX ? LFIX : len); ++q)
                if (!FIX || q < len) {
                    pr += xs[q];
                    qv += pr;
                    qdst[q] = qv;
                }
            if (len > 0 && a0 + len == ce) {
                ptot[seg.chr] = plast;
                qtot[seg.chr] = qv;
            }
            __syncthreads();
            // Q continues linearly past a chromosome's last gene (x is taken as 0 there): Q(n-1+k) = Qn + k*Pn, k = 1..h
            if (PADQ) {
                // a warp per chromosome, lanes over its 2h + 2 pad entries (no integer division per entry)
                const int padw = 2 * h + 2;
                for (int c = warp; c < p.K; c += NW) {
                    const int nc = chr_n[c];
                    if (nc >= 2) {
                        const int base = chr_cs[c] + c * padw;
                        const double pt = ptot[c], qt = qtot[c];
                        for (int e = lane; e < padw; e += 32) {
                            if (e < h + 2) in[base + e] = 0.0;
                            else in[base + nc + e] = fma((double)(e - (h + 1)), pt, qt);
                        }
                    }
                }
            } else {
                for (int idx = tid; idx < p.K * h; idx += NT) {
                    const int c = idx / h, k = idx - c * h + 1;
                    rext[idx] = fma((double)k, ptot[c], qtot[c]);
                }
            }
            __syncthreads();
            lap(2);
            // outputs: N(j) = (Q(j+h) - Q(j-1)) - (Q(j-1) - Q(j-h-2)), one code path for interior and edge genes -
            // out-of-range Q come from the pads (PADQ) or, by index selection, from the continuation table / the zero slot
            if (n >= 2 && PADQ) {
                const double *__restrict__ P = in + pbase + (a0 - cs);   // &Q(j0)
                double *__restrict__ O = oth + a0;
                const int j0 = a0 - cs;
                if (pad_fast) {
                    // the reciprocal denominators of the slice are consecutive entries of the padded table (interior
                    // genes: the constant entries in front of index 0), read through a pointer that moves by dI per gene
                    const double *__restrict__ pa = P + h, *__restrict__ pb = P - 1, *__restrict__ pc = P - h - 2;
                    const double *__restrict__ pI = invD + r0I;
#pragma unroll 2   // (fully unrolled with a predicate per gene this loop turns into branches: 22.5 against 18.5 per gene)
                    for (int q = 0; q < len; ++q) {
                        const double qb = pb[q];
                        const double N = (pa[q] - qb) - (qb - pc[q]);
                        const double out = N * *pI;
                        pI += dI;
                        O[q] = out;
                        ys1 += out;
                        ys2 = fma(out, out, ys2);
                    }
                } else {
                    for (int q = 0; q < len; ++q) {
                        const int j = j0 + q;
                        const double qb = P[q - 1];
                        const double N = (P[q + h] - qb) - (qb - P[q - h - 2]);
                        const int rl = max(h - j, 0), rr = max(h - (n - 1 - j), 0);
                        double out;
                        if (rl > 0 && rr > 0) {
                            const double D = (double)(h + 1) * (double)(h + 1) - 0.5 * (double)rl * (double)(rl + 1) -
                                             0.5 * (double)rr * (double)(rr + 1);
                            out = N / D;
                        } else {
                            out = N * invD[rl + rr];
                        }
                        O[q] = out;
                        ys1 += out;
                        ys2 = fma(out, out, ys2);
                    }
                }
            } else if (n >= 2) {
                const int qoff = (int)(oth - sm) + cs;                       // Q(j) lives at sm[qoff + j], 0 <= j < n
                const int roff = (int)(rext - sm) + seg.chr * h - n;         // Q(j) at sm[roff + j], n <= j < n + h
                const int zoff = (int)(zslot - sm);
                const bool short_chr = n < 2 * h + 1;                        // both ends inside one window
                int j = a0 - cs;
#pragma unroll 2
                for (int q = 0; q < len; ++q, ++j) {
                    const int ja = j + h, jb = j - 1, jc = j - h - 2;
                    const double qa = sm[(ja <= n - 1 ? qoff : roff) + ja];
                    const double qb = sm[jb >= 0 ? qoff + jb : zoff];
                    const double qc = sm[jc >= 0 ? qoff + jc : zoff];
                    const double N = (qa - qb) - (qb - qc);
                    const int rl = max(h - j, 0), rr = max(h - (n - 1 - j), 0);
                    double out;
                    if (short_chr && rl > 0 && rr > 0) {
                        const double D = (double)(h + 1) * (double)(h + 1) - 0.5 * (double)rl * (double)(rl + 1) -
                                         0.5 * (double)rr * (double)(rr + 1);
                        out = N / D;
                    } else {
                        out = N * invD[rl + rr];
                    }
                    in[a0 + q] = out;
                    ys1 += out;
                    ys2 = fma(out, out, ys2);
                }
            } else {
                // single-gene chromosome: left untouched (ops.R:2417); Q of a single element is the element, and with
                // PADQ x' itself is still in place in `oth`
                for (int q = 0; q < len; ++q) {
                    const double out = oth[a0 + q];
                    if (!PADQ) in[a0 + q] = out;
                    ys1 += out;
                    ys2 = fma(out, out, ys2);
                }
            }
        }
        ys1 = warp_sum_d(ys1);
        ys2 = warp_sum_d(ys2);
        if (lane == 0) {
            red.d[phase][0][warp] = ys1;
            red.d[phase][1][warp] = ys2;
        }
        __syncthreads();   // smoothed values complete in `in` (PADQ: in `oth`); Q no longer needed
        double *const sv = PADQ ? oth : in;   // the smoothed column stages C and D read
        double S1 = (lane < NW) ? red.d[phase][0][lane] : 0.0, S2 = (lane < NW) ? red.d[phase][1][lane] : 0.0;
        S1 = warp_sum_d(S1);
        S2 = warp_sum_d(S2);
        phase ^= 1;
        lap(3);
        if (tid == 0) {    // next cell's column lands where Q was (`oth`; PADQ: `in`) while the median and the epilogue run
            const int64_t cn = ci + gridDim.x;
            if (cn < p.n_cols) {
                const int64_t coln = p.cols ? (int64_t)p.cols[cn] : cn;
                if (tma_ok(coln)) {
                    fence_proxy_async();
                    mbar_expect_tx(bar, col_bytes);
                    bulk_g2s(PADQ ? in : oth, p.X + p.ldx * coln, col_bytes, bar);
                }
            }
        }

        // ---- C: per-cell centre --------------------------------------------------------------------------------
        double centre = 0.0;
        if (p.center == 1) {
            if (tid == 0) atomicAdd(&g_stats[1], 1ull);
            if (block_median_hist<NT>(sv, G, inv_G, S1, S2, hist, (int)(hdump - hist), hres, wcnt, cand, cand_n, centre)) {
                if (tid == 0) atomicAdd(&g_stats[10], 1ull);
            } else {   // tiny or degenerate columns, > CAND_MAX ties in the middle bin: bracketing selection
                double s1 = 0.0, s2 = 0.0;
                for (int q = 0; q < len; ++q) {
                    const double v = sv[a0 + q];
                    s1 += v;
                    s2 = fma(v, v, s2);
                }
                centre = block_median_smem<NT>(sv, a0, len, G, s1, s2, red, phase, cand, cand_n);
            }
        } else if (p.center == 2) {
            centre = S1 / (double)G;
        }

        lap(4);
        // ---- D: centre, second reference subtraction, 2^x fused into the one coalesced write ----------------
        if (p.lo2 && p.apply_exp2) {
            int g0 = tid;
            for (; g0 + 3 * NT < G; g0 += 4 * NT) stage_d_group<4, NT>(sv, dst, p.lo2, p.hi2, g0, centre, etab);
            if (g0 + NT < G) {
                stage_d_group<2, NT>(sv, dst, p.lo2, p.hi2, g0, centre, etab);
                g0 += 2 * NT;
            }
            if (g0 < G) stage_d_group<1, NT>(sv, dst, p.lo2, p.hi2, g0, centre, etab);
        } else {
            for (int g = tid; g < G; g += NT) {
                double x = sv[g] - centre;
                if (p.lo2) x = sub_bounds(x, p.lo2[g], p.hi2[g]);
                else if (p.mid2) x = x - p.mid2[g];
                if (p.apply_exp2) x = fast_exp2(x, etab);
                dst[g] = x;
            }
        }
        __syncthreads();   // the smoothed column is rewritten by the next cell's stage A
        lap(5);
        if (!PADQ) {       // the next cell landed (or will be loaded) in `oth`
            double *t = in;
            in = oth;
            oth = t;
        }
    }
#ifdef ICNV_STAGE_TIMERS
    if (tid == 0 && blockIdx.x == 0)
        for (int i = 0; i < 6; ++i) atomicAdd(&g_stats[4 + i], tacc[i]);
#endif
    if (bad && p.err_flag) atomicExch(p.err_flag, 1);
}

// =================================================================================================
// K2 v4: ONE shared-memory buffer per cell, so that two cells are in flight on every SM
// =================================================================================================
//
// v3 is bound by the latency of its barrier-separated phases and by shared-memory wavefronts, not by HBM: 512 threads
// per CTA run a cell in almost the time 1024 threads need (measured: 1.21 against 1.14 ms per 9 000 cells x 10 000
// genes), but its two 80 KB buffers allow one CTA per SM.  v4 keeps a single padded copy of the column and runs every
// stage in place, which fits two 512-thread CTAs (two cells) per SM at 10 000 genes; their phases interleave and fill
// each other's bubbles.
//
// Layout: per chromosome c a frame  [slack 0..1][h + 2 front pad][n_c values][h back pad]  (slack makes the value
// region's parity equal the parity of the chromosome's first gene, so every chromosome lands by its own 16-byte
// aligned bulk copy).  Stages:
//   A   x -> x' in place (log2(x+1), dead-band subtraction, clamp); warps walk 32-gene chunks (a descriptor table in
//       shared memory: slot, gene, count), so global reads of the bounds are coalesced and shared-memory accesses
//       conflict free
//   B1  prefix sums P, Q in place over the thread's own slice (three short passes + two segmented warp scans), pads
//   B2  outputs N(j) = (Q(j+h) - Q(j-1)) - (Q(j-1) - Q(j-h-2)) / D(j) written IN PLACE, shifted down by h + 2 slots:
//       slot u is last read by output u + h + 2, which is the output stored there.  Outputs are produced in rounds
//       of V4_R chunks per warp held in registers, one barrier per round; a round's stores only touch slots below
//       every slot a later round reads.
//   C   median over the whole buffer (the slots that hold no value are set to +inf, which the histogram ignores)
//   D   centring, second dead-band subtraction, 2^x, coalesced store of the column
// The next cell's bulk copies are issued when stage D has drained the buffer; the CTA's wait for them is covered by
// the other CTA on the SM.
struct Chr4 {
    int cs;   // first gene of the chromosome
    int n;    // genes
    int fs;   // first slot of the frame
    int vb;   // slot of the first value while x' / Q live in the frame
    int fb;   // slot of the first smoothed value (vb - h - 2; vb when nothing is smoothed)
    int q0;   // index of the chromosome's first 32-gene chunk (entry K: the total)
};

struct Cell4Params {
    const double *X;
    int64_t G, ldx;
    const int32_t *cols;
    int64_t n_cols;
    double *Y;
    int64_t ldy;
    const Seg *segs;
    const Chr4 *chr;    // K + 1 entries (the last one: n = 0, fs = nb, q0 = number of chunks)
    const int4 *chunks; // per 32-gene chunk: x = slot of its first value (x' / Q layout), y = first gene, z = genes in it,
                        // w = chromosome | 0x40000000 when every window of the chunk is a full one
    int apply_log;
    const double *lo1, *hi1, *mid1;
    double threshold;
    int window, h;
    int center;
    const double *lo2, *hi2, *mid2;
    int apply_exp2;
    int *err_flag;
    int K;
    int nb;            // slots of the buffer (even)
    int n_chunks;
};

__device__ __forceinline__ void bulk_g2s_multi(void *dst, const void *src, unsigned bytes, void *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// (a hook for host-side execution models of the copy engine: completes the phase after the issuing thread's copies; the
// GPU's mbarrier completes by transaction bytes and needs nothing here)
__device__ __forceinline__ void mbar_host_commit(void *bar) { (void)bar; }

constexpr int V4_R = 6;   // chunks per warp and output round (registers: 2 per chunk and thread)
constexpr int V4_U = 2;   // chunks per straight-line group of stages A and D (64 registers per thread: 4 spill)

// LFIX > 0: every busy thread's slice has at most LFIX genes: the scan passes are fully unrolled with a predicate per gene.
template <int NT, int MINB, int NB, int LFIX>
__global__ void __launch_bounds__(NT, MINB) cell_pipeline4_kernel(const Cell4Params p) {
    constexpr bool FIX = LFIX > 0;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NW = NT / 32;
    double2 *ltab = reinterpret_cast<double2 *>(smem_raw);
    double *etab = reinterpret_cast<double *>(ltab + 128);
    double *buf = etab + 128;
    double *invD = buf + p.nb;
    double *ptot = invD + (p.h + 2);
    double *qtot = ptot + p.K;
    double *tails = qtot + p.K;                               // [2][NW]
    double *cand = tails + 2 * NW;
    Red<NW> &red = *reinterpret_cast<Red<NW> *>(cand + CAND_MAX + 2);
    unsigned long long *bar = reinterpret_cast<unsigned long long *>(&red + 1);
    // [n_chunks] chunk descriptors, read and written as int4: 16-byte aligned (an odd h leaves `bar` 8 bytes past a 16-byte
    // boundary, the doubles in front of it being nb + h + 2 + 2 K + 2 NW + CAND_MAX + 2 with nb even)
    int4 *ctab = reinterpret_cast<int4 *>(bar + 2 + (p.h & 1));
    int *hist = reinterpret_cast<int *>(ctab + p.n_chunks);   // NB bins, zero between cells
    int *hres = hist + NB;
    int *wcnt = hres + 8;                                     // [2][NW]
    int *cand_n = wcnt + 2 * NW;
    int *hdump = cand_n + 2;                                  // [32] per-lane spare words of the histogram pass
    Chr4 *chr = reinterpret_cast<Chr4 *>(hdump + 32);         // [K + 1]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = (int)p.G, h = p.h, K = p.K, nb = p.nb, NCH = p.n_chunks;
    const bool do_smooth = p.window >= 2;
    const int sh = do_smooth ? h + 2 : 0;   // smoothed values sit this many slots below x' / Q
    const double inv_G = 1.0 / (double)G;
    int phase = 0;
    unsigned parity = 0;
    if (do_smooth) {
        const double full = (double)(h + 1) * (double)(h + 1);
        for (int r = tid; r <= h; r += NT) invD[r] = 1.0 / (full - 0.5 * (double)r * (double)(r + 1));
    }
    if (tid == 0) mbar_init(bar, 1);
    for (int i = tid; i < NB; i += NT) hist[i] = 0;
    for (int i = tid; i < 128; i += NT) {
        ltab[i] = make_double2(g_log_tab[i][0], g_log_tab[i][1]);
        etab[i] = g_exp_tab[i];
    }
    for (int i = tid; i <= K; i += NT) chr[i] = p.chr[i];
    for (int i = tid; i < NCH; i += NT) ctab[i] = p.chunks[i];
    const Seg seg = p.segs[tid];
    const int len = seg.len, a0 = seg.start, cs = seg.cs, ce = seg.ce;
    const int lane_first = max(seg.tfirst - (tid - lane), 0);
    const int wfirst = seg.tfirst >> 5;
    bool bad = false;
    const unsigned col_bytes = (unsigned)(p.G * sizeof(double));
    auto tma_ok = [&](int64_t col) {
        return ((col_bytes & 15u) == 0) && ((reinterpret_cast<uintptr_t>(p.X + p.ldx * col) & 15u) == 0);
    };
    __syncthreads();
    const int my_vb = chr[seg.chr].vb + (a0 - cs);   // slot of this thread's slice while x' / Q live in the frame
    const int my_fb = my_vb - sh;                    // ... of its smoothed values
    const double inv0 = do_smooth ? invD[0] : 1.0;
    // the column of cell `col` -> value slots of the frames: one 16-byte aligned bulk copy per chromosome (the element in
    // front of an odd first gene / behind an odd end lands in a pad slot, which is rewritten before it is read)
    auto issue_column = [&](int64_t col) {
        const double *src = p.X + p.ldx * col;
        unsigned total = 0;
        for (int c = 0; c < K; ++c) {
            const int nc = chr[c].n;
            if (nc > 0) total += (unsigned)((((chr[c].cs + nc + 1) & ~1) - (chr[c].cs & ~1)) * (int)sizeof(double));
        }
        fence_proxy_async();
        mbar_expect_tx(bar, total);
        for (int c = 0; c < K; ++c) {
            const int nc = chr[c].n;
            if (nc > 0) {
                const int e0 = chr[c].cs & ~1, e1 = (chr[c].cs + nc + 1) & ~1;
                bulk_g2s_multi(buf + chr[c].vb - (chr[c].cs & 1), src + e0, (unsigned)((e1 - e0) * (int)sizeof(double)), bar);
            }
        }
        mbar_host_commit(bar);
    };
    if (tid == 0 && (int64_t)blockIdx.x < p.n_cols) {
        const int64_t col0 = p.cols ? (int64_t)p.cols[blockIdx.x] : (int64_t)blockIdx.x;
        if (tma_ok(col0)) issue_column(col0);
    }
    const bool fast_a = p.apply_log && p.lo1 && p.threshold > 0.0;
    const bool fast_d = p.lo2 && p.apply_exp2;
    const int n_it = (NCH - warp + NW - 1) / NW;   // chunks of this warp: warp, warp + NW, ...
    const int n_it_cta = (NCH + NW - 1) / NW;      // ... of warp 0: the most any warp has

    for (int64_t ci = blockIdx.x; ci < p.n_cols; ci += gridDim.x) {
        const int64_t col = p.cols ? (int64_t)p.cols[ci] : ci;
        double *__restrict__ dst = p.Y + p.ldy * ci;
        // ---- the column is in the frames -----------------------------------------------------------------------------
        if (tma_ok(col)) {
            mbar_wait(bar, parity);
            parity ^= 1u;
        } else {
            const double *__restrict__ src = p.X + p.ldx * col;
            for (int it = 0; it < n_it; ++it) {
                const int4 d = ctab[warp + NW * it];
                if (lane < d.z) buf[d.x + lane] = src[d.y + lane];
            }
            __syncthreads();
        }
        // ---- A: x -> x' in place ------------------------------------------------------------------------------------------
        {
            const double thr = p.threshold;
            int it = 0;
            if (fast_a) {
                // V4_U chunks per step as one straight-line block (no range branch per value: the group is re-evaluated
                // through the library path when an argument leaves the fast path's domain)
                for (; it + V4_U <= n_it; it += V4_U) {
                    int4 d[V4_U];
#pragma unroll
                    for (int u = 0; u < V4_U; ++u) d[u] = ctab[warp + NW * (it + u)];
                    double v[V4_U], lo[V4_U], hi[V4_U], x[V4_U];
#pragma unroll
                    for (int u = 0; u < V4_U; ++u) {
                        const bool ok = lane < d[u].z;
                        v[u] = buf[d[u].x + lane];           // slots behind a chromosome's last gene are pad slots
                        lo[u] = ok ? p.lo1[d[u].y + lane] : 0.0;
                        hi[u] = ok ? p.hi1[d[u].y + lane] : 0.0;
                        v[u] = ok ? v[u] : 0.0;
                    }
                    bool slow = false;
#pragma unroll
                    for (int u = 0; u < V4_U; ++u) x[u] = fast_log2_1p_nc(v[u], ltab, slow);
                    if (slow) {
#pragma unroll
                        for (int u = 0; u < V4_U; ++u) {
                            if (!is_finite_d(v[u])) bad = true;
                            x[u] = fast_log2_1p(v[u], ltab);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < V4_U; ++u)
                        if (lane < d[u].z) buf[d[u].x + lane] = clamp_sym(sub_bounds(x[u], lo[u], hi[u]), thr);
                }
            }
            for (; it < n_it; ++it) {
                const int4 d = ctab[warp + NW * it];
                if (lane < d.z) {
                    const int g = d.y + lane;
                    double x = buf[d.x + lane];
                    if (!is_finite_d(x)) bad = true;
                    if (p.apply_log) x = fast_log2_1p(x, ltab);
                    if (p.lo1) x = sub_bounds(x, p.lo1[g], p.hi1[g]);
                    else if (p.mid1) x = x - p.mid1[g];
                    if (thr > 0.0) x = clamp_sym(x, thr);
                    buf[d.x + lane] = x;
                }
            }
        }
        __syncthreads();

        // ---- B: pyramid smooth in place --------------------------------------------------------------------------------------
        double ys1 = 0.0, ys2 = 0.0;   // sum / sum of squares of the outputs (bin geometry of the median)
        if (!do_smooth) {
            const double *xs = buf + my_fb;
            for (int q = 0; q < len; ++q) {
                const double out = xs[q];
                ys1 += out;
                ys2 = fma(out, out, ys2);
            }
        } else {
            double *xs = buf + my_vb;
            // pass 1: slice total of x
            double tot = 0.0;
#pragma unroll(FIX ? LFIX : 4)
            for (int q = 0; q < (FIX ? LFIX : len); ++q)
                if (!FIX || q < len) tot += xs[q];
            double inc = tot;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double t = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane - d >= lane_first) inc += t;
            }
            double exc = __shfl_up_sync(0xffffffffu, inc, 1);
            if (lane <= lane_first) exc = 0.0;
            if (lane == 31) tails[warp] = inc;
            __syncthreads();
            double carry = 0.0;
            for (int u = wfirst; u < warp; ++u) carry += tails[u];
            const double offP = exc + carry;   // P just before this slice
            // pass 2: slice total of P (P = prefix of x inside the chromosome)
            double pr = offP, qsum = 0.0;
#pragma unroll(FIX ? LFIX : 4)
            for (int q = 0; q < (FIX ? LFIX : len); ++q)
                if (!FIX || q < len) {
                    pr += xs[q];
                    qsum += pr;
                }
            const double plast = pr;
            inc = qsum;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double t = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane - d >= lane_first) inc += t;
            }
            exc = __shfl_up_sync(0xffffffffu, inc, 1);
            if (lane <= lane_first) exc = 0.0;
            if (lane == 31) tails[NW + warp] = inc;
            __syncthreads();
            carry = 0.0;
            for (int u = wfirst; u < warp; ++u) carry += tails[NW + u];
            const double offQ = exc + carry;   // Q just before this slice
            // pass 3: Q in place (each thread touches only its own slice)
            pr = offP;
            double qv = offQ;
#pragma unroll(FIX ? LFIX : 4)
            for (int q = 0; q < (FIX ? LFIX : len); ++q)
                if (!FIX || q < len) {
                    pr += xs[q];
                    qv += pr;
                    xs[q] = qv;
                }
            if (len > 0 && a0 + len == ce) {
                ptot[seg.chr] = plast;
                qtot[seg.chr] = qv;
            }
            __syncthreads();
            // pads, a warp per chromosome: h + 2 zeros in front (Q(-1) .. Q(-h-2)), behind the last gene the linear
            // continuation Q(n-1+k) = Qn + k Pn, k = 1..h (x is taken as 0 there)
            for (int c = warp; c < K; c += NW) {
                const int nc = chr[c].n;
                if (nc >= 2) {
                    const int vb = chr[c].vb;
                    const double pt = ptot[c], qt = qtot[c];
                    for (int e = lane; e < 2 * h + 2; e += 32) {
                        if (e < h + 2) buf[vb - 1 - e] = 0.0;
                        else buf[vb + nc + (e - (h + 2))] = fma((double)(e - (h + 1)), pt, qt);
                    }
                }
            }
            __syncthreads();
            // outputs, V4_R chunks per warp and round
            for (int it0 = 0; it0 < n_it_cta; it0 += V4_R) {   // the same number of rounds (barriers) in every warp
                double o[V4_R];
                int wpos[V4_R];
#pragma unroll
                for (int r = 0; r < V4_R; ++r) {
                    wpos[r] = -1;
                    o[r] = 0.0;
                    if (it0 + r < n_it) {
                        const int4 d = ctab[warp + NW * (it0 + r)];
                        const double *__restrict__ P = buf + d.x + lane;
                        if (d.w & 0x40000000) {   // every window of the chunk is a full one (a full chunk, too)
                            const double qb = P[-1];
                            const double N = (P[h] - qb) - (qb - P[-h - 2]);
                            const double out = N * inv0;
                            o[r] = out;
                            wpos[r] = d.x + lane - sh;
                            ys1 += out;
                            ys2 = fma(out, out, ys2);
                        } else if (lane < d.z) {
                            const int c = d.w & 0xffff;
                            const int nc = chr[c].n, j = d.y + lane - chr[c].cs;
                            double out;
                            if (nc >= 2) {
                                const double qb = P[-1];
                                const double N = (P[h] - qb) - (qb - P[-h - 2]);
                                const int rl = max(h - j, 0), rr = max(h - (nc - 1 - j), 0);
                                if (rl > 0 && rr > 0) {   // both ends inside the window (chromosome shorter than it)
                                    const double D = (double)(h + 1) * (double)(h + 1) - 0.5 * (double)rl * (double)(rl + 1) -
                                                     0.5 * (double)rr * (double)(rr + 1);
                                    out = N / D;
                                } else {
                                    out = N * invD[rl + rr];
                                }
                            } else {
                                out = P[0];   // single-gene chromosome: left untouched (ops.R:2417); Q of one element is the element
                            }
                            o[r] = out;
                            wpos[r] = d.x + lane - sh;
                            ys1 += out;
                            ys2 = fma(out, out, ys2);
                        }
                    }
                }
                __syncthreads();   // every read of this round is done; its stores touch no slot a later round reads
#pragma unroll
                for (int r = 0; r < V4_R; ++r)
                    if (wpos[r] >= 0) buf[wpos[r]] = o[r];
            }
        }
        // slots that hold no smoothed value -> +inf (the median pass walks the whole buffer)
        if (p.center == 1) {
            for (int c = warp; c < K; c += NW) {
                const int f0 = chr[c].fs, f1 = chr[c].fb, f2 = chr[c].fb + chr[c].n, f3 = chr[c + 1].fs;
                for (int e = f0 + lane; e < f1; e += 32) buf[e] = INFINITY;
                for (int e = f2 + lane; e < f3; e += 32) buf[e] = INFINITY;
            }
        }
        ys1 = warp_sum_d(ys1);
        ys2 = warp_sum_d(ys2);
        if (lane == 0) {
            red.d[phase][0][warp] = ys1;
            red.d[phase][1][warp] = ys2;
        }
        __syncthreads();   // smoothed values complete at frame start + j
        double S1 = (lane < NW) ? red.d[phase][0][lane] : 0.0, S2 = (lane < NW) ? red.d[phase][1][lane] : 0.0;
        S1 = warp_sum_d(S1);
        S2 = warp_sum_d(S2);
        phase ^= 1;

        // ---- C: per-cell centre --------------------------------------------------------------------------------------------
        double centre = 0.0;
        if (p.center == 1) {
            if (tid == 0) atomicAdd(&g_stats[1], 1ull);
            if (block_median_hist<NT, NB>(buf, G, inv_G, S1, S2, hist, (int)(hdump - hist), hres, wcnt, cand, cand_n, centre, nb)) {
                if (tid == 0) atomicAdd(&g_stats[10], 1ull);
            } else {   // tiny or degenerate columns, > CAND_MAX ties in the middle bin: bracketing selection
                double s1 = 0.0, s2 = 0.0;
                for (int q = 0; q < len; ++q) {
                    const double v = buf[my_fb + q];
                    s1 += v;
                    s2 = fma(v, v, s2);
                }
                centre = block_median_smem<NT>(buf, my_fb, len, G, s1, s2, red, phase, cand, cand_n);
            }
        } else if (p.center == 2) {
            centre = S1 / (double)G;
        }

        // ---- D: centre, second reference subtraction, 2^x fused into the one coalesced write --------------------------------
        {
            int it = 0;
            if (fast_d) {
                for (; it + V4_U <= n_it; it += V4_U) {
                    int4 d[V4_U];
#pragma unroll
                    for (int u = 0; u < V4_U; ++u) d[u] = ctab[warp + NW * (it + u)];
                    double v[V4_U], lo[V4_U], hi[V4_U], x[V4_U];
#pragma unroll
                    for (int u = 0; u < V4_U; ++u) {
                        const bool ok = lane < d[u].z;
                        v[u] = buf[d[u].x + lane - sh];
                        lo[u] = ok ? p.lo2[d[u].y + lane] : 0.0;
                        hi[u] = ok ? p.hi2[d[u].y + lane] : 0.0;
                        v[u] = ok ? v[u] : 0.0;
                    }
                    bool slow = false;
#pragma unroll
                    for (int u = 0; u < V4_U; ++u) {
                        v[u] = sub_bounds(v[u] - centre, lo[u], hi[u]);
                        x[u] = fast_exp2_nc(v[u], etab, slow);
                    }
                    if (slow) {
#pragma unroll
                        for (int u = 0; u < V4_U; ++u) x[u] = fast_exp2(v[u], etab);
                    }
#pragma unroll
                    for (int u = 0; u < V4_U; ++u)
                        if (lane < d[u].z) dst[d[u].y + lane] = x[u];
                }
            }
            for (; it < n_it; ++it) {
                const int4 d = ctab[warp + NW * it];
                if (lane < d.z) {
                    const int g = d.y + lane;
                    double x = buf[d.x + lane - sh] - centre;
                    if (p.lo2) x = sub_bounds(x, p.lo2[g], p.hi2[g]);
                    else if (p.mid2) x = x - p.mid2[g];
                    if (p.apply_exp2) x = fast_exp2(x, etab);
                    dst[g] = x;
                }
            }
        }
        __syncthreads();   // the buffer is free: the next cell's column may land
        if (tid == 0) {
            const int64_t cn = ci + gridDim.x;
            if (cn < p.n_cols) {
                const int64_t coln = p.cols ? (int64_t)p.cols[cn] : cn;
                if (tma_ok(coln)) issue_column(coln);
            }
        }
    }
    if (bad && p.err_flag) atomicExch(p.err_flag, 1);
}

// =================================================================================================
// host-side launchers (device-pointer ABI)
// =================================================================================================

static int build_segments(int64_t G, const int32_t *chr_start, const int32_t *chr_len, int K, int NT, int lmax,
                          std::vector<Seg> &segs) {
    // cover every gene exactly once; genes outside every chromosome range are an argument error
    int64_t covered = 0;
    for (int k = 0; k < K; ++k) {
        if (chr_len[k] < 0 || chr_start[k] < 0 || (int64_t)chr_start[k] + chr_len[k] > G) return -1;
        if (k > 0 && chr_start[k] != chr_start[k - 1] + chr_len[k - 1]) return -1;
        covered += chr_len[k];
    }
    if (K > 0 && chr_start[0] != 0) return -1;
    if (covered != G) return -1;
    // every non-empty chromosome needs a thread of its own, whatever the segment length
    int nonempty = 0;
    for (int k = 0; k < K; ++k) nonempty += chr_len[k] > 0 ? 1 : 0;
    if (nonempty > NT) return 0;
    // L odd: adjacent threads then start an odd number of 8-byte words apart, so the strided
    // 64-bit shared-memory accesses are bank-conflict free within a half-warp.
    for (int L = 1; L < lmax; L += 2) {
        int64_t n = 0;
        for (int k = 0; k < K; ++k) n += (chr_len[k] + L - 1) / L;
        if (n <= NT) {
            segs.resize(NT);
            int t = 0;
            for (int k = 0; k < K; ++k) {
                int pos = chr_start[k], end = chr_start[k] + chr_len[k];
                const int tfirst = t;
                while (pos < end) {
                    int len = end - pos < L ? end - pos : L;
                    segs[t] = Seg{pos, len, chr_start[k], end, tfirst, k};
                    ++t;
                    pos += len;
                }
            }
            for (; t < NT; ++t) segs[t] = Seg{0, 0, 0, 0, t, 0};
            return L;
        }
    }
    return 0;  // does not fit
}

}  // namespace icnv

using namespace icnv;

extern "C" {

int icnv_dev_group_partial_sums_f64(const double *X, int64_t G, int64_t ldx, const int32_t *cells, int64_t n_cells,
                                    int chunk, int apply_log, double *partial, void *stream) {
    ICNV_REQUIRE_READY();
    if (!X || !cells || !partial || G <= 0 || n_cells <= 0 || chunk <= 0)
        return set_error(ICNV_E_BAD_ARG, "icnv_dev_group_partial_sums_f64: bad argument");
    int64_t n_chunks = (n_cells + chunk - 1) / chunk;
    if (n_chunks > 65535) return set_error(ICNV_E_BAD_ARG, "too many chunks (%lld)", (long long)n_chunks);
    dim3 grid((unsigned)((G + 255) / 256), (unsigned)n_chunks);
    if (apply_log == 2)
        group_partial_sums_invlog_kernel<<<grid, 256, 0, pick_stream(stream)>>>(X, G, ldx, cells, n_cells, chunk,
                                                                              partial);
    else
        group_partial_sums_kernel<<<grid, 256, 0, pick_stream(stream)>>>(X, G, ldx, cells, n_cells, chunk, apply_log,
                                                                       partial);
    ICNV_CHECK_LAUNCH("group_partial_sums_kernel");
    return ICNV_OK;
}

int icnv_dev_combine_partials_f64(const double *partial, int64_t G, int64_t n_chunks, int64_t count, double *means,
                                  void *stream) {
    ICNV_REQUIRE_READY();
    if (!partial || !means || G <= 0 || n_chunks <= 0 || count <= 0)
        return set_error(ICNV_E_BAD_ARG, "icnv_dev_combine_partials_f64: bad argument");
    combine_partials_kernel<<<(unsigned)((G + 255) / 256), 256, 0, pick_stream(stream)>>>(partial, G, n_chunks,
                                                                                          (double)count, means);
    ICNV_CHECK_LAUNCH("combine_partials_kernel");
    return ICNV_OK;
}

static int launch_partials(const double *partials, int64_t G, int world, int64_t tot_rows, int n_grp, const int32_t *row_off,
                           const int64_t *counts, double *lo, double *hi, double *mid, double *means, void *stream, const char *who) {
    if (!partials || !row_off || !counts || G <= 0 || world <= 0 || n_grp <= 0 || n_grp > 32 || tot_rows <= 0)
        return set_error(ICNV_E_BAD_ARG, "%s: bad argument (at most 32 groups per call)", who);
    PartialBoundsParams p;
    p.part = partials;
    p.G = G;
    p.tot_rows = tot_rows;
    p.world = world;
    p.n_grp = n_grp;
    for (int k = 0; k <= n_grp; ++k) p.row_off[k] = row_off[k];
    for (int k = 0; k < n_grp; ++k) {
        if (counts[k] <= 0 || row_off[k + 1] < row_off[k] || row_off[k + 1] > tot_rows)
            return set_error(ICNV_E_BAD_ARG, "%s: bad group %d", who, k);
        p.count[k] = (double)counts[k];
    }
    p.lo = lo;
    p.hi = hi;
    p.mid = mid;
    p.means = means;
    bounds_from_partials_kernel<<<(unsigned)((G + 255) / 256), 256, 0, pick_stream(stream)>>>(p);
    ICNV_CHECK_LAUNCH("bounds_from_partials_kernel");
    return ICNV_OK;
}

int icnv_dev_bounds_from_partials_f64(const double *partials, int64_t G, int world, int64_t tot_rows, int n_grp,
                                      const int32_t *row_off, const int64_t *counts, double *lo, double *hi, double *mid,
                                      void *stream) {
    ICNV_REQUIRE_READY();
    if (!lo || !hi) return set_error(ICNV_E_BAD_ARG, "icnv_dev_bounds_from_partials_f64: bad argument");
    return launch_partials(partials, G, world, tot_rows, n_grp, row_off, counts, lo, hi, mid, nullptr, stream,
                           "icnv_dev_bounds_from_partials_f64");
}

int icnv_dev_means_from_partials_f64(const double *partials, int64_t G, int world, int64_t tot_rows, int n_grp,
                                     const int32_t *row_off, const int64_t *counts, double *means, void *stream) {
    ICNV_REQUIRE_READY();
    if (!means) return set_error(ICNV_E_BAD_ARG, "icnv_dev_means_from_partials_f64: bad argument");
    return launch_partials(partials, G, world, tot_rows, n_grp, row_off, counts, nullptr, nullptr, nullptr, means, stream,
                           "icnv_dev_means_from_partials_f64");
}

int icnv_dev_bounds_from_means_f64(const double *means, int64_t G, int n_grp, double *lo, double *hi, double *mid,
                                   void *stream) {
    ICNV_REQUIRE_READY();
    if (!means || !lo || !hi || G <= 0 || n_grp <= 0)
        return set_error(ICNV_E_BAD_ARG, "icnv_dev_bounds_from_means_f64: bad argument");
    bounds_from_means_kernel<<<(unsigned)((G + 255) / 256), 256, 0, pick_stream(stream)>>>(means, G, n_grp, lo, hi, mid);
    ICNV_CHECK_LAUNCH("bounds_from_means_kernel");
    return ICNV_OK;
}

// the compiled kernel the last icnv_dev_cell_pipeline_f64 call launched (host side; read by icnv_debug_cell_launch)
static int g_cell_launch[8];

static void record_cell_launch(int version, int nt, int padq, int lfix, int minb, int seg_len, int64_t grid, int64_t resident) {
    const int v[8] = {version, nt, padq, lfix, minb, seg_len, (int)grid, (int)resident};
    memcpy(g_cell_launch, v, sizeof(v));
}

// test hook, not part of the public header: {version (3 / 4), threads, padded Q, fixed slice length, min CTAs per SM,
// segment length, grid, CTAs the launcher lets run at once (the grid of a launch with enough cells)} of the last
// cell-pipeline launch
ICNV_API int icnv_debug_cell_launch(int *out) {
    if (!out) return set_error(ICNV_E_BAD_ARG, "icnv_debug_cell_launch: bad argument");
    memcpy(out, g_cell_launch, sizeof(g_cell_launch));
    return ICNV_OK;
}

ICNV_API int icnv_debug_stats(unsigned long long *out4, int reset) {
    ICNV_REQUIRE_READY();
    ICNV_CUDA(cudaDeviceSynchronize());
    ICNV_CUDA(cudaMemcpyFromSymbol(out4, g_stats, sizeof(unsigned long long) * 16));
    if (reset) {
        unsigned long long z[16] = {};
        ICNV_CUDA(cudaMemcpyToSymbol(g_stats, z, sizeof(z)));
    }
    return ICNV_OK;
}

int icnv_dev_invlog_finish_f64(double *means, int64_t n, void *stream) {
    ICNV_REQUIRE_READY();
    invlog_finish_kernel<<<(unsigned)((n + 255) / 256), 256, 0, pick_stream(stream)>>>(means, n);
    ICNV_CHECK_LAUNCH("invlog_finish_kernel");
    return ICNV_OK;
}

int icnv_dev_cell_pipeline_f64(const double *X, int64_t G, int64_t ldx, const int32_t *cols, int64_t n_cols, double *Y,
                               int64_t ldy, const int32_t *chr_start, const int32_t *chr_len, int K, int apply_log,
                               const double *lo1, const double *hi1, const double *mid1, double threshold, int window,
                               int center, const double *lo2, const double *hi2, const double *mid2, int apply_exp2,
                               int *err_flag, void *stream) {
    ICNV_REQUIRE_READY();
    Ctx &c = ctx();
    if (!X || !Y || G <= 0 || n_cols < 0 || ldx < G || ldy < G || !chr_start || !chr_len || K <= 0)
        return set_error(ICNV_E_BAD_ARG, "icnv_dev_cell_pipeline_f64: bad argument");
    if ((lo1 == nullptr) != (hi1 == nullptr) || (lo2 == nullptr) != (hi2 == nullptr))
        return set_error(ICNV_E_BAD_ARG, "lo/hi bounds must be given in pairs");
    if (window >= 2 && (window & 1) == 0)
        return set_error(ICNV_E_BAD_ARG, "window_length %d is even: the reference's behaviour is accidental there", window);
    if (center < 0 || center > 2) return set_error(ICNV_E_BAD_ARG, "center must be 0, 1 or 2");
    if (n_cols == 0) return ICNV_OK;
    int h = window >= 2 ? (window - 1) / 2 : 0;
    int s_elems = (int)((G + 1) & ~(int64_t)1);
    std::vector<Seg> segs;
    cudaStream_t st = pick_stream(stream);
    if (!c.math_tables_uploaded) {
        ICNV_CUDA(cudaMemcpyToSymbol(g_log_tab, icnv_log_tab, sizeof(icnv_log_tab)));
        ICNV_CUDA(cudaMemcpyToSymbol(g_exp_tab, icnv_exp_tab, sizeof(icnv_exp_tab)));
        c.math_tables_uploaded = true;
    }
    CellParams p;
    p.X = X; p.G = G; p.ldx = ldx; p.cols = cols; p.n_cols = n_cols; p.Y = Y; p.ldy = ldy;
    p.apply_log = apply_log; p.lo1 = lo1; p.hi1 = hi1; p.mid1 = mid1; p.threshold = threshold;
    p.window = window; p.h = h; p.center = center; p.lo2 = lo2; p.hi2 = hi2; p.mid2 = mid2;
    p.apply_exp2 = apply_exp2; p.err_flag = err_flag; p.s_elems = s_elems; p.K = K;

    // ---- v3 (values stay in shared memory, two ping-pong buffers) whenever both buffers fit -----------------
    if (c.opt_cell_kernel != 4) {
        const int want_v2 = 0;
        int nt3 = (G <= 2048) ? 256 : (G <= 6144 ? 512 : 1024);
        if (ctx().opt_cell_nt) nt3 = ctx().opt_cell_nt;
        if (nt3 != 256 && nt3 != 512 && nt3 != 1024) nt3 = 1024;
        int L3 = want_v2 ? 0 : build_segments(G, chr_start, chr_len, K, nt3, 1 << 20, segs);
        if (L3 < 0) return set_error(ICNV_E_BAD_ARG, "chromosome ranges must tile [0, G) contiguously");
        // more chromosomes than the gene count's thread count: the next larger CTA (one thread per chromosome at least)
        while (L3 == 0 && !ctx().opt_cell_nt && nt3 < 1024) {
            nt3 *= 2;
            L3 = build_segments(G, chr_start, chr_len, K, nt3, 1 << 20, segs);
        }
        const int NW3 = nt3 / 32;
        const size_t red3 = (nt3 == 256) ? sizeof(Red<8>) : (nt3 == 512 ? sizeof(Red<16>) : sizeof(Red<32>));
        // padded-Q layout (see the kernel) whenever it fits; ICNV_CELL_PADQ=0 keeps the ping-pong layout (A/B switch)
        int padq = 1;
        padq = padq && ctx().opt_cell_padq != 0;
        const int q_elems = (int)(((int64_t)G + (int64_t)K * (2 * h + 2) + 1) & ~(int64_t)1);
        const int ipad = (L3 + 2) & ~1;   // front pad of the reciprocal-denominator table: >= the longest slice, even
        auto smem_for = [&](bool pq) {
            const size_t cols = pq ? (size_t)q_elems + (size_t)s_elems + (size_t)ipad
                                   : 2 * (size_t)s_elems + (size_t)K * (size_t)h;
            return 128 * 24 + sizeof(double) * (cols + (size_t)(h + 2) + 2 * (size_t)K + 2 * (size_t)NW3 + CAND_MAX + 2 + 2 + 2) +
                   red3 + sizeof(int) * (HIST_NB + 8 + 2 * (size_t)NW3 + 2 + 2 * (size_t)K + 2 + 32) + 64;
        };
        if (padq && smem_for(true) > (size_t)c.smem_optin) padq = 0;
        const size_t smem3 = smem_for(padq != 0);
        p.q_elems = q_elems;
        p.ipad = ipad;
        if (L3 > 0 && smem3 <= (size_t)c.smem_optin) {
            Seg *d_segs3 = (Seg *)scratch(SLOT_SEGS, sizeof(Seg) * 1024);
            if (!d_segs3) return ICNV_E_NOMEM;
            ICNV_CUDA(upload_if_changed(c.up_segs, c.up_segs_stream, d_segs3, segs.data(), sizeof(Seg) * nt3, st));
            p.segs = d_segs3;
            const int64_t grid3 = std::min<int64_t>(n_cols, c.sm_count);
            auto launch3 = [&](auto kern) -> int {
                ICNV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem3));
                kern<<<(unsigned)grid3, nt3, smem3, st>>>(p);
                return ICNV_OK;
            };
            int rc3;
            // fully unrolled slice loops for the segment length of the 10 000-gene configurations (ICNV_CELL_LFIX=0: generic)
            int lfix = (padq && nt3 == 1024 && L3 == 11) ? 11 : 0;
            if (ctx().opt_cell_lfix == 0) lfix = 0;
            record_cell_launch(3, nt3, padq, lfix, 1, L3, grid3, c.sm_count);
            if (lfix == 11)
                rc3 = launch3(cell_pipeline3_kernel<1024, true, 11>);
            else if (padq)
                rc3 = (nt3 == 256) ? launch3(cell_pipeline3_kernel<256, true, 0>)
                                   : (nt3 == 512 ? launch3(cell_pipeline3_kernel<512, true, 0>) : launch3(cell_pipeline3_kernel<1024, true, 0>));
            else
                rc3 = (nt3 == 256) ? launch3(cell_pipeline3_kernel<256, false, 0>)
                                   : (nt3 == 512 ? launch3(cell_pipeline3_kernel<512, false, 0>) : launch3(cell_pipeline3_kernel<1024, false, 0>));
            if (rc3) return rc3;
            ICNV_CHECK_LAUNCH("cell_pipeline3_kernel");
            return ICNV_OK;
        }
    }

    // ---- v4 (single padded buffer, stages in place): columns too long for v3's two buffers (> ~12 400 genes at window
    // 101; config c5's 20 000 genes run here, one 1024-thread CTA per SM), or everywhere with ICNV_CELL_KERNEL=4 (read at
    // icnv_init): two 512-thread CTAs per SM when a CTA's buffer allows it, four 256-thread CTAs for small columns.
    // Measured at 10 000 genes (profiles/r02_*): v4 with two cells per SM 1.21 ms per 9 000 cells against v3's 1.14 ms -
    // its chunk-descriptor loops cost more instructions than the second cell in flight wins back - so v3 stays the default
    // where it fits; at 20 000 genes v4 runs 62 500 cells in 13.8 ms where the register-resident v2 kernel it replaced
    // took 25.4 ms.
    {
        const int pad = 2 * h + 2;
        std::vector<Chr4> chr((size_t)K + 1);
        int pos = 0, nch = 0;
        for (int k = 0; k < K; ++k) {
            Chr4 &e = chr[(size_t)k];
            e.cs = chr_start[k];
            e.n = chr_len[k];
            e.fs = pos;
            int vb = pos + h + 2;
            if ((vb ^ e.cs) & 1) ++vb;          // value region and first gene of the same parity: 16-byte aligned bulk copies
            e.vb = vb;
            e.fb = window >= 2 ? vb - (h + 2) : vb;
            e.q0 = nch;
            nch += (e.n + 31) / 32;
            pos = vb + e.n + h;
        }
        const int nb = (pos + 2 + 1) & ~1;      // + 2: the element behind an odd chromosome end of the last frame
        chr[(size_t)K] = Chr4{(int)G, 0, nb, nb, nb, nch};
        (void)pad;
        std::vector<int4> chunks((size_t)nch);
        for (int k = 0; k < K; ++k)
            for (int q = 0; q * 32 < chr[(size_t)k].n; ++q) {
                const int j0 = q * 32, cnt = std::min(32, chr[(size_t)k].n - j0), nc = chr[(size_t)k].n;
                const bool full = window >= 2 && cnt == 32 && j0 >= h && j0 + 31 <= nc - 1 - h;
                chunks[(size_t)(chr[(size_t)k].q0 + q)] = make_int4(chr[(size_t)k].vb + j0, chr[(size_t)k].cs + j0, cnt, k | (full ? 0x40000000 : 0));
            }
        auto smem4 = [&](int nt) {
            const int nw = nt / 32;
            const size_t red = (nt == 256) ? sizeof(Red<8>) : (nt == 512 ? sizeof(Red<16>) : sizeof(Red<32>));
            return 128 * 24 + sizeof(double) * ((size_t)nb + (size_t)(h + 2) + 2 * (size_t)K + 2 * (size_t)nw + CAND_MAX + 2) + red + 16 +
                   sizeof(double) * (size_t)(h & 1) +   // alignment of the chunk table (see the kernel)
                   sizeof(int) * (1024 + 8 + 2 * (size_t)nw + 2 + 32) + sizeof(Chr4) * ((size_t)K + 1) + sizeof(int4) * (size_t)nch + 16;
        };
        const size_t sm_total = 228 * 1024;     // shared memory of an SM; every resident CTA also reserves 1 KB
        int nt4 = 0, minb = 1;
        if (c.opt_cell_nt == 256 || c.opt_cell_nt == 512 || c.opt_cell_nt == 1024) {
            nt4 = c.opt_cell_nt;
            minb = std::max(1, std::min(nt4 == 256 ? 4 : (nt4 == 512 ? 2 : 1), (int)(sm_total / (smem4(nt4) + 1024))));
        } else if (4 * (smem4(256) + 1024) <= sm_total && G <= 6144) {
            nt4 = 256;
            minb = 4;
        } else if (2 * (smem4(512) + 1024) <= sm_total) {
            nt4 = 512;
            minb = 2;
        } else {
            nt4 = 1024;
            minb = 1;
        }
        int L4 = build_segments(G, chr_start, chr_len, K, nt4, 1 << 20, segs);
        if (L4 < 0) return set_error(ICNV_E_BAD_ARG, "chromosome ranges must tile [0, G) contiguously");
        // more chromosomes than threads: the next larger CTA, with as many CTAs per SM as its shared memory allows
        while (L4 == 0 && !c.opt_cell_nt && nt4 < 1024) {
            nt4 *= 2;
            minb = std::max(1, std::min(nt4 == 512 ? 2 : 1, (int)(sm_total / (smem4(nt4) + 1024))));
            L4 = build_segments(G, chr_start, chr_len, K, nt4, 1 << 20, segs);
        }
        const size_t smem = smem4(nt4);
        if (L4 > 0 && smem <= (size_t)c.smem_optin) {
            const size_t off_chr = sizeof(Seg) * 1024, off_chunks = (off_chr + sizeof(Chr4) * ((size_t)K + 1) + 15) & ~(size_t)15;
            const size_t tab_bytes = off_chunks + sizeof(int4) * (size_t)nch;
            char *d_tab = (char *)scratch(SLOT_SEGS, tab_bytes);
            if (!d_tab) return ICNV_E_NOMEM;
            std::vector<unsigned char> tab(tab_bytes, 0);
            memcpy(tab.data(), segs.data(), sizeof(Seg) * (size_t)nt4);
            memcpy(tab.data() + off_chr, chr.data(), sizeof(Chr4) * ((size_t)K + 1));
            memcpy(tab.data() + off_chunks, chunks.data(), sizeof(int4) * (size_t)nch);
            ICNV_CUDA(upload_if_changed(c.up_segs, c.up_segs_stream, d_tab, tab.data(), tab.size(), st));
            Cell4Params q;
            q.X = X; q.G = G; q.ldx = ldx; q.cols = cols; q.n_cols = n_cols; q.Y = Y; q.ldy = ldy;
            q.segs = (const Seg *)d_tab;
            q.chr = (const Chr4 *)(d_tab + off_chr);
            q.chunks = (const int4 *)(d_tab + off_chunks);
            q.apply_log = apply_log; q.lo1 = lo1; q.hi1 = hi1; q.mid1 = mid1; q.threshold = threshold;
            q.window = window; q.h = h; q.center = center; q.lo2 = lo2; q.hi2 = hi2; q.mid2 = mid2;
            q.apply_exp2 = apply_exp2; q.err_flag = err_flag; q.K = K; q.nb = nb; q.n_chunks = nch;
            auto launch4 = [&](auto kern, int kminb, int klfix) -> int {
                ICNV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                int per_sm = 1;
                ICNV_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, nt4, smem));
                const int64_t resident = (int64_t)c.sm_count * std::max(per_sm, 1);
                const int64_t grid = std::min<int64_t>(n_cols, resident);
                record_cell_launch(4, nt4, 0, klfix, kminb, L4, grid, resident);
                kern<<<(unsigned)grid, nt4, smem, st>>>(q);
                return ICNV_OK;
            };
            int rc4;
            // the slice length of the 10 000-gene / 20 000-gene layouts (21 genes per thread) gets fully unrolled scan passes
            const bool fix21 = L4 == 21 && c.opt_cell_lfix != 0;
            if (nt4 == 256) rc4 = (minb >= 4) ? launch4(cell_pipeline4_kernel<256, 4, 1024, 0>, 4, 0) : launch4(cell_pipeline4_kernel<256, 1, 1024, 0>, 1, 0);
            else if (nt4 == 512 && minb >= 2) rc4 = fix21 ? launch4(cell_pipeline4_kernel<512, 2, 1024, 21>, 2, 21) : launch4(cell_pipeline4_kernel<512, 2, 1024, 0>, 2, 0);
            else if (nt4 == 512) rc4 = launch4(cell_pipeline4_kernel<512, 1, 1024, 0>, 1, 0);
            else rc4 = fix21 ? launch4(cell_pipeline4_kernel<1024, 1, 1024, 21>, 1, 21) : launch4(cell_pipeline4_kernel<1024, 1, 1024, 0>, 1, 0);
            if (rc4) return rc4;
            ICNV_CHECK_LAUNCH("cell_pipeline4_kernel");
            return ICNV_OK;
        }
        if (!(L4 > 0)) {
            int nonempty = 0;
            for (int k = 0; k < K; ++k) nonempty += chr_len[k] > 0 ? 1 : 0;
            return set_error(ICNV_E_UNSUPPORTED, "%d non-empty chromosomes need a thread each, more than the %d threads of a CTA",
                             nonempty, nt4);
        }
        return set_error(ICNV_E_UNSUPPORTED, "G = %lld genes in %d chromosomes, window %d: a cell's padded column needs %lld B of "
                         "shared memory, more than the %d B a CTA can have", (long long)G, K, window, (long long)smem, c.smem_optin);
    }
}

}  // extern "C"
