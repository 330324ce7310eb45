// K12: Pareto-smoothed importance-sampling leave-one-out (PSIS-LOO) and WAIC of a run over its per-bin births and deaths, on the
// device, without copying the records.  literate_b200.loo.loo_host is the definition, step for step.
//
// The observation is the count A of side s in bin j (the unit K11 checks): given a record, every sampler here models it as
// Poisson(rate_sj B_sj) with the exposure B at its observed value, so the pointwise log-likelihood of column (s, j) with B > 0 is
//   l_sj = A log(r B) - r B - lgamma(A + 1)          (A log(r B) = 0 for A = 0)
// Rows, ladders and the rates of bin j are those of K11 (lr_chain_row; lr_k3_stage / lr_k3_slot for K3 records).  A record is used
// under K11's rule and when every l_sj of it is finite; the S used records of all chains are pooled.
//
// Work, per batch of columns:
//   1. (once) a scan pass (one warp per record) marks the used records, and one CTA numbers them (pos = their index among the used).
//   2. pointwise: one warp per record, lane = column of the batch: l into L [records][batch] (NaN for an unused record) and the
//      order-preserving key of v = -l (-0 as +0) to the column's segment at the record's number.
//   3. K10's segmented radix sort (lr_k10_sort) of the segments: max, cutoff and the tail of v come out exactly, ties included.
//   4. L becomes exp(l - max l) in place, and lr_k9_run gives its "mean" ESS over the chains (NaN for a column with an unused
//      record or a constant one): r_eff = ESS / S, or 1 when the ESS is NaN.
//   5. tail: one CTA per column, from the sorted keys alone -- lppd and WAIC, the cutoff and the tail, whose exceedances y go to
//      the key buffer the sort left free; grid: the grid points of Zhang and Stephens' GPD fit, a warp each and several CTAs per
//      column, lanes over y; fit: one CTA per column, the fit's weights, k_hat, the smoothed tail and the two log-sum-exps.  The
//      smoothed weights pair with the sorted draws, so no draw needs its unsorted place.
// Every sum is compensated and done in a fixed order (lanes strided, butterflies, then the warps in order): repeated calls are
// bit-identical.
#include <math_constants.h>
#include <algorithm>
#include <cmath>
#include <vector>
#include "lr_common.cuh"

namespace {

constexpr int K12_RB = 256;             // threads of the record kernels
constexpr int K12_FT = 256;             // threads of the fit kernel
constexpr int K12_FW = K12_FT / 32;
constexpr int K12_QL = 4;               // batch columns per lane of the pointwise kernel
constexpr int K12_MAX_BATCH = 32 * K12_QL;
constexpr size_t K12_BUDGET = (size_t)1 << 30;   // K12's own batch scratch (a batch holds at least one column)
constexpr double K12_LOG_TINY = -708.3964185322641;    // log(DBL_MIN), as numpy rounds it
constexpr double K12_EPS = 2.220446049250313e-16;      // DBL_EPSILON

// the tail of one batch column (k12_tail_kernel), read by the grid and fit kernels
struct K12Col {
    double lppd, p_waic, reff, vmax, ec;
    long long i0, T;                // first tail place, tail length
    int m;                          // grid points of the GPD fit (0: T <= 4, no fit)
    int used;                       // 0: fewer than 2 records used
};

struct K12Args {
    lr_chain_rows src;
    int layout, rate_col, nb, s0f;
    const double* terms;            // [4][nb]: A^b, B^b, A^d, B^d
    long long R;                    // S M logical records
    const int* col;                 // [n_act] side nb + j of the columns with B > 0
    const double* lg;               // [n_act] lgamma(A + 1) of each
    int n_act;
    unsigned char* flag;            // [R] 0 used, 1 skipped, 2 no member at beta = 1
    long long* pos;                 // [R] number of a used record among the used ones
    long long* n_used;              // [1]
    unsigned long long* status;     // [2] the caller's
    // the batch
    int c0, bc;                     // its first active column, its columns
    long long n;                    // used records (segment length)
    double* L;                      // [R][bc] l, then exp(l - max l)
    unsigned long long* key[2];     // [bc][n] keys of v = -l, ping-pong
    unsigned long long* band;       // [bc] AND / OR of the keys of a column
    unsigned long long* bor;
    double* r9;                     // [5][bc] K9 on exp(l - max l)
    double* gp;                     // [bc][3][mcap] b_i, k_i then w_i, L_i of the GPD fit
    long long mcap;
    K12Col* cs;                     // [bc]
    double* out;                    // [9][2][nb]
};

__device__ __forceinline__ void k12_column(const K12Args& p, int a, int* side, int* j) {
    const int sj = p.col[a];
    *side = sj >= p.nb;
    *j = sj - *side * p.nb;
}

__device__ __forceinline__ double k12_rate(const K12Args& p, const double* row, int side, int j, const int* sjb, int K) {
    return p.layout == 0 ? row[(side ? 80 : 16) + lr_k3_slot(sjb, K, j)] : row[p.rate_col + side * p.nb + j];
}

// the Poisson log pmf of A at mu
__device__ __forceinline__ double k12_ll(double A, double mu, double lg) {
    const double a = A == 0.0 ? 0.0 : __dmul_rn(A, log(mu));
    return __dsub_rn(__dsub_rn(a, mu), lg);
}

// compensated butterfly over the warp: every lane ends with the same value
__device__ __forceinline__ double k12_warp_sum(double v) {
    double s = v, c = 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double so = __shfl_xor_sync(0xffffffffu, s, o), co = __shfl_xor_sync(0xffffffffu, c, o);
        const double t = __dadd_rn(s, so), bv = __dsub_rn(t, s);
        const double e = __dadd_rn(__dsub_rn(s, __dsub_rn(t, bv)), __dsub_rn(so, bv));
        c = __dadd_rn(__dadd_rn(c, co), e);
        s = t;
    }
    return isfinite(s) ? __dadd_rn(s, c) : s;
}
// the larger of two values, NaN if either is NaN (numpy's max)
__device__ __forceinline__ double k12_max(double a, double b) { return (a != a || b != b) ? CUDART_NAN : fmax(a, b); }

// block-wide sum of every thread's v (warps by butterfly, then the warps in order); every thread gets it
__device__ __forceinline__ double k12_block_sum(double v, double* sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = k12_warp_sum(v);
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        lr_sum a;
        for (int w = 0; w < K12_FW; ++w) a.add(sh[w]);
        sh[K12_FW] = a.value();
    }
    __syncthreads();
    const double r = sh[K12_FW];
    __syncthreads();
    return r;
}
__device__ __forceinline__ double k12_block_max(double v, double* sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = k12_max(v, __shfl_xor_sync(0xffffffffu, v, o));
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double m = sh[0];
        for (int w = 1; w < K12_FW; ++w) m = k12_max(m, sh[w]);
        sh[K12_FW] = m;
    }
    __syncthreads();
    const double r = sh[K12_FW];
    __syncthreads();
    return r;
}

// one warp per logical record: K11's rule, and every l finite
__global__ void __launch_bounds__(K12_RB) k12_scan_kernel(const K12Args p) {
    __shared__ int sjb[K12_RB / 32][2][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long r = (long long)blockIdx.x * (K12_RB / 32) + warp;
    if (r >= p.R) return;
    const long long s = r / p.src.M, c = r - s * p.src.M;
    bool missing = false;
    const double* row = lr_chain_row(p.src, s, c, lane, &missing);
    unsigned char f = 0;
    if (missing) {
        f = 2;
    } else {
        int K[2] = {0, 0};
        if (p.layout == 0) {
            K[0] = lr_k3_stage(p.s0f, p.nb, row, 0, lane, sjb[warp][0]);
            K[1] = lr_k3_stage(p.s0f, p.nb, row, 1, lane, sjb[warp][1]);
        }
        bool ok = (p.layout != 0 || (K[0] > 0 && K[1] > 0)) && row[0] >= 0.0 && row[0] < 9.2e18;
        if (ok) {
            for (int a = lane; a < p.n_act; a += 32) {
                int side, j;
                k12_column(p, a, &side, &j);
                const double B = p.terms[(2 * side + 1) * p.nb + j];
                const double mu = __dmul_rn(k12_rate(p, row, side, j, sjb[warp][side], K[side]), B);
                ok &= mu >= 0.0 && mu <= LR_POIS_MU_MAX && isfinite(k12_ll(p.terms[2 * side * p.nb + j], mu, p.lg[a]));
            }
        }
        f = __all_sync(0xffffffffu, ok) ? 0 : 1;
    }
    if (lane == 0) {
        p.flag[r] = f;
        if (f) atomicAdd(p.status + (f == 1 ? 0 : 1), 1ull);
    }
}

// one CTA: pos = exclusive prefix count of the used records (contiguous ranges per thread, in order), n_used
__global__ void __launch_bounds__(1024) k12_number_kernel(const K12Args p) {
    __shared__ long long ws[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long per = (p.R + 1023) / 1024, r0 = min(p.R, (long long)tid * per), r1 = min(p.R, r0 + per);
    long long cnt = 0;
    for (long long r = r0; r < r1; ++r) cnt += p.flag[r] == 0;
    long long x = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) ws[warp] = x;
    __syncthreads();
    if (warp == 0) {
        long long w = ws[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += y; }
        ws[lane] = w;
    }
    __syncthreads();
    long long run = x - cnt + (warp ? ws[warp - 1] : 0);
    for (long long r = r0; r < r1; ++r) { p.pos[r] = run; run += p.flag[r] == 0; }
    if (tid == 1023) *p.n_used = run;
}

__global__ void k12_init_kernel(const K12Args p) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < p.bc) { p.band[q] = ~0ull; p.bor[q] = 0ull; }
}

// warps over records (grid-stride), lane = columns lane, lane + 32, ... of the batch
__global__ void __launch_bounds__(K12_RB) k12_point_kernel(const K12Args p) {
    __shared__ int sjb[K12_RB / 32][2][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int side[K12_QL], jj[K12_QL];
    double A[K12_QL], B[K12_QL], lg[K12_QL];
    unsigned long long kand[K12_QL], kor[K12_QL];
#pragma unroll
    for (int u = 0; u < K12_QL; ++u) {
        const int q = lane + 32 * u;
        side[u] = 0; jj[u] = 0; A[u] = 0.0; B[u] = 0.0; lg[u] = 0.0;
        kand[u] = ~0ull; kor[u] = 0ull;
        if (q < p.bc) {
            k12_column(p, p.c0 + q, &side[u], &jj[u]);
            A[u] = p.terms[2 * side[u] * p.nb + jj[u]];
            B[u] = p.terms[(2 * side[u] + 1) * p.nb + jj[u]];
            lg[u] = p.lg[p.c0 + q];
        }
    }
    const long long step = (long long)gridDim.x * (K12_RB / 32);
    for (long long r = (long long)blockIdx.x * (K12_RB / 32) + warp; r < p.R; r += step) {
        const bool used = p.flag[r] == 0;                          // warp-uniform
        const long long s = r / p.src.M, c = r - s * p.src.M;
        const double* row = lr_chain_row(p.src, s, c, lane, nullptr);
        int K[2] = {0, 0};
        if (used && p.layout == 0) {
            K[0] = lr_k3_stage(p.s0f, p.nb, row, 0, lane, sjb[warp][0]);
            K[1] = lr_k3_stage(p.s0f, p.nb, row, 1, lane, sjb[warp][1]);
        }
        const long long at = used ? p.pos[r] : 0;
#pragma unroll
        for (int u = 0; u < K12_QL; ++u) {
            const int q = lane + 32 * u;
            if (q >= p.bc) continue;
            double l = CUDART_NAN;
            if (used) {
                l = k12_ll(A[u], __dmul_rn(k12_rate(p, row, side[u], jj[u], sjb[warp][side[u]], K[side[u]]), B[u]), lg[u]);
                const double v = -l;
                const unsigned long long k = lr_key(v == 0.0 ? 0.0 : v);
                p.key[0][(size_t)q * p.n + at] = k;
                kand[u] &= k; kor[u] |= k;
            }
            p.L[(size_t)r * p.bc + q] = l;
        }
    }
#pragma unroll
    for (int u = 0; u < K12_QL; ++u) {
        const int q = lane + 32 * u;
        if (q < p.bc && kand[u] != ~0ull) atomicAnd(p.band + q, kand[u]);
        if (q < p.bc && kor[u]) atomicOr(p.bor + q, kor[u]);
    }
}

// the sorted keys of batch column q
__device__ __forceinline__ const unsigned long long* k12_sorted(const K12Args& p, int q) {
    return p.key[lr_radix_src(lr_radix_passes(p.band[q], p.bor[q]), 8)] + (size_t)q * p.n;
}

// L = exp(l - max l) in place (NaN stays NaN)
__global__ void k12_exp_kernel(const K12Args p) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.R * p.bc) return;
    const int q = (int)(i % p.bc);
    const double lmax = -lr_val(k12_sorted(p, q)[0]);
    p.L[i] = exp(__dsub_rn(p.L[i], lmax));
}

// the smoothed tail value of 0-based tail place t: log(sigma expm1(-k log1p(-p)) / k + exp(cutoff)), truncated at 0
__device__ __forceinline__ double k12_smooth(long long t, long long T, double kh, double sigma, double ec) {
    if (!(sigma > 0.0)) return CUDART_NAN;
    const double pr = __ddiv_rn(__dadd_rn((double)t, 0.5), (double)T);
    const double g = fabs(kh) < K12_EPS ? -log1p(-pr) : __ddiv_rn(expm1(__dmul_rn(-kh, log1p(-pr))), kh);
    const double x = log(__dadd_rn(__dmul_rn(g, sigma), ec));
    return x > 0.0 ? 0.0 : x;
}

// the sorted keys' other buffer of batch column q, free once the sort is done: the tail's exceedances y
__device__ __forceinline__ double* k12_ybuf(const K12Args& p, int q) {
    return (double*)(p.key[1 - lr_radix_src(lr_radix_passes(p.band[q], p.bor[q]), 8)] + (size_t)q * p.n);
}

// one CTA per batch column: lppd, p_waic, r_eff, the cutoff and the tail, and y_t = exp(x_{i0 + t}) - exp(cutoff) (ascending)
__global__ void __launch_bounds__(K12_FT) k12_tail_kernel(const K12Args p) {
    __shared__ double sh[K12_FW + 1];
    const int q = blockIdx.x, tid = threadIdx.x;
    K12Col c;
    memset(&c, 0, sizeof(c));
    const long long n = p.n;
    if (n < 2) {
        if (tid == 0) p.cs[q] = c;
        return;
    }
    const unsigned long long* ks = k12_sorted(p, q);
    const double vmin = lr_val(ks[0]), vmax = lr_val(ks[n - 1]);
    const double lmax = -vmin;
    const double dn = (double)n;
    // lppd and WAIC: l = -v
    lr_sum se, sl;
    for (long long i = tid; i < n; i += K12_FT) {
        const double l = -lr_val(ks[i]);
        se.add(exp(__dsub_rn(l, lmax)));
        sl.add(l);
    }
    const double sum_e = k12_block_sum(se.value(), sh);
    const double mean = __ddiv_rn(k12_block_sum(sl.value(), sh), dn);
    lr_sum sv;
    for (long long i = tid; i < n; i += K12_FT) {
        const double d = __dsub_rn(-lr_val(ks[i]), mean);
        sv.add(__dmul_rn(d, d));
    }
    c.p_waic = __ddiv_rn(k12_block_sum(sv.value(), sh), dn - 1.0);
    c.lppd = __dsub_rn(__dadd_rn(log(sum_e), lmax), log(dn));
    // r_eff, tail length, cutoff
    const double ess = p.r9[3 * p.bc + q];
    c.reff = ess != ess ? 1.0 : __ddiv_rn(ess, dn);
    const long long Mt = (long long)ceil(fmin(__dmul_rn(0.2, dn), __dmul_rn(3.0, sqrt(__ddiv_rn(dn, c.reff)))));
    const long long ci = n - Mt - 1;
    const double cutoff = fmax(__dsub_rn(lr_val(ks[ci < 0 ? 0 : ci]), vmax), K12_LOG_TINY);
    long long lo = 0, hi = n;                                        // first place with x > cutoff
    while (lo < hi) {
        const long long m = (lo + hi) >> 1;
        if (__dsub_rn(lr_val(ks[m]), vmax) > cutoff) hi = m; else lo = m + 1;
    }
    c.i0 = lo; c.T = n - lo;
    c.vmax = vmax;
    c.ec = exp(cutoff);
    c.used = 1;
    c.m = c.T > 4 ? 30 + (int)floor(sqrt((double)c.T)) : 0;
    if (c.m) {
        double* y = k12_ybuf(p, q);
        for (long long t = tid; t < c.T; t += K12_FT) y[t] = __dsub_rn(exp(__dsub_rn(lr_val(ks[c.i0 + t]), vmax)), c.ec);
    }
    if (tid == 0) p.cs[q] = c;
}

// grid (block of K12_FW grid points, batch column): warp w takes grid point i of Zhang and Stephens' fit, lanes over the tail
__global__ void __launch_bounds__(K12_FT) k12_grid_kernel(const K12Args p) {
    const int q = blockIdx.y, lane = threadIdx.x & 31;
    const int i = blockIdx.x * K12_FW + (threadIdx.x >> 5);
    const K12Col& c = p.cs[q];
    const int m = c.m;
    if (i >= m) return;
    const long long T = c.T;
    const double* y = k12_ybuf(p, q);
    const double yq = y[(long long)(__dadd_rn(__ddiv_rn((double)T, 4.0), 0.5)) - 1], ylast = y[T - 1];
    const double dT = (double)T;
    double b = __dsub_rn(1.0, sqrt(__ddiv_rn((double)m, __dsub_rn((double)(i + 1), 0.5))));
    b = __ddiv_rn(b, __dmul_rn(3.0, yq));
    b = __dadd_rn(b, __ddiv_rn(1.0, ylast));
    lr_sum s;
    for (long long t = lane; t < T; t += 32) s.add(log1p(__dmul_rn(-b, y[t])));
    const double k = __ddiv_rn(k12_warp_sum(s.value()), dT);
    if (lane == 0) {
        double* gb = p.gp + (size_t)q * 3 * p.mcap;
        gb[i] = b; gb[p.mcap + i] = k;
        gb[2 * p.mcap + i] = __dmul_rn(dT, __dsub_rn(__dsub_rn(log(-__ddiv_rn(b, k)), k), 1.0));
    }
}

// one CTA per batch column: the fit's weights, k_hat and sigma, the smoothed log weights, elpd_loo and the outputs
__global__ void __launch_bounds__(K12_FT) k12_fit_kernel(const K12Args p) {
    __shared__ double sh[K12_FW + 1];
    __shared__ double sfit[1];
    const int q = blockIdx.x, tid = threadIdx.x;
    int side, j;
    k12_column(p, p.c0 + q, &side, &j);
    const size_t ob = (size_t)2 * p.nb, oj = (size_t)side * p.nb + j;
    double* o = p.out + oj;
    const K12Col c = p.cs[q];
    if (tid == 0) o[0] = p.terms[2 * side * p.nb + j];
    if (!c.used) {
        if (tid == 0) for (int f = 1; f < 9; ++f) o[f * ob] = CUDART_NAN;
        return;
    }
    const long long n = p.n, i0 = c.i0, T = c.T;
    const unsigned long long* ks = k12_sorted(p, q);
    const double vmax = c.vmax, ec = c.ec;
    double kh = CUDART_INF, sigma = 0.0;
    if (c.m) {
        const int m = c.m;
        const double* y = k12_ybuf(p, q);
        double* gb = p.gp + (size_t)q * 3 * p.mcap;
        double* gk = gb + p.mcap;
        const double* gl = gk + p.mcap;
        for (int i = tid; i < m; i += K12_FT) {
            lr_sum s;
            for (int l = 0; l < m; ++l) s.add(exp(__dsub_rn(gl[l], gl[i])));
            gk[i] = __ddiv_rn(1.0, s.value());                    // k_i is no longer needed: w_i takes its place
        }
        __syncthreads();
        if (tid == 0) {
            lr_sum ws;
            for (int i = 0; i < m; ++i) if (gk[i] >= 10.0 * K12_EPS) ws.add(gk[i]);
            const double wt = ws.value();
            lr_sum bs;
            for (int i = 0; i < m; ++i) if (gk[i] >= 10.0 * K12_EPS) bs.add(__dmul_rn(gb[i], __ddiv_rn(gk[i], wt)));
            sfit[0] = bs.value();
        }
        __syncthreads();
        const double bh = sfit[0];
        const double dT = (double)T;
        lr_sum s;
        for (long long t = tid; t < T; t += K12_FT) s.add(log1p(__dmul_rn(-bh, y[t])));
        const double k = __ddiv_rn(k12_block_sum(s.value(), sh), dT);
        sigma = __ddiv_rn(-k, bh);
        kh = __ddiv_rn(__dadd_rn(__dmul_rn(dT, k), 5.0), __dadd_rn(dT, 10.0));
    }
    const bool smooth = isfinite(kh);
    // the log weights x~ (x below the tail, the smoothed tail when k is finite) and their log-sum-exp
    auto xs = [=](long long i) {
        return (smooth && i >= i0) ? k12_smooth(i - i0, T, kh, sigma, ec) : __dsub_rn(lr_val(ks[i]), vmax);
    };
    double mx = -CUDART_INF;
    for (long long i = tid; i < n; i += K12_FT) mx = k12_max(mx, xs(i));
    mx = k12_block_max(mx, sh);
    lr_sum sx;
    for (long long i = tid; i < n; i += K12_FT) sx.add(exp(__dsub_rn(xs(i), mx)));
    const double lse = __dadd_rn(log(k12_block_sum(sx.value(), sh)), mx);
    // elpd_loo = logsumexp(l + lw), lw = x~ - lse
    auto val = [=](long long i) { return __dadd_rn(-lr_val(ks[i]), __dsub_rn(xs(i), lse)); };
    double mv = -CUDART_INF;
    for (long long i = tid; i < n; i += K12_FT) mv = k12_max(mv, val(i));
    mv = k12_block_max(mv, sh);
    lr_sum sz;
    for (long long i = tid; i < n; i += K12_FT) sz.add(exp(__dsub_rn(val(i), mv)));
    const double elpd = __dadd_rn(log(k12_block_sum(sz.value(), sh)), mv);
    if (tid == 0) {
        o[1 * ob] = c.lppd;
        o[2 * ob] = elpd;
        o[3 * ob] = __dsub_rn(c.lppd, elpd);
        o[4 * ob] = __dsub_rn(c.lppd, c.p_waic);
        o[5 * ob] = c.p_waic;
        o[6 * ob] = kh;
        o[7 * ob] = c.reff;
        o[8 * ob] = (double)T;
    }
}

__global__ void k12_fill_kernel(double* out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = CUDART_NAN;
}

// the workspace: per call the flags, numbers, columns; per batch of bc columns L, the keys, the sort's counts, K9's outputs and
// status, the GPD grid, then K9's scratch.  Placed from `base` (null: only measured); returns its bytes.
struct K12Ws { int* col; double* lg; int64_t* k9status; unsigned* ghist; char* k9; };

size_t k12_layout(char* base, K12Args* p, K12Ws* w9, long long R, int n_act, int bc, long long M) {
    lr_carve w{base};
    p->flag = w.take<unsigned char>(R);
    p->pos = w.take<long long>(R);
    p->n_used = w.take<long long>(1);
    w9->col = w.take<int>(n_act);
    w9->lg = w.take<double>(n_act);
    p->L = w.take<double>((size_t)R * bc);
    p->key[0] = w.take<unsigned long long>((size_t)R * bc);
    p->key[1] = w.take<unsigned long long>((size_t)R * bc);
    w9->ghist = w.take<unsigned>(lr_k10_sort_ghist(R) * bc);
    p->band = w.take<unsigned long long>(bc);
    p->bor = w.take<unsigned long long>(bc);
    p->r9 = w.take<double>((size_t)5 * bc);
    w9->k9status = w.take<int64_t>(1);
    p->gp = w.take<double>((size_t)3 * p->mcap * bc);
    p->cs = w.take<K12Col>(bc);
    w9->k9 = w.take<char>(lr_k9_scratch_bytes(M, bc));
    return w.used;
}

}  // namespace

extern "C" int lr_loo(lr_handle_t h, const double* d_rows, int64_t n_samples, int64_t n_chains, int32_t ladder, int32_t beta_col,
                      int64_t row_stride, int32_t layout, int32_t rate_col, double start_time, int32_t n_bins, const double* d_terms,
                      double* d_out, int64_t* d_n, int64_t* d_status, void* stream) {
    const char* who = "lr_loo";
    const int32_t col0 = 0;
    int rc = lr_check_chain_rows(who, h, d_terms && d_out && d_n && d_status, d_rows, n_samples, n_chains, ladder, beta_col, row_stride,
                                 1, &col0, nullptr, nullptr);
    if (rc != LR_OK) return rc;
    LR_REQUIRE(n_bins >= 1 && n_bins <= (1 << 30), "%s: n_bins must be 1 .. 2^30", who);
    LR_REQUIRE(layout == 0 || layout == 1, "%s: layout must be 0 (RJMCMC records) or 1 (dense per-bin rates)", who);
    if (layout == 0) {
        LR_REQUIRE(row_stride >= LR_REC_DOUBLES, "%s: RJMCMC records hold %d doubles; the row holds %lld", who, LR_REC_DOUBLES,
                   (long long)row_stride);
        LR_REQUIRE(start_time >= 0.0 && start_time < 2147483647.0, "%s: start_time must be in [0, 2^31)", who);
    } else {
        LR_REQUIRE(rate_col >= 1 && (int64_t)rate_col + 2 * (int64_t)n_bins <= row_stride,
                   "%s: the rates [rate_col, rate_col + 2 n_bins) = [%d, %lld) lie outside the row of %lld doubles", who, rate_col,
                   (long long)rate_col + 2 * n_bins, (long long)row_stride);
    }
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;

    // the columns with B > 0 and lgamma(A + 1) of each
    std::vector<double> ht((size_t)4 * n_bins);
    LR_CUDA(cudaMemcpyAsync(ht.data(), d_terms, ht.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    LR_CUDA(cudaStreamSynchronize(st));
    std::vector<int> hcol;
    std::vector<double> hlg;
    for (int side = 0; side < 2; ++side)
        for (int j = 0; j < n_bins; ++j)
            if (ht[(size_t)(2 * side + 1) * n_bins + j] > 0.0) {
                hcol.push_back(side * n_bins + j);
                hlg.push_back(std::lgamma(ht[(size_t)2 * side * n_bins + j] + 1.0));
            }
    const int n_act = (int)hcol.size();

    K12Args p;
    memset(&p, 0, sizeof(p));
    p.src = {d_rows, n_samples, n_chains, row_stride, ladder, beta_col};
    p.layout = layout; p.rate_col = rate_col; p.nb = n_bins; p.s0f = (int)floor(start_time);
    p.terms = d_terms; p.R = n_samples * n_chains; p.n_act = n_act;
    p.status = (unsigned long long*)d_status;
    p.out = d_out;
    p.mcap = 32 + (long long)std::sqrt(0.2 * (double)p.R);
    const size_t per_col = (size_t)p.R * 24 + lr_k10_sort_ghist(p.R) * 4 + (size_t)p.mcap * 24 + 64;
    const int bc = (int)std::max<size_t>(1, std::min<size_t>({(size_t)std::max(n_act, 1), (size_t)K12_MAX_BATCH, K12_BUDGET / per_col}));
    K12Ws w9;
    rc = lr_ws_acquire(h, k12_layout(nullptr, &p, &w9, p.R, std::max(n_act, 1), bc, n_chains), st);
    if (rc != LR_OK) return rc;
    k12_layout((char*)h->ws, &p, &w9, p.R, std::max(n_act, 1), bc, n_chains);
    p.col = w9.col; p.lg = w9.lg;
    if (n_act) {
        LR_CUDA(cudaMemcpyAsync(w9.col, hcol.data(), n_act * sizeof(int), cudaMemcpyHostToDevice, st));
        LR_CUDA(cudaMemcpyAsync(w9.lg, hlg.data(), n_act * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    LR_CUDA(cudaMemsetAsync(d_status, 0, 2 * sizeof(int64_t), st));
    const long long n_out = 9LL * 2 * n_bins;
    k12_fill_kernel<<<(unsigned)((n_out + 255) / 256), 256, 0, st>>>(d_out, n_out);
    k12_scan_kernel<<<(unsigned)((p.R + K12_RB / 32 - 1) / (K12_RB / 32)), K12_RB, 0, st>>>(p);
    k12_number_kernel<<<1, 1024, 0, st>>>(p);
    LR_CUDA(cudaGetLastError());
    h->launches += 3;
    long long n = 0;
    LR_CUDA(cudaMemcpyAsync(&n, p.n_used, sizeof(long long), cudaMemcpyDeviceToHost, st));
    LR_CUDA(cudaMemcpyAsync(d_n, p.n_used, sizeof(long long), cudaMemcpyDeviceToDevice, st));
    LR_CUDA(cudaStreamSynchronize(st));
    p.n = n;
    std::vector<int32_t> zcols(bc);
    for (int q = 0; q < bc; ++q) zcols[q] = q;
    const int point_blocks = (int)std::min<long long>((p.R + K12_RB / 32 - 1) / (K12_RB / 32), 16LL * h->sm_count);
    for (int c0 = 0; c0 < n_act; c0 += bc) {
        p.c0 = c0;
        p.bc = std::min(bc, n_act - c0);
        k12_init_kernel<<<(p.bc + 127) / 128, 128, 0, st>>>(p);
        k12_point_kernel<<<point_blocks, K12_RB, 0, st>>>(p);
        LR_CUDA(cudaGetLastError());
        h->launches += 2;
        rc = lr_k10_sort(h, p.key[0], p.key[1], n, p.bc, p.band, p.bor, w9.ghist, st);
        if (rc != LR_OK) return rc;
        const long long cells = p.R * p.bc;
        k12_exp_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(p);
        LR_CUDA(cudaGetLastError());
        h->launches += 1;
        rc = lr_k9_run(h, w9.k9, who, p.L, n_samples, n_chains, 1, -1, p.bc, p.bc, zcols.data(), nullptr, nullptr, nullptr, p.r9,
                       w9.k9status, st);
        if (rc != LR_OK) return rc;
        k12_tail_kernel<<<p.bc, K12_FT, 0, st>>>(p);
        k12_grid_kernel<<<dim3((unsigned)((p.mcap + K12_FW - 1) / K12_FW), p.bc), K12_FT, 0, st>>>(p);
        k12_fit_kernel<<<p.bc, K12_FT, 0, st>>>(p);
        LR_CUDA(cudaGetLastError());
        h->launches += 3;
    }
    LR_CUDA(cudaStreamSynchronize(st));
    return LR_OK;
}
