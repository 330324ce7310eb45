// K9: split R-hat and effective sample size ("mean" ESS; Vehtari et al. 2021, section 3, as Stan and ArviZ compute them) of every
// column of the sample records of a run, over its chains, on the device -- without copying the records.
//
// Rows are lr_chain_rows of lr_common.cuh: the records of K3 / K6 / K7, or the matrices of lr_marginal_rates (ladder 1), read
// through the cold member of each ladder.  A column is a spec of lr_common.cuh (row[a] +- row[b] + add).
//
// Estimator (literate_b200.diagnostics.rhat_ess is its host restatement, step for step).  n = floor(S / 2); split chain 2c is
// draws [0, n) of chain c, split chain 2c + 1 draws [S - n, S) (the middle draw of an odd S is dropped); m = 2 M split chains.
//   mean_j    the mean of split chain j; exactly its value when all its draws are equal
//   acov_j(t) = (1/n) sum_{i < n - t} (x_ij - mean_j)(x_{i+t,j} - mean_j)
//   W = n/(n-1) mean_j acov_j(0);  var+ = (n-1)/n W + var_j(mean_j, ddof 1) (exactly 0 when all mean_j are equal)
//   R-hat = sqrt(var+ / W), sd = sqrt(var+), mean = the mean of the m n draws used
//   rho_t = 1 - (W - mean_j acov_j(t)) / var+, truncated by Geyer's initial positive sequence and made monotone (a running
//   minimum of the pair sums), tau = -1 + 2 sum_{t <= max_t} rho_t + rho_{max_t + 1} >= 1 / log10(m n), ESS = m n / tau,
//   lag = max_t.
// Degenerate columns: a non-finite draw -> every output NaN, lag -1; W = 0 and var+ = 0 (constant) -> R-hat NaN, ESS NaN, lag -1;
// W = 0 and var+ > 0 (every split chain stuck on its own value) -> R-hat +inf, ESS NaN, lag -1.
//
// Work.  A moments pass (32 columns per group, lane = column, one warp per split chain) writes every split chain's sum and mean
// and whether it is finite and constant.  Then lag blocks of doubling width (16, 32, 64, ... up to 4096 lags): one CTA per (column
// group, 64 lags of the block, slice of split chains) streams the draws of its split chains through shared memory in tiles of 64
// draws plus a halo of its lags, centred on the split chain's mean, and sums the lag products (a tile in registers, the tiles
// and split chains compensated, in a fixed order).  One thread per column then adds the slices in order, forms rho_t and advances
// Geyer's sequence over the block's lags with O(1) state; a finished column writes its outputs and counts itself.  The host reads
// that count once per block and stops when every column of the batch is done: the work follows the largest truncation lag
// reached, not n^2, and a record field is read about twice per lag block (once per 64 lags beyond 64).  Repeated calls are
// bit-identical; everything is fp64.  Scratch (per split chain moments, partial sums) comes from the handle's workspace, at
// most ~256 MB: columns are processed in batches.
#include <math_constants.h>
#include <algorithm>
#include "lr_common.cuh"

namespace {

constexpr int K9_G = 32;            // columns per group: lane c owns column c of its group
constexpr int K9_WARPS = 8;         // warps of the moments and lag kernels
constexpr int K9_TI = 64;           // draws per tile of the lag kernel
constexpr int K9_CTA_LAGS = 64;     // lags of one CTA (8 warps x 8 lags) once a block is 64 lags wide
constexpr int K9_MAX_BLOCK = 4096;  // widest lag block
constexpr int K9_PART_LAGS = 8192;  // slices x block width: the partial sums of one column, at most

struct K9Col {                      // per column of the batch
    lr_sum acc;                     // sum of the monotone pair sums confirmed so far
    double mean, W, varp;           // the mean of the draws, within variance, var+ (between-chain variance until block 0)
    double mono, ev, od;            // running minimum of the pair sums, the last pair (even, odd)
    long long t;                    // Geyer's t (odd)
    int stored, finite, constant, equal, done;
};

struct K9Args {
    lr_chain_rows src;
    long long n;                    // draws per split chain
    lr_col_specs cols;              // column specs of this batch
    int n_cols;                     // columns of this batch
    long long m;                    // split chains
    double* sum;                    // [m][n_cols] sum of each split chain
    double* mean;                   // [m][n_cols] mean of each split chain (exact for a constant one)
    int* flag;                      // [m][n_cols] bit 0: a non-finite draw, bit 1: not constant
    double* part;                   // [slices][block lags][n_cols] lag sums of the slices
    K9Col* col;                     // [n_cols]
    int* done;                      // [n_cols]
    unsigned* finished;             // columns of the batch finished
    unsigned long long* missing;    // (sample, ladder) pairs without a member at beta = 1 (first batch only)
    double* out;                    // [5][n_out] of this batch: mean, sd, rhat, ess, lag
    long long n_out;
};

// row of draw i of split chain j (lr_chain_row: a warp-wide call)
__device__ __forceinline__ const double* k9_row(const K9Args& p, long long j, long long i, int lane, bool* missing) {
    return lr_chain_row(p.src, (j & 1) ? p.src.S - p.n + i : i, j >> 1, lane, missing);
}

// grid (block of K9_WARPS split chains, group): warp w takes split chain blockIdx.x K9_WARPS + w, lane c column c of the group
__global__ void __launch_bounds__(K9_WARPS * 32) k9_moments_kernel(const K9Args p) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long j = (long long)blockIdx.x * K9_WARPS + warp;
    if (j >= p.m) return;
    const int col = blockIdx.y * K9_G + lane;
    const bool has = col < p.n_cols;
    lr_col_spec spec;
    if (has) spec = p.cols.load(col);
    lr_sum sum;
    double lo = CUDART_INF, hi = -CUDART_INF, first = 0.0;
    bool finite = true;
    unsigned long long miss = 0;
    for (long long i = 0; i < p.n; ++i) {
        bool m = false;
        const double* row = k9_row(p, j, i, lane, &m);
        miss += m;
        if (has) {
            const double v = spec.value(row);
            if (i == 0) first = v;
            sum.add(v);
            finite &= isfinite(v);
            lo = fmin(lo, v); hi = fmax(hi, v);
        }
    }
    if (miss && lane == 0 && blockIdx.y == 0 && p.missing) atomicAdd(p.missing, miss);
    if (!has) return;
    const size_t o = (size_t)j * p.n_cols + col;
    const double sv = sum.value();
    const bool constant = finite && lo == hi;
    p.sum[o] = sv;
    p.mean[o] = constant ? first : sv / (double)p.n;
    p.flag[o] = (finite ? 0 : 1) | (constant ? 0 : 2);
}

__device__ __forceinline__ void k9_finish(const K9Args& p, int col, K9Col& st, double mean, double sd, double rhat, double ess, double lag) {
    p.out[col] = mean; p.out[p.n_out + col] = sd; p.out[2 * p.n_out + col] = rhat; p.out[3 * p.n_out + col] = ess; p.out[4 * p.n_out + col] = lag;
    st.done = 1;
    p.done[col] = 1;
    atomicAdd(p.finished, 1u);
}

// one thread per column: finiteness, the mean of the draws, the between-chain variance, whether W = 0 must follow
__global__ void k9_init_kernel(const K9Args p) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= p.n_cols) return;
    K9Col st;
    memset(&st, 0, sizeof(st));
    lr_sum tot, mm;
    int fl_or = 0, fl_and = 2;
    bool equal = true;
    const double m0 = p.mean[col];
    for (long long j = 0; j < p.m; ++j) {
        const size_t o = (size_t)j * p.n_cols + col;
        tot.add(p.sum[o]);
        mm.add(p.mean[o]);
        fl_or |= p.flag[o]; fl_and &= p.flag[o];
        equal &= p.mean[o] == m0;
    }
    st.finite = !(fl_or & 1);
    st.constant = !(fl_or & 2);               // every split chain constant
    st.equal = equal;
    if (!st.finite) {
        k9_finish(p, col, st, CUDART_NAN, CUDART_NAN, CUDART_NAN, CUDART_NAN, -1.0);
    } else {
        const double xbar = mm.value() / (double)p.m;
        double between = 0.0;
        if (!equal) {
            lr_sum d2;
            for (long long j = 0; j < p.m; ++j) {
                const double d = p.mean[(size_t)j * p.n_cols + col] - xbar;
                d2.add(d * d);
            }
            between = d2.value() / (double)(p.m - 1);
        }
        st.varp = between;                      // completed with W by the first lag block
        st.mean = tot.value() / ((double)p.m * (double)p.n);
        p.done[col] = 0;
    }
    p.col[col] = st;
}

// grid (group, CTA of the block, slice): sums over the slice's split chains of the lag products for the lags
// tc0 + 8 LPT .. of this CTA; warp w owns lags tc0 + w LPT + q, q < LPT, lane c column c of the group
template <int LPT>
__global__ void __launch_bounds__(K9_WARPS * 32) k9_lag_kernel(const K9Args p, long long t0, long long t1, int width, long long per_slice) {
    constexpr int CL = K9_WARPS * LPT;                    // lags of this CTA
    __shared__ double sa[K9_TI][K9_G];                    // x[i0 + r] - mean, r < TI
    __shared__ double sb[K9_TI + CL][K9_G];               // x[i0 + tc0 + r] - mean, r < TI + CL
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int col = blockIdx.x * K9_G + lane;
    const bool has = col < p.n_cols;
    if (!__syncthreads_or(has && !p.done[col])) return;  // every column of the group finished
    const long long tc0 = t0 + (long long)blockIdx.y * CL;
    const long long j0 = (long long)blockIdx.z * per_slice, j1 = min(p.m, j0 + per_slice);
    lr_col_spec spec;
    if (has) spec = p.cols.load(col);
    lr_sum acc[LPT];
    for (long long j = j0; j < j1; ++j) {
        const double mu = has ? p.mean[(size_t)j * p.n_cols + col] : 0.0;
        for (long long i0 = 0; i0 < p.n - tc0; i0 += K9_TI) {
            for (int r = warp; r < 2 * K9_TI + CL; r += K9_WARPS) {
                const long long i = r < K9_TI ? i0 + r : i0 + tc0 + (r - K9_TI);
                double v = 0.0;
                if (i < p.n) {                            // warp-uniform
                    const double* row = k9_row(p, j, i, lane, nullptr);
                    if (has) v = __dsub_rn(spec.value(row), mu);
                }
                if (r < K9_TI) sa[r][lane] = v; else sb[r - K9_TI][lane] = v;
            }
            __syncthreads();
            double part[LPT], w[LPT];
#pragma unroll
            for (int q = 0; q < LPT; ++q) { part[q] = 0.0; w[q] = sb[warp * LPT + q][lane]; }
#pragma unroll 4
            for (int i = 0; i < K9_TI; ++i) {
                const double x = sa[i][lane];
#pragma unroll
                for (int q = 0; q < LPT; ++q) part[q] = fma(x, w[q], part[q]);
#pragma unroll
                for (int q = 0; q < LPT - 1; ++q) w[q] = w[q + 1];
                w[LPT - 1] = sb[i + warp * LPT + LPT][lane];       // at most TI + CL - 1
            }
#pragma unroll
            for (int q = 0; q < LPT; ++q) acc[q].add(part[q]);
            __syncthreads();
        }
    }
    if (!has) return;
#pragma unroll
    for (int q = 0; q < LPT; ++q) {
        const long long t = tc0 + warp * LPT + q;
        if (t < t1) p.part[((size_t)blockIdx.z * width + (size_t)(t - t0)) * p.n_cols + col] = acc[q].value();
    }
}

// one thread per column: the lag sums of [t0, t1) (slices added in order), then Geyer's sequence as far as they reach
__global__ void k9_step_kernel(const K9Args p, long long t0, long long t1, int width, int slices) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= p.n_cols || p.done[col]) return;
    K9Col st = p.col[col];
    const double mn = (double)p.m * (double)p.n;
    auto lagsum = [&](long long t) {
        lr_sum s;
        for (int z = 0; z < slices; ++z) s.add(p.part[((size_t)z * width + (size_t)(t - t0)) * p.n_cols + col]);
        return s.value();
    };
    auto rho = [&](long long t) { return 1.0 - (st.W - lagsum(t) / mn) / st.varp; };
    if (t0 == 0) {
        const double mean = st.mean;
        const double nn = (double)p.n;
        st.W = nn / (nn - 1.0) * (lagsum(0) / mn);
        st.varp = (nn - 1.0) / nn * st.W + st.varp;
        const double sd = sqrt(st.varp);
        if (st.W == 0.0) {
            k9_finish(p, col, st, mean, sd, st.varp == 0.0 ? CUDART_NAN : CUDART_INF, CUDART_NAN, -1.0);
            p.col[col] = st;
            return;
        }
        st.t = 1; st.ev = 1.0; st.od = rho(1); st.stored = 1; st.mono = CUDART_INF;
        st.acc = lr_sum();
    }
    for (;;) {
        if (!(st.t < p.n - 3 && st.ev + st.od > 0.0)) {               // Geyer's sequence ends: max_t = t - 2
            const double extra = (st.stored || st.ev > 0.0) ? st.ev : 0.0;
            double tau = -1.0 + 2.0 * st.acc.value() + extra;
            tau = fmax(tau, 1.0 / log10(mn));
            k9_finish(p, col, st, st.mean, sqrt(st.varp), sqrt(st.varp / st.W), mn / tau, (double)(st.t - 2));
            break;
        }
        if (st.t + 2 >= t1) break;                                    // the next pair lies in the next block
        const double s = st.ev + st.od;                               // the pair (t - 1, t) is inside [0, max_t]
        st.mono = fmin(st.mono, s);
        st.acc.add(st.mono);
        st.ev = rho(st.t + 1); st.od = rho(st.t + 2);
        st.stored = st.ev + st.od >= 0.0;
        st.t += 2;
    }
    p.col[col] = st;
}

template <int LPT>
void k9_launch_lag(const K9Args& p, int groups, long long t0, long long t1, int width, int slices, long long per_slice, cudaStream_t st) {
    const int ctas = (width + K9_WARPS * LPT - 1) / (K9_WARPS * LPT);
    k9_lag_kernel<LPT><<<dim3(groups, ctas, slices), K9_WARPS * 32, 0, st>>>(p, t0, t1, width, per_slice);
}

}  // namespace

// columns per batch: the per split chain moments (20 B) and the partial lag sums of a column within ~256 MB
static int k9_batch_cols(long long m, int n_cols) {
    const size_t per_col = (size_t)m * 20 + (size_t)K9_PART_LAGS * 8 + sizeof(K9Col) + 4;
    return (int)std::max<size_t>(1, std::min<size_t>((size_t)n_cols, ((size_t)256 << 20) / per_col));
}

// K9's scratch: the staged specs, the finished count, then one batch's buffers, placed from `base` (null: only measured) for p.m
// split chains; returns its bytes
static size_t k9_layout(char* base, K9Args& p, lr_col_specs& spec, int n_cols) {
    const int batch_cols = k9_batch_cols(p.m, n_cols);
    lr_carve w{base};
    spec = lr_col_specs::carve(w, n_cols);
    p.finished = w.take<unsigned>(1);
    p.sum = w.take<double>((size_t)p.m * batch_cols);
    p.mean = w.take<double>((size_t)p.m * batch_cols);
    p.flag = w.take<int>((size_t)p.m * batch_cols);
    p.part = w.take<double>((size_t)K9_PART_LAGS * batch_cols);
    p.col = w.take<K9Col>(batch_cols);
    p.done = w.take<int>(batch_cols);
    return w.used;
}

size_t lr_k9_scratch_bytes(int64_t n_chains, int32_t n_cols) {
    K9Args p;
    lr_col_specs spec;
    p.m = 2 * n_chains;
    return k9_layout(nullptr, p, spec, n_cols);
}

int lr_k9_run(lr_handle_t h, char* w, const char* who, const double* d_rows, int64_t n_samples, int64_t n_chains, int32_t ladder,
              int32_t beta_col, int64_t row_stride, int32_t n_cols, const int32_t* h_col_a, const int32_t* h_col_b,
              const int32_t* h_col_sign, const double* h_col_add, double* d_out, int64_t* d_status, cudaStream_t st) {
    const long long n = n_samples / 2, m = 2 * n_chains;
    const int batch_cols = k9_batch_cols(m, n_cols);
    K9Args p;
    memset(&p, 0, sizeof(p));
    p.src = {d_rows, n_samples, n_chains, row_stride, ladder, beta_col};
    p.n = n; p.m = m; p.n_out = n_cols;
    lr_col_specs spec;
    k9_layout(w, p, spec, n_cols);
    int rc = lr_stage_col_specs(who, spec, n_cols, h_col_a, h_col_b, h_col_sign, h_col_add, st);
    if (rc != LR_OK) return rc;
    LR_CUDA(cudaMemsetAsync(d_status, 0, sizeof(int64_t), st));
    for (int c0 = 0; c0 < n_cols; c0 += batch_cols) {
        p.n_cols = std::min(batch_cols, n_cols - c0);
        p.cols = spec.from(c0);
        p.out = d_out + c0;
        p.missing = c0 == 0 ? (unsigned long long*)d_status : nullptr;
        const int groups = (p.n_cols + K9_G - 1) / K9_G;
        LR_CUDA(cudaMemsetAsync(p.finished, 0, sizeof(unsigned), st));
        k9_moments_kernel<<<dim3((unsigned)((m + K9_WARPS - 1) / K9_WARPS), groups), K9_WARPS * 32, 0, st>>>(p);
        const int cb = 128, cg = (p.n_cols + cb - 1) / cb;
        k9_init_kernel<<<cg, cb, 0, st>>>(p);
        h->launches += 2;
        long long t0 = 0;
        int width = 16;
        for (;;) {
            const long long t1 = std::min<long long>(t0 + width, n);
            const int lpt = width >= K9_CTA_LAGS ? 8 : width / K9_WARPS;
            const int ctas = (width + K9_WARPS * lpt - 1) / (K9_WARPS * lpt);
            // slices of split chains: enough CTAs for 4 per SM, at most K9_PART_LAGS / width partial sums per column
            long long slices = std::max<long long>(1, (4LL * h->sm_count + (long long)groups * ctas - 1) / ((long long)groups * ctas));
            slices = std::min<long long>(std::min<long long>(slices, m), std::max(1, K9_PART_LAGS / width));
            const long long per_slice = (m + slices - 1) / slices;
            slices = (m + per_slice - 1) / per_slice;
            if (lpt == 2) k9_launch_lag<2>(p, groups, t0, t1, width, (int)slices, per_slice, st);
            else if (lpt == 4) k9_launch_lag<4>(p, groups, t0, t1, width, (int)slices, per_slice, st);
            else k9_launch_lag<8>(p, groups, t0, t1, width, (int)slices, per_slice, st);
            k9_step_kernel<<<cg, cb, 0, st>>>(p, t0, t1, width, (int)slices);
            LR_CUDA(cudaGetLastError());
            h->launches += 2;
            unsigned fin = 0;
            LR_CUDA(cudaMemcpyAsync(&fin, p.finished, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
            LR_CUDA(cudaStreamSynchronize(st));
            if ((int)fin >= p.n_cols) break;
            LR_REQUIRE(t1 < n, "%s: %d columns unfinished after every lag (internal error)", who, p.n_cols - (int)fin);
            t0 = t1;
            width = std::min(2 * width, K9_MAX_BLOCK);
        }
    }
    return LR_OK;
}

extern "C" int lr_chain_diagnostics(lr_handle_t h, const double* d_rows, int64_t n_samples, int64_t n_chains, int32_t ladder, int32_t beta_col,
                                    int64_t row_stride, int32_t n_cols, const int32_t* h_col_a, const int32_t* h_col_b,
                                    const int32_t* h_col_sign, const double* h_col_add, double* d_out, int64_t* d_status, void* stream) {
    int rc = lr_check_chain_rows("lr_chain_diagnostics", h, d_out && d_status, d_rows, n_samples, n_chains, ladder, beta_col, row_stride,
                                 n_cols, h_col_a, h_col_b, h_col_sign);
    if (rc != LR_OK) return rc;
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    rc = lr_ws_acquire(h, lr_k9_scratch_bytes(n_chains, n_cols), st);
    if (rc != LR_OK) return rc;
    return lr_k9_run(h, (char*)h->ws, "lr_chain_diagnostics", d_rows, n_samples, n_chains, ladder, beta_col, row_stride, n_cols,
                     h_col_a, h_col_b, h_col_sign, h_col_add, d_out, d_status, st);
}
