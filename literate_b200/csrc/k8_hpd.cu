// K8: per-column means and exact HPD intervals of a row-major fp64 matrix on the device -- the sample records of K3 / K6 / K7
// (the columns a log would hold, built from up to two record fields and a constant) or K5's expanded per-sample matrices.
//
// calcHPD (plotRJforward.v3.py:12-28, summary.hpd_columns) only looks at the lowest and the highest m = n - n_in + 1 order
// statistics of a column (n_in = rint(level n)): the narrowest window is x[i + n_in - 1] - x[i], i < m.  So instead of sorting
// whole columns:
//   1. every value becomes an order-preserving 64-bit key (NaN -> the largest key, as np.sort puts NaN last);
//   2. eight radix-select passes (8-bit digits, most significant first) over a group of 32 columns find, per column, the key of
//      rank m - 1 (top of the lower tail) and of rank n_in - 1 (bottom of the upper tail); the first pass also sums the columns;
//   3. one more pass gathers the keys strictly beyond each threshold; each tail is padded to m with copies of its threshold
//      (equal keys are equal values);
//   4. one CTA per tail sorts it (LSD radix, 8-bit digits, skipping digits in which every key agrees);
//   5. one CTA per column takes the first narrowest window (a NaN width wins, as in numpy's argmin) and the mean.
// The records are never copied; the scratch (tails, histograms) is bounded, columns are processed in batches of groups.
// Everything is integer counting except the widths and the sums, which are compensated and have a fixed order: repeated calls
// are bit-identical.
#include <math_constants.h>
#include <algorithm>
#include <climits>
#include "lr_common.cuh"

namespace {

constexpr int K8_G = 32;                    // columns per group: lane c of a warp owns column c of its group
constexpr int K8_WARPS = 16;                // warps of the pass kernel (one row per warp at a time)
constexpr int K8_HB = 257;                  // padded bins per histogram row: bank = (column + digit) % 32, no conflicts for equal digits
constexpr int K8_PASS_SMEM = 2 * K8_G * K8_HB * 4 + K8_WARPS * K8_G * 8;
constexpr int K8_SORT_WARPS = 16;
constexpr int K8_WIN_THREADS = 256;

struct K8Ctrl { long long n, n_in, m; int ok; };

struct K8Args {
    const double* rows;
    long long n_rows, stride;
    int mask_col;
    lr_col_specs cols;              // column specs of this batch
    int n_cols;                     // columns of this batch
    long long rows_per_slice;
    int n_slices;
    double level;
    K8Ctrl* ctrl;
    unsigned long long* sel;        // [n_cols][4]: threshold prefix (lower, upper), rank left to find (lower, upper)
    unsigned* ghist;                // [n_cols][2][256]
    double* part;                   // [n_slices][n_cols] partial sums
    unsigned* cnt;                  // [2 n_cols] keys gathered per tail
    unsigned long long* tail0;      // [2 n_cols][m_stride]: tail t of column c is segment t n_cols + c
    unsigned long long* tail1;      // ping-pong buffer of the sort
    int* where;                     // [2 n_cols] buffer holding the sorted tail
    long long m_stride;
    double* mean; double* lo; double* hi; long long* n_out;
};

// pass < 8: histogram of digit `pass` (most significant first) of the keys that share each threshold's prefix so far (pass 0 also
// writes the partial sums); pass 8: gathers the keys below the lower / above the upper threshold.  grid (slice, group).
__global__ void __launch_bounds__(K8_WARPS * 32) k8_pass_kernel(const K8Args p, int pass) {
    extern __shared__ __align__(16) unsigned char k8_smem[];
    unsigned* hist = reinterpret_cast<unsigned*>(k8_smem);                              // [2][32][K8_HB]
    double* red = reinterpret_cast<double*>(k8_smem + 2 * K8_G * K8_HB * 4);           // [K8_WARPS][32]
    if (pass > 0 && !p.ctrl->ok) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int col = blockIdx.y * K8_G + lane;
    const bool has = col < p.n_cols;
    if (pass < 8)
        for (int i = threadIdx.x; i < 2 * K8_G * K8_HB; i += blockDim.x) hist[i] = 0;
    lr_col_spec spec;
    unsigned long long pre0 = 0, pre1 = 0, mhi = 0;
    const int shift = pass < 8 ? 56 - 8 * pass : 0;
    if (has) {
        spec = p.cols.load(col);
        if (pass > 0) { pre0 = p.sel[4 * col]; pre1 = p.sel[4 * col + 1]; }
    }
    if (pass > 0 && pass < 8) mhi = ~0ull << (shift + 8);
    __syncthreads();
    const long long r0 = (long long)blockIdx.x * p.rows_per_slice;
    const long long r1 = min(p.n_rows, r0 + p.rows_per_slice);
    lr_sum sum;
    if (has) {
        unsigned* h0 = hist + lane * K8_HB;
        unsigned* h1 = hist + (K8_G + lane) * K8_HB;
#pragma unroll 4
        for (long long r = r0 + warp; r < r1; r += K8_WARPS) {
            const double* row = p.rows + r * p.stride;
            if (p.mask_col >= 0 && row[p.mask_col] != 1.0) continue;
            const double v = spec.value(row);
            const unsigned long long k = lr_key(v);
            if (pass < 8) {
                if (pass == 0) sum.add(v);
                const unsigned d = (unsigned)(k >> shift) & 255u;
                if ((k & mhi) == pre0) atomicAdd(h0 + d, 1u);
                if ((k & mhi) == pre1) atomicAdd(h1 + d, 1u);
            } else {
                if (k < pre0) p.tail0[(size_t)col * p.m_stride + atomicAdd(p.cnt + col, 1u)] = k;
                if (k > pre1) p.tail0[(size_t)(p.n_cols + col) * p.m_stride + atomicAdd(p.cnt + p.n_cols + col, 1u)] = k;
            }
        }
    }
    if (pass == 8) return;
    if (pass == 0) red[warp * K8_G + lane] = sum.value();
    __syncthreads();
    if (pass == 0 && warp == 0 && has) {                 // fixed order: rows of a warp in order, then the warps in order
        lr_sum t;
        for (int w = 0; w < K8_WARPS; ++w) t.add(red[w * K8_G + lane]);
        p.part[(size_t)blockIdx.x * p.n_cols + col] = t.value();
    }
    for (int i = threadIdx.x; i < 2 * K8_G * 256; i += blockDim.x) {
        const int t = i / (K8_G * 256), lc = (i / 256) % K8_G, d = i % 256;
        const unsigned v = hist[(t * K8_G + lc) * K8_HB + d];
        const int cc = blockIdx.y * K8_G + lc;
        if (v && cc < p.n_cols) atomicAdd(p.ghist + ((size_t)cc * 2 + t) * 256 + d, v);
    }
}

// One thread per (column, threshold): picks the digit of the bin holding the rank still to be found, and clears the histogram.
// After pass 0 the histogram totals give n (every counted row adds one key to every column), hence n_in and m.
__global__ void k8_select_kernel(const K8Args p, int pass) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * p.n_cols) return;
    const int col = i >> 1, t = i & 1;
    unsigned* h = p.ghist + (size_t)i * 256;
    if (pass == 0) {
        long long n = 0;
        for (int d = 0; d < 256; ++d) n += h[d];
        const long long n_in = (long long)rint(p.level * (double)n);
        const long long m = n - n_in + 1;
        const int ok = n_in >= 2 && m <= p.m_stride;
        if (i == 0) { p.ctrl->n = n; p.ctrl->n_in = n_in; p.ctrl->m = m; p.ctrl->ok = ok; }
        if (!ok) { for (int d = 0; d < 256; ++d) h[d] = 0; return; }
        p.sel[4 * col + t] = 0;
        p.sel[4 * col + 2 + t] = t == 0 ? (unsigned long long)(m - 1) : (unsigned long long)(n_in - 1);
    } else if (!p.ctrl->ok) {
        return;
    }
    const unsigned long long k = p.sel[4 * col + 2 + t];
    unsigned long long cum = 0;
    int dig = 255;
    for (int d = 0; d < 256; ++d) {
        const unsigned c = h[d];
        if (k < cum + c) { dig = d; break; }
        cum += c;
    }
    for (int d = 0; d < 256; ++d) h[d] = 0;
    p.sel[4 * col + t] |= (unsigned long long)dig << (56 - 8 * pass);
    p.sel[4 * col + 2 + t] = k - cum;
}

// every tail starts as m copies of its threshold key; grid (chunk, segment)
__global__ void k8_fill_kernel(const K8Args p) {
    if (!p.ctrl->ok) return;
    const int seg = blockIdx.y;
    const unsigned long long key = seg < p.n_cols ? p.sel[4 * seg] : p.sel[4 * (seg - p.n_cols) + 1];
    unsigned long long* out = p.tail0 + (size_t)seg * p.m_stride;
    const long long m = p.ctrl->m;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (long long)gridDim.x * blockDim.x) out[i] = key;
    if (blockIdx.x == 0 && threadIdx.x == 0) p.cnt[seg] = 0;
}

// LSD radix sort of one tail (one CTA per segment) between tail0 and tail1.  A tile of 512 keys per step: each warp ranks its
// keys by digit with __match_any_sync (stable: lane order), 256 threads turn the per-warp counts into offsets (warp order), and
// the keys go to their places -- two barriers per tile.
__global__ void __launch_bounds__(K8_SORT_WARPS * 32) k8_sort_kernel(const K8Args p) {
    __shared__ unsigned hist[8][256];
    __shared__ unsigned cnt[K8_SORT_WARPS][256];
    __shared__ unsigned off[K8_SORT_WARPS][256];
    __shared__ unsigned base[256];
    __shared__ int skip;
    if (!p.ctrl->ok) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nt = blockDim.x;
    const long long m = p.ctrl->m;
    const int seg = blockIdx.x;
    unsigned long long* buf[2] = {p.tail0 + (size_t)seg * p.m_stride, p.tail1 + (size_t)seg * p.m_stride};
    const unsigned lt = (1u << lane) - 1u;
    for (int i = tid; i < 8 * 256; i += nt) (&hist[0][0])[i] = 0;
    for (int i = tid; i < K8_SORT_WARPS * 256; i += nt) (&cnt[0][0])[i] = 0;
    __syncthreads();
    for (long long t0 = 0; t0 < m; t0 += nt) {          // the histograms of all eight digits in one read
        const long long i = t0 + tid;
        const bool valid = i < m;
        const unsigned long long k = valid ? buf[0][i] : 0ull;
#pragma unroll
        for (int d = 0; d < 8; ++d) {
            const unsigned dig = valid ? (unsigned)(k >> (8 * d)) & 255u : 256u;
            const unsigned peers = __match_any_sync(0xffffffffu, dig);
            if (valid && (peers & lt) == 0) atomicAdd(&hist[d][dig], __popc(peers));
        }
    }
    __syncthreads();
    int src = 0;
    for (int d = 0; d < 8; ++d) {
        __syncthreads();                                  // the previous digit's keys are in place, `skip` has been read
        if (tid == 0) {
            skip = hist[d][(unsigned)(buf[src][0] >> (8 * d)) & 255u] == (unsigned)m;
            if (!skip) {
                unsigned run = 0;
                for (int q = 0; q < 256; ++q) { base[q] = run; run += hist[d][q]; }
            }
        }
        __syncthreads();
        if (skip) continue;
        const unsigned long long* in = buf[src];
        unsigned long long* out = buf[src ^ 1];
        for (long long t0 = 0; t0 < m; t0 += nt) {
            const long long i = t0 + tid;
            const bool valid = i < m;
            const unsigned long long k = valid ? in[i] : 0ull;
            const unsigned dig = valid ? (unsigned)(k >> (8 * d)) & 255u : 256u;
            const unsigned peers = __match_any_sync(0xffffffffu, dig);
            const unsigned rank = __popc(peers & lt);
            if (valid && rank == 0) cnt[warp][dig] = __popc(peers);
            __syncthreads();
            if (tid < 256) {
                unsigned run = base[tid];
                for (int w = 0; w < K8_SORT_WARPS; ++w) { const unsigned c = cnt[w][tid]; off[w][tid] = run; run += c; cnt[w][tid] = 0; }
                base[tid] = run;
            }
            __syncthreads();
            if (valid) out[off[warp][dig] + rank] = k;
        }
        src ^= 1;
    }
    if (tid == 0) p.where[seg] = src;
}

// (NaN first, then the smaller width, then the smaller index): numpy's argmin over the widths, a total order, so the reduction
// order does not matter
__device__ __forceinline__ bool k8_better(double wa, long long ia, double wb, long long ib) {
    const bool na = wa != wa, nb = wb != wb;
    if (na != nb) return na;
    if (!na && wa != wb) return wa < wb;
    return ia < ib;
}

// one CTA per column: the first narrowest window over the two sorted tails, and the mean from the partial sums in slice order
__global__ void __launch_bounds__(K8_WIN_THREADS) k8_window_kernel(const K8Args p) {
    __shared__ double sw[K8_WIN_THREADS];
    __shared__ long long si[K8_WIN_THREADS];
    const int col = blockIdx.x, tid = threadIdx.x;
    const K8Ctrl c = *p.ctrl;
    if (col == 0 && tid == 0 && p.n_out) *p.n_out = c.n;
    if (!c.ok) {
        if (tid == 0) { p.mean[col] = CUDART_NAN; p.lo[col] = CUDART_NAN; p.hi[col] = CUDART_NAN; }
        return;
    }
    const unsigned long long* L = (p.where[col] ? p.tail1 : p.tail0) + (size_t)col * p.m_stride;
    const unsigned long long* U = (p.where[p.n_cols + col] ? p.tail1 : p.tail0) + (size_t)(p.n_cols + col) * p.m_stride;
    double bw = CUDART_INF;
    long long bi = LLONG_MAX;
    for (long long i = tid; i < c.m; i += K8_WIN_THREADS) {
        const double w = __dsub_rn(lr_val(U[i]), lr_val(L[i]));
        if (k8_better(w, i, bw, bi)) { bw = w; bi = i; }
    }
    sw[tid] = bw; si[tid] = bi;
    __syncthreads();
    for (int o = K8_WIN_THREADS / 2; o > 0; o >>= 1) {
        if (tid < o && k8_better(sw[tid + o], si[tid + o], sw[tid], si[tid])) { sw[tid] = sw[tid + o]; si[tid] = si[tid + o]; }
        __syncthreads();
    }
    if (tid == 0) {
        const long long i = si[0];
        p.lo[col] = lr_val(L[i]);
        p.hi[col] = lr_val(U[i]);
        lr_sum t;
        for (int q = 0; q < p.n_slices; ++q) t.add(p.part[(size_t)q * p.n_cols + col]);
        p.mean[col] = t.value() / (double)c.n;
    }
}

// the workspace of lr_column_hpd: the staged specs, the control block, then one batch's buffers, placed from `base` (null: only
// measured) for p.n_slices and p.m_stride; returns its bytes
size_t k8_layout(char* base, K8Args& p, lr_col_specs& spec, int n_cols, int batch_cols) {
    lr_carve w{base};
    spec = lr_col_specs::carve(w, n_cols);
    p.ctrl = w.take<K8Ctrl>(1);
    p.sel = w.take<unsigned long long>((size_t)batch_cols * 4);
    p.ghist = w.take<unsigned>((size_t)batch_cols * 2 * 256);
    p.part = w.take<double>((size_t)p.n_slices * batch_cols);
    p.cnt = w.take<unsigned>((size_t)batch_cols * 2);
    p.where = w.take<int>((size_t)batch_cols * 2);
    p.tail0 = w.take<unsigned long long>((size_t)2 * batch_cols * p.m_stride);
    p.tail1 = w.take<unsigned long long>((size_t)2 * batch_cols * p.m_stride);
    return w.used;
}

}  // namespace

extern "C" int lr_column_hpd(lr_handle_t h, const double* d_rows, int64_t n_rows, int64_t row_stride, int32_t mask_col, int32_t n_cols,
                             const int32_t* h_col_a, const int32_t* h_col_b, const int32_t* h_col_sign, const double* h_col_add,
                             double level, double* d_mean, double* d_lo, double* d_hi, int64_t* d_n, void* stream) {
    LR_REQUIRE(h && d_mean && d_lo && d_hi && h_col_a && (n_rows == 0 || d_rows), "lr_column_hpd: null pointer");
    LR_REQUIRE(n_rows >= 0 && n_rows < ((int64_t)1 << 31) && n_cols >= 1 && row_stride >= 1, "lr_column_hpd: bad sizes");
    LR_REQUIRE(mask_col < row_stride, "lr_column_hpd: mask column %d outside the row of %lld doubles", mask_col, (long long)row_stride);
    LR_REQUIRE(level > 0.0 && level <= 1.0, "lr_column_hpd: level must be in (0, 1]");
    { int rc0 = lr_check_col_specs("lr_column_hpd", n_cols, row_stride, h_col_a, h_col_b, h_col_sign); if (rc0 != LR_OK) return rc0; }
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    static bool attr[64] = {};
    if (h->device >= 64 || !attr[h->device]) {
        LR_CUDA(cudaFuncSetAttribute(k8_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, K8_PASS_SMEM));
        if (h->device < 64) attr[h->device] = true;
    }
    // m can only be smaller for fewer (masked) rows, by at most one more than for n_rows (rounding of level n)
    const long long m_stride = std::max<long long>(1, n_rows - (long long)rint(level * (double)n_rows) + 2);
    const int n_slices = (int)std::max<long long>(1, std::min<long long>((n_rows + 1023) / 1024, 2LL * h->sm_count));
    const long long rows_per_slice = std::max<long long>(1, (n_rows + n_slices - 1) / n_slices);
    const int n_groups = (n_cols + K8_G - 1) / K8_G;
    // columns per batch: tails (two, ping-pong) of at most ~512 MB per batch, at least one group, at most 1023 (the fill kernel's
    // grid.y holds a batch's 2 x columns tails)
    const size_t per_group = (size_t)K8_G * (4 * (size_t)m_stride * 8 + 32 + 2048 + 16 + (size_t)n_slices * 8);
    const int groups_per_batch = (int)std::max<size_t>(1, std::min<size_t>(std::min(n_groups, 1023), ((size_t)512 << 20) / per_group));
    const int batch_cols = std::min(n_cols, groups_per_batch * K8_G);
    K8Args p;
    memset(&p, 0, sizeof(p));
    p.rows = d_rows; p.n_rows = n_rows; p.stride = row_stride; p.mask_col = mask_col;
    p.rows_per_slice = rows_per_slice; p.n_slices = n_slices; p.level = level; p.m_stride = m_stride;
    lr_col_specs spec;
    int rc = lr_ws_acquire(h, k8_layout(nullptr, p, spec, n_cols, batch_cols), st);
    if (rc != LR_OK) return rc;
    k8_layout((char*)h->ws, p, spec, n_cols, batch_cols);
    rc = lr_stage_col_specs("lr_column_hpd", spec, n_cols, h_col_a, h_col_b, h_col_sign, h_col_add, st);
    if (rc != LR_OK) return rc;
    LR_CUDA(cudaMemsetAsync(p.ghist, 0, (size_t)batch_cols * 2 * 256 * 4, st));
    for (int c0 = 0; c0 < n_cols; c0 += batch_cols) {
        p.n_cols = std::min(batch_cols, n_cols - c0);
        p.cols = spec.from(c0);
        p.mean = d_mean + c0; p.lo = d_lo + c0; p.hi = d_hi + c0;
        p.n_out = c0 == 0 ? (long long*)d_n : nullptr;
        const dim3 grid(n_slices, (p.n_cols + K8_G - 1) / K8_G);
        const int sel_blocks = (2 * p.n_cols + 63) / 64;
        for (int pass = 0; pass < 8; ++pass) {
            k8_pass_kernel<<<grid, K8_WARPS * 32, K8_PASS_SMEM, st>>>(p, pass);
            k8_select_kernel<<<sel_blocks, 64, 0, st>>>(p, pass);
        }
        k8_fill_kernel<<<dim3((unsigned)std::min<long long>(64, (m_stride + 255) / 256), 2 * p.n_cols), 256, 0, st>>>(p);
        k8_pass_kernel<<<grid, K8_WARPS * 32, K8_PASS_SMEM, st>>>(p, 8);
        k8_sort_kernel<<<2 * p.n_cols, K8_SORT_WARPS * 32, 0, st>>>(p);
        k8_window_kernel<<<p.n_cols, K8_WIN_THREADS, 0, st>>>(p);
        LR_CUDA(cudaGetLastError());
        h->launches += 20;
    }
    return LR_OK;
}
