// K10: the rank-normalised split R-hat and the bulk and tail effective sample sizes (Vehtari et al. 2021; ArviZ's _rhat_rank,
// _ess_bulk, _ess_tail) of every column of the sample records of a run, over its chains, on the device.
// literate_b200.diagnostics.rank_rhat_ess is the host restatement and the definition.
//
// Rows, ladders and column specs are those of K9 (k9_diag.cu).  n = floor(S / 2); the split draws of chain c are its draws [0, n)
// and [S - n, S); N = 2 M n of them per column.  Split position i < 2n of chain c is row i M + c of Z (i >= n: draw S - 2n + i).
//
// lr_rank_transform, per batch of columns:
//   1. gather: every draw of the column (the middle draw of an odd S too) becomes an order-preserving key (lr_key; -0 as +0); the
//      split draws go to a segment of N keys in Z-row order, the middle draws to a segment of M keys, and the value of each split
//      draw to its z slot of Z.  The AND and OR of all keys of a column give the digits every key shares (their sort passes are
//      skipped: integer columns such as K_l need two or three of eight); flags say whether a split draw is non-finite or NaN.
//   2. a segmented LSD radix sort of the keys (8-bit digits), many CTAs per segment: per pass a tile histogram, one scan per
//      segment over (digit, tile), and a stable scatter in which each warp ranks its keys with __match_any_sync (K8's scheme).
//   3. median of the sorted split draws ((a + b) / 2 of the middle two), q05 and q95 of all M S draws (numpy's "linear" method,
//      the order statistics from the sorted split and middle segments), NaN as numpy gives it.
//   4. rank pass: each split draw's key is looked up in its sorted segment (two binary searches give the count of draws below it
//      and of its ties), so the average rank before + (ties + 1) / 2 is exact, also for runs of a million equal draws; z =
//      Phi^-1((r - 3/8) / (N + 1/4)), evaluated from the smaller tail so that extreme ranks keep full precision.  The same pass
//      writes I_0.05, I_0.95 and |x - median| and its key.
//   5. the folded values are sorted (step 2) and ranked (step 4) into z_f.
// lr_rank_diagnostics runs the transform on a batch into the workspace, K9 (lr_k9_run, on the workspace behind K10's buffers) on
// the batch's 4 columns per column of Z, and a last kernel that applies the degenerate rules.  Everything is integer counting,
// order statistics and per-draw arithmetic, so repeated calls are bit-identical.
#include <math_constants.h>
#include <algorithm>
#include <vector>
#include "lr_common.cuh"

namespace {

constexpr int K10_G = 32;               // columns per group: lane c owns column c of its group
constexpr int K10_TW = 4;               // warps of the gather and rank kernels (a 32 x 32 key tile each in shared memory)
constexpr int K10_ST = 256;             // threads of the sort kernels
constexpr int K10_SW = K10_ST / 32;
constexpr int K10_ITEMS = 16;           // keys per thread of a sort tile
constexpr int K10_TILE = K10_ST * K10_ITEMS;
constexpr size_t K10_BUDGET = (size_t)1 << 30;   // K10's own scratch per batch (a batch holds at least one column)
constexpr int K10_MAX_BATCH = 8192;

struct K10Args {
    lr_chain_rows src;
    long long n;                    // split draws per chain and half
    lr_col_specs cols;              // column specs of this batch
    int n_cols;                     // columns of this batch
    long long N, Nmid;              // split draws, middle draws (M or 0) per column
    double* Z; long long zs, zq;    // Z row stride, distance of the slots z, z_f, I_05, I_95; Z points at the batch's first column
    unsigned long long* kx[2];      // [n_cols][N] split keys, ping-pong
    unsigned long long* km[2];      // [n_cols][Nmid] middle keys
    unsigned long long* kf[2];      // [n_cols][N] folded keys
    unsigned long long* band;       // [n_cols] AND, OR of every key of the column; then of the folded keys
    unsigned long long* bor;
    unsigned long long* fand;
    unsigned long long* f_or;
    int* flag;                      // [n_cols] bit 0: a non-finite split draw, 1: a NaN split draw, 2: a NaN draw
    double* quant; long long qn;    // [3][qn]: median, q05, q95 of the batch's first column
    unsigned long long* missing;    // (sample, ladder) pairs without a member at beta = 1
};

__device__ __forceinline__ unsigned long long k10_key(double v) { return lr_key(v == 0.0 ? 0.0 : v); }

__global__ void k10_init_kernel(const K10Args p) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.n_cols) return;
    p.band[c] = ~0ull; p.bor[c] = 0ull; p.fand[c] = ~0ull; p.f_or[c] = 0ull; p.flag[c] = 0;
}

// where row r = (s, chain) goes: its split position i M + chain, or -1 - chain for the middle draw of an odd S
__device__ __forceinline__ long long k10_pos(const K10Args& p, long long r) {
    const long long M = p.src.M, s = r / M, ch = r - s * M;
    if (s < p.n) return s * M + ch;
    if (s >= p.src.S - p.n) return (s - (p.src.S - 2 * p.n)) * M + ch;
    return -1 - ch;
}

// grid (row tiles, group): warp w takes 32 rows at a time; lane = column while reading the records (a row's fields are adjacent),
// lane = row while writing the keys (a column's segment is contiguous)
__global__ void __launch_bounds__(K10_TW * 32) k10_gather_kernel(const K10Args p) {
    __shared__ unsigned long long sk[K10_TW][32][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int col = blockIdx.y * K10_G + lane;
    const bool has = col < p.n_cols;
    lr_col_spec spec;
    if (has) spec = p.cols.load(col);
    const long long R = p.src.S * p.src.M;
    unsigned long long kand = ~0ull, kor = 0ull, miss = 0;
    int fl = 0;
    for (long long r0 = ((long long)blockIdx.x * K10_TW + warp) * 32; r0 < R; r0 += (long long)gridDim.x * K10_TW * 32) {
        for (int j = 0; j < 32; ++j) {
            const long long r = r0 + j;
            if (r >= R) break;                                       // warp-uniform
            const long long sm = r / p.src.M;
            bool m = false;
            const double* row = lr_chain_row(p.src, sm, r - sm * p.src.M, lane, &m);
            miss += m;
            unsigned long long k = 0;
            if (has) {
                const double v = spec.value(row);
                k = k10_key(v);
                kand &= k; kor |= k;
                const long long pos = k10_pos(p, r);
                if (v != v) fl |= 4;
                if (pos >= 0) {
                    if (!isfinite(v)) fl |= 1;
                    if (v != v) fl |= 2;
                    p.Z[pos * p.zs + col] = v;
                }
            }
            sk[warp][j][lane] = k;
        }
        __syncwarp();
        const long long r = r0 + lane;
        if (r < R) {
            const long long pos = k10_pos(p, r);
            for (int q = 0; q < K10_G; ++q) {
                const int cq = blockIdx.y * K10_G + q;
                if (cq >= p.n_cols) break;
                const unsigned long long k = sk[warp][lane][q];
                if (pos >= 0) p.kx[0][(size_t)cq * p.N + pos] = k;
                else p.km[0][(size_t)cq * p.Nmid + (-1 - pos)] = k;
            }
        }
        __syncwarp();
    }
    if (has) {
        atomicAnd(p.band + col, kand); atomicOr(p.bor + col, kor);
        if (fl) atomicOr(p.flag + col, fl);
    }
    if (miss && lane == 0 && blockIdx.y == 0 && p.missing) atomicAdd(p.missing, miss);
}

// ---- segmented LSD radix sort of [segs][L] keys between b0 and b1; segment s skips the digits its AND / OR say agree
struct K10Sort {
    unsigned long long* b0; unsigned long long* b1;
    long long L; int tiles;
    const unsigned long long* band; const unsigned long long* bor;
    unsigned* ghist;                // [segs][256][tiles] counts, then their exclusive scan
};

// grid (tile, segment): the digit counts of one tile
__global__ void __launch_bounds__(K10_ST) k10_hist_kernel(const K10Sort q, int d) {
    __shared__ unsigned h[256];
    const int seg = blockIdx.y, tid = threadIdx.x;
    const unsigned passes = lr_radix_passes(q.band[seg], q.bor[seg]);
    if (!((passes >> d) & 1u)) return;
    const unsigned long long* in = (lr_radix_src(passes, d) ? q.b1 : q.b0) + (size_t)seg * q.L;
    h[tid] = 0;
    __syncthreads();
    const unsigned lt = (1u << (tid & 31)) - 1u;
    const long long t0 = (long long)blockIdx.x * K10_TILE;
    for (int it = 0; it < K10_ITEMS; ++it) {
        const long long i = t0 + (long long)it * K10_ST + tid;
        const bool valid = i < q.L;
        const unsigned dig = valid ? (unsigned)(in[i] >> (8 * d)) & 255u : 256u;
        const unsigned peers = __match_any_sync(0xffffffffu, dig);
        if (valid && (peers & lt) == 0) atomicAdd(&h[dig], __popc(peers));
    }
    __syncthreads();
    q.ghist[((size_t)seg * 256 + tid) * q.tiles + blockIdx.x] = h[tid];
}

// one CTA per segment: exclusive scan of its 256 x tiles counts in (digit, tile) order
__global__ void __launch_bounds__(1024) k10_scan_kernel(const K10Sort q, int d) {
    __shared__ unsigned ws[32];
    const int seg = blockIdx.x, tid = threadIdx.x;
    const unsigned passes = lr_radix_passes(q.band[seg], q.bor[seg]);
    if (!((passes >> d) & 1u)) return;
    unsigned* g = q.ghist + (size_t)seg * 256 * q.tiles;
    const long long E = 256LL * q.tiles, per = (E + 1023) / 1024;
    const long long e0 = min(E, (long long)tid * per), e1 = min(E, e0 + per);
    unsigned sum = 0;
    for (long long e = e0; e < e1; ++e) sum += g[e];
    unsigned x = sum;                                              // inclusive scan over the block
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) ws[warp] = x;
    __syncthreads();
    if (warp == 0) {
        unsigned w = ws[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned y = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += y; }
        ws[lane] = w;
    }
    __syncthreads();
    unsigned run = x - sum + (warp ? ws[warp - 1] : 0u);
    for (long long e = e0; e < e1; ++e) { const unsigned v = g[e]; g[e] = run; run += v; }
}

// grid (tile, segment): the tile's keys to their places, in order (sub-tiles of 256 one after the other, warps in order, lanes in
// order), two barriers per sub-tile
__global__ void __launch_bounds__(K10_ST) k10_scatter_kernel(const K10Sort q, int d) {
    __shared__ unsigned base[256];
    __shared__ unsigned cnt[K10_SW][256];
    __shared__ unsigned off[K10_SW][256];
    const int seg = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned passes = lr_radix_passes(q.band[seg], q.bor[seg]);
    if (!((passes >> d) & 1u)) return;
    const int src = lr_radix_src(passes, d);
    const unsigned long long* in = (src ? q.b1 : q.b0) + (size_t)seg * q.L;
    unsigned long long* out = (src ? q.b0 : q.b1) + (size_t)seg * q.L;
    base[tid] = q.ghist[((size_t)seg * 256 + tid) * q.tiles + blockIdx.x];
    for (int w = 0; w < K10_SW; ++w) cnt[w][tid] = 0;
    __syncthreads();
    const unsigned lt = (1u << lane) - 1u;
    const long long t0 = (long long)blockIdx.x * K10_TILE;
    for (int it = 0; it < K10_ITEMS; ++it) {
        const long long i = t0 + (long long)it * K10_ST + tid;
        if (t0 + (long long)it * K10_ST >= q.L) break;             // block-uniform
        const bool valid = i < q.L;
        const unsigned long long k = valid ? in[i] : 0ull;
        const unsigned dig = valid ? (unsigned)(k >> (8 * d)) & 255u : 256u;
        const unsigned peers = __match_any_sync(0xffffffffu, dig);
        const unsigned rank = __popc(peers & lt);
        if (valid && rank == 0) cnt[warp][dig] = __popc(peers);
        __syncthreads();
        {
            unsigned run = base[tid];
            for (int w = 0; w < K10_SW; ++w) { const unsigned cw = cnt[w][tid]; off[w][tid] = run; run += cw; cnt[w][tid] = 0; }
            base[tid] = run;
        }
        __syncthreads();
        if (valid) out[off[warp][dig] + rank] = k;
    }
}

int k10_sort(lr_handle_t h, const K10Sort& q, int segs, cudaStream_t st) {
    if (q.L == 0 || segs == 0) return LR_OK;
    for (int d = 0; d < 8; ++d) {
        k10_hist_kernel<<<dim3(q.tiles, segs), K10_ST, 0, st>>>(q, d);
        k10_scan_kernel<<<segs, 1024, 0, st>>>(q, d);
        k10_scatter_kernel<<<dim3(q.tiles, segs), K10_ST, 0, st>>>(q, d);
    }
    LR_CUDA(cudaGetLastError());
    h->launches += 24;
    return LR_OK;
}

// the k-th smallest (0-based) of the sorted keys a[0, na) and b[0, nb), k < na + nb
__device__ unsigned long long k10_kth(const unsigned long long* a, long long na, const unsigned long long* b, long long nb, long long k) {
    long long lo = max(0LL, k + 1 - na), hi = min(k + 1, nb);      // keys taken from b
    while (lo < hi) {
        const long long jb = (lo + hi) >> 1, ja = k + 1 - jb;       // jb < nb, ja >= 1
        if (b[jb] < a[ja - 1]) lo = jb + 1; else hi = jb;
    }
    const long long ja = k + 1 - lo;
    unsigned long long x = ja > 0 ? a[ja - 1] : 0ull;
    if (lo > 0) x = max(x, b[lo - 1]);
    return x;
}

// np.quantile(x, p) ("linear"): h = (n - 1) p, the order statistics below and above it, numpy's two-sided lerp
__device__ double k10_quantile(const unsigned long long* a, long long na, const unsigned long long* b, long long nb, double p) {
    const long long n = na + nb;
    const double hv = __dmul_rn((double)(n - 1), p);
    double lo_v, hi_v, g;
    if (hv >= (double)(n - 1)) {                                     // numpy: both neighbours the last, gamma = h + 1
        lo_v = hi_v = lr_val(k10_kth(a, na, b, nb, n - 1));
        g = __dadd_rn(hv, 1.0);
    } else {
        const double fl = floor(hv);
        const long long lo = (long long)fl;
        lo_v = lr_val(k10_kth(a, na, b, nb, lo));
        hi_v = lr_val(k10_kth(a, na, b, nb, lo + 1));
        g = __dsub_rn(hv, fl);
    }
    const double diff = __dsub_rn(hi_v, lo_v);
    if (g >= 0.5) return __dsub_rn(hi_v, __dmul_rn(diff, __dsub_rn(1.0, g)));
    return __dadd_rn(lo_v, __dmul_rn(diff, g));
}

// one thread per column: median of the split draws, q05 and q95 of all draws
__global__ void k10_quant_kernel(const K10Args p) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.n_cols) return;
    const unsigned passes = lr_radix_passes(p.band[c], p.bor[c]);
    const unsigned long long* a = p.kx[lr_radix_src(passes, 8)] + (size_t)c * p.N;
    const unsigned long long* b = p.km[lr_radix_src(passes, 8)] + (size_t)c * p.Nmid;
    const int fl = p.flag[c];
    const double med = (fl & 2) ? CUDART_NAN : __dadd_rn(lr_val(a[p.N / 2 - 1]), lr_val(a[p.N / 2])) / 2.0;
    const double q05 = (fl & 4) ? CUDART_NAN : k10_quantile(a, p.N, b, p.Nmid, 0.05);
    const double q95 = (fl & 4) ? CUDART_NAN : k10_quantile(a, p.N, b, p.Nmid, 0.95);
    p.quant[c] = med; p.quant[p.qn + c] = q05; p.quant[2 * p.qn + c] = q95;
}

// z of the average rank of `key` among the sorted keys s[0, N): (r - 3/8) / (N + 1/4) and its complement are exact ratios of
// exact numerators, so the smaller one goes to Phi^-1
__device__ __forceinline__ double k10_z(const unsigned long long* s, long long N, unsigned long long key) {
    long long lo = 0, hi = N;
    while (lo < hi) { const long long m = (lo + hi) >> 1; if (s[m] < key) lo = m + 1; else hi = m; }
    const long long before = lo;
    hi = N;
    while (lo < hi) { const long long m = (lo + hi) >> 1; if (s[m] <= key) lo = m + 1; else hi = m; }
    const double r = (double)before + 0.5 * (double)(lo - before + 1);
    const double num = r - 0.375, den = (double)N + 0.25, rest = den - num;
    return num <= rest ? normcdfinv(num / den) : -normcdfinv(rest / den);
}

// grid (position tiles, group): z, I_05, I_95 and |x - median| (its key written transposed like the gather's) of every split draw
__global__ void __launch_bounds__(K10_TW * 32) k10_rank_kernel(const K10Args p) {
    __shared__ unsigned long long sk[K10_TW][32][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int col = blockIdx.y * K10_G + lane;
    const bool has = col < p.n_cols;
    const unsigned long long* sorted = nullptr;
    double med = 0.0, q05 = 0.0, q95 = 0.0;
    if (has) {
        sorted = p.kx[lr_radix_src(lr_radix_passes(p.band[col], p.bor[col]), 8)] + (size_t)col * p.N;
        med = p.quant[col]; q05 = p.quant[p.qn + col]; q95 = p.quant[2 * p.qn + col];
    }
    unsigned long long kand = ~0ull, kor = 0ull;
    for (long long p0 = ((long long)blockIdx.x * K10_TW + warp) * 32; p0 < p.N; p0 += (long long)gridDim.x * K10_TW * 32) {
        for (int j = 0; j < 32; ++j) {
            const long long pos = p0 + j;
            if (pos >= p.N) break;                                   // warp-uniform
            unsigned long long k = 0;
            if (has) {
                double* zr = p.Z + pos * p.zs + col;
                const double v = zr[0];
                zr[0] = k10_z(sorted, p.N, k10_key(v));
                zr[2 * p.zq] = v <= q05 ? 1.0 : 0.0;
                zr[3 * p.zq] = v <= q95 ? 1.0 : 0.0;
                const double f = fabs(__dsub_rn(v, med));
                zr[p.zq] = f;
                k = k10_key(f);
                kand &= k; kor |= k;
            }
            sk[warp][j][lane] = k;
        }
        __syncwarp();
        const long long pos = p0 + lane;
        if (pos < p.N) {
            for (int q = 0; q < K10_G; ++q) {
                const int cq = blockIdx.y * K10_G + q;
                if (cq >= p.n_cols) break;
                p.kf[0][(size_t)cq * p.N + pos] = sk[warp][lane][q];
            }
        }
        __syncwarp();
    }
    if (has) { atomicAnd(p.fand + col, kand); atomicOr(p.f_or + col, kor); }
}

// grid (position tiles, group): z_f of every split draw
__global__ void __launch_bounds__(K10_TW * 32) k10_rank_fold_kernel(const K10Args p) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int col = blockIdx.y * K10_G + lane;
    if (col >= p.n_cols) return;
    const unsigned long long* sorted = p.kf[lr_radix_src(lr_radix_passes(p.fand[col], p.f_or[col]), 8)] + (size_t)col * p.N;
    for (long long pos = (long long)blockIdx.x * K10_TW + warp; pos < p.N; pos += (long long)gridDim.x * K10_TW) {
        double* zr = p.Z + pos * p.zs + p.zq + col;
        zr[0] = k10_z(sorted, p.N, k10_key(zr[0]));
    }
}

// one thread per column of the batch: rules 2 and 4-6 of diagnostics.rank_rhat_ess on K9's outputs r9 [5][4 n_cols] of Z
__global__ void k10_finish_kernel(const K10Args p, const double* r9, double* out, long long n_out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.n_cols) return;
    const long long w = 4LL * p.n_cols;
    const double* rhat = r9 + 2 * w;
    const double* ess = r9 + 3 * w;
    const double rb = rhat[c], rt = rhat[p.n_cols + c];
    double v[5];
    if ((p.flag[c] & 1) || !isfinite(rb)) {                           // non-finite, constant or stuck column
        for (int k = 0; k < 8; ++k) out[k * n_out + c] = CUDART_NAN;
        return;
    }
    double e[2];
    for (int t = 0; t < 2; ++t) {                                     // a constant indicator (R-hat NaN) has N effective draws
        const int ci = (2 + t) * p.n_cols + c;
        e[t] = rhat[ci] != rhat[ci] ? (double)p.N : ess[ci];
    }
    v[0] = rb;
    v[1] = rt;
    v[2] = rt != rt ? rb : fmax(rb, rt);
    v[3] = ess[c];
    v[4] = (e[0] != e[0] || e[1] != e[1]) ? CUDART_NAN : fmin(e[0], e[1]);
    for (int k = 0; k < 5; ++k) out[(3 + k) * n_out + c] = v[k];
}

struct K10Plan {
    long long n, N, Nmid;
    int tiles, mid_tiles;
    size_t per_col;
};

K10Plan k10_plan(long long S, long long M, bool with_z) {
    K10Plan pl;
    pl.n = S / 2; pl.N = 2 * M * pl.n; pl.Nmid = (S & 1) ? M : 0;
    pl.tiles = (int)((pl.N + K10_TILE - 1) / K10_TILE);
    pl.mid_tiles = (int)((pl.Nmid + K10_TILE - 1) / K10_TILE);
    pl.per_col = (size_t)pl.N * 8 * 4 + (size_t)pl.Nmid * 8 * 2 + (size_t)pl.tiles * 256 * 4 + 64
                 + (with_z ? (size_t)pl.N * 32 + 5 * 4 * 8 : 0);
    return pl;
}

// lr_rank_diagnostics' buffers besides the transform's: K9's status, Z of a batch, K9's outputs on it, and K9's scratch
struct K10Diag { int64_t* status; double* Z; double* r9; char* k9; };

// The workspace of one call: the staged specs; with dg (lr_rank_diagnostics) K9's status, Z of a batch and K9's outputs on it;
// the sort buffers of a batch of bc columns; with dg K9's scratch last.  Placed from `base` (null: only measured) for p's chains;
// returns its bytes.
size_t k10_layout(char* base, K10Args* p, K10Sort* sx, K10Sort* sm, K10Sort* sf, lr_col_specs* spec, K10Diag* dg, const K10Plan& pl,
                  int n_cols, int bc) {
    lr_carve w{base};
    *spec = lr_col_specs::carve(w, n_cols);
    if (dg) {
        dg->status = w.take<int64_t>(1);
        dg->Z = w.take<double>((size_t)pl.N * 4 * bc);
        dg->r9 = w.take<double>((size_t)5 * 4 * bc);
    }
    const size_t keys = (size_t)bc * pl.N, mids = (size_t)bc * std::max<long long>(pl.Nmid, 1);
    p->kx[0] = w.take<unsigned long long>(keys); p->kx[1] = w.take<unsigned long long>(keys);
    p->kf[0] = w.take<unsigned long long>(keys); p->kf[1] = w.take<unsigned long long>(keys);
    p->km[0] = w.take<unsigned long long>(mids); p->km[1] = w.take<unsigned long long>(mids);
    unsigned* ghist = w.take<unsigned>((size_t)bc * 256 * std::max(pl.tiles, 1));
    p->band = w.take<unsigned long long>(bc); p->bor = w.take<unsigned long long>(bc);
    p->fand = w.take<unsigned long long>(bc); p->f_or = w.take<unsigned long long>(bc);
    p->flag = w.take<int>(bc);
    *sx = {p->kx[0], p->kx[1], pl.N, pl.tiles, p->band, p->bor, ghist};
    *sm = {p->km[0], p->km[1], pl.Nmid, pl.mid_tiles, p->band, p->bor, ghist};
    *sf = {p->kf[0], p->kf[1], pl.N, pl.tiles, p->fand, p->f_or, ghist};
    if (dg) dg->k9 = w.take<char>(lr_k9_scratch_bytes(p->src.M, 4 * bc));
    return w.used;
}

// steps 1-5 on the batch of p (its specs, Z and quant set)
int k10_transform_batch(lr_handle_t h, K10Args& p, K10Sort& sx, K10Sort& sm, K10Sort& sf, cudaStream_t st) {
    const int groups = (p.n_cols + K10_G - 1) / K10_G;
    const int cb = 128, cg = (p.n_cols + cb - 1) / cb;
    const long long want = std::max<long long>(1, 8LL * h->sm_count / groups);
    k10_init_kernel<<<cg, cb, 0, st>>>(p);
    const long long rtiles = (p.src.S * p.src.M + K10_TW * 32 - 1) / (K10_TW * 32);
    k10_gather_kernel<<<dim3((unsigned)std::min<long long>(rtiles, want), groups), K10_TW * 32, 0, st>>>(p);
    LR_CUDA(cudaGetLastError());
    int rc = k10_sort(h, sx, p.n_cols, st);
    if (rc == LR_OK) rc = k10_sort(h, sm, p.n_cols, st);
    if (rc != LR_OK) return rc;
    k10_quant_kernel<<<cg, cb, 0, st>>>(p);
    const long long ptiles = (p.N + K10_TW * 32 - 1) / (K10_TW * 32);
    k10_rank_kernel<<<dim3((unsigned)std::min<long long>(ptiles, want), groups), K10_TW * 32, 0, st>>>(p);
    LR_CUDA(cudaGetLastError());
    rc = k10_sort(h, sf, p.n_cols, st);
    if (rc != LR_OK) return rc;
    const long long ftiles = (p.N + K10_TW - 1) / K10_TW;
    k10_rank_fold_kernel<<<dim3((unsigned)std::min<long long>(ftiles, want), groups), K10_TW * 32, 0, st>>>(p);
    LR_CUDA(cudaGetLastError());
    h->launches += 5;
    return LR_OK;
}

void k10_args(K10Args* p, const double* d_rows, int64_t n_samples, int64_t n_chains, int32_t ladder, int32_t beta_col, int64_t row_stride,
              const K10Plan& pl) {
    memset(p, 0, sizeof(*p));
    p->src = {d_rows, n_samples, n_chains, row_stride, ladder, beta_col};
    p->n = pl.n; p->N = pl.N; p->Nmid = pl.Nmid;
}

}  // namespace

size_t lr_k10_sort_ghist(int64_t L) { return (size_t)256 * std::max<int64_t>(1, (L + K10_TILE - 1) / K10_TILE); }

int lr_k10_sort(lr_handle_t h, unsigned long long* b0, unsigned long long* b1, int64_t L, int segs, const unsigned long long* band,
                const unsigned long long* bor, unsigned* ghist, cudaStream_t st) {
    const K10Sort q{b0, b1, L, (int)((L + K10_TILE - 1) / K10_TILE), band, bor, ghist};
    return k10_sort(h, q, segs, st);
}

extern "C" int lr_rank_transform(lr_handle_t h, const double* d_rows, int64_t n_samples, int64_t n_chains, int32_t ladder, int32_t beta_col,
                                 int64_t row_stride, int32_t n_cols, const int32_t* h_col_a, const int32_t* h_col_b,
                                 const int32_t* h_col_sign, const double* h_col_add, double* d_z, double* d_quant, int64_t* d_status,
                                 void* stream) {
    const char* who = "lr_rank_transform";
    int rc = lr_check_chain_rows(who, h, d_z && d_quant && d_status, d_rows, n_samples, n_chains, ladder, beta_col, row_stride, n_cols,
                                 h_col_a, h_col_b, h_col_sign);
    if (rc != LR_OK) return rc;
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    const K10Plan pl = k10_plan(n_samples, n_chains, false);
    const int bc = (int)std::max<size_t>(1, std::min<size_t>({(size_t)n_cols, (size_t)K10_MAX_BATCH, K10_BUDGET / pl.per_col}));
    K10Args p;
    k10_args(&p, d_rows, n_samples, n_chains, ladder, beta_col, row_stride, pl);
    K10Sort sx, sm, sf;
    lr_col_specs spec;
    rc = lr_ws_acquire(h, k10_layout(nullptr, &p, &sx, &sm, &sf, &spec, nullptr, pl, n_cols, bc), st);
    if (rc != LR_OK) return rc;
    k10_layout((char*)h->ws, &p, &sx, &sm, &sf, &spec, nullptr, pl, n_cols, bc);
    rc = lr_stage_col_specs(who, spec, n_cols, h_col_a, h_col_b, h_col_sign, h_col_add, st);
    if (rc != LR_OK) return rc;
    LR_CUDA(cudaMemsetAsync(d_status, 0, sizeof(int64_t), st));
    p.zs = 4LL * n_cols; p.zq = n_cols; p.qn = n_cols;
    for (int c0 = 0; c0 < n_cols; c0 += bc) {
        p.n_cols = std::min(bc, n_cols - c0);
        p.cols = spec.from(c0);
        p.Z = d_z + c0; p.quant = d_quant + c0;
        p.missing = c0 == 0 ? (unsigned long long*)d_status : nullptr;
        rc = k10_transform_batch(h, p, sx, sm, sf, st);
        if (rc != LR_OK) return rc;
    }
    return LR_OK;
}

extern "C" int lr_rank_diagnostics(lr_handle_t h, const double* d_rows, int64_t n_samples, int64_t n_chains, int32_t ladder, int32_t beta_col,
                                   int64_t row_stride, int32_t n_cols, const int32_t* h_col_a, const int32_t* h_col_b,
                                   const int32_t* h_col_sign, const double* h_col_add, double* d_out, int64_t* d_status, void* stream) {
    const char* who = "lr_rank_diagnostics";
    int rc = lr_check_chain_rows(who, h, d_out && d_status, d_rows, n_samples, n_chains, ladder, beta_col, row_stride, n_cols, h_col_a,
                                 h_col_b, h_col_sign);
    if (rc != LR_OK) return rc;
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    const K10Plan pl = k10_plan(n_samples, n_chains, true);
    const int bc = (int)std::max<size_t>(1, std::min<size_t>({(size_t)n_cols, (size_t)K10_MAX_BATCH, K10_BUDGET / pl.per_col}));
    K10Args p;
    k10_args(&p, d_rows, n_samples, n_chains, ladder, beta_col, row_stride, pl);
    K10Sort sx, sm, sf;
    K10Diag dg;
    lr_col_specs spec;
    rc = lr_ws_acquire(h, k10_layout(nullptr, &p, &sx, &sm, &sf, &spec, &dg, pl, n_cols, bc), st);
    if (rc != LR_OK) return rc;
    k10_layout((char*)h->ws, &p, &sx, &sm, &sf, &spec, &dg, pl, n_cols, bc);
    rc = lr_stage_col_specs(who, spec, n_cols, h_col_a, h_col_b, h_col_sign, h_col_add, st);
    if (rc != LR_OK) return rc;
    std::vector<int32_t> zcols(4 * (size_t)bc);
    for (int j = 0; j < 4 * bc; ++j) zcols[j] = j;
    LR_CUDA(cudaMemsetAsync(d_status, 0, sizeof(int64_t), st));
    for (int c0 = 0; c0 < n_cols; c0 += bc) {
        p.n_cols = std::min(bc, n_cols - c0);
        p.cols = spec.from(c0);
        p.Z = dg.Z; p.zs = 4LL * p.n_cols; p.zq = p.n_cols;
        p.quant = d_out + c0; p.qn = n_cols;
        p.missing = c0 == 0 ? (unsigned long long*)d_status : nullptr;
        rc = k10_transform_batch(h, p, sx, sm, sf, st);
        if (rc != LR_OK) return rc;
        rc = lr_k9_run(h, dg.k9, who, dg.Z, 2 * pl.n, n_chains, 1, -1, 4LL * p.n_cols, 4 * p.n_cols, zcols.data(), nullptr, nullptr,
                       nullptr, dg.r9, dg.status, st);
        if (rc != LR_OK) return rc;
        k10_finish_kernel<<<(p.n_cols + 127) / 128, 128, 0, st>>>(p, dg.r9, d_out + c0, n_cols);
        LR_CUDA(cudaGetLastError());
        h->launches += 1;
    }
    return LR_OK;
}
