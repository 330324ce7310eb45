// K11: posterior predictive check of the per-bin births and deaths of a run, on the device, without copying the records.
//
// Every likelihood of the samplers is  C + sum_j [A^b_j log lambda_j - B^b_j lambda_j] + sum_j [A^d_j log mu_j - B^d_j mu_j]:
// event weights A and exposures B per bin and side (K3: lr_dataset_bin_terms; K6 / K7: sp, br, ex, br of their statistics).  The
// model it states is y_j ~ Poisson(rate_j B_j) per side and bin, with the exposure B held at its observed value (no new lineage
// table is simulated).  For each record (posterior draw) and each bin with B > 0 K11 draws one replicate count from that model
// and compares it with the observed A, bin by bin and through the Poisson deviance of the whole record.
//
// Rows are lr_chain_rows of lr_common.cuh (the (s, k) layout, ladder and beta_col of lr_chain_diagnostics: tempered runs are
// checked over their cold members).  Rates per bin: K3 records (layout 0) take the rate of the segment bin j falls in under the
// likelihood's own mapping (side_stats in chain_device.cuh: segment k starts at bin floor(t_k) - floor(start_time), clamped to
// [0, n_bins]; bin j takes the last segment starting at or before it); dense records (layout 1) hold the birth rates at
// [rate_col, rate_col + n_bins) and the death rates after them.
//
// Work.  A pre-pass (one warp per record) marks the records that cannot be used.  The draw kernel runs one CTA per (chunk of
// K11_CHUNK records, block of bins, side): thread = bin, records in order; each thread keeps its bin's counts and compensated sums
// in registers and writes them once per chunk, and the per-record deviance sums over the CTA's bins are reduced per batch of
// K11_BATCH records (compensated butterflies, then the warps in order).  Small kernels then add the chunks, the bin blocks and the
// records in a fixed order.  Integer counts are exact and the fp64 sums are compensated in a fixed order: repeated calls are
// bit-identical.
#include <algorithm>
#include "lr_common.cuh"

namespace {

constexpr int K11_CHUNK = 1024;     // records of one draw CTA: the per-bin partials are [records / K11_CHUNK][2][n_bins]
constexpr int K11_BATCH = 8;        // records per deviance reduction of the draw kernel
constexpr int K11_NI = 4;           // int64 fields per side and bin: used, sum y_rep, #(y_rep > A), #(y_rep == A)
constexpr int K11_NF = 3;           // fp64 fields: sum mu, sum mu^2, sum A
constexpr int K11_RB = 256;         // threads of the record kernels
constexpr int K11_MAX_BINS = 65535 * 256;   // the draw grid's bin blocks of 256 stay within gridDim.y; < 2^24 (the counter's bin field)

struct K11Args {
    lr_chain_rows src;
    int layout, rate_col, nb, s0f;
    const double* terms;            // [n_rep][4][nb]: A^b, B^b, A^d, B^d
    const int* rep;                 // [M]
    long long chain_id0;
    uint32_t k0, k1;
    long long R;                    // S M logical records
    int bb;                         // bin blocks per side
    unsigned char* flag;            // [R] 0 used, 1 skipped (a rate, a mean or a K3 segment unusable), 2 no member at beta = 1
    long long* part_i;              // [chunks][2][nb][K11_NI]
    double* part_f;                 // [chunks][2][nb][K11_NF]
    double* dev_part;               // [R][2][bb][2]: deviance sums (observed, replicate) of each bin block
    double* dev;                    // [R][4]: D_obs^b, D_rep^b, D_obs^d, D_rep^d (NaN when not used)
    double* glob_part;              // [record blocks][6]
    unsigned long long* count;      // [4] the caller's global counts
    unsigned long long* status;     // [3]
};

// the deviance term of one bin, 0 log 0 = 0: y log(y / mu) - (y - mu)
__device__ __forceinline__ double k11_dev_term(double y, double mu) {
    return y == 0.0 ? mu : __dsub_rn(__dmul_rn(y, log(__ddiv_rn(y, mu))), __dsub_rn(y, mu));
}

// compensated butterfly over the warp: every lane ends with the same (s, c) (TwoSum's error term is exact, so symmetric)
__device__ __forceinline__ double k11_warp_sum(double v) {
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

// one warp per logical record: which records are used
__global__ void __launch_bounds__(K11_RB) k11_scan_kernel(const K11Args p) {
    __shared__ int sjb[K11_RB / 32][2][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long r = (long long)blockIdx.x * (K11_RB / 32) + warp;
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
        bool ok = (p.layout != 0 || (K[0] > 0 && K[1] > 0)) && row[0] >= 0.0 && row[0] < 9.2e18;   // the iteration keys the draws
        if (ok) {
            const double* T = p.terms + (size_t)p.rep[c] * 4 * p.nb;
            for (int side = 0; side < 2; ++side)
                for (int j = lane; j < p.nb; j += 32) {
                    const double B = T[(2 * side + 1) * p.nb + j];
                    if (!(B > 0.0)) continue;
                    const double rate = p.layout == 0 ? row[(side ? 80 : 16) + lr_k3_slot(sjb[warp][side], K[side], j)]
                                                      : row[p.rate_col + side * p.nb + j];
                    const double mu = __dmul_rn(rate, B);
                    ok &= mu >= 0.0 && mu <= LR_POIS_MU_MAX;
                }
        }
        f = __all_sync(0xffffffffu, ok) ? 0 : 1;
    }
    if (lane == 0) {
        p.flag[r] = f;
        if (f) atomicAdd(p.status + (f == 1 ? 0 : 2), 1ull);
    }
}

// grid (chunk, bin block, side), blockDim.x = bins of a block (a multiple of 32)
__global__ void __launch_bounds__(256) k11_draw_kernel(const K11Args p) {
    extern __shared__ double k11_smem[];
    const int nw = blockDim.x >> 5, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* sdev = k11_smem;                                   // [K11_BATCH][nw][2]
    int* sjb = (int*)(sdev + K11_BATCH * nw * 2) + warp * 32;  // [nw][32]
    const int side = blockIdx.z;
    const int j = blockIdx.y * blockDim.x + threadIdx.x;
    const bool on = j < p.nb;
    const long long r_begin = (long long)blockIdx.x * K11_CHUNK, r_end = min(p.R, r_begin + K11_CHUNK);
    long long n = 0, sy = 0, gt = 0, eq = 0;
    lr_sum smu, smu2, sA;
    unsigned exhausted = 0;
    for (long long r0 = r_begin; r0 < r_end; r0 += K11_BATCH) {
        for (int q = 0; q < K11_BATCH; ++q) {
            const long long r = r0 + q;
            double obs = 0.0, rep = 0.0;
            if (r < r_end && p.flag[r] == 0) {                  // uniform over the CTA
                const long long s = r / p.src.M, c = r - s * p.src.M;
                const double* row = lr_chain_row(p.src, s, c, lane, nullptr);
                int K = 0;
                if (p.layout == 0) K = lr_k3_stage(p.s0f, p.nb, row, side, lane, sjb);
                const double* T = p.terms + (size_t)p.rep[c] * 4 * p.nb;
                if (on) {
                    const double A = T[2 * side * p.nb + j], B = T[(2 * side + 1) * p.nb + j];
                    if (B > 0.0) {
                        const double rate = p.layout == 0 ? row[(side ? 80 : 16) + lr_k3_slot(sjb, K, j)] : row[p.rate_col + side * p.nb + j];
                        const double mu = __dmul_rn(rate, B);
                        const long long it = (long long)row[0];
                        const unsigned long long g = (unsigned long long)(p.chain_id0 + c);
                        const long long y = lr_poisson(mu, (uint32_t)it, (uint32_t)((unsigned long long)it >> 32), (uint32_t)j | ((uint32_t)side << 24),
                                                       (uint32_t)g, p.k0, p.k1, &exhausted);
                        const double yd = (double)y;
                        n += 1; sy += y; gt += yd > A; eq += yd == A;
                        smu.add(mu); smu2.add(__dmul_rn(mu, mu)); sA.add(A);
                        obs = k11_dev_term(A, mu);
                        rep = k11_dev_term(yd, mu);
                    }
                }
            }
            obs = k11_warp_sum(obs);
            rep = k11_warp_sum(rep);
            if (lane == 0) { sdev[(q * nw + warp) * 2] = obs; sdev[(q * nw + warp) * 2 + 1] = rep; }
        }
        __syncthreads();
        if (threadIdx.x < 2 * K11_BATCH) {
            const int q = threadIdx.x >> 1, v = threadIdx.x & 1;
            const long long r = r0 + q;
            if (r < r_end && p.flag[r] == 0) {
                lr_sum acc;
                for (int w = 0; w < nw; ++w) acc.add(sdev[(q * nw + w) * 2 + v]);
                p.dev_part[(((size_t)r * 2 + side) * p.bb + blockIdx.y) * 2 + v] = acc.value();
            }
        }
        __syncthreads();
    }
    if (on) {
        const size_t o = ((size_t)blockIdx.x * 2 + side) * p.nb + j;
        long long* pi = p.part_i + o * K11_NI;
        double* pf = p.part_f + o * K11_NF;
        pi[0] = n; pi[1] = sy; pi[2] = gt; pi[3] = eq;
        pf[0] = smu.value(); pf[1] = smu2.value(); pf[2] = sA.value();
    }
    if (exhausted) atomicAdd(p.status + 1, (unsigned long long)exhausted);
}

// one thread per (side, bin): the chunks in order
__global__ void k11_bins_kernel(const K11Args p, long long chunks, long long* __restrict__ out_i, double* __restrict__ out_f) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 2 * p.nb) return;
    long long acc_i[K11_NI] = {0, 0, 0, 0};
    lr_sum acc_f[K11_NF];
    for (long long k = 0; k < chunks; ++k) {
        const size_t o = (size_t)k * 2 * p.nb + t;
#pragma unroll
        for (int f = 0; f < K11_NI; ++f) acc_i[f] += p.part_i[o * K11_NI + f];
#pragma unroll
        for (int f = 0; f < K11_NF; ++f) acc_f[f].add(p.part_f[o * K11_NF + f]);
    }
    const int side = t / p.nb, j = t - side * p.nb;
#pragma unroll
    for (int f = 0; f < K11_NI; ++f) out_i[((size_t)side * K11_NI + f) * p.nb + j] = acc_i[f];
#pragma unroll
    for (int f = 0; f < K11_NF; ++f) out_f[((size_t)side * K11_NF + f) * p.nb + j] = acc_f[f].value();
}

// one thread per record: the deviances, the global counts, one block's partial sums
__global__ void __launch_bounds__(K11_RB) k11_records_kernel(const K11Args p) {
    __shared__ double sp[K11_RB / 32][6];
    const long long r = (long long)blockIdx.x * K11_RB + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool used = r < p.R && p.flag[r] == 0;
    double D[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};              // obs b, rep b, obs d, rep d, obs total, rep total
    if (used) {
        for (int side = 0; side < 2; ++side)
            for (int v = 0; v < 2; ++v) {
                lr_sum acc;
                for (int b = 0; b < p.bb; ++b) acc.add(p.dev_part[(((size_t)r * 2 + side) * p.bb + b) * 2 + v]);
                D[2 * side + v] = 2.0 * acc.value();
            }
        D[4] = __dadd_rn(D[0], D[2]);
        D[5] = __dadd_rn(D[1], D[3]);
    }
    if (r < p.R) {
        double* o = p.dev + (size_t)r * 4;
        for (int k = 0; k < 4; ++k) o[k] = used ? D[k] : __longlong_as_double(0x7ff8000000000000ll);
    }
    const unsigned cu = __popc(__ballot_sync(0xffffffffu, used));
    const unsigned cb = __popc(__ballot_sync(0xffffffffu, used && D[1] >= D[0]));
    const unsigned cd = __popc(__ballot_sync(0xffffffffu, used && D[3] >= D[2]));
    const unsigned ct = __popc(__ballot_sync(0xffffffffu, used && D[5] >= D[4]));
    if (lane == 0) {
        if (cu) atomicAdd(p.count, (unsigned long long)cu);
        if (cb) atomicAdd(p.count + 1, (unsigned long long)cb);
        if (cd) atomicAdd(p.count + 2, (unsigned long long)cd);
        if (ct) atomicAdd(p.count + 3, (unsigned long long)ct);
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const double v = k11_warp_sum(D[k]);
        if (lane == 0) sp[warp][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        lr_sum acc;
        for (int w = 0; w < K11_RB / 32; ++w) acc.add(sp[w][threadIdx.x]);
        p.glob_part[(size_t)blockIdx.x * 6 + threadIdx.x] = acc.value();
    }
}

// six warps: warp k adds field k of the record blocks (lane-strided, then a compensated butterfly)
__global__ void k11_global_kernel(const K11Args p, long long blocks, double* __restrict__ out) {
    const int lane = threadIdx.x & 31, k = threadIdx.x >> 5;
    lr_sum acc;
    for (long long b = lane; b < blocks; b += 32) acc.add(p.glob_part[(size_t)b * 6 + k]);
    const double v = k11_warp_sum(acc.value());
    if (lane == 0) out[k] = v;
}

}  // namespace

extern "C" int lr_predictive_check(lr_handle_t h, const double* d_rows, int64_t n_samples, int64_t n_chains, int32_t ladder, int32_t beta_col,
                                   int64_t row_stride, int32_t layout, int32_t rate_col, double start_time, int32_t n_bins,
                                   const double* d_terms, int32_t n_rep, const int32_t* h_rep_of_chain, int64_t chain_id0, uint64_t seed,
                                   int64_t* d_bin_count, double* d_bin_sum, int64_t* d_glob_count, double* d_glob_sum, double* d_dev,
                                   int64_t* d_status, void* stream) {
    const char* who = "lr_predictive_check";
    const int32_t col0 = 0;
    int rc = lr_check_chain_rows(who, h, d_terms && d_bin_count && d_bin_sum && d_glob_count && d_glob_sum && d_status, d_rows, n_samples,
                                 n_chains, ladder, beta_col, row_stride, 1, &col0, nullptr, nullptr);
    if (rc != LR_OK) return rc;
    // bins go to bits 0..23 of the counter and blocks of 256 bins to gridDim.y (at most 65535)
    LR_REQUIRE(n_bins >= 1 && n_bins <= K11_MAX_BINS, "%s: n_bins must be 1 .. %d", who, K11_MAX_BINS);
    LR_REQUIRE(n_rep >= 1, "%s: n_rep must be at least 1", who);
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
    if (h_rep_of_chain)
        for (int64_t c = 0; c < n_chains; ++c)
            LR_REQUIRE(h_rep_of_chain[c] >= 0 && h_rep_of_chain[c] < n_rep, "%s: chain %lld uses replicate %d; the terms hold %d", who,
                       (long long)c, h_rep_of_chain[c], n_rep);
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;

    K11Args p;
    memset(&p, 0, sizeof(p));
    p.src = {d_rows, n_samples, n_chains, row_stride, ladder, beta_col};
    p.layout = layout; p.rate_col = rate_col; p.nb = n_bins; p.s0f = (int)floor(start_time);
    p.terms = d_terms; p.chain_id0 = chain_id0;
    p.k0 = (uint32_t)seed; p.k1 = (uint32_t)(seed >> 32);
    p.R = n_samples * n_chains;
    const int threads = (int)std::min<long long>(256, ((long long)n_bins + 31) / 32 * 32);
    p.bb = (n_bins + threads - 1) / threads;
    const long long chunks = (p.R + K11_CHUNK - 1) / K11_CHUNK;
    const long long rblocks = (p.R + K11_RB - 1) / K11_RB;
    auto layout_ws = [&](char* base) {
        lr_carve w{base};
        p.rep = w.take<int>(n_chains);
        p.flag = w.take<unsigned char>(p.R);
        p.part_i = w.take<long long>((size_t)chunks * 2 * n_bins * K11_NI);
        p.part_f = w.take<double>((size_t)chunks * 2 * n_bins * K11_NF);
        p.dev_part = w.take<double>((size_t)p.R * 2 * p.bb * 2);
        p.dev = d_dev ? d_dev : w.take<double>((size_t)p.R * 4);
        p.glob_part = w.take<double>((size_t)rblocks * 6);
        return w.used;
    };
    rc = lr_ws_acquire(h, layout_ws(nullptr), st);
    if (rc != LR_OK) return rc;
    layout_ws((char*)h->ws);
    p.count = (unsigned long long*)d_glob_count;
    p.status = (unsigned long long*)d_status;

    int* hrep = (int*)calloc((size_t)n_chains, sizeof(int));
    LR_REQUIRE(hrep, "%s: out of host memory", who);
    if (h_rep_of_chain) memcpy(hrep, h_rep_of_chain, (size_t)n_chains * sizeof(int));
    const cudaError_t e = cudaMemcpyAsync((void*)p.rep, hrep, (size_t)n_chains * sizeof(int), cudaMemcpyHostToDevice, st);
    free(hrep);                                                  // pageable source: staged when the call returns
    LR_CUDA(e);
    LR_CUDA(cudaMemsetAsync(d_status, 0, 3 * sizeof(int64_t), st));
    LR_CUDA(cudaMemsetAsync(d_glob_count, 0, 4 * sizeof(int64_t), st));

    k11_scan_kernel<<<(unsigned)((p.R + K11_RB / 32 - 1) / (K11_RB / 32)), K11_RB, 0, st>>>(p);
    const size_t smem = (size_t)K11_BATCH * (threads / 32) * 2 * sizeof(double) + (size_t)(threads / 32) * 32 * sizeof(int);
    k11_draw_kernel<<<dim3((unsigned)chunks, (unsigned)p.bb, 2), threads, smem, st>>>(p);
    k11_bins_kernel<<<(2 * n_bins + 127) / 128, 128, 0, st>>>(p, chunks, (long long*)d_bin_count, d_bin_sum);
    k11_records_kernel<<<(unsigned)rblocks, K11_RB, 0, st>>>(p);
    k11_global_kernel<<<1, 6 * 32, 0, st>>>(p, rblocks, d_glob_sum);
    LR_CUDA(cudaGetLastError());
    h->launches += 5;
    return LR_OK;
}
