// Shared device/host helpers for the literate_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "../../include/literate_b200.h"

#ifndef __CUDACC__
#error "literate_b200 is CUDA-only: there is no CPU path"
#endif

#define LR_WARP 32
#define LR_SLOTS 32            // register slots per side of one chain (one per lane)
#define LR_FIX_SHIFT 52        // fractions of a year are accumulated in 2^-52 fixed point
#define LR_FIX_SCALE 4503599627370496.0   // 2^52

// ---- error plumbing ------------------------------------------------------------------------
void lr_set_error(const char* fmt, ...);
#define LR_CUDA(call)                                                                        \
    do {                                                                                     \
        cudaError_t e__ = (call);                                                            \
        if (e__ != cudaSuccess) {                                                            \
            lr_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return LR_ERR_CUDA;                                                              \
        }                                                                                    \
    } while (0)
// same, running `cleanup` (free what the function has allocated so far) before returning
#define LR_CUDA_CLEAN(call, cleanup)                                                         \
    do {                                                                                     \
        cudaError_t e__ = (call);                                                            \
        if (e__ != cudaSuccess) {                                                            \
            lr_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            cleanup;                                                                         \
            return LR_ERR_CUDA;                                                              \
        }                                                                                    \
    } while (0)
#define LR_REQUIRE(cond, ...)                                                                \
    do {                                                                                     \
        if (!(cond)) {                                                                       \
            lr_set_error(__VA_ARGS__);                                                       \
            return LR_ERR_INVALID;                                                           \
        }                                                                                    \
    } while (0)

// staging buffers of the host-buffer entry points: enough in flight that the copy engine never waits for a K1 batch, even when
// another kernel (the chains of the previous table) leaves K1 only a few SMs
#define LR_NSTAGE 4

struct lr_handle_s {
    int device;
    int sm_count;
    int max_smem_optin;
    cudaStream_t stream;        // compute
    cudaStream_t copy_stream;   // host<->device staging
    cudaEvent_t ev[2 * LR_NSTAGE];   // [buf] copy of a batch done, [LR_NSTAGE + buf] its kernel done
    int64_t launches;           // kernels launched through this handle
    // grow-only workspace, handed from one entry point to the next IN STREAM ORDER (lr_ws_acquire)
    void* ws;
    size_t ws_bytes;
    cudaStream_t ws_stream;     // stream of the workspace's last user
    int ws_used;
    cudaEvent_t ev_order;       // scratch event of lr_order
    void* stage[LR_NSTAGE];
    size_t stage_bytes;
    // K1's memory of the last table's kind: one int in mapped pinned host memory that the kernel's CTA 0 writes (1 = the table
    // carries fractional times, 0 = integer years) and the NEXT lr_bin_accumulate reads without synchronising to choose between
    // its two bit-identical builds (k1_binstats.cu); a stale value costs speed only
    int* k1_hint;
    int k1_hint_used;
    // set by the host-buffer entry points around their per-batch passes: those are bound by the host link (K1 at 4.8 TB/s hides
    // behind 55 GB/s of copies) and run beside the chain kernels of the previous table, whose 64 KB shared-memory carve-out the
    // lane-private build (2 x 105 KB per SM) cannot share an SM with -- it would wait for whole SMs to drain
    int k1_general_only;
    int k1_last_build;          // what the last lr_bin_accumulate launched: 0 k1_bin_kernel, 1 k1_bin_lanes_kernel (lr_bin_last_build)
};

// Cross-stream ordering without host synchronisation.  Entry points take a caller stream or fall back to the handle's
// own; objects (datasets, chains, trend / dd samplers) and the workspace remember the stream that touched them last.
// lr_order makes `now` wait for everything submitted so far to `*last` (an event recorded there and waited for here) when
// the two differ, and moves `*last` to `now`.
struct lr_last_stream { cudaStream_t s; int valid; };
int lr_order(lr_handle_t h, lr_last_stream* last, cudaStream_t now);
// the workspace, at least `bytes` large, for work submitted to `stream` (ordered after its previous user)
int lr_ws_acquire(lr_handle_t h, size_t bytes, cudaStream_t stream);

// ---- host plumbing of the chain objects (K3 lr_chains_t, K6 lr_trend_t, K7 lr_dd_t) -------------------------------------------
// launch grid of the one-warp-per-chain kernels: few chains get one warp per CTA so that they spread over all SMs, many chains 4
inline int lr_chain_grid(int n, int& threads) {
    const int wpb = n <= 1024 ? 1 : 4;
    threads = wpb * 32;
    return (n + wpb - 1) / wpb;
}

// Warps per chain of the K6 / K7 chain loop.  W warps (one CTA) share a chain's bins when one warp per chain would leave most
// of the GPU idle and there are bins to share.  The environment variable `env` overrides the population rule (development):
// 0 one warp per chain, anything else the width by the bins.
inline int lr_chain_width(int n_bins, int n_chains, int sm_count, const char* env) {
    const int W = n_bins > 128 ? 4 : (n_bins > 64 ? 2 : 1);
    if (const char* e = getenv(env)) return atoi(e) ? W : 1;
    return (long long)n_chains * W > (long long)sm_count * 8 ? 1 : W;
}

// records a run of n_iter iterations from iteration it0 writes: one per multiple of sample_every in [it0, it0 + n_iter)
inline long long lr_records_per_run(long long it0, long long n_iter, long long sample_every) {
    const long long first = (it0 + sample_every - 1) / sample_every * sample_every;
    const long long it1 = it0 + n_iter;
    return first < it1 ? (it1 - 1 - first) / sample_every + 1 : 0;
}

// iteration counter of a chain, read from the device after everything submitted to the object so far; false on failure
inline bool lr_read_counter(lr_handle_t h, lr_last_stream* last, const long long* d_it, long long* it) {
    cudaSetDevice(h->device);
    lr_order(h, last, h->stream);
    cudaStreamSynchronize(h->stream);
    return cudaMemcpy(it, d_it, sizeof(long long), cudaMemcpyDeviceToHost) == cudaSuccess;
}

// The *_run_host entry points: `nrec` samples of `sample_bytes` each (nrec < 0: the iteration counter could not be read) are
// recorded into the workspace by run(d_records) -- d_records null: no records -- and copied to h_records; returns when done.
template <class Run>
int lr_run_into_host(lr_handle_t h, const char* fn, int64_t nrec, size_t sample_bytes, double* h_records, Run run) {
    LR_REQUIRE(nrec >= 0, "%s: could not read the iteration counter", fn);
    const size_t bytes = (size_t)nrec * sample_bytes;
    double* d_rec = nullptr;
    if (bytes) {
        int rc = lr_ws_acquire(h, bytes, h->stream);
        if (rc != LR_OK) return rc;
        d_rec = (double*)h->ws;
    }
    int rc = run(d_rec);
    if (rc != LR_OK) return rc;
    if (bytes) LR_CUDA(cudaMemcpyAsync(h_records, d_rec, bytes, cudaMemcpyDeviceToHost, h->stream));
    LR_CUDA(cudaStreamSynchronize(h->stream));
    return LR_OK;
}

// One launch on `stream` (null: the handle's own), ordered after everything submitted to the object so far (lr_order)
template <class Launch>
int lr_launch_ordered(lr_handle_t h, lr_last_stream* last, void* stream, Launch launch) {
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    { int rc0 = lr_order(h, last, st); if (rc0 != LR_OK) return rc0; }
    launch(st);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    return LR_OK;
}

// ---- tempered ladders of the chain objects (K3, K6, K7) ------------------------------------------------------------------------
// The swap_apply entry points: shard [first, first + n_chains) of global chain ids, gathered (lik, beta) table d_info_all[n_all][2]
// whose row 0 is global chain table_first.  launch(blocks, threads, stream) starts the sampler's apply kernel, one warp per chain.
template <class Launch>
int lr_swap_apply(lr_handle_t h, lr_last_stream* last, int n_chains, const double* d_info_all, int64_t table_first, int64_t n_all,
                  int64_t first, int32_t ladder, void* stream, const char* who, Launch launch) {
    LR_REQUIRE(d_info_all, "%s: null pointer", who);
    LR_REQUIRE(ladder >= 2 && ladder <= 32, "%s: ladder size must be 2..32", who);
    LR_REQUIRE(first >= table_first && first + n_chains <= table_first + n_all,
               "%s: this shard [first, first + n_chains) lies outside the gathered table", who);
    int threads;
    const int blocks = lr_chain_grid(n_chains, threads);
    return lr_launch_ordered(h, last, stream, [&](cudaStream_t st) { launch(blocks, threads, st); });
}

// The swap_step entry points (`prefix` lr_chains, lr_trend, lr_dd): one round for ladders that all live on this shard, on the
// handle's stream.  info(d_info) fills the (lik, beta) table of the shard in the workspace, apply(d_info) applies the round.
// rep_of_chain (host, may be null): a ladder whose members run on different replicates is refused -- its swaps would mix two
// posteriors.
template <class Info, class Apply>
int lr_swap_step(lr_handle_t h, int64_t chain_id0, int n_chains, int32_t ladder, const int* rep_of_chain, const char* prefix, Info info,
                 Apply apply) {
    LR_REQUIRE(ladder >= 2 && chain_id0 % ladder == 0 && n_chains % ladder == 0,
               "%s_swap_step: the shard must hold whole ladders (chain_id0 and n_chains multiples of the ladder size); "
               "use %s_swap_info + an all-gather + %s_swap_apply for ladders that span devices", prefix, prefix, prefix);
    if (rep_of_chain)
        for (int c = 0; c < n_chains; ++c)
            LR_REQUIRE(rep_of_chain[c] == rep_of_chain[c - c % ladder],
                       "%s_swap_step: the ladder of chain %lld runs on replicates %d and %d; swaps would mix two posteriors", prefix,
                       (long long)(chain_id0 + c), rep_of_chain[c - c % ladder], rep_of_chain[c]);
    int rc = lr_ws_acquire(h, (size_t)n_chains * 16, h->stream);
    if (rc != LR_OK) return rc;
    rc = info((double*)h->ws);
    if (rc != LR_OK) return rc;
    return apply((const double*)h->ws);
}

// lr_trend_set_beta_host / lr_dd_set_beta_host: every beta in [0, 1], staged through the workspace; set(d_beta, stream) launches
// the sampler's kernel.  Returns when the betas are in place.
template <class Set>
int lr_set_beta(lr_handle_t h, lr_last_stream* last, int n_chains, const double* h_beta, const char* who, Set set) {
    for (int c = 0; c < n_chains; ++c)
        LR_REQUIRE(h_beta[c] >= 0.0 && h_beta[c] <= 1.0, "%s: beta of chain %d = %g outside [0, 1]", who, c, h_beta[c]);
    LR_CUDA(cudaSetDevice(h->device));
    { int rc0 = lr_order(h, last, h->stream); if (rc0 != LR_OK) return rc0; }
    int rc = lr_ws_acquire(h, (size_t)n_chains * 8, h->stream);
    if (rc != LR_OK) return rc;
    LR_CUDA(cudaMemcpyAsync(h->ws, h_beta, (size_t)n_chains * 8, cudaMemcpyHostToDevice, h->stream));
    set((const double*)h->ws, h->stream);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    LR_CUDA(cudaStreamSynchronize(h->stream));
    return LR_OK;
}

// lr_trend_temper_host / lr_dd_temper_host: beta [n] and swaps proposed / accepted [n][2] of the chain states d_st (K6 TrendChain,
// K7 DDChain: fields beta and swaps); either output may be null
template <class Chain>
int lr_temper_host(lr_handle_t h, lr_last_stream* last, const Chain* d_st, int n_chains, double* h_beta, int64_t* h_swaps, const char* who) {
    LR_CUDA(cudaSetDevice(h->device));
    { int rc0 = lr_order(h, last, h->stream); if (rc0 != LR_OK) return rc0; }
    LR_CUDA(cudaStreamSynchronize(h->stream));
    Chain* tmp = new Chain[n_chains];
    cudaError_t e = cudaMemcpy(tmp, d_st, (size_t)n_chains * sizeof(Chain), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { delete[] tmp; lr_set_error("%s: %s", who, cudaGetErrorString(e)); return LR_ERR_CUDA; }
    for (int c = 0; c < n_chains; ++c) {
        if (h_beta) h_beta[c] = tmp[c].beta;
        if (h_swaps) { h_swaps[2 * c] = tmp[c].swaps[0]; h_swaps[2 * c + 1] = tmp[c].swaps[1]; }
    }
    delete[] tmp;
    return LR_OK;
}

// The *_create_host entry points of K6 / K7: the per-bin statistics sp, ex, br [cnt] from the host into the workspace, on the
// handle's stream
inline int lr_upload_bin_stats(lr_handle_t h, size_t cnt, const int64_t* h_sp, const int64_t* h_ex, const double* h_br, int64_t** d_sp,
                               int64_t** d_ex, double** d_br) {
    LR_CUDA(cudaSetDevice(h->device));
    int rc = lr_ws_acquire(h, cnt * 24, h->stream);
    if (rc != LR_OK) return rc;
    *d_sp = (int64_t*)h->ws;
    *d_ex = *d_sp + cnt;
    *d_br = (double*)(*d_ex + cnt);
    LR_CUDA(cudaMemcpyAsync(*d_sp, h_sp, cnt * 8, cudaMemcpyHostToDevice, h->stream));
    LR_CUDA(cudaMemcpyAsync(*d_ex, h_ex, cnt * 8, cudaMemcpyHostToDevice, h->stream));
    LR_CUDA(cudaMemcpyAsync(*d_br, h_br, cnt * 8, cudaMemcpyHostToDevice, h->stream));
    return LR_OK;
}

// ---- workspace layout ----------------------------------------------------------------------------------------------------------
inline size_t lr_align256(size_t x) { return (x + 255) & ~(size_t)255; }
// Buffers placed one after the other from `base`, each 256-byte aligned.  A null base only measures: every buffer is null and
// `used` ends as the bytes the same calls need from a real base, so one layout function both sizes a workspace and places it.
struct lr_carve {
    char* base;
    size_t used = 0;
    template <class T> T* take(size_t n) {
        T* p = base ? (T*)(base + used) : nullptr;
        used += lr_align256(n * sizeof(T));
        return p;
    }
};

// ---- record consumers (K8 lr_column_hpd, K9 lr_chain_diagnostics, K10 lr_rank_*) --------------------------------------------------
// order-preserving key of a double: negative values bit-inverted, the sign bit set on the others; every NaN -> the largest key
__device__ __forceinline__ unsigned long long lr_key(double x) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    if (x != x) return ~0ull;
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double lr_val(unsigned long long k) {
    return __longlong_as_double((long long)((k & 0x8000000000000000ull) ? (k ^ 0x8000000000000000ull) : ~k));
}
// Compensated (Neumaier) sum: the running sum s and the rounding errors c of its additions, so that a mean over millions of rows
// stays within a few units in the last place of the correctly rounded one (a plain sum in any order drifts by up to n ulp when the
// rounding errors share a sign, e.g. a column of the values 0.1, 0.2, 0.3).  A sum that became +-inf or NaN stays so and is
// returned as it is, as a plain sum would.
struct lr_sum {
    double s = 0.0, c = 0.0;
    __device__ __forceinline__ void add(double v) {
        const double t = __dadd_rn(s, v);
        c = __dadd_rn(c, fabs(s) >= fabs(v) ? __dadd_rn(__dsub_rn(s, t), v) : __dadd_rn(__dsub_rn(v, t), s));
        s = t;
    }
    __device__ __forceinline__ double value() const { return isfinite(s) ? __dadd_rn(s, c) : s; }
};

// Column specs.  Output column j of a row is row[a_j], then + or - row[b_j] (b_j >= 0, sign_j = +-1), then + add_j (if non-zero):
// one fp64 operation each, in this order -- what the logs hold (the net rate l_j - m_j, DDRate's midpoint_x0 and maxCarryingCap).
// (a default spec reads field 0: what a lane without a column of its group holds, whose values it never uses)
struct lr_col_spec {
    int a = 0, b = -1, s = 1;
    double c = 0.0;
    __device__ __forceinline__ double value(const double* row) const {
        double v = row[a];
        if (b >= 0) v = s > 0 ? __dadd_rn(v, row[b]) : __dsub_rn(v, row[b]);
        if (c != 0.0) v = __dadd_rn(v, c);
        return v;
    }
};
// the specs staged on the device: add [n] fp64, then a, b, sign [n] int32, one block in the workspace
struct lr_col_specs {
    int* a; int* b; int* sign; double* add;
    static lr_col_specs carve(lr_carve& w, int n_cols) {
        lr_col_specs s;
        s.add = w.take<double>(n_cols); s.a = w.take<int>(n_cols); s.b = w.take<int>(n_cols); s.sign = w.take<int>(n_cols);
        return s;
    }
    // the specs of a batch of columns from column c0
    lr_col_specs from(int c0) const { return {a + c0, b + c0, sign + c0, add + c0}; }
    __device__ __forceinline__ lr_col_spec load(int col) const { return {a[col], b[col], sign[col], add[col]}; }
};

// every field inside the row and every sign +-1 (b, sign and add may be NULL: -1, 1, 0)
inline int lr_check_col_specs(const char* who, int n_cols, int64_t row_stride, const int32_t* h_col_a, const int32_t* h_col_b,
                              const int32_t* h_col_sign) {
    for (int j = 0; j < n_cols; ++j) {
        const int a = h_col_a[j], b = h_col_b ? h_col_b[j] : -1, s = h_col_sign ? h_col_sign[j] : 1;
        LR_REQUIRE(a >= 0 && a < row_stride && b >= -1 && b < row_stride && (s == 1 || s == -1),
                   "%s: column %d = (%d, %d, %d) names a field outside the row of %lld doubles or a sign other than +-1", who, j, a, b, s,
                   (long long)row_stride);
    }
    return LR_OK;
}

// the specs, staged in one host block (defaults for the optional arrays) and copied to the block `spec` (device, carved by
// lr_col_specs::carve) in one piece on `st`; the copy is from pageable memory, so it has been staged when this returns
inline int lr_stage_col_specs(const char* who, const lr_col_specs& spec, int n_cols, const int32_t* h_col_a, const int32_t* h_col_b,
                              const int32_t* h_col_sign, const double* h_col_add, cudaStream_t st) {
    char* base = (char*)spec.add;
    const size_t bytes = (char*)(spec.sign + n_cols) - base;
    char* stage = (char*)calloc(1, bytes);
    LR_REQUIRE(stage, "%s: out of host memory", who);
    double* hc = (double*)stage;
    int* ha = (int*)(stage + ((char*)spec.a - base));
    int* hb = (int*)(stage + ((char*)spec.b - base));
    int* hs = (int*)(stage + ((char*)spec.sign - base));
    for (int j = 0; j < n_cols; ++j) {
        ha[j] = h_col_a[j]; hb[j] = h_col_b ? h_col_b[j] : -1; hs[j] = h_col_sign ? h_col_sign[j] : 1;
        hc[j] = h_col_add ? h_col_add[j] : 0.0;
    }
    const cudaError_t e = cudaMemcpyAsync(base, stage, bytes, cudaMemcpyHostToDevice, st);
    free(stage);
    LR_CUDA(e);
    return LR_OK;
}

// Rows of the chains of a run (K9, K10): row (s, k) is at rows + (s M T + k) stride -- [sample][chain][record], or a matrix
// [S M][bins] (T = 1).  With ladders (T > 1) logical chain c at sample s is the first of the rows (s, cT) .. (s, cT + T - 1) whose
// field beta_col holds 1.0 (the cold member of its ladder).
struct lr_chain_rows {
    const double* rows;
    long long S, M, stride;
    int T, beta_col;
};
// row of logical chain c at sample s; with ladders the cold member is found by the warp (lanes 0..T-1 test one member each) and
// *missing (if not null) says whether the ladder has none at this sample
__device__ __forceinline__ const double* lr_chain_row(const lr_chain_rows& r, long long s, long long c, int lane, bool* missing) {
    const double* base = r.rows + (s * r.M * r.T + c * r.T) * r.stride;
    if (r.T == 1) return base;
    const bool cold = lane < r.T && base[(long long)lane * r.stride + r.beta_col] == 1.0;
    const unsigned b = __ballot_sync(0xffffffffu, cold);
    if (missing) *missing = b == 0;
    return base + (long long)(b ? __ffs(b) - 1 : 0) * r.stride;
}

// the arguments of the entry points that read chain rows (lr_chain_diagnostics, lr_rank_transform, lr_rank_diagnostics); outs:
// every output pointer of the entry point is set
inline int lr_check_chain_rows(const char* who, lr_handle_t h, bool outs, const double* d_rows, int64_t n_samples, int64_t n_chains,
                               int32_t ladder, int32_t beta_col, int64_t row_stride, int32_t n_cols, const int32_t* h_col_a,
                               const int32_t* h_col_b, const int32_t* h_col_sign) {
    LR_REQUIRE(h && outs && h_col_a && d_rows, "%s: null pointer", who);
    LR_REQUIRE(n_samples >= 4, "%s: not enough data (%lld samples per chain; at least 4)", who, (long long)n_samples);
    LR_REQUIRE(n_chains >= 1 && ladder >= 1 && ladder <= 32 && n_cols >= 1 && row_stride >= 1,
               "%s: bad sizes (n_chains >= 1, ladder 1..32, n_cols >= 1, row_stride >= 1)", who);
    LR_REQUIRE(n_samples * n_chains * ladder < ((int64_t)1 << 31), "%s: %lld rows; at most 2^31 - 1", who,
               (long long)(n_samples * n_chains * ladder));
    LR_REQUIRE(ladder == 1 || (beta_col >= 0 && beta_col < row_stride), "%s: beta column %d outside the row of %lld doubles", who,
               beta_col, (long long)row_stride);
    return lr_check_col_specs(who, n_cols, row_stride, h_col_a, h_col_b, h_col_sign);
}

// ---- the likelihood's record-to-bin rate mapping of K3 records (K11, K12): segment k of a side starts at bin
// floor(t_k) - floor(start_time) (s0f), clamped to [0, nb]; bin j takes the last segment starting at or before it.
// lr_k3_stage stages the first bin of every segment of `side` in sjb[32] (the warp's) and returns K (0: the side is unusable --
// K outside 1..32, a non-finite shift time or segments out of order); a warp-wide call.
__device__ __forceinline__ int lr_k3_stage(int s0f, int nb, const double* row, int side, int lane, int* sjb) {
    __syncwarp();                                              // the previous record's searches are done with sjb
    const double kd = row[side ? 6 : 5];
    const int K = (kd >= 1.0 && kd <= 32.0 && kd == floor(kd)) ? (int)kd : 0;
    const double t = row[(side ? 112 : 48) + lane];
    bool ok = true;
    int jb = 0;
    if (lane > 0 && lane < K) {
        ok = isfinite(t);
        jb = ok ? (int)fmin(fmax(floor(t) - (double)s0f, 0.0), (double)nb) : 0;
    }
    sjb[lane] = jb;
    __syncwarp();
    if (lane > 0 && lane < K && jb < sjb[lane - 1]) ok = false;
    const bool all = __all_sync(0xffffffffu, ok);
    __syncwarp();
    return all ? K : 0;
}
// slot of bin j: the last k < K with sjb[k] <= j (sjb[0] = 0)
__device__ __forceinline__ int lr_k3_slot(const int* sjb, int K, int j) {
    int lo = 0, hi = K - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (sjb[mid] <= j) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// ---- K10's segmented LSD radix sort of 64-bit keys (k10_rank.cu) on a caller's buffers: segment s of length L sits at b0 + s L;
// its digit d is sorted only when some of its keys differ there (band / bor: the AND and OR of the segment's keys, bit d of
// lr_radix_passes), so the sorted segment ends in b0 or b1 as lr_radix_src(passes, 8) says.  ghist holds lr_k10_sort_ghist(L)
// words per segment.  Asynchronous on st.
__device__ __forceinline__ unsigned lr_radix_passes(unsigned long long a, unsigned long long o) {
    const unsigned long long d = a ^ o;
    unsigned m = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) m |= ((d >> (8 * q)) & 255ull) ? (1u << q) : 0u;
    return m;
}
// the buffer (0 / 1) that holds a segment before pass d, and after the last pass (d = 8)
__device__ __forceinline__ int lr_radix_src(unsigned passes, int d) { return __popc(passes & ((1u << d) - 1u)) & 1; }
size_t lr_k10_sort_ghist(int64_t L);
int lr_k10_sort(lr_handle_t h, unsigned long long* b0, unsigned long long* b1, int64_t L, int segs, const unsigned long long* band,
                const unsigned long long* bor, unsigned* ghist, cudaStream_t st);

// ---- K9's host driver on a caller's scratch (k9_diag.cu): lr_chain_diagnostics runs it on the workspace, K10 on the part of the
// workspace behind its own buffers.  lr_k9_scratch_bytes is what lr_k9_run uses from `w` (the staged specs and at most ~256 MB);
// the arguments are those of lr_chain_diagnostics, already checked, `who` names the entry point in errors.
size_t lr_k9_scratch_bytes(int64_t n_chains, int32_t n_cols);
int lr_k9_run(lr_handle_t h, char* w, const char* who, const double* d_rows, int64_t n_samples, int64_t n_chains, int32_t ladder,
              int32_t beta_col, int64_t row_stride, int32_t n_cols, const int32_t* h_col_a, const int32_t* h_col_b,
              const int32_t* h_col_sign, const double* h_col_add, double* d_out, int64_t* d_status, cudaStream_t st);

// ---- small device helpers --------------------------------------------------------------------
__device__ __forceinline__ double2 ld_stream_f64x2(const double2* p) {
    double2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ double ld_stream_f64(const double* p) {
    double v;
    asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// warp_sum of a value that is zero in every lane >= K (the slots a side does not use), K warp-uniform: the butterfly steps that
// would only add zeros are skipped -- the bits are those of warp_sum -- and lane 0's total is broadcast.  One shuffle for a
// single-rate side instead of five.
__device__ __forceinline__ double warp_sum_first(double v, int K) {
    if (K > 8) return warp_sum(v);
    if (K > 1) {
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    }
    return __shfl_sync(0xffffffffu, v, 0);
}
__device__ __forceinline__ double warp_prod(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v *= __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- Philox-4x32-10 (Salmon et al., SC'11); counter-based, one call = 128 random bits --------
struct Philox4 { uint32_t x, y, z, w; };
__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    Philox4 o; o.x = c0; o.y = c1; o.z = c2; o.w = c3;
    return o;
}
// uniform strictly inside (0,1) from 52 random bits: the bits become the mantissa of a double in [1,2) (no integer to
// floating-point conversion), shifted down by 1 and up by half a step: values (k + 1/2) 2^-52, k = 0 .. 2^52-1
__device__ __forceinline__ double u01(uint32_t hi, uint32_t lo) {
    const double x = __hiloint2double((int)(0x3ff00000u | (hi >> 12)), (int)((hi << 20) | (lo >> 12)));
    return (x - 1.0) + 1.1102230246251565e-16;
}

// ---- Poisson counts from a Philox stream (K11) -----------------------------------------------------------------------------------
// lr_poisson(mu) draws one Poisson(mu) count.  The draw takes Philox-4x32-10 blocks at counter (c0, c1, c2 | a << 25, c3) and key
// (k0, k1) for attempt a = 0, 1, .. (c2 must leave bits 25..31 clear); each block gives the uniforms U1 = u01(x, y), U2 = u01(z, w).
//   mu == 0          0, no draw
//   mu < 10          inversion by sequential search (attempt 0, U1): p = exp(-mu), F = p, k = 0; while U1 > F: k += 1, p = p mu / k,
//                    F = F + p.  More than LR_POIS_SEARCH steps exhaust the search.
//   10 <= mu         Hormann's PTRS (transformed rejection with squeeze, 1993), the algorithm and constants of numpy's
//                    random_poisson_ptrs: U = U1 - 1/2, V = U2 of attempt a; LR_POIS_ATTEMPTS attempts at most.
// Every operation is one IEEE double operation in the order written (no contraction), so a host restatement with the same
// exp / log / lgamma gives the same count; only those three functions can differ by a few ulp (literate_b200.predictive).
// Returns -1 for a mu outside [0, LR_POIS_MU_MAX] or NaN (no draw) and 0 with *exhausted incremented when the loop ran out.
#define LR_POIS_SEARCH 256
#define LR_POIS_ATTEMPTS 64
#define LR_POIS_MU_MAX 4503599627370496.0     // 2^52: every candidate count and k log(mu) stays exact in int64 / fp64
__device__ __forceinline__ long long lr_poisson(double mu, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                                unsigned* exhausted) {
    if (!(mu >= 0.0 && mu <= LR_POIS_MU_MAX)) return -1;
    if (mu == 0.0) return 0;
    if (mu < 10.0) {
        const Philox4 r = philox4x32_10(c0, c1, c2, c3, k0, k1);
        const double u = u01(r.x, r.y);
        double p = exp(-mu), F = p;
        long long k = 0;
        while (u > F) {
            if (k == LR_POIS_SEARCH) { ++*exhausted; return 0; }
            k += 1;
            p = __ddiv_rn(__dmul_rn(p, mu), (double)k);
            F = __dadd_rn(F, p);
        }
        return k;
    }
    const double slam = sqrt(mu), loglam = log(mu);
    const double b = __dadd_rn(0.931, __dmul_rn(2.53, slam));
    const double a = __dadd_rn(-0.059, __dmul_rn(0.02483, b));
    const double invalpha = __dadd_rn(1.1239, __ddiv_rn(1.1328, __dsub_rn(b, 3.4)));
    const double vr = __dsub_rn(0.9277, __ddiv_rn(3.6224, __dsub_rn(b, 2.0)));
    const double lia = log(invalpha);
    for (uint32_t att = 0; att < LR_POIS_ATTEMPTS; ++att) {
        const Philox4 r = philox4x32_10(c0, c1, c2 | (att << 25), c3, k0, k1);
        const double U = __dsub_rn(u01(r.x, r.y), 0.5), V = u01(r.z, r.w);
        const double us = __dsub_rn(0.5, fabs(U));
        const double kd = floor(__dadd_rn(__dadd_rn(__dmul_rn(__dadd_rn(__ddiv_rn(__dmul_rn(2.0, a), us), b), U), mu), 0.43));
        if (us >= 0.07 && V <= vr) return (long long)kd;
        if (kd < 0.0 || (us < 0.013 && V > us)) continue;
        const double lhs = __dsub_rn(__dadd_rn(log(V), lia), log(__dadd_rn(__ddiv_rn(a, __dmul_rn(us, us)), b)));
        const double rhs = __dsub_rn(__dadd_rn(-mu, __dmul_rn(kd, loglam)), lgamma(__dadd_rn(kd, 1.0)));
        if (lhs <= rhs) return (long long)kd;
    }
    ++*exhausted;
    return 0;
}

// exp(x) for |x| <= 0.1 (the log-multipliers of update_multiplier_proposal_vec: |2 log(1.1) (u - .5)| <= 0.0954): Taylor series to
// x^11, truncation error < 2e-21, i.e. rounding only.  The coefficients sit in constant memory: as literals every one costs
// two UMOV before its DFMA (17 extra instructions per call); from the constant bank two arrive per LDCU.128.
__constant__ double c_exp_small[12] = {2.505210838544172e-8 /* 1/11! */, 2.755731922398589e-7, 2.755731922398589e-6, 2.48015873015873e-5,
                                       1.984126984126984e-4, 1.388888888888889e-3, 8.333333333333333e-3, 4.166666666666666e-2,
                                       1.666666666666667e-1, 0.5, 1.0, 1.0};
__device__ __forceinline__ double exp_small(double x) {
    double p = c_exp_small[0];
#pragma unroll
    for (int k = 1; k < 12; ++k) p = fma(p, x, c_exp_small[k]);
    return p;
}

// Single-precision bracket [*lo, *hi] of the double log(u) of a uniform u in (0, 1) (error bound: __logf <= 2^-21.4 absolute on
// [.5, 2], 3 ulp elsewhere, plus the rounding of u to float).  The Metropolis-Hastings tests below evaluate the double-precision
// logarithm only when x falls inside it; their decision is always the one the exact comparison with log(u) gives.
__device__ __forceinline__ void mh_bracket(double u, double* lo, double* hi) {
    const float lf = __logf((float)u);
    const float err = 2e-6f * (1.0f + fabsf(lf));
    *hi = (double)(lf + err); *lo = (double)(lf - err);
}
// `x > log(u)` (K6, K7).  NaN and -inf are rejected.
__device__ __forceinline__ bool mh_accept_gt(double x, double u) {
    double lo, hi;
    mh_bracket(u, &lo, &hi);
    if (x > hi) return true;
    if (!(x >= lo)) return false;
    return x > log(u);
}
// `x >= log(u)` (K3) from the bracket [lo, hi] of mh_bracket, which K3 computes with its other draws; log_fn(u) is the
// double-precision logarithm (K3 passes its out-of-line one).  -inf is rejected by the bracket, NaN by the last comparison.
template <class Log>
__device__ __forceinline__ bool mh_accept_ge(double x, double u, double lo, double hi, Log log_fn) {
    if (x >= hi) return true;
    if (x < lo) return false;
    return x >= log_fn(u);
}

// standard normal from two uniforms in single precision (Box-Muller); a proposal step, not a likelihood term: 24 bits suffice
__device__ __forceinline__ double normal_f32(double u1, uint32_t bits) {
    const float r = sqrtf(-2.0f * __logf((float)u1));
    return (double)(r * cospif(((float)(bits >> 8) + 0.5f) * 1.1920929e-7f));     // angle 2 pi k / 2^24 as cospi(2 k / 2^24)
}

// ---- the swap rule of the tempered ladders (K3, K6, K7) ----------------------------------------------------------------------
// One swap round.  Chains are grouped into ladders of `ladder` consecutive GLOBAL chain ids; within a ladder the members are
// ordered by temperature and neighbours (2p + parity, 2p + 1 + parity) exchange their TEMPERATURES with probability
// min(1, exp((beta_i - beta_j)(lik_j - lik_i))).  Every rank holding a member of a ladder recomputes the whole ladder's decisions
// from the gathered (lik, beta) table and a Philox draw keyed by (seed, ladder, round, pair), so the outcome is identical
// everywhere and no state crosses the interconnect.  Only the likelihood is tempered, so lik is the untempered log-likelihood.
// Called by one warp for global chain g (table row of global chain m: m - table_first); one lane then calls
// write(paired, accept, beta_p) for that chain: paired = it has a partner this round, accept = the two exchange, beta_p = the
// partner's beta.  The sampler's write stores beta and its swap counters.
template <class Write>
__device__ __forceinline__ void lr_swap_round(const double* __restrict__ info_all, long long table_first, long long n_all, long long g,
                                              int ladder, unsigned long long round, uint32_t k0, uint32_t k1, int lane, Write write) {
    const long long lad = g / ladder;
    const int me = (int)(g - lad * ladder);
    const long long m = lad * ladder + lane;
    const bool on = lane < ladder && m >= table_first && m < table_first + n_all;
    const double lik = on ? info_all[2 * (m - table_first)] : 0.0;
    const double beta = on ? info_all[2 * (m - table_first) + 1] : -1.0;
    // rank by temperature: 0 = coldest (largest beta); ties broken by position
    int rank = 0;
    for (int k = 0; k < ladder; ++k) {
        const double bk = __shfl_sync(0xffffffffu, beta, k);
        if (bk > beta || (bk == beta && k < lane)) rank++;
    }
    const int parity = (int)(round & 1ull);
    const int q = rank - parity;
    int partner_rank = -1;
    if (on && q >= 0) {
        partner_rank = (q ^ 1) + parity;
        if (partner_rank >= ladder) partner_rank = -1;
    }
    int partner = -1;
    for (int k = 0; k < ladder; ++k) {
        const int rk = __shfl_sync(0xffffffffu, rank, k);
        const bool onk = __shfl_sync(0xffffffffu, (int)on, k) != 0;
        if (onk && rk == partner_rank) partner = k;
    }
    const double lik_p = __shfl_sync(0xffffffffu, lik, partner < 0 ? 0 : partner);
    const double beta_p = __shfl_sync(0xffffffffu, beta, partner < 0 ? 0 : partner);
    bool accept = false;
    if (partner >= 0) {
        const int pair = (rank < partner_rank ? rank : partner_rank);
        const Philox4 r = philox4x32_10((uint32_t)round, (uint32_t)(round >> 32), (uint32_t)pair | (0x5157u << 16), (uint32_t)lad, k0, k1 ^ 0x7e3a9u);
        const double u = u01(r.x, r.y);
        accept = log(u) <= (beta - beta_p) * (lik_p - lik);
    }
    if (lane == me) write(partner >= 0, accept, beta_p);
}
