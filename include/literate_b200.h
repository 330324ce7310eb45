/*
 * literate_b200 -- C ABI of the B200-native LiteRate RJMCMC birth-death hot path.
 *
 * The reference (dsilvestro/LiteRate) is a single Python script with no FFI seam; the three
 * seams below are the module-level functions of LiteRateForward.py that a maintainer would
 * rebind (INTEGRATION.md shows the ctypes stubs).  All file:line citations are relative to the
 * reference checkout.
 *
 *   L2  precompute_events()/get_br() loop        LiteRateForward.py:111-123, :514-549
 *         -> lr_bin_stats / lr_bin_stats_host / lr_bin_accumulate + lr_bin_finalize
 *   L3  calc_likelihood() + priors of runMCMC    LiteRateForward.py:137-162, :198-202, :296-306
 *         -> lr_dataset_create + lr_state_eval
 *   L4  runMCMC()                                LiteRateForward.py:216-373
 *         -> lr_chains_create / lr_chains_run / lr_chains_get_state / lr_chains_destroy
 *   and, on the same statistics, the loops of the two sibling fixed-dimension samplers (SURVEY 8 f-4):
 *       trend_rate.py:102-196 -> lr_trend_*          DDRatev3.py:242-292 -> lr_dd_*
 *
 * Conventions
 *   - plain C, no torch / CUDA types in signatures; `stream` is a cudaStream_t passed as void*
 *     (NULL = the handle's own stream).
 *   - pointers named d_* are DEVICE pointers owned by the caller; h_* are HOST pointers.
 *   - every function returns LR_OK (0) or a negative lr_status; lr_last_error() returns the
 *     message of the last failure on the calling thread.  Nothing throws, nothing falls back
 *     to a CPU implementation.
 *   - device-pointer entry points are asynchronous on `stream`; *_host entry points are
 *     synchronous (they copy host->device, run, copy device->host and wait).
 *   - one handle per (device, host thread); a handle is not thread-safe, distinct handles are.
 */
#ifndef LITERATE_B200_H
#define LITERATE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LR_ABI_VERSION 1

typedef enum lr_status {
    LR_OK = 0,
    LR_ERR_INVALID = -1,      /* bad argument */
    LR_ERR_CUDA = -2,         /* CUDA runtime error, see lr_last_error() */
    LR_ERR_UNSUPPORTED = -3,  /* size outside what the kernels implement */
    LR_ERR_NOMEM = -4
} lr_status;

typedef struct lr_handle_s*  lr_handle_t;   /* one per device */
typedef struct lr_dataset_s* lr_dataset_t;  /* per-replicate binned statistics + prefix tables, on device */
typedef struct lr_chains_s*  lr_chains_t;   /* a population of independent chains, on device */

/* ---------------------------------------------------------------- runtime */
int lr_abi_version(void);
const char* lr_last_error(void);
int lr_create(int device, lr_handle_t* out);
int lr_destroy(lr_handle_t h);
/* number of SMs, kernels launched through this handle so far, device id */
int lr_info(lr_handle_t h, int32_t* sm_count, int64_t* kernel_launches, int32_t* device);
int lr_sync(lr_handle_t h);

/* ---------------------------------------------------------------- L2: lineages -> per-bin statistics
 *
 * Replaces the loop `for i in range(int(min ts), int(max te)): precompute_events([i, i+1])`
 * (LiteRateForward.py:519-523) and its extinct-only twin (:529-549).
 *
 *   ts, te     [n_rep][ld] fp64, ld >= n; replicate r occupies ts[r*ld .. r*ld+n)
 *   first_bin  int(min ts); bin j is [first_bin+j, first_bin+j+1]
 *   n_bins     int(max te) - int(min ts)
 *   fe_ref     expected fractional part of te above its bin edge, in (0, 1]
 *              (0.5 for integer years with the default -death_jitter .5; 1.0 for integer te).
 *              It only selects the fast path; any value gives the same result.
 *   dead_only  1: keep only lineages with te < end_time (:531-532), else 0
 *   sp, ex     int64 [n_rep][n_bins]  births  ts in [t0,t1), deaths te in (t0,t1]   (:120-121)
 *   br         fp64  [n_rep][n_bins]  sum_i max(0, min(te_i,t1) - max(ts_i,t0))      (:111-116)
 *
 * Counts are exact (from the raw doubles).  br is the correctly rounded exact sum of the clipped lifetimes, with every
 * endpoint on the 2^-52 grid: fractions are accumulated in 2^-52 fixed point, a birth as
 * floor(ts) + rint((ts - floor(ts)) * 2^52) / 2^52 and a death as c + rint((te - c) * 2^52) / 2^52, c = ceil(te) - 1, both
 * differences taken in fp64 (ties to even).  For |t| >= 1 that is the time itself (the difference is exact and on the grid),
 * so br is the exact sum there; times in (-1, 1) are first rounded to the grid.  Hence bit-identical to the reference for
 * dyadic data and run-to-run deterministic for any data (oracle/k1_exact.py restates this definition).
 */
#define LR_ACC_ROWS 8
/* row stride (in int64) of the raw accumulator block of one replicate */
int64_t lr_acc_stride(int32_t n_bins);
/* raw accumulators: int64 [n_rep][LR_ACC_ROWS][lr_acc_stride(n_bins)], must be zeroed by the caller.
 * Rows: 0 births, 1 deaths, 2/3 low-32/high parts of sum frac(ts)*2^52, 4/5 low-32/high parts of
 * sum (fe-fe_ref)*2^52, 6/7 births/deaths of lineages that carry no time at risk (te<=ts);
 * [6][n_bins] counts lineages alive before bin 0.
 * All rows are plain integer sums, so lineage shards combine with an int64 SUM all-reduce. */
int lr_bin_accumulate(lr_handle_t h, const double* d_ts, const double* d_te, int64_t n, int64_t ld,
                      int32_t n_rep, int64_t first_bin, int32_t n_bins, double fe_ref,
                      int32_t dead_only, double end_time, int64_t* d_acc, void* stream);
/* Two builds of the pass produce these accumulators -- the same integer sums, hence the same finalized statistics bit for bit
 * (how a 96-bit sum is split over its row pair depends on where a pass flushed): the general one (any n_bins; the only one the
 * host-buffer entry points use: they are bound by the host link and run beside the chain kernels), and the lane-private one
 * (fraction words once per lane in shared memory, one CTA of 1024 threads per SM): every table of at least 250 000 lineages per
 * replicate up to 310 bins -- 1.05 of the copy bandwidth against 1.02 on integer years and against 0.74 on real-valued times --
 * and real-valued tables of at least 50 000 lineages per replicate up to 439 bins.
 * The pass itself records which kind of table it saw (its first 32 lineages) and the NEXT lr_bin_accumulate
 * through the handle uses that to choose -- no synchronisation, a stale answer costs speed only.  lr_bin_table_hint reads the
 * record (1 = fractional times, 0 = integer years) as of the last finished pass, lr_bin_last_build which build the last call
 * launched (0 general, 1 lane-private); the environment variable LR_K1_LANES=0 / 1 forces the choice. */
int lr_bin_table_hint(lr_handle_t h, int32_t* out);
int lr_bin_last_build(lr_handle_t h, int32_t* out);
int lr_bin_finalize(lr_handle_t h, const int64_t* d_acc, int32_t n_rep, int32_t n_bins, double fe_ref,
                    int64_t* d_sp, int64_t* d_ex, double* d_br, void* stream);
/* zero + accumulate + finalize using the handle's workspace */
int lr_bin_stats(lr_handle_t h, const double* d_ts, const double* d_te, int64_t n, int64_t ld,
                 int32_t n_rep, int64_t first_bin, int32_t n_bins, double fe_ref,
                 int32_t dead_only, double end_time,
                 int64_t* d_sp, int64_t* d_ex, double* d_br, void* stream);
/* same with host buffers; copies are pipelined per replicate against the kernel */
int lr_bin_stats_host(lr_handle_t h, const double* h_ts, const double* h_te, int64_t n, int64_t ld,
                      int32_t n_rep, int64_t first_bin, int32_t n_bins, double fe_ref,
                      int32_t dead_only, double end_time,
                      int64_t* h_sp, int64_t* h_ex, double* h_br);

/* The same pass for tables of INTEGER YEARS held as int32 (8 bytes per lineage instead of 16 -- every table the
 * reference ships is of this kind once parsed, LiteRateForward.py:440-451): ts = year, te = year + death_jitter (:471),
 * i.e. what the fp64 entry points see after `te = te + death_jitter`.  Every regular death is counted with the fraction
 * death_jitter itself, which is what fl(year + death_jitter) leaves for every |year| < 2^31 only when death_jitter is a
 * multiple of 2^-22 in [0, 1] (0, 0.25, 0.5, 1; not 0.1 or 1e-14): other jitters are refused (LR_ERR_INVALID) -- bin
 * those tables through the fp64 entry points.  Same accumulators, bit for bit; finalize them with
 * fe_ref = lr_fe_ref_of_jitter(death_jitter).  Pad ragged replicates with INT32_MIN in both columns (a lineage that ends
 * before the window: no contribution). */
int lr_bin_accumulate_i32(lr_handle_t h, const int32_t* d_ts, const int32_t* d_te, int64_t n, int64_t ld,
                          int32_t n_rep, int64_t first_bin, int32_t n_bins, double death_jitter,
                          int32_t dead_only, double end_time, int64_t* d_acc, void* stream);
double lr_fe_ref_of_jitter(double death_jitter);
/* host buffers (pinned for asynchronous copies), copies pipelined per batch of replicates against the kernel */
int lr_bin_stats_host_i32(lr_handle_t h, const int32_t* h_ts, const int32_t* h_te, int64_t n, int64_t ld,
                          int32_t n_rep, int64_t first_bin, int32_t n_bins, double death_jitter,
                          int32_t dead_only, double end_time,
                          int64_t* h_sp, int64_t* h_ex, double* h_br);

/* ---------------------------------------------------------------- L3: likelihood + priors on a state
 *
 * A dataset holds, per replicate, the binned statistics and the prefix tables the likelihood of a
 * piecewise-constant state needs (globals sp_events_bin / ex_events_bin / br_length_bin [/ *_dead]
 * of LiteRateForward.py:566-574).  model_BDI as the reference's -model_BDI (0 BD, 1 ID, 2 Keiding,
 * 3 Keiding extinct-only; :421-431).  d_ex_dead/d_br_dead may be NULL unless model_BDI == 3.
 */
int lr_dataset_create(lr_handle_t h, int32_t n_rep, int32_t n_bins, int32_t model_BDI,
                      double start_time, double end_time,
                      const int64_t* d_sp, const int64_t* d_ex, const double* d_br,
                      const int64_t* d_ex_dead, const double* d_br_dead,
                      void* stream, lr_dataset_t* out);
int lr_dataset_create_host(lr_handle_t h, int32_t n_rep, int32_t n_bins, int32_t model_BDI,
                           double start_time, double end_time,
                           const int64_t* h_sp, const int64_t* h_ex, const double* h_br,
                           const int64_t* h_ex_dead, const double* h_br_dead, lr_dataset_t* out);
/* The general form behind the four -model_BDI tables: per bin and side an event weight A_j and an exposure B_j,
 *     likelihood = C + sum_j [A_birth_j log(lambda_j) - B_birth_j lambda_j] + sum_j [A_death_j log(mu_j) - B_death_j mu_j]
 * with lambda_j / mu_j the rate of the segment bin j falls in.  HOST arrays [n_rep][n_bins] (h_C [n_rep] or NULL = 0);
 * x_birth / x_death are the per-bin vectors calculate_r_squared regresses the rates on (literate_library.py:268-279).
 * Replaces the `-proportion 1` likelihood of LiteRateForward-proportion.py:157-162 (A = interpolated yearly counts of a
 * series where its running total is positive, B = that mask, x = the counts, :585-598, :627-628); model_tag is what
 * lr_chain_config.model_BDI must then be (1 there, :442-444). */
int lr_dataset_create_general_host(lr_handle_t h, int32_t n_rep, int32_t n_bins, int32_t model_tag, double start_time, double end_time,
                                   const double* h_A_birth, const double* h_B_birth, const double* h_A_death, const double* h_B_death,
                                   const double* h_x_birth, const double* h_x_death, const double* h_C, lr_dataset_t* out);
int lr_dataset_destroy(lr_dataset_t ds);

#define LR_KMAX 30   /* most rates per side a state can hold (slots of one warp minus two control lanes) */

/* Batched evaluation of states, HOST buffers (parity/diagnostic entry point).
 *   rep[n]                replicate of each state
 *   K_l[n], K_m[n]        number of birth / death rates (1..LR_KMAX)
 *   L, M       [n][LR_KMAX]  rates
 *   tL, tM     [n][LR_KMAX]  slot 0 ignored (= start_time), slots 1..K-1 interior shift times, ascending
 *   gamma_rate [n][2], poi_lambda[n]   hyper-parameters (Gamma_rate, Poi_lambda_rjHP of :220-222)
 * Outputs (any may be NULL):
 *   lik[n]         calc_likelihood(L[indL], M[indM])            (:306, :137-162)
 *   prior_rates[n] prior_gamma(L)+prior_gamma(M) + time prior   (:296-298)
 *   prior_poi[n]   Poisson_prior(K_l)+Poisson_prior(K_m)        (:279)
 *   adequacy[n][3] calculate_r_squared                           (literate_library.py:268-279)
 */
int lr_state_eval_host(lr_dataset_t ds, int32_t n, const int32_t* rep, const int32_t* K_l, const int32_t* K_m,
                       const double* L, const double* M, const double* tL, const double* tM,
                       const double* gamma_rate, const double* poi_lambda,
                       double* lik, double* prior_rates, double* prior_poi, double* adequacy);

/* One reversible-jump proposal per explicit state with EXPLICIT draws, HOST buffers (parity entry point for the proposal
 * arithmetic of add_shift_RJ_weighted_mean / remove_shift_RJ_weighted_mean, LiteRateForward.py:29-69, and the acceptance
 * ratio of :296-313).  State arrays as lr_state_eval_host; additionally per state
 *   beta (NULL: 1), poiA   inverse temperature and the stored (possibly stale) Poisson prior term priorPoiA (:300-304)
 *   side                   1 birth side, 0 death side
 *   kind, idx              0 rate multiplier (update_multiplier_freq, :165-176); 2 add-shift inside segment idx (0-based);
 *                          3 remove interior shift idx (1..K-1)
 *   u_t, u_beta            add-shift: position inside the segment as a fraction, Beta(10,10) variate
 *   mult_on, mult_u        kind 0: [n][LR_KMAX] Bernoulli mask and uniforms of the multipliers (may be NULL otherwise)
 * Outputs: ok (0 = rejected by the spacing guard :290 or at capacity), K_new, rates_new / times_new [n][LR_KMAX] of the proposed
 * side, hasting = log q-ratio + log Jacobian (:47, :69), x = beta (lik' - lik) + (prior' - prior) + hasting with the new
 * Poisson prior term against poiA (:279, :313). */
int lr_proposal_eval_host(lr_dataset_t ds, int32_t n, const int32_t* rep, const int32_t* K_l, const int32_t* K_m,
                          const double* L, const double* M, const double* tL, const double* tM,
                          const double* gamma_rate, const double* poi_lambda, const double* beta, const double* poiA,
                          const int32_t* side, const int32_t* kind, const int32_t* idx, const double* u_t, const double* u_beta,
                          const int32_t* mult_on, const double* mult_u,
                          int32_t* ok, int32_t* K_new, double* rates_new, double* times_new, double* hasting, double* x);

/* Validation path: the Keiding log-likelihood (BD_lik_Keiding, :137-148; -model_BDI 2) of n_states states evaluated DIRECTLY
 * over the lineages without binning -- the per-lineage formulation of the reference's ancestor
 * (other/LiteRateBDI_ext.py:124-160, get_BDlik) -- to cross-check lr_bin_stats + lr_state_eval at full size.
 *   d_lam, d_mu  [n_states][n_bins] per-bin rates (a state expanded with get_rate_index, :125-135)
 *   d_out        [n_states]
 * Reads the lineages once per group of 8 states (16 B per lineage per group); deterministic; asynchronous on `stream`. */
int lr_loglik_direct(lr_handle_t h, const double* d_ts, const double* d_te, int64_t n, int64_t first_bin, int32_t n_bins,
                     const double* d_lam, const double* d_mu, int32_t n_states, double* d_out, void* stream);

/* ---------------------------------------------------------------- L4: the chains (runMCMC) */
typedef struct lr_chain_config {
    int32_t model_BDI;          /* must equal the dataset's */
    int32_t const_rates;        /* -const_rates        (:274, :386) */
    int32_t const_death_rate;   /* -const_death_rate   (:243-247, :387) */
    int32_t use_rate_HP;        /* -use_rate_HP        (:285, :395) */
    double  poisson_prior;      /* -Poisson_prior, 0 = sample the hyper-prior (:220-221, :283, :396) */
    double  update_fraction;    /* -update_fraction    (:252, :399) */
    int32_t real_move_shift;    /* 0 = reference behaviour (move-shift proposes the current state, :184-185);
                                   1 = reflected sliding window d=1 (opt-in, deviates from the reference) */
    int32_t loop_variant;       /* build of the chain loop: 0 choose by population size (4 up to four chains per SM, 3 up to
                                   seven, else 2); 1 warp-specialised, one chain per CTA (a chain warp fed by three producer
                                   warps); 3 warp-specialised, four chains per CTA (one producer each, registers re-balanced
                                   with setmaxnreg); 2 compact (one warp per chain, thousands of resident chains);
                                   4 speculative teams (16 / 8 / 4 warps evaluate consecutive iterations of ONE chain ahead
                                   of time, the first state change commits and the others roll back selectively) with a
                                   continuation pass of build 1 / 3 for chains whose state changes more than once in eight
                                   iterations (small tables, burn-in).  Results are identical, bit for bit */
    double  beta;               /* likelihood tempering exponent of every chain unless set per chain; 1 = reference */
} lr_chain_config;

/* Creates n_chains chains; chain c uses replicate rep_of_chain[c] (NULL: all use replicate 0) and the
 * Philox-4x32-10 stream keyed by (seed, chain_id0 + c), so results do not depend on how chains are
 * sharded over devices.  Initial state as :580-583 (rates ~ Gamma(2, scale 2), no shifts) with the
 * initial prior of :227-230. */
int lr_chains_create(lr_handle_t h, lr_dataset_t ds, int32_t n_chains, const lr_chain_config* cfg,
                     uint64_t seed, int64_t chain_id0, const int32_t* h_rep_of_chain, lr_chains_t* out);
int lr_chains_destroy(lr_chains_t c);

/* One sample record = LR_REC_DOUBLES doubles:
 *   [0] iteration  [1] likA  [2] priorA  [3] mean(L)  [4] mean(M)  [5] K_l  [6] K_m
 *   [7] Gamma_rate[0]  [8] Gamma_rate[1]  [9] Poi_lambda  [10..12] adequacy (coeff, r2, gelman_r2)
 *   [13] poi_lambda_is_initial (1 while Poi_lambda_rjHP still is the constant of :220-221)
 *   [14] beta (inverse temperature of the chain when the record was written; 1 = the reference's chain)
 *   [15] priorPoiA: the Poisson-prior term inside [2], refreshed only by accepted RJ proposals (:279, :300-304, :319)
 *   [16 .. 16+32)  L slots   [48 .. 80) birth shift times (slot 0 = start_time)
 *   [80 .. 112)    M slots   [112 .. 144) death shift times
 */
#define LR_REC_DOUBLES 144
/* Runs n_iter iterations of every chain, continuing from the current iteration counter `it`.
 * A record is written after every iteration with it % sample_every == 0 (as :321), i.e.
 * ceil-count of multiples of sample_every in [it0, it0+n_iter).  d_records must hold
 * lr_chains_records_per_run() * n_chains records, laid out [sample][chain][LR_REC_DOUBLES].
 * Asynchronous on `stream`. */
/* (host-side arithmetic on the iteration counter the library tracks: does NOT wait for launches in flight) */
int64_t lr_chains_records_per_run(lr_chains_t c, int64_t n_iter, int64_t sample_every);
int lr_chains_run(lr_chains_t c, int64_t n_iter, int64_t sample_every, double* d_records, void* stream);
/* same, records delivered to host memory; synchronous */
int lr_chains_run_host(lr_chains_t c, int64_t n_iter, int64_t sample_every, double* h_records);
/* per-chain counters since creation: [n_chains][LR_NCOUNTERS] int64 =
 *   iterations, accepted, likelihood evaluations, rate-updates, move-shifts, RJ proposals,
 *   Gibbs draws, capacity rejections (add-shift at K == LR_KMAX), temperature swaps proposed, swaps accepted */
#define LR_NCOUNTERS 10
int lr_chains_counters_host(lr_chains_t c, int64_t* h_counters);
/* diagnostics of the speculative team build (loop_variant 4), per chain since creation: [n_chains][6] int64 =
 *   state versions committed, evaluations dropped by rollbacks, polls while waiting to become the frontier,
 *   polls at the lead limit, iterations done by teams, hand-overs to the continuation pass.
 *   Zero for the other builds.  No reference counterpart. */
int lr_chains_team_stats_host(lr_chains_t c, int64_t* h_stats);
/* current state of every chain as one record each (iteration = number of iterations done) */
int lr_chains_get_state_host(lr_chains_t c, double* h_records);
/* overwrite the state of every chain from records (fields 1,2 and 10-12 are recomputed) */
int lr_chains_set_state_host(lr_chains_t c, const double* h_records);

/* ---------------------------------------------------------------- tempered ensembles (Metropolis-coupled MCMC)
 * New; the reference has no tempering.  A chain with beta = 1 is the reference's chain; a heated chain raises the
 * likelihood to the power beta < 1.  Chains are grouped into ladders of `ladder` consecutive GLOBAL chain ids; a swap
 * round exchanges TEMPERATURES (not states) between temperature neighbours of a ladder with the usual MC3 rule.
 */
/* per-chain inverse temperatures */
int lr_chains_set_beta_host(lr_chains_t c, const double* h_beta);
/* d_info[n_chains][2] = (likelihood, beta) of every chain: the 16 bytes per chain a swap round exchanges; async on `stream` */
int lr_chains_swap_info(lr_chains_t c, double* d_info, void* stream);
/* apply swap round `round` to this shard (global chain ids [first, first + n_chains)) given the gathered table
 * d_info_all[n_all][2] of the whole ensemble (an all-gather of every rank's lr_chains_swap_info when ladders span
 * devices; the shard's own table when they do not).  Even rounds pair temperature ranks (0,1)(2,3).., odd rounds (1,2)(3,4)..;
 * the decision of a pair is a Philox draw keyed by (seed, ladder, round, pair), identical on every rank.  Async on `stream`. */
int lr_chains_swap_apply(lr_chains_t c, const double* d_info_all, int64_t n_all, int64_t first, int32_t ladder,
                         uint64_t round, void* stream);
/* single-device convenience: swap_info + swap_apply on the handle's stream for ladders that live on this device */
int lr_chains_swap_step(lr_chains_t c, int32_t ladder, uint64_t round);

/* ---------------------------------------------------------------- posterior accumulators (SURVEY 8 f-1)
 * From device-resident sample records (any [n_records][LR_REC_DOUBLES] slice, e.g. the cold chains after the burn-in) the
 * sums behind plotRJforward.v3.py's per-bin summaries (get_marginal_rates :92-139, get_r_plot :166-176, get_K_values :292-305):
 *   d_sum_rate    [2][n_bins] fp64   sum over records of the marginal birth / death rate of every unit bin from first_edge
 *                                     (np.histogram semantics: half-open bins, last one closed); mean = sum / n_records
 *   d_shift_count [2][n_bins] int64  number of sampled shift times per bin (frequency = count / n_records)
 *   d_k_count     [2][32]     int64  number of records with K = index + 1 rates
 * Deterministic (fixed summation order); asynchronous on `stream`. */
int lr_summarize_records(lr_handle_t h, const double* d_records, int64_t n_records, double first_edge, int32_t n_bins,
                         double* d_sum_rate, int64_t* d_shift_count, int64_t* d_k_count, void* stream);
/* Envelopes over imputation replicates (utilities/imputation_averager.py:23-61): per bin, mean / min / max over the n_rep
 * replicates of ex/br, sp/br and br, from the outputs of lr_bin_stats (device pointers).  d_out [9][n_bins] =
 * death mean, min, max; birth mean, min, max; diversity mean, min, max.  Means accumulate in replicate order (numpy's
 * mean(axis=0) over the stacked div.log tables); min / max propagate NaN like numpy.  Asynchronous on `stream`. */
int lr_imputation_envelope(lr_handle_t h, const int64_t* d_sp, const int64_t* d_ex, const double* d_br, int32_t n_rep, int32_t n_bins,
                           double* d_out, void* stream);
/* The per-sample matrix behind the 95 % HPD intervals (get_marginal_rates :92-139, calcHPD :12-28): the marginal birth and death
 * rate of every record in the unit bins [bin_lo, bin_lo + bin_cnt) of the n_bins from first_edge, record-major:
 *   d_birth, d_death  [n_records][bin_cnt] fp64
 * (sort the columns and take the narrowest window holding 95 % of the rows: literate_b200.summary.hpd_device does it with
 * torch.sort on the device, a bin range at a time so that the matrix of a large ensemble need not exist as a whole). */
int lr_marginal_rates(lr_handle_t h, const double* d_records, int64_t n_records, double first_edge, int32_t n_bins,
                      int32_t bin_lo, int32_t bin_cnt, double* d_birth, double* d_death, void* stream);
/* K8: per-column means and exact HPD intervals of a row-major fp64 matrix d_rows[n_rows][row_stride] on the device -- the sample
 * records of any sampler (after the burn-in rows) or the matrices of lr_marginal_rates -- without copying it.
 *   mask_col     < 0: every row counts; otherwise only rows with row[mask_col] == 1.0 (the cold members of tempered ladders:
 *                the beta field of the records, e.g. 15 for TrendRate, 21 for DDRate)
 *   column j     value = row[h_col_a[j]], then + row[b] (h_col_sign[j] = 1) or - row[b] (-1) if b = h_col_b[j] >= 0, then
 *                + h_col_add[j] if that is non-zero: one fp64 operation each, in this order (the log's net rate l_j - m_j, DDRate's
 *                maxCarryingCap L + div_0 and midpoint_x0 x0 + origin).  HOST arrays [n_cols]; b, sign and add may be NULL (-1, 1, 0).
 *   level        in (0, 1]
 * Outputs [n_cols] fp64: d_mean (compensated sums in a fixed order: within a few ulp of the correctly rounded mean, and repeated calls are
 * bit-identical) and the HPD bounds d_lo, d_hi under
 * calcHPD (plotRJforward.v3.py:12-28): n_in = rint(level n), widths x[i + n_in - 1] - x[i] over the sorted column, the first
 * minimum wins; NaN sorts last as in np.sort and a NaN width wins as in np.argmin; +-inf are ordered normally.  The bounds equal
 * a host sort's bit for bit up to the sign of a zero.  d_n (int64 [1], may be NULL): the number of rows used.  When
 * rint(level n) < 2 every output column is NaN.  Scratch (at most ~512 MB of tails at a time) comes from the handle's workspace;
 * rejects bad sizes and column indices; asynchronous on `stream` (the column specs are staged before it returns). */
int lr_column_hpd(lr_handle_t h, const double* d_rows, int64_t n_rows, int64_t row_stride, int32_t mask_col, int32_t n_cols,
                  const int32_t* h_col_a, const int32_t* h_col_b, const int32_t* h_col_sign, const double* h_col_add,
                  double level, double* d_mean, double* d_lo, double* d_hi, int64_t* d_n, void* stream);
/* K9: split R-hat and "mean" effective sample size (Vehtari et al. 2021, section 3; Stan's and ArviZ's rhat(method="split") and
 * ess(method="mean")) of every column over the chains of a run, without copying the records.
 *   rows         row (s, k) at d_rows + (s n_chains ladder + k) row_stride: [sample][chain][record] for the records of K3 / K6 / K7,
 *                [n_samples n_chains][bins] for the matrices of lr_marginal_rates (ladder 1).  Burn-in: offset the pointer.
 *   ladder       1..32; T > 1: logical chain c at sample s is the first of the rows (s, cT .. cT + T - 1) with row[beta_col] == 1.0
 *   columns      the specs of lr_column_hpd (HOST arrays [n_cols]; b, sign, add may be NULL)
 * Split chains: n = floor(n_samples / 2), split chain 2c = draws [0, n) of chain c, 2c + 1 = draws [n_samples - n, n_samples) (an
 * odd n_samples drops the middle draw).  A split chain whose draws are all equal has that value as its mean, exactly; the
 * between-chain variance is exactly 0 when all split-chain means are equal.  Otherwise literate_b200.diagnostics.rhat_ess is the
 * definition, step for step: W, var+, rho_t, Geyer's initial positive and monotone sequences, tau >= 1/log10(m n).
 *   d_out        fp64 [5][n_cols]: mean (of the draws used), sd = sqrt(var+), R-hat, ESS, lag (Geyer's max_t, as a double)
 *   degenerate   a non-finite draw: every output NaN, lag -1; W = 0, var+ = 0 (constant): R-hat NaN, ESS NaN, lag -1;
 *                W = 0, var+ > 0 (every split chain stuck on its own value): R-hat +inf, ESS NaN, lag -1
 *   d_status     int64 [1]: (sample, ladder) pairs among the draws used with no member at beta = 1 (0 when ladder = 1)
 * Sums are compensated and in a fixed order: repeated calls are bit-identical.  The work follows the largest truncation lag
 * (lag blocks of doubling width, the count of unfinished columns read once per block), so the call returns when the outputs are
 * written.  Scratch (at most ~256 MB; columns in batches) comes from the handle's workspace.  Rejects bad sizes, fields outside
 * the row, n_samples < 4 ("not enough data") and more than 2^31 - 1 rows. */
int lr_chain_diagnostics(lr_handle_t h, const double* d_rows, int64_t n_samples, int64_t n_chains, int32_t ladder, int32_t beta_col,
                         int64_t row_stride, int32_t n_cols, const int32_t* h_col_a, const int32_t* h_col_b,
                         const int32_t* h_col_sign, const double* h_col_add, double* d_out, int64_t* d_status, void* stream);
/* K10: rank-normalised split R-hat and bulk and tail effective sample sizes (Vehtari et al. 2021; ArviZ's rhat(method="rank"),
 * ess(method="bulk"), ess(method="tail")) of every column over the chains of a run, without copying the records.  Rows, ladder,
 * columns, d_status and the split of lr_chain_diagnostics; n = floor(n_samples / 2), N = 2 n n_chains split draws per column.
 * literate_b200.diagnostics.rank_rhat_ess is the definition.
 * lr_rank_transform writes
 *   d_z          fp64 [2n][n_chains][4 n_cols]: row i n_chains + c holds split draw i of chain c (i >= n: draw n_samples - 2n + i);
 *                slot q n_cols + j of column j: q = 0 z = Phi^-1((r - 3/8) / (N + 1/4)) of the draw's average rank r (1-based)
 *                among the N split draws, q = 1 the same of |x - median|, q = 2 / 3 the indicator x <= q05 / x <= q95 (0.0 / 1.0)
 *   d_quant      fp64 [3][n_cols]: median of the split draws (np.median), q05 and q95 of all n_samples n_chains draws
 *                (np.quantile, method "linear"), bit for bit as numpy computes them up to the sign of a zero (NaN if a NaN is among them)
 * lr_rank_diagnostics writes d_out fp64 [8][n_cols]: median, q05, q95, rhat_bulk, rhat_tail, rhat_rank, ess_bulk, ess_tail; every
 * output NaN for a column lr_chain_diagnostics finds non-finite, constant or stuck.  Ties get their average rank; -0 ranks as +0.
 * Scratch comes from the handle's workspace: at most ~1 GiB of K10 buffers (columns in batches, at least one column per batch)
 * plus lr_chain_diagnostics' own.  Repeated calls are bit-identical.  lr_rank_transform is asynchronous on `stream`;
 * lr_rank_diagnostics returns when its outputs are written.  Rejects what lr_chain_diagnostics rejects, under its own name. */
int lr_rank_transform(lr_handle_t h, const double* d_rows, int64_t n_samples, int64_t n_chains, int32_t ladder, int32_t beta_col,
                      int64_t row_stride, int32_t n_cols, const int32_t* h_col_a, const int32_t* h_col_b, const int32_t* h_col_sign,
                      const double* h_col_add, double* d_z, double* d_quant, int64_t* d_status, void* stream);
int lr_rank_diagnostics(lr_handle_t h, const double* d_rows, int64_t n_samples, int64_t n_chains, int32_t ladder, int32_t beta_col,
                        int64_t row_stride, int32_t n_cols, const int32_t* h_col_a, const int32_t* h_col_b, const int32_t* h_col_sign,
                        const double* h_col_add, double* d_out, int64_t* d_status, void* stream);

/* ---------------------------------------------------------------- TrendRate (SURVEY 8 f-4): fixed-dimension chains on the same statistics
 *
 * Replaces the Metropolis-Hastings loop of trend_rate.py:102-196 (likelihood_function :73-91, calc_prior :93-100) and the
 * literate_library.py functions it calls (update_normal_nobound_vec :140-146, update_multiplier_proposal_vec :156-165,
 * prior_gamma/prior_norm :182-187, calculate_r_squared :268-279).  Rates follow an exogenous trend,
 *   lambda_j = l_min + alpha * trend_j ** delta,   mu_j = m_min + beta * trend_j ** gamma   (values <= 0 become 1e-15),
 * and the likelihood is the Keiding form over the bins of literate_library.create_bins (:231-257: unit bins from the
 * first birth time, the last one dropped) -- the statistics lr_bin_stats delivers for n_bins = that count.
 *
 *   sp, ex, br   [n_rep][n_bins]  statistics (device pointers: the outputs of lr_bin_stats; host pointers for *_host)
 *   h_trend      [n_bins] HOST    the min-max normalised trend with zeros replaced by 1e-15 (trend_rate.py:61-69)
 *   const_birth / const_death     -const_B / -const_D (-no_death implies -const_D, :44); both together are refused
 *                                 (the reference stops in np.random.binomial(p = nan), :129-134)
 * Chain c uses replicate h_rep_of_chain[c] (NULL: 0) and the Philox-4x32-10 stream keyed by (seed, chain_id0 + c).  The
 * initial state is :141-147; as in the reference the proposal of iteration 0 is always accepted (:176). */
typedef struct lr_trend_s* lr_trend_t;
int lr_trend_create(lr_handle_t h, int32_t n_rep, int32_t n_bins, const int64_t* d_sp, const int64_t* d_ex,
                    const double* d_br, const double* h_trend, int32_t const_birth, int32_t const_death,
                    int32_t n_chains, uint64_t seed, int64_t chain_id0, const int32_t* h_rep_of_chain,
                    void* stream, lr_trend_t* out);
int lr_trend_create_host(lr_handle_t h, int32_t n_rep, int32_t n_bins, const int64_t* h_sp, const int64_t* h_ex,
                         const double* h_br, const double* h_trend, int32_t const_birth, int32_t const_death,
                         int32_t n_chains, uint64_t seed, int64_t chain_id0, const int32_t* h_rep_of_chain,
                         lr_trend_t* out);
int lr_trend_destroy(lr_trend_t t);
/* One sample record = lr_trend_record_doubles(n_bins) = LR_TREND_REC_HEAD + 2 n_bins doubles (the row of :191):
 *   [0] iteration  [1] likelihood  [2] likelihood_birth  [3] likelihood_death  [4] prior
 *   [5..10] l_min, m_min, alpha, beta, delta, gamma  [11..13] adequacy (coeff, r2, gelman_r2)
 *   [14] proposals accepted so far  [15] inverse temperature beta of the chain (1 unless tempered, lr_trend_set_beta_host)
 *   [16 .. 16+n_bins) birth rates  [16+n_bins .. 16+2 n_bins) death rates */
#define LR_TREND_REC_HEAD 16
int64_t lr_trend_record_doubles(int32_t n_bins);
/* A record is written after every iteration `it` with it % sample_every == 0 (:184: the sample follows the accept step, so
 * the record of iteration 0 already holds the first proposal).  Layout [sample][chain][record]; asynchronous on `stream`. */
int64_t lr_trend_records_per_run(lr_trend_t t, int64_t n_iter, int64_t sample_every);
int lr_trend_run(lr_trend_t t, int64_t n_iter, int64_t sample_every, double* d_records, void* stream);
int lr_trend_run_host(lr_trend_t t, int64_t n_iter, int64_t sample_every, double* h_records);
/* Parity entry point, HOST buffers: evaluates n explicit parameter vectors params[n][6] on replicate rep[n] (NULL: 0).
 * With kind != NULL one proposal with EXPLICIT draws is applied first: kind[n] 0 multiplier (draw = uniform) / 1 additive
 * normal (draw = standard normal), on[n][6] the Bernoulli mask, draw[n][6]; out_params[n][6], out_hast[n] receive it.
 * Outputs (any may be NULL): lik[n][2] birth and death log-likelihood, prior[n], rates[n][2][n_bins], adequacy[n][3]. */
int lr_trend_eval_host(lr_trend_t t, int32_t n, const int32_t* rep, const double* params, const int32_t* kind,
                       const int32_t* on, const double* draw, double* out_params, double* out_hast, double* lik,
                       double* prior, double* rates, double* adequacy);
/* current state of every chain: [n_chains][LR_TREND_STATE_DOUBLES] = six parameters, likelihood_birth, likelihood_death,
 * prior, iterations done, proposals accepted, replicate */
#define LR_TREND_STATE_DOUBLES 12
int lr_trend_state_host(lr_trend_t t, double* h_state);
/* Tempered ladders, as lr_chains_set_beta_host .. lr_chains_swap_step (new; the reference has no tempering).  A chain at
 * beta = 1 is the reference's chain; a heated chain raises the likelihood (not the prior) to the power beta < 1.  Swap rounds
 * exchange temperatures between neighbours of a ladder of `ladder` consecutive GLOBAL chain ids by the rule of
 * lr_chains_swap_apply; the exchanged likelihood is the stored one of the current state.
 *   set_beta_host: beta[n_chains] (HOST), each in [0, 1]; chains start at 1.
 *   swap_info / swap_apply: as lr_chains_swap_info / lr_chains_swap_apply, async on `stream`.
 *   swap_step: one round on the handle's stream for a shard that holds whole ladders, each on a single replicate.
 *   temper_host: current beta[n_chains] and swaps proposed / accepted [n_chains][2] (HOST; either may be NULL). */
int lr_trend_set_beta_host(lr_trend_t t, const double* h_beta);
int lr_trend_swap_info(lr_trend_t t, double* d_info, void* stream);
int lr_trend_swap_apply(lr_trend_t t, const double* d_info_all, int64_t n_all, int64_t first, int32_t ladder, uint64_t round,
                        void* stream);
int lr_trend_swap_step(lr_trend_t t, int32_t ladder, uint64_t round);
int lr_trend_temper_host(lr_trend_t t, double* h_beta, int64_t* h_swaps);

/* ---------------------------------------------------------------- DDRate (SURVEY 8 f-4): diversity-dependent rates on the same statistics
 *
 * Replaces the Metropolis-Hastings loop of DDRatev3.py:242-292 (likelihood_function :82-124, calc_prior :127-141, proposals
 * literate_library.py:124-128, :156-165).  Parameters (:83): l_f, l_mul, k, x0, div_0, L, m_mul, nuB, nuD, g_lambda1,
 * g_lambda2.  m_birth: 0 constant, 1 constant carrying capacity, 2 logistic carrying capacity, 3 = 2 plus the genre-birth term of
 * :99-102 (needs the genre table h_gts/h_gte[n_genre], HOST, as parse_ts_te leaves it); m_death: 0 death rate 1 (:105-106),
 * 1 constant, 2 logistic carrying capacity.  -m_birth -1 / -m_death -1 stop with NameError in the reference (:192-195) and are
 * refused.  sp, ex, br [n_rep][n_bins] are the statistics of literate_library.create_bins' window (as for lr_trend_create; replicates =
 * stochastic imputations of one data set over a common window); origin/present = min ts / max te (:35).  Chain c runs on replicate
 * h_rep_of_chain[c] (NULL: 0) and draws from the Philox-4x32-10 stream keyed by (seed, chain_id0 + c). */
typedef struct lr_dd_s* lr_dd_t;
#define LR_DD_NPAR 11
int lr_dd_create(lr_handle_t h, int32_t n_rep, int32_t n_bins, const int64_t* d_sp, const int64_t* d_ex, const double* d_br,
                 double origin, double present, int32_t m_birth, int32_t m_death,
                 const double* h_gts, const double* h_gte, int32_t n_genre,
                 int32_t n_chains, uint64_t seed, int64_t chain_id0, const int32_t* h_rep_of_chain, void* stream, lr_dd_t* out);
int lr_dd_create_host(lr_handle_t h, int32_t n_rep, int32_t n_bins, const int64_t* h_sp, const int64_t* h_ex, const double* h_br,
                      double origin, double present, int32_t m_birth, int32_t m_death,
                      const double* h_gts, const double* h_gte, int32_t n_genre,
                      int32_t n_chains, uint64_t seed, int64_t chain_id0, const int32_t* h_rep_of_chain, lr_dd_t* out);
int lr_dd_destroy(lr_dd_t t);
/* One sample record = lr_dd_record_doubles(n_bins) = LR_DD_REC_HEAD + 4 n_bins doubles (the row of :285-287):
 *   [0] iteration  [1] likelihood (sum of the three terms; the genre term is the constant 1 unless m_birth = 3, :84)
 *   [2] likelihood_birth  [3] likelihood_death  [4] prior  [5..15] the 11 parameters as the chain holds them (x0 relative to
 *   origin, L without div_0: the log row adds them, :278-279)  [16] genre term  [17..19] adequacy  [20] proposals accepted
 *   [21] inverse temperature beta of the chain (1 unless tempered, lr_dd_set_beta_host)  [22..23] reserved  then birth rates, death rates, niche, niche fraction, n_bins each */
#define LR_DD_REC_HEAD 24
int64_t lr_dd_record_doubles(int32_t n_bins);
int64_t lr_dd_records_per_run(lr_dd_t t, int64_t n_iter, int64_t sample_every);
int lr_dd_run(lr_dd_t t, int64_t n_iter, int64_t sample_every, double* d_records, void* stream);
int lr_dd_run_host(lr_dd_t t, int64_t n_iter, int64_t sample_every, double* h_records);
/* Parity entry point, HOST buffers: n explicit parameter vectors params[n][11] on replicate rep[n] (NULL: 0); with kind != NULL one proposal with EXPLICIT
 * draws is applied first: kind[n] 0 multiplier move (on[n][11] mask, draw[n][11] uniforms), 1 sliding window on x0 (uniform
 * draw[n][3]), 2 sliding window on m_mul (uniform draw[n][6]).  Outputs (any may be NULL): out_params[n][11], out_hast[n],
 * lik[n][3] (birth, death, genre), prior[n], series[n][4][n_bins], adequacy[n][3], genre[n][4] (births and time at risk of the
 * genre table before / after origin + x0). */
int lr_dd_eval_host(lr_dd_t t, int32_t n, const int32_t* rep, const double* params, const int32_t* kind, const int32_t* on, const double* draw,
                    double* out_params, double* out_hast, double* lik, double* prior, double* series, double* adequacy,
                    double* genre);
/* [n_chains][LR_DD_STATE_DOUBLES]: 11 parameters, the three likelihood terms, prior, iterations done, proposals accepted,
 * the four cached genre statistics, replicate, 2 reserved */
#define LR_DD_STATE_DOUBLES 24
int lr_dd_state_host(lr_dd_t t, double* h_state);
/* Tempered ladders: as the lr_trend_* calls of the same names; the tempered likelihood includes the genre term. */
int lr_dd_set_beta_host(lr_dd_t t, const double* h_beta);
int lr_dd_swap_info(lr_dd_t t, double* d_info, void* stream);
int lr_dd_swap_apply(lr_dd_t t, const double* d_info_all, int64_t n_all, int64_t first, int32_t ladder, uint64_t round, void* stream);
int lr_dd_swap_step(lr_dd_t t, int32_t ladder, uint64_t round);
int lr_dd_temper_host(lr_dd_t t, double* h_beta, int64_t* h_swaps);

#ifdef __cplusplus
}
#endif
#endif /* LITERATE_B200_H */
