// K2 (dataset tables + batched state evaluation) and K3 (the multi-chain RJMCMC loop, whole loop on device).
//
// K3 replaces runMCMC (LiteRateForward.py:216-373).  A chain lives in the registers of one warp (lane k = slot k of the
// birth and of the death side); per iteration it takes its random numbers from a Philox-4x32-10 stream keyed by
// (seed, global chain id, iteration), builds the proposal with register shuffles, forms the Metropolis-Hastings ratio as
// one warp reduction of per-lane differences and commits or not -- no host round trip, no memory traffic besides the
// read-only prefix tables and the sample records.  Two builds of the loop (specialised: producer warps feed the chain
// warp through a shared-memory ring; compact: one warp does everything) are described where they are defined.
// Reference quirks kept on purpose (SURVEY Appendix A): no-op move-shift (:184-185), stale priorPoiA (:300-304,:319),
// initial prior with Gamma rate 2 (:227), `>=` accept test (:313), min-spacing guard (:290).
#include <stdlib.h>
#include "chain_device.cuh"

namespace {

__constant__ double c_lnfact[LR_SLOTS + 2];

struct ChainState {
    long long it;
    long long counters[LR_NCOUNTERS];   // 0..7 maintained by k3_run_kernel, 8..9 by the tempered-swap kernel
    long long team[6];                  // diagnostics of the speculative team build (k3_team.cuh)
    long long solo_until;               // the team build leaves the chain to the continuation pass while it < solo_until
    unsigned win_iters, win_commits;    // the team build's current observation window (state changes per iteration)
    long long solo_span;                // how long the next hand-over lasts (doubles while the teams keep stopping)
    int K_l, K_m, rep, poi_is_init;
    unsigned chain_id, consistent;
    double priorA, poiA, gL, gM, poi, beta;
    double rL[LR_SLOTS], lrL[LR_SLOTS], tL[LR_SLOTS];
    double rM[LR_SLOTS], lrM[LR_SLOTS], tM[LR_SLOTS];
};

}  // namespace

struct lr_chains_s {
    lr_handle_t h;
    lr_dataset_t ds;
    int n_chains;
    lr_chain_config cfg;
    uint64_t seed;
    int64_t chain_id0;    // global id of chain 0 of this shard
    ChainState* st;       // device [n_chains]
    lr_last_stream last;  // stream that touched the chains last (lr_order)
    long long it_host;    // iteration counter of every chain as the host knows it (-1: chains differ, set through set_state)
};

namespace {

// ------------------------------------------------------------------------------------------------
// dataset tables
// ------------------------------------------------------------------------------------------------
__global__ void k2_build_tables(const long long* __restrict__ sp, const long long* __restrict__ ex,
                                const double* __restrict__ br, const long long* __restrict__ exd,
                                const double* __restrict__ brd, int nb, int model, double* __restrict__ tab_all,
                                double* __restrict__ cst_all) {
    const int rep = blockIdx.x, t = threadIdx.x;
    const long long* U = sp + (size_t)rep * nb;
    const long long* D = ex + (size_t)rep * nb;
    const double* K = br + (size_t)rep * nb;
    const long long* Dd = exd ? exd + (size_t)rep * nb : D;
    const double* Kd = brd ? brd + (size_t)rep * nb : K;
    double* tab = tab_all + (size_t)rep * LR_NTAB * (nb + 1);
    if (t < LR_NTAB) {
        double acc = 0.0;
        double* T = tab + (size_t)t * (nb + 1);
        T[0] = 0.0;
        for (int j = 0; j < nb; ++j) {
            const bool m = (model <= 1) ? (K[j] > 0.0) : true;
            double v = 0.0;
            switch (t) {
                case T_AB: v = m ? (double)U[j] : 0.0; break;
                case T_BB: v = (model == 1) ? (m ? 1.0 : 0.0) : (m ? K[j] : 0.0); break;
                case T_AD: v = (model == 3) ? (double)Dd[j] : (m ? (double)D[j] : 0.0); break;
                case T_BD: v = (model == 3) ? Kd[j] : (m ? K[j] : 0.0); break;
                case T_XB: v = (double)U[j] / K[j]; break;
                case T_XD: v = (double)D[j] / K[j]; break;
            }
            acc += v;
            T[j + 1] = acc;
        }
    } else if (t == 32) {
        double c = 0.0, sx = 0.0, sxx = 0.0;
        for (int j = 0; j < nb; ++j) {
            if (model <= 1 && K[j] > 0.0) {
                const double lk = log(K[j]);
                c += (model == 0 ? (double)(U[j] + D[j]) : (double)D[j]) * lk;
            }
            const double xb = (double)U[j] / K[j], xd = (double)D[j] / K[j];
            sx += xb + xd;
            sxx += xb * xb + xd * xd;
        }
        cst_all[rep * LR_NCST + 0] = c;
        cst_all[rep * LR_NCST + 1] = sx;
        cst_all[rep * LR_NCST + 2] = sxx;
        cst_all[rep * LR_NCST + 3] = 0.0;
    }
}

// General form of the same tables: per bin and side an event weight A_j and an exposure B_j, the likelihood being
//     C + sum_j [ A^b_j log(lambda_j) - B^b_j lambda_j ] + sum_j [ A^d_j log(mu_j) - B^d_j mu_j ]
// (every likelihood of the reference has this shape; the four -model_BDI tables above are instances).  Used for the
// `-proportion 1` variant (LiteRateForward-proportion.py:157-162): A = interpolated yearly counts of a series masked by its
// running total > 0, B = that mask, C = 0; x_b / x_d are the vectors calculate_r_squared regresses on (:627-628: the counts).
__global__ void k2_build_tables_general(const double* __restrict__ Ab, const double* __restrict__ Bb, const double* __restrict__ Ad,
                                        const double* __restrict__ Bd, const double* __restrict__ xb, const double* __restrict__ xd,
                                        const double* __restrict__ C, int nb, double* __restrict__ tab_all, double* __restrict__ cst_all) {
    const int rep = blockIdx.x, t = threadIdx.x;
    double* tab = tab_all + (size_t)rep * LR_NTAB * (nb + 1);
    const size_t o = (size_t)rep * nb;
    if (t < LR_NTAB) {
        const double* src = t == T_AB ? Ab : (t == T_BB ? Bb : (t == T_AD ? Ad : (t == T_BD ? Bd : (t == T_XB ? xb : xd))));
        double acc = 0.0;
        double* T = tab + (size_t)t * (nb + 1);
        T[0] = 0.0;
        for (int j = 0; j < nb; ++j) { acc += src[o + j]; T[j + 1] = acc; }
    } else if (t == 32) {
        double sx = 0.0, sxx = 0.0;
        for (int j = 0; j < nb; ++j) { sx += xb[o + j] + xd[o + j]; sxx += xb[o + j] * xb[o + j] + xd[o + j] * xd[o + j]; }
        cst_all[rep * LR_NCST + 0] = C ? C[rep] : 0.0;
        cst_all[rep * LR_NCST + 1] = sx;
        cst_all[rep * LR_NCST + 2] = sxx;
        cst_all[rep * LR_NCST + 3] = 0.0;
    }
}

// ------------------------------------------------------------------------------------------------
// per-warp random numbers
// ------------------------------------------------------------------------------------------------
struct Rng {
    uint32_t k0, k1, chain;
    __device__ __forceinline__ void draw(long long it, uint32_t purpose, int lane, double& ua, double& ub) const {
        Philox4 p = philox4x32_10((uint32_t)it, (uint32_t)((unsigned long long)it >> 32), (uint32_t)lane | (purpose << 8), chain, k0, k1);
        ua = u01(p.x, p.y);
        ub = u01(p.z, p.w);
    }
};

// Gamma(a, 1), 1 <= a < 2 (Marsaglia & Tsang 2000), 32 attempts per round, first accepted lane wins
__device__ __noinline__ double warp_gamma_mt(double a, const Rng rng, long long it, uint32_t purpose, int lane) {
    const double d = a - 1.0 / 3.0, c = rsqrt(9.0 * d);
    for (uint32_t round = 0;; ++round) {
        double u1, u2, u3, u4;
        rng.draw(it, purpose + 2 * round, lane, u1, u2);
        rng.draw(it, purpose + 2 * round + 1, lane, u3, u4);
        const double z = sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
        double v = 1.0 + c * z;
        bool ok = v > 0.0;
        v = v * v * v;
        ok = ok && (log(u3) < 0.5 * z * z + d - d * v + d * log(v));
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (m) return __shfl_sync(0xffffffffu, d * v, __ffs(m) - 1);
        if (round > 64) return d;   // unreachable in practice (p ~ 0.05^2048)
    }
}

// ------------------------------------------------------------------------------------------------
// state <-> registers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void load_sides(const ChainState* S, Side& L, Side& M, int lane) {
    L.K = S->K_l; M.K = S->K_m;
    L.r = S->rL[lane]; L.lr = S->lrL[lane]; L.t = S->tL[lane];
    M.r = S->rM[lane]; M.lr = S->lrM[lane]; M.t = S->tM[lane];
}
__device__ __forceinline__ void store_sides(ChainState* S, const Side& L, const Side& M, int lane) {
    S->rL[lane] = L.r; S->lrL[lane] = L.lr; S->tL[lane] = L.t;
    S->rM[lane] = M.r; S->lrM[lane] = M.lr; S->tM[lane] = M.t;
    if (lane == 0) { S->K_l = L.K; S->K_m = M.K; }
}

struct Hyper {
    double gL, gM, lgL, lgM, poi, lpoi;
};

__device__ __forceinline__ double full_prior(const Side& L, const Side& M, const Hyper& hp, const DataView& d, double poi_term) {
    // :296-303
    return rates_prior(L, hp.gL, hp.lgL) + rates_prior(M, hp.gM, hp.lgM) - d.log_span * (double)(L.K + M.K - 2) + poi_term;
}

// (cold functions take their arguments BY VALUE: a reference into a __noinline__ callee would make the caller keep the
// chain's state in local memory for the whole loop)
__device__ __noinline__ void write_record(double* rec, long long it, Side L, Side M, const Hyper hp, const DataView d,
                                          double priorA, double poiA, int consistent, int poi_is_init, double beta, int lane, bool with_adequacy) {
    side_sums(L, lane); side_sums(M, lane);
    if (consistent) priorA = full_prior(L, M, hp, d, poiA);     // the stored prior IS the prior of the state (with the stale poiA, :300-304)
    double adq[3] = {0.0, 0.0, 0.0};
    if (with_adequacy) adequacy3(L, M, d, lane, adq);
    if (lane == 0) {
        rec[0] = (double)it;
        rec[1] = d.C + L.lik + M.lik;
        rec[2] = priorA;
        rec[3] = L.sumr / (double)L.K;
        rec[4] = M.sumr / (double)M.K;
        rec[5] = (double)L.K;
        rec[6] = (double)M.K;
        rec[7] = hp.gL; rec[8] = hp.gM; rec[9] = hp.poi;
        rec[10] = adq[0]; rec[11] = adq[1]; rec[12] = adq[2];
        rec[13] = (double)poi_is_init; rec[14] = beta; rec[15] = poiA;      // [15]: the stored (possibly stale) priorPoiA of :300-304
    }
    rec[16 + lane] = lane < L.K ? L.r : 0.0;
    rec[48 + lane] = lane < L.K ? (lane == 0 ? d.start_time : L.t) : 0.0;
    rec[80 + lane] = lane < M.K ? M.r : 0.0;
    rec[112 + lane] = lane < M.K ? (lane == 0 ? d.start_time : M.t) : 0.0;
}

// branch frequencies and update fractions of the loop (:243-252), computed once on the host: as kernel parameters they are
// constant-bank operands instead of per-iteration selects
struct LoopConsts {
    double shift_mu, b_freq, d_freq, fL, fM;
    int const_rates, real_move_shift;
};
__host__ __device__ inline LoopConsts loop_consts(const lr_chain_config& cfg) {
    LoopConsts k;
    k.shift_mu = cfg.const_death_rate ? 0.0 : 0.5;          // :243-252
    k.b_freq = cfg.const_death_rate ? 0.7 : 0.4; k.d_freq = 0.8;
    k.fL = cfg.update_fraction; k.fM = cfg.const_death_rate ? 1.0 : cfg.update_fraction;
    k.const_rates = cfg.const_rates; k.real_move_shift = cfg.real_move_shift;
    return k;
}

struct RunParams {
    ChainState* st;
    int n_chains;
    const double* tab; const double* cst;
    int nb, s0f, model;
    double start_time, end_time;
    lr_chain_config cfg;
    LoopConsts lc;
    uint32_t k0, k1;
    long long n_iter, sample_every;
    long long it_begin;  // first iteration of this launch (every chain's, as the host tracks it); -1: take each chain's own counter
    int team_bail;       // team build: may hand a chain with frequent state changes to the continuation pass
    int cont_mode;       // k3_run_kernel as continuation pass: 1 = only handed-over chains, up to the end of their hand-over; 0 = to the end
    double* records;     // [sample][chain][LR_REC_DOUBLES] or null
    int with_adequacy;
};

// ------------------------------------------------------------------------------------------------
// The loop, in two builds of one source.
//
// Everything an iteration takes from the random stream is independent of the chain's state: the branch uniforms, the
// per-rate multipliers exp(2 ln 1.1 (u - .5)) of the rate update, the Beta(10,10) variate of the add-shift move with
// its logarithms, a single-precision bracket of log(u) for the accept test.  make_draws() computes all of it from the
// counter-based Philox stream of (seed, chain, iteration).
//
//   SPECIALISED (few chains; ncu: one warp per scheduler, 54 % of stall samples on fixed-latency dependencies):
//       one CTA of 4 warps per chain.  Warps 1-3 are PRODUCERS: each runs make_draws() for every third iteration and
//       publishes it into a shared-memory ring (release/acquire flags).  Warp 0 is the CHAIN warp: it only does the
//       state-dependent part (segment statistics, sums, prior, accept, commit), so Philox, the exponentials of the
//       multipliers and the five logarithms of the add-shift move leave its dependency chain.
//   COMPACT (thousands of chains resident; ncu: 54 % no_inst with a 45 KB hot footprint): one warp per chain calls
//       make_draws() inline, one out-of-line copy of log/exp, side selected at run time, 92 registers.
// Both run the same arithmetic on the same random numbers: identical chains, bit for bit (tested).
// ------------------------------------------------------------------------------------------------
__device__ __noinline__ double ool_log(double x) { return log(x); }
__device__ __noinline__ double ool_exp(double x) { return exp(x); }
template <bool C> __device__ __forceinline__ double xlog(double x) { if constexpr (C) return ool_log(x); else return log(x); }
template <bool C> __device__ __forceinline__ double xexp(double x) { if constexpr (C) return ool_exp(x); else return exp(x); }

struct Draws {
    double u_acc;                  // the accept uniform (:313)
    double thr_hi, thr_lo;         // single-precision bracket of log(u_acc): x >= thr_hi accepts, x < thr_lo rejects
    int kind;                      // proposal type decided by the branch uniforms alone (:234, :74): DK_* << 1 | birth side
    double u_idx, u_t;             // RJMCMC / move: segment or shift index, position inside the segment
    double w, ln_beta;             // add-shift: log((1-u)/u) and beta.logpdf(u; 10, 10) of the Beta variate u (:22-23, :41-42)
    double m, dlt;                 // this lane's rate multiplier and its logarithm (1, 0 when the rate is not touched) (:165-176)
};

// proposal kinds (Draws::kind >> 1)
#define DK_BLOCK_RATE 0     // birth/death block, rate multiplier (:258, :268)
#define DK_BLOCK_MOVE 1     // birth/death block, move-shift unless the side has a single rate (:261, :271)
#define DK_RJ_ADD 2
#define DK_RJ_REMOVE 3
#define DK_GIBBS 4

// K_l / K_m: the chain's current numbers of rates if the caller knows them (compact build), -1 otherwise (producers): a
// block iteration that will be a move-shift (r1 >= .5 on a side with more than one rate) does not need the multipliers.
template <bool C>
__device__ __forceinline__ Draws make_draws(const Rng& rng, long long it, int lane, const LoopConsts& k, int K_l = -1, int K_m = -1) {
    Draws q;
    double ua, ub;
    rng.draw(it, 0, lane, ua, ub);
    const double r0 = __shfl_sync(0xffffffffu, ua, 31), r1 = __shfl_sync(0xffffffffu, ub, 31);   // np.random.random(2) of :234
    q.u_acc = __shfl_sync(0xffffffffu, ua, 30);
    // bracket of log(u) for the accept test (error bound: __logf <= 2^-21.4 absolute on [.5,2], 3 ulp elsewhere, plus the
    // rounding of u to float)
    const float lf = __logf((float)q.u_acc);
    const float err = 2e-6f * (1.0f + fabsf(lf));
    q.thr_hi = (double)(lf + err); q.thr_lo = (double)(lf - err);
    q.u_idx = 0.0; q.u_t = 0.0; q.w = 0.0; q.ln_beta = 0.0; q.m = 1.0; q.dlt = 0.0;
    if (r0 < k.d_freq) {
        // update_multiplier_freq (:165-176): each rate w.p. f times exp(2 ln(1.1) (u - .5))
        const bool birth = r0 < k.b_freq;
        const double f = birth ? k.fL : k.fM;
        const int K_side = birth ? K_l : K_m;
        if (r1 < 0.5 || K_side <= 1) {
            const bool touched = ua < f;
            q.dlt = touched ? LR_LN_MULT * (ub - 0.5) : 0.0;
            q.m = exp_small(q.dlt);                         // |dlt| <= 0.0954: 11-term polynomial, inline; exp_small(0) = 1 exactly
        }
        q.kind = ((r1 < 0.5 ? DK_BLOCK_RATE : DK_BLOCK_MOVE) << 1) | (birth ? 1 : 0);
        if (k.real_move_shift) { q.u_idx = __shfl_sync(0xffffffffu, ua, 28); q.u_t = __shfl_sync(0xffffffffu, ub, 28); }
    } else if (r0 < 0.999 && !k.const_rates) {
        const double rs = __shfl_sync(0xffffffffu, ua, 29), ra = __shfl_sync(0xffffffffu, ub, 29);   // np.random.random(2) of :74
        q.u_idx = __shfl_sync(0xffffffffu, ua, 28); q.u_t = __shfl_sync(0xffffffffu, ub, 28);
        const bool birth = rs > k.shift_mu;
        if (ra > 0.5) {
            // Beta(10,10) = G1/(G1+G2), Gamma(10,1) = -log(prod of 10 uniforms); every logarithm of u the reference takes
            // is assembled from log g1, log g2, log(g1+g2)
            // (the five logarithms are of warp-uniform values: lanes 0-2 take one each, two calls instead of five)
            const double p1 = warp_prod(lane < 10 ? ua : 1.0), p2 = warp_prod(lane < 10 ? ub : 1.0);
            const double lp = xlog<C>(lane == 1 ? p2 : p1);
            const double g1 = -__shfl_sync(0xffffffffu, lp, 0), g2 = -__shfl_sync(0xffffffffu, lp, 1);
            const double lg = xlog<C>(lane == 0 ? g1 : (lane == 1 ? g2 : g1 + g2));
            const double lg1 = __shfl_sync(0xffffffffu, lg, 0), lg2 = __shfl_sync(0xffffffffu, lg, 1), lgs = __shfl_sync(0xffffffffu, lg, 2);
            q.w = lg2 - lg1;
            q.ln_beta = (LR_SHAPE_BETA - 1.0) * (lg1 + lg2 - 2.0 * lgs) - LR_BETA_NORM;
            q.kind = (DK_RJ_ADD << 1) | (birth ? 1 : 0);
        } else {
            q.kind = (DK_RJ_REMOVE << 1) | (birth ? 1 : 0);
        }
    } else {
        q.kind = DK_GIBBS << 1;
    }
    return q;
}

// ---- shared-memory ring between the producer warps and the chain warp (SPECIALISED build).
// The unit of hand-off is a BATCH of RING_BATCH consecutive iterations: batch b is produced by producer b % PPC of the
// chain into slot b % DEPTH and published with one release store; the chain warp acquires once per batch and releases the slot
// when it has taken the batch's last iteration.
constexpr int RING_BATCH = 8;
struct RingIter {
    double m[32], dlt[32];
    double sc[16];                     // u_acc u_idx u_t w ln_beta thr_hi thr_lo kind
};
template <int DEPTH>
struct Ring {
    RingIter it[DEPTH][RING_BATCH];
    unsigned long long full[DEPTH];        // b + 1 once batch b is published
    unsigned long long done[DEPTH];        // b + 1 once batch b has been consumed
};
// register re-balancing between the warpgroups of the 4-chains-per-CTA build (PTX setmaxnreg, sm_90+): the kernel is
// launched at 128 registers per thread (2 CTAs of 256 threads per SM); the producer warpgroup gives registers back, the
// chain warpgroup takes them
template <int N> __device__ __forceinline__ void reg_dealloc() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" :: "n"(N)); }
template <int N> __device__ __forceinline__ void reg_alloc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" :: "n"(N)); }
__device__ __forceinline__ unsigned long long ld_acquire_cta(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.cta.shared.u64 %0, [%1];" : "=l"(v) : "r"((unsigned)__cvta_generic_to_shared(p)) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_cta(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.cta.shared.u64 [%0], %1;" :: "r"((unsigned)__cvta_generic_to_shared(p)), "l"(v) : "memory");
}
__device__ __forceinline__ void ring_store(RingIter& S, const Draws& q, int lane) {
    S.m[lane] = q.m; S.dlt[lane] = q.dlt;
    double v = q.u_acc;
    v = lane == 1 ? q.u_idx : v; v = lane == 2 ? q.u_t : v; v = lane == 3 ? q.w : v; v = lane == 4 ? q.ln_beta : v;
    v = lane == 5 ? q.thr_hi : v; v = lane == 6 ? q.thr_lo : v; v = lane == 7 ? __longlong_as_double((long long)q.kind) : v;
    if (lane < 8) S.sc[lane] = v;
}
__device__ __forceinline__ Draws ring_load(const RingIter& S, int lane) {
    Draws q;
    q.m = S.m[lane]; q.dlt = S.dlt[lane];
    q.u_acc = S.sc[0]; q.u_idx = S.sc[1]; q.u_t = S.sc[2]; q.w = S.sc[3]; q.ln_beta = S.sc[4];
    q.thr_hi = S.sc[5]; q.thr_lo = S.sc[6]; q.kind = (int)__double_as_longlong(S.sc[7]);
    return q;
}

// ------------------------------------------------------------------------------------------------
// proposals on one side (all warp-uniform control flow)
// ------------------------------------------------------------------------------------------------
// add_shift_RJ_weighted_mean (:29-47).  Returns false if the proposal violates the spacing guard (:290).
template <bool C, bool SUMS>
__device__ __forceinline__ bool propose_add(const Side& cur, Side& nw, const DataView& d, int tabA, int tabB,
                                            const Draws& q, int lane, double& hasting) {
    const int K = cur.K;
    int i = (int)(q.u_idx * (double)K);
    if (i > K - 1) i = K - 1;
    const double t_raw = (lane == 0) ? d.start_time : cur.t;
    const double t_i = __shfl_sync(0xffffffffu, t_raw, i);
    double t_n = __shfl_sync(0xffffffffu, t_raw, (i + 1) & 31);
    if (i + 1 >= K) t_n = d.end_time;
    const double gap = t_n - t_i;
    const double tp = t_i + q.u_t * gap;                     // np.random.uniform(0, gap)
    if ((tp - t_i) <= LR_MIN_DT || (t_n - tp) <= LR_MIN_DT) return false;
    const double p1 = (t_i - tp) / (t_i - t_n);
    const double p2 = (tp - t_n) / (t_i - t_n);
    const double lr_i = __shfl_sync(0xffffffffu, cur.lr, i);
    const double lr1 = lr_i - p2 * q.w, lr2 = lr_i + p1 * q.w;
    const double er = xexp<C>(lane == 1 ? lr2 : lr1);              // both exponentials in one call (lanes 0 and 1)
    const double r1 = __shfl_sync(0xffffffffu, er, 0), r2 = __shfl_sync(0xffffffffu, er, 1);
    const double rs = r1 + r2;
    // log|gap| + 2 log(r1 + r2): one logarithm (two where the square would leave fp64)
    hasting = ((rs > 1e-150 && rs < 1e150) ? xlog<C>(fabs(gap) * rs * rs) : xlog<C>(fabs(gap)) + 2.0 * xlog<C>(rs)) - q.ln_beta - lr_i;
    // shift slots above i up by one
    const double ur = __shfl_up_sync(0xffffffffu, cur.r, 1);
    const double ulr = __shfl_up_sync(0xffffffffu, cur.lr, 1);
    const double ut = __shfl_up_sync(0xffffffffu, cur.t, 1);
    nw = cur;
    nw.K = K + 1;
    if (lane == i) { nw.r = r1; nw.lr = lr1; }
    else if (lane == i + 1) { nw.r = r2; nw.lr = lr2; nw.t = tp; }
    else if (lane > i + 1) { nw.r = ur; nw.lr = ulr; nw.t = ut; }
    side_stats(nw, d, tabA, tabB, lane);
    if constexpr (SUMS) side_sums(nw, lane);
    return true;
}

// remove_shift_RJ_weighted_mean (:49-69); caller guarantees K > 1.  u = ra/(ra+rb): log u and log(1-u) come from the
// stored log-rates and the one logarithm of (ra+rb) the Jacobian needs anyway.
template <bool C, bool SUMS>
__device__ __forceinline__ void propose_remove(const Side& cur, Side& nw, const DataView& d, int tabA, int tabB,
                                               const Draws& q, int lane, double& hasting) {
    const int K = cur.K;
    int j = 1 + (int)(q.u_idx * (double)(K - 1));
    if (j > K - 1) j = K - 1;
    const double t_raw = (lane == 0) ? d.start_time : cur.t;
    const double t_rm = __shfl_sync(0xffffffffu, t_raw, j);
    const double t_a = __shfl_sync(0xffffffffu, t_raw, j - 1);
    double t_b = __shfl_sync(0xffffffffu, t_raw, (j + 1) & 31);
    if (j + 1 >= K) t_b = d.end_time;
    const double dT = fabs(t_b - t_a);
    const double p1 = (t_a - t_rm) / (t_a - t_b);
    const double p2 = (t_rm - t_b) / (t_a - t_b);
    const double lra = __shfl_sync(0xffffffffu, cur.lr, j - 1), lrb = __shfl_sync(0xffffffffu, cur.lr, j);
    const double ra = __shfl_sync(0xffffffffu, cur.r, j - 1), rb = __shfl_sync(0xffffffffu, cur.r, j);
    const double lm = p1 * lra + p2 * lrb;
    const double merged = xexp<C>(lm);
    // -log dT + lnBeta(u) + lm - 2 log(ra + rb), lnBeta(u) = 9 (lra + lrb - 2 log(ra + rb)) - norm: the three logarithms of
    // the reference collapse into  -log(dT (ra + rb)^20)  (rates within 1e-15 .. 1e15 keep the power inside fp64)
    const double s1 = ra + rb, s2 = s1 * s1, s4 = s2 * s2, s8 = s4 * s4, s16 = s8 * s8;
    // (s1^20 leaves fp64 for rates beyond ~1e-15 .. 1e15: there the two logarithms are taken separately, as the reference does)
    const double lg = (s1 > 1e-14 && s1 < 1e14) ? xlog<C>(dT * (s16 * s4)) : xlog<C>(dT) + 20.0 * xlog<C>(s1);
    hasting = (LR_SHAPE_BETA - 1.0) * (lra + lrb) - LR_BETA_NORM + lm - lg;
    const double dr = __shfl_down_sync(0xffffffffu, cur.r, 1);
    const double dlr = __shfl_down_sync(0xffffffffu, cur.lr, 1);
    const double dt = __shfl_down_sync(0xffffffffu, cur.t, 1);
    nw = cur;
    nw.K = K - 1;
    if (lane == j - 1) { nw.r = merged; nw.lr = lm; }
    else if (lane >= j) { nw.r = dr; nw.lr = dlr; nw.t = dt; }
    side_stats(nw, d, tabA, tabB, lane);
    if constexpr (SUMS) side_sums(nw, lane);
}

// opt-in real move-shift: reflected sliding window of width 1 on one interior shift (what
// update_sliding_win :178-186 computes before it overwrites the result)
template <bool SUMS>
__device__ __forceinline__ bool propose_move(const Side& cur, Side& nw, const DataView& d, int tabA, int tabB,
                                             const Draws& q, int lane) {
    const int K = cur.K;
    int j = 1 + (int)(q.u_idx * (double)(K - 1));
    if (j > K - 1) j = K - 1;
    const double t_raw = (lane == 0) ? d.start_time : cur.t;
    const double t_j = __shfl_sync(0xffffffffu, t_raw, j);
    const double t_a = __shfl_sync(0xffffffffu, t_raw, j - 1);
    double t_b = __shfl_sync(0xffffffffu, t_raw, (j + 1) & 31);
    if (j + 1 >= K) t_b = d.end_time;
    double tp = t_j + (q.u_t - 0.5) * 1.0;
    if (tp < d.start_time) tp = d.start_time + (d.start_time - tp);
    if (tp > d.end_time) tp = d.end_time - (tp - d.end_time);
    nw = cur;
    if (lane == j) nw.t = tp;
    if ((tp - t_a) <= LR_MIN_DT || (t_b - tp) <= LR_MIN_DT) return false;
    side_stats(nw, d, tabA, tabB, lane);
    if constexpr (SUMS) side_sums(nw, lane);
    return true;
}

// Metropolis-Hastings test `x >= log(u)` (:313).  The double-precision logarithm is only evaluated when the
// single-precision bracket [thr_lo, thr_hi] of log(u) cannot decide; the decision is the one the exact comparison gives.
__device__ __forceinline__ bool mh_accept(double x, const Draws& q) {
    if (x >= q.thr_hi) return true;
    if (x < q.thr_lo) return false;                // also taken for x = -inf
    return x >= ool_log(q.u_acc);                  // NaN lands here and is rejected
}

// everything of a chain that is not one of the two sides
struct ChainRegs {
    Hyper hp;
    double priorA, poiA, beta;
    int poi_is_init;
    int consistent;                // priorA is the prior of the current state under the current hyper-parameters and poiA
                                   // (false only between the initial state of :227 and the first accepted proposal)
};
// per-launch event counters (added to the chain's 64-bit counters when the launch ends; kept apart from ChainRegs so that
// they stay in registers in both builds)
struct Counters { unsigned v[8]; };
// hyper-parameters and table ids as seen from the side a proposal works on
struct SideView {
    double g_cur, lg_cur, g_oth, lg_oth;
    int tabA, tabB;
};
__device__ __forceinline__ SideView side_view(const Hyper& hp, bool birth) {
    SideView v;
    v.g_cur = birth ? hp.gL : hp.gM; v.lg_cur = birth ? hp.lgL : hp.lgM;
    v.g_oth = birth ? hp.gM : hp.gL; v.lg_oth = birth ? hp.lgM : hp.lgL;
    v.tabA = birth ? T_AB : T_AD; v.tabB = birth ? T_BB : T_BD;
    return v;
}

// ------------------------------------------------------------------------------------------------
// The accept ratio in DELTA form.  With e_k = (beta A_k + 1) lr_k - (beta B_k + g) r_k summed over the K slots of a side,
//     beta * lik_side + rates_prior_side = sum_k e_k + K * 2 log g            (:150-162 / :137-148, :201-202)
// so every proposal's  beta (lik' - lik) + (prior' - prior) + hasting  is ONE warp reduction of per-lane differences plus a
// few scalars; no sum of the current state is cached between iterations (nothing to keep consistent when the
// hyper-parameters or the temperature change), and the difference of two 1e5-sized likelihoods is never formed.
// This needs the stored prior to BE the prior of the current state (c.consistent), which holds from the first accepted
// proposal on; before that -- the reference compares against the initial prior computed with Gamma rate 2, :227 -- and for
// degenerate windows (every proposal rejected by the guard of :290) the absolute form below (slow_step) is used.
// ------------------------------------------------------------------------------------------------

// birth block (:254-262) / death block (:264-272) on side `cur`, delta form.  Returns false if the caller must use slow_step.
template <bool C>
__device__ __forceinline__ bool block_step(Side& cur, const SideView v, ChainRegs& c, Counters& n, const DataView& d,
                                           const lr_chain_config& cfg, const Draws& q, bool frozen, int lane) {
    if (!c.consistent || frozen) return false;
    const bool rate = (q.kind >> 1) == DK_BLOCK_RATE || cur.K == 1;
    if (rate) {
        // update_multiplier_freq (:165-176): q * m as the reference does; the log-rate follows by addition.
        // x = sum_k (beta A_k + 1) dlt_k - (beta B_k + g)(r'_k - r_k)  +  hasting (= sum_k dlt_k)
        n.v[3]++; n.v[2]++;
        const bool on = lane < cur.K;
        const double dl = on ? q.dlt : 0.0;
        const double rn = cur.r * (on ? q.m : 1.0);
        const double x = warp_sum_first((c.beta * cur.A + 2.0) * dl - (c.beta * cur.B + v.g_cur) * (rn - cur.r), cur.K);
        if (mh_accept(x, q)) { cur.r = rn; cur.lr += dl; n.v[1]++; }
    } else if (!cfg.real_move_shift) {
        // The reference's move proposes the current state (:184-185): prior - priorA = 0, always accepted, nothing changes.
        n.v[4]++; n.v[2]++; n.v[1]++;
    } else {
        n.v[4]++;
        Side nw;
        if (propose_move<false>(cur, nw, d, v.tabA, v.tabB, q, lane)) {
            n.v[2]++;
            const bool on = lane < cur.K;
            const double x = warp_sum(on ? c.beta * ((nw.A - cur.A) * cur.lr - (nw.B - cur.B) * cur.r) : 0.0);
            if (mh_accept(x, q)) { cur.t = nw.t; cur.A = nw.A; cur.B = nw.B; cur.jb = nw.jb; n.v[1]++; }
        }
    }
    return true;
}

// One RJ proposal in delta form: the proposed side `nw`, its Hastings/Jacobian term, the new Poisson prior and the log
// acceptance ratio x.  Shared by the loop (rj_step) and by the parity entry point lr_proposal_eval_host.
// Returns false if nothing is to be evaluated (capacity reached: *cap set; or spacing guard :290).
template <bool C>
__device__ __forceinline__ bool rj_propose(const Side& cur, const Side& oth, const SideView v, const Hyper& hp, double beta, double poiA,
                                           const DataView& d, const Draws& q, int lane, Side& nw, double& hasting, double& poiN, double& x,
                                           bool& cap) {
    nw = cur;
    hasting = 0.0;
    cap = false;
    bool ok = true;
    if ((q.kind >> 1) == DK_RJ_ADD) {
        if (cur.K >= LR_KMAX) { ok = false; cap = true; }
        else ok = propose_add<C, false>(cur, nw, d, v.tabA, v.tabB, q, lane, hasting);
    } else if (cur.K > 1) {
        propose_remove<C, false>(cur, nw, d, v.tabA, v.tabB, q, lane, hasting);
    }
    if (!ok) return false;
    poiN = poisson_prior(nw.K, hp.poi, hp.lpoi, c_lnfact) + poisson_prior(oth.K, hp.poi, hp.lpoi, c_lnfact);   // :279
    const double e_new = lane < nw.K ? (beta * nw.A + 1.0) * nw.lr - (beta * nw.B + v.g_cur) * nw.r : 0.0;
    const double e_old = lane < cur.K ? (beta * cur.A + 1.0) * cur.lr - (beta * cur.B + v.g_cur) * cur.r : 0.0;
    x = warp_sum_first(e_new - e_old, nw.K > cur.K ? nw.K : cur.K) + (double)(nw.K - cur.K) * (2.0 * v.lg_cur - d.log_span) + (poiN - poiA) + hasting;
    return true;
}

// RJMCMC (:71-97, :274-279) on side `cur`, delta form.  Returns false if the caller must use slow_step.
template <bool C>
__device__ __forceinline__ bool rj_step(Side& cur, const Side& oth, const SideView v, ChainRegs& c, Counters& n, const DataView& d,
                                        const Draws& q, bool frozen, int lane) {
    if (!c.consistent || frozen) return false;
    Side nw;
    double hasting, poiN, x;
    bool cap;
    if (rj_propose<C>(cur, oth, v, c.hp, c.beta, c.poiA, d, q, lane, nw, hasting, poiN, x, cap)) {
        n.v[2]++;
        if (mh_accept(x, q)) { cur = nw; c.poiA = poiN; n.v[1]++; }
    } else if (cap) {
        n.v[7]++;
    }
    return true;
}

// Absolute form of one block / RJ iteration: the arithmetic of :296-313 term by term, on copies with freshly computed
// sums.  Used while the stored prior is not the prior of the state (the first iterations of a chain) and for degenerate
// windows; out of line and by value (see write_record).
struct SlowOut {
    Side cur;
    double priorA, poiA;
    int consistent, accepted, evaluated, cap_reject;
};
__device__ __noinline__ SlowOut slow_step(Side cur, Side oth, const SideView v, const Hyper hp, double priorA, double poiA, double beta,
                                          int consistent, const DataView d, int real_move_shift, const Draws q, bool frozen, int lane) {
    SlowOut o;
    o.priorA = priorA; o.poiA = poiA; o.consistent = consistent; o.accepted = 0; o.evaluated = 0; o.cap_reject = 0;
    side_sums(cur, lane); side_sums(oth, lane);
    const int kind = q.kind >> 1;
    if (kind <= DK_BLOCK_MOVE) {
        const double p_oth = rates_prior(oth, v.g_oth, v.lg_oth) - d.log_span * (double)(cur.K + oth.K - 2) + poiA;   // :296-303
        if (kind == DK_BLOCK_RATE || cur.K == 1) {
            Side nw = cur;
            const bool on = lane < cur.K;
            nw.lr = cur.lr + (on ? q.dlt : 0.0);
            nw.r = cur.r * (on ? q.m : 1.0);
            side_sums(nw, lane);
            const double hasting = nw.sumlr - cur.sumlr;
            if (!frozen) {
                o.evaluated = 1;
                const double prior = rates_prior(nw, v.g_cur, v.lg_cur) + p_oth;
                if (mh_accept(beta * (nw.lik - cur.lik) + (prior - priorA) + hasting, q)) { cur = nw; o.priorA = prior; o.consistent = 1; o.accepted = 1; }
            }
        } else if (!real_move_shift) {
            // the no-op move while priorA still is the initial prior of :227: only the prior bookkeeping can differ
            if (!frozen) {
                o.evaluated = 1;
                const double prior = rates_prior(cur, v.g_cur, v.lg_cur) + p_oth;
                if (mh_accept(prior - priorA, q)) { o.priorA = prior; o.consistent = 1; o.accepted = 1; }
            }
        } else {
            Side nw;
            const bool ok = propose_move<true>(cur, nw, d, v.tabA, v.tabB, q, lane);
            if (ok && !frozen) {
                o.evaluated = 1;
                const double prior = rates_prior(nw, v.g_cur, v.lg_cur) + p_oth;
                if (mh_accept(beta * (nw.lik - cur.lik) + (prior - priorA), q)) { cur = nw; o.priorA = prior; o.consistent = 1; o.accepted = 1; }
            }
        }
    } else {
        Side nw = cur;
        double hasting = 0.0;
        bool ok = true;
        if (kind == DK_RJ_ADD) {
            if (cur.K >= LR_KMAX) { ok = false; o.cap_reject = 1; }
            else ok = propose_add<true, true>(cur, nw, d, v.tabA, v.tabB, q, lane, hasting);
        } else if (cur.K > 1) {
            propose_remove<true, true>(cur, nw, d, v.tabA, v.tabB, q, lane, hasting);
        }
        if (ok && !frozen) {
            o.evaluated = 1;
            const double poiN = poisson_prior(nw.K, hp.poi, hp.lpoi, c_lnfact) + poisson_prior(oth.K, hp.poi, hp.lpoi, c_lnfact);   // :279
            const double prior = rates_prior(nw, v.g_cur, v.lg_cur) + rates_prior(oth, v.g_oth, v.lg_oth)
                                 - d.log_span * (double)(nw.K + oth.K - 2) + poiN;
            if (mh_accept(beta * (nw.lik - cur.lik) + (prior - priorA) + hasting, q)) {
                cur = nw; o.priorA = prior; o.poiA = poiN; o.consistent = 1; o.accepted = 1;
            }
        }
    }
    o.cur = cur;
    return o;
}
__device__ __forceinline__ void run_slow(Side& cur, const Side& oth, const SideView v, ChainRegs& c, Counters& n, const DataView& d,
                                         const lr_chain_config& cfg, const Draws& q, bool frozen, int lane) {
    const int kind = q.kind >> 1;
    const SlowOut o = slow_step(cur, oth, v, c.hp, c.priorA, c.poiA, c.beta, c.consistent, d, cfg.real_move_shift, q, frozen, lane);
    cur = o.cur; c.priorA = o.priorA; c.poiA = o.poiA; c.consistent = o.consistent;
    if (kind <= DK_BLOCK_MOVE) n.v[(kind == DK_BLOCK_RATE || cur.K == 1) ? 3 : 4]++;
    n.v[2] += o.evaluated; n.v[1] += o.accepted; n.v[7] += o.cap_reject;
}

// Gibbs on the hyper-priors (:281-287), always accepted (:313); one iteration in a thousand, kept out of line.
// Arguments and result by value (see write_record).
struct GibbsOut { Hyper hp; double priorA; int poi_is_init; };
__device__ __noinline__ GibbsOut gibbs_step(Side L, Side M, Hyper hp, double poiA, int poi_is_init, const DataView d,
                                            int sample_poisson, int use_rate_HP, const Rng rng, long long it, bool frozen, int lane) {
    side_sums(L, lane); side_sums(M, lane);
    if (sample_poisson) {
        // get_post_rj_HP (:99-108): Gamma(2 + K_l + K_m, scale 1/3), integer shape
        double ga, gb;
        rng.draw(it, 1, lane, ga, gb);
        const int n = 2 + L.K + M.K;
        const double pr = warp_prod((lane < n ? ga : 1.0) * (lane + 32 < n ? gb : 1.0));
        hp.poi = -log(pr) / 3.0;
        hp.lpoi = log(hp.poi);
        poi_is_init = 0;
    }
    if (use_rate_HP) {
        // get_rate_HP (:210-213): Gamma(1.2 + 2K, scale 1/(0.1 + sum rates)) = (Gamma(1.2) + Gamma(2K)) * scale
        double ga, gb;
        rng.draw(it, 2, lane, ga, gb);
        const double eL = -log(warp_prod(lane < L.K ? ga * gb : 1.0));
        const double fracL = warp_gamma_mt(1.2, rng, it, 8, lane);
        hp.gL = (eL + fracL) / (0.1 + L.sumr);
        rng.draw(it, 3, lane, ga, gb);
        const double eM = -log(warp_prod(lane < M.K ? ga * gb : 1.0));
        const double fracM = warp_gamma_mt(1.2, rng, it, 160, lane);
        hp.gM = (eM + fracM) / (0.1 + M.sumr);
        hp.lgL = log(hp.gL); hp.lgM = log(hp.gM);
    }
    GibbsOut o;
    o.hp = hp; o.poi_is_init = poi_is_init;
    o.priorA = frozen ? -INFINITY : full_prior(L, M, hp, d, poiA);      // :291 with gibbs == 1 (:313) stores -inf
    return o;
}

// log-rates follow the rates by addition inside the loop; every LR_RESYNC iterations they are re-derived from the rates
// (at fixed iteration numbers, so that a chain does not depend on how a run is split into launches or sampled)
// The COMPACT build calls the cold functions through these by-reference wrappers ON PURPOSE: the escaping addresses make
// the compiler keep the two Sides and the ChainRegs in local memory (L1-resident) instead of registers, and the kernel is
// capped at 128 registers (4 CTAs of 4 warps per SM).  With thousands of chains resident the extra warps hide more latency
// than the local loads cost (B200, 4096 / 16384 chains: 1.67 / 1.87 G it/s at 128 registers, 1.42 / 1.67 at the 152 the
// compiler would take, 1.62 / 1.92 at 96); the SPECIALISED build wants the opposite and calls the by-value functions.
__device__ __noinline__ void gibbs_step_ref(const Side& L, const Side& M, ChainRegs& c, const DataView& d, int sample_poisson,
                                            int use_rate_HP, const Rng& rng, long long it, bool frozen, int lane) {
    const GibbsOut g = gibbs_step(L, M, c.hp, c.poiA, c.poi_is_init, d, sample_poisson, use_rate_HP, rng, it, frozen, lane);
    c.hp = g.hp; c.priorA = g.priorA; c.poi_is_init = g.poi_is_init;
}
__device__ __noinline__ void write_record_ref(double* rec, long long it, const Side& L, const Side& M, const ChainRegs& c, const DataView& d,
                                              int lane, bool with_adequacy) {
    write_record(rec, it, L, M, c.hp, d, c.priorA, c.poiA, c.consistent, c.poi_is_init, c.beta, lane, with_adequacy);
}

#define LR_RESYNC 1024
__device__ __forceinline__ void resync_log_rates(Side& L, Side& M, int lane) {
    const double a = ool_log(L.r), b = ool_log(M.r);      // inactive lanes hold 0: -inf, discarded
    L.lr = lane < L.K ? a : 0.0;
    M.lr = lane < M.K ? b : 0.0;
}

// ------------------------------------------------------------------------------------------------
// K3: the chains.  SPEC = warp-specialised build (blockDim = 128: chain warp + 3 producer warps, one chain per CTA);
// otherwise compact build (one warp per chain, any blockDim that is a multiple of 32).
// ------------------------------------------------------------------------------------------------
// MODE 0  compact: one warp per chain, any blockDim that is a multiple of 32
// MODE 1  specialised, one chain per CTA of 4 warps: chain warp + 3 producer warps (2 CTAs per SM at ~210 registers)
// MODE 2  specialised, four chains per CTA of 8 warps: warpgroup 0 = 4 chain warps, warpgroup 1 = their 4 producers (one
//         each, which keeps up: ~390 cycles per produced iteration against ~900 consumed); setmaxnreg moves registers from
//         the producers (72) to the chain warps (184), 2 CTAs = 8 chains per SM
// last iteration (exclusive) of this launch for one chain (see lr_chains_run for the sequence of passes)
__device__ __forceinline__ long long chain_end(const RunParams& P, const ChainState* S, long long it0) {
    long long it1 = (P.it_begin >= 0 ? P.it_begin : it0) + P.n_iter;
    if (P.cont_mode == 1) { const long long su = S->solo_until; it1 = su > it0 ? (su < it1 ? su : it1) : it0; }
    return it1;
}

template <int MODE>
__global__ void __launch_bounds__(MODE == 2 ? 256 : 128, MODE == 0 ? 4 : (MODE == 2 ? 2 : 1)) k3_run_kernel(const RunParams P) {
    constexpr bool SPEC = MODE != 0;
    constexpr bool C = !SPEC;
    constexpr int CPB = MODE == 2 ? 4 : 1;             // chains per CTA
    constexpr int PPC = MODE == 2 ? 1 : 3;             // producer warps per chain
    constexpr int DEPTH = MODE == 2 ? 3 : 6;           // ring slots (batches in flight) per chain
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const bool producer = SPEC && warp >= CPB;
    const int slot_in_cta = !SPEC ? 0 : (producer ? (warp - CPB) / PPC : warp);
    const int chain = SPEC ? (int)blockIdx.x * CPB + slot_in_cta : (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);

    extern __shared__ __align__(16) unsigned char ring_raw[];
    Ring<DEPTH>* ring_p = nullptr;
    const lr_chain_config& cfg = P.cfg;
    const LoopConsts& K = P.lc;
    if constexpr (SPEC) {
        Ring<DEPTH>* rings = reinterpret_cast<Ring<DEPTH>*>(ring_raw);
        if (threadIdx.x < CPB * DEPTH) { rings[threadIdx.x / DEPTH].full[threadIdx.x % DEPTH] = 0ull; rings[threadIdx.x / DEPTH].done[threadIdx.x % DEPTH] = 0ull; }
        __syncthreads();
        ring_p = rings + slot_in_cta;
        if (producer) {
            // ---------------- producer warp `pid` of this chain: batches b = pid, pid + PPC, ... of RING_BATCH iterations each.
            // (The whole producer role sits inside this branch and returns: the register re-balancing below applies to
            // code that only one of the two warpgroups can reach.)
            if constexpr (MODE == 2) reg_dealloc<72>();
            if (chain >= P.n_chains) return;
            const ChainState* S = P.st + chain;
            Rng rng; rng.k0 = P.k0; rng.k1 = P.k1; rng.chain = S->chain_id;
            const long long it0 = S->it;                  // the chain warp rewrites S->it only at the very end
            const long long n_own = chain_end(P, S, it0) - it0;          // what this pass does of this launch for this chain
            Ring<DEPTH>& ring = *ring_p;
            const int pid = (warp - CPB) % PPC;
            const long long n_batches = (n_own + RING_BATCH - 1) / RING_BATCH;
            int s = pid % DEPTH;                    // slot of batch b is b % DEPTH, tracked without a division
            for (long long b = pid; b < n_batches; b += PPC) {
                // wait until the previous occupant of the slot (batch b - DEPTH) has been consumed; back off while
                // waiting so that the polling does not compete with the chain warp for the shared-memory pipe
                while ((long long)ld_acquire_cta(&ring.done[s]) < b - DEPTH + 1) __nanosleep(200);
                const long long j0 = b * RING_BATCH;
#pragma unroll 1
                for (int i = 0; i < RING_BATCH; ++i) {
                    if (j0 + i < n_own) ring_store(ring.it[s][i], make_draws<false>(rng, it0 + j0 + i, lane, K), lane);
                }
                __syncwarp();
                if (lane == 0) st_release_cta(&ring.full[s], (unsigned long long)(b + 1));
                s += PPC; if (s >= DEPTH) s -= DEPTH;
            }
            return;
        } else {
            if constexpr (MODE == 2) reg_alloc<184>();
        }
    }
    if (chain >= P.n_chains) return;
    ChainState* S = P.st + chain;
    Rng rng; rng.k0 = P.k0; rng.k1 = P.k1; rng.chain = S->chain_id;
    const long long it0 = S->it, it_begin = P.it_begin >= 0 ? P.it_begin : it0, it1 = chain_end(P, S, it0);
    if (it0 >= it1) return;                       // continuation pass: nothing left for this chain in this pass

    // ---------------- the chain warp
    const DataView d = make_view(P.tab, P.cst, S->rep, P.nb, P.s0f, P.start_time, P.end_time);
    Side L, M;
    load_sides(S, L, M, lane);
    side_stats(L, d, T_AB, T_BB, lane);
    side_stats(M, d, T_AD, T_BD, lane);
    ChainRegs c;
    c.hp.gL = S->gL; c.hp.gM = S->gM; c.hp.lgL = log(c.hp.gL); c.hp.lgM = log(c.hp.gM); c.hp.poi = S->poi; c.hp.lpoi = log(c.hp.poi);
    c.priorA = S->priorA; c.poiA = S->poiA; c.beta = S->beta; c.poi_is_init = S->poi_is_init; c.consistent = (int)S->consistent;
    Counters n;
#pragma unroll
    for (int i = 0; i < 8; ++i) n.v[i] = 0u;
    const bool frozen = (d.end_time - d.start_time) <= LR_MIN_DT;      // guard :290 rejects everything

    const long long s_every = P.sample_every > 0 ? P.sample_every : 1;
    long long next_sample = P.records != nullptr ? (it0 + s_every - 1) / s_every * s_every : it1;   // no 64-bit division in the loop
    long long next_resync = (it0 + LR_RESYNC - 1) / LR_RESYNC * LR_RESYNC;
    long long next_event = next_resync < next_sample ? next_resync : next_sample;
    // records of this launch written before it0 (by the team build, when this is the continuation pass)
    const long long rec_done = (it0 + s_every - 1) / s_every - (it_begin + s_every - 1) / s_every;
    double* rec = P.records + ((size_t)rec_done * P.n_chains + chain) * LR_REC_DOUBLES;
    int slot = 0, in_batch = 0;
    long long batch = 0;

    for (long long it = it0; it < it1; ++it) {
        Draws q;
        if constexpr (SPEC) {
            Ring<DEPTH>& R = *ring_p;
            if (in_batch == 0) { while (ld_acquire_cta(&R.full[slot]) != (unsigned long long)(batch + 1)) { } }
            q = ring_load(R.it[slot][in_batch], lane);
            if (++in_batch == RING_BATCH || it + 1 == it1) {
                __syncwarp();
                if (lane == 0) st_release_cta(&R.done[slot], (unsigned long long)(batch + 1));
                in_batch = 0; ++batch; if (++slot == DEPTH) slot = 0;
            }
        }
        else q = make_draws<true>(rng, it, lane, K, L.K, M.K);

        const int kind = q.kind >> 1;
        const bool birth = (q.kind & 1) != 0;
        if (kind <= DK_BLOCK_MOVE) {
            if constexpr (C) {
                Side& cur = birth ? L : M;
                if (!block_step<C>(cur, side_view(c.hp, birth), c, n, d, cfg, q, frozen, lane))
                    run_slow(cur, birth ? M : L, side_view(c.hp, birth), c, n, d, cfg, q, frozen, lane);
            } else {
                if (birth) { if (!block_step<C>(L, side_view(c.hp, true), c, n, d, cfg, q, frozen, lane)) run_slow(L, M, side_view(c.hp, true), c, n, d, cfg, q, frozen, lane); }
                else { if (!block_step<C>(M, side_view(c.hp, false), c, n, d, cfg, q, frozen, lane)) run_slow(M, L, side_view(c.hp, false), c, n, d, cfg, q, frozen, lane); }
            }
        } else if (kind != DK_GIBBS) {
            n.v[5]++;
            if constexpr (C) {
                Side& cur = birth ? L : M;
                const Side& oth = birth ? M : L;
                if (!rj_step<C>(cur, oth, side_view(c.hp, birth), c, n, d, q, frozen, lane))
                    run_slow(cur, oth, side_view(c.hp, birth), c, n, d, cfg, q, frozen, lane);
            } else {
                if (birth) { if (!rj_step<C>(L, M, side_view(c.hp, true), c, n, d, q, frozen, lane)) run_slow(L, M, side_view(c.hp, true), c, n, d, cfg, q, frozen, lane); }
                else { if (!rj_step<C>(M, L, side_view(c.hp, false), c, n, d, q, frozen, lane)) run_slow(M, L, side_view(c.hp, false), c, n, d, cfg, q, frozen, lane); }
            }
        } else {
            n.v[6]++;
            if constexpr (C) {
                gibbs_step_ref(L, M, c, d, cfg.poisson_prior == 0.0 ? 1 : 0, cfg.use_rate_HP, rng, it, frozen, lane);
            } else {
                const GibbsOut g = gibbs_step(L, M, c.hp, c.poiA, c.poi_is_init, d, cfg.poisson_prior == 0.0 ? 1 : 0, cfg.use_rate_HP, rng, it, frozen, lane);
                c.hp = g.hp; c.priorA = g.priorA; c.poi_is_init = g.poi_is_init;
            }
            c.consistent = 1;
            n.v[1]++;
        }

        if (it == next_event) {                     // one comparison per iteration for the two rare events
            if (it == next_resync) { resync_log_rates(L, M, lane); next_resync += LR_RESYNC; }
            if (it == next_sample) {                // it % sample_every == 0 (:321)
                if constexpr (C) write_record_ref(rec, it, L, M, c, d, lane, P.with_adequacy != 0);
                else write_record(rec, it, L, M, c.hp, d, c.priorA, c.poiA, c.consistent, c.poi_is_init, c.beta, lane, P.with_adequacy != 0);
                rec += (size_t)P.n_chains * LR_REC_DOUBLES;
                next_sample += s_every;
            }
            next_event = next_resync < next_sample ? next_resync : next_sample;
        }
    }

    store_sides(S, L, M, lane);
    if (lane == 0) {
        S->it = it1;
        S->priorA = c.priorA; S->poiA = c.poiA; S->gL = c.hp.gL; S->gM = c.hp.gM; S->poi = c.hp.poi; S->poi_is_init = c.poi_is_init; S->consistent = (unsigned)c.consistent;
        S->counters[0] += it1 - it0;
#pragma unroll
        for (int i = 1; i < 8; ++i) S->counters[i] += (long long)n.v[i];
    }
}

#include "k3_team.cuh"

// initial state (:580-583) and initial bookkeeping (:220-230)
__global__ void k3_init_kernel(ChainState* st, int n_chains, const int* __restrict__ rep_of_chain, long long chain_id0,
                               uint32_t k0, uint32_t k1, double start_time, double poisson_prior_cfg, double beta) {
    const int lane = threadIdx.x & 31;
    const int chain = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
    if (chain >= n_chains) return;
    ChainState* S = st + chain;
    Rng rng; rng.k0 = k0; rng.k1 = k1; rng.chain = (uint32_t)(chain_id0 + chain);
    double ua, ub;
    rng.draw(-1, 15, lane, ua, ub);
    // Gamma(shape 2, scale 2) = -2 log(u1 u2)
    const double l0 = -2.0 * log(__shfl_sync(0xffffffffu, ua, 0) * __shfl_sync(0xffffffffu, ub, 0));
    const double m0 = -2.0 * log(__shfl_sync(0xffffffffu, ua, 1) * __shfl_sync(0xffffffffu, ub, 1));
    S->rL[lane] = lane == 0 ? l0 : 0.0; S->lrL[lane] = lane == 0 ? log(l0) : 0.0; S->tL[lane] = lane == 0 ? start_time : 0.0;
    S->rM[lane] = lane == 0 ? m0 : 0.0; S->lrM[lane] = lane == 0 ? log(m0) : 0.0; S->tM[lane] = lane == 0 ? start_time : 0.0;
    if (lane == 0) {
        S->it = 0;
        for (int i = 0; i < LR_NCOUNTERS; ++i) S->counters[i] = 0;
        for (int i = 0; i < 6; ++i) S->team[i] = 0;
        S->solo_until = TEAM_INITIAL_SOLO; S->win_iters = 0u; S->win_commits = 0u; S->solo_span = 0;   // burn-in: nearly every proposal moves the state
        S->K_l = 1; S->K_m = 1; S->rep = rep_of_chain ? rep_of_chain[chain] : 0;
        S->chain_id = rng.chain; S->consistent = 0;     // the initial prior uses Gamma rate 2 (:227), the loop rate 1
        const double poi = poisson_prior_cfg == 0.0 ? 1.0 : poisson_prior_cfg;       // :220-221
        S->poi = poi; S->poi_is_init = 1;
        S->gL = 1.0; S->gM = 1.0;                                                     // :222
        const double lpoi = log(poi);
        const double poiA = 2.0 * (1.0 * lpoi - poi - 0.0);                            // :229, K = 1 on both sides
        // prior_gamma defaults a=2, b=2 (:227): 2 log 2 + log x - 2 x per rate; no shifts yet (:228)
        const double lg2 = log(2.0);
        S->priorA = (2.0 * lg2 + log(l0) - 2.0 * l0) + (2.0 * lg2 + log(m0) - 2.0 * m0) + poiA;
        S->poiA = poiA;
        S->beta = beta;
    }
}

// record -> state (tests, checkpoint/resume).  priorA becomes the consistent prior of the state.
__global__ void k3_set_state_kernel(ChainState* st, int n_chains, const double* __restrict__ recs, const double* tab,
                                    const double* cst, int nb, int s0f, double start_time, double end_time) {
    const int lane = threadIdx.x & 31;
    const int chain = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
    if (chain >= n_chains) return;
    ChainState* S = st + chain;
    const double* rec = recs + (size_t)chain * LR_REC_DOUBLES;
    const int Kl = (int)rec[5], Km = (int)rec[6];
    const double rl = rec[16 + lane], rm = rec[80 + lane];
    S->rL[lane] = lane < Kl ? rl : 0.0; S->lrL[lane] = lane < Kl ? log(rl) : 0.0;
    S->tL[lane] = lane == 0 ? start_time : (lane < Kl ? rec[48 + lane] : 0.0);
    S->rM[lane] = lane < Km ? rm : 0.0; S->lrM[lane] = lane < Km ? log(rm) : 0.0;
    S->tM[lane] = lane == 0 ? start_time : (lane < Km ? rec[112 + lane] : 0.0);
    __syncwarp();
    const DataView d = make_view(tab, cst, S->rep, nb, s0f, start_time, end_time);
    Side L, M;
    L.K = Kl; M.K = Km;
    L.r = S->rL[lane]; L.lr = S->lrL[lane]; L.t = S->tL[lane];
    M.r = S->rM[lane]; M.lr = S->lrM[lane]; M.t = S->tM[lane];
    side_stats(L, d, T_AB, T_BB, lane); side_sums(L, lane);
    side_stats(M, d, T_AD, T_BD, lane); side_sums(M, lane);
    Hyper hp;
    hp.gL = rec[7]; hp.gM = rec[8]; hp.poi = rec[9]; hp.lgL = log(hp.gL); hp.lgM = log(hp.gM); hp.lpoi = log(hp.poi);
    const double poiA = poisson_prior(Kl, hp.poi, hp.lpoi, c_lnfact) + poisson_prior(Km, hp.poi, hp.lpoi, c_lnfact);
    if (lane == 0) {
        S->it = (long long)rec[0];
        S->K_l = Kl; S->K_m = Km;
        S->gL = hp.gL; S->gM = hp.gM; S->poi = hp.poi; S->poi_is_init = (int)rec[13];
        S->poiA = poiA;
        S->priorA = full_prior(L, M, hp, d, poiA);
        S->consistent = 1;
        S->solo_until = 0; S->win_iters = 0u; S->win_commits = 0u; S->solo_span = 0;
    }
}

__global__ void k3_get_state_kernel(const ChainState* st, int n_chains, double* __restrict__ recs, const double* tab,
                                    const double* cst, int nb, int s0f, double start_time, double end_time) {
    const int lane = threadIdx.x & 31;
    const int chain = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
    if (chain >= n_chains) return;
    const ChainState* S = st + chain;
    const DataView d = make_view(tab, cst, S->rep, nb, s0f, start_time, end_time);
    Side L, M;
    load_sides(S, L, M, lane);
    side_stats(L, d, T_AB, T_BB, lane); side_sums(L, lane);
    side_stats(M, d, T_AD, T_BD, lane); side_sums(M, lane);
    Hyper hp;
    hp.gL = S->gL; hp.gM = S->gM; hp.poi = S->poi; hp.lgL = log(hp.gL); hp.lgM = log(hp.gM); hp.lpoi = log(hp.poi);
    write_record(recs + (size_t)chain * LR_REC_DOUBLES, S->it, L, M, hp, d, S->priorA, S->poiA, (int)S->consistent, S->poi_is_init, S->beta, lane, true);
}

// K2: one warp per state
__global__ void k2_state_eval_kernel(int n, const int* __restrict__ rep, const int* __restrict__ K_l, const int* __restrict__ K_m,
                                     const double* __restrict__ Lr, const double* __restrict__ Mr,
                                     const double* __restrict__ tL, const double* __restrict__ tM,
                                     const double* __restrict__ gamma_rate, const double* __restrict__ poi_lambda,
                                     const double* tab, const double* cst, int nb, int s0f, double start_time, double end_time,
                                     double* __restrict__ lik, double* __restrict__ prior_rates, double* __restrict__ prior_poi,
                                     double* __restrict__ adequacy) {
    const int lane = threadIdx.x & 31;
    const int i = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
    if (i >= n) return;
    const DataView d = make_view(tab, cst, rep ? rep[i] : 0, nb, s0f, start_time, end_time);
    Side L, M;
    L.K = K_l[i]; M.K = K_m[i];
    const bool inL = lane < L.K && lane < LR_KMAX, inM = lane < M.K && lane < LR_KMAX;
    L.r = inL ? Lr[(size_t)i * LR_KMAX + lane] : 0.0; L.lr = inL ? log(L.r) : 0.0;
    L.t = lane == 0 ? start_time : (inL ? tL[(size_t)i * LR_KMAX + lane] : 0.0);
    M.r = inM ? Mr[(size_t)i * LR_KMAX + lane] : 0.0; M.lr = inM ? log(M.r) : 0.0;
    M.t = lane == 0 ? start_time : (inM ? tM[(size_t)i * LR_KMAX + lane] : 0.0);
    side_stats(L, d, T_AB, T_BB, lane); side_sums(L, lane);
    side_stats(M, d, T_AD, T_BD, lane); side_sums(M, lane);
    Hyper hp;
    hp.gL = gamma_rate ? gamma_rate[2 * i] : 1.0; hp.gM = gamma_rate ? gamma_rate[2 * i + 1] : 1.0;
    hp.poi = poi_lambda ? poi_lambda[i] : 1.0;
    hp.lgL = log(hp.gL); hp.lgM = log(hp.gM); hp.lpoi = log(hp.poi);
    double adq[3];
    if (adequacy) adequacy3(L, M, d, lane, adq);
    if (lane == 0) {
        if (lik) lik[i] = d.C + L.lik + M.lik;
        if (prior_rates) prior_rates[i] = full_prior(L, M, hp, d, 0.0);
        if (prior_poi) prior_poi[i] = poisson_prior(L.K, hp.poi, hp.lpoi, c_lnfact) + poisson_prior(M.K, hp.poi, hp.lpoi, c_lnfact);
        if (adequacy) { adequacy[3 * i] = adq[0]; adequacy[3 * i + 1] = adq[1]; adequacy[3 * i + 2] = adq[2]; }
    }
}

// K2b: one RJ proposal per explicit state with explicit draws (parity entry point; one warp per state).
// kind 2 = add-shift on segment idx at t_idx + u_t * gap with Beta variate u_beta; kind 3 = remove interior shift idx.
__global__ void k2_proposal_eval_kernel(int n, const int* __restrict__ rep, const int* __restrict__ K_l, const int* __restrict__ K_m,
                                        const double* __restrict__ Lr, const double* __restrict__ Mr,
                                        const double* __restrict__ tL, const double* __restrict__ tM,
                                        const double* __restrict__ gamma_rate, const double* __restrict__ poi_lambda,
                                        const double* __restrict__ beta_in, const double* __restrict__ poiA_in,
                                        const int* __restrict__ side, const int* __restrict__ kind, const int* __restrict__ idx,
                                        const double* __restrict__ u_t, const double* __restrict__ u_beta,
                                        const int* __restrict__ mult_on, const double* __restrict__ mult_u,
                                        const double* tab, const double* cst, int nb, int s0f, double start_time, double end_time,
                                        int* __restrict__ ok_out, int* __restrict__ K_new, double* __restrict__ rates_new,
                                        double* __restrict__ times_new, double* __restrict__ hasting_out, double* __restrict__ x_out) {
    const int lane = threadIdx.x & 31;
    const int i = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
    if (i >= n) return;
    const DataView d = make_view(tab, cst, rep ? rep[i] : 0, nb, s0f, start_time, end_time);
    Side L, M;
    L.K = K_l[i]; M.K = K_m[i];
    const bool inL = lane < L.K && lane < LR_KMAX, inM = lane < M.K && lane < LR_KMAX;
    L.r = inL ? Lr[(size_t)i * LR_KMAX + lane] : 0.0; L.lr = inL ? log(L.r) : 0.0;
    L.t = lane == 0 ? start_time : (inL ? tL[(size_t)i * LR_KMAX + lane] : 0.0);
    M.r = inM ? Mr[(size_t)i * LR_KMAX + lane] : 0.0; M.lr = inM ? log(M.r) : 0.0;
    M.t = lane == 0 ? start_time : (inM ? tM[(size_t)i * LR_KMAX + lane] : 0.0);
    side_stats(L, d, T_AB, T_BB, lane);
    side_stats(M, d, T_AD, T_BD, lane);
    Hyper hp;
    hp.gL = gamma_rate ? gamma_rate[2 * i] : 1.0; hp.gM = gamma_rate ? gamma_rate[2 * i + 1] : 1.0;
    hp.poi = poi_lambda ? poi_lambda[i] : 1.0;
    hp.lgL = log(hp.gL); hp.lgM = log(hp.gM); hp.lpoi = log(hp.poi);
    const bool birth = side[i] != 0;
    const Side& cur = birth ? L : M;
    const Side& oth = birth ? M : L;
    Draws q;
    q.u_acc = 0.5; q.thr_hi = 0.0; q.thr_lo = 0.0; q.m = 1.0; q.dlt = 0.0;
    Side nw;
    double hasting = 0.0, poiN = 0.0, x = 0.0;
    bool cap = false, ok = true;
    if (kind[i] == 0) {
        // update_multiplier_freq (:165-176) with the given Bernoulli mask and uniforms: m = exp(2 ln(1.1) (u - .5)) on the
        // touched rates, Hastings = sum log m; the acceptance ratio exactly as block_step forms it
        const bool on = lane < cur.K && lane < LR_KMAX;
        const bool touched = on && mult_on[(size_t)i * LR_KMAX + lane] != 0;
        const double dl = touched ? LR_LN_MULT * (mult_u[(size_t)i * LR_KMAX + lane] - 0.5) : 0.0;
        const double rn = cur.r * exp_small(dl);
        const SideView v = side_view(hp, birth);
        const double b = beta_in ? beta_in[i] : 1.0;
        x = warp_sum((b * cur.A + 2.0) * dl - (b * cur.B + v.g_cur) * (rn - cur.r));
        hasting = warp_sum(dl);
        nw = cur; nw.r = rn; nw.lr = cur.lr + dl;
    } else {
        q.kind = ((kind[i] == 2 ? DK_RJ_ADD : DK_RJ_REMOVE) << 1) | (birth ? 1 : 0);
        // the index draws that select exactly segment / shift idx (propose_add: (int)(u K); propose_remove: 1 + (int)(u (K-1)))
        q.u_idx = kind[i] == 2 ? ((double)idx[i] + 0.5) / (double)cur.K : ((double)(idx[i] - 1) + 0.5) / (double)(cur.K > 1 ? cur.K - 1 : 1);
        q.u_t = u_t[i];
        const double ub = u_beta[i];
        q.w = log((1.0 - ub) / ub);                                                           // :41-42
        q.ln_beta = (LR_SHAPE_BETA - 1.0) * (log(ub) + log1p(-ub)) - LR_BETA_NORM;            // beta.logpdf(u; 10, 10), :22-23
        ok = rj_propose<false>(cur, oth, side_view(hp, birth), hp, beta_in ? beta_in[i] : 1.0, poiA_in[i], d, q, lane, nw, hasting, poiN, x, cap);
    }
    if (lane == 0) { ok_out[i] = ok ? 1 : 0; K_new[i] = ok ? nw.K : cur.K; hasting_out[i] = ok ? hasting : 0.0; x_out[i] = ok ? x : 0.0; }
    if (lane < LR_KMAX) {
        rates_new[(size_t)i * LR_KMAX + lane] = (ok && lane < nw.K) ? nw.r : 0.0;
        times_new[(size_t)i * LR_KMAX + lane] = (ok && lane < nw.K) ? (lane == 0 ? start_time : nw.t) : 0.0;
    }
}

__global__ void k3_set_beta_kernel(ChainState* st, int n, const double* beta) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) st[i].beta = beta[i];
}

// ------------------------------------------------------------------------------------------------
// tempered ensembles (Metropolis-coupled MCMC).  New: the reference has no tempering (SURVEY A-15); a chain with
// beta = 1 is the reference's chain, heated chains raise the likelihood to the power beta < 1.
// ------------------------------------------------------------------------------------------------
// (likelihood, beta) of every chain: the 16 bytes per chain a swap round exchanges
__global__ void k3_swap_info_kernel(const ChainState* st, int n_chains, double* __restrict__ info, const double* tab, const double* cst,
                                    int nb, int s0f, double start_time, double end_time) {
    const int lane = threadIdx.x & 31;
    const int chain = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
    if (chain >= n_chains) return;
    const ChainState* S = st + chain;
    const DataView d = make_view(tab, cst, S->rep, nb, s0f, start_time, end_time);
    Side L, M;
    load_sides(S, L, M, lane);
    side_stats(L, d, T_AB, T_BB, lane); side_sums(L, lane);
    side_stats(M, d, T_AD, T_BD, lane); side_sums(M, lane);
    if (lane == 0) { info[2 * chain] = d.C + L.lik + M.lik; info[2 * chain + 1] = S->beta; }
}

// One swap round (lr_swap_round): beta and the swap counters of K3's chain state
__global__ void k3_swap_apply_kernel(ChainState* st, int n_local, const double* __restrict__ info_all, long long table_first,
                                     long long n_all, long long first, int ladder, unsigned long long round, uint32_t k0, uint32_t k1) {
    const int lane = threadIdx.x & 31;
    const int local = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
    if (local >= n_local) return;
    lr_swap_round(info_all, table_first, n_all, first + local, ladder, round, k0, k1, lane, [&](bool paired, bool accept, double beta_p) {
        ChainState* S = st + local;
        if (paired) {
            S->counters[8] += 1;
            if (accept) { S->counters[9] += 1; S->beta = beta_p; }
        }
    });
}

int upload_lnfact() {
    static bool done[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 64 && done[dev]) return LR_OK;
    double t[LR_SLOTS + 2];
    t[0] = 0.0;
    for (int k = 1; k < LR_SLOTS + 2; ++k) t[k] = t[k - 1] + log((double)k);     // sum(log(arange(1,k+1))) (:199)
    LR_CUDA(cudaMemcpyToSymbol(c_lnfact, t, sizeof(t)));
    if (dev < 64) done[dev] = true;
    return LR_OK;
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" int lr_dataset_create(lr_handle_t h, int32_t n_rep, int32_t n_bins, int32_t model_BDI,
                                 double start_time, double end_time,
                                 const int64_t* d_sp, const int64_t* d_ex, const double* d_br,
                                 const int64_t* d_ex_dead, const double* d_br_dead, void* stream, lr_dataset_t* out) {
    LR_REQUIRE(h && out && d_sp && d_ex && d_br, "lr_dataset_create: null pointer");
    LR_REQUIRE(n_rep >= 1 && n_bins >= 1, "lr_dataset_create: bad sizes");
    LR_REQUIRE(model_BDI >= 0 && model_BDI <= 3, "lr_dataset_create: model_BDI must be 0..3");
    LR_REQUIRE(model_BDI != 3 || (d_ex_dead && d_br_dead), "lr_dataset_create: model_BDI 3 needs the extinct-only statistics");
    LR_REQUIRE(end_time > start_time, "lr_dataset_create: end_time must exceed start_time");
    LR_REQUIRE(start_time >= 0.0, "lr_dataset_create: negative start_time is not supported (the reference's rate index breaks there too)");
    LR_REQUIRE((long long)floor(end_time) - (long long)floor(start_time) == n_bins,
               "lr_dataset_create: n_bins must equal floor(end_time) - floor(start_time) (LiteRateForward.py:519, :125-135)");
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    int rc = upload_lnfact();
    if (rc != LR_OK) return rc;
    lr_dataset_t ds = new lr_dataset_s();
    ds->h = h; ds->n_rep = n_rep; ds->n_bins = n_bins; ds->model = model_BDI;
    ds->start_time = start_time; ds->end_time = end_time; ds->s0f = (int)floor(start_time);
    ds->tab = nullptr; ds->cst = nullptr;
    ds->last.s = st; ds->last.valid = 1;
    // stream-ordered allocation: creating/destroying datasets and chains never synchronises the device, so a pipeline can
    // set up batch k+1 while the chains of batch k are still running (cudaFree would wait for them)
    cudaError_t e = cudaMallocAsync((void**)&ds->tab, (size_t)n_rep * LR_NTAB * (n_bins + 1) * sizeof(double), st);
    if (e == cudaSuccess) e = cudaMallocAsync((void**)&ds->cst, (size_t)n_rep * LR_NCST * sizeof(double), st);
    if (e != cudaSuccess) {
        lr_set_error("lr_dataset_create: cudaMallocAsync failed: %s", cudaGetErrorString(e));
        if (ds->tab) cudaFreeAsync(ds->tab, st);
        delete ds;
        return LR_ERR_NOMEM;
    }
    k2_build_tables<<<n_rep, 64, 0, st>>>((const long long*)d_sp, (const long long*)d_ex, d_br, (const long long*)d_ex_dead,
                                           d_br_dead, n_bins, model_BDI, ds->tab, ds->cst);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    *out = ds;
    return LR_OK;
}

extern "C" int lr_dataset_create_host(lr_handle_t h, int32_t n_rep, int32_t n_bins, int32_t model_BDI,
                                      double start_time, double end_time,
                                      const int64_t* h_sp, const int64_t* h_ex, const double* h_br,
                                      const int64_t* h_ex_dead, const double* h_br_dead, lr_dataset_t* out) {
    LR_REQUIRE(h && out && h_sp && h_ex && h_br, "lr_dataset_create_host: null pointer");
    LR_REQUIRE(n_rep >= 1 && n_bins >= 1, "lr_dataset_create_host: bad sizes");
    LR_CUDA(cudaSetDevice(h->device));
    const size_t cnt = (size_t)n_rep * n_bins;
    const bool dead = h_ex_dead && h_br_dead;
    const size_t bytes = cnt * 8 * (dead ? 5 : 3);
    int rc = lr_ws_acquire(h, bytes, h->stream);
    if (rc != LR_OK) return rc;
    char* w = (char*)h->ws;
    LR_CUDA(cudaMemcpyAsync(w, h_sp, cnt * 8, cudaMemcpyHostToDevice, h->stream));
    LR_CUDA(cudaMemcpyAsync(w + cnt * 8, h_ex, cnt * 8, cudaMemcpyHostToDevice, h->stream));
    LR_CUDA(cudaMemcpyAsync(w + cnt * 16, h_br, cnt * 8, cudaMemcpyHostToDevice, h->stream));
    if (dead) {
        LR_CUDA(cudaMemcpyAsync(w + cnt * 24, h_ex_dead, cnt * 8, cudaMemcpyHostToDevice, h->stream));
        LR_CUDA(cudaMemcpyAsync(w + cnt * 32, h_br_dead, cnt * 8, cudaMemcpyHostToDevice, h->stream));
    }
    rc = lr_dataset_create(h, n_rep, n_bins, model_BDI, start_time, end_time, (const int64_t*)w, (const int64_t*)(w + cnt * 8),
                           (const double*)(w + cnt * 16), dead ? (const int64_t*)(w + cnt * 24) : nullptr,
                           dead ? (const double*)(w + cnt * 32) : nullptr, h->stream, out);
    if (rc != LR_OK) return rc;
    LR_CUDA(cudaStreamSynchronize(h->stream));
    return LR_OK;
}

extern "C" int lr_dataset_create_general_host(lr_handle_t h, int32_t n_rep, int32_t n_bins, int32_t model_tag, double start_time, double end_time,
                                              const double* h_A_birth, const double* h_B_birth, const double* h_A_death, const double* h_B_death,
                                              const double* h_x_birth, const double* h_x_death, const double* h_C, lr_dataset_t* out) {
    LR_REQUIRE(h && out && h_A_birth && h_B_birth && h_A_death && h_B_death && h_x_birth && h_x_death, "lr_dataset_create_general_host: null pointer");
    LR_REQUIRE(n_rep >= 1 && n_bins >= 1, "lr_dataset_create_general_host: bad sizes");
    LR_REQUIRE(model_tag >= 0 && model_tag <= 3, "lr_dataset_create_general_host: model_tag must be 0..3 (what lr_chain_config.model_BDI will be checked against)");
    LR_REQUIRE(end_time > start_time && start_time >= 0.0, "lr_dataset_create_general_host: need 0 <= start_time < end_time");
    LR_REQUIRE((long long)floor(end_time) - (long long)floor(start_time) == n_bins,
               "lr_dataset_create_general_host: n_bins must equal floor(end_time) - floor(start_time)");
    LR_CUDA(cudaSetDevice(h->device));
    int rc = upload_lnfact();
    if (rc != LR_OK) return rc;
    const size_t cnt = (size_t)n_rep * n_bins;
    rc = lr_ws_acquire(h, (6 * cnt + n_rep) * sizeof(double), h->stream);
    if (rc != LR_OK) return rc;
    double* w = (double*)h->ws;
    const double* src[6] = {h_A_birth, h_B_birth, h_A_death, h_B_death, h_x_birth, h_x_death};
    for (int k = 0; k < 6; ++k) LR_CUDA(cudaMemcpyAsync(w + k * cnt, src[k], cnt * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    if (h_C) LR_CUDA(cudaMemcpyAsync(w + 6 * cnt, h_C, (size_t)n_rep * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    lr_dataset_t ds = new lr_dataset_s();
    ds->h = h; ds->n_rep = n_rep; ds->n_bins = n_bins; ds->model = model_tag;
    ds->start_time = start_time; ds->end_time = end_time; ds->s0f = (int)floor(start_time);
    ds->tab = nullptr; ds->cst = nullptr;
    ds->last.s = h->stream; ds->last.valid = 1;
    cudaError_t e = cudaMallocAsync((void**)&ds->tab, (size_t)n_rep * LR_NTAB * (n_bins + 1) * sizeof(double), h->stream);
    if (e == cudaSuccess) e = cudaMallocAsync((void**)&ds->cst, (size_t)n_rep * LR_NCST * sizeof(double), h->stream);
    if (e != cudaSuccess) {
        lr_set_error("lr_dataset_create_general_host: cudaMallocAsync failed: %s", cudaGetErrorString(e));
        if (ds->tab) cudaFreeAsync(ds->tab, h->stream);
        delete ds;
        return LR_ERR_NOMEM;
    }
    k2_build_tables_general<<<n_rep, 64, 0, h->stream>>>(w, w + cnt, w + 2 * cnt, w + 3 * cnt, w + 4 * cnt, w + 5 * cnt, h_C ? w + 6 * cnt : nullptr,
                                                           n_bins, ds->tab, ds->cst);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    LR_CUDA(cudaStreamSynchronize(h->stream));
    *out = ds;
    return LR_OK;
}

extern "C" int lr_dataset_destroy(lr_dataset_t ds) {
    if (!ds) return LR_OK;
    cudaSetDevice(ds->h->device);
    lr_order(ds->h, &ds->last, ds->h->stream);        // readers on caller streams finish before the block returns to the pool
    cudaFreeAsync(ds->tab, ds->h->stream); cudaFreeAsync(ds->cst, ds->h->stream);
    delete ds;
    return LR_OK;
}

extern "C" int lr_state_eval_host(lr_dataset_t ds, int32_t n, const int32_t* rep, const int32_t* K_l, const int32_t* K_m,
                                  const double* L, const double* M, const double* tL, const double* tM,
                                  const double* gamma_rate, const double* poi_lambda,
                                  double* lik, double* prior_rates, double* prior_poi, double* adequacy) {
    LR_REQUIRE(ds && K_l && K_m && L && M && tL && tM, "lr_state_eval_host: null pointer");
    LR_REQUIRE(n >= 0, "lr_state_eval_host: n < 0");
    if (n == 0) return LR_OK;
    for (int i = 0; i < n; ++i) {
        LR_REQUIRE(K_l[i] >= 1 && K_l[i] <= LR_KMAX && K_m[i] >= 1 && K_m[i] <= LR_KMAX, "lr_state_eval_host: K out of 1..%d at state %d", LR_KMAX, i);
        LR_REQUIRE(!rep || (rep[i] >= 0 && rep[i] < ds->n_rep), "lr_state_eval_host: replicate index out of range at state %d", i);
    }
    lr_handle_t h = ds->h;
    LR_CUDA(cudaSetDevice(h->device));
    { int rc0 = lr_order(h, &ds->last, h->stream); if (rc0 != LR_OK) return rc0; }
    const size_t nK = (size_t)n * LR_KMAX * 8;
    // layout in workspace
    size_t off = 0;
    auto take = [&](size_t b) { size_t o = off; off += (b + 255) & ~(size_t)255; return o; };
    const size_t o_rep = take((size_t)n * 4), o_kl = take((size_t)n * 4), o_km = take((size_t)n * 4);
    const size_t o_L = take(nK), o_M = take(nK), o_tL = take(nK), o_tM = take(nK);
    const size_t o_g = take((size_t)n * 16), o_p = take((size_t)n * 8);
    const size_t o_lik = take((size_t)n * 8), o_pr = take((size_t)n * 8), o_pp = take((size_t)n * 8), o_ad = take((size_t)n * 24);
    int rc = lr_ws_acquire(h, off, h->stream);
    if (rc != LR_OK) return rc;
    char* w = (char*)h->ws;
    cudaStream_t st = h->stream;
    if (rep) LR_CUDA(cudaMemcpyAsync(w + o_rep, rep, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    LR_CUDA(cudaMemcpyAsync(w + o_kl, K_l, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    LR_CUDA(cudaMemcpyAsync(w + o_km, K_m, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    LR_CUDA(cudaMemcpyAsync(w + o_L, L, nK, cudaMemcpyHostToDevice, st));
    LR_CUDA(cudaMemcpyAsync(w + o_M, M, nK, cudaMemcpyHostToDevice, st));
    LR_CUDA(cudaMemcpyAsync(w + o_tL, tL, nK, cudaMemcpyHostToDevice, st));
    LR_CUDA(cudaMemcpyAsync(w + o_tM, tM, nK, cudaMemcpyHostToDevice, st));
    if (gamma_rate) LR_CUDA(cudaMemcpyAsync(w + o_g, gamma_rate, (size_t)n * 16, cudaMemcpyHostToDevice, st));
    if (poi_lambda) LR_CUDA(cudaMemcpyAsync(w + o_p, poi_lambda, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    const int wpb = 4;
    k2_state_eval_kernel<<<(n + wpb - 1) / wpb, wpb * 32, 0, st>>>(
        n, rep ? (const int*)(w + o_rep) : nullptr, (const int*)(w + o_kl), (const int*)(w + o_km),
        (const double*)(w + o_L), (const double*)(w + o_M), (const double*)(w + o_tL), (const double*)(w + o_tM),
        gamma_rate ? (const double*)(w + o_g) : nullptr, poi_lambda ? (const double*)(w + o_p) : nullptr,
        ds->tab, ds->cst, ds->n_bins, ds->s0f, ds->start_time, ds->end_time,
        lik ? (double*)(w + o_lik) : nullptr, prior_rates ? (double*)(w + o_pr) : nullptr,
        prior_poi ? (double*)(w + o_pp) : nullptr, adequacy ? (double*)(w + o_ad) : nullptr);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    if (lik) LR_CUDA(cudaMemcpyAsync(lik, w + o_lik, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    if (prior_rates) LR_CUDA(cudaMemcpyAsync(prior_rates, w + o_pr, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    if (prior_poi) LR_CUDA(cudaMemcpyAsync(prior_poi, w + o_pp, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    if (adequacy) LR_CUDA(cudaMemcpyAsync(adequacy, w + o_ad, (size_t)n * 24, cudaMemcpyDeviceToHost, st));
    LR_CUDA(cudaStreamSynchronize(st));
    return LR_OK;
}

extern "C" int lr_proposal_eval_host(lr_dataset_t ds, int32_t n, const int32_t* rep, const int32_t* K_l, const int32_t* K_m,
                                     const double* L, const double* M, const double* tL, const double* tM,
                                     const double* gamma_rate, const double* poi_lambda, const double* beta, const double* poiA,
                                     const int32_t* side, const int32_t* kind, const int32_t* idx, const double* u_t, const double* u_beta,
                                     const int32_t* mult_on, const double* mult_u,
                                     int32_t* ok, int32_t* K_new, double* rates_new, double* times_new, double* hasting, double* x) {
    LR_REQUIRE(ds && K_l && K_m && L && M && tL && tM && poiA && side && kind && idx && u_t && u_beta && ok && K_new && rates_new && times_new && hasting && x,
               "lr_proposal_eval_host: null pointer");
    LR_REQUIRE(n >= 0, "lr_proposal_eval_host: n < 0");
    if (n == 0) return LR_OK;
    for (int i = 0; i < n; ++i) {
        LR_REQUIRE(K_l[i] >= 1 && K_l[i] <= LR_KMAX && K_m[i] >= 1 && K_m[i] <= LR_KMAX, "lr_proposal_eval_host: K out of 1..%d at state %d", LR_KMAX, i);
        LR_REQUIRE(!rep || (rep[i] >= 0 && rep[i] < ds->n_rep), "lr_proposal_eval_host: replicate index out of range at state %d", i);
        const int K = side[i] ? K_l[i] : K_m[i];
        LR_REQUIRE(kind[i] == 0 || kind[i] == 2 || kind[i] == 3, "lr_proposal_eval_host: kind must be 0 (rate multiplier), 2 (add-shift) or 3 (remove-shift) at state %d", i);
        LR_REQUIRE(kind[i] != 0 || (mult_on && mult_u), "lr_proposal_eval_host: kind 0 needs mult_on and mult_u");
        if (kind[i] == 0) continue;
        LR_REQUIRE(kind[i] == 2 ? (idx[i] >= 0 && idx[i] < K) : (K > 1 && idx[i] >= 1 && idx[i] <= K - 1), "lr_proposal_eval_host: index out of range at state %d", i);
        LR_REQUIRE(u_beta[i] > 0.0 && u_beta[i] < 1.0 && u_t[i] >= 0.0 && u_t[i] <= 1.0, "lr_proposal_eval_host: draws outside (0,1) at state %d", i);
    }
    lr_handle_t h = ds->h;
    LR_CUDA(cudaSetDevice(h->device));
    { int rc0 = lr_order(h, &ds->last, h->stream); if (rc0 != LR_OK) return rc0; }
    const size_t nK = (size_t)n * LR_KMAX * 8, n4 = (size_t)n * 4, n8 = (size_t)n * 8;
    size_t off = 0;
    auto take = [&](size_t b) { size_t o = off; off += (b + 255) & ~(size_t)255; return o; };
    const size_t o_rep = take(n4), o_kl = take(n4), o_km = take(n4), o_L = take(nK), o_M = take(nK), o_tL = take(nK), o_tM = take(nK);
    const size_t o_g = take(2 * n8), o_p = take(n8), o_b = take(n8), o_pa = take(n8), o_sd = take(n4), o_kd = take(n4), o_ix = take(n4);
    const size_t o_mo = take((size_t)n * LR_KMAX * 4), o_mu = take(nK);
    const size_t o_ut = take(n8), o_ub = take(n8), o_ok = take(n4), o_kn = take(n4), o_rn = take(nK), o_tn = take(nK), o_h = take(n8), o_x = take(n8);
    int rc = lr_ws_acquire(h, off, h->stream);
    if (rc != LR_OK) return rc;
    char* w = (char*)h->ws;
    cudaStream_t st = h->stream;
    auto up = [&](size_t o, const void* src, size_t b) { return src ? cudaMemcpyAsync(w + o, src, b, cudaMemcpyHostToDevice, st) : cudaSuccess; };
    LR_CUDA(up(o_rep, rep, n4)); LR_CUDA(up(o_kl, K_l, n4)); LR_CUDA(up(o_km, K_m, n4));
    LR_CUDA(up(o_L, L, nK)); LR_CUDA(up(o_M, M, nK)); LR_CUDA(up(o_tL, tL, nK)); LR_CUDA(up(o_tM, tM, nK));
    LR_CUDA(up(o_g, gamma_rate, 2 * n8)); LR_CUDA(up(o_p, poi_lambda, n8)); LR_CUDA(up(o_b, beta, n8)); LR_CUDA(up(o_pa, poiA, n8));
    LR_CUDA(up(o_sd, side, n4)); LR_CUDA(up(o_kd, kind, n4)); LR_CUDA(up(o_ix, idx, n4)); LR_CUDA(up(o_ut, u_t, n8)); LR_CUDA(up(o_ub, u_beta, n8));
    LR_CUDA(up(o_mo, mult_on, (size_t)n * LR_KMAX * 4)); LR_CUDA(up(o_mu, mult_u, nK));
    const int wpb = 4;
    k2_proposal_eval_kernel<<<(n + wpb - 1) / wpb, wpb * 32, 0, st>>>(
        n, rep ? (const int*)(w + o_rep) : nullptr, (const int*)(w + o_kl), (const int*)(w + o_km), (const double*)(w + o_L), (const double*)(w + o_M),
        (const double*)(w + o_tL), (const double*)(w + o_tM), gamma_rate ? (const double*)(w + o_g) : nullptr,
        poi_lambda ? (const double*)(w + o_p) : nullptr, beta ? (const double*)(w + o_b) : nullptr, (const double*)(w + o_pa),
        (const int*)(w + o_sd), (const int*)(w + o_kd), (const int*)(w + o_ix), (const double*)(w + o_ut), (const double*)(w + o_ub),
        mult_on ? (const int*)(w + o_mo) : nullptr, mult_u ? (const double*)(w + o_mu) : nullptr,
        ds->tab, ds->cst, ds->n_bins, ds->s0f, ds->start_time, ds->end_time,
        (int*)(w + o_ok), (int*)(w + o_kn), (double*)(w + o_rn), (double*)(w + o_tn), (double*)(w + o_h), (double*)(w + o_x));
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    LR_CUDA(cudaMemcpyAsync(ok, w + o_ok, n4, cudaMemcpyDeviceToHost, st));
    LR_CUDA(cudaMemcpyAsync(K_new, w + o_kn, n4, cudaMemcpyDeviceToHost, st));
    LR_CUDA(cudaMemcpyAsync(rates_new, w + o_rn, nK, cudaMemcpyDeviceToHost, st));
    LR_CUDA(cudaMemcpyAsync(times_new, w + o_tn, nK, cudaMemcpyDeviceToHost, st));
    LR_CUDA(cudaMemcpyAsync(hasting, w + o_h, n8, cudaMemcpyDeviceToHost, st));
    LR_CUDA(cudaMemcpyAsync(x, w + o_x, n8, cudaMemcpyDeviceToHost, st));
    LR_CUDA(cudaStreamSynchronize(st));
    return LR_OK;
}

extern "C" int lr_chains_create(lr_handle_t h, lr_dataset_t ds, int32_t n_chains, const lr_chain_config* cfg,
                                uint64_t seed, int64_t chain_id0, const int32_t* h_rep_of_chain, lr_chains_t* out) {
    LR_REQUIRE(h && ds && cfg && out, "lr_chains_create: null pointer");
    LR_REQUIRE(ds->h == h, "lr_chains_create: dataset belongs to another handle");
    LR_REQUIRE(n_chains >= 1, "lr_chains_create: n_chains must be >= 1");
    LR_REQUIRE(cfg->model_BDI == ds->model, "lr_chains_create: cfg.model_BDI differs from the dataset's");
    LR_REQUIRE(cfg->update_fraction >= 0.0 && cfg->update_fraction <= 1.0, "lr_chains_create: update_fraction outside [0,1]");
    LR_REQUIRE(cfg->poisson_prior >= 0.0, "lr_chains_create: poisson_prior must be >= 0");
    LR_REQUIRE(cfg->loop_variant >= 0 && cfg->loop_variant <= 4, "lr_chains_create: loop_variant must be 0..4");
    LR_REQUIRE(chain_id0 >= 0 && chain_id0 + n_chains <= 0xffffffffll, "lr_chains_create: chain ids must fit 32 bits");
    if (h_rep_of_chain)
        for (int i = 0; i < n_chains; ++i)
            LR_REQUIRE(h_rep_of_chain[i] >= 0 && h_rep_of_chain[i] < ds->n_rep, "lr_chains_create: replicate of chain %d out of range", i);
    LR_CUDA(cudaSetDevice(h->device));
    { int rc0 = lr_order(h, &ds->last, h->stream); if (rc0 != LR_OK) return rc0; }
    lr_chains_t c = new lr_chains_s();
    c->last.s = h->stream; c->last.valid = 1;
    c->h = h; c->ds = ds; c->n_chains = n_chains; c->cfg = *cfg; c->seed = seed; c->chain_id0 = chain_id0; c->st = nullptr; c->it_host = 0;
    if (c->cfg.beta == 0.0) c->cfg.beta = 1.0;
    cudaError_t e = cudaMallocAsync((void**)&c->st, (size_t)n_chains * sizeof(ChainState), h->stream);
    if (e != cudaSuccess) { lr_set_error("lr_chains_create: cudaMallocAsync: %s", cudaGetErrorString(e)); delete c; return LR_ERR_NOMEM; }
    int* d_rep = nullptr;
    if (h_rep_of_chain) {
        int rc = lr_ws_acquire(h, (size_t)n_chains * 4, h->stream);
        if (rc != LR_OK) { cudaFreeAsync(c->st, h->stream); delete c; return rc; }
        d_rep = (int*)h->ws;
        LR_CUDA(cudaMemcpyAsync(d_rep, h_rep_of_chain, (size_t)n_chains * 4, cudaMemcpyHostToDevice, h->stream));
    }
    int threads;
    const int blocks = lr_chain_grid(n_chains, threads);
    k3_init_kernel<<<blocks, threads, 0, h->stream>>>(c->st, n_chains, d_rep, chain_id0, (uint32_t)seed, (uint32_t)(seed >> 32),
                                                      ds->start_time, cfg->poisson_prior, c->cfg.beta);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    LR_CUDA(cudaStreamSynchronize(h->stream));
    *out = c;
    return LR_OK;
}

extern "C" int lr_chains_destroy(lr_chains_t c) {
    if (!c) return LR_OK;
    cudaSetDevice(c->h->device);
    lr_order(c->h, &c->last, c->h->stream);
    cudaFreeAsync(c->st, c->h->stream);
    delete c;
    return LR_OK;
}

extern "C" int64_t lr_chains_records_per_run(lr_chains_t c, int64_t n_iter, int64_t sample_every) {
    if (!c || n_iter <= 0 || sample_every <= 0) return 0;
    long long it0 = c->it_host;
    // chains were given different iteration counters through set_state: chain 0's counts, as before
    if (it0 < 0 && !lr_read_counter(c->h, &c->last, &c->st[0].it, &it0)) return -1;
    return lr_records_per_run(it0, n_iter, sample_every);
}

extern "C" int lr_chains_run(lr_chains_t c, int64_t n_iter, int64_t sample_every, double* d_records, void* stream) {
    LR_REQUIRE(c != nullptr, "lr_chains_run: null chains");
    LR_REQUIRE(n_iter >= 0 && sample_every >= 0, "lr_chains_run: negative count");
    LR_REQUIRE(n_iter <= 2000000000ll, "lr_chains_run: at most 2e9 iterations per launch (32-bit per-launch counters); split the run");
    if (n_iter == 0) return LR_OK;
    lr_handle_t h = c->h;
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    { int rc0 = lr_order(h, &c->last, st); if (rc0 == LR_OK) rc0 = lr_order(h, &c->ds->last, st); if (rc0 != LR_OK) return rc0; }
    RunParams P;
    P.st = c->st; P.n_chains = c->n_chains; P.tab = c->ds->tab; P.cst = c->ds->cst;
    P.nb = c->ds->n_bins; P.s0f = c->ds->s0f; P.model = c->ds->model;
    P.start_time = c->ds->start_time; P.end_time = c->ds->end_time;
    P.cfg = c->cfg; P.lc = loop_consts(c->cfg); P.k0 = (uint32_t)c->seed; P.k1 = (uint32_t)(c->seed >> 32);
    P.n_iter = n_iter; P.sample_every = sample_every > 0 ? sample_every : 1;
    P.it_begin = c->it_host; P.team_bail = 0; P.cont_mode = 0;
    P.records = sample_every > 0 ? d_records : nullptr;
    P.with_adequacy = 1;
    int threads;
    const int blocks = lr_chain_grid(c->n_chains, threads);
    // loop_variant: 0 = choose by population size (measured cross-over on B200), 1 = warp-specialised build
    // (one CTA of 4 warps per chain), 2 = compact build (one warp per chain)
    // loop_variant 0 picks by population size (measured on B200, 148 SMs; M it/s for one-chain CTAs / four-chain CTAs / compact):
    //   296 chains 572 / 506 / 325;  512: - / 873 / 557;  1024: - / 1094 / 1027;  1184: - / 1119 / 1161;  2048: - / 1051 / 1547
    // loop_variant 4 (speculative team, k3_team.cuh) and the automatic choice: teams of W warps by how many chains an SM has
    // to hold (M it/s on the bench statistics, 1M lineages x 200 bins: 148 chains W=16 852 against 358 for one-chain CTAs;
    // 256 chains W=8 1000 against 584; 512 chains W=4 1151 against 1041 for four-chain CTAs), followed by a CONTINUATION pass of
    // the latency-optimised build for the chains whose teams stopped because their state changes too often for speculation to
    // pay (example table, 75 lineages: 40 % of the iterations change the state -- team 55 M it/s, one-chain CTAs 145 M).
    int variant = c->cfg.loop_variant;
    const int sm = h->sm_count;
    if (variant == 0) {
        if (c->it_host >= 0 && c->n_chains <= 4 * sm) variant = 4;
        else variant = c->n_chains <= 2 * sm ? 1 : (c->n_chains <= 7 * sm ? 3 : 2);
    }
    auto launch_plain = [&](int var) {
        if (var == 1) {
            const size_t smem = sizeof(Ring<6>);
            cudaFuncSetAttribute(k3_run_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            k3_run_kernel<1><<<c->n_chains, 128, smem, st>>>(P);
        } else if (var == 3) {
            const size_t smem = 4 * sizeof(Ring<3>);
            cudaFuncSetAttribute(k3_run_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            k3_run_kernel<2><<<(c->n_chains + 3) / 4, 256, smem, st>>>(P);
        } else {
            k3_run_kernel<0><<<blocks, threads, 0, st>>>(P);
        }
        h->launches += 1;
    };
    if (variant == 4) {
        const char* e_w = getenv("LR_TEAM_W");              // development overrides (tests sweep them)
        const char* e_lead = getenv("LR_TEAM_LEAD");
        const char* e_nobail = getenv("LR_TEAM_NOBAIL");
        const int env_w = e_w ? atoi(e_w) : 0, env_lead = e_lead ? atoi(e_lead) : 0;
        const int W = env_w ? env_w : (c->n_chains <= sm ? 16 : (c->n_chains <= 2 * sm ? 8 : 4));
        int lead = env_lead ? env_lead : 4;
        if (lead < 1) lead = 1;
        if (lead > 7) lead = 7;
        P.team_bail = (c->it_host >= 0 && !(e_nobail && atoi(e_nobail))) ? 1 : 0;
        // Shared-memory carve-out: an SM serves kernels of different streams side by side only if its configured carve-out
        // already holds all of them; a K1 batch of the NEXT table (41 KB for five CTAs) launched while teams run on the default
        // 16 KB configuration waits for whole SMs to drain -- measured: one K1 launch delayed by 16 ms, the copy engine idle
        // for 13 of the 87 ms of a table.  Ask for 64 KB (28 % of 228) so that K1 fits next to the teams.
        static bool carve_set = false;
        if (!carve_set) {
            cudaFuncSetAttribute(k3_team_kernel<16>, cudaFuncAttributePreferredSharedMemoryCarveout, 30);
            cudaFuncSetAttribute(k3_team_kernel<8>, cudaFuncAttributePreferredSharedMemoryCarveout, 30);
            cudaFuncSetAttribute(k3_team_kernel<10>, cudaFuncAttributePreferredSharedMemoryCarveout, 30);
            cudaFuncSetAttribute(k3_team_kernel<12>, cudaFuncAttributePreferredSharedMemoryCarveout, 30);
            cudaFuncSetAttribute(k3_team_kernel<4>, cudaFuncAttributePreferredSharedMemoryCarveout, 30);
            carve_set = true;
        }
        auto launch_team = [&]() {
            if (W >= 16) k3_team_kernel<16><<<c->n_chains, 512, 0, st>>>(P, lead);
            else if (W == 12) k3_team_kernel<12><<<c->n_chains, 384, 0, st>>>(P, lead);
            else if (W == 10) k3_team_kernel<10><<<c->n_chains, 320, 0, st>>>(P, lead);
            else if (W >= 8) k3_team_kernel<8><<<c->n_chains, 256, 0, st>>>(P, lead);
            else k3_team_kernel<4><<<c->n_chains, 128, 0, st>>>(P, lead);
            h->launches += 1;
        };
        // Four passes over the same launch window; every kernel skips the chains that have nothing to do in it.
        //   A  teams; a team whose chain changes state too often stops early and hands the chain over for a while
        //   B  latency-optimised build: handed-over chains, up to the end of their hand-over
        //   C  teams again for the chains whose hand-over ended inside the window (burn-in is over: speculation pays now)
        //   D  latency-optimised build: whatever is left
        launch_team();
        if (P.team_bail) {
            const int cont = c->n_chains <= 2 * sm ? 1 : 3;
            LR_CUDA(cudaGetLastError());
            P.cont_mode = 1; launch_plain(cont);
            LR_CUDA(cudaGetLastError());
            P.cont_mode = 0; launch_team();
            LR_CUDA(cudaGetLastError());
            launch_plain(cont);
        }
    } else {
        launch_plain(variant);
    }
    LR_CUDA(cudaGetLastError());
    if (c->it_host >= 0) c->it_host += n_iter;
    return LR_OK;
}

extern "C" int lr_chains_run_host(lr_chains_t c, int64_t n_iter, int64_t sample_every, double* h_records) {
    LR_REQUIRE(c != nullptr, "lr_chains_run_host: null chains");
    const int64_t nrec = (h_records && sample_every > 0) ? lr_chains_records_per_run(c, n_iter, sample_every) : 0;
    return lr_run_into_host(c->h, "lr_chains_run_host", nrec, (size_t)c->n_chains * LR_REC_DOUBLES * sizeof(double), h_records,
                            [&](double* d_rec) { return lr_chains_run(c, n_iter, d_rec ? sample_every : 0, d_rec, c->h->stream); });
}

extern "C" int lr_chains_counters_host(lr_chains_t c, int64_t* h_counters) {
    LR_REQUIRE(c && h_counters, "lr_chains_counters_host: null pointer");
    LR_CUDA(cudaSetDevice(c->h->device));
    { int rc0 = lr_order(c->h, &c->last, c->h->stream); if (rc0 != LR_OK) return rc0; }
    LR_CUDA(cudaStreamSynchronize(c->h->stream));
    LR_CUDA(cudaMemcpy2D(h_counters, LR_NCOUNTERS * sizeof(int64_t), &c->st[0].counters[0], sizeof(ChainState), LR_NCOUNTERS * sizeof(int64_t),
                         c->n_chains, cudaMemcpyDeviceToHost));
    return LR_OK;
}

extern "C" int lr_chains_team_stats_host(lr_chains_t c, int64_t* h_stats) {
    LR_REQUIRE(c && h_stats, "lr_chains_team_stats_host: null pointer");
    LR_CUDA(cudaSetDevice(c->h->device));
    { int rc0 = lr_order(c->h, &c->last, c->h->stream); if (rc0 != LR_OK) return rc0; }
    LR_CUDA(cudaStreamSynchronize(c->h->stream));
    LR_CUDA(cudaMemcpy2D(h_stats, 6 * sizeof(int64_t), &c->st[0].team[0], sizeof(ChainState), 6 * sizeof(int64_t), c->n_chains, cudaMemcpyDeviceToHost));
    return LR_OK;
}

extern "C" int lr_chains_get_state_host(lr_chains_t c, double* h_records) {
    LR_REQUIRE(c && h_records, "lr_chains_get_state_host: null pointer");
    lr_handle_t h = c->h;
    LR_CUDA(cudaSetDevice(h->device));
    { int rc0 = lr_order(h, &c->last, h->stream); if (rc0 == LR_OK) rc0 = lr_order(h, &c->ds->last, h->stream); if (rc0 != LR_OK) return rc0; }
    const size_t bytes = (size_t)c->n_chains * LR_REC_DOUBLES * sizeof(double);
    int rc = lr_ws_acquire(h, bytes, h->stream);
    if (rc != LR_OK) return rc;
    int threads;
    const int blocks = lr_chain_grid(c->n_chains, threads);
    k3_get_state_kernel<<<blocks, threads, 0, h->stream>>>(c->st, c->n_chains, (double*)h->ws, c->ds->tab, c->ds->cst, c->ds->n_bins,
                                                           c->ds->s0f, c->ds->start_time, c->ds->end_time);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    LR_CUDA(cudaMemcpyAsync(h_records, h->ws, bytes, cudaMemcpyDeviceToHost, h->stream));
    LR_CUDA(cudaStreamSynchronize(h->stream));
    return LR_OK;
}

extern "C" int lr_chains_set_state_host(lr_chains_t c, const double* h_records) {
    LR_REQUIRE(c && h_records, "lr_chains_set_state_host: null pointer");
    lr_handle_t h = c->h;
    long long it_all = (long long)h_records[0];
    for (int i = 0; i < c->n_chains; ++i) {
        const double* r = h_records + (size_t)i * LR_REC_DOUBLES;
        LR_REQUIRE(r[5] >= 1 && r[5] <= LR_KMAX && r[6] >= 1 && r[6] <= LR_KMAX, "lr_chains_set_state_host: K out of range in chain %d", i);
        if ((long long)r[0] != it_all) it_all = -1;
    }
    c->it_host = it_all;
    LR_CUDA(cudaSetDevice(h->device));
    { int rc0 = lr_order(h, &c->last, h->stream); if (rc0 == LR_OK) rc0 = lr_order(h, &c->ds->last, h->stream); if (rc0 != LR_OK) return rc0; }
    const size_t bytes = (size_t)c->n_chains * LR_REC_DOUBLES * sizeof(double);
    int rc = lr_ws_acquire(h, bytes, h->stream);
    if (rc != LR_OK) return rc;
    LR_CUDA(cudaMemcpyAsync(h->ws, h_records, bytes, cudaMemcpyHostToDevice, h->stream));
    int threads;
    const int blocks = lr_chain_grid(c->n_chains, threads);
    k3_set_state_kernel<<<blocks, threads, 0, h->stream>>>(c->st, c->n_chains, (const double*)h->ws, c->ds->tab, c->ds->cst,
                                                           c->ds->n_bins, c->ds->s0f, c->ds->start_time, c->ds->end_time);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    LR_CUDA(cudaStreamSynchronize(h->stream));
    return LR_OK;
}

extern "C" int lr_chains_set_beta_host(lr_chains_t c, const double* h_beta) {
    LR_REQUIRE(c && h_beta, "lr_chains_set_beta_host: null pointer");
    lr_handle_t h = c->h;
    LR_CUDA(cudaSetDevice(h->device));
    { int rc0 = lr_order(h, &c->last, h->stream); if (rc0 != LR_OK) return rc0; }
    int rc = lr_ws_acquire(h, (size_t)c->n_chains * 8, h->stream);
    if (rc != LR_OK) return rc;
    LR_CUDA(cudaMemcpyAsync(h->ws, h_beta, (size_t)c->n_chains * 8, cudaMemcpyHostToDevice, h->stream));
    k3_set_beta_kernel<<<(c->n_chains + 127) / 128, 128, 0, h->stream>>>(c->st, c->n_chains, (const double*)h->ws);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    LR_CUDA(cudaStreamSynchronize(h->stream));
    return LR_OK;
}

extern "C" int lr_chains_swap_info(lr_chains_t c, double* d_info, void* stream) {
    LR_REQUIRE(c && d_info, "lr_chains_swap_info: null pointer");
    lr_handle_t h = c->h;
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    { int rc0 = lr_order(h, &c->last, st); if (rc0 == LR_OK) rc0 = lr_order(h, &c->ds->last, st); if (rc0 != LR_OK) return rc0; }
    int threads;
    const int blocks = lr_chain_grid(c->n_chains, threads);
    k3_swap_info_kernel<<<blocks, threads, 0, st>>>(c->st, c->n_chains, d_info, c->ds->tab, c->ds->cst, c->ds->n_bins, c->ds->s0f,
                                                    c->ds->start_time, c->ds->end_time);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    return LR_OK;
}

static int swap_apply(lr_chains_t c, const double* d_info_all, int64_t table_first, int64_t n_all, int64_t first, int32_t ladder,
                      uint64_t round, void* stream, const char* who) {
    LR_REQUIRE(c, "%s: null pointer", who);
    return lr_swap_apply(c->h, &c->last, c->n_chains, d_info_all, table_first, n_all, first, ladder, stream, who,
                         [&](int blocks, int threads, cudaStream_t st) {
                             k3_swap_apply_kernel<<<blocks, threads, 0, st>>>(c->st, c->n_chains, d_info_all, table_first, n_all, first,
                                                                              ladder, round, (uint32_t)c->seed, (uint32_t)(c->seed >> 32));
                         });
}

extern "C" int lr_chains_swap_apply(lr_chains_t c, const double* d_info_all, int64_t n_all, int64_t first, int32_t ladder,
                                    uint64_t round, void* stream) {
    return swap_apply(c, d_info_all, 0, n_all, first, ladder, round, stream, "lr_chains_swap_apply");
}

extern "C" int lr_chains_swap_step(lr_chains_t c, int32_t ladder, uint64_t round) {
    LR_REQUIRE(c != nullptr, "lr_chains_swap_step: null chains");
    // ladders and their Philox keys are numbered by GLOBAL chain id, so the outcome does not depend on the sharding
    return lr_swap_step(c->h, c->chain_id0, c->n_chains, ladder, nullptr, "lr_chains",
                        [&](double* d_info) { return lr_chains_swap_info(c, d_info, c->h->stream); },
                        [&](const double* d_info) {
                            return swap_apply(c, d_info, c->chain_id0, c->n_chains, c->chain_id0, ladder, round, c->h->stream,
                                              "lr_chains_swap_step");
                        });
}
