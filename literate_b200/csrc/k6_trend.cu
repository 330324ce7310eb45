// K6: TrendRate (SURVEY 8 f-4) -- fixed-dimension Metropolis-Hastings chains on the binned statistics of K1 with
// birth and death rates that follow an exogenous trend.  Replaces the loop of trend_rate.py:102-196 and the
// literate_library.py functions it calls (proposals :140-165, priors :182-187, adequacy :268-279).
//
//   lambda_j = l_min + alpha * trend_j ** delta      mu_j = m_min + beta * trend_j ** gamma        (trend_rate.py:73-91)
//   log-lik  = sum_j log(lambda_j) sp_j - lambda_j br_j  +  sum_j log(mu_j) ex_j - mu_j br_j       (Keiding form, :82, :88)
//
// One warp = one chain, whole loop on device.  Lane p < 6 owns parameter p: it draws the parameter's Bernoulli mask and
// its multiplier / normal step from one Philox call keyed by (seed, chain, iteration, lane), evaluates the parameter's
// prior difference (no logarithm: the Gamma(3) parameters only move by multipliers), and the six values are broadcast by
// shuffles; lane 6 draws the branch uniform and the acceptance uniform (accept test through a single-precision bracket of log u).
// Bins are strided over the 32 lanes (bin j lives in lane j % 32; the first 32 bins' statistics stay in registers), the
// two side sums come out of one butterfly.  A side none of whose parameters was touched keeps its stored likelihood (the
// reference recomputes the identical number).  Nothing but the read-only per-bin table (L1-resident) is read inside the
// loop; the only global writes are the sample records.
#include "lr_common.cuh"

#define TR_NPAR 6
#define TR_ROWS 6          // per replicate: sp, ex, br, ln(trend), empirical birth rate, empirical death rate
#define TR_SP 0
#define TR_EX 1
#define TR_BR 2
#define TR_LNT 3
#define TR_XB 4
#define TR_XD 5
#define TR_SMALL 0.000000000000001      // SMALL_NUMBER, trend_rate.py:55
#define TR_LN_MULT 0.19062035960864987  // 2*log(1.1): update_multiplier_proposal_vec(d=1.1), literate_library.py:160
#define TR_NORM_SD 0.001                // update_normal_nobound_vec(d=.001), trend_rate.py:168

struct TrendChain {
    double p[TR_NPAR];     // l_min, m_min, alpha, beta, delta, gamma (trend_rate.py:74)
    double likB, likD, prior;
    long long it;          // iterations done
    long long accepted;
    unsigned chain;        // global chain id (Philox key)
    int rep;
    double beta;           // inverse temperature of a tempered ladder (1: the reference's chain)
    long long swaps[2];    // temperature swaps proposed, accepted
};

struct lr_trend_s {
    lr_handle_t h;
    lr_last_stream last;           // stream that touched the object last (lr_order)
    int n_rep, n_bins, nbp;        // nbp: row pitch of the table
    int const_b, const_d;
    double* tab;                   // device [n_rep][TR_ROWS][nbp]
    double* cst;                   // device [n_rep][2]: sum x, sum x^2 of the empirical rates (adequacy)
    int n_chains;
    uint64_t seed;
    int64_t chain_id0;             // global id of chain 0 (ladders are numbered by global id)
    int* rep_of_chain;             // host [n_chains]: replicate of every chain (swap_step refuses ladders that mix replicates)
    TrendChain* st;                // device [n_chains]
    double f_mult[TR_NPAR], f_norm[TR_NPAR];
};

namespace {

struct TrendView {
    const double* tab;
    int nb, nbp, const_b, const_d;
    double Sx, Sxx;
    // the bins of the likelihood sums this warp owns: first + lane (statistics in registers), then every `stride`-th after it.
    // One warp per chain: first = 0, stride = 32.  W warps per chain: first = 32 w, stride = 32 W.
    int first, stride;
    double sp0, ex0, br0, lnT0;
};

__device__ __forceinline__ TrendView trend_view(const double* tab_all, const double* cst_all, int rep, int nb, int nbp,
                                                int const_b, int const_d, int lane, int first = 0, int stride = 32) {
    TrendView v;
    v.tab = tab_all + (size_t)rep * TR_ROWS * nbp;
    v.nb = nb; v.nbp = nbp; v.const_b = const_b; v.const_d = const_d;
    v.Sx = cst_all[2 * rep]; v.Sxx = cst_all[2 * rep + 1];
    v.first = first; v.stride = stride;
    const int j = first + lane;
    const bool on = j < nb;
    v.sp0 = on ? v.tab[TR_SP * nbp + j] : 0.0;
    v.ex0 = on ? v.tab[TR_EX * nbp + j] : 0.0;
    v.br0 = on ? v.tab[TR_BR * nbp + j] : 0.0;
    v.lnT0 = on ? v.tab[TR_LNT * nbp + j] : 0.0;
    return v;
}

// rate of one bin (trend_rate.py:75-80 / :83-87): floor = a + b * T**c, values <= 0 become SMALL_NUMBER
__device__ __forceinline__ double trend_rate(double a, double b, double c, double lnT, int is_const) {
    if (is_const) return a;
    double r = a + b * exp(c * lnT);
    return r > 0.0 ? r : TR_SMALL;
}

// T**delta and T**gamma of the first 32 bins (one per lane): they change only when delta / gamma are proposed
struct PowCache { double b, d; };

// partial sums over the bins this warp owns (per lane, not yet reduced)
// termB / termD (W > 1): if not null, every bin's term is also stored at its bin index
__device__ __forceinline__ void trend_lik_partial(const TrendView& v, const double* p, int lane, bool doB, bool doD, bool newPowB, bool newPowD,
                                                  PowCache& pc, double& sB, double& sD, double* termB = nullptr, double* termD = nullptr) {
    sB = 0.0; sD = 0.0;
    if (doB) {
        double lam = p[0];
        if (!v.const_b) {
            if (newPowB) pc.b = exp(p[4] * v.lnT0);
            lam = p[0] + p[2] * pc.b;
            lam = lam > 0.0 ? lam : TR_SMALL;
        }
        sB = log(lam) * v.sp0 - lam * v.br0;
    }
    if (doD) {
        double mu = p[1];
        if (!v.const_d) {
            if (newPowD) pc.d = exp(p[5] * v.lnT0);
            mu = p[1] + p[3] * pc.d;
            mu = mu > 0.0 ? mu : TR_SMALL;
        }
        sD = log(mu) * v.ex0 - mu * v.br0;
    }
    if (termB != nullptr && v.first + lane < v.nb) { termB[v.first + lane] = sB; termD[v.first + lane] = sD; }
    for (int j = v.first + lane + v.stride; j < v.nb; j += v.stride) {
        const double lnT = __ldg(v.tab + TR_LNT * v.nbp + j), br = __ldg(v.tab + TR_BR * v.nbp + j);
        double tB = 0.0, tD = 0.0;
        if (doB) {
            const double lam = trend_rate(p[0], p[2], p[4], lnT, v.const_b);
            tB = log(lam) * __ldg(v.tab + TR_SP * v.nbp + j) - lam * br;
            sB += tB;
        }
        if (doD) {
            const double mu = trend_rate(p[1], p[3], p[5], lnT, v.const_d);
            tD = log(mu) * __ldg(v.tab + TR_EX * v.nbp + j) - mu * br;
            sD += tD;
        }
        if (termB != nullptr) { termB[j] = tB; termD[j] = tD; }
    }
}

// both side likelihoods (uniform over the warp); a side with do_* == false keeps the value passed in.  newPowB/newPowD: the
// exponent of that side differs from the one `pc` was computed for (pc is updated in place)
// `extra`: a per-lane term (Hastings share + prior difference of the lane's parameter) that rides the same butterfly; its
// warp total comes back in place.
// W warps per chain (W > 1): termB / termD are this iteration's [nbp] buffers of shared memory.  Every warp stores the terms
// of its bins there and then adds up all bins exactly as one warp per chain does -- lane l its bins l, l + 32, ... in
// ascending order (0.0 for a side that was not evaluated), then one butterfly -- so the chain does not depend on W.
template <int W = 1>
__device__ __forceinline__ void trend_lik(const TrendView& v, const double* p, int lane, bool doB, bool doD, bool newPowB, bool newPowD,
                                          PowCache& pc, double& likB, double& likD, double& extra, double* termB = nullptr,
                                          double* termD = nullptr) {
    double sB, sD;
    if constexpr (W == 1) {
        trend_lik_partial(v, p, lane, doB, doD, newPowB, newPowD, pc, sB, sD);
    } else {
        trend_lik_partial(v, p, lane, doB, doD, newPowB, newPowD, pc, sB, sD, termB, termD);
        __syncthreads();
        sB = 0.0; sD = 0.0;
        for (int j = lane; j < v.nb; j += 32) { sB += termB[j]; sD += termD[j]; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sB += __shfl_xor_sync(0xffffffffu, sB, o);
        sD += __shfl_xor_sync(0xffffffffu, sD, o);
        extra += __shfl_xor_sync(0xffffffffu, extra, o);
    }
    if (doB) likB = sB;
    if (doD) likD = sD;
}

// prior term of parameter `lane` (calc_prior, trend_rate.py:93-100; closed forms of scipy's gamma/norm logpdf)
__device__ __forceinline__ double trend_prior_term(int lane, double x) {
    if (lane < 2) {                         // Gamma(a=1, scale 10, loc .001)
        const double y = x - 0.001;
        return y < 0.0 ? -INFINITY : -2.302585092994046 - y / 10.0;
    }
    if (lane < 4) return -(x * x) / 50.0 - 2.528376445638773;      // Normal(0, 5): -log(5) - log(2 pi)/2
    if (lane < 6) return x > 0.0 ? 2.0 * log(2.0 * x) - 2.0 * x : -INFINITY;     // Gamma(a=3, scale .5): lgamma(3) = -log(.5)
    return 0.0;
}

// prior(x') - prior(x) of parameter `lane` inside the loop, without logarithms: the Gamma(3) parameters (delta, gamma) only move
// by multipliers, where log x' - log x is the log-multiplier `lm` itself.  `x` lies in the support (it is an accepted state).
__device__ __forceinline__ double trend_prior_delta(int lane, double x, double xn, double lm) {
    const double d = xn - x;
    if (lane < 2) return xn < 0.001 ? -INFINITY : -d / 10.0;
    if (lane < 4) return -(d * (xn + x)) / 50.0;
    if (lane < 6) return xn > 0.0 ? 2.0 * lm - 2.0 * d : -INFINITY;
    return 0.0;
}

// One proposal (trend_rate.py:166-171).  Lane p < 6 returns the proposed value of parameter p given the parameter's own
// value `x`, its mask bit and its draw (uniform for the multiplier, standard normal for the additive step); `hast` receives
// the lane's share of the Hastings ratio.
__device__ __forceinline__ double trend_propose(int kind_normal, double x, bool on, double draw, double& hast) {
    hast = 0.0;
    if (!on) return x;
    if (kind_normal) return x + TR_NORM_SD * draw;          // literate_library.py:140-146
    const double lm = TR_LN_MULT * (draw - 0.5);            // literate_library.py:156-165: m = exp(l (u - .5)), U = sum log m
    hast = lm;
    return x * exp_small(lm);
}

__device__ __forceinline__ void bcast6(double mine, double* p) {
#pragma unroll
    for (int k = 0; k < TR_NPAR; ++k) p[k] = __shfl_sync(0xffffffffu, mine, k);
}

// calculate_r_squared (literate_library.py:268-279) in closed form; x = empirical rates, y = the model's rates
__device__ __forceinline__ void trend_adequacy(const TrendView& v, const double* p, int lane, double out[3]) {
    double sy = 0, syy = 0, sxy = 0;
    for (int j = lane; j < v.nb; j += 32) {
        const double lnT = __ldg(v.tab + TR_LNT * v.nbp + j);
        const double lam = trend_rate(p[0], p[2], p[4], lnT, v.const_b), mu = trend_rate(p[1], p[3], p[5], lnT, v.const_d);
        const double xb = __ldg(v.tab + TR_XB * v.nbp + j), xd = __ldg(v.tab + TR_XD * v.nbp + j);
        sy += lam + mu; syy += lam * lam + mu * mu; sxy += lam * xb + mu * xd;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sy += __shfl_xor_sync(0xffffffffu, sy, o);
        syy += __shfl_xor_sync(0xffffffffu, syy, o);
        sxy += __shfl_xor_sync(0xffffffffu, sxy, o);
    }
    const double n = 2.0 * v.nb;
    const double c = sxy / v.Sxx;
    const double ssres = syy - c * sxy;
    const double var_f = c * c * (v.Sxx - v.Sx * v.Sx / n) / (n - 1.0);
    const double sres = sy - c * v.Sx;
    const double var_r = (ssres - sres * sres / n) / (n - 1.0);
    out[0] = c; out[1] = 1.0 - ssres / syy; out[2] = var_f / (var_f + var_r);
}

// record: [0] it [1] likelihood [2] likelihood_birth [3] likelihood_death [4] prior [5..10] parameters [11..13] adequacy
//         [14] accepted so far [15] beta [16 .. 16+nb) birth rates [16+nb .. 16+2nb) death rates
__device__ __forceinline__ void trend_record(double* rec, const TrendView& v, const double* p, double mine, double likB, double likD,
                                             long long it, long long accepted, double beta, int lane) {
    double adq[3];
    trend_adequacy(v, p, lane, adq);
    const double prior = warp_sum(trend_prior_term(lane, mine));
    if (lane == 0) {
        rec[0] = (double)it; rec[1] = likB + likD; rec[2] = likB; rec[3] = likD; rec[4] = prior;
        rec[11] = adq[0]; rec[12] = adq[1]; rec[13] = adq[2]; rec[14] = (double)accepted; rec[15] = beta;
    }
#pragma unroll
    for (int k = 0; k < TR_NPAR; ++k)
        if (lane == k) rec[5 + k] = p[k];
    for (int j = lane; j < v.nb; j += 32) {
        const double lnT = __ldg(v.tab + TR_LNT * v.nbp + j);
        rec[LR_TREND_REC_HEAD + j] = trend_rate(p[0], p[2], p[4], lnT, v.const_b);
        rec[LR_TREND_REC_HEAD + v.nb + j] = trend_rate(p[1], p[3], p[5], lnT, v.const_d);
    }
}

struct TrendRun {
    TrendChain* st;
    int n_chains;
    const double* tab;
    const double* cst;
    int nb, nbp, const_b, const_d;
    uint32_t k0, k1;
    long long n_iter, sample_every;
    double* records;       // [sample][chain][rec_doubles] or null
    int rec_doubles;
    double fd_mult[TR_NPAR], fd_norm[TR_NPAR];  // Bernoulli probability of every parameter under the two proposal kinds
};

// W == 1: one warp per chain, four chains per CTA.  W = 2 or 4 (the wide build): one CTA of W warps per chain.  With a few
// hundred chains and hundreds of bins one warp per chain leaves the GPU idle (ncu, round 1: sm__throughput 10 %, 7 bins per
// lane in series, each an exp -> log chain).  There warp w evaluates bins 32 w + lane (+ 32 W k) -- at 200 bins and W = 4 two
// per lane instead of seven.  Every warp draws the same random numbers, builds the same proposal and takes the same accept
// decision; the warps exchange their per-bin terms through shared memory (double-buffered by iteration parity: one
// __syncthreads per iteration) and add them up in the one-warp order (trend_lik), so the chain is the one-warp chain, bit for
// bit (tests/test_gpu_trend.py), and does not depend on scheduling.
template <int W>
__global__ void __launch_bounds__(W == 1 ? 128 : 32 * W, W == 1 ? 4 : 2) k6_trend_kernel(const TrendRun P) {
    extern __shared__ double terms[];                  // W > 1: [2 parities][2 sides][nbp]
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int c = W == 1 ? blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5) : blockIdx.x;
    if (c >= P.n_chains) return;
    TrendChain* S = P.st + c;
    const TrendView v = trend_view(P.tab, P.cst, S->rep, P.nb, P.nbp, P.const_b, P.const_d, lane, W == 1 ? 0 : 32 * w, 32 * W);
    const unsigned chain = S->chain;
    double mine = lane < TR_NPAR ? S->p[lane] : 0.0;       // this lane's parameter; p[] = the broadcast copies
    double p[TR_NPAR];
    bcast6(mine, p);
    double likB = S->likB, likD = S->likD;
    PowCache pc;
    pc.b = v.const_b ? 1.0 : exp(p[4] * v.lnT0);
    pc.d = v.const_d ? 1.0 : exp(p[5] * v.lnT0);
    long long it = S->it, accepted = S->accepted;
    const long long it_end = it + P.n_iter;
    const double beta = S->beta;                           // read by every warp before warp 0 may rewrite the state
    // this lane's Bernoulli probabilities (lanes >= 6: never on)
    const double fm = lane < TR_NPAR ? P.fd_mult[lane] : 0.0, fn = lane < TR_NPAR ? P.fd_norm[lane] : 0.0;
    long long next_sample = (it + P.sample_every - 1) / P.sample_every * P.sample_every;
    long long rec_idx = 0;
    if constexpr (W > 1) __syncthreads();              // every warp has read the chain's state before warp 0 may rewrite it

    for (; it < it_end; ++it) {
        const Philox4 r = philox4x32_10((uint32_t)it, (uint32_t)((unsigned long long)it >> 32), (uint32_t)lane | (0x60u << 8), chain, P.k0, P.k1);
        // lane 6: branch and acceptance uniforms
        const double ua = u01(r.x, r.y), ub = u01(r.z, r.w);
        const double rr = __shfl_sync(0xffffffffu, ua, 6);
        const double u_acc = __shfl_sync(0xffffffffu, ub, 6);
        const int kind_normal = rr < 0.33;                                  // trend_rate.py:167
        // lanes 0..5: mask from 32 bits, draw from 52 bits (+ 24 bits for the angle of Box-Muller)
        const double um = ((double)r.x + 0.5) * 2.3283064365386963e-10;
        const bool on = um < (kind_normal ? fn : fm);
        double draw = u01(r.y, r.z);
        if (kind_normal) draw = normal_f32(draw, r.w);
        double h;
        const double prop = trend_propose(kind_normal, mine, on, draw, h);
        const unsigned touched = __ballot_sync(0xffffffffu, on);
        double q[TR_NPAR];
        bcast6(prop, q);
        // Hastings share and prior difference of this lane's parameter: summed in the butterfly of the likelihood
        double hp = h + trend_prior_delta(lane, mine, prop, h);
        double nB = likB, nD = likD;
        PowCache npc = pc;
        double* tB = terms + (size_t)(it & 1) * 2 * P.nbp;
        double* tD = tB + P.nbp;
        trend_lik<W>(v, q, lane, (touched & 0x15u) != 0, (touched & 0x2au) != 0, (touched & 0x10u) != 0, (touched & 0x20u) != 0, npc, nB, nD, hp, tB, tD);
        // tempered: only the likelihood is raised to the power beta (1.0 * d == d: at beta = 1 this is the untempered test)
        const double x = beta * ((nB + nD) - (likB + likD)) + hp;
        if (it == 0 || mh_accept_gt(x, u_acc)) {                            // trend_rate.py:176
#pragma unroll
            for (int k = 0; k < TR_NPAR; ++k) p[k] = q[k];
            mine = prop;
            likB = nB; likD = nD; pc = npc;
            ++accepted;
        }
        if (it == next_sample) {                                             // trend_rate.py:184
            if (P.records && (W == 1 || w == 0)) {
                // W > 1: re-reading the view here keeps its constants out of registers across the loop (142, not 146)
                const TrendView v0 = W == 1 ? v : trend_view(P.tab, P.cst, S->rep, P.nb, P.nbp, P.const_b, P.const_d, lane);
                trend_record(P.records + ((size_t)rec_idx * P.n_chains + c) * P.rec_doubles, v0, p, mine, likB, likD, it, accepted, beta, lane);
            }
            ++rec_idx;
            next_sample += P.sample_every;
        }
    }
    if (W == 1 || w == 0) {
        const double prior = warp_sum(trend_prior_term(lane, mine));
        if (lane < TR_NPAR) S->p[lane] = mine;
        if (lane == 0) { S->likB = likB; S->likD = likD; S->prior = prior; S->it = it; S->accepted = accepted; }
    }
}

// initial state (trend_rate.py:141-156)
__global__ void k6_init_kernel(TrendChain* st, int n_chains, const int* rep_of_chain, long long chain_id0, const double* tab,
                               const double* cst, int nb, int nbp, int const_b, int const_d) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n_chains) return;
    const int rep = rep_of_chain ? rep_of_chain[c] : 0;
    const TrendView v = trend_view(tab, cst, rep, nb, nbp, const_b, const_d, lane);
    const double mine = lane < 2 ? 0.1 : (lane < 4 ? 0.0 : (lane < 6 ? 1.0 : 0.0));
    double p[TR_NPAR];
    bcast6(mine, p);
    double likB = 0, likD = 0;
    PowCache pc;
    double unused = 0.0;
    trend_lik(v, p, lane, true, true, true, true, pc, likB, likD, unused);
    double pr = trend_prior_term(lane, mine);
    pr = warp_sum(pr);
    if (lane < TR_NPAR) st[c].p[lane] = mine;
    if (lane == 0) {
        st[c].likB = likB; st[c].likD = likD; st[c].prior = pr; st[c].it = 0; st[c].accepted = 0;
        st[c].chain = (unsigned)(chain_id0 + c); st[c].rep = rep;
        st[c].beta = 1.0; st[c].swaps[0] = 0; st[c].swaps[1] = 0;
    }
}

// ---- tempered ladders (new: the reference has no tempering, SURVEY A-15; the swap rule is lr_swap_round, shared with K3)
__global__ void k6_set_beta_kernel(TrendChain* st, int n, const double* beta) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) st[i].beta = beta[i];
}

// (likelihood, beta) of every chain, as stored: the untempered likelihood of the current state
__global__ void k6_swap_info_kernel(const TrendChain* st, int n, double* __restrict__ info) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { info[2 * i] = st[i].likB + st[i].likD; info[2 * i + 1] = st[i].beta; }
}

__global__ void k6_swap_apply_kernel(TrendChain* st, int n_local, const double* __restrict__ info_all, long long table_first,
                                     long long n_all, long long first, int ladder, unsigned long long round, uint32_t k0, uint32_t k1) {
    const int lane = threadIdx.x & 31;
    const int local = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
    if (local >= n_local) return;
    lr_swap_round(info_all, table_first, n_all, first + local, ladder, round, k0, k1, lane, [&](bool paired, bool accept, double beta_p) {
        TrendChain* S = st + local;
        if (paired) {
            S->swaps[0] += 1;
            if (accept) { S->swaps[1] += 1; S->beta = beta_p; }
        }
    });
}

// per-replicate table: statistics as doubles, ln(trend), empirical rates and their sums
__global__ void k6_build_tables(const long long* __restrict__ sp, const long long* __restrict__ ex, const double* __restrict__ br,
                                const double* __restrict__ trend, int nb, int nbp, double* __restrict__ tab_all, double* __restrict__ cst_all) {
    const int rep = blockIdx.x;
    double* tab = tab_all + (size_t)rep * TR_ROWS * nbp;
    for (int j = threadIdx.x; j < nbp; j += blockDim.x) {
        const bool in = j < nb;
        const double U = in ? (double)sp[(size_t)rep * nb + j] : 0.0, D = in ? (double)ex[(size_t)rep * nb + j] : 0.0;
        const double K = in ? br[(size_t)rep * nb + j] : 0.0;
        tab[TR_SP * nbp + j] = U; tab[TR_EX * nbp + j] = D; tab[TR_BR * nbp + j] = K;
        tab[TR_LNT * nbp + j] = in ? log(trend[j]) : 0.0;
        tab[TR_XB * nbp + j] = in ? U / K : 0.0;
        tab[TR_XD * nbp + j] = in ? D / K : 0.0;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double sx = 0, sxx = 0;
        for (int j = 0; j < nb; ++j) {
            const double xb = tab[TR_XB * nbp + j], xd = tab[TR_XD * nbp + j];
            sx += xb + xd; sxx += xb * xb + xd * xd;
        }
        cst_all[2 * rep] = sx; cst_all[2 * rep + 1] = sxx;
    }
}

// parity entry: one warp per explicit parameter vector, optionally after one proposal with explicit draws
__global__ void k6_eval_kernel(const double* tab, const double* cst, int nb, int nbp, int const_b, int const_d, int n,
                               const int* rep, const double* params, const int* kind, const int* on, const double* draw,
                               double* out_params, double* out_hast, double* lik, double* prior, double* rates, double* adequacy) {
    const int lane = threadIdx.x & 31;
    const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (s >= n) return;
    const TrendView v = trend_view(tab, cst, rep ? rep[s] : 0, nb, nbp, const_b, const_d, lane);
    double mine = lane < TR_NPAR ? params[s * TR_NPAR + lane] : 0.0, h = 0.0;
    if (kind) mine = trend_propose(kind[s], mine, lane < TR_NPAR && on[s * TR_NPAR + lane] != 0, lane < TR_NPAR ? draw[s * TR_NPAR + lane] : 0.0, h);
    h = warp_sum(h);
    double p[TR_NPAR];
    bcast6(mine, p);
    double likB = 0, likD = 0;
    PowCache pc;
    double unused = 0.0;
    trend_lik(v, p, lane, true, true, true, true, pc, likB, likD, unused);
    const double pr = warp_sum(trend_prior_term(lane, mine));
    double adq[3];
    trend_adequacy(v, p, lane, adq);
    if (lane == 0) {
        if (lik) { lik[2 * s] = likB; lik[2 * s + 1] = likD; }
        if (prior) prior[s] = pr;
        if (out_hast) out_hast[s] = h;
        if (adequacy) { adequacy[3 * s] = adq[0]; adequacy[3 * s + 1] = adq[1]; adequacy[3 * s + 2] = adq[2]; }
    }
    if (out_params && lane < TR_NPAR) out_params[s * TR_NPAR + lane] = mine;
    if (rates)
        for (int j = lane; j < nb; j += 32) {
            const double lnT = v.tab[TR_LNT * nbp + j];
            rates[(size_t)s * 2 * nb + j] = trend_rate(p[0], p[2], p[4], lnT, const_b);
            rates[(size_t)s * 2 * nb + nb + j] = trend_rate(p[1], p[3], p[5], lnT, const_d);
        }
}

// per-parameter Bernoulli probabilities of the two proposal kinds (trend_rate.py:122-134)
void move_weights(int const_b, int const_d, double* f_mult, double* f_norm) {
    double m[TR_NPAR] = {1, 1, 0, 0, 1, 1}, nn[TR_NPAR] = {0, 0, 1, 1, 0, 0};
    if (const_b) { m[4] = 0; nn[2] = 0; }
    if (const_d) { m[5] = 0; nn[3] = 0; }
    double sm = 0, sn = 0;
    for (int k = 0; k < TR_NPAR; ++k) { sm += m[k]; sn += nn[k]; }
    for (int k = 0; k < TR_NPAR; ++k) { f_mult[k] = m[k] / sm; f_norm[k] = nn[k] / sn; }
}

}  // namespace

extern "C" int64_t lr_trend_record_doubles(int32_t n_bins) { return LR_TREND_REC_HEAD + 2 * (int64_t)n_bins; }

extern "C" int lr_trend_create(lr_handle_t h, int32_t n_rep, int32_t n_bins, const int64_t* d_sp, const int64_t* d_ex,
                               const double* d_br, const double* h_trend, int32_t const_birth, int32_t const_death,
                               int32_t n_chains, uint64_t seed, int64_t chain_id0, const int32_t* h_rep_of_chain,
                               void* stream, lr_trend_t* out) {
    LR_REQUIRE(h && d_sp && d_ex && d_br && h_trend && out, "lr_trend_create: null pointer");
    LR_REQUIRE(n_rep >= 1 && n_bins >= 1 && n_chains >= 1, "lr_trend_create: n_rep, n_bins, n_chains must be >= 1");
    LR_REQUIRE(chain_id0 >= 0 && chain_id0 + n_chains <= 0xffffffffll, "lr_trend_create: chain ids must fit 32 bits");
    if (const_birth && const_death) {
        lr_set_error("lr_trend_create: constant birth AND death rates leave the additive move without a parameter; the reference "
                     "stops in np.random.binomial(p = nan) on its first such move (trend_rate.py:129-134, :168)");
        return LR_ERR_UNSUPPORTED;
    }
    for (int j = 0; j < n_bins; ++j)
        LR_REQUIRE(h_trend[j] > 0.0 && h_trend[j] <= 1.0, "lr_trend_create: trend[%d] = %g outside (0, 1]; pass the min-max normalised trend "
                   "with zeros replaced by 1e-15 (trend_rate.py:65-68)", j, h_trend[j]);
    if (h_rep_of_chain)
        for (int i = 0; i < n_chains; ++i)
            LR_REQUIRE(h_rep_of_chain[i] >= 0 && h_rep_of_chain[i] < n_rep, "lr_trend_create: replicate of chain %d out of range", i);
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    lr_trend_t t = new lr_trend_s();
    memset(t, 0, sizeof(*t));
    t->last.s = st; t->last.valid = 1;
    t->h = h; t->n_rep = n_rep; t->n_bins = n_bins; t->nbp = (n_bins + 3) & ~3;
    t->const_b = const_birth != 0; t->const_d = const_death != 0; t->n_chains = n_chains; t->seed = seed; t->chain_id0 = chain_id0;
    t->rep_of_chain = new int[n_chains];
    for (int i = 0; i < n_chains; ++i) t->rep_of_chain[i] = h_rep_of_chain ? h_rep_of_chain[i] : 0;
    move_weights(t->const_b, t->const_d, t->f_mult, t->f_norm);
    const size_t tab_bytes = (size_t)n_rep * TR_ROWS * t->nbp * sizeof(double);
    cudaError_t e = cudaMallocAsync((void**)&t->tab, tab_bytes, st);
    if (e == cudaSuccess) e = cudaMallocAsync((void**)&t->cst, (size_t)n_rep * 2 * sizeof(double), st);
    if (e == cudaSuccess) e = cudaMallocAsync((void**)&t->st, (size_t)n_chains * sizeof(TrendChain), st);
    if (e != cudaSuccess) { lr_set_error("lr_trend_create: cudaMallocAsync: %s", cudaGetErrorString(e)); lr_trend_destroy(t); return LR_ERR_NOMEM; }
    // trend and replicate map through stream-ordered scratch
    double* d_trend = nullptr;
    int* d_rep = nullptr;
    e = cudaMallocAsync((void**)&d_trend, (size_t)n_bins * sizeof(double), st);
    if (e == cudaSuccess && h_rep_of_chain) e = cudaMallocAsync((void**)&d_rep, (size_t)n_chains * sizeof(int), st);
    if (e != cudaSuccess) { lr_set_error("lr_trend_create: cudaMallocAsync: %s", cudaGetErrorString(e)); lr_trend_destroy(t); return LR_ERR_NOMEM; }
    auto undo = [&]() { if (d_trend) cudaFreeAsync(d_trend, st); if (d_rep) cudaFreeAsync(d_rep, st); lr_trend_destroy(t); };
    LR_CUDA_CLEAN(cudaMemcpyAsync(d_trend, h_trend, (size_t)n_bins * sizeof(double), cudaMemcpyHostToDevice, st), undo());
    if (d_rep) LR_CUDA_CLEAN(cudaMemcpyAsync(d_rep, h_rep_of_chain, (size_t)n_chains * sizeof(int), cudaMemcpyHostToDevice, st), undo());
    k6_build_tables<<<n_rep, 128, 0, st>>>((const long long*)d_sp, (const long long*)d_ex, d_br, d_trend, n_bins, t->nbp, t->tab, t->cst);
    LR_CUDA_CLEAN(cudaGetLastError(), undo());
    int threads;
    const int blocks = lr_chain_grid(n_chains, threads);
    k6_init_kernel<<<blocks, threads, 0, st>>>(t->st, n_chains, d_rep, chain_id0, t->tab, t->cst, n_bins, t->nbp, t->const_b, t->const_d);
    LR_CUDA_CLEAN(cudaGetLastError(), undo());
    h->launches += 2;
    LR_CUDA_CLEAN(cudaStreamSynchronize(st), undo());       // h_trend / h_rep_of_chain may be pageable: they are consumed when this returns
    cudaFreeAsync(d_trend, st);
    if (d_rep) cudaFreeAsync(d_rep, st);
    *out = t;
    return LR_OK;
}

extern "C" int lr_trend_create_host(lr_handle_t h, int32_t n_rep, int32_t n_bins, const int64_t* h_sp, const int64_t* h_ex,
                                    const double* h_br, const double* h_trend, int32_t const_birth, int32_t const_death,
                                    int32_t n_chains, uint64_t seed, int64_t chain_id0, const int32_t* h_rep_of_chain,
                                    lr_trend_t* out) {
    LR_REQUIRE(h && h_sp && h_ex && h_br, "lr_trend_create_host: null pointer");
    LR_REQUIRE(n_rep >= 1 && n_bins >= 1, "lr_trend_create_host: bad sizes");
    int64_t *d_sp, *d_ex;
    double* d_br;
    int rc = lr_upload_bin_stats(h, (size_t)n_rep * n_bins, h_sp, h_ex, h_br, &d_sp, &d_ex, &d_br);
    if (rc != LR_OK) return rc;
    return lr_trend_create(h, n_rep, n_bins, d_sp, d_ex, d_br, h_trend, const_birth, const_death, n_chains, seed, chain_id0,
                           h_rep_of_chain, h->stream, out);
}

extern "C" int lr_trend_destroy(lr_trend_t t) {
    if (!t) return LR_OK;
    cudaSetDevice(t->h->device);
    lr_order(t->h, &t->last, t->h->stream);
    if (t->tab) cudaFreeAsync(t->tab, t->h->stream);
    if (t->cst) cudaFreeAsync(t->cst, t->h->stream);
    if (t->st) cudaFreeAsync(t->st, t->h->stream);
    delete[] t->rep_of_chain;
    delete t;
    return LR_OK;
}

extern "C" int64_t lr_trend_records_per_run(lr_trend_t t, int64_t n_iter, int64_t sample_every) {
    if (!t || n_iter <= 0 || sample_every <= 0) return 0;
    long long it0 = 0;
    if (!lr_read_counter(t->h, &t->last, &t->st[0].it, &it0)) return -1;
    return lr_records_per_run(it0, n_iter, sample_every);
}

extern "C" int lr_trend_run(lr_trend_t t, int64_t n_iter, int64_t sample_every, double* d_records, void* stream) {
    LR_REQUIRE(t != nullptr, "lr_trend_run: null chains");
    LR_REQUIRE(n_iter >= 0 && sample_every >= 0, "lr_trend_run: negative count");
    if (n_iter == 0) return LR_OK;
    lr_handle_t h = t->h;
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    { int rc0 = lr_order(h, &t->last, st); if (rc0 != LR_OK) return rc0; }
    TrendRun P;
    P.st = t->st; P.n_chains = t->n_chains; P.tab = t->tab; P.cst = t->cst; P.nb = t->n_bins; P.nbp = t->nbp;
    P.const_b = t->const_b; P.const_d = t->const_d; P.k0 = (uint32_t)t->seed; P.k1 = (uint32_t)(t->seed >> 32);
    P.n_iter = n_iter; P.sample_every = sample_every > 0 ? sample_every : (int64_t)1 << 62;
    P.records = sample_every > 0 ? d_records : nullptr;
    P.rec_doubles = (int)lr_trend_record_doubles(t->n_bins);
    for (int k = 0; k < TR_NPAR; ++k) { P.fd_mult[k] = t->f_mult[k]; P.fd_norm[k] = t->f_norm[k]; }
    int threads;
    const int blocks = lr_chain_grid(t->n_chains, threads);
    // wide build (one warp per canonical group of bins) when one warp per chain would leave most of the GPU idle: measured on
    // B200 at 200 bins, M it/s one-warp / wide: 256 chains 82 / 141, 2048 chains 454 / 213.  Same chains either way.
    int W = lr_chain_width(t->n_bins, t->n_chains, h->sm_count, "LR_TREND_WIDE");
    const size_t smem = (size_t)4 * t->nbp * sizeof(double);
    if (W > 1 && smem > 40 * 1024) W = 1;
    if (W == 4) k6_trend_kernel<4><<<t->n_chains, 128, smem, st>>>(P);
    else if (W == 2) k6_trend_kernel<2><<<t->n_chains, 64, smem, st>>>(P);
    else k6_trend_kernel<1><<<blocks, threads, 0, st>>>(P);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    return LR_OK;
}

extern "C" int lr_trend_run_host(lr_trend_t t, int64_t n_iter, int64_t sample_every, double* h_records) {
    LR_REQUIRE(t != nullptr, "lr_trend_run_host: null chains");
    const int64_t nrec = (h_records && sample_every > 0) ? lr_trend_records_per_run(t, n_iter, sample_every) : 0;
    return lr_run_into_host(t->h, "lr_trend_run_host", nrec, (size_t)t->n_chains * lr_trend_record_doubles(t->n_bins) * sizeof(double),
                            h_records, [&](double* d_rec) { return lr_trend_run(t, n_iter, d_rec ? sample_every : 0, d_rec, t->h->stream); });
}

extern "C" int lr_trend_eval_host(lr_trend_t t, int32_t n, const int32_t* rep, const double* params, const int32_t* kind,
                                  const int32_t* on, const double* draw, double* out_params, double* out_hast, double* lik,
                                  double* prior, double* rates, double* adequacy) {
    LR_REQUIRE(t && params, "lr_trend_eval_host: null pointer");
    LR_REQUIRE(n >= 1, "lr_trend_eval_host: n must be >= 1");
    LR_REQUIRE(!kind || (on && draw), "lr_trend_eval_host: kind needs on and draw");
    if (rep)
        for (int i = 0; i < n; ++i) LR_REQUIRE(rep[i] >= 0 && rep[i] < t->n_rep, "lr_trend_eval_host: replicate of state %d out of range", i);
    lr_handle_t h = t->h;
    LR_CUDA(cudaSetDevice(h->device));
    { int rc0 = lr_order(t->h, &t->last, t->h->stream); if (rc0 != LR_OK) return rc0; }
    const int nb = t->n_bins;
    // workspace layout (doubles unless noted)
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_par = take((size_t)n * TR_NPAR * 8), o_rep = take((size_t)n * 4), o_kind = take((size_t)n * 4),
                 o_on = take((size_t)n * TR_NPAR * 4), o_draw = take((size_t)n * TR_NPAR * 8), o_np = take((size_t)n * TR_NPAR * 8),
                 o_h = take((size_t)n * 8), o_lik = take((size_t)n * 16), o_pr = take((size_t)n * 8),
                 o_rates = take((size_t)n * 2 * nb * 8), o_adq = take((size_t)n * 24);
    int rc = lr_ws_acquire(h, off, h->stream);
    if (rc != LR_OK) return rc;
    char* W = (char*)h->ws;
    cudaStream_t st = h->stream;
    LR_CUDA(cudaMemcpyAsync(W + o_par, params, (size_t)n * TR_NPAR * 8, cudaMemcpyHostToDevice, st));
    if (rep) LR_CUDA(cudaMemcpyAsync(W + o_rep, rep, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    if (kind) {
        LR_CUDA(cudaMemcpyAsync(W + o_kind, kind, (size_t)n * 4, cudaMemcpyHostToDevice, st));
        LR_CUDA(cudaMemcpyAsync(W + o_on, on, (size_t)n * TR_NPAR * 4, cudaMemcpyHostToDevice, st));
        LR_CUDA(cudaMemcpyAsync(W + o_draw, draw, (size_t)n * TR_NPAR * 8, cudaMemcpyHostToDevice, st));
    }
    k6_eval_kernel<<<(n + 3) / 4, 128, 0, st>>>(t->tab, t->cst, nb, t->nbp, t->const_b, t->const_d, n, rep ? (const int*)(W + o_rep) : nullptr,
                                                (const double*)(W + o_par), kind ? (const int*)(W + o_kind) : nullptr,
                                                (const int*)(W + o_on), (const double*)(W + o_draw), (double*)(W + o_np), (double*)(W + o_h),
                                                (double*)(W + o_lik), (double*)(W + o_pr), (double*)(W + o_rates), (double*)(W + o_adq));
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    if (out_params) LR_CUDA(cudaMemcpyAsync(out_params, W + o_np, (size_t)n * TR_NPAR * 8, cudaMemcpyDeviceToHost, st));
    if (out_hast) LR_CUDA(cudaMemcpyAsync(out_hast, W + o_h, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    if (lik) LR_CUDA(cudaMemcpyAsync(lik, W + o_lik, (size_t)n * 16, cudaMemcpyDeviceToHost, st));
    if (prior) LR_CUDA(cudaMemcpyAsync(prior, W + o_pr, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    if (rates) LR_CUDA(cudaMemcpyAsync(rates, W + o_rates, (size_t)n * 2 * nb * 8, cudaMemcpyDeviceToHost, st));
    if (adequacy) LR_CUDA(cudaMemcpyAsync(adequacy, W + o_adq, (size_t)n * 24, cudaMemcpyDeviceToHost, st));
    LR_CUDA(cudaStreamSynchronize(st));
    return LR_OK;
}

extern "C" int lr_trend_state_host(lr_trend_t t, double* h_state) {
    LR_REQUIRE(t && h_state, "lr_trend_state_host: null pointer");
    LR_CUDA(cudaSetDevice(t->h->device));
    { int rc0 = lr_order(t->h, &t->last, t->h->stream); if (rc0 != LR_OK) return rc0; }
    LR_CUDA(cudaStreamSynchronize(t->h->stream));
    // [n_chains][LR_TREND_STATE_DOUBLES]: parameters, likB, likD, prior, then iteration and accepted as doubles
    TrendChain* tmp = new TrendChain[t->n_chains];
    cudaError_t e = cudaMemcpy(tmp, t->st, (size_t)t->n_chains * sizeof(TrendChain), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { delete[] tmp; lr_set_error("lr_trend_state_host: %s", cudaGetErrorString(e)); return LR_ERR_CUDA; }
    for (int c = 0; c < t->n_chains; ++c) {
        double* o = h_state + (size_t)c * LR_TREND_STATE_DOUBLES;
        for (int k = 0; k < TR_NPAR; ++k) o[k] = tmp[c].p[k];
        o[6] = tmp[c].likB; o[7] = tmp[c].likD; o[8] = tmp[c].prior; o[9] = (double)tmp[c].it; o[10] = (double)tmp[c].accepted;
        o[11] = (double)tmp[c].rep;
    }
    delete[] tmp;
    return LR_OK;
}

extern "C" int lr_trend_set_beta_host(lr_trend_t t, const double* h_beta) {
    LR_REQUIRE(t && h_beta, "lr_trend_set_beta_host: null pointer");
    return lr_set_beta(t->h, &t->last, t->n_chains, h_beta, "lr_trend_set_beta_host", [&](const double* d_beta, cudaStream_t st) {
        k6_set_beta_kernel<<<(t->n_chains + 127) / 128, 128, 0, st>>>(t->st, t->n_chains, d_beta);
    });
}

extern "C" int lr_trend_swap_info(lr_trend_t t, double* d_info, void* stream) {
    LR_REQUIRE(t && d_info, "lr_trend_swap_info: null pointer");
    return lr_launch_ordered(t->h, &t->last, stream, [&](cudaStream_t st) {
        k6_swap_info_kernel<<<(t->n_chains + 127) / 128, 128, 0, st>>>(t->st, t->n_chains, d_info);
    });
}

static int trend_swap_apply(lr_trend_t t, const double* d_info_all, int64_t table_first, int64_t n_all, int64_t first, int32_t ladder,
                            uint64_t round, void* stream, const char* who) {
    LR_REQUIRE(t, "%s: null pointer", who);
    return lr_swap_apply(t->h, &t->last, t->n_chains, d_info_all, table_first, n_all, first, ladder, stream, who,
                         [&](int blocks, int threads, cudaStream_t st) {
                             k6_swap_apply_kernel<<<blocks, threads, 0, st>>>(t->st, t->n_chains, d_info_all, table_first, n_all, first,
                                                                              ladder, round, (uint32_t)t->seed, (uint32_t)(t->seed >> 32));
                         });
}

extern "C" int lr_trend_swap_apply(lr_trend_t t, const double* d_info_all, int64_t n_all, int64_t first, int32_t ladder, uint64_t round,
                                   void* stream) {
    return trend_swap_apply(t, d_info_all, 0, n_all, first, ladder, round, stream, "lr_trend_swap_apply");
}

extern "C" int lr_trend_swap_step(lr_trend_t t, int32_t ladder, uint64_t round) {
    LR_REQUIRE(t != nullptr, "lr_trend_swap_step: null chains");
    return lr_swap_step(t->h, t->chain_id0, t->n_chains, ladder, t->rep_of_chain, "lr_trend",
                        [&](double* d_info) { return lr_trend_swap_info(t, d_info, t->h->stream); },
                        [&](const double* d_info) {
                            return trend_swap_apply(t, d_info, t->chain_id0, t->n_chains, t->chain_id0, ladder, round, t->h->stream,
                                                    "lr_trend_swap_step");
                        });
}

extern "C" int lr_trend_temper_host(lr_trend_t t, double* h_beta, int64_t* h_swaps) {
    LR_REQUIRE(t != nullptr, "lr_trend_temper_host: null chains");
    return lr_temper_host(t->h, &t->last, t->st, t->n_chains, h_beta, h_swaps, "lr_trend_temper_host");
}
