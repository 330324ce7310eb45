// K7: DDRate (SURVEY 8 f-4) -- fixed-dimension Metropolis-Hastings chains on the binned statistics of K1 with
// diversity-dependent birth and death rates against a constant or logistic carrying capacity.  Replaces the loop of
// DDRatev3.py:242-292 with likelihood_function (:82-124), calc_prior (:127-141) and the literate_library.py proposals
// (update_sliding_win :124-128, update_multiplier_proposal_vec :156-165).
//
//   niche_j  = div_0 + L / (1 + exp(-k (j - x0)))   (-m_birth >= 2 / -m_death 2)   or   L + div_0   (-m_* 1)
//   lambda_j = l_max - (l_max - l_f) (br_j / niche_j) ** nuB,   l_max = l_f + l_f l_mul               (:70-74)
//   mu_j     = m_min + (l_f - m_min) (br_j / niche_j) ** nuD,   m_min = l_f - l_f m_mul               (:76-80)
//   log-lik  = sum_j log(lambda_j) sp_j - lambda_j br_j + sum_j log(mu_j) ex_j - mu_j br_j  [+ genre term, -m_birth 3, :99-102]
//
// One warp = one chain, whole loop on device (the layout of K6): lane p < 11 owns parameter p (Philox draw, multiplier,
// prior difference without logarithms), lane 11 draws the two branch uniforms, lane 12 the sliding-window and the acceptance
// uniform (accept test through a single-precision bracket of log u); bins are strided over the lanes.  A term none of whose
// parameters was touched keeps its stored value, and so do the logarithms of the niche of the first 32 bins.  The genre term of
// -m_birth 3 needs births and time at risk of the genre table inside [origin, origin + x0) and [origin + x0, present):
// one strided pass over the (small, L1-resident) genre table whenever x0 is proposed, cached otherwise.
#include "lr_common.cuh"

#define DD_NPAR LR_DD_NPAR
#define DD_ROWS 6
#define DD_SP 0
#define DD_EX 1
#define DD_BR 2
#define DD_LNBR 3          // log(br): niche_frac ** nu = exp(nu (log br - log niche))
#define DD_XB 4
#define DD_XD 5
#define DD_SMALL 0.000000000000001      // SMALL_NUMBER, DDRatev3.py:54
#define DD_LN_MULT 0.19062035960864987  // 2 log(1.1)
// parameter indices (:83)
#define P_LF 0
#define P_LMUL 1
#define P_K 2
#define P_X0 3
#define P_DIV0 4
#define P_L 5
#define P_MMUL 6
#define P_NUB 7
#define P_NUD 8
#define P_G1 9
#define P_G2 10

struct DDChain {
    double p[DD_NPAR];
    double likB, likD, likG, prior;
    double g[4];           // genre statistics of the current x0: births and time at risk in the two windows
    long long it, accepted;
    unsigned chain;
    int rep;
    double beta;           // inverse temperature of a tempered ladder (1: the reference's chain)
    long long swaps[2];    // temperature swaps proposed, accepted
};

struct lr_dd_s {
    lr_handle_t h;
    lr_last_stream last;           // stream that touched the object last (lr_order)
    int n_rep, n_bins, nbp, m_birth, m_death, n_genre;
    double origin, present;
    double* tab;           // device [n_rep][DD_ROWS][nbp]
    double* cst;           // device [n_rep][4]: sum x, sum x^2 (adequacy), -sum br (death likelihood of -m_death <= 0), max br
    double* genre;         // device [2][n_genre] (ts, te) or null
    int n_chains;
    uint64_t seed;
    int64_t chain_id0;     // global id of chain 0 (ladders are numbered by global id)
    int* rep_of_chain;     // host [n_chains]: replicate of every chain (swap_step refuses ladders that mix replicates)
    DDChain* st;
    double f[DD_NPAR];     // Bernoulli probability of every parameter in the multiplier move (:208-225)
    unsigned depB, depD;   // parameters the birth side / the death side depend on
};

namespace {

struct DDView {
    const double* tab;         // as a kernel argument: the tables of all replicates; after dd_select(): this chain's replicate
    const double* cst;
    const double* genre;
    int nb, nbp, mb, md, ng;
    double origin, present, ln_k0l, k0l, Sx, Sxx, likD_const;      // the last five are filled by dd_select()
};

// the view of one replicate (statistics table and its constants; PRIOR_K0_L = max br of that replicate, DDRatev3.py:53)
__device__ __forceinline__ DDView dd_select(DDView v, int rep) {
    v.tab += (size_t)rep * DD_ROWS * v.nbp;
    const double* c = v.cst + 4 * rep;
    v.Sx = c[0]; v.Sxx = c[1]; v.likD_const = c[2]; v.k0l = c[3]; v.ln_k0l = log(c[3]);
    return v;
}

__device__ __forceinline__ double dd_floor(double r) { return r > 0.0 ? r : DD_SMALL; }

// niche of bin j for the two kinds of carrying capacity (:64-68)
__device__ __forceinline__ double dd_niche_logistic(const double* p, int j) {
    return p[P_DIV0] + p[P_L] / (1.0 + exp(-p[P_K] * ((double)j - p[P_X0])));
}

// rates, niche and niche fraction of bin j as likelihood_function leaves them (:86-116)
__device__ __forceinline__ void dd_bin(const DDView& v, const double* p, int j, double br, double lnbr, bool doB, bool doD,
                                       double& lam, double& mu, double& niche_out, double& nf_out) {
    const bool needL = (doB && v.mb >= 2) || (doD && v.md == 2), needC = (doB && v.mb == 1) || (doD && v.md == 1);
    const double nicheC = p[P_L] + p[P_DIV0];
    const double nicheL = needL ? dd_niche_logistic(p, j) : 1.0;
    const double ln_nicheL = needL ? log(nicheL) : 0.0, ln_nicheC = needC ? log(nicheC) : 0.0;
    lam = 0.0; mu = 1.0; niche_out = 1.0; nf_out = 1.0;
    if (doB) {
        if (v.mb == 0) {
            lam = p[P_LF] * p[P_LMUL];                                   // :87 (no floor in the reference)
        } else {
            const double x = exp(p[P_NUB] * (lnbr - (v.mb == 1 ? ln_nicheC : ln_nicheL)));
            const double rmax = p[P_LF] + p[P_LF] * p[P_LMUL];
            lam = dd_floor(rmax - (rmax - p[P_LF]) * x);
            niche_out = v.mb == 1 ? nicheC : nicheL;
            nf_out = br / niche_out;
        }
    }
    if (doD && v.md >= 1) {
        const double x = exp(p[P_NUD] * (lnbr - (v.md == 1 ? ln_nicheC : ln_nicheL)));
        const double rmin = p[P_LF] - p[P_LF] * p[P_MMUL];
        mu = dd_floor(rmin + (p[P_LF] - rmin) * x);
        niche_out = v.md == 1 ? nicheC : nicheL;
        nf_out = br / niche_out;
    }
}

// Logarithms that survive from one iteration to the next: log niche of bin `lane` (the first 32 bins, one per lane) for the
// logistic carrying capacity, log(L + div_0) for the constant one, log g_lambda1/2.  They are recomputed only when one of the
// parameters they depend on is proposed.
struct DDCache {
    double lnL0, lnC, lg1, lg2;
    // log logistic niche of the bins beyond the first 32 (bin j lives in lane j % 32, which alone reads and writes entry j - 32):
    // per warp in shared memory, two buffers; sel = the buffer that holds the values of the accepted state.  Null: no cache.
    double* tail;          // [2][nt]
    int nt, sel;
};

// this lane's bin of the first 32: statistics held in registers for the whole launch
struct DDBin0 { double sp, ex, br, lnbr; };

// (first: the bin of lane 0 -- 0 for one warp per chain, 32 w for warp w of the wide build)
__device__ __forceinline__ DDBin0 dd_bin0(const DDView& v, int lane, int first = 0) {
    DDBin0 b;
    const int j = first + lane;
    const bool in = j < v.nb;
    b.sp = in ? v.tab[DD_SP * v.nbp + j] : 0.0;
    b.ex = in ? v.tab[DD_EX * v.nbp + j] : 0.0;
    b.br = in ? v.tab[DD_BR * v.nbp + j] : 0.0;
    b.lnbr = in ? v.tab[DD_LNBR * v.nbp + j] : 0.0;
    return b;
}

// Per-lane partial sums over the bins first + lane, first + lane + stride, ... (one warp per chain: first 0, stride 32; warp w of
// W per chain: first 32 w, stride 32 W).  termB / termD (W > 1): every bin's term is also stored at its bin index.
__device__ __forceinline__ void dd_lik_partial(const DDView& v, const DDBin0& b0, int first, int stride, const double* p, int lane, bool doB,
                                               bool doD, bool newL, bool newC, DDCache& c, double& sB, double& sD,
                                               double* termB = nullptr, double* termD = nullptr) {
    const bool evalD = doD && v.md >= 1;
    sB = 0.0; sD = 0.0;
    if (doB || evalD) {
        const bool needL = (doB && v.mb >= 2) || (evalD && v.md == 2), needC = (doB && v.mb == 1) || (evalD && v.md == 1);
        if (needL && newL) c.lnL0 = log(dd_niche_logistic(p, first + lane));
        if (needC && newC) c.lnC = log(p[P_L] + p[P_DIV0]);
        if (doB) {
            double lam = p[P_LF] * p[P_LMUL];                            // :87 (no floor in the reference)
            if (v.mb >= 1) {
                const double x = exp(p[P_NUB] * (b0.lnbr - (v.mb == 1 ? c.lnC : c.lnL0)));
                const double rmax = p[P_LF] + p[P_LF] * p[P_LMUL];
                lam = dd_floor(rmax - (rmax - p[P_LF]) * x);
            }
            sB = log(lam) * b0.sp - lam * b0.br;
        }
        if (evalD) {
            const double x = exp(p[P_NUD] * (b0.lnbr - (v.md == 1 ? c.lnC : c.lnL0)));
            const double rmin = p[P_LF] - p[P_LF] * p[P_MMUL];
            const double mu = dd_floor(rmin + (p[P_LF] - rmin) * x);
            sD = log(mu) * b0.ex - mu * b0.br;
        }
    }
    if (termB != nullptr && first + lane < v.nb) { termB[first + lane] = sB; termD[first + lane] = sD; }
    if (doB || evalD) {
        const bool needL = (doB && v.mb >= 2) || (evalD && v.md == 2);
        for (int j = first + lane + stride; j < v.nb; j += stride) {
            const double br = __ldg(v.tab + DD_BR * v.nbp + j), lnbr = __ldg(v.tab + DD_LNBR * v.nbp + j);
            double lnL = 0.0, tB = 0.0, tD = 0.0;
            if (needL) {
                if (c.tail == nullptr) lnL = log(dd_niche_logistic(p, j));
                else if (newL) { lnL = log(dd_niche_logistic(p, j)); c.tail[(c.sel ^ 1) * c.nt + j - 32] = lnL; }
                else lnL = c.tail[c.sel * c.nt + j - 32];
            }
            if (doB) {
                double lam = p[P_LF] * p[P_LMUL];
                if (v.mb >= 1) {
                    const double x = exp(p[P_NUB] * (lnbr - (v.mb == 1 ? c.lnC : lnL)));
                    const double rmax = p[P_LF] + p[P_LF] * p[P_LMUL];
                    lam = dd_floor(rmax - (rmax - p[P_LF]) * x);
                }
                tB = log(lam) * __ldg(v.tab + DD_SP * v.nbp + j) - lam * br;
                sB += tB;
            }
            if (evalD) {
                const double x = exp(p[P_NUD] * (lnbr - (v.md == 1 ? c.lnC : lnL)));
                const double rmin = p[P_LF] - p[P_LF] * p[P_MMUL];
                const double mu = dd_floor(rmin + (p[P_LF] - rmin) * x);
                tD = log(mu) * __ldg(v.tab + DD_EX * v.nbp + j) - mu * br;
                sD += tD;
            }
            if (termB != nullptr) { termB[j] = tB; termD[j] = tD; }
        }
        if (c.tail != nullptr && needL && newL) c.sel ^= 1;       // the recomputed values sit in the other buffer
    } else if (termB != nullptr) {
        for (int j = first + lane + stride; j < v.nb; j += stride) { termB[j] = 0.0; termD[j] = 0.0; }
    }
}

// newL / newC: a parameter of the logistic / constant carrying capacity differs from the one `c` was computed for
// `extra`: a per-lane term (Hastings share + prior difference of the lane's parameter) that rides the same butterfly; its warp
// total comes back in place.
// W warps per chain (W > 1): this warp's bins start at `first`; termB / termD are this iteration's [nbp] buffers of shared
// memory.  Every warp stores the terms of its bins there and then adds up all bins in the one-warp order (lane l its bins l,
// l + 32, ... ascending, then one butterfly), so the chain does not depend on W.
template <int W = 1>
__device__ __forceinline__ void dd_lik(const DDView& v, const DDBin0& b0, const double* p, int lane, bool doB, bool doD, bool newL,
                                       bool newC, DDCache& c, double& likB, double& likD, double& extra, int first = 0,
                                       double* termB = nullptr, double* termD = nullptr) {
    double sB, sD;
    if constexpr (W == 1) {
        dd_lik_partial(v, b0, 0, 32, p, lane, doB, doD, newL, newC, c, sB, sD);
    } else {
        dd_lik_partial(v, b0, first, 32 * W, p, lane, doB, doD, newL, newC, c, sB, sD, termB, termD);
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
    if (doD) likD = v.md >= 1 ? sD : v.likD_const;                   // death rate 1 in every bin (:105-106)
}

// births and time at risk of the genre table in [origin, c) and [c, present)   (precompute_events, :100-101)
__device__ __forceinline__ void dd_genre_stats(const DDView& v, double x0, int lane, double g[4]) {
    const double O = v.origin, c = v.origin + x0, Pn = v.present;
    double s1 = 0, b1 = 0, s2 = 0, b2 = 0;
    for (int i = lane; i < v.ng; i += 32) {
        const double ts = __ldg(v.genre + i), te = __ldg(v.genre + v.ng + i);
        if (ts >= O && ts < c) s1 += 1.0;
        if (ts >= c && ts < Pn) s2 += 1.0;
        const double d1 = fmin(te, c) - fmax(ts, O), d2 = fmin(te, Pn) - fmax(ts, c);
        if (d1 > 0.0) b1 += d1;
        if (d2 > 0.0) b2 += d2;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, o); b1 += __shfl_xor_sync(0xffffffffu, b1, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o); b2 += __shfl_xor_sync(0xffffffffu, b2, o);
    }
    g[0] = s1; g[1] = b1; g[2] = s2; g[3] = b2;
}

__device__ __forceinline__ double dd_genre_lik(const double* p, const double g[4], bool new1, bool new2, DDCache& c) {
    if (new1) c.lg1 = log(p[P_G1]);
    if (new2) c.lg2 = log(p[P_G2]);
    return (c.lg1 * g[0] - p[P_G1] * g[1]) + (c.lg2 * g[2] - p[P_G2] * g[3]);                    // :102
}

// prior term of parameter `lane` (calc_prior :127-141; closed forms of scipy's gamma / beta logpdf)
__device__ __forceinline__ double dd_prior_term(const DDView& v, int lane, double x) {
    switch (lane) {
        case P_LF: case P_K: case P_G1: case P_G2: return x < 0.0 ? -INFINITY : -x / 10.0 - 2.302585092994046;      // Gamma(1, scale 10)
        case P_LMUL: return x < 0.0 ? -INFINITY : -x;                                                                  // Gamma(1, scale 1)
        case P_X0: return (v.origin + x >= v.present) ? -INFINITY : 0.0;                                               // :139-140
        case P_DIV0: case P_L: return x < 0.0 ? -INFINITY : -x / v.k0l - v.ln_k0l;                                     // Gamma(1, scale max br)
        case P_MMUL: return (x >= 0.0 && x < 1.0) ? 0.1823215567939546 + 0.2 * log1p(-x) : -INFINITY;                  // Beta(1, 1.2)
        case P_NUB: case P_NUD: return x > 0.0 ? 2.0 * log(2.0 * x) - 2.0 * x : -INFINITY;                            // Gamma(3, scale .5)
        default: return 0.0;
    }
}

// Per-lane constants of the prior difference used inside the loop (no logarithm except for the rare m_mul window move):
// prior(x') - prior(x) = -coef (x' - x) [+ 2 lm for the Gamma(3) parameters, which only move by multipliers with log-multiplier lm]
struct DDPriorLane { double coef; int cls; };      // cls 0 Gamma(1, .), 1 Gamma(3, .5), 2 x0, 3 m_mul, 4 none
__device__ __forceinline__ DDPriorLane dd_prior_lane(const DDView& v, int lane) {
    DDPriorLane r; r.coef = 0.0; r.cls = 4;
    if (lane == P_LF || lane == P_K || lane == P_G1 || lane == P_G2) { r.coef = 0.1; r.cls = 0; }
    if (lane == P_LMUL) { r.coef = 1.0; r.cls = 0; }
    if (lane == P_DIV0 || lane == P_L) { r.coef = 1.0 / v.k0l; r.cls = 0; }
    if (lane == P_NUB || lane == P_NUD) { r.coef = 2.0; r.cls = 1; }
    if (lane == P_X0) r.cls = 2;
    if (lane == P_MMUL) r.cls = 3;
    return r;
}
__device__ __forceinline__ double dd_prior_delta(const DDView& v, const DDPriorLane& pl, double x, double xn, double lm) {
    double d = -pl.coef * (xn - x);
    if (pl.cls == 1) d += 2.0 * lm;
    bool bad = false;
    if (pl.cls == 0) bad = xn < 0.0;
    if (pl.cls == 1) bad = !(xn > 0.0);
    if (pl.cls == 2) bad = v.origin + xn >= v.present;                                     // :139-140
    if (pl.cls == 3) {
        bad = !(xn >= 0.0 && xn < 1.0);
        if (!bad && xn != x) d = 0.2 * (log1p(-xn) - log1p(-x));                           // Beta(1, 1.2)
    }
    return bad ? -INFINITY : d;
}

// update_sliding_win (literate_library.py:124-128) with m = 0
__device__ __forceinline__ double dd_slide(double x, double u, double M, double d) {
    double y = x + (u - 0.5) * d;
    if (y > M) y = M - (y - M);
    return fabs(y);
}

__device__ __forceinline__ void dd_bcast(double mine, double* p) {
#pragma unroll
    for (int k = 0; k < DD_NPAR; ++k) p[k] = __shfl_sync(0xffffffffu, mine, k);
}

// kind: 0 multiplier move (mask `on`, uniform `draw`), 1 sliding window on x0, 2 sliding window on m_mul (uniform `draw`)
__device__ __forceinline__ double dd_propose(const DDView& v, int lane, int kind, double x, bool on, double draw, double& hast) {
    hast = 0.0;
    if (kind == 1) return lane == P_X0 ? dd_slide(x, draw, v.present, 1.5) : x;        // :251
    if (kind == 2) return lane == P_MMUL ? dd_slide(x, draw, 1.0, 0.05) : x;           // :253
    if (!on) return x;
    const double lm = DD_LN_MULT * (draw - 0.5);
    hast = lm;
    return x * exp_small(lm);
}

__device__ __forceinline__ void dd_adequacy(const DDView& v, const double* p, int lane, double out[3]) {
    double sy = 0, syy = 0, sxy = 0;
    for (int j = lane; j < v.nb; j += 32) {
        double lam, mu, ni, nf;
        dd_bin(v, p, j, __ldg(v.tab + DD_BR * v.nbp + j), __ldg(v.tab + DD_LNBR * v.nbp + j), true, true, lam, mu, ni, nf);
        const double xb = __ldg(v.tab + DD_XB * v.nbp + j), xd = __ldg(v.tab + DD_XD * v.nbp + j);
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

// the four per-bin series of the log row (:287): birth rates, death rates, niche, niche fraction
__device__ __forceinline__ void dd_series(double* out, const DDView& v, const double* p, int lane) {
    for (int j = lane; j < v.nb; j += 32) {
        const double br = __ldg(v.tab + DD_BR * v.nbp + j);
        double lam, mu, ni, nf;
        dd_bin(v, p, j, br, __ldg(v.tab + DD_LNBR * v.nbp + j), true, true, lam, mu, ni, nf);
        out[j] = lam; out[v.nb + j] = mu; out[2 * v.nb + j] = ni; out[3 * v.nb + j] = nf;
    }
}

__device__ __forceinline__ void dd_record(double* rec, const DDView& v, const double* p, double mine, double likB, double likD,
                                          double likG, long long it, long long accepted, double beta, int lane) {
    double adq[3];
    dd_adequacy(v, p, lane, adq);
    const double prior = warp_sum(dd_prior_term(v, lane, mine));
    if (lane == 0) {
        rec[0] = (double)it; rec[1] = likB + likD + likG; rec[2] = likB; rec[3] = likD; rec[4] = prior; rec[16] = likG;
        rec[17] = adq[0]; rec[18] = adq[1]; rec[19] = adq[2]; rec[20] = (double)accepted; rec[21] = beta; rec[22] = 0.0; rec[23] = 0.0;
    }
#pragma unroll
    for (int k = 0; k < DD_NPAR; ++k)
        if (lane == k) rec[5 + k] = p[k];
    dd_series(rec + LR_DD_REC_HEAD, v, p, lane);
}

struct DDRun {
    DDChain* st;
    int n_chains;
    DDView v;
    uint32_t k0, k1;
    long long n_iter, sample_every;
    double* records;
    int rec_doubles;
    double f[DD_NPAR];
    unsigned depB, depD;
    int tail_n;            // entries per buffer of the shared-memory log-niche cache of the bins beyond the first 32 (0: none)
};

// W == 1: one warp per chain, four chains per CTA.  W = 2 or 4 (the wide build, as k6_trend_kernel<W>): one CTA of W warps per
// chain; warp w evaluates bins 32 w + lane (+ 32 W k), every warp draws the same random numbers and takes the same decision, the
// per-bin terms are exchanged through shared memory (double-buffered by iteration parity, one __syncthreads per iteration) and
// added in the one-warp order (dd_lik) -- the same chain, bit for bit.
template <int W>
__global__ void __launch_bounds__(W == 1 ? 128 : 32 * W, W == 1 ? 3 : 2) k7_dd_kernel(const DDRun P) {
    const int lane = threadIdx.x & 31, wq = threadIdx.x >> 5;
    const int first = W == 1 ? 0 : 32 * wq, stride = 32 * W;
    const int c = W == 1 ? blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5) : blockIdx.x;
    if (c >= P.n_chains) return;
    DDChain* S = P.st + c;
    const DDView v = dd_select(P.v, S->rep);
    const unsigned chain = S->chain;
    double mine = lane < DD_NPAR ? S->p[lane] : 0.0;
    double p[DD_NPAR];
    dd_bcast(mine, p);
    double likB = S->likB, likD = S->likD, likG = S->likG;
    double g[4] = {S->g[0], S->g[1], S->g[2], S->g[3]};
    const DDBin0 b0 = dd_bin0(v, lane, first);
    const DDPriorLane pl = dd_prior_lane(v, lane);
    const unsigned maskL = (1u << P_K) | (1u << P_X0) | (1u << P_DIV0) | (1u << P_L), maskC = (1u << P_DIV0) | (1u << P_L);
    // the log-niche cache of the bins beyond each warp's register bin: W == 1 [warp][2][tail_n], W > 1 one CTA-wide [2][tail_n]
    // indexed by bin, followed by the per-bin terms [2 parities][2 sides][nbp]
    extern __shared__ double tail_s[];
    double* terms = tail_s + 2 * (size_t)P.tail_n;
    DDCache cache;
    cache.nt = P.tail_n; cache.sel = 0;
    cache.tail = P.tail_n > 0 ? (W == 1 ? tail_s + (size_t)(threadIdx.x >> 5) * 2 * P.tail_n : tail_s) : nullptr;
    if (cache.tail != nullptr)
        for (int j = first + lane + stride; j < v.nb; j += stride) cache.tail[j - 32] = log(dd_niche_logistic(p, j));
    cache.lnL0 = log(dd_niche_logistic(p, first + lane));
    cache.lnC = log(p[P_L] + p[P_DIV0]);
    cache.lg1 = log(p[P_G1]); cache.lg2 = log(p[P_G2]);
    long long it = S->it, accepted = S->accepted;
    const long long it_end = it + P.n_iter;
    double fmine = 0.0;
#pragma unroll
    for (int k = 0; k < DD_NPAR; ++k)
        if (lane == k) fmine = P.f[k];
    const bool can_slide = v.mb >= 1 || v.md >= 1;
    long long next_sample = (it + P.sample_every - 1) / P.sample_every * P.sample_every;
    long long rec_idx = 0;
    if constexpr (W > 1) __syncthreads();              // every warp has read the chain's state before warp 0 may rewrite it

    for (; it < it_end; ++it) {
        const Philox4 r = philox4x32_10((uint32_t)it, (uint32_t)((unsigned long long)it >> 32), (uint32_t)lane | (0x70u << 8), chain, P.k0, P.k1);
        const double ua = u01(r.x, r.y), ub = u01(r.z, r.w);
        const double rr1 = __shfl_sync(0xffffffffu, ua, 11), rr2 = __shfl_sync(0xffffffffu, ub, 11);
        const double us = __shfl_sync(0xffffffffu, ua, 12);
        const double u_acc = __shfl_sync(0xffffffffu, ub, 12);
        const int kind = (rr1 < 0.1 && can_slide) ? (rr2 < 0.5 ? 1 : 2) : 0;                  // :248-258
        const bool on = kind == 0 && (((double)r.x + 0.5) * 2.3283064365386963e-10) < fmine;
        double h;
        const double prop = dd_propose(v, lane, kind, mine, on, kind == 0 ? u01(r.y, r.z) : us, h);
        unsigned touched = __ballot_sync(0xffffffffu, on);
        if (kind == 1) touched = 1u << P_X0;
        if (kind == 2) touched = 1u << P_MMUL;
        double q[DD_NPAR];
        dd_bcast(prop, q);
        double hp = h + dd_prior_delta(v, pl, mine, prop, h);       // summed in the butterfly of the likelihood
        double nB = likB, nD = likD, nG = likG;
        double ng[4] = {g[0], g[1], g[2], g[3]};
        DDCache nc = cache;
        const bool doB = (touched & P.depB) != 0, doD = (touched & P.depD) != 0;
        double* tB = terms + (size_t)(it & 1) * 2 * v.nbp;
        double* tD = tB + v.nbp;
        dd_lik<W>(v, b0, q, lane, doB, doD, (touched & maskL) != 0, (touched & maskC) != 0, nc, nB, nD, hp, first, tB, tD);
        if (v.mb == 3) {
            if (touched & (1u << P_X0)) dd_genre_stats(v, q[P_X0], lane, ng);
            if (touched & ((1u << P_X0) | (1u << P_G1) | (1u << P_G2)))
                nG = dd_genre_lik(q, ng, (touched & (1u << P_G1)) != 0, (touched & (1u << P_G2)) != 0, nc);
        }
        // tempered: only the likelihood (genre term included) is raised to the power beta (1.0 * d == d at beta = 1).  beta is
        // read from the state here rather than held from before the loop: with the register copy nvcc contracts the rate
        // bound l_f + l_f l_mul of the one-warp build into an fma, which moves an untempered chain by an ulp
        const double x = S->beta * ((nB + nD + nG) - (likB + likD + likG)) + hp;
        if (it == 0 || mh_accept_gt(x, u_acc)) {                                                 // :263
#pragma unroll
            for (int k = 0; k < DD_NPAR; ++k) p[k] = q[k];
            mine = prop;
            likB = nB; likD = nD; likG = nG; cache = nc;
            g[0] = ng[0]; g[1] = ng[1]; g[2] = ng[2]; g[3] = ng[3];
            ++accepted;
        }
        if (it == next_sample) {                                                                 // :274
            if (P.records && (W == 1 || wq == 0))
                dd_record(P.records + ((size_t)rec_idx * P.n_chains + c) * P.rec_doubles, v, p, mine, likB, likD, likG, it, accepted, S->beta, lane);
            ++rec_idx;
            next_sample += P.sample_every;
        }
    }
    if (W > 1 && wq != 0) return;
    const double prior = warp_sum(dd_prior_term(v, lane, mine));
    if (lane < DD_NPAR) S->p[lane] = mine;
    if (lane == 0) {
        S->likB = likB; S->likD = likD; S->likG = likG; S->prior = prior; S->it = it; S->accepted = accepted;
        S->g[0] = g[0]; S->g[1] = g[1]; S->g[2] = g[2]; S->g[3] = g[3];
    }
}

__device__ __forceinline__ void dd_eval_all(const DDView& v, const double* p, double mine, int lane, double& likB, double& likD,
                                            double& likG, double& prior, double g[4]) {
    likB = 0; likD = 0;
    DDCache c;
    c.lnL0 = c.lnC = c.lg1 = c.lg2 = 0.0;
    c.tail = nullptr; c.nt = 0; c.sel = 0;
    double unused = 0.0;
    dd_lik(v, dd_bin0(v, lane), p, lane, true, true, true, true, c, likB, likD, unused);
    likG = 1.0;                                                    // g_birth_lik = 1 unless -m_birth 3 (:84)
    g[0] = g[1] = g[2] = g[3] = 0.0;
    if (v.mb == 3) { dd_genre_stats(v, p[P_X0], lane, g); likG = dd_genre_lik(p, g, true, true, c); }
    prior = warp_sum(dd_prior_term(v, lane, mine));
}

// initial state (:187-201, :229-240)
__global__ void k7_init_kernel(DDChain* st, int n_chains, const int* rep_of_chain, long long chain_id0, const DDView v_all) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n_chains) return;
    const int rep = rep_of_chain ? rep_of_chain[c] : 0;
    const DDView v = dd_select(v_all, rep);
    const double init[DD_NPAR] = {0.5, 1.01, 1.5, v.present - (v.origin + v.present) / 2.0, 10.0, 20000.0, 0.99, 1.0, 1.0, 1.0, 1.0};
    double mine = 0.0;
#pragma unroll
    for (int k = 0; k < DD_NPAR; ++k)
        if (lane == k) mine = init[k];
    double p[DD_NPAR];
    dd_bcast(mine, p);
    double likB, likD, likG, prior, g[4];
    dd_eval_all(v, p, mine, lane, likB, likD, likG, prior, g);
    if (lane < DD_NPAR) st[c].p[lane] = mine;
    if (lane == 0) {
        st[c].likB = likB; st[c].likD = likD; st[c].likG = likG; st[c].prior = prior;
        st[c].g[0] = g[0]; st[c].g[1] = g[1]; st[c].g[2] = g[2]; st[c].g[3] = g[3];
        st[c].it = 0; st[c].accepted = 0; st[c].chain = (unsigned)(chain_id0 + c); st[c].rep = rep;
        st[c].beta = 1.0; st[c].swaps[0] = 0; st[c].swaps[1] = 0;
    }
}

// ---- tempered ladders (new: the reference has no tempering, SURVEY A-15; the swap rule is lr_swap_round, shared with K3)
__global__ void k7_set_beta_kernel(DDChain* st, int n, const double* beta) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) st[i].beta = beta[i];
}

// (likelihood, beta) of every chain, as stored: the untempered likelihood of the current state, genre term included
__global__ void k7_swap_info_kernel(const DDChain* st, int n, double* __restrict__ info) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { info[2 * i] = st[i].likB + st[i].likD + st[i].likG; info[2 * i + 1] = st[i].beta; }
}

__global__ void k7_swap_apply_kernel(DDChain* st, int n_local, const double* __restrict__ info_all, long long table_first,
                                     long long n_all, long long first, int ladder, unsigned long long round, uint32_t k0, uint32_t k1) {
    const int lane = threadIdx.x & 31;
    const int local = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
    if (local >= n_local) return;
    lr_swap_round(info_all, table_first, n_all, first + local, ladder, round, k0, k1, lane, [&](bool paired, bool accept, double beta_p) {
        DDChain* S = st + local;
        if (paired) {
            S->swaps[0] += 1;
            if (accept) { S->swaps[1] += 1; S->beta = beta_p; }
        }
    });
}

__global__ void k7_build_tables(const long long* __restrict__ sp_all, const long long* __restrict__ ex_all, const double* __restrict__ br_all,
                                int nb, int nbp, double* __restrict__ tab_all, double* __restrict__ cst_all) {
    const int rep = blockIdx.x;
    const long long* sp = sp_all + (size_t)rep * nb;
    const long long* ex = ex_all + (size_t)rep * nb;
    const double* br = br_all + (size_t)rep * nb;
    double* tab = tab_all + (size_t)rep * DD_ROWS * nbp;
    double* cst = cst_all + 4 * rep;
    for (int j = threadIdx.x; j < nbp; j += blockDim.x) {
        const bool in = j < nb;
        const double U = in ? (double)sp[j] : 0.0, D = in ? (double)ex[j] : 0.0, K = in ? br[j] : 0.0;
        tab[DD_SP * nbp + j] = U; tab[DD_EX * nbp + j] = D; tab[DD_BR * nbp + j] = K;
        tab[DD_LNBR * nbp + j] = in ? log(K) : 0.0;
        tab[DD_XB * nbp + j] = in ? U / K : 0.0;
        tab[DD_XD * nbp + j] = in ? D / K : 0.0;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double sx = 0, sxx = 0, sk = 0, mx = 0;
        for (int j = 0; j < nb; ++j) {
            const double xb = tab[DD_XB * nbp + j], xd = tab[DD_XD * nbp + j];
            sx += xb + xd; sxx += xb * xb + xd * xd;
            sk += log(1.0) * tab[DD_EX * nbp + j] - 1.0 * tab[DD_BR * nbp + j];      // death rate 1 (:105-106, :118)
            mx = fmax(mx, tab[DD_BR * nbp + j]);
        }
        cst[0] = sx; cst[1] = sxx; cst[2] = sk; cst[3] = mx;        // mx = PRIOR_K0_L (:53)
    }
}

__global__ void k7_eval_kernel(const DDView v_all, int n, const int* rep, const double* params, const int* kind, const int* on, const double* draw,
                               double* out_params, double* out_hast, double* lik, double* prior, double* series, double* adequacy,
                               double* genre) {
    const int lane = threadIdx.x & 31;
    const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (s >= n) return;
    const DDView v = dd_select(v_all, rep ? rep[s] : 0);
    double mine = lane < DD_NPAR ? params[s * DD_NPAR + lane] : 0.0, h = 0.0;
    if (kind) mine = dd_propose(v, lane, kind[s], mine, lane < DD_NPAR && on[s * DD_NPAR + lane] != 0,
                                lane < DD_NPAR ? draw[s * DD_NPAR + lane] : 0.0, h);
    h = warp_sum(h);
    double p[DD_NPAR];
    dd_bcast(mine, p);
    double likB, likD, likG, pr, g[4];
    dd_eval_all(v, p, mine, lane, likB, likD, likG, pr, g);
    double adq[3];
    dd_adequacy(v, p, lane, adq);
    if (lane == 0) {
        if (lik) { lik[3 * s] = likB; lik[3 * s + 1] = likD; lik[3 * s + 2] = likG; }
        if (prior) prior[s] = pr;
        if (out_hast) out_hast[s] = h;
        if (adequacy) { adequacy[3 * s] = adq[0]; adequacy[3 * s + 1] = adq[1]; adequacy[3 * s + 2] = adq[2]; }
        if (genre) { genre[4 * s] = g[0]; genre[4 * s + 1] = g[1]; genre[4 * s + 2] = g[2]; genre[4 * s + 3] = g[3]; }
    }
    if (out_params && lane < DD_NPAR) out_params[s * DD_NPAR + lane] = mine;
    if (series) dd_series(series + (size_t)s * 4 * v.nb, v, p, lane);
}

// update_multiplier (:208-225) and the parameters every term depends on
void dd_model_tables(int mb, int md, double* f, unsigned& depB, unsigned& depD) {
    double w[DD_NPAR];
    const double w0[DD_NPAR] = {1, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0}, w2[DD_NPAR] = {1, 1, 1, 0, 1, 1, 0, 1, 1, 0, 0},
                 w1[DD_NPAR] = {1, 1, 0, 0, 0, 1, 0, 1, 1, 0, 0}, w3[DD_NPAR] = {1, 1, 1, 0, 1, 1, 0, 1, 1, 1, 1};
    const double* src = (mb == 0 && md <= 0) ? w0 : ((mb == 2 || md == 2) ? w2 : w1);
    if (mb == 3) src = w3;
    double s = 0;
    for (int k = 0; k < DD_NPAR; ++k) { w[k] = src[k]; s += w[k]; }
    for (int k = 0; k < DD_NPAR; ++k) f[k] = w[k] / s;
    const unsigned logistic = (1u << P_K) | (1u << P_X0) | (1u << P_DIV0) | (1u << P_L), constK = (1u << P_DIV0) | (1u << P_L);
    depB = (1u << P_LF) | (1u << P_LMUL);
    if (mb >= 1) depB |= (1u << P_NUB) | (mb == 1 ? constK : logistic);
    depD = 0;
    if (md >= 1) depD = (1u << P_LF) | (1u << P_MMUL) | (1u << P_NUD) | (md == 1 ? constK : logistic);
}

DDView dd_view(lr_dd_t t) {
    DDView v;
    v.tab = t->tab; v.cst = t->cst; v.genre = t->genre; v.nb = t->n_bins; v.nbp = t->nbp; v.mb = t->m_birth; v.md = t->m_death;
    v.ng = t->n_genre; v.origin = t->origin; v.present = t->present;
    v.k0l = 0.0; v.ln_k0l = 0.0; v.Sx = 0.0; v.Sxx = 0.0; v.likD_const = 0.0;
    return v;
}

}  // namespace

extern "C" int64_t lr_dd_record_doubles(int32_t n_bins) { return LR_DD_REC_HEAD + 4 * (int64_t)n_bins; }

extern "C" int lr_dd_create(lr_handle_t h, int32_t n_rep, int32_t n_bins, const int64_t* d_sp, const int64_t* d_ex, const double* d_br,
                            double origin, double present, int32_t m_birth, int32_t m_death,
                            const double* h_gts, const double* h_gte, int32_t n_genre,
                            int32_t n_chains, uint64_t seed, int64_t chain_id0, const int32_t* h_rep_of_chain,
                            void* stream, lr_dd_t* out) {
    LR_REQUIRE(h && d_sp && d_ex && d_br && out, "lr_dd_create: null pointer");
    LR_REQUIRE(n_rep >= 1 && n_bins >= 1 && n_chains >= 1, "lr_dd_create: n_rep, n_bins and n_chains must be >= 1");
    LR_REQUIRE(present > origin, "lr_dd_create: present must be later than origin");
    LR_REQUIRE(chain_id0 >= 0 && chain_id0 + n_chains <= 0xffffffffll, "lr_dd_create: chain ids must fit 32 bits");
    if (m_birth < 0 || m_birth > 3 || m_death < 0 || m_death > 2) {
        lr_set_error("lr_dd_create: -m_birth must be 0..3 and -m_death 0..2 (the fixed-rate models -1 stop with NameError in the "
                     "reference, DDRatev3.py:192-195)");
        return LR_ERR_UNSUPPORTED;
    }
    LR_REQUIRE(m_birth != 3 || (h_gts && h_gte && n_genre >= 1), "lr_dd_create: -m_birth 3 needs the genre table (DDRatev3.py:36-38)");
    if (h_rep_of_chain)
        for (int i = 0; i < n_chains; ++i)
            LR_REQUIRE(h_rep_of_chain[i] >= 0 && h_rep_of_chain[i] < n_rep, "lr_dd_create: replicate of chain %d out of range", i);
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    lr_dd_t t = new lr_dd_s();
    memset(t, 0, sizeof(*t));
    t->last.s = st; t->last.valid = 1;
    t->h = h; t->n_rep = n_rep; t->n_bins = n_bins; t->nbp = (n_bins + 3) & ~3; t->m_birth = m_birth; t->m_death = m_death;
    t->n_genre = m_birth == 3 ? n_genre : 0; t->origin = origin; t->present = present; t->n_chains = n_chains; t->seed = seed;
    t->chain_id0 = chain_id0;
    t->rep_of_chain = new int[n_chains];
    for (int i = 0; i < n_chains; ++i) t->rep_of_chain[i] = h_rep_of_chain ? h_rep_of_chain[i] : 0;
    dd_model_tables(m_birth, m_death, t->f, t->depB, t->depD);
    int* d_rep = nullptr;
    cudaError_t e = cudaMallocAsync((void**)&t->tab, (size_t)n_rep * DD_ROWS * t->nbp * sizeof(double), st);
    if (e == cudaSuccess) e = cudaMallocAsync((void**)&t->cst, (size_t)n_rep * 4 * sizeof(double), st);
    if (e == cudaSuccess) e = cudaMallocAsync((void**)&t->st, (size_t)n_chains * sizeof(DDChain), st);
    if (e == cudaSuccess && t->n_genre) e = cudaMallocAsync((void**)&t->genre, (size_t)2 * t->n_genre * sizeof(double), st);
    if (e == cudaSuccess && h_rep_of_chain) e = cudaMallocAsync((void**)&d_rep, (size_t)n_chains * sizeof(int), st);
    if (e != cudaSuccess) { lr_set_error("lr_dd_create: cudaMallocAsync: %s", cudaGetErrorString(e)); lr_dd_destroy(t); return LR_ERR_NOMEM; }
    auto undo = [&]() { if (d_rep) cudaFreeAsync(d_rep, st); lr_dd_destroy(t); };
    if (t->n_genre) {
        LR_CUDA_CLEAN(cudaMemcpyAsync(t->genre, h_gts, (size_t)t->n_genre * sizeof(double), cudaMemcpyHostToDevice, st), undo());
        LR_CUDA_CLEAN(cudaMemcpyAsync(t->genre + t->n_genre, h_gte, (size_t)t->n_genre * sizeof(double), cudaMemcpyHostToDevice, st), undo());
    }
    if (d_rep) LR_CUDA_CLEAN(cudaMemcpyAsync(d_rep, h_rep_of_chain, (size_t)n_chains * sizeof(int), cudaMemcpyHostToDevice, st), undo());
    k7_build_tables<<<n_rep, 128, 0, st>>>((const long long*)d_sp, (const long long*)d_ex, d_br, n_bins, t->nbp, t->tab, t->cst);
    LR_CUDA_CLEAN(cudaGetLastError(), undo());
    // every replicate needs some time at risk: its largest br is the scale of two priors (PRIOR_K0_L, DDRatev3.py:53)
    double* h_cst = new double[(size_t)n_rep * 4];
    cudaError_t ce = cudaMemcpyAsync(h_cst, t->cst, (size_t)n_rep * 4 * sizeof(double), cudaMemcpyDeviceToHost, st);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
    int bad = -1;
    for (int r = 0; ce == cudaSuccess && r < n_rep; ++r)
        if (!(h_cst[4 * r + 3] > 0.0)) { bad = r; break; }
    delete[] h_cst;
    if (ce != cudaSuccess) { lr_set_error("lr_dd_create: %s", cudaGetErrorString(ce)); undo(); return LR_ERR_CUDA; }
    if (bad >= 0) { lr_set_error("lr_dd_create: replicate %d has no time at risk in any bin", bad); undo(); return LR_ERR_INVALID; }
    int threads;
    const int blocks = lr_chain_grid(n_chains, threads);
    k7_init_kernel<<<blocks, threads, 0, st>>>(t->st, n_chains, d_rep, chain_id0, dd_view(t));
    LR_CUDA_CLEAN(cudaGetLastError(), undo());
    h->launches += 2;
    LR_CUDA_CLEAN(cudaStreamSynchronize(st), undo());
    if (d_rep) cudaFreeAsync(d_rep, st);
    *out = t;
    return LR_OK;
}

extern "C" int lr_dd_create_host(lr_handle_t h, int32_t n_rep, int32_t n_bins, const int64_t* h_sp, const int64_t* h_ex, const double* h_br,
                                 double origin, double present, int32_t m_birth, int32_t m_death,
                                 const double* h_gts, const double* h_gte, int32_t n_genre,
                                 int32_t n_chains, uint64_t seed, int64_t chain_id0, const int32_t* h_rep_of_chain, lr_dd_t* out) {
    LR_REQUIRE(h && h_sp && h_ex && h_br, "lr_dd_create_host: null pointer");
    LR_REQUIRE(n_rep >= 1 && n_bins >= 1, "lr_dd_create_host: bad sizes");
    int64_t *d_sp, *d_ex;
    double* d_br;
    int rc = lr_upload_bin_stats(h, (size_t)n_rep * n_bins, h_sp, h_ex, h_br, &d_sp, &d_ex, &d_br);
    if (rc != LR_OK) return rc;
    return lr_dd_create(h, n_rep, n_bins, d_sp, d_ex, d_br, origin, present, m_birth, m_death, h_gts, h_gte, n_genre, n_chains, seed,
                        chain_id0, h_rep_of_chain, h->stream, out);
}

extern "C" int lr_dd_destroy(lr_dd_t t) {
    if (!t) return LR_OK;
    cudaSetDevice(t->h->device);
    lr_order(t->h, &t->last, t->h->stream);
    if (t->tab) cudaFreeAsync(t->tab, t->h->stream);
    if (t->cst) cudaFreeAsync(t->cst, t->h->stream);
    if (t->st) cudaFreeAsync(t->st, t->h->stream);
    if (t->genre) cudaFreeAsync(t->genre, t->h->stream);
    delete[] t->rep_of_chain;
    delete t;
    return LR_OK;
}

extern "C" int64_t lr_dd_records_per_run(lr_dd_t t, int64_t n_iter, int64_t sample_every) {
    if (!t || n_iter <= 0 || sample_every <= 0) return 0;
    long long it0 = 0;
    if (!lr_read_counter(t->h, &t->last, &t->st[0].it, &it0)) return -1;
    return lr_records_per_run(it0, n_iter, sample_every);
}

extern "C" int lr_dd_run(lr_dd_t t, int64_t n_iter, int64_t sample_every, double* d_records, void* stream) {
    LR_REQUIRE(t != nullptr, "lr_dd_run: null chains");
    LR_REQUIRE(n_iter >= 0 && sample_every >= 0, "lr_dd_run: negative count");
    if (n_iter == 0) return LR_OK;
    lr_handle_t h = t->h;
    LR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    { int rc0 = lr_order(h, &t->last, st); if (rc0 != LR_OK) return rc0; }
    DDRun P;
    P.st = t->st; P.n_chains = t->n_chains; P.v = dd_view(t);
    P.k0 = (uint32_t)t->seed; P.k1 = (uint32_t)(t->seed >> 32);
    P.n_iter = n_iter; P.sample_every = sample_every > 0 ? sample_every : (int64_t)1 << 62;
    P.records = sample_every > 0 ? d_records : nullptr;
    P.rec_doubles = (int)lr_dd_record_doubles(t->n_bins);
    for (int k = 0; k < DD_NPAR; ++k) P.f[k] = t->f[k];
    P.depB = t->depB; P.depD = t->depD;
    int threads;
    const int blocks = lr_chain_grid(t->n_chains, threads);
    // Shared memory, up to 48 KB: the log-niche cache of the bins beyond the first 32 (W == 1: [warp][2 buffers][tail_n]
    // doubles, left out if it does not fit), and for W > 1 one [2][tail_n] cache plus the per-bin terms [2][2][nbp] (one warp
    // per chain if they do not fit)
    int W = lr_chain_width(t->n_bins, t->n_chains, h->sm_count, "LR_DD_WIDE");
    P.tail_n = t->n_bins > 32 ? t->nbp - 32 : 0;
    size_t smem = ((size_t)2 * P.tail_n + (size_t)4 * t->nbp) * sizeof(double);
    if (W > 1 && smem > 48 * 1024) W = 1;
    if (W == 1) {
        smem = (size_t)(threads / 32) * 2 * P.tail_n * sizeof(double);
        if (smem > 48 * 1024) { P.tail_n = 0; smem = 0; }
    }
    if (W == 4) k7_dd_kernel<4><<<t->n_chains, 128, smem, st>>>(P);
    else if (W == 2) k7_dd_kernel<2><<<t->n_chains, 64, smem, st>>>(P);
    else k7_dd_kernel<1><<<blocks, threads, smem, st>>>(P);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    return LR_OK;
}

extern "C" int lr_dd_run_host(lr_dd_t t, int64_t n_iter, int64_t sample_every, double* h_records) {
    LR_REQUIRE(t != nullptr, "lr_dd_run_host: null chains");
    const int64_t nrec = (h_records && sample_every > 0) ? lr_dd_records_per_run(t, n_iter, sample_every) : 0;
    return lr_run_into_host(t->h, "lr_dd_run_host", nrec, (size_t)t->n_chains * lr_dd_record_doubles(t->n_bins) * sizeof(double),
                            h_records, [&](double* d_rec) { return lr_dd_run(t, n_iter, d_rec ? sample_every : 0, d_rec, t->h->stream); });
}

extern "C" int lr_dd_eval_host(lr_dd_t t, int32_t n, const int32_t* rep, const double* params, const int32_t* kind, const int32_t* on,
                               const double* draw, double* out_params, double* out_hast, double* lik, double* prior,
                               double* series, double* adequacy, double* genre) {
    LR_REQUIRE(t && params, "lr_dd_eval_host: null pointer");
    LR_REQUIRE(n >= 1, "lr_dd_eval_host: n must be >= 1");
    LR_REQUIRE(!kind || (on && draw), "lr_dd_eval_host: kind needs on and draw");
    if (rep)
        for (int i = 0; i < n; ++i) LR_REQUIRE(rep[i] >= 0 && rep[i] < t->n_rep, "lr_dd_eval_host: replicate of state %d out of range", i);
    lr_handle_t h = t->h;
    LR_CUDA(cudaSetDevice(h->device));
    { int rc0 = lr_order(t->h, &t->last, t->h->stream); if (rc0 != LR_OK) return rc0; }
    const int nb = t->n_bins;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_par = take((size_t)n * DD_NPAR * 8), o_rep = take((size_t)n * 4), o_kind = take((size_t)n * 4), o_on = take((size_t)n * DD_NPAR * 4),
                 o_draw = take((size_t)n * DD_NPAR * 8), o_np = take((size_t)n * DD_NPAR * 8), o_h = take((size_t)n * 8),
                 o_lik = take((size_t)n * 24), o_pr = take((size_t)n * 8), o_ser = take((size_t)n * 4 * nb * 8),
                 o_adq = take((size_t)n * 24), o_g = take((size_t)n * 32);
    int rc = lr_ws_acquire(h, off, h->stream);
    if (rc != LR_OK) return rc;
    char* W = (char*)h->ws;
    cudaStream_t st = h->stream;
    LR_CUDA(cudaMemcpyAsync(W + o_par, params, (size_t)n * DD_NPAR * 8, cudaMemcpyHostToDevice, st));
    if (rep) LR_CUDA(cudaMemcpyAsync(W + o_rep, rep, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    if (kind) {
        LR_CUDA(cudaMemcpyAsync(W + o_kind, kind, (size_t)n * 4, cudaMemcpyHostToDevice, st));
        LR_CUDA(cudaMemcpyAsync(W + o_on, on, (size_t)n * DD_NPAR * 4, cudaMemcpyHostToDevice, st));
        LR_CUDA(cudaMemcpyAsync(W + o_draw, draw, (size_t)n * DD_NPAR * 8, cudaMemcpyHostToDevice, st));
    }
    k7_eval_kernel<<<(n + 3) / 4, 128, 0, st>>>(dd_view(t), n, rep ? (const int*)(W + o_rep) : nullptr, (const double*)(W + o_par), kind ? (const int*)(W + o_kind) : nullptr,
                                                (const int*)(W + o_on), (const double*)(W + o_draw), (double*)(W + o_np), (double*)(W + o_h),
                                                (double*)(W + o_lik), (double*)(W + o_pr), (double*)(W + o_ser), (double*)(W + o_adq),
                                                (double*)(W + o_g));
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    if (out_params) LR_CUDA(cudaMemcpyAsync(out_params, W + o_np, (size_t)n * DD_NPAR * 8, cudaMemcpyDeviceToHost, st));
    if (out_hast) LR_CUDA(cudaMemcpyAsync(out_hast, W + o_h, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    if (lik) LR_CUDA(cudaMemcpyAsync(lik, W + o_lik, (size_t)n * 24, cudaMemcpyDeviceToHost, st));
    if (prior) LR_CUDA(cudaMemcpyAsync(prior, W + o_pr, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    if (series) LR_CUDA(cudaMemcpyAsync(series, W + o_ser, (size_t)n * 4 * nb * 8, cudaMemcpyDeviceToHost, st));
    if (adequacy) LR_CUDA(cudaMemcpyAsync(adequacy, W + o_adq, (size_t)n * 24, cudaMemcpyDeviceToHost, st));
    if (genre) LR_CUDA(cudaMemcpyAsync(genre, W + o_g, (size_t)n * 32, cudaMemcpyDeviceToHost, st));
    LR_CUDA(cudaStreamSynchronize(st));
    return LR_OK;
}

extern "C" int lr_dd_state_host(lr_dd_t t, double* h_state) {
    LR_REQUIRE(t && h_state, "lr_dd_state_host: null pointer");
    LR_CUDA(cudaSetDevice(t->h->device));
    { int rc0 = lr_order(t->h, &t->last, t->h->stream); if (rc0 != LR_OK) return rc0; }
    LR_CUDA(cudaStreamSynchronize(t->h->stream));
    DDChain* tmp = new DDChain[t->n_chains];
    cudaError_t e = cudaMemcpy(tmp, t->st, (size_t)t->n_chains * sizeof(DDChain), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { delete[] tmp; lr_set_error("lr_dd_state_host: %s", cudaGetErrorString(e)); return LR_ERR_CUDA; }
    for (int c = 0; c < t->n_chains; ++c) {
        double* o = h_state + (size_t)c * LR_DD_STATE_DOUBLES;
        for (int k = 0; k < DD_NPAR; ++k) o[k] = tmp[c].p[k];
        o[11] = tmp[c].likB; o[12] = tmp[c].likD; o[13] = tmp[c].likG; o[14] = tmp[c].prior;
        o[15] = (double)tmp[c].it; o[16] = (double)tmp[c].accepted;
        for (int k = 0; k < 4; ++k) o[17 + k] = tmp[c].g[k];
        o[21] = (double)tmp[c].rep; o[22] = 0.0; o[23] = 0.0;
    }
    delete[] tmp;
    return LR_OK;
}

extern "C" int lr_dd_set_beta_host(lr_dd_t t, const double* h_beta) {
    LR_REQUIRE(t && h_beta, "lr_dd_set_beta_host: null pointer");
    return lr_set_beta(t->h, &t->last, t->n_chains, h_beta, "lr_dd_set_beta_host", [&](const double* d_beta, cudaStream_t st) {
        k7_set_beta_kernel<<<(t->n_chains + 127) / 128, 128, 0, st>>>(t->st, t->n_chains, d_beta);
    });
}

extern "C" int lr_dd_swap_info(lr_dd_t t, double* d_info, void* stream) {
    LR_REQUIRE(t && d_info, "lr_dd_swap_info: null pointer");
    return lr_launch_ordered(t->h, &t->last, stream, [&](cudaStream_t st) {
        k7_swap_info_kernel<<<(t->n_chains + 127) / 128, 128, 0, st>>>(t->st, t->n_chains, d_info);
    });
}

static int dd_swap_apply(lr_dd_t t, const double* d_info_all, int64_t table_first, int64_t n_all, int64_t first, int32_t ladder,
                         uint64_t round, void* stream, const char* who) {
    LR_REQUIRE(t, "%s: null pointer", who);
    return lr_swap_apply(t->h, &t->last, t->n_chains, d_info_all, table_first, n_all, first, ladder, stream, who,
                         [&](int blocks, int threads, cudaStream_t st) {
                             k7_swap_apply_kernel<<<blocks, threads, 0, st>>>(t->st, t->n_chains, d_info_all, table_first, n_all, first,
                                                                              ladder, round, (uint32_t)t->seed, (uint32_t)(t->seed >> 32));
                         });
}

extern "C" int lr_dd_swap_apply(lr_dd_t t, const double* d_info_all, int64_t n_all, int64_t first, int32_t ladder, uint64_t round,
                                void* stream) {
    return dd_swap_apply(t, d_info_all, 0, n_all, first, ladder, round, stream, "lr_dd_swap_apply");
}

extern "C" int lr_dd_swap_step(lr_dd_t t, int32_t ladder, uint64_t round) {
    LR_REQUIRE(t != nullptr, "lr_dd_swap_step: null chains");
    return lr_swap_step(t->h, t->chain_id0, t->n_chains, ladder, t->rep_of_chain, "lr_dd",
                        [&](double* d_info) { return lr_dd_swap_info(t, d_info, t->h->stream); },
                        [&](const double* d_info) {
                            return dd_swap_apply(t, d_info, t->chain_id0, t->n_chains, t->chain_id0, ladder, round, t->h->stream,
                                                 "lr_dd_swap_step");
                        });
}

extern "C" int lr_dd_temper_host(lr_dd_t t, double* h_beta, int64_t* h_swaps) {
    LR_REQUIRE(t != nullptr, "lr_dd_temper_host: null chains");
    return lr_temper_host(t->h, &t->last, t->st, t->n_chains, h_beta, h_swaps, "lr_dd_temper_host");
}
