// Device-side building blocks shared by K2 (state evaluation) and K3 (the RJMCMC chains).
//
// One chain (or one state) lives in ONE WARP: lane k holds slot k of the birth side and slot k of
// the death side in registers (rate, log-rate, start time of the segment, the segment's sufficient
// statistics).  Every branch on the proposal type is therefore warp-uniform, insert/delete of a
// rate shift is a register shuffle, and nothing but the read-only prefix tables is touched in
// memory inside the loop.
//
// Likelihood in prefix form.  With piecewise-constant rates the per-bin sums of the reference
// collapse to per-segment sums:
//   BDI_partial_lik (LiteRateForward.py:150-162), model_BDI = 0, mask m = (br > 0), Tk = 1:
//       sum_j m_j [ U_j log(k_j L_j) + D_j log(M_j k_j) - k_j (L_j + M_j) ]
//     = C0 + sum_seg [ logL * U_seg - L * K_seg ] + sum_seg [ logM * D_seg - M * K_seg ],
//       C0 = sum_j m_j (U_j + D_j) log k_j
//   model_BDI = 1 (L -> 0, I = lambda):  log(I) U - I  per bin  ->  [ logL * U_seg - L * N_seg ],  N = #bins with k>0
//       C1 = sum_j m_j D_j log k_j
//   BD_lik_Keiding (:137-148), model_BDI = 2/3: the same two segment sums without mask or constant
//       (model 3 takes the death side from the extinct-only statistics).
// Tables per replicate, each a prefix sum over bins with n_bins+1 entries:
//   T_AB events of the birth side, T_BB exposure of the birth side, T_AD, T_BD same for deaths,
//   T_XB / T_XD prefix sums of the empirical rates sp/br, ex/br (adequacy, literate_library.py:260-279).
#pragma once
#include "lr_common.cuh"

#define LR_NTAB 6
#define T_AB 0
#define T_BB 1
#define T_AD 2
#define T_BD 3
#define T_XB 4
#define T_XD 5
#define LR_NCST 4      // per replicate: C (likelihood constant), sum x, sum x^2, unused

struct lr_dataset_s {
    lr_handle_t h;
    int n_rep, n_bins, model;
    double start_time, end_time;
    int s0f;               // floor(start_time): a shift at time t starts bin floor(t) - s0f (:262, :125-135)
    double* tab;           // device [n_rep][LR_NTAB][n_bins+1]
    double* cst;           // device [n_rep][LR_NCST]
    double* terms;         // device [n_rep][4][n_bins]: A^b, B^b, A^d, B^d of every bin, the terms the tables sum
    lr_last_stream last;   // stream that built or read the tables last (lr_order)
};

// constants of the sampler (LiteRateForward.py:165, :586-590, :101-102)
#define LR_LN_MULT 0.19062035960864987      // 2*log(1.1), window of update_multiplier_freq (:165,:169)
#define LR_BETA_NORM (-13.73622922703656)   // 2*lgamma(10) - lgamma(20): log B(10,10)
#define LR_SHAPE_BETA 10.0
#define LR_MIN_DT 1.0                       // min_allowed_t (:587)

struct DataView {
    const double* tab;     // this replicate's tables
    int nb, s0f;
    double C, Sx, Sxx;
    double start_time, end_time, log_span;
};

__device__ __forceinline__ DataView make_view(const double* tab_all, const double* cst_all, int rep, int nb, int s0f,
                                              double start_time, double end_time) {
    DataView d;
    d.tab = tab_all + (size_t)rep * LR_NTAB * (nb + 1);
    d.nb = nb; d.s0f = s0f;
    d.C = cst_all[rep * LR_NCST + 0]; d.Sx = cst_all[rep * LR_NCST + 1]; d.Sxx = cst_all[rep * LR_NCST + 2];
    d.start_time = start_time; d.end_time = end_time; d.log_span = log(end_time - start_time);
    return d;
}

// One side (birth or death) of a state, distributed over the lanes of a warp.
struct Side {
    double r, lr, t;       // slot `lane`: rate, log(rate), start of the segment (slot 0: start_time)
    double A, B;           // the segment's event count and exposure
    int jb;                // first bin of the segment
    int K;                 // number of rates (uniform)
    // Filled by side_sums() where absolute values are needed (records, Gibbs, the slow path, K2); the loop itself works
    // on per-lane differences and never reads them:
    double sumlr, sumr;    // sum of log-rates / rates over the K slots (uniform)
    double lik;            // sum_k A*lr - r*B (uniform)
};

__device__ __forceinline__ int bin_of_time(const DataView& d, double t) {
    int j = __double2int_rd(t) - d.s0f;
    return j < 0 ? 0 : (j > d.nb ? d.nb : j);
}

// segment statistics of every slot from the prefix tables (two table lookups per lane)
__device__ __forceinline__ void side_stats(Side& s, const DataView& d, int tabA, int tabB, int lane) {
    s.jb = (lane == 0) ? 0 : bin_of_time(d, s.t);
    int nxt = __shfl_down_sync(0xffffffffu, s.jb, 1);
    if (lane >= s.K - 1) nxt = d.nb;
    if (lane < s.K) {
        const double* PA = d.tab + (size_t)tabA * (d.nb + 1);
        const double* PB = d.tab + (size_t)tabB * (d.nb + 1);
        s.A = __ldg(PA + nxt) - __ldg(PA + s.jb);
        s.B = __ldg(PB + nxt) - __ldg(PB + s.jb);
    } else {
        s.A = 0.0; s.B = 0.0;
    }
}

// the three sums every evaluation needs, in one butterfly
__device__ __forceinline__ void side_sums(Side& s, int lane) {
    const bool on = lane < s.K;
    double a = on ? s.lr : 0.0, b = on ? s.r : 0.0, c = on ? (s.A * s.lr - s.r * s.B) : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
        c += __shfl_xor_sync(0xffffffffu, c, o);
    }
    s.sumlr = a; s.sumr = b; s.lik = c;
}

// sum_k lnGammaPdf(rate_k; shape 2, rate g)   (prior_gamma, :201-202; lgamma(2) = 0)
__device__ __forceinline__ double rates_prior(const Side& s, double g, double log_g) {
    return (double)s.K * (2.0 * log_g) + s.sumlr - g * s.sumr;
}
// Poisson_prior(k, lambda) (:198-199)
__device__ __forceinline__ double poisson_prior(int k, double lam, double log_lam, const double* lnfact) {
    return (double)k * log_lam - lam - lnfact[k];
}

// calculate_r_squared (literate_library.py:268-279) in closed form from segment sums
__device__ __forceinline__ void adequacy3(const Side& L, const Side& M, const DataView& d, int lane, double out[3]) {
    const double* XB = d.tab + (size_t)T_XB * (d.nb + 1);
    const double* XD = d.tab + (size_t)T_XD * (d.nb + 1);
    double sy = 0, syy = 0, sxy = 0;
    {
        int nxt = __shfl_down_sync(0xffffffffu, L.jb, 1);
        if (lane >= L.K - 1) nxt = d.nb;
        if (lane < L.K) {
            double n = (double)(nxt - L.jb), x = __ldg(XB + nxt) - __ldg(XB + L.jb);
            sy += L.r * n; syy += L.r * L.r * n; sxy += L.r * x;
        }
    }
    {
        int nxt = __shfl_down_sync(0xffffffffu, M.jb, 1);
        if (lane >= M.K - 1) nxt = d.nb;
        if (lane < M.K) {
            double n = (double)(nxt - M.jb), x = __ldg(XD + nxt) - __ldg(XD + M.jb);
            sy += M.r * n; syy += M.r * M.r * n; sxy += M.r * x;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sy += __shfl_xor_sync(0xffffffffu, sy, o);
        syy += __shfl_xor_sync(0xffffffffu, syy, o);
        sxy += __shfl_xor_sync(0xffffffffu, sxy, o);
    }
    const double n = 2.0 * d.nb;
    const double c = sxy / d.Sxx;
    const double ssres = syy - c * sxy;
    const double var_f = c * c * (d.Sxx - d.Sx * d.Sx / n) / (n - 1.0);
    const double sres = sy - c * d.Sx;
    const double var_r = (ssres - sres * sres / n) / (n - 1.0);
    out[0] = c; out[1] = 1.0 - ssres / syy; out[2] = var_f / (var_f + var_r);
}
