"""Host-side mirror of the three seams of LiteRateForward.py, over the C ABI.

  precompute_events loop (:514-549)  -> Device.bin_stats / bin_stats_device
  calc_likelihood + priors (:137-162, :296-306) -> Dataset + Dataset.evaluate
  runMCMC (:216-373)                 -> Chains

Everything here is plumbing: argument checking, numpy/torch buffers, ctypes calls.  All arithmetic
runs in the CUDA kernels of libliterate_b200.so; there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass

import numpy as np

from . import _native as N
from ._native import ChainConfig, LR_KMAX, LR_REC_DOUBLES, NativeError  # noqa: F401


def _stream_ptr(stream, device=None):
    """cudaStream_t for the C ABI.  NULL means "the handle's own stream" there, so torch's legacy default
    stream (handle 0) is passed as cudaStreamLegacy (0x1)."""
    if stream is None:
        import torch
        stream = torch.cuda.current_stream(device).cuda_stream
    return C.c_void_p(int(stream) if int(stream) != 0 else 1)


def fe_ref_for_jitter(death_jitter: float) -> float:
    """Fractional part (in (0,1]) that te = integer + death_jitter leaves above its bin's lower edge."""
    f = death_jitter - math.ceil(death_jitter) + 1.0
    return f if 0.0 < f <= 1.0 else 1.0


@dataclass
class BinStats:
    """sp_events_bin / ex_events_bin / br_length_bin (LiteRateForward.py:566-568) for n_rep replicates."""
    first_bin: int
    sp: np.ndarray                 # int64 [n_rep, n_bins]
    ex: np.ndarray
    br: np.ndarray                 # float64
    ex_dead: np.ndarray = None     # -model_BDI 3 (:529-549)
    br_dead: np.ndarray = None

    @property
    def n_bins(self):
        return self.sp.shape[-1]

    @property
    def n_rep(self):
        return self.sp.shape[0]


YEAR_PAD = np.iinfo(np.int32).min      # padding of ragged int32 year tables (both columns): contributes nothing


def year_jitter_ok(death_jitter) -> bool:
    """Whether an int32 year table with this death jitter gives the fp64 table's statistics exactly.

    The int32 pass counts every regular death's fraction as exactly `death_jitter`; the fp64 pass sees fl(year + jitter).  The
    two agree for every |year| < 2^31 iff year + jitter is exact there, i.e. 0 <= jitter <= 1 and jitter * 2^22 is an integer
    (0, 0.25, 0.5, 1 are; 0.1 and 1e-14 are not).  The same check guards lr_bin_accumulate_i32."""
    j = float(death_jitter)
    return 0.0 <= j <= 1.0 and math.ldexp(j, 22).is_integer()


def window(ts, te):
    """(first_bin, n_bins) = range(int(min ts), int(max te)) of :519 for host arrays."""
    first = int(np.min(ts))
    return first, int(np.max(te)) - first


class Device:
    """One lr_handle_t: a B200 and its streams/workspace."""

    def __init__(self, index: int = 0):
        self.lib = N.load(build_if_missing=True)     # compiles the CUDA library with nvcc if it is not there; no other path exists
        h = C.c_void_p()
        N.check(self.lib.lr_create(int(index), C.byref(h)), "lr_create")
        self.h = h
        self.index = index

    def close(self):
        if getattr(self, "h", None):
            self.lib.lr_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        N.check(self.lib.lr_sync(self.h), "lr_sync")

    @property
    def sm_count(self):
        sm = C.c_int32()
        N.check(self.lib.lr_info(self.h, C.byref(sm), None, None))
        return sm.value

    @property
    def kernel_launches(self):
        n = C.c_int64()
        N.check(self.lib.lr_info(self.h, None, C.byref(n), None))
        return n.value

    # ------------------------------------------------------------------ L2
    def bin_stats(self, ts, te, first_bin=None, n_bins=None, death_jitter=0.5, only_dead=False, end_time=None,
                  fe_ref=None) -> BinStats:
        """HOST arrays in, host arrays out (lr_bin_stats_host).

        ``ts``/``te`` are float64 arrays of shape [n] or [n_rep, n] (te already jittered, as after
        LiteRateForward.py:471) -- or int32 arrays of YEARS (te before the jitter, which ``death_jitter``
        then supplies): half the bytes over PCIe, the same statistics bit for bit as the float64 table
        (ts, te + death_jitter).  That holds only for jitters that are multiples of 2^-22 in [0, 1]
        (year_jitter_ok); any other jitter raises ValueError for int32 tables -- pass the float64 table.
        With ``only_dead`` the extinct-only statistics of :529-549 are added, for lineages with te < end_time.
        """
        years = np.asarray(ts).dtype == np.int32 and np.asarray(te).dtype == np.int32
        if years:
            # compact tables: integer YEARS as int32 (8 bytes per lineage over PCIe instead of 16); te is the year BEFORE the
            # jitter of :471, which the kernel adds (lr_bin_stats_host_i32).  Pad ragged replicates with YEAR_PAD.
            if not year_jitter_ok(death_jitter):
                raise ValueError("int32 year tables need a death_jitter in [0, 1] that is a multiple of 2^-22 (year + jitter "
                                 "exact); bin the float64 table instead")
            ts = np.ascontiguousarray(ts); te = np.ascontiguousarray(te)
        else:
            ts = np.ascontiguousarray(ts, dtype=np.float64)
            te = np.ascontiguousarray(te, dtype=np.float64)
        if ts.shape != te.shape or ts.ndim not in (1, 2):
            raise ValueError("ts and te must have the same shape, [n] or [n_rep, n]")
        if ts.ndim == 1:
            ts, te = ts[None, :], te[None, :]
        n_rep, n = ts.shape
        if n == 0:
            raise ValueError("no lineages")
        if first_bin is None or n_bins is None:
            if years:
                real = ts != YEAR_PAD
                first_bin = int(ts[real].min())
                n_bins = int(float(te[real].max()) + death_jitter) - first_bin
            else:
                first_bin, n_bins = window(ts, te)
        if n_bins < 1:
            raise ValueError("the time window holds no complete bin (int(max te) <= int(min ts))")
        if fe_ref is None:
            fe_ref = fe_ref_for_jitter(death_jitter)
        if end_time is None:
            end_time = float(te[ts != YEAR_PAD].max()) + death_jitter if years else float(np.max(te))

        def run(dead):
            sp = np.empty((n_rep, n_bins), dtype=np.int64)
            ex = np.empty((n_rep, n_bins), dtype=np.int64)
            br = np.empty((n_rep, n_bins), dtype=np.float64)
            if years:
                N.check(self.lib.lr_bin_stats_host_i32(self.h, N.np_ptr(ts), N.np_ptr(te), n, n, n_rep, int(first_bin), int(n_bins),
                                                       float(death_jitter), 1 if dead else 0, float(end_time),
                                                       N.np_ptr(sp), N.np_ptr(ex), N.np_ptr(br)), "lr_bin_stats_host_i32")
            else:
                N.check(self.lib.lr_bin_stats_host(self.h, N.np_ptr(ts), N.np_ptr(te), n, n, n_rep, int(first_bin), int(n_bins),
                                                   float(fe_ref), 1 if dead else 0, float(end_time),
                                                   N.np_ptr(sp), N.np_ptr(ex), N.np_ptr(br)), "lr_bin_stats_host")
            return sp, ex, br

        sp, ex, br = run(False)
        out = BinStats(int(first_bin), sp, ex, br)
        if only_dead:
            _, out.ex_dead, out.br_dead = run(True)
        return out

    def bin_stats_device(self, ts, te, first_bin, n_bins, fe_ref=0.5, dead_only=False, end_time=0.0, stream=None, out=None):
        """torch CUDA tensors in, torch CUDA tensors out (lr_bin_stats); asynchronous on `stream`.

        ts/te: float64 CUDA tensors [n_rep, n] (row stride may exceed n).  Returns (sp, ex, br).
        """
        import torch
        assert ts.is_cuda and te.is_cuda and ts.dtype == torch.float64 and te.dtype == torch.float64
        if ts.dim() == 1:
            ts, te = ts[None, :], te[None, :]
        assert ts.stride(-1) == 1 and te.stride(-1) == 1 and ts.shape == te.shape
        n_rep, n = ts.shape
        ld = ts.stride(0) if n_rep > 1 else n
        assert n_rep == 1 or te.stride(0) == ld
        if out is None:
            sp = torch.empty((n_rep, n_bins), dtype=torch.int64, device=ts.device)
            ex = torch.empty_like(sp)
            br = torch.empty((n_rep, n_bins), dtype=torch.float64, device=ts.device)
        else:
            sp, ex, br = out
        st = _stream_ptr(stream, ts.device)
        N.check(self.lib.lr_bin_stats(self.h, C.c_void_p(ts.data_ptr()), C.c_void_p(te.data_ptr()), n, ld, n_rep,
                                      int(first_bin), int(n_bins), float(fe_ref), 1 if dead_only else 0, float(end_time),
                                      C.c_void_p(sp.data_ptr()), C.c_void_p(ex.data_ptr()), C.c_void_p(br.data_ptr()), st),
                "lr_bin_stats")
        return sp, ex, br

    def bin_accumulate_device(self, ts, te, first_bin, n_bins, acc, fe_ref=0.5, dead_only=False, end_time=0.0, stream=None,
                              death_jitter=None):
        """Raw integer accumulators only (lr_bin_accumulate) -- the lineage-sharded multi-GPU path all-reduces
        `acc` (int64 [n_rep, 8, lr_acc_stride]) before bin_finalize_device."""
        import torch
        if ts.dim() == 1:
            ts, te = ts[None, :], te[None, :]
        n_rep, n = ts.shape
        ld = ts.stride(0) if n_rep > 1 else max(n, 1)
        st = _stream_ptr(stream, ts.device)
        if ts.dtype == torch.int32:
            # int32 YEARS: `death_jitter` takes the place of fe_ref (te = year + jitter); finalize with fe_ref_for_jitter(death_jitter)
            jit = fe_ref if death_jitter is None else death_jitter
            if not year_jitter_ok(jit):
                raise ValueError("int32 year tables need a death_jitter in [0, 1] that is a multiple of 2^-22 (year + jitter exact)")
            N.check(self.lib.lr_bin_accumulate_i32(self.h, C.c_void_p(ts.data_ptr()), C.c_void_p(te.data_ptr()), n, ld, n_rep,
                                                   int(first_bin), int(n_bins), float(jit), 1 if dead_only else 0, float(end_time),
                                                   C.c_void_p(acc.data_ptr()), st), "lr_bin_accumulate_i32")
            return acc
        N.check(self.lib.lr_bin_accumulate(self.h, C.c_void_p(ts.data_ptr()), C.c_void_p(te.data_ptr()), n, ld, n_rep,
                                           int(first_bin), int(n_bins), float(fe_ref), 1 if dead_only else 0, float(end_time),
                                           C.c_void_p(acc.data_ptr()), st), "lr_bin_accumulate")
        return acc

    def bin_table_hint(self):
        """What the last finished K1 pass saw (lr_bin_table_hint): 1 = fractional times, 0 = integer years.  The next pass
        through this handle picks its build from it."""
        out = C.c_int32(0)
        N.check(self.lib.lr_bin_table_hint(self.h, C.byref(out)), "lr_bin_table_hint")
        return int(out.value)

    def bin_last_build(self):
        """Which build of K1 the last bin_accumulate_device / bin_stats_device call launched (lr_bin_last_build)."""
        out = C.c_int32(0)
        N.check(self.lib.lr_bin_last_build(self.h, C.byref(out)), "lr_bin_last_build")
        return "k1_bin_lanes_kernel" if out.value == 1 else "k1_bin_kernel"

    def loglik_direct_device(self, ts, te, first_bin, n_bins, lam, mu, stream=None):
        """Validation path (lr_loglik_direct): Keiding log-likelihood of states given as per-bin rates, straight from the
        lineages.  ts/te: float64 CUDA tensors [n]; lam/mu: float64 CUDA tensors [n_states, n_bins].  Returns [n_states]."""
        import torch
        assert ts.is_cuda and lam.is_cuda and lam.shape == mu.shape and lam.shape[1] == n_bins and lam.is_contiguous() and mu.is_contiguous()
        out = torch.empty(lam.shape[0], dtype=torch.float64, device=lam.device)
        N.check(self.lib.lr_loglik_direct(self.h, C.c_void_p(ts.data_ptr()), C.c_void_p(te.data_ptr()), ts.numel(), int(first_bin), int(n_bins),
                                          C.c_void_p(lam.data_ptr()), C.c_void_p(mu.data_ptr()), lam.shape[0], C.c_void_p(out.data_ptr()),
                                          _stream_ptr(stream, lam.device)), "lr_loglik_direct")
        return out

    def summarize_records_device(self, records, first_edge, n_bins, stream=None):
        """Posterior accumulators of device-resident records (lr_summarize_records): `records` is a contiguous float64 CUDA
        tensor [..., 144]; returns (sum_rate [2, n_bins] float64, shift_count [2, n_bins] int64, k_count [2, 32] int64, n_records)."""
        import torch
        assert records.is_cuda and records.dtype == torch.float64 and records.is_contiguous() and records.shape[-1] == LR_REC_DOUBLES
        n = records.numel() // LR_REC_DOUBLES
        sr = torch.empty((2, n_bins), dtype=torch.float64, device=records.device)
        sc = torch.empty((2, n_bins), dtype=torch.int64, device=records.device)
        kc = torch.empty((2, 32), dtype=torch.int64, device=records.device)
        N.check(self.lib.lr_summarize_records(self.h, C.c_void_p(records.data_ptr()), n, float(first_edge), int(n_bins),
                                              C.c_void_p(sr.data_ptr()), C.c_void_p(sc.data_ptr()), C.c_void_p(kc.data_ptr()),
                                              _stream_ptr(stream, records.device)), "lr_summarize_records")
        return sr, sc, kc, n

    def marginal_rates_device(self, records, first_edge, n_bins, bin_lo=0, bin_cnt=None, stream=None):
        """Per-sample marginal rates of device-resident records (lr_marginal_rates): `records` a contiguous float64 CUDA tensor
        [..., 144]; returns (birth, death), float64 CUDA tensors [n_records, bin_cnt] for the bins [bin_lo, bin_lo + bin_cnt)."""
        import torch
        assert records.is_cuda and records.dtype == torch.float64 and records.is_contiguous() and records.shape[-1] == LR_REC_DOUBLES
        n = records.numel() // LR_REC_DOUBLES
        if bin_cnt is None:
            bin_cnt = n_bins - bin_lo
        b = torch.empty((n, bin_cnt), dtype=torch.float64, device=records.device)
        d = torch.empty((n, bin_cnt), dtype=torch.float64, device=records.device)
        N.check(self.lib.lr_marginal_rates(self.h, C.c_void_p(records.data_ptr()), n, float(first_edge), int(n_bins), int(bin_lo), int(bin_cnt),
                                           C.c_void_p(b.data_ptr()), C.c_void_p(d.data_ptr()), _stream_ptr(stream, records.device)),
                "lr_marginal_rates")
        return b, d

    def new_accumulators(self, n_rep, n_bins, device):
        import torch
        return torch.zeros((n_rep, N.LR_ACC_ROWS, int(self.lib.lr_acc_stride(int(n_bins)))), dtype=torch.int64, device=device)

    def imputation_envelope_device(self, sp, ex, br, stream=None):
        """Mean / min / max over the replicates of ex/br, sp/br and br (lr_imputation_envelope; utilities/imputation_averager.py:23-61).
        sp, ex: int64, br: float64 CUDA tensors [n_rep, n_bins] (the outputs of bin_stats_device).  Returns float64 [9, n_bins]."""
        import torch
        n_rep, nb = sp.shape
        out = torch.empty((9, nb), dtype=torch.float64, device=sp.device)
        N.check(self.lib.lr_imputation_envelope(self.h, C.c_void_p(sp.data_ptr()), C.c_void_p(ex.data_ptr()), C.c_void_p(br.data_ptr()),
                                                int(n_rep), int(nb), C.c_void_p(out.data_ptr()), _stream_ptr(stream, sp.device)),
                "lr_imputation_envelope")
        return out

    def bin_finalize_device(self, acc, n_bins, fe_ref=0.5, stream=None):
        import torch
        n_rep = acc.shape[0]
        sp = torch.empty((n_rep, n_bins), dtype=torch.int64, device=acc.device)
        ex = torch.empty_like(sp)
        br = torch.empty((n_rep, n_bins), dtype=torch.float64, device=acc.device)
        st = _stream_ptr(stream, acc.device)
        N.check(self.lib.lr_bin_finalize(self.h, C.c_void_p(acc.data_ptr()), n_rep, int(n_bins), float(fe_ref),
                                         C.c_void_p(sp.data_ptr()), C.c_void_p(ex.data_ptr()), C.c_void_p(br.data_ptr()), st),
                "lr_bin_finalize")
        return sp, ex, br


class Dataset:
    """Binned statistics of n_rep replicates resident on the device, plus the prefix tables of the likelihood."""

    def __init__(self, dev: Device, stats: BinStats, model_BDI: int, start_time: float, end_time: float):
        self.dev, self.model_BDI = dev, int(model_BDI)
        self.start_time, self.end_time = float(start_time), float(end_time)
        self.n_rep, self.n_bins = stats.n_rep, stats.n_bins
        sp = np.ascontiguousarray(stats.sp, dtype=np.int64).reshape(self.n_rep, self.n_bins)
        ex = np.ascontiguousarray(stats.ex, dtype=np.int64).reshape(self.n_rep, self.n_bins)
        br = np.ascontiguousarray(stats.br, dtype=np.float64).reshape(self.n_rep, self.n_bins)
        exd = brd = None
        if self.model_BDI == 3:
            if stats.ex_dead is None or stats.br_dead is None:
                raise ValueError("-model_BDI 3 needs the extinct-only statistics (bin_stats(only_dead=True))")
            exd = np.ascontiguousarray(stats.ex_dead, dtype=np.int64).reshape(self.n_rep, self.n_bins)
            brd = np.ascontiguousarray(stats.br_dead, dtype=np.float64).reshape(self.n_rep, self.n_bins)
        ds = C.c_void_p()
        N.check(dev.lib.lr_dataset_create_host(dev.h, self.n_rep, self.n_bins, self.model_BDI, self.start_time, self.end_time,
                                               N.np_ptr(sp), N.np_ptr(ex), N.np_ptr(br), N.np_ptr(exd), N.np_ptr(brd),
                                               C.byref(ds)), "lr_dataset_create_host")
        self.ds = ds

    @classmethod
    def from_device(cls, dev: Device, sp, ex, br, model_BDI, start_time, end_time, ex_dead=None, br_dead=None, stream=None):
        """Same from torch CUDA tensors already on the device (no host round trip)."""
        import torch
        self = cls.__new__(cls)
        self.dev, self.model_BDI = dev, int(model_BDI)
        self.start_time, self.end_time = float(start_time), float(end_time)
        self.n_rep, self.n_bins = sp.shape
        st = _stream_ptr(stream, sp.device)
        ds = C.c_void_p()
        N.check(dev.lib.lr_dataset_create(dev.h, self.n_rep, self.n_bins, self.model_BDI, self.start_time, self.end_time,
                                          C.c_void_p(sp.data_ptr()), C.c_void_p(ex.data_ptr()), C.c_void_p(br.data_ptr()),
                                          C.c_void_p(ex_dead.data_ptr()) if ex_dead is not None else None,
                                          C.c_void_p(br_dead.data_ptr()) if br_dead is not None else None, st, C.byref(ds)),
                "lr_dataset_create")
        self.ds = ds
        return self

    @classmethod
    def from_tables(cls, dev: Device, A_birth, B_birth, A_death, B_death, x_birth, x_death, start_time, end_time, model_tag=1, C_const=None):
        """General piecewise-constant Poisson likelihood (lr_dataset_create_general_host): per bin and side an event weight A and
        an exposure B, likelihood = C + sum A_b log(lambda) - B_b lambda + sum A_d log(mu) - B_d mu.  Host arrays [n_bins] or
        [n_rep, n_bins]; x_* are the vectors the adequacy regression uses.  The `-proportion 1` variant is built this way."""
        self = cls.__new__(cls)
        arrs = [np.atleast_2d(np.ascontiguousarray(a, dtype=np.float64)) for a in (A_birth, B_birth, A_death, B_death, x_birth, x_death)]
        self.dev, self.model_BDI = dev, int(model_tag)
        self.start_time, self.end_time = float(start_time), float(end_time)
        self.n_rep, self.n_bins = arrs[0].shape
        if any(a.shape != arrs[0].shape for a in arrs):
            raise ValueError("the six tables must have the same shape")
        cc = None if C_const is None else np.ascontiguousarray(np.broadcast_to(np.asarray(C_const, np.float64), (self.n_rep,)))
        ds = C.c_void_p()
        N.check(dev.lib.lr_dataset_create_general_host(dev.h, self.n_rep, self.n_bins, self.model_BDI, self.start_time, self.end_time,
                                                       *[N.np_ptr(np.ascontiguousarray(a)) for a in arrs], N.np_ptr(cc), C.byref(ds)),
                "lr_dataset_create_general_host")
        self.ds = ds
        return self

    def close(self):
        if getattr(self, "ds", None):
            self.dev.lib.lr_dataset_destroy(self.ds)
            self.ds = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def evaluate(self, states, gamma_rate=None, poi_lambda=None, rep=None):
        """Likelihood / prior / adequacy of explicit states (lr_state_eval_host).

        ``states``: list of (L, M, timesL, timesM) with times = [start, shifts..., end] as in the reference.
        Returns dict of arrays: lik, prior_rates (gamma + time prior), prior_poi, adequacy[n,3].
        """
        n = len(states)
        K_l = np.zeros(n, np.int32); K_m = np.zeros(n, np.int32)
        L = np.zeros((n, LR_KMAX)); M = np.zeros((n, LR_KMAX)); tL = np.zeros((n, LR_KMAX)); tM = np.zeros((n, LR_KMAX))
        for i, (l, m, tl, tm) in enumerate(states):
            l, m, tl, tm = (np.asarray(x, dtype=np.float64) for x in (l, m, tl, tm))
            if len(tl) != len(l) + 1 or len(tm) != len(m) + 1:
                raise ValueError("times must hold one more entry than rates")
            K_l[i], K_m[i] = len(l), len(m)
            L[i, :len(l)], M[i, :len(m)] = l, m
            tL[i, :len(l)], tM[i, :len(m)] = tl[:-1], tm[:-1]
        g = None if gamma_rate is None else np.ascontiguousarray(np.broadcast_to(np.asarray(gamma_rate, np.float64), (n, 2)))
        p = None if poi_lambda is None else np.ascontiguousarray(np.broadcast_to(np.asarray(poi_lambda, np.float64), (n,)))
        r = None if rep is None else np.ascontiguousarray(np.broadcast_to(np.asarray(rep, np.int32), (n,)))
        lik = np.empty(n); pr = np.empty(n); pp = np.empty(n); ad = np.empty((n, 3))
        N.check(self.dev.lib.lr_state_eval_host(self.ds, n, N.np_ptr(r), N.np_ptr(K_l), N.np_ptr(K_m), N.np_ptr(L), N.np_ptr(M),
                                                N.np_ptr(tL), N.np_ptr(tM), N.np_ptr(g), N.np_ptr(p),
                                                N.np_ptr(lik), N.np_ptr(pr), N.np_ptr(pp), N.np_ptr(ad)), "lr_state_eval_host")
        return {"lik": lik, "prior_rates": pr, "prior_poi": pp, "adequacy": ad}


def _pack_states(states):
    n = len(states)
    K_l = np.zeros(n, np.int32); K_m = np.zeros(n, np.int32)
    L = np.zeros((n, LR_KMAX)); M = np.zeros((n, LR_KMAX)); tL = np.zeros((n, LR_KMAX)); tM = np.zeros((n, LR_KMAX))
    for i, (l, m, tl, tm) in enumerate(states):
        l, m, tl, tm = (np.asarray(x, dtype=np.float64) for x in (l, m, tl, tm))
        if len(tl) != len(l) + 1 or len(tm) != len(m) + 1:
            raise ValueError("times must hold one more entry than rates")
        K_l[i], K_m[i] = len(l), len(m)
        L[i, :len(l)], M[i, :len(m)] = l, m
        tL[i, :len(l)], tM[i, :len(m)] = tl[:-1], tm[:-1]
    return K_l, K_m, L, M, tL, tM


def evaluate_proposals(ds: "Dataset", states, side, kind, idx, u_t, u_beta, gamma_rate=None, poi_lambda=None, beta=None, poiA=None, rep=None,
                       mult_on=None, mult_u=None):
    """One reversible-jump proposal per state with explicit draws (lr_proposal_eval_host; parity entry point).
    kind: 0 rate multiplier with mask mult_on / uniforms mult_u [n, LR_KMAX]; 2 add-shift inside segment idx; 3 remove interior shift idx.  Returns dict: ok, K_new, rates, times (lists of
    arrays: the proposed side in the reference's layout [start, shifts..., end]), hasting, x."""
    n = len(states)
    K_l, K_m, L, M, tL, tM = _pack_states(states)
    b = lambda a, dt, shape: None if a is None else np.ascontiguousarray(np.broadcast_to(np.asarray(a, dt), shape))
    g, p, be = b(gamma_rate, np.float64, (n, 2)), b(poi_lambda, np.float64, (n,)), b(beta, np.float64, (n,))
    pa = b(0.0 if poiA is None else poiA, np.float64, (n,))
    r = b(rep, np.int32, (n,))
    sd, kd, ix = b(side, np.int32, (n,)), b(kind, np.int32, (n,)), b(idx, np.int32, (n,))
    ut, ub = b(u_t, np.float64, (n,)), b(u_beta, np.float64, (n,))
    mo, mu = b(mult_on, np.int32, (n, LR_KMAX)), b(mult_u, np.float64, (n, LR_KMAX))
    ok = np.empty(n, np.int32); kn = np.empty(n, np.int32)
    rn = np.empty((n, LR_KMAX)); tn = np.empty((n, LR_KMAX)); hs = np.empty(n); x = np.empty(n)
    N.check(ds.dev.lib.lr_proposal_eval_host(ds.ds, n, N.np_ptr(r), N.np_ptr(K_l), N.np_ptr(K_m), N.np_ptr(L), N.np_ptr(M), N.np_ptr(tL),
                                             N.np_ptr(tM), N.np_ptr(g), N.np_ptr(p), N.np_ptr(be), N.np_ptr(pa), N.np_ptr(sd), N.np_ptr(kd),
                                             N.np_ptr(ix), N.np_ptr(ut), N.np_ptr(ub), N.np_ptr(mo), N.np_ptr(mu), N.np_ptr(ok), N.np_ptr(kn), N.np_ptr(rn), N.np_ptr(tn),
                                             N.np_ptr(hs), N.np_ptr(x)), "lr_proposal_eval_host")
    rates = [rn[i, :kn[i]].copy() for i in range(n)]
    times = [np.concatenate([tn[i, :kn[i]], [ds.end_time]]) for i in range(n)]
    return {"ok": ok.astype(bool), "K_new": kn, "rates": rates, "times": times, "hasting": hs, "x": x}


# field offsets of a sample record (include/literate_b200.h)
REC_IT, REC_LIK, REC_PRIOR, REC_LAVG, REC_MAVG, REC_KL, REC_KM, REC_GL, REC_GM, REC_POI = range(10)
REC_ADQ, REC_POI_INIT, REC_BETA, REC_POIA = 10, 13, 14, 15
REC_L, REC_TL, REC_M, REC_TM = 16, 48, 80, 112
COUNTER_NAMES = ["iterations", "accepted", "lik_evals", "rate_updates", "move_shifts", "rj_proposals", "gibbs", "capacity_rejects",
                 "swaps_proposed", "swaps_accepted"]


class Chains:
    """A population of independent RJMCMC chains on one device (runMCMC, LiteRateForward.py:216-373)."""

    def __init__(self, ds: Dataset, n_chains: int, seed: int, cfg: ChainConfig = None, chain_id0: int = 0, rep_of_chain=None):
        self.ds, self.dev, self.n_chains = ds, ds.dev, int(n_chains)
        if cfg is None:
            cfg = default_config(ds.model_BDI)
        self.cfg = cfg
        rep = None
        if rep_of_chain is not None:
            rep = np.ascontiguousarray(rep_of_chain, dtype=np.int32)
            if rep.shape != (self.n_chains,):
                raise ValueError("rep_of_chain must have one entry per chain")
        c = C.c_void_p()
        N.check(self.dev.lib.lr_chains_create(self.dev.h, ds.ds, self.n_chains, C.byref(cfg), C.c_uint64(int(seed) & (2**64 - 1)),
                                              int(chain_id0), N.np_ptr(rep), C.byref(c)), "lr_chains_create")
        self.c = c

    def close(self):
        if getattr(self, "c", None):
            self.dev.lib.lr_chains_destroy(self.c)
            self.c = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def records_per_run(self, n_iter, sample_every):
        return int(self.dev.lib.lr_chains_records_per_run(self.c, int(n_iter), int(sample_every)))

    def run(self, n_iter: int, sample_every: int = 0, out=None):
        """n_iter iterations of every chain; returns records [n_samples, n_chains, 144] (host) or None."""
        if sample_every and sample_every > 0:
            nrec = self.records_per_run(n_iter, sample_every)
            if out is None:
                out = np.empty((nrec, self.n_chains, LR_REC_DOUBLES), dtype=np.float64)
            assert out.shape == (nrec, self.n_chains, LR_REC_DOUBLES) and out.flags["C_CONTIGUOUS"]
            N.check(self.dev.lib.lr_chains_run_host(self.c, int(n_iter), int(sample_every), N.np_ptr(out)), "lr_chains_run_host")
            return out
        N.check(self.dev.lib.lr_chains_run_host(self.c, int(n_iter), 0, None), "lr_chains_run_host")
        return None

    def run_device(self, n_iter: int, sample_every: int, records, stream=None):
        """Asynchronous variant: `records` is a float64 CUDA tensor [n_samples, n_chains, 144] (or None).
        stream: a cudaStream_t, None = torch's current stream, "handle" = the Device's own compute stream."""
        import torch
        st = C.c_void_p(None) if isinstance(stream, str) and stream == "handle" else _stream_ptr(stream)
        ptr = C.c_void_p(records.data_ptr()) if records is not None else None
        N.check(self.dev.lib.lr_chains_run(self.c, int(n_iter), int(sample_every) if records is not None else 0, ptr, st),
                "lr_chains_run")

    def state(self):
        out = np.empty((self.n_chains, LR_REC_DOUBLES), dtype=np.float64)
        N.check(self.dev.lib.lr_chains_get_state_host(self.c, N.np_ptr(out)), "lr_chains_get_state_host")
        return out

    def set_state(self, records):
        records = np.ascontiguousarray(records, dtype=np.float64)
        assert records.shape == (self.n_chains, LR_REC_DOUBLES)
        N.check(self.dev.lib.lr_chains_set_state_host(self.c, N.np_ptr(records)), "lr_chains_set_state_host")

    def counters(self):
        out = np.empty((self.n_chains, N.LR_NCOUNTERS), dtype=np.int64)
        N.check(self.dev.lib.lr_chains_counters_host(self.c, N.np_ptr(out)), "lr_chains_counters_host")
        return out

    def team_stats(self):
        """Diagnostics of the speculative team build (loop_variant 4): int64 [n_chains, 6] = state versions committed,
        evaluations dropped by rollbacks, polls waiting for the frontier, polls at the lead limit, iterations done by
        teams, hand-overs to the continuation pass."""
        out = np.empty((self.n_chains, 6), dtype=np.int64)
        N.check(self.dev.lib.lr_chains_team_stats_host(self.c, N.np_ptr(out)), "lr_chains_team_stats_host")
        return out

    # ---- tempered ensembles (new; the reference has no MC3)
    def set_beta(self, beta):
        beta = np.ascontiguousarray(np.broadcast_to(np.asarray(beta, np.float64), (self.n_chains,)))
        N.check(self.dev.lib.lr_chains_set_beta_host(self.c, N.np_ptr(beta)), "lr_chains_set_beta_host")

    def swap_step(self, ladder: int, round_: int):
        """One swap round for ladders of `ladder` consecutive chains that all live on this device."""
        N.check(self.dev.lib.lr_chains_swap_step(self.c, int(ladder), C.c_uint64(int(round_))), "lr_chains_swap_step")

    def run_tempered(self, n_iter: int, sample_every: int, ladder: int, swap_every: int, round0: int = 0, swap=None):
        """n_iter iterations with a swap round every `swap_every` iterations (ladders on this device unless `swap`
        -- a callable round -> None, e.g. parallel.tempered_swap bound to this shard -- is given).
        Returns (records of ALL chains [n_samples, n_chains, 144], number of swap rounds done); filter on
        records[..., REC_BETA] == 1 for the cold chains (cold_records())."""
        out, done, rnd = [], 0, int(round0)
        while done < n_iter:
            n = min(int(swap_every), n_iter - done)
            r = self.run(n, sample_every)
            if r is not None and len(r):
                out.append(r)
            done += n
            if done < n_iter or n == swap_every:
                if swap is None:
                    self.swap_step(ladder, rnd)
                else:
                    swap(rnd)
                rnd += 1
        recs = np.concatenate(out) if out else np.empty((0, self.n_chains, LR_REC_DOUBLES))
        return recs, rnd - int(round0)

    def swap_info_device(self, info, stream=None):
        """(likelihood, beta) of every chain into the float64 CUDA tensor info[n_chains, 2]."""
        N.check(self.dev.lib.lr_chains_swap_info(self.c, C.c_void_p(info.data_ptr()), _stream_ptr(stream, info.device)), "lr_chains_swap_info")
        return info

    def swap_apply_device(self, info_all, first: int, ladder: int, round_: int, stream=None):
        """Apply a swap round given the gathered table info_all[n_all, 2] of the whole ensemble (see parallel.tempered_swap)."""
        N.check(self.dev.lib.lr_chains_swap_apply(self.c, C.c_void_p(info_all.data_ptr()), int(info_all.shape[0]), int(first), int(ladder),
                                                  C.c_uint64(int(round_)), _stream_ptr(stream, info_all.device)), "lr_chains_swap_apply")


def default_config(model_BDI=0, const_rates=0, const_death_rate=0, use_rate_HP=1, Poisson_prior=0.0, update_fraction=0.75,
                   real_move_shift=0, beta=1.0, loop_variant=0) -> ChainConfig:
    """Defaults of LiteRateForward.py:386-399."""
    return ChainConfig(int(model_BDI), int(const_rates), int(const_death_rate), int(use_rate_HP), float(Poisson_prior),
                       float(update_fraction), int(real_move_shift), int(loop_variant), float(beta))


def cold_records(records, ladder: int):
    """[n_samples, n_chains, 144] of a tempered run -> [n_samples, n_chains // ladder, 144]: per ladder and sample, the
    record of the member that held beta = 1 when the sample was written."""
    ns, nc, w = records.shape
    r = records.reshape(ns, nc // ladder, ladder, w)
    idx = np.argmax(r[..., REC_BETA], axis=2)
    out = np.take_along_axis(r, idx[:, :, None, None], axis=2)[:, :, 0, :]
    if not np.all(out[..., REC_BETA] == 1.0):
        raise ValueError("a ladder has no chain at beta = 1")
    return out


def record_to_state(rec, end_time):
    """One sample record -> (L, M, timesL, timesM) in the reference's layout."""
    kl, km = int(rec[REC_KL]), int(rec[REC_KM])
    L = rec[REC_L:REC_L + kl].copy()
    M = rec[REC_M:REC_M + km].copy()
    tL = np.concatenate([rec[REC_TL:REC_TL + kl], [end_time]])
    tM = np.concatenate([rec[REC_TM:REC_TM + km], [end_time]])
    return L, M, tL, tM


def run_rjmcmc(dev: Device, ts, te, n_chains, n_iter, sample_every, seed=1, cfg: ChainConfig = None, model_BDI=0,
               first_bin=None, n_bins=None, death_jitter=0.5, start_time=None, end_time=None, rep_of_chain=None,
               chain_id0=0, out=None):
    """Host tables in, sample records out: the whole hot path in one call (what forward.py does per input file).

    ts/te: float64 host arrays [n] or [n_rep, n] (te already jittered).  Binning (K1), tables (K2) and the chains (K3)
    run on the device; the copies of the lineages to the device are pipelined against K1.  Returns
    (records [n_samples, n_chains, 144], BinStats).
    """
    ts = np.asarray(ts); te = np.asarray(te)
    if first_bin is None or n_bins is None:
        first_bin, n_bins = window(ts, te)
    if start_time is None:
        start_time = float(np.min(ts))
    if end_time is None:
        end_time = float(np.max(te))
    if cfg is None:
        cfg = default_config(model_BDI)
    stats = dev.bin_stats(ts, te, first_bin=first_bin, n_bins=n_bins, death_jitter=death_jitter,
                          only_dead=(cfg.model_BDI == 3), end_time=end_time)
    ds = Dataset(dev, stats, cfg.model_BDI, start_time, end_time)
    try:
        ch = Chains(ds, n_chains, seed, cfg, chain_id0=chain_id0, rep_of_chain=rep_of_chain)
        try:
            rec = ch.run(n_iter, sample_every, out=out)
        finally:
            ch.close()
    finally:
        ds.close()
    return rec, stats


def bind_host_to_gpu(index: int):
    """Pin this process to the CPUs NVML reports as local to GPU `index` (same NUMA node / PCIe root), so that pinned host
    buffers allocated afterwards are first-touched on that node and the copy engine does not cross the inter-socket link.
    Returns the CPU list, or None when NVML has nothing better than "all CPUs" to offer.  Plumbing; call it before allocating."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(index))
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if not cpus or len(cpus) == len(allowed):
            return None
        os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:                    # noqa: BLE001 -- no NVML / not permitted: leave the affinity alone
        return None


class Pipeline:
    """The hot path over a stream of batches, double-buffered: while the chains of batch k run (K3: no memory traffic),
    the tables of batch k+1 are copied to the device and binned (PCIe + K1: hardly any SM time).  Two handles on the same
    GPU keep the two halves on independent streams; allocation is stream-ordered, so nothing synchronises the device.

        pipe = Pipeline(0)
        for ts, te in batches:
            done = pipe.push(ts, te, n_chains, n_iter, sample_every, ...)   # -> (records, BinStats) of the PREVIOUS batch, or None
        last = pipe.flush()
    """

    def __init__(self, device_index: int = 0):
        self.dev_bin = Device(device_index)
        self.dev_run = Device(device_index)
        self.index = device_index
        self._inflight = None

    def _collect(self, out):
        import torch
        t, self._inflight = self._inflight, None
        if t is None:
            return None
        self.dev_run.sync()                          # the chains of the previous batch (normally long finished)
        host = None
        if t["rec"] is not None:
            if out is not None:                      # numpy array or (pinned) torch tensor
                (out if isinstance(out, torch.Tensor) else torch.from_numpy(out)).copy_(t["rec"])
                host = out
            else:
                host = t["rec"].cpu().numpy()
        t["ch"].close(); t["ds"].close()
        return host, t["stats"]

    def push(self, ts, te, n_chains, n_iter, sample_every, seed=1, cfg: ChainConfig = None, model_BDI=0, first_bin=None,
             n_bins=None, death_jitter=0.5, start_time=None, end_time=None, rep_of_chain=None, chain_id0=0, out=None):
        """Bin this batch (overlapping the chains of the previous one), hand back the previous batch's result (copied into
        `out` if given), then launch this batch's chains asynchronously."""
        import torch
        ts = np.asarray(ts); te = np.asarray(te)
        years = ts.dtype == np.int32 and te.dtype == np.int32          # compact year tables: te is the year before the jitter
        if first_bin is None or n_bins is None:
            if years:
                first_bin = int(ts[ts != YEAR_PAD].min()); n_bins = int(float(te[ts != YEAR_PAD].max()) + death_jitter) - first_bin
            else:
                first_bin, n_bins = window(ts, te)
        if start_time is None:
            start_time = float(ts[ts != YEAR_PAD].min()) if years else float(np.min(ts))
        if end_time is None:
            end_time = float(te[ts != YEAR_PAD].max()) + death_jitter if years else float(np.max(te))
        if cfg is None:
            cfg = default_config(model_BDI)
        stats = self.dev_bin.bin_stats(ts, te, first_bin=first_bin, n_bins=n_bins, death_jitter=death_jitter,
                                       only_dead=(cfg.model_BDI == 3), end_time=end_time)          # H2D + K1, synchronous
        prev = self._collect(out)
        ds = Dataset(self.dev_run, stats, cfg.model_BDI, start_time, end_time)
        ch = Chains(ds, n_chains, seed, cfg, chain_id0=chain_id0, rep_of_chain=rep_of_chain)
        n_rec = ch.records_per_run(n_iter, sample_every) if sample_every else 0
        rec = torch.empty((n_rec, n_chains, LR_REC_DOUBLES), dtype=torch.float64, device=torch.device("cuda", self.index)) if n_rec else None
        ch.run_device(n_iter, sample_every, rec, stream="handle")                                   # asynchronous
        self._inflight = {"ds": ds, "ch": ch, "rec": rec, "stats": stats}
        return prev

    def flush(self, out=None):
        """Result of the last pushed batch."""
        return self._collect(out)

    def close(self):
        self._collect(None)
        self.dev_bin.close(); self.dev_run.close()
