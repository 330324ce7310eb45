// K3, SPECULATIVE TEAM build of the chain loop (loop_variant 4).  Included by k3_chains.cu inside its anonymous namespace.
//
// Why: at a few hundred chains one warp per chain leaves the SMs four-fifths idle (ncu, round 1: 0.19 of issue peak): an
// iteration is ~900 cycles of DEPENDENT fp64 work.  But most iterations do not change the chain's state -- the
// reference's move-shift proposes the current state (LiteRateForward.py:184-185), a rate update that touches no rate or
// a remove-shift on a single-rate side leaves it as it is, and on large tables nearly every real proposal is rejected
// (:313) -- and everything an iteration draws is independent of the state (make_draws).  So a TEAM of W warps works on
// one chain: warp w evaluates iterations w, w + W, w + 2W, ... against its own register copy of the state, without
// waiting for the iterations before it.  An evaluation that leaves the state unchanged is simply published
// ("iterations below n of mine are done under state version v").  A warp whose iteration would CHANGE the state
// (accepted proposal, Gibbs step :281-287, the periodic log-rate resync) or must observe it (sample record :321) first
// waits until every earlier iteration is published under the same version -- it is then the chain's frontier, its
// evaluation is the one the sequential loop would have made -- applies the change, writes the new state to shared memory
// and bumps the version.  The others notice the new version at their next iteration, reload, and resume at the iteration
// after the commit; whatever they had evaluated beyond it is dropped.  The chain is the SAME chain, bit for bit, as in
// the other builds (tests/test_gpu_chains.py::test_loop_builds_give_identical_chains): same draws, same arithmetic on the
// same state, only evaluated early.
//
// Protocol (shared memory of the CTA = one chain):
//   verword          version (24 bits, wraps) | what the commit changed (8 bits) | offset of the iteration after the commit (32 bits)
//   prog[w]          (version << 32) | offset of warp w's next unevaluated iteration
//   buf[version & 1] the state of that version (written by the committing warp before the release store of verword)
// A commit at iteration j under version v needs every other warp's prog to carry version v and an offset > j; so every warp has
// acknowledged v (nobody still reads the buffer of v - 1, which v + 1 overwrites), versions never skip a warp, and there is
// one frontier at a time.  A warp may run at most `lead` own iterations ahead of the slowest one (bounds the dropped
// work and keeps the per-warp history of counter increments -- 8 iterations deep -- exact under rollback).
// Rollbacks are selective: every evaluation records WHAT it read (values / number of rates of either side, the stored
// Poisson prior), every commit says what it changed, and a warp only goes back to its first evaluation beyond the commit
// that read something the commit changed -- a death-rate update survives an accepted add-shift on the birth side, the
// reference's no-op move survives everything that keeps its side's number of rates.

template <int W>
struct TeamShared {
    unsigned long long verword;
    unsigned long long prog[W];
    unsigned n_eff;            // iterations of this launch the team does (lowered when it hands the chain over or its time slice ends)
    unsigned stopped;          // n_eff was lowered because the time slice ended (not a hand-over)
    int chain;                 // time-sliced teams: the chain and the end of the slice (global timer, 0: none), kept here
    unsigned long long t_stop; // and not in registers, which the loop needs all of
    unsigned win_i, win_c;     // observation window: first offset, state changes since then (only the frontier touches them)
    unsigned cnt[W][8];
    unsigned dbg[W][4];        // commits, evaluations dropped by rollbacks, polls while waiting to be the frontier, polls at the lead limit
    struct Buf {
        double r[2][32], lr[2][32], t[2][32], A[2][32], B[2][32];
        int jb[2][32];
        double sc[8];          // gL gM lgL lgM poi lpoi priorA poiA
        int isc[4];            // K_l K_m poi_is_init consistent
    } buf[2];
};

// what an evaluation read / what a commit changed
#define TD_LV 1u          // rates, log-rates, shift times (and segment statistics) of the birth side
#define TD_LK 2u          // number of birth rates
#define TD_MV 4u
#define TD_MK 8u
#define TD_P 16u          // the stored Poisson prior priorPoiA (:300-304)
#define TD_ALL 31u        // + hyper-parameters, stored prior, consistency flag (Gibbs step, absolute-form iterations)
#define TEAM_VMASK 0xffffffu
__device__ __forceinline__ unsigned tv_version(unsigned long long vw) { return (unsigned)(vw >> 40); }
__device__ __forceinline__ unsigned tv_changed(unsigned long long vw) { return (unsigned)(vw >> 32) & 0xffu; }

__device__ __forceinline__ unsigned long long ld_volatile_shared(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.volatile.shared.u64 %0, [%1];" : "=l"(v) : "r"((unsigned)__cvta_generic_to_shared(p)) : "memory");
    return v;
}
__device__ __forceinline__ void st_volatile_shared(unsigned long long* p, unsigned long long v) {
    asm volatile("st.volatile.shared.u64 [%0], %1;" :: "r"((unsigned)__cvta_generic_to_shared(p)), "l"(v) : "memory");
}

// per-warp event counters of the team build: the increments of one iteration are a bit mask (bit k = counter k); the
// last eight masks wait in `hist` (newest in the low byte) and are only counted when they leave it -- by then the
// iteration is older than any possible rollback
struct TeamCounters {
    unsigned long long hist;
    unsigned long long dep;            // what each of those eight evaluations read (TD_* bits), same order
    unsigned lo, hi, pushes;
    unsigned n[8];
};
__device__ __noinline__ void tc_flush(TeamCounters& t) {
#pragma unroll
    for (int k = 0; k < 4; ++k) { t.n[k] += (t.lo >> (8 * k)) & 0xffu; t.n[4 + k] += (t.hi >> (8 * k)) & 0xffu; }
    t.lo = 0u; t.hi = 0u;
}
__device__ __forceinline__ void tc_push(TeamCounters& t, unsigned mask, unsigned dep) {
    const unsigned out = (unsigned)(t.hist >> 56);
    t.hist = (t.hist << 8) | (unsigned long long)mask;
    t.dep = (t.dep << 8) | (unsigned long long)dep;
    t.lo += ((out & 0xfu) * 0x00204081u) & 0x01010101u;       // bit k of the mask -> byte k
    t.hi += ((out >> 4) * 0x00204081u) & 0x01010101u;
    if ((++t.pushes & 127u) == 0u) tc_flush(t);
}

// event iterations (sample record :321, log-rate resync) as offsets from the launch's first iteration
struct TeamEvents {
    unsigned long long first_sample, s_every, first_resync;     // first_sample = ~0 when no records are written
    unsigned long long rec_done;                                // records of this launch written before the team's first iteration
    unsigned next_sample, next_resync, next_event;
};
__device__ __noinline__ void team_events_from(TeamEvents& e, unsigned i) {
    unsigned long long ns = ~0ull, nr;
    if (e.first_sample != ~0ull) ns = i <= e.first_sample ? e.first_sample : e.first_sample + (i - e.first_sample + e.s_every - 1) / e.s_every * e.s_every;
    nr = i <= e.first_resync ? e.first_resync : e.first_resync + ((unsigned long long)i - e.first_resync + LR_RESYNC - 1) / LR_RESYNC * LR_RESYNC;
    e.next_sample = ns > 0xffffffffull ? 0xffffffffu : (unsigned)ns;
    e.next_resync = nr > 0xffffffffull ? 0xffffffffu : (unsigned)nr;
    e.next_event = e.next_sample < e.next_resync ? e.next_sample : e.next_resync;
}

template <int W>
__device__ __noinline__ void team_publish_state(TeamShared<W>& T, unsigned v_new, unsigned changed, unsigned restart, const Side& L, const Side& M,
                                                const ChainRegs& c, int lane) {
    typename TeamShared<W>::Buf& b = T.buf[v_new & 1u];
    b.r[0][lane] = L.r; b.lr[0][lane] = L.lr; b.t[0][lane] = L.t; b.A[0][lane] = L.A; b.B[0][lane] = L.B; b.jb[0][lane] = L.jb;
    b.r[1][lane] = M.r; b.lr[1][lane] = M.lr; b.t[1][lane] = M.t; b.A[1][lane] = M.A; b.B[1][lane] = M.B; b.jb[1][lane] = M.jb;
    if (lane == 0) {
        b.sc[0] = c.hp.gL; b.sc[1] = c.hp.gM; b.sc[2] = c.hp.lgL; b.sc[3] = c.hp.lgM; b.sc[4] = c.hp.poi; b.sc[5] = c.hp.lpoi;
        b.sc[6] = c.priorA; b.sc[7] = c.poiA;
        b.isc[0] = L.K; b.isc[1] = M.K; b.isc[2] = c.poi_is_init; b.isc[3] = c.consistent;
    }
    __syncwarp();
    if (lane == 0) st_release_cta(&T.verword, ((unsigned long long)((v_new << 8) | changed) << 32) | restart);
}
template <int W>
__device__ __noinline__ void team_load_state(const TeamShared<W>& T, unsigned v, Side& L, Side& M, ChainRegs& c, int lane) {
    const typename TeamShared<W>::Buf& b = T.buf[v & 1u];
    L.r = b.r[0][lane]; L.lr = b.lr[0][lane]; L.t = b.t[0][lane]; L.A = b.A[0][lane]; L.B = b.B[0][lane]; L.jb = b.jb[0][lane];
    M.r = b.r[1][lane]; M.lr = b.lr[1][lane]; M.t = b.t[1][lane]; M.A = b.A[1][lane]; M.B = b.B[1][lane]; M.jb = b.jb[1][lane];
    c.hp.gL = b.sc[0]; c.hp.gM = b.sc[1]; c.hp.lgL = b.sc[2]; c.hp.lgM = b.sc[3]; c.hp.poi = b.sc[4]; c.hp.lpoi = b.sc[5];
    c.priorA = b.sc[6]; c.poiA = b.sc[7];
    L.K = b.isc[0]; M.K = b.isc[1]; c.poi_is_init = b.isc[2]; c.consistent = b.isc[3];
}

// true once every earlier iteration is published under version v (this warp is the chain's frontier at offset i);
// false if the version changed while waiting (the caller's evaluation is void)
template <int W>
__device__ __forceinline__ bool team_wait_frontier(const TeamShared<W>& T, unsigned v, unsigned i, int w, int lane, unsigned& polls) {
    for (;;) {
        const unsigned long long vw = ld_volatile_shared(&T.verword);
        if (tv_version(vw) != v) return false;
        const unsigned long long pw = ld_volatile_shared(&T.prog[lane % W]);
        const bool ok = (lane % W) == w || ((unsigned)(pw >> 32) == v && (unsigned)pw >= i);
        if (__all_sync(0xffffffffu, ok)) return true;
        ++polls;
        __nanosleep(20);
    }
}

// speculative evaluation of one block iteration (:254-272) on side `cur`: block_step's arithmetic without the commit.
// Returns 0 if the state stays as it is, else the kind of pending change with the proposed side in `nw`.
#define TEAM_WINDOW 2048u
#define TEAM_BAIL_DEN 8u
#define TEAM_INITIAL_SOLO 2048           // a fresh chain's first iterations go to the latency-optimised build
#define TEAM_SOLO_SPAN_MIN 8192
#define TEAM_SOLO_SPAN_MAX 262144
#define TEAM_PEND_NONE 0
#define TEAM_PEND_SIDE 1       // cur = nw
#define TEAM_PEND_RJ 2         // cur = nw, poiA = poiN
template <bool C>
__device__ __forceinline__ int team_block_eval(const Side& cur, const SideView v, const ChainRegs& c, const DataView& d,
                                               const lr_chain_config& cfg, const Draws& q, int lane, unsigned& mask, unsigned& dep, Side& nw) {
    const bool rate = (q.kind >> 1) == DK_BLOCK_RATE || cur.K == 1;
    const unsigned xv = (q.kind & 1) ? TD_LV : TD_MV, xk = (q.kind & 1) ? TD_LK : TD_MK;
    dep = (rate || cfg.real_move_shift) ? (xv | xk) : xk;
    if (rate) {
        mask |= (1u << 3) | (1u << 2);
        const bool on = lane < cur.K;
        const double dl = on ? q.dlt : 0.0;
        const double rn = cur.r * (on ? q.m : 1.0);
        const double x = warp_sum_first((c.beta * cur.A + 2.0) * dl - (c.beta * cur.B + v.g_cur) * (rn - cur.r), cur.K);
        if (mh_accept(x, q)) {
            mask |= 1u << 1;
            // no rate touched (Binomial(1, f) of :170 came out 0 everywhere): r * 1 and lr + 0 are the state's own bits
            if (__any_sync(0xffffffffu, dl != 0.0)) { nw = cur; nw.r = rn; nw.lr = cur.lr + dl; return TEAM_PEND_SIDE; }
        }
    } else if (!cfg.real_move_shift) {
        mask |= (1u << 4) | (1u << 2) | (1u << 1);
    } else {
        mask |= 1u << 4;
        if (propose_move<false>(cur, nw, d, v.tabA, v.tabB, q, lane)) {
            mask |= 1u << 2;
            const bool on = lane < cur.K;
            const double x = warp_sum(on ? c.beta * ((nw.A - cur.A) * cur.lr - (nw.B - cur.B) * cur.r) : 0.0);
            if (mh_accept(x, q)) { mask |= 1u << 1; return TEAM_PEND_SIDE; }
        }
    }
    return TEAM_PEND_NONE;
}
template <bool C>
__device__ __forceinline__ int team_rj_eval(const Side& cur, const Side& oth, const SideView v, const ChainRegs& c, const DataView& d,
                                            const Draws& q, int lane, unsigned& mask, unsigned& dep, Side& nw, double& poiN) {
    double hasting, x;
    bool cap;
    mask |= 1u << 5;
    dep = (q.kind & 1) ? (TD_LV | TD_LK | TD_MK | TD_P) : (TD_MV | TD_MK | TD_LK | TD_P);
    if (rj_propose<C>(cur, oth, v, c.hp, c.beta, c.poiA, d, q, lane, nw, hasting, poiN, x, cap)) {
        mask |= 1u << 2;
        if (mh_accept(x, q)) {
            mask |= 1u << 1;
            // remove-shift on a single-rate side proposes the state itself (:81-86); only the stored Poisson prior may move (:279, :319)
            if (nw.K != cur.K || poiN != c.poiA) return TEAM_PEND_RJ;
        }
    } else if (cap) {
        mask |= 1u << 7;
    }
    return TEAM_PEND_NONE;
}

// barrier of the W warps of one team: the whole CTA, or named barrier 1 / 2 for the two teams of 8 of a slot CTA
template <int W, bool SLICED>
__device__ __forceinline__ void team_sync() {
    if (SLICED && W == 8) asm volatile("bar.sync %0, 256;" :: "r"(1 + (int)(threadIdx.x >> 8)) : "memory");
    else __syncthreads();
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// One team of W warps runs `chain` for this launch: the CTA (one chain per CTA), or with SLICED one time slice of the slot
// kernel below, where a CTA of 16 warps is one team of 16 or two teams of 8 (threads 0-255 and 256-511).  There the chain's
// first iteration of the run is S->run_begin (set by the placement kernel), and once the global timer passes t_stop (0: no
// limit) the team stops at an iteration no commit has passed and leaves the rest to the next slice.
template <int W, bool SLICED>
__device__ __forceinline__ void team_run(const RunParams& P, const int lead, const int chain_arg, const unsigned long long t_stop) {
    constexpr bool C = true;
    __shared__ TeamShared<W> T_all[SLICED && W == 8 ? 2 : 1];
    TeamShared<W>& T = T_all[SLICED && W == 8 ? (threadIdx.x >> 8) : 0];
    const int lane = (int)(threadIdx.x & 31);
    const int w = (int)(SLICED ? (threadIdx.x >> 5) % W : threadIdx.x >> 5);
    ChainState* S = P.st + chain_arg;
    const long long it0 = S->it;
    const long long it_begin = P.it_begin >= 0 ? P.it_begin : (SLICED ? S->run_begin : it0);
    const long long n_own = it_begin + P.n_iter - it0;
    if (n_own <= 0 || (P.team_bail && it0 < S->solo_until)) return;      // whole team: nothing to do / left to the continuation pass
    if (w == 0 && lane == 0) {
        T.verword = 0ull; T.n_eff = (unsigned)n_own; T.stopped = 0u; T.win_i = 0u - S->win_iters; T.win_c = S->win_commits;
        T.chain = chain_arg; T.t_stop = t_stop;
    }
    if (w == 0 && lane < W) T.prog[lane] = (unsigned long long)lane;
    team_sync<W, SLICED>();

    const lr_chain_config& cfg = P.cfg;
    const LoopConsts& K = P.lc;
    Rng rng; rng.k0 = P.k0; rng.k1 = P.k1; rng.chain = S->chain_id;
    unsigned n = (unsigned)n_own;
    const DataView d = make_view(P.tab, P.cst, S->rep, P.nb, P.s0f, P.start_time, P.end_time);
    Side L, M;
    load_sides(S, L, M, lane);
    side_stats(L, d, T_AB, T_BB, lane);
    side_stats(M, d, T_AD, T_BD, lane);
    ChainRegs c;
    c.hp.gL = S->gL; c.hp.gM = S->gM; c.hp.lgL = log(c.hp.gL); c.hp.lgM = log(c.hp.gM); c.hp.poi = S->poi; c.hp.lpoi = log(c.hp.poi);
    c.priorA = S->priorA; c.poiA = S->poiA; c.beta = S->beta; c.poi_is_init = S->poi_is_init; c.consistent = (int)S->consistent;
    const bool frozen = (d.end_time - d.start_time) <= LR_MIN_DT;
    team_sync<W, SLICED>();           // every warp has read the chain's global state before anybody may finish and rewrite it

    TeamEvents ev;
    {
        const unsigned long long s_every = (unsigned long long)(P.sample_every > 0 ? P.sample_every : 1);
        ev.s_every = s_every;
        ev.first_sample = P.records != nullptr ? (s_every - (unsigned long long)it0 % s_every) % s_every : ~0ull;
        ev.rec_done = (unsigned long long)((it0 + (long long)s_every - 1) / (long long)s_every - (it_begin + (long long)s_every - 1) / (long long)s_every);
        ev.first_resync = (LR_RESYNC - (unsigned long long)it0 % LR_RESYNC) % LR_RESYNC;
    }
    TeamCounters tc;
    tc.hist = 0ull; tc.dep = 0ull; tc.lo = 0u; tc.hi = 0u; tc.pushes = 0u;
#pragma unroll
    for (int k = 0; k < 8; ++k) tc.n[k] = 0u;

    unsigned v = 0u, base = 0u, i = (unsigned)w;
    unsigned F_seen = 0u;             // a lower bound of the slowest warp's next iteration (it only grows)
    unsigned n_commit = 0u, n_drop = 0u, n_fwait = 0u, n_lead = 0u;
    team_events_from(ev, i);
    const unsigned lead_span = (unsigned)lead * W;

    for (;;) {
        // ---- has the chain moved on?  (a commit by another warp: reload; go back to the first own evaluation beyond the
        // commit that read something the commit changed)
        {
            const unsigned long long vw0 = ld_volatile_shared(&T.verword);
            if (tv_version(vw0) != v) {
                const unsigned long long vw = ld_acquire_cta(&T.verword);
                const unsigned v_new = tv_version(vw), changed = tv_changed(vw), base_new = (unsigned)vw;
                team_load_state<W>(T, v_new, L, M, c, lane);
                const unsigned i_first = base_new + ((unsigned)w + W - base_new % W) % W;
                const unsigned beyond = (i - i_first) / W;             // own evaluations at or after base_new (<= lead)
                unsigned long long conf = tc.dep & ((unsigned long long)changed * 0x0101010101010101ull);
                if (beyond < 8u) conf &= (1ull << (8u * beyond)) - 1ull;
                const unsigned dropped = conf ? (unsigned)(63 - __clzll((long long)conf)) / 8u + 1u : 0u;
                tc.hist >>= 8u * dropped; tc.dep >>= 8u * dropped;
                n_drop += dropped;
                i -= dropped * W; v = v_new; base = base_new;
                n = *(volatile unsigned*)&T.n_eff;
                if (F_seen < base) F_seen = base;
                team_events_from(ev, i);
                __syncwarp();
                if (lane == 0) st_volatile_shared(&T.prog[w], ((unsigned long long)v << 32) | i);
                continue;
            }
        }
        if (i >= n) {
            // my share is done; the launch ends when everybody's is (a rollback can still hand me iterations again)
            const unsigned long long pw = ld_volatile_shared(&T.prog[lane % W]);
            if (__all_sync(0xffffffffu, (unsigned)(pw >> 32) == v && (unsigned)pw >= n)) break;
            __nanosleep(200);
            continue;
        }
        if (i > F_seen + lead_span) {
            // not more than `lead` own iterations ahead of the slowest warp
            const unsigned long long pw = ld_volatile_shared(&T.prog[lane % W]);
            const unsigned nxt = (unsigned)(pw >> 32) == v ? (unsigned)pw : base;
            F_seen = __reduce_min_sync(0xffffffffu, nxt);
            if (i > F_seen + lead_span) { ++n_lead; __nanosleep(100); continue; }
        }
        if (SLICED && w == 0 && (i & (16u * W - 1u)) == 15u * W && *(volatile unsigned long long*)&T.t_stop != 0ull &&
            __shfl_sync(0xffffffffu, global_ns(), 0) >= *(volatile unsigned long long*)&T.t_stop) {
            // the slice is over (the timer is read every 16th own iteration: a slice does at least 15 W iterations): once every
            // earlier iteration is published, the team stops BEFORE iteration i, which nobody has committed or observed.  The
            // state stays as it is; the new version only carries the lowered n_eff to the others, which trim what they
            // evaluated at or beyond i as after a hand-over.
            if (!team_wait_frontier<W>(T, v, i, w, lane, n_fwait)) continue;
            v = (v + 1u) & TEAM_VMASK; base = i; n = i;
            if (lane == 0) { *(volatile unsigned*)&T.n_eff = i; *(volatile unsigned*)&T.stopped = 1u; }
            __syncwarp();
            team_publish_state<W>(T, v, 0u, i, L, M, c, lane);
            if (lane == 0) st_volatile_shared(&T.prog[w], ((unsigned long long)v << 32) | i);
            continue;
        }

        const long long it = it0 + (long long)i;
        const Draws q = make_draws<true>(rng, it, lane, K, L.K, M.K);
        const int kind = q.kind >> 1;
        const bool birth = (q.kind & 1) != 0;
        const bool event = i == ev.next_event;
        const bool serial = !c.consistent || frozen || kind == DK_GIBBS;
        unsigned mask = 0u, dep = TD_ALL;
        int pend = TEAM_PEND_NONE;
        Side nw;
        double poiN = 0.0;
        Side& cur = birth ? L : M;
        const Side& oth = birth ? M : L;
        if (!serial) {
            if (kind <= DK_BLOCK_MOVE) pend = team_block_eval<C>(cur, side_view(c.hp, birth), c, d, cfg, q, lane, mask, dep, nw);
            else pend = team_rj_eval<C>(cur, oth, side_view(c.hp, birth), c, d, q, lane, mask, dep, nw, poiN);
            if (pend == TEAM_PEND_NONE && !event) {
                // the common case: the state stays as it is
                tc_push(tc, mask, dep);
                i += W;
                if (lane == 0) st_volatile_shared(&T.prog[w], ((unsigned long long)v << 32) | i);
                if (i > ev.next_event) team_events_from(ev, i);
                continue;
            }
        }
        // ---- this iteration changes or observes the state: it has to be the chain's frontier
        if (!team_wait_frontier<W>(T, v, i, w, lane, n_fwait)) { ++n_drop; continue; }
        unsigned changed = 0u;
        if (serial) {
            Counters ns;
#pragma unroll
            for (int k = 0; k < 8; ++k) ns.v[k] = 0u;
            if (kind == DK_GIBBS) {
                ns.v[6]++;
                gibbs_step_ref(L, M, c, d, cfg.poisson_prior == 0.0 ? 1 : 0, cfg.use_rate_HP, rng, it, frozen, lane);
                c.consistent = 1;
                ns.v[1]++;
            } else {
                if (kind > DK_BLOCK_MOVE) ns.v[5]++;
                run_slow(cur, oth, side_view(c.hp, birth), c, ns, d, cfg, q, frozen, lane);
            }
#pragma unroll
            for (int k = 1; k < 8; ++k) mask |= ns.v[k] ? (1u << k) : 0u;
            changed = TD_ALL;
        } else if (pend != TEAM_PEND_NONE) {
            const unsigned xv = birth ? TD_LV : TD_MV, xk = birth ? TD_LK : TD_MK;
            changed = pend == TEAM_PEND_RJ ? (TD_P | (nw.K != cur.K ? (xv | xk) : 0u)) : xv;
            cur = nw;
            if (pend == TEAM_PEND_RJ) c.poiA = poiN;
        }
        if (event) {
            if (i == ev.next_resync) { resync_log_rates(L, M, lane); changed |= TD_LV | TD_MV; }
            if (i == ev.next_sample) {
                const unsigned long long k = ev.rec_done + ((unsigned long long)i - ev.first_sample) / ev.s_every;
                const int chain = SLICED ? *(volatile int*)&T.chain : chain_arg;
                write_record_ref(P.records + ((size_t)k * P.n_chains + chain) * LR_REC_DOUBLES, it, L, M, c, d, lane, P.with_adequacy != 0);
            }
        }
        if (changed) {
            v = (v + 1u) & TEAM_VMASK; base = i + 1u; ++n_commit;
            // Does speculation pay on this chain?  More than one state change in TEAM_BAIL_DEN iterations over a window of
            // TEAM_WINDOW: evaluating ahead mostly produces rollbacks (small tables, burn-in); the team stops after this
            // iteration and the continuation pass (the latency-optimised build) runs the rest of the launch.
            const unsigned wc = *(volatile unsigned*)&T.win_c + 1u, wlen = base - *(volatile unsigned*)&T.win_i;
            if (wlen >= TEAM_WINDOW) {
                if (P.team_bail && wc * TEAM_BAIL_DEN > wlen && base < n) { n = base; if (lane == 0) *(volatile unsigned*)&T.n_eff = base; }
                if (lane == 0) { *(volatile unsigned*)&T.win_i = base; *(volatile unsigned*)&T.win_c = 0u; }
            } else if (lane == 0) {
                *(volatile unsigned*)&T.win_c = wc;
            }
            __syncwarp();
            team_publish_state<W>(T, v, changed, base, L, M, c, lane);
        }
        tc_push(tc, mask, dep);
        i += W;
        if (lane == 0) st_volatile_shared(&T.prog[w], ((unsigned long long)v << 32) | i);
        if (i > ev.next_event) team_events_from(ev, i);
    }

    // ---- every warp holds the final state; warp 0 stores it, all add their counters
    {
        // evaluations kept through the rollbacks but beyond the iteration the team stopped at belong to the continuation pass
        const unsigned i_first = n + ((unsigned)w + W - n % W) % W;
        const unsigned beyond = i > i_first ? (i - i_first) / W : 0u;
        tc.hist = beyond >= 8u ? 0ull : (tc.hist >> (8u * beyond));
    }
    for (int k = 0; k < 8; ++k) tc_push(tc, 0u, 0u);
    tc_flush(tc);
    if (lane < 8) T.cnt[w][lane] = tc.n[lane];
    if (lane == 0) { T.dbg[w][0] = n_commit; T.dbg[w][1] = n_drop; T.dbg[w][2] = n_fwait; T.dbg[w][3] = n_lead; }
    team_sync<W, SLICED>();
    if (w == 0) {
        ChainState* S = P.st + (SLICED ? *(volatile int*)&T.chain : chain_arg);
        store_sides(S, L, M, lane);
        if (lane == 0) {
            const unsigned n_done = *(volatile unsigned*)&T.n_eff;
            S->it = it0 + (long long)n_done;
            S->team[4] += (long long)n_done;
            if (n_done < (unsigned)n_own && !*(volatile unsigned*)&T.stopped) {
                S->team[5] += 1;
                // handed over: for solo_span iterations, twice as long the next time
                const long long span = S->solo_span < TEAM_SOLO_SPAN_MIN ? TEAM_SOLO_SPAN_MIN : S->solo_span;
                S->solo_until = it0 + (long long)n_done + span;
                S->solo_span = 2 * span > TEAM_SOLO_SPAN_MAX ? TEAM_SOLO_SPAN_MAX : 2 * span;
            } else if (n_done >= 4u * TEAM_WINDOW) {
                S->solo_span = 0;
            }
            S->win_iters = n_done - *(volatile unsigned*)&T.win_i; S->win_commits = *(volatile unsigned*)&T.win_c;
            S->priorA = c.priorA; S->poiA = c.poiA; S->gL = c.hp.gL; S->gM = c.hp.gM; S->poi = c.hp.poi; S->poi_is_init = c.poi_is_init; S->consistent = (unsigned)c.consistent;
            S->counters[0] += (long long)n_done;
            for (int k = 1; k < 8; ++k) {
                long long s = 0;
                for (int ww = 0; ww < W; ++ww) s += (long long)T.cnt[ww][k];
                S->counters[k] += s;
            }
            for (int k = 0; k < 4; ++k) {
                long long s = 0;
                for (int ww = 0; ww < W; ++ww) s += (long long)T.dbg[ww][k];
                S->team[k] += s;
            }
        }
    }
}

template <int W>
__global__ void __launch_bounds__(W * 32, W >= 16 ? 1 : (W >= 8 ? 2 : 4)) k3_team_kernel(const RunParams P, const int lead) {
    if ((int)blockIdx.x >= P.n_chains) return;                       // whole CTA
    team_run<W, false>(P, lead, (int)blockIdx.x, 0ull);
}

// ---- time-sliced teams (between one and two chains per SM).  One CTA per SM of 16 warps hosts either ONE chain as a team
// of 16 or TWO chains as two teams of 8 (with their own shared state and barrier), as the placement kernel says.  A team of 8
// that shares its SM runs at about 4 iterations per microsecond, a team of 16 alone at about 6: with one CTA per chain the
// chains that share an SM set the launch's time while the SMs of the lone chains run out of work.  Slices of a fixed time
// (measured from the CTA's start) with the chains furthest behind moved to the lone slots in between keep every SM busy to the
// end; a chain is the same chain however its launch is cut (event iterations sit at absolute iteration numbers).
#define TEAM_SLICE_PLAN_RATE 6.0     // chain iterations per microsecond and SM the number of slices is planned with (bench statistics:
                                     // about 8 for two teams of 8, 6 for one of 16; a slower table leaves more to the last slice)
// The two layouts are two kernels, launched side by side on two streams over all slots; each CTA runs only the slots of its
// layout and returns at once from the others, so the SMs end up with one CTA each.  (One kernel with both bodies costs the
// registers of both: spills that made either layout 5 - 8 % slower than the one-chain-per-CTA kernels.)
template <int W>
__global__ void __launch_bounds__(512, 1) k3_team_slot_kernel(const RunParams P, const int lead, const int* __restrict__ place, const long long budget_ns) {
    const int a = place[2 * blockIdx.x], b = place[2 * blockIdx.x + 1];
    if (a < 0 || (b < 0) != (W == 16)) return;                      // no chain, or the other layout's slot
    const unsigned long long t_stop = budget_ns > 0 ? global_ns() + (unsigned long long)budget_ns : 0ull;
    team_run<W, true>(P, lead, W == 16 || threadIdx.x < 256 ? a : b, t_stop);
}

// Placement of the next slice: slot CTA s runs chain place[2 s] (-1: none), alone if place[2 s + 1] is -1, else beside it.  The
// chains furthest behind the end of the launch get the lone slots (every chain gets one once at most n_slots are left); chains
// that are done or inside a hand-over span get none.  first: the first slice of the launch, which records where each chain starts.
#define TEAM_PLACE_MAX 1024
__global__ void __launch_bounds__(TEAM_PLACE_MAX) k3_team_place_kernel(const RunParams P, int* __restrict__ place, const int n_slots, const int first) {
    __shared__ long long left[TEAM_PLACE_MAX];
    __shared__ int n_active;
    const int n = P.n_chains;                                        // <= 2 n_slots and <= TEAM_PLACE_MAX (lr_chains_run)
    if (threadIdx.x == 0) n_active = 0;
    for (int s = threadIdx.x; s < 2 * n_slots; s += blockDim.x) place[s] = -1;
    __syncthreads();
    for (int c = threadIdx.x; c < n; c += blockDim.x) {
        ChainState* S = P.st + c;
        const long long it = S->it;
        if (first) S->run_begin = it;
        const long long end = (P.it_begin >= 0 ? P.it_begin : S->run_begin) + P.n_iter;
        const bool active = it < end && !(P.team_bail && it < S->solo_until);
        left[c] = active ? end - it : -1;
        if (active) atomicAdd(&n_active, 1);
    }
    __syncthreads();
    const int m = n_active;
    const int n_lone = m <= n_slots ? m : 2 * n_slots - m;
    for (int c = threadIdx.x; c < n; c += blockDim.x) {
        const long long k = left[c];
        if (k < 0) continue;
        int r = 0;                                                   // rank: chains with more left go first, ties by index
        for (int j = 0; j < n; ++j) r += (left[j] > k || (left[j] == k && j < c)) ? 1 : 0;
        if (r < n_lone) place[2 * r] = c;
        else { const int q = r - n_lone; place[2 * (n_lone + q / 2) + (q & 1)] = c; }
    }
}
