// K1: lineages -> per-bin sufficient statistics, one streaming pass over (ts, te).
//
// Replaces the reference's per-bin loop over precompute_events()/get_br()
// (LiteRateForward.py:111-123, :519-523; extinct-only twin :529-549), which makes ~10 full
// passes over the lineages for EVERY bin.  Here every lineage is read once (16 B) and touches
// O(1) accumulators, using the identity of SURVEY 7.3:
//
//   a = floor(ts) - first_bin                         birth bin   (rule ts >= t0 && ts < t1, :120)
//   b = ceil(te) - 1 - first_bin                      death bin   (rule te >  t0 && te <= t1, :121)
//   br[j] = FS[j] + FE[j] + pre + sum_{i<=j} (D[i-1] - E[i])
//   FS[a] += floor(ts)+1-ts,  FE[b] += te-(ceil(te)-1),  D/E = births/deaths that carry time at risk
//
// Fractions are accumulated in 2^-52 fixed point (integers), so every accumulator is an integer
// sum: order-independent, run-to-run deterministic, and lineage shards of several GPUs combine
// with an int64 SUM all-reduce.  br is recovered by lr_bin_finalize as the correctly rounded
// exact sum.
//
// Kernel shape (B200, HBM-bound: 16 B/lineage, no reuse):
//   - grid = 5 CTAs of 256 threads per SM (48 registers/thread), each CTA owns one contiguous slice of the
//     flattened [replicate][lineage] space -> perfectly balanced, 2-3 flushes per CTA per launch;
//   - 128-bit coalesced streaming loads (ld.global.nc.L1::no_allocate.v2.f64), 2 deep per array per thread
//     = 80 KB in flight per SM (measured: 4 CTAs x 4 deep 6.06 TB/s, 5 x 2 deep 6.69 TB/s, 6 x 2 deep 5.88, 8 x 1 deep
//     5.49, 3 x 4 deep 4.57, 4 x 3 deep 6.75 but slower on real-valued tables);
//   - block-shared u32 histograms updated with shared-memory atomics (ATOMS.POPC.INC: lanes that hit the same bin
//     are merged by the hardware, so year-sorted tables cost the same as shuffled ones); fractional parts that
//     differ from the expected ones (integer ts, te = int + fe_ref) go through a 96-bit carry chain of 32-bit
//     shared atomics;
//   - measured on B200 (1M lineages x 256 replicates x 200 bins): 6.7 TB/s on integer-year tables
//     (dram__bytes_read = the algorithmic 16 B/lineage), 4.75 TB/s on real-valued times (stalls on the returning
//     atomics of the carry chain; overlapping the chains of four lineages by hand cost registers and was slower).  Two designs were measured and dropped: lane-private u16 histograms without
//     atomics (2.1 TB/s: 8 warps/SM cannot hide the serialised read-modify-write chains) and a joint
//     (birth bin, lifetime) table with one atomic per lineage (5.8 TB/s: more index arithmetic than it saves).
#include "lr_common.cuh"

namespace {


constexpr int K1_UNROLL = 2;                        // double2 loads in flight per array per thread
constexpr int K1_TILE = 64 * K1_UNROLL;             // lineages one warp consumes per tile
constexpr int ROW_SP = 0, ROW_EX = 1, ROW_CS_LO = 2, ROW_CS_HI = 3, ROW_CE_LO = 4, ROW_CE_HI = 5,
              ROW_SPX = 6, ROW_EXX = 7;

struct K1Params {
    const double* ts;
    const double* te;
    const int* ts_i;       // int32 years (lr_bin_accumulate_i32): ts = ts_i, te = te_i + jitter
    const int* te_i;
    double jitter;         // death_jitter of the int32 path, in [0, 1]
    int b_off;             // death bin of an int32 lineage = te_i + b_off - first_bin (0 for jitter > 0, -1 for jitter == 0)
    long long n, ld;
    int n_rep;
    int fb;                // first_bin
    unsigned nb;           // n_bins
    double fe_ref;
    long long fe_ref_fix;
    int dead_only;
    double end_time;
    long long* acc;
    long long acc_stride;  // int64 per row
    long long chunk;       // flattened lineages per CTA
    long long seg_max;     // forced flush period
    int vec_ok;
    int* hint;             // mapped host int: CTA 0 records whether its first tile carried fractional times (may be null)
};

// 96-bit unsigned accumulation out of 32-bit shared atomics: words [idx], [nb+idx], [2nb+idx]
__device__ __forceinline__ void add96(unsigned* arr, unsigned nb, unsigned idx, long long v) {
    unsigned lo = (unsigned)v, hi = (unsigned)((unsigned long long)v >> 32);
    unsigned old = atomicAdd(&arr[idx], lo);
    unsigned add2 = hi + (((unsigned)(old + lo) < lo) ? 1u : 0u);
    if (add2) {
        unsigned old2 = atomicAdd(&arr[nb + idx], add2);
        if ((unsigned)(old2 + add2) < add2) atomicAdd(&arr[2 * nb + idx], 1u);
    }
}

// ---- tables sorted by time (real-valued): the lanes of a warp, and the warp's consecutive tiles, sit on ONE bin for thousands
// of lineages, and 32 carry chains per lineage on one shared-memory word serialise (measured 1.8 TB/s; a per-lineage warp
// reduction with MATCH + REDUX reached 3.5 TB/s).  A RUN keeps the bin the warp is on and sums the fractions of every lineage
// that falls into it in REGISTERS, per lane; it touches shared memory only when the bin changes (or every 1023 lineages per lane,
// so that the 52-bit fractions cannot overflow the 64-bit lane sums).
struct K1Run {
    unsigned bin;                 // 0xffffffff: no run open
    unsigned cnt;                 // lineages per lane in the run (warp-uniform: lanes only ever advance together)
    unsigned long long acc;       // this lane's sum of fractions, 2^-52 fixed point
};
__device__ __forceinline__ void run_flush(K1Run& r, unsigned* cnt_arr, unsigned* frac_arr, unsigned nb) {
    if (r.cnt) {
        const unsigned p0 = __reduce_add_sync(0xffffffffu, (unsigned)r.acc & 0x3fffffu);
        const unsigned p1 = __reduce_add_sync(0xffffffffu, (unsigned)(r.acc >> 22) & 0x3fffffu);
        const unsigned p2 = __reduce_add_sync(0xffffffffu, (unsigned)(r.acc >> 44));
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&cnt_arr[r.bin], 32u * r.cnt);
            // total < 2^67: low 64 bits through the carry chain, the rest straight into the top word
            // total < 2^70, into the 96-bit accumulator word by word with explicit carries
            const unsigned __int128 t = (unsigned __int128)p0 + ((unsigned __int128)p1 << 22) + ((unsigned __int128)p2 << 44);
            if (t) {
                const unsigned w0 = (unsigned)t, w1 = (unsigned)(t >> 32), w2 = (unsigned)(t >> 64);
                const unsigned old0 = atomicAdd(&frac_arr[r.bin], w0);
                const unsigned long long s1 = (unsigned long long)w1 + (((unsigned)(old0 + w0) < w0) ? 1ull : 0ull);
                unsigned c1 = (unsigned)(s1 >> 32);
                if ((unsigned)s1) {
                    const unsigned old1 = atomicAdd(&frac_arr[nb + r.bin], (unsigned)s1);
                    c1 += ((unsigned)(old1 + (unsigned)s1) < (unsigned)s1) ? 1u : 0u;
                }
                if (w2 + c1) atomicAdd(&frac_arr[2 * nb + r.bin], w2 + c1);
            }
        }
    }
    r.cnt = 0u; r.acc = 0ull;
}

struct K1Smem {
    unsigned* hs32;       // [nb] births
    unsigned* he32;       // [nb] deaths whose fraction is the expected one (fe == fe_ref)
    unsigned* cS;         // [3][nb]
    unsigned* cE;         // [3][nb]
    unsigned* exC;        // [nb] deaths with any other fraction: every death takes exactly ONE of the two counters
};

// Lineages that are not (alive for a positive time, born inside the window): rare, global atomics.
// (the five fields it needs by value: a reference to the kernel's parameter block would make every CTA copy the block to
// local memory at entry)
__device__ __noinline__ void k1_irregular(int p_fb, unsigned p_nb, long long S, long long p_fe_ref_fix, long long* acc, double ts, double te) {
    const struct { int fb; unsigned nb; long long fe_ref_fix; } p = {p_fb, p_nb, p_fe_ref_fix};
    const double T0 = (double)p.fb, T1 = (double)p.fb + (double)p.nb;
    unsigned long long* row = (unsigned long long*)acc;
    bool live = te > ts;   // false for NaNs
    if (live) {
        if (ts >= T1) return;                 // born after the window: nothing
        // here ts < T0: alive before bin 0
        if (!(te > T0)) return;               // died before the window
        atomicAdd(&row[ROW_SPX * S + p.nb], 1ull);      // `pre`: present in every bin until its death
        if (te <= T1) {
            long long ci = (long long)ceil(te);
            unsigned b = (unsigned)(ci - 1 - p.fb);
            atomicAdd(&row[ROW_EX * S + b], 1ull);
            double fe = te - (double)(ci - 1);
            long long d = __double2ll_rn(fe * LR_FIX_SCALE) - p.fe_ref_fix;
            atomicAdd(&row[ROW_CE_LO * S + b], (unsigned long long)(d & 0xffffffffll));
            atomicAdd(&row[ROW_CE_HI * S + b], (unsigned long long)(d >> 32));
        }
        return;
    }
    // no time at risk (te <= ts or NaN): the reference still counts the events (:120-121)
    if (ts >= T0 && ts < T1) {
        unsigned a = (unsigned)((long long)floor(ts) - p.fb);
        atomicAdd(&row[ROW_SP * S + a], 1ull);
        atomicAdd(&row[ROW_SPX * S + a], 1ull);
    }
    if (te > T0 && te <= T1) {
        unsigned b = (unsigned)((long long)ceil(te) - 1 - p.fb);
        atomicAdd(&row[ROW_EX * S + b], 1ull);
        atomicAdd(&row[ROW_EXX * S + b], 1ull);
    }
}

__device__ __forceinline__ void k1_lineage(const K1Params& p, const K1Smem& s, long long* acc, double ts, double te) {
    if (p.dead_only) {
        if (!(te < p.end_time)) return;      // :531-532
    }
    const int ti = __double2int_rd(ts);
    const int ci = __double2int_ru(te);
    const unsigned a = (unsigned)(ti - p.fb);
    const unsigned b = (unsigned)(ci - 1 - p.fb);
    if ((te > ts) && (a < p.nb)) {
        atomicAdd(&s.hs32[a], 1u);
        const double fr = ts - (double)ti;
        if (fr != 0.0) add96(s.cS, p.nb, a, __double2ll_rn(fr * LR_FIX_SCALE));
        if (b < p.nb) {
            const double fe = te - (double)(ci - 1);
            if (fe != p.fe_ref) {
                atomicAdd(&s.exC[b], 1u);
                add96(s.cE, p.nb, b, __double2ll_rn(fe * LR_FIX_SCALE));
            } else {
                atomicAdd(&s.he32[b], 1u);
            }
        }
    } else {
        k1_irregular(p.fb, p.nb, p.acc_stride, p.fe_ref_fix, acc, ts, te);
    }
}

// the same lineage with run-length accumulation on the side(s) the segment's probe found sorted (warp-uniform flags); all 32
// lanes call it together
__device__ __forceinline__ void k1_lineage_runs(const K1Params& p, const K1Smem& s, long long* acc, double ts, double te,
                                                bool runS_on, bool runE_on, K1Run& rS, K1Run& rE) {
    const bool keep = !p.dead_only || (te < p.end_time);
    const int ti = __double2int_rd(ts);
    const int ci = __double2int_ru(te);
    const unsigned a = (unsigned)(ti - p.fb);
    const unsigned b = (unsigned)(ci - 1 - p.fb);
    const bool regular = keep && (te > ts) && (a < p.nb);
    const double fr = ts - (double)ti;
    const double fe = te - (double)(ci - 1);
    // ---- birth side
    bool doneS = false;
    if (runS_on) {
        if (__all_sync(0xffffffffu, regular && a == rS.bin)) {
            rS.cnt++; rS.acc += (unsigned long long)__double2ll_rn(fr * LR_FIX_SCALE);
            if (rS.cnt == 1023u) run_flush(rS, s.hs32, s.cS, p.nb);
            doneS = true;
        } else {
            run_flush(rS, s.hs32, s.cS, p.nb);
            const unsigned m = __ballot_sync(0xffffffffu, regular);
            rS.bin = m ? __shfl_sync(0xffffffffu, a, 31 - __clz(m)) : 0xffffffffu;     // the bin a sorted table moves on to
        }
    }
    if (regular && !doneS) {
        atomicAdd(&s.hs32[a], 1u);
        if (fr != 0.0) add96(s.cS, p.nb, a, __double2ll_rn(fr * LR_FIX_SCALE));
    }
    // ---- death side (only lineages that are regular on the birth side carry a death with time at risk here)
    const bool death = regular && b < p.nb;
    bool doneE = false;
    if (runE_on) {
        if (__all_sync(0xffffffffu, death && b == rE.bin && fe != p.fe_ref)) {
            rE.cnt++; rE.acc += (unsigned long long)__double2ll_rn(fe * LR_FIX_SCALE);
            if (rE.cnt == 1023u) run_flush(rE, s.exC, s.cE, p.nb);
            doneE = true;
        } else {
            run_flush(rE, s.exC, s.cE, p.nb);
            const unsigned m = __ballot_sync(0xffffffffu, death && fe != p.fe_ref);
            rE.bin = m ? __shfl_sync(0xffffffffu, b, 31 - __clz(m)) : 0xffffffffu;
        }
    }
    if (death && !doneE) {
        if (fe != p.fe_ref) {
            atomicAdd(&s.exC[b], 1u);
            add96(s.cE, p.nb, b, __double2ll_rn(fe * LR_FIX_SCALE));
        } else {
            atomicAdd(&s.he32[b], 1u);
        }
    }
    if (keep && !regular) k1_irregular(p.fb, p.nb, p.acc_stride, p.fe_ref_fix, acc, ts, te);
}

// the full tiles of one segment; RUNS = false is the plain stream (no per-lineage warp votes)
template <bool RUNS>
__device__ __forceinline__ void k1_tiles(const K1Params& p, const K1Smem& s, long long* acc, const double* ts, const double* te,
                                         long long A, long long ntiles, int warp, int W, int lane, bool runS_on, bool runE_on) {
    K1Run rS, rE;
    rS.bin = 0xffffffffu; rS.cnt = 0u; rS.acc = 0ull; rE = rS;
    if (p.vec_ok) {
        for (long long k = warp; k < ntiles; k += W) {
            const double2* t2 = (const double2*)(ts + A + k * K1_TILE) + lane;
            const double2* e2 = (const double2*)(te + A + k * K1_TILE) + lane;
            double2 sv[K1_UNROLL], ev[K1_UNROLL];
#pragma unroll
            for (int u = 0; u < K1_UNROLL; ++u) { sv[u] = ld_stream_f64x2(t2 + u * 32); ev[u] = ld_stream_f64x2(e2 + u * 32); }
#pragma unroll
            for (int u = 0; u < K1_UNROLL; ++u) {
                if constexpr (RUNS) {
                    k1_lineage_runs(p, s, acc, sv[u].x, ev[u].x, runS_on, runE_on, rS, rE);
                    k1_lineage_runs(p, s, acc, sv[u].y, ev[u].y, runS_on, runE_on, rS, rE);
                } else {
                    k1_lineage(p, s, acc, sv[u].x, ev[u].x);
                    k1_lineage(p, s, acc, sv[u].y, ev[u].y);
                }
            }
        }
    } else {
        for (long long k = warp; k < ntiles; k += W) {
            const double* t1 = ts + A + k * K1_TILE + lane;
            const double* e1 = te + A + k * K1_TILE + lane;
            double sv[2 * K1_UNROLL], ev[2 * K1_UNROLL];
#pragma unroll
            for (int u = 0; u < 2 * K1_UNROLL; ++u) { sv[u] = ld_stream_f64(t1 + u * 32); ev[u] = ld_stream_f64(e1 + u * 32); }
#pragma unroll
            for (int u = 0; u < 2 * K1_UNROLL; ++u) {
                if constexpr (RUNS) k1_lineage_runs(p, s, acc, sv[u], ev[u], runS_on, runE_on, rS, rE);
                else k1_lineage(p, s, acc, sv[u], ev[u]);
            }
        }
    }
    if constexpr (RUNS) { run_flush(rS, s.hs32, s.cS, p.nb); run_flush(rE, s.exC, s.cE, p.nb); }
}

// ---- int32 years (8 B per lineage): ts is an integer year, te an integer year plus the constant death jitter, so every
// fraction is the expected one and a regular lineage is exactly two ATOMS.POPC.INC
__device__ __forceinline__ void k1_lineage_i32(const K1Params& p, const K1Smem& s, long long* acc, int ts, int te) {
    const bool live = p.b_off == 0 ? (te >= ts) : (te > ts);          // te + jitter > ts
    if (p.dead_only) {
        if (!((double)te + p.jitter < p.end_time)) return;            // :531-532
    }
    const unsigned a = (unsigned)(ts - p.fb);
    const unsigned b = (unsigned)(te + p.b_off - p.fb);
    if (live && a < p.nb) {
        atomicAdd(&s.hs32[a], 1u);
        if (b < p.nb) atomicAdd(&s.he32[b], 1u);
    } else {
        k1_irregular(p.fb, p.nb, p.acc_stride, p.fe_ref_fix, acc, (double)ts, (double)te + p.jitter);
    }
}
__device__ __forceinline__ int4 ld_stream_s32x4(const int4* q) {
    int4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(q));
    return v;
}
__device__ __forceinline__ int ld_stream_s32(const int* q) {
    int v;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(q));
    return v;
}
constexpr int K1I_TILE = 128 * K1_UNROLL;           // lineages one warp consumes per tile of the int32 path (int4 loads)

__global__ void __launch_bounds__(256, 5) k1_bin_i32_kernel(const K1Params p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, W = blockDim.x >> 5;
    const unsigned nb = p.nb;
    K1Smem s;
    s.hs32 = (unsigned*)smem_raw; s.he32 = s.hs32 + nb; s.cS = nullptr; s.cE = nullptr; s.exC = nullptr;
    const long long total = p.n * (long long)p.n_rep;
    long long g0 = (long long)blockIdx.x * p.chunk;
    long long g1 = g0 + p.chunk;
    if (g1 > total) g1 = total;
    while (g0 < g1) {
        const long long rep = g0 / p.n;
        const long long s0 = g0 - rep * p.n;
        long long s1 = p.n;
        if (s1 - s0 > g1 - g0) s1 = s0 + (g1 - g0);
        if (s1 - s0 > p.seg_max) s1 = s0 + p.seg_max;
        g0 += s1 - s0;
        const int* ts = p.ts_i + rep * p.ld;
        const int* te = p.te_i + rep * p.ld;
        long long* acc = p.acc + rep * (LR_ACC_ROWS * p.acc_stride);
        for (unsigned i = tid; i < 2 * nb; i += blockDim.x) s.hs32[i] = 0u;
        __syncthreads();
        long long A = (s0 + K1I_TILE - 1) / K1I_TILE * K1I_TILE;
        if (A > s1) A = s1;
        const long long ntiles = p.vec_ok ? (s1 - A) / K1I_TILE : 0;
        const long long B = A + ntiles * K1I_TILE;
        for (long long i = s0 + tid; i < A; i += blockDim.x) k1_lineage_i32(p, s, acc, ld_stream_s32(ts + i), ld_stream_s32(te + i));
        for (long long i = B + tid; i < s1; i += blockDim.x) k1_lineage_i32(p, s, acc, ld_stream_s32(ts + i), ld_stream_s32(te + i));
        for (long long k = warp; k < ntiles; k += W) {
            const int4* t4 = (const int4*)(ts + A + k * K1I_TILE) + lane;
            const int4* e4 = (const int4*)(te + A + k * K1I_TILE) + lane;
            int4 sv[K1_UNROLL], ev[K1_UNROLL];
#pragma unroll
            for (int u = 0; u < K1_UNROLL; ++u) { sv[u] = ld_stream_s32x4(t4 + u * 32); ev[u] = ld_stream_s32x4(e4 + u * 32); }
#pragma unroll
            for (int u = 0; u < K1_UNROLL; ++u) {
                k1_lineage_i32(p, s, acc, sv[u].x, ev[u].x);
                k1_lineage_i32(p, s, acc, sv[u].y, ev[u].y);
                k1_lineage_i32(p, s, acc, sv[u].z, ev[u].z);
                k1_lineage_i32(p, s, acc, sv[u].w, ev[u].w);
            }
        }
        __syncthreads();
        unsigned long long* g = (unsigned long long*)acc;
        for (unsigned i = tid; i < nb; i += blockDim.x) {
            if (s.hs32[i]) atomicAdd(&g[ROW_SP * p.acc_stride + i], (unsigned long long)s.hs32[i]);
            if (s.he32[i]) atomicAdd(&g[ROW_EX * p.acc_stride + i], (unsigned long long)s.he32[i]);
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256, 5) k1_bin_kernel(const K1Params p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, W = blockDim.x >> 5;
    const unsigned nb = p.nb;

    // ---- carve shared memory: [2][nb] histograms, [7][nb] fraction accumulators
    K1Smem s;
    unsigned* hist32 = (unsigned*)smem_raw;
    s.hs32 = hist32;
    s.he32 = hist32 + nb;
    unsigned* corr = hist32 + 2 * nb;
    s.cS = corr;
    s.cE = corr + 3 * nb;
    s.exC = corr + 6 * nb;
    const size_t zero_words = 9 * (size_t)nb;

    const long long total = p.n * (long long)p.n_rep;
    long long g0 = (long long)blockIdx.x * p.chunk;
    long long g1 = g0 + p.chunk;
    if (g1 > total) g1 = total;

    while (g0 < g1) {
        // ---- one segment: a run of lineages of ONE replicate, at most seg_max long
        const long long rep = g0 / p.n;
        const long long s0 = g0 - rep * p.n;
        long long s1 = p.n;
        if (s1 - s0 > g1 - g0) s1 = s0 + (g1 - g0);
        if (s1 - s0 > p.seg_max) s1 = s0 + p.seg_max;
        g0 += s1 - s0;
        const double* ts = p.ts + rep * p.ld;
        const double* te = p.te + rep * p.ld;
        long long* acc = p.acc + rep * (LR_ACC_ROWS * p.acc_stride);

        for (size_t i = tid; i < zero_words; i += blockDim.x) ((unsigned*)smem_raw)[i] = 0u;
        __syncthreads();

        // head (up to the first tile boundary), full tiles, tail
        long long A = (s0 + K1_TILE - 1) / K1_TILE * K1_TILE;
        if (A > s1) A = s1;
        const long long ntiles = (s1 - A) / K1_TILE;
        const long long B = A + ntiles * K1_TILE;
        for (long long i = s0 + tid; i < A; i += blockDim.x) k1_lineage(p, s, acc, ld_stream_f64(ts + i), ld_stream_f64(te + i));
        for (long long i = B + tid; i < s1; i += blockDim.x) k1_lineage(p, s, acc, ld_stream_f64(ts + i), ld_stream_f64(te + i));
        // Sorted-looking table?  One probe per warp and segment: the first lineage of each lane's first tile.
        bool mergeS = false, mergeE = false;
        if (warp < ntiles) {
            const long long i0 = A + (long long)warp * K1_TILE + lane;
            const double t0 = ld_stream_f64(ts + i0), e0 = ld_stream_f64(te + i0);
            int sameS, sameE;
            __match_all_sync(0xffffffffu, __double2int_rd(t0), &sameS);
            __match_all_sync(0xffffffffu, __double2int_ru(e0), &sameE);
            // only tables that carry fractions reach the carry chains at all: integer-year tables keep the plain stream
            const bool fracS = __any_sync(0xffffffffu, t0 != floor(t0));
            const bool fracE = __any_sync(0xffffffffu, e0 - (ceil(e0) - 1.0) != p.fe_ref);
            mergeS = sameS != 0 && fracS; mergeE = sameE != 0 && fracE;
            if (blockIdx.x == 0 && tid == 0 && s0 == 0 && p.hint) *(volatile int*)p.hint = (fracS || fracE) ? 1 : 0;
        }
        if (mergeS || mergeE) k1_tiles<true>(p, s, acc, ts, te, A, ntiles, warp, W, lane, mergeS, mergeE);
        else k1_tiles<false>(p, s, acc, ts, te, A, ntiles, warp, W, lane, false, false);
        __syncthreads();

        // ---- flush this segment into the replicate's global accumulators
        unsigned long long* g = (unsigned long long*)acc;
        for (unsigned i = tid; i < nb; i += blockDim.x) {
            if (s.hs32[i]) atomicAdd(&g[ROW_SP * p.acc_stride + i], (unsigned long long)s.hs32[i]);
            if (s.he32[i] | s.exC[i]) atomicAdd(&g[ROW_EX * p.acc_stride + i], (unsigned long long)s.he32[i] + (unsigned long long)s.exC[i]);
        }
        for (unsigned i = tid; i < nb; i += blockDim.x) {
            const unsigned a0 = s.cS[i], a1 = s.cS[nb + i], a2 = s.cS[2 * nb + i];
            if (a0 | a1 | a2) {
                atomicAdd(&g[ROW_CS_LO * p.acc_stride + i], (unsigned long long)a0);
                atomicAdd(&g[ROW_CS_HI * p.acc_stride + i], (unsigned long long)a1 + ((unsigned long long)a2 << 32));
            }
            const unsigned n = s.exC[i];
            if (n) {
                // sum(fix(fe)) - n*fe_ref_fix, split into (low 32 bits, signed high part)
                __int128 v = ((__int128)s.cE[2 * nb + i] << 64) + ((__int128)s.cE[nb + i] << 32) + (__int128)s.cE[i];
                v -= (__int128)n * (__int128)p.fe_ref_fix;
                atomicAdd(&g[ROW_CE_LO * p.acc_stride + i], (unsigned long long)(v & 0xffffffff));
                atomicAdd(&g[ROW_CE_HI * p.acc_stride + i], (unsigned long long)(long long)(v >> 32));
            }
        }
        __syncthreads();
    }
}

// ---- LANE-PRIVATE fraction words: the build for real-valued tables, and the faster one for every table up to 310 bins ----
// On real-valued tables k1_bin_kernel is bound by the shared-memory data stage and by issue: its six atomics per lineage hit
// random bins, 32 random words fall on the 32 banks 3.1 deep on average (ncu, 1M x 256 shuffled: 168 M atomic wavefronts for
// 53.8 M atomic instructions, l1tex 83 % busy, 97 warp instructions per lineage at 69 % issue, 0.74 of the copy peak), and on
// sorted tables 32 carry chains per instruction land on ONE word.
// Here the two low words of each side's fraction sum exist once per LANE ([bin][2][32]: lane l only ever touches bank l), so a
// fraction atomic is one wavefront whatever the bins are, shuffled or sorted, and only the warps of the CTA contend for a word;
// the third word (one carry in >= 4096 additions) and the counters (ATOMS.POPC.INC, merged by the hardware) stay shared.
// 2 x 256 B per bin: 200 bins = 105 KB, ONE CTA of 1024 threads per SM (up to 439 bins; the L1 keeps what shared memory leaves:
// two CTAs of 512 threads, 210 KB of shared memory at 200 bins, ran 8 % slower).  Every birth adds its fraction and every death
// goes through the "other fraction" counter (sum(fix(fe)) - n * fix(fe_ref) is zero for the expected ones); a death outside
// the window lands in a spare bin; fix(x) is the mantissa of 1 + x (one DADD and an integer subtraction, identical to
// rn(x * 2^52) including ties and x == 1); the carries are add.cc / addc.  A regular lineage is straight-line code, 36 warp
// instructions against 60, and the two lineages of a 128-bit load issue their four carry chains together.
// Loads in flight: 4 double2 per array and thread (128 KB per SM) up to 310 bins, 2 beyond (the L1 is what shared memory leaves).
// Measured (tools/k1_bench.py 256, GB/s of 16 B per lineage, 200 bins; k1_bin_kernel in brackets): real-valued shuffled 6 890
// (4 850), sorted by birth 7 000 (4 500), integer years 6 940 (6 690), sorted 7 050 (6 710) -- 1.05 - 1.08 of the copy peak, a
// read-only stream; 300 bins 6 410 / 6 930, 400 bins 5 760 / 5 940.  Flushing every 128 000 lineages (which would make the high
// word's carry unnecessary) cost 8 %: each flush drains the CTA's loads.  Integer sums: the accumulators hold the same totals as
// k1_bin_kernel's, the finalized statistics are bit-identical.
constexpr int K1L_THREADS = 1024;                    // ONE CTA per SM: two of 512 leave the L1 18 KB at 200 bins and run 8 % slower
constexpr size_t K1L_WORDS_PER_BIN = 4 * 32 + 4;

struct K1Lanes {
    unsigned* hs32; unsigned* exC;      // [nb + 1] births, deaths (generic pointers: ATOMS.POPC.INC)
    unsigned S0, E0;                    // shared-window byte addresses of THIS LANE's low word of bin 0 in [nb + 1][2][32] (high word: + 128)
    unsigned topS, topE;                // ... of the [nb + 1] third words, shared by the lanes
};

// 2^-52 fixed point of x in [0, 1]: the mantissa of 1 + x (exponent step included when 1 + x rounds to 2)
__device__ __forceinline__ void fix_of(double x, unsigned& lo, unsigned& hi) {
    const long long b = __double_as_longlong(x + 1.0);
    lo = (unsigned)b; hi = (unsigned)((unsigned long long)b >> 32) - 0x3ff00000u;
}
__device__ __forceinline__ void add_lanes(unsigned addr, unsigned top_addr, unsigned lo, unsigned hi) {
    unsigned old, old2, c;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(addr), "r"(lo) : "memory");
    asm("{ .reg .u32 t; add.cc.u32 t, %1, %2; addc.u32 %0, %0, 0; }" : "+r"(hi) : "r"(old), "r"(lo));      // carry of the low word
    asm volatile("atom.shared.add.u32 %0, [%1+128], %2;" : "=r"(old2) : "r"(addr), "r"(hi) : "memory");
    asm("{ .reg .u32 t; add.cc.u32 t, %1, %2; addc.u32 %0, 0, 0; }" : "=r"(c) : "r"(old2), "r"(hi));       // of the high word: once in >= 4096 additions
    if (c) asm volatile("red.shared.add.u32 [%0], 1;" :: "r"(top_addr) : "memory");
}

// a lineage born inside the window and alive for a positive time, straight-line: a death outside the window (an extant lineage)
// goes to the spare bin nb, which the flush ignores
__device__ __forceinline__ void k1_regular_lanes(const K1Params& p, const K1Lanes& s, double ts, double te, int ti, unsigned a, int c1, unsigned b) {
    unsigned lo, hi, lo2, hi2;
    b = min(b, p.nb);
    atomicAdd(&s.hs32[a], 1u);
    atomicAdd(&s.exC[b], 1u);
    fix_of(ts - (double)ti, lo, hi);
    fix_of(te - (double)c1, lo2, hi2);
    add_lanes(s.S0 + a * 256u, s.topS + a * 4u, lo, hi);
    add_lanes(s.E0 + b * 256u, s.topE + b * 4u, lo2, hi2);
}

template <bool DEAD_ONLY>
__device__ __forceinline__ void k1_lineage_lanes(const K1Params& p, const K1Lanes& s, long long* acc, double ts, double te) {
    if constexpr (DEAD_ONLY) {
        if (!(te < p.end_time)) return;      // :531-532
    }
    const int ti = __double2int_rd(ts);
    const int c1 = __double2int_ru(te) - 1;
    const unsigned a = (unsigned)(ti - p.fb);
    const unsigned b = (unsigned)(c1 - p.fb);
    if ((te > ts) && (a < p.nb)) k1_regular_lanes(p, s, ts, te, ti, a, c1, b);
    else k1_irregular(p.fb, p.nb, p.acc_stride, p.fe_ref_fix, acc, ts, te);
}

// the two lineages of one 128-bit load: when both are regular (nearly always) their four carry chains are issued together
template <bool DEAD_ONLY>
__device__ __forceinline__ void k1_pair_lanes(const K1Params& p, const K1Lanes& s, long long* acc, double2 ts, double2 te) {
    const int t0 = __double2int_rd(ts.x), t1 = __double2int_rd(ts.y);
    const int c0 = __double2int_ru(te.x) - 1, c1 = __double2int_ru(te.y) - 1;
    const unsigned a0 = (unsigned)(t0 - p.fb), a1 = (unsigned)(t1 - p.fb);
    bool r0 = (te.x > ts.x) && (a0 < p.nb), r1 = (te.y > ts.y) && (a1 < p.nb);
    if constexpr (DEAD_ONLY) { r0 = r0 && (te.x < p.end_time); r1 = r1 && (te.y < p.end_time); }
    if (r0 && r1) {
        k1_regular_lanes(p, s, ts.x, te.x, t0, a0, c0, (unsigned)(c0 - p.fb));
        k1_regular_lanes(p, s, ts.y, te.y, t1, a1, c1, (unsigned)(c1 - p.fb));
    } else {
        k1_lineage_lanes<DEAD_ONLY>(p, s, acc, ts.x, te.x);
        k1_lineage_lanes<DEAD_ONLY>(p, s, acc, ts.y, te.y);
    }
}

// sum over the 32 lane copies of one bin's two words: sum(low) + (sum(high) << 32), as a 128-bit value (all lanes get it)
__device__ __forceinline__ unsigned __int128 lanes_total(const unsigned* w, unsigned bin, unsigned lane) {
    const unsigned x0 = w[bin * 64u + lane], x1 = w[bin * 64u + 32u + lane];
    const unsigned long long t0 = (unsigned long long)__reduce_add_sync(0xffffffffu, x0 & 0xffffu) +
                                  ((unsigned long long)__reduce_add_sync(0xffffffffu, x0 >> 16) << 16);
    const unsigned long long t1 = (unsigned long long)__reduce_add_sync(0xffffffffu, x1 & 0xffffu) +
                                  ((unsigned long long)__reduce_add_sync(0xffffffffu, x1 >> 16) << 16);
    return (unsigned __int128)t0 + ((unsigned __int128)t1 << 32);
}

// K1L_UNROLL: double2 loads in flight per array per thread (32 KB per SM each)
template <bool DEAD_ONLY, int K1L_UNROLL>
__global__ void __launch_bounds__(K1L_THREADS, 1) k1_bin_lanes_kernel(const K1Params p) {
    constexpr int K1L_TILE = 64 * K1L_UNROLL;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, warp = tid >> 5, W = blockDim.x >> 5;
    const unsigned lane = (unsigned)tid & 31u;
    const unsigned nb = p.nb;
    unsigned* const wS = (unsigned*)smem_raw;              // [nb + 1][2][32]
    unsigned* const wE = wS + 64 * (size_t)(nb + 1);       // [nb + 1][2][32]
    K1Lanes s;
    s.hs32 = wE + 64 * (size_t)(nb + 1); s.exC = s.hs32 + (nb + 1);
    unsigned* const tS_top = s.exC + (nb + 1); unsigned* const tE_top = tS_top + (nb + 1);
    s.topS = (unsigned)__cvta_generic_to_shared(tS_top); s.topE = (unsigned)__cvta_generic_to_shared(tE_top);
    s.S0 = (unsigned)__cvta_generic_to_shared(wS) + lane * 4u; s.E0 = (unsigned)__cvta_generic_to_shared(wE) + lane * 4u;
    asm volatile("" : "+r"(s.S0), "+r"(s.E0));       // opaque: kept in two registers instead of being recomputed per lineage
    const size_t zero_words = K1L_WORDS_PER_BIN * (size_t)(nb + 1);
    const size_t zero_vec = zero_words / 4;

    const long long total = p.n * (long long)p.n_rep;
    long long g0 = (long long)blockIdx.x * p.chunk;
    long long g1 = g0 + p.chunk;
    if (g1 > total) g1 = total;

    while (g0 < g1) {
        const long long rep = g0 / p.n;
        const long long s0 = g0 - rep * p.n;
        long long s1 = p.n;
        if (s1 - s0 > g1 - g0) s1 = s0 + (g1 - g0);
        if (s1 - s0 > p.seg_max) s1 = s0 + p.seg_max;
        g0 += s1 - s0;
        const double* ts = p.ts + rep * p.ld;
        const double* te = p.te + rep * p.ld;
        long long* acc = p.acc + rep * (LR_ACC_ROWS * p.acc_stride);

        for (size_t i = tid; i < zero_vec; i += blockDim.x) ((uint4*)smem_raw)[i] = make_uint4(0u, 0u, 0u, 0u);
        for (size_t i = zero_vec * 4 + tid; i < zero_words; i += blockDim.x) ((unsigned*)smem_raw)[i] = 0u;
        __syncthreads();

        long long A = (s0 + K1L_TILE - 1) / K1L_TILE * K1L_TILE;
        if (A > s1) A = s1;
        const long long ntiles = (s1 - A) / K1L_TILE;
        const long long B = A + ntiles * K1L_TILE;
        for (long long i = s0 + tid; i < A; i += blockDim.x) k1_lineage_lanes<DEAD_ONLY>(p, s, acc, ld_stream_f64(ts + i), ld_stream_f64(te + i));
        for (long long i = B + tid; i < s1; i += blockDim.x) k1_lineage_lanes<DEAD_ONLY>(p, s, acc, ld_stream_f64(ts + i), ld_stream_f64(te + i));
        if (blockIdx.x == 0 && warp == 0 && s0 == 0 && p.hint && s1 - s0 >= 32) {      // the kind of table, for the next call
            const double t0 = ld_stream_f64(ts + s0 + lane), e0 = ld_stream_f64(te + s0 + lane);
            const bool frac = __any_sync(0xffffffffu, t0 != floor(t0) || e0 - (ceil(e0) - 1.0) != p.fe_ref);
            if (lane == 0) *(volatile int*)p.hint = frac ? 1 : 0;
        }
        for (long long k = warp; k < ntiles; k += W) {
            const double2* t2 = (const double2*)(ts + A + k * K1L_TILE) + lane;
            const double2* e2 = (const double2*)(te + A + k * K1L_TILE) + lane;
            double2 sv[K1L_UNROLL], ev[K1L_UNROLL];
#pragma unroll
            for (int u = 0; u < K1L_UNROLL; ++u) { sv[u] = ld_stream_f64x2(t2 + u * 32); ev[u] = ld_stream_f64x2(e2 + u * 32); }
#pragma unroll
            for (int u = 0; u < K1L_UNROLL; ++u) {
                k1_pair_lanes<DEAD_ONLY>(p, s, acc, sv[u], ev[u]);
            }
        }
        __syncthreads();

        // ---- flush: counters as in k1_bin_kernel; one warp per bin folds the 32 lane copies
        unsigned long long* g = (unsigned long long*)acc;
        for (unsigned i = tid; i < nb; i += blockDim.x) {
            if (s.hs32[i]) atomicAdd(&g[ROW_SP * p.acc_stride + i], (unsigned long long)s.hs32[i]);
            if (s.exC[i]) atomicAdd(&g[ROW_EX * p.acc_stride + i], (unsigned long long)s.exC[i]);
        }
        for (unsigned i = warp; i < nb; i += W) {
            const unsigned nS = s.hs32[i], nE = s.exC[i];                                     // warp-uniform
            unsigned __int128 tS = 0, tE = 0;
            if (nS) tS = lanes_total(wS, i, lane) + ((unsigned __int128)tS_top[i] << 64);
            if (nE) tE = lanes_total(wE, i, lane) + ((unsigned __int128)tE_top[i] << 64);
            if (lane == 0) {
                if (tS) {
                    atomicAdd(&g[ROW_CS_LO * p.acc_stride + i], (unsigned long long)(tS & 0xffffffffu));
                    atomicAdd(&g[ROW_CS_HI * p.acc_stride + i], (unsigned long long)(tS >> 32));
                }
                if (nE) {
                    const __int128 v = (__int128)tE - (__int128)nE * (__int128)p.fe_ref_fix;
                    if (v != 0) {
                        atomicAdd(&g[ROW_CE_LO * p.acc_stride + i], (unsigned long long)(v & 0xffffffff));
                        atomicAdd(&g[ROW_CE_HI * p.acc_stride + i], (unsigned long long)(long long)(v >> 32));
                    }
                }
            }
        }
        __syncthreads();
    }
}

// exact conversion of a non-negative 128-bit fixed-point value (2^-52 units) to the nearest double
__device__ double fix128_to_double(unsigned __int128 f) {
    unsigned long long hi = (unsigned long long)(f >> 64), lo = (unsigned long long)f;
    if (hi == 0) {
        if (lo < (1ull << 53)) return (double)lo * (1.0 / LR_FIX_SCALE);
        return __ull2double_rn(lo) * (1.0 / LR_FIX_SCALE);     // single rounding, scaling by 2^-52 is exact
    }
    int sh = 64 - __clzll(hi);                                  // bits above the low word
    unsigned long long top = (unsigned long long)(f >> sh);
    bool sticky = (f & ((((unsigned __int128)1) << sh) - 1)) != 0;
    top |= sticky ? 1ull : 0ull;
    return ldexp(__ull2double_rn(top), sh - LR_FIX_SHIFT);
}

// one CTA per replicate: integer prefix scan + exact reconstruction of br
__global__ void __launch_bounds__(256) k1_finalize_kernel(const long long* __restrict__ acc_all, long long acc_stride, int nb,
                                                          long long fe_ref_fix, long long* __restrict__ sp_out,
                                                          long long* __restrict__ ex_out, double* __restrict__ br_out) {
    __shared__ long long warp_tot[8];
    __shared__ long long carry_s;
    const int rep = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long* acc = acc_all + (long long)rep * LR_ACC_ROWS * acc_stride;
    if (tid == 0) carry_s = acc[ROW_SPX * acc_stride + nb];     // lineages alive before bin 0
    __syncthreads();
    for (int base = 0; base < nb; base += blockDim.x) {
        const int j = base + tid;
        long long D = 0, E = 0, x = 0;
        if (j < nb) {
            D = acc[ROW_SP * acc_stride + j] - acc[ROW_SPX * acc_stride + j];
            E = acc[ROW_EX * acc_stride + j] - acc[ROW_EXX * acc_stride + j];
            long long Dprev = j > 0 ? acc[ROW_SP * acc_stride + j - 1] - acc[ROW_SPX * acc_stride + j - 1] : 0;
            x = Dprev - E;
        }
        // inclusive block scan of x
        long long v = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            long long t = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += t;
        }
        if (lane == 31) warp_tot[warp] = v;
        __syncthreads();
        long long off = carry_s;
        for (int w = 0; w < warp; ++w) off += warp_tot[w];
        const long long c = v + off;                              // lineages spanning all of bin j ... minus deaths in j
        __syncthreads();
        if (tid == blockDim.x - 1) carry_s = c;
        if (j < nb) {
            __int128 cS = (__int128)acc[ROW_CS_LO * acc_stride + j] + ((__int128)acc[ROW_CS_HI * acc_stride + j] << 32);
            __int128 cE = (__int128)acc[ROW_CE_LO * acc_stride + j] + ((__int128)acc[ROW_CE_HI * acc_stride + j] << 32);
            __int128 F = ((__int128)(c + D) << LR_FIX_SHIFT) - cS + (__int128)E * (__int128)fe_ref_fix + cE;
            if (F < 0) F = 0;
            sp_out[(long long)rep * nb + j] = acc[ROW_SP * acc_stride + j];
            ex_out[(long long)rep * nb + j] = acc[ROW_EX * acc_stride + j];
            br_out[(long long)rep * nb + j] = fix128_to_double((unsigned __int128)F);
        }
        __syncthreads();
    }
}

}  // namespace

extern "C" int64_t lr_acc_stride(int32_t n_bins) { return ((int64_t)n_bins + 1 + 7) / 8 * 8; }

static long long fe_fix(double fe_ref) { return (long long)llrint(fe_ref * LR_FIX_SCALE); }

extern "C" int lr_bin_accumulate(lr_handle_t h, const double* d_ts, const double* d_te, int64_t n, int64_t ld,
                                 int32_t n_rep, int64_t first_bin, int32_t n_bins, double fe_ref,
                                 int32_t dead_only, double end_time, int64_t* d_acc, void* stream) {
    LR_REQUIRE(h != nullptr, "lr_bin_accumulate: null handle");
    LR_REQUIRE(n >= 0 && n_rep >= 1 && ld >= n, "lr_bin_accumulate: need n >= 0, n_rep >= 1, ld >= n");
    LR_REQUIRE(n_bins >= 1, "lr_bin_accumulate: n_bins must be >= 1");
    LR_REQUIRE(fe_ref > 0.0 && fe_ref <= 1.0, "lr_bin_accumulate: fe_ref must lie in (0, 1]");
    LR_REQUIRE(d_acc != nullptr && (n == 0 || (d_ts != nullptr && d_te != nullptr)), "lr_bin_accumulate: null pointer");
    const size_t smem_need = 9 * (size_t)n_bins * sizeof(unsigned);
    if (first_bin <= -(1ll << 30) || first_bin >= (1ll << 30) || smem_need + 1024 > (size_t)h->max_smem_optin) {
        lr_set_error("lr_bin_accumulate: |first_bin| must be < 2^30 and the 9 x n_bins shared-memory counters must fit one SM (n_bins <= %d)",
                     (int)(((size_t)h->max_smem_optin - 1024) / (9 * sizeof(unsigned))));
        return LR_ERR_UNSUPPORTED;
    }
    if (n == 0) return LR_OK;
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    LR_CUDA(cudaSetDevice(h->device));

    K1Params p;
    p.ts = d_ts; p.te = d_te; p.n = n; p.ld = ld; p.n_rep = n_rep;
    p.fb = (int)first_bin; p.nb = (unsigned)n_bins; p.fe_ref = fe_ref; p.fe_ref_fix = fe_fix(fe_ref);
    p.dead_only = dead_only; p.end_time = end_time;
    p.acc = (long long*)d_acc; p.acc_stride = lr_acc_stride(n_bins);
    p.vec_ok = (((uintptr_t)d_ts | (uintptr_t)d_te) & 15) == 0 && (ld % 2 == 0 || n_rep == 1);

    const size_t smem = 9 * (size_t)n_bins * sizeof(unsigned);
    const size_t budget = (size_t)h->max_smem_optin - 1024;
    int per_sm = (int)(budget / (smem + 1024));
    if (per_sm > 5) per_sm = 5;
    if (per_sm < 1) per_sm = 1;
    const int threads = 256, blocks = h->sm_count * per_sm;
    p.seg_max = 1ll << 31;             // u32 counters: at most 2^31 lineages between flushes
    const long long total = n * (long long)n_rep;
    long long chunk = (total + blocks - 1) / blocks;
    chunk = (chunk + K1_TILE - 1) / K1_TILE * K1_TILE;
    p.chunk = chunk;
    const int used = (int)((total + chunk - 1) / chunk);
    p.hint = h->k1_hint;
    h->k1_hint_used = 1;
    // The lane-private build (k1_bin_lanes_kernel): every kind of table up to 310 bins (164 KB of shared memory: it is the faster
    // build there, 4 loads deep) with at least 250 000 lineages per replicate, real-valued tables up to 439 bins (2 deep beyond 310)
    // with at least 50 000 (the previous pass through the handle tells the kind of table, K1Params::hint); the general build
    // otherwise, and always for the host-buffer entry points (lr_common.cuh).
    // LR_K1_LANES=0 / 1 forces the choice.
    const size_t smem_l = K1L_WORDS_PER_BIN * ((size_t)n_bins + 1) * sizeof(unsigned);
    const char* e_l = getenv("LR_K1_LANES");
    const bool lanes_fit = smem_l <= (size_t)h->max_smem_optin && p.vec_ok;
    const bool lanes_deep = n_bins <= 310;                      // 164 KB of shared memory: 4 loads deep still pays (measured at 300, not at 400)
    // (a CTA zeroes and folds its 528 B per bin once per replicate it touches: below a quarter of a million lineages per replicate --
    // 50 000 for real-valued tables -- the general build's 36 B per bin win; measured at 1 000 / 10 000 / 100 000 lineages per replicate)
    const bool real_seen = *(volatile int*)h->k1_hint == 1;
    const bool lanes_pay = (lanes_deep && n >= 250000) || (real_seen && n >= 50000);
    const bool lanes = lanes_fit && (e_l ? atoi(e_l) != 0 : (!h->k1_general_only && lanes_pay));
    h->k1_last_build = lanes ? 1 : 0;
    if (lanes) {
        const int blocks_l = h->sm_count;
        const int unroll = lanes_deep ? 4 : 2;
        const int tile_l = 64 * unroll;
        long long chunk_l = (total + blocks_l - 1) / blocks_l;
        chunk_l = (chunk_l + tile_l - 1) / tile_l * tile_l;
        p.chunk = chunk_l;
        const int used_l = (int)((total + chunk_l - 1) / chunk_l);
#define LR_K1L(D, U) do { LR_CUDA(cudaFuncSetAttribute(k1_bin_lanes_kernel<D, U>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_l)); \
                          k1_bin_lanes_kernel<D, U><<<used_l, K1L_THREADS, smem_l, st>>>(p); } while (0)
        if (dead_only) { if (unroll == 2) LR_K1L(true, 2); else LR_K1L(true, 4); }
        else { if (unroll == 2) LR_K1L(false, 2); else LR_K1L(false, 4); }
#undef LR_K1L
        LR_CUDA(cudaGetLastError());
        h->launches += 1;
        return LR_OK;
    }
    LR_CUDA(cudaFuncSetAttribute(k1_bin_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k1_bin_kernel<<<used, threads, smem, st>>>(p);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    return LR_OK;
}

extern "C" int lr_bin_accumulate_i32(lr_handle_t h, const int32_t* d_ts, const int32_t* d_te, int64_t n, int64_t ld,
                                     int32_t n_rep, int64_t first_bin, int32_t n_bins, double death_jitter,
                                     int32_t dead_only, double end_time, int64_t* d_acc, void* stream) {
    LR_REQUIRE(h != nullptr, "lr_bin_accumulate_i32: null handle");
    LR_REQUIRE(n >= 0 && n_rep >= 1 && ld >= n, "lr_bin_accumulate_i32: need n >= 0, n_rep >= 1, ld >= n");
    LR_REQUIRE(n_bins >= 1, "lr_bin_accumulate_i32: n_bins must be >= 1");
    // every regular death is counted with the fraction death_jitter: the fp64 table's fl(year + jitter) has it for every
    // |year| < 2^31 iff the jitter is a multiple of 2^-22
    LR_REQUIRE(death_jitter >= 0.0 && death_jitter <= 1.0 && ldexp(death_jitter, 22) == floor(ldexp(death_jitter, 22)),
               "lr_bin_accumulate_i32: death_jitter must be a multiple of 2^-22 in [0, 1] (year + jitter exact for every int32 year); "
               "bin other jitters as fp64 tables");
    LR_REQUIRE(d_acc != nullptr && (n == 0 || (d_ts != nullptr && d_te != nullptr)), "lr_bin_accumulate_i32: null pointer");
    const size_t smem = 2 * (size_t)n_bins * sizeof(unsigned);
    if (first_bin <= -(1ll << 30) || first_bin >= (1ll << 30) || smem + 1024 > (size_t)h->max_smem_optin) {
        lr_set_error("lr_bin_accumulate_i32: |first_bin| must be < 2^30 and the 2 x n_bins shared-memory counters must fit one SM");
        return LR_ERR_UNSUPPORTED;
    }
    if (n == 0) return LR_OK;
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    LR_CUDA(cudaSetDevice(h->device));
    K1Params p;
    memset(&p, 0, sizeof(p));
    p.ts_i = d_ts; p.te_i = d_te; p.jitter = death_jitter; p.b_off = death_jitter > 0.0 ? 0 : -1;
    p.n = n; p.ld = ld; p.n_rep = n_rep;
    p.fb = (int)first_bin; p.nb = (unsigned)n_bins;
    p.fe_ref = death_jitter > 0.0 ? death_jitter : 1.0;           // finalize with this fe_ref (lr_fe_ref_of_jitter)
    p.fe_ref_fix = fe_fix(p.fe_ref);
    p.dead_only = dead_only; p.end_time = end_time;
    p.acc = (long long*)d_acc; p.acc_stride = lr_acc_stride(n_bins);
    p.vec_ok = (((uintptr_t)d_ts | (uintptr_t)d_te) & 15) == 0 && (ld % 4 == 0 || n_rep == 1);
    const int threads = 256, blocks = h->sm_count * 5;
    p.seg_max = 1ll << 31;
    const long long total = n * (long long)n_rep;
    long long chunk = (total + blocks - 1) / blocks;
    chunk = (chunk + K1I_TILE - 1) / K1I_TILE * K1I_TILE;
    p.chunk = chunk;
    const int used = (int)((total + chunk - 1) / chunk);
    LR_CUDA(cudaFuncSetAttribute(k1_bin_i32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k1_bin_i32_kernel<<<used, threads, smem, st>>>(p);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    return LR_OK;
}

extern "C" int lr_bin_table_hint(lr_handle_t h, int32_t* out) {
    LR_REQUIRE(h != nullptr && out != nullptr, "lr_bin_table_hint: null pointer");
    *out = *(volatile int*)h->k1_hint;
    return LR_OK;
}

extern "C" int lr_bin_last_build(lr_handle_t h, int32_t* out) {
    LR_REQUIRE(h != nullptr && out != nullptr, "lr_bin_last_build: null pointer");
    *out = h->k1_last_build;
    return LR_OK;
}

extern "C" double lr_fe_ref_of_jitter(double death_jitter) { return death_jitter > 0.0 && death_jitter <= 1.0 ? death_jitter : 1.0; }

extern "C" int lr_bin_finalize(lr_handle_t h, const int64_t* d_acc, int32_t n_rep, int32_t n_bins, double fe_ref,
                               int64_t* d_sp, int64_t* d_ex, double* d_br, void* stream) {
    LR_REQUIRE(h != nullptr && d_acc && d_sp && d_ex && d_br, "lr_bin_finalize: null pointer");
    LR_REQUIRE(n_rep >= 1 && n_bins >= 1, "lr_bin_finalize: bad sizes");
    LR_REQUIRE(fe_ref > 0.0 && fe_ref <= 1.0, "lr_bin_finalize: fe_ref must lie in (0, 1]");
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    LR_CUDA(cudaSetDevice(h->device));
    k1_finalize_kernel<<<n_rep, 256, 0, st>>>((const long long*)d_acc, lr_acc_stride(n_bins), n_bins, fe_fix(fe_ref),
                                               (long long*)d_sp, (long long*)d_ex, d_br);
    LR_CUDA(cudaGetLastError());
    h->launches += 1;
    return LR_OK;
}

extern "C" int lr_bin_stats(lr_handle_t h, const double* d_ts, const double* d_te, int64_t n, int64_t ld,
                            int32_t n_rep, int64_t first_bin, int32_t n_bins, double fe_ref,
                            int32_t dead_only, double end_time,
                            int64_t* d_sp, int64_t* d_ex, double* d_br, void* stream) {
    LR_REQUIRE(h != nullptr, "lr_bin_stats: null handle");
    LR_REQUIRE(n_rep >= 1 && n_bins >= 1, "lr_bin_stats: bad sizes");
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    const size_t acc_bytes = (size_t)n_rep * LR_ACC_ROWS * lr_acc_stride(n_bins) * sizeof(int64_t);
    int rc = lr_ws_acquire(h, acc_bytes, st);
    if (rc != LR_OK) return rc;
    LR_CUDA(cudaMemsetAsync(h->ws, 0, acc_bytes, st));
    rc = lr_bin_accumulate(h, d_ts, d_te, n, ld, n_rep, first_bin, n_bins, fe_ref, dead_only, end_time, (int64_t*)h->ws, st);
    if (rc != LR_OK) return rc;
    return lr_bin_finalize(h, (const int64_t*)h->ws, n_rep, n_bins, fe_ref, d_sp, d_ex, d_br, st);
}
