// sm_100a kernels of the marginal-likelihood path.
//
//   geometry_tp/eb_kernel  one thread per prior draw: Kepler's-law semi-major axis, transit
//                          probability, collision and inclination masks (reference
//                          marginal_likelihoods.py:107-123 for TP-type, :254-299 for EB-type),
//                          and compaction of the surviving draws into a work list.
//   lnl_kernel             persistent warps; one warp per surviving draw.  The lanes sweep the
//                          time stamps inside the draw's transit window, each lane averaging its
//                          own sub-exposures; a shuffle tree reduces chi^2.  Points outside the
//                          window have model == 1 exactly and are added from a prefix sum of
//                          (flux-1)^2.  EB-type draws first evaluate the 25-point secondary
//                          eclipse (one point per lane) and its depth cut
//                          (likelihoods.py:417-438, :535-538).
//   lse_partial/final      log-mean-exp of lnL + lnprior as per-thread running (max, scaled sum)
//                          pairs merged per block and then across blocks (_numerics.py:12-51).
//
// FP64 CUDA-core work throughout: the path is not a contraction, so no tensor cores.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "tri_model.cuh"

namespace tri {

// pointer + stride (0 = one value broadcast to every sample, 1 = per-sample array)
struct Col {
    const double* p;
    int64_t stride;
    __device__ __forceinline__ double at(int64_t i) const { return __ldg(p + i * stride); }
};

// ---- geometry ------------------------------------------------------------------------------
struct GeomTp {
    int64_t N;
    Col rp, P, inc, ecc, argp, mtot, rhost;
    const uint8_t* extra_mask;  // optional AND term (qs_comp != 0, logg/Teff cuts)
    double* a_out;              // [N] semi-major axis [cm] of surviving draws
    double* lnl_out;            // [N] pre-filled with -inf for the rejected draws
    uint8_t* mask_out;          // optional [N]
    int64_t* items;             // work list (sample index << 1), capacity N: long items are
                                // appended from the front, short ones from the back
    unsigned long long* n_items;  // [0] items at the front, [3] items at the back
};

struct GeomEb {
    int64_t N;
    Col reb, q, P, inc, ecc, argp, mtot, rhost;
    const uint8_t* extra_mask;
    int scalar_loop;    // parallel=False loop: Ptra(P) > 1 skips the twin branch too
    double* a_out;      // a (q < 0.95) or a_twin (q >= 0.95) of surviving draws
    double* p_out;      // P or 2P
    double* lnl_out;    // [N] EB branch, -inf default
    double* lnl_twin_out;  // [N] twin branch, -inf default
    uint8_t* mask_out;       // optional [N]: mask of the EB branch
    uint8_t* mask_twin_out;  // optional [N]: mask of the twin branch
    int64_t* items;     // (sample index << 1) | twin; front / back as in GeomTp
    unsigned long long* n_items;  // [0] items at the front, [1] twins, [3] items at the back
};

__device__ __forceinline__ double neg_inf() { return -INFINITY; }

// a = ((G*M*Msun)/(4*pi**2)*(P*86400)**2)**(1/3)        marginal_likelihoods.py:75
__device__ __forceinline__ double semi_major_axis(double mtot, double P) {
    double ps = P * 86400.0;
    return pow((kG * mtot * kMsun) / (4.0 * (kPi * kPi)) * (ps * ps), 1.0 / 3.0);
}

// inc_min = arccos(Ptra)*180/pi where Ptra <= 1 else 90          marginal_likelihoods.py:120-121
__device__ __forceinline__ bool transits(double inc_deg, double Ptra) {
    double inc_min = 90.0;
    if (Ptra <= 1.0) inc_min = acos(Ptra) * 180.0 / kPi;
    return inc_deg >= inc_min;
}

// A draw whose chord is short (cos i > 0.92 Ptra, i.e. impact parameter above 0.92 (1 + k):
// at most 40 % of the central transit duration) is cheap to evaluate.  Such draws go to the back
// of the work list and are handed out last, so that the warps that finish the launch are busy
// with short items and the tail of the persistent kernel is short (longest-first scheduling
// with two classes; the result does not depend on the order).
__device__ __forceinline__ bool short_chord(double inc_deg, double Ptra) {
    return Ptra <= 1.0 && cos(inc_deg * (kPi / 180.0)) > 0.92 * Ptra;
}

__device__ __forceinline__ void push_one(unsigned ballot, bool mine, int64_t item, int64_t* slot0,
                                         int dir, unsigned long long* counter) {
    if (ballot == 0) return;
    int lane = threadIdx.x & 31;
    int leader = __ffs(ballot) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(counter, (unsigned long long)__popc(ballot));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (mine) {
        long long off = (long long)(base + __popc(ballot & ((1u << lane) - 1u)));
        slot0[dir * off] = item;
    }
}

__device__ __forceinline__ void push_item(bool take, bool is_short, int64_t item, int64_t* items,
                                          int64_t cap, unsigned long long* n_items) {
    const unsigned front = __ballot_sync(0xffffffffu, take && !is_short);
    const unsigned back = __ballot_sync(0xffffffffu, take && is_short);
    push_one(front, take && !is_short, item, items, +1, n_items + 0);
    push_one(back, take && is_short, item, items + (cap - 1), -1, n_items + 3);
}

__global__ void geometry_tp_kernel(GeomTp g) {
    int64_t n_round = (g.N + 31) / 32 * 32;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_round;
         i += (int64_t)gridDim.x * blockDim.x) {
        bool take = false, brief = false;
        if (i < g.N) {
            double rp = g.rp.at(i), P = g.P.at(i), inc = g.inc.at(i), ecc = g.ecc.at(i);
            double argp = g.argp.at(i), rhost = g.rhost.at(i);
            double a = semi_major_axis(g.mtot.at(i), P);
            // e_corr, Ptra, coll                      marginal_likelihoods.py:111-115
            double e_corr = (1.0 + ecc * sin(argp * kPi / 180.0)) / (1.0 - ecc * ecc);
            double rsum = rp * kRearth + rhost * kRsun;
            double Ptra = rsum / a * e_corr;
            bool coll = rsum > a * (1.0 - ecc);
            take = transits(inc, Ptra) && !coll;
            if (g.extra_mask) take = take && (g.extra_mask[i] != 0);
            g.lnl_out[i] = neg_inf();
            if (take) {
                g.a_out[i] = a;
                brief = short_chord(inc, Ptra);
            }
            if (g.mask_out) g.mask_out[i] = take ? 1 : 0;
        }
        push_item(take, brief, i << 1, g.items, g.N, g.n_items);
    }
}

__global__ void geometry_eb_kernel(GeomEb g) {
    int64_t n_round = (g.N + 31) / 32 * 32;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_round;
         i += (int64_t)gridDim.x * blockDim.x) {
        bool take = false, brief = false;
        int twin = 0;
        if (i < g.N) {
            double reb = g.reb.at(i), q = g.q.at(i), P = g.P.at(i), inc = g.inc.at(i);
            double ecc = g.ecc.at(i), argp = g.argp.at(i), rhost = g.rhost.at(i);
            double mtot = g.mtot.at(i);
            // marginal_likelihoods.py:254-268
            double e_corr = (1.0 + ecc * sin(argp * kPi / 180.0)) / (1.0 - ecc * ecc);
            double rsum = reb * kRsun + rhost * kRsun;
            twin = (q >= 0.95) ? 1 : 0;
            double a, Ptra;
            bool coll;
            if (!twin) {
                a = semi_major_axis(mtot, P);
                Ptra = rsum / a * e_corr;
                coll = rsum > a * (1.0 - ecc);
            } else {
                a = semi_major_axis(mtot, 2.0 * P);
                Ptra = rsum / a * e_corr;
                coll = (2.0 * rhost * kRsun) > a * (1.0 - ecc);
            }
            take = transits(inc, Ptra) && !coll;
            // marginal_likelihoods.py:316-319: the scalar loop `continue`s before it reaches the
            // twin branch when the period-P transit probability exceeds 1
            if (twin && g.scalar_loop && !(rsum / semi_major_axis(mtot, P) * e_corr <= 1.0))
                take = false;
            if (g.extra_mask) take = take && (g.extra_mask[i] != 0);
            g.lnl_out[i] = neg_inf();
            g.lnl_twin_out[i] = neg_inf();
            if (take) {
                g.a_out[i] = a;
                g.p_out[i] = twin ? 2.0 * P : P;
                brief = short_chord(inc, Ptra);
            }
            if (g.mask_out) g.mask_out[i] = (take && !twin) ? 1 : 0;
            if (g.mask_twin_out) g.mask_twin_out[i] = (take && twin) ? 1 : 0;
        }
        push_item(take, brief, (i << 1) | twin, g.items, g.N, g.n_items);
        unsigned bt = __ballot_sync(0xffffffffu, take && twin);
        if ((threadIdx.x & 31) == 0 && bt) atomicAdd(g.n_items + 1, (unsigned long long)__popc(bt));
    }
}

// ---- log-mean-exp pieces (used by the light-curve kernel's epilogue) ---------------------------
struct LsePartial {
    double m;      // running max of the finite entries (-inf if none)
    double s;      // sum of exp(x - m)
    unsigned long long n_finite, n_posinf;
};

__device__ __forceinline__ void lse_push(LsePartial& a, double x) {
    if (isinf(x) && x > 0) { a.n_posinf++; return; }
    if (!isfinite(x)) return;  // -inf and NaN: zero weight
    a.n_finite++;
    if (x > a.m) {
        a.s = a.s * exp(a.m - x) + 1.0;   // exp(-inf) = 0 on the first finite entry
        a.m = x;
    } else {
        a.s += exp(x - a.m);
    }
}

__device__ __forceinline__ void lse_merge(LsePartial& a, const LsePartial& b) {
    a.n_finite += b.n_finite;
    a.n_posinf += b.n_posinf;
    if (b.m == -INFINITY) return;
    if (a.m == -INFINITY) { a.m = b.m; a.s = b.s; return; }
    if (b.m > a.m) {
        a.s = a.s * exp(a.m - b.m) + b.s;
        a.m = b.m;
    } else {
        a.s += b.s * exp(b.m - a.m);
    }
}

// order-preserving integer image of a double: larger double -> larger key
__device__ __forceinline__ unsigned long long topk_key(double x) {
    unsigned long long u = (unsigned long long)__double_as_longlong(x);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

constexpr int kTopkBins = 1 << 16;   // histogram over the leading 16 key bits (sign, exponent,
                                     // four mantissa bits), filled by the light-curve kernel

// ---- light curve + chi^2 ---------------------------------------------------------------------
// Mixed cadence (tri_set_lightcurve_cadence): the stamps are sorted by (group, time) and group g
// owns the sorted stamps [off[g], off[g+1]) of the one light curve (one prefix-sum array over
// the concatenation).  Read by lnl_kernel<*, true> only; with one cadence the table is unused.
constexpr int kMaxCadences = 8;   // TRI_MAX_CADENCES
struct CadenceTable {
    int n;                           // groups
    int off[kMaxCadences + 1];
    int nsamples[kMaxCadences];
    double exptime[kMaxCadences];
    double tmin[kMaxCadences], tmax[kMaxCadences];   // first and last stamp of the group
};

struct LnlArgs {
    LightCurve lc;
    OrbitTable tab;
    int eb;                  // 0 TP-type, 1 EB-type
    int companion_is_host;
    int raw;                 // 1: store +0.5 chi^2 (the lnL_*_p seam), +inf on the depth cut
                             // 0: store -0.5 ln(2 pi) - ln(sigma) - 0.5 chi^2 (marginal_likelihoods.py:130)
    int twin_uniform;        // twin flag when items == nullptr
    Col body;                // R_p [R_earth] (TP) or R_EB [R_sun] (EB)
    Col ebfr;                // EB flux ratio (EB only)
    Col P, inc, a, rhost, u1, u2, ecc, argp, cfr;
    const int64_t* items;    // nullptr: identity list 0..count-1
    int64_t count;             // number of work items when count_dev == nullptr
    const unsigned long long* count_dev;  // else read from device memory (written by geometry):
                                          // count_dev[0] items at the front of `items`,
                                          // count_dev[3] at the back (handed out last)
    int64_t items_cap;         // capacity of `items` (the back grows down from items_cap - 1)
    unsigned long long* next;  // work-queue cursor
    double* out;             // lnL of the (EB) branch, indexed by sample
    double* out_twin;        // lnL of the twin branch (fused EB only)
    unsigned long long* counters;  // optional [4]: stamps inside transit windows, stamps whose
                                   // sub-exposures were evaluated (window minus centre-probe
                                   // skips), interior-case points, limb/edge-case points
    // fused evidence epilogue (marginal_likelihoods.py:154 / :568, _numerics.py:12-51): every warp
    // keeps a running (max, scaled sum) of lnL + lnprior over the draws it evaluates, the block
    // merges its warps and writes one record per branch; finalize_kernel merges the blocks
    Col lnprior;             // ptr nullptr: none
    LsePartial* lse_partials;  // nullptr: off; else [2][gridDim.x] (branch-major)
    double* cval;            // optional [items_cap]: lnL of work item `slot`, in the slot order of
                             // `items` (the dense input of the best-draw selection)
    unsigned int* hist16;    // optional [2][kTopkBins]: counts of finite lnL per leading key bits
    // simulate mode (simulate_TP_transit_p / simulate_EB_transit_p, likelihoods.py:302-439):
    double* model_out;       // optional [count][npts] diluted model flux, caller's stamp order
    double* secdepth_out;    // optional [count] secondary-eclipse depth (EB-type)
    const int* perm;         // sorted stamp j -> caller's stamp index
    int scalar_rule;         // 1: radius-ratio rules of the scalar simulate_EB_transit
                             // (likelihoods.py:121-123, :137) instead of the vectorised ones
    CadenceTable cad;        // cadence groups (lnl_kernel<*, true>); lc.exptime is then the largest
                             // exposure of the groups, which transit_window's image check uses
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// One warp per block: the per-draw record of the warp then sits at compile-time constant
// shared-memory addresses.  32 resident blocks per SM = 64 registers per thread (A/B on B200,
// ms per step of the headline workload: 128 threads x 6 blocks: 166.7, 32 x 24: 165.6,
// 32 x 28: 163.8, 32 x 32: 163.8 -- the kernel is bound by the issue port, not by the number
// of warps, see DESIGN.md).
#ifndef TRI_LNL_THREADS
#define TRI_LNL_THREADS 32
#endif
constexpr int kLnlThreads = TRI_LNL_THREADS;
constexpr int kLnlWarps = kLnlThreads / 32;
#ifndef TRI_LNL_MIN_BLOCKS
#define TRI_LNL_MIN_BLOCKS (1024 / TRI_LNL_THREADS)
#endif
constexpr int kLnlMinBlocks = TRI_LNL_MIN_BLOCKS;

constexpr int kToffTable = 64;

// One draw's constants, ONE copy per warp in shared memory.  Every lane of the warp works on
// the same draw, so these values are warp-uniform; held in registers they cost 32 copies and
// (at 6 resident blocks per SM) ~45 doubles of local-memory spills per thread.  The hot loop
// reads them through a volatile reference: one LDS broadcast per use, on the load/store pipe,
// which the FP64-bound loop leaves idle.
struct WarpDraw {
    Orbit o;
    Limb L;
    double skip_beyond;   // centre probe: |z| beyond which a whole exposure is out of transit
    double half_ma;       // half an exposure in mean anomaly (+ margin): n * exptime / 2
    double d1, d2;        // dilution (likelihoods.py:352-357 / :427-438)
    int two_stage;
};

struct LnlShared {
    WarpDraw draw[kLnlWarps];
    LsePartial lse[kLnlWarps][2];
    unsigned long long cnt[kLnlWarps][4];   // diagnostic counters of the warp
    double toff[kLnlWarps][kToffTable];   // sub-exposure offsets: row 0 for the whole block
                                          // with one cadence, else the warp's current group
    const double* time;
    const double* flux;
    const double* prefix;
    double lnorm;
};

// Per-draw state of the segmented instantiation: the transit window, found once and used by
// every cadence group, the current group's stamps, and the sums over the groups.
struct SegDraw {
    double red = 0.0;       // per lane: chi^2 of the groups' window stamps
    double pre_chi = 0.0;   // chi^2 of the groups' stamps outside the window
    bool have_win = false;
    double t_lo = 0.0, t_hi = 0.0, speed = 0.0;   // the window, max_projected_speed
    int n_win = 0;          // the groups' window stamps
    int g0, g1;             // the current group's stamps [g0, g1)
};

// kCount: also count the work classes of SURVEY.md 8(d) (window stamps, evaluated stamps,
// interior and limb points) into A.counters -- the roofline accounting of bench.py and the
// n_stamps / n_interior / n_limb diagnostics; the production instantiation leaves them out of
// the hot loop.
// kSeg: the light curve has several cadence groups (A.cad).  Per draw the orbit, limb and
// dilution set-up, the transit window and (EB-type) the secondary pass run once, as with one
// cadence; then each group in turn takes its stamp range inside the window (its own half
// exposure), its own centre-probe radius and sub-exposure half-width in the warp's record, its
// own sub-exposure offsets in the warp's row of S.toff, the round loop with its own sample
// count, and the prefix terms of its stamps outside the window.  A compile-time switch, so that
// the single-cadence instantiation carries none of the per-group bookkeeping.  Where the two are
// written differently below for the same arithmetic (the pass index, where exptime is set, the
// per-pass reductions, the segmented state in one SegDraw), the single-cadence form is the one
// whose SASS is unchanged: which locals exist and where they are defined moves the compiler's
// register assignment (DESIGN.md section 4h).
template <bool kCount, bool kSeg>
__global__ void __launch_bounds__(kLnlThreads, kLnlMinBlocks) lnl_kernel(LnlArgs A) {
    extern __shared__ double smem[];
    __shared__ LnlShared S;
    if (A.lc.time == nullptr) return;
    const int npts = A.lc.npts;
    // Stage the folded light curve once per block when it fits (else read through L1/L2).
    {
        size_t need = (size_t)(3 * npts + 1) * sizeof(double);
        unsigned dyn;
        asm volatile("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn));
        if (need <= dyn) {
            double* st = smem;
            double* sf = smem + npts;
            double* sp = smem + 2 * npts;
            for (int j = threadIdx.x; j < npts; j += blockDim.x) {
                st[j] = A.lc.time[j];
                sf[j] = A.lc.flux[j];
            }
            for (int j = threadIdx.x; j <= npts; j += blockDim.x) sp[j] = A.lc.prefix[j];
            if (threadIdx.x == 0) { S.time = st; S.flux = sf; S.prefix = sp; }
        } else if (threadIdx.x == 0) {
            S.time = A.lc.time; S.flux = A.lc.flux; S.prefix = A.lc.prefix;
        }
    }
    // sub-exposure offsets of the observed light curve (the same for every draw) in row 0; with
    // cadence groups every warp fills its own row per group instead, and toff_tab follows the
    // group
    bool toff_tab = A.lc.nsamples < kToffTable;
    if (!kSeg && toff_tab) {
        const double inv = 1.0 / A.lc.nsamples;
        for (int is = threadIdx.x; is <= A.lc.nsamples; is += blockDim.x)
            S.toff[0][is] = is ? A.lc.exptime * ((is - 0.5) * inv - 0.5) : 0.0;
    }
    const int lane = threadIdx.x & 31;
    // (one warp per block: every shared-memory address is a compile-time constant)
    const int warp = kLnlWarps == 1 ? 0 : (int)(threadIdx.x >> 5);
    if (lane == 0) {
        S.lse[warp][0] = LsePartial{-INFINITY, 0.0, 0, 0};
        S.lse[warp][1] = LsePartial{-INFINITY, 0.0, 0, 0};
        for (int c = 0; c < 4; ++c) S.cnt[warp][c] = 0;
    }
    // the Gaussian constant, once per light curve (marginal_likelihoods.py:130)
    if (threadIdx.x == 0) S.lnorm = -0.5 * log(2.0 * kPi) - log(A.lc.sigma);
    __syncthreads();
    WarpDraw& wd = S.draw[warp];
    const volatile WarpDraw& vd = S.draw[warp];
    const volatile LnlShared& VS = S;
    const int64_t n_front = A.count_dev ? (int64_t)A.count_dev[0] : A.count;
    const int64_t count = n_front + (A.count_dev ? (int64_t)A.count_dev[3] : 0);
    constexpr int kPass1 = kSeg ? 0 : 1;   // the first pass over the observed light curve

#pragma unroll 1
    for (;;) {
        unsigned long long w = 0;
        if (lane == 0) w = atomicAdd(A.next, 1ull);
        w = __shfl_sync(0xffffffffu, w, 0);
        if ((int64_t)w >= count) break;
        // slot of this work item in `items` (and in `cval`)
        const int64_t slot = ((int64_t)w < n_front) ? (int64_t)w
                                                    : A.items_cap - 1 - ((int64_t)w - n_front);
        const int64_t item = !A.items ? (((int64_t)w << 1) | A.twin_uniform) : A.items[slot];
        const int64_t i = item >> 1;
        const int twin = (int)(item & 1);

        // Passes through ONE copy of the model code: pass kPass1 - 1 (EB-type only) is the
        // 25-stamp secondary eclipse on [-0.05, 0.05] d with the roles swapped and no
        // supersampling (likelihoods.py:417-423), reduced with a minimum; pass kPass1 + g is
        // cadence group g of the observed light curve (the whole curve without kSeg), reduced to
        // chi^2.
        double chi = 0.0;
        SegDraw sg;   // kSeg only
        bool cut = false;
        int jlo = 0, jhi = 0;
        unsigned n_interior = 0, n_limb = 0;   // per lane, this draw
        unsigned n_skip = 0;                    // per lane: stamps the centre probe dismissed
#pragma unroll 1
        for (int pass = A.eb ? kPass1 - 1 : kPass1; pass < kPass1 + (kSeg ? A.cad.n : 1); ++pass) {
            const bool primary = pass >= kPass1;
            const int grp = pass - kPass1;
            const int ns = primary ? (kSeg ? A.cad.nsamples[grp] : A.lc.nsamples) : 1;
            // (one cadence: set with the per-sample constants below)
            double exptime = kSeg && primary ? A.cad.exptime[grp] : 0.0;
            if constexpr (kSeg) {
                sg.g0 = primary ? A.cad.off[grp] : 0;
                sg.g1 = primary ? A.cad.off[grp + 1] : 25;
            }
            bool probe;
            if (!kSeg || grp <= 0) {
                // ---- per-sample constants (every lane computes the same values); nothing of
                // this block stays in registers across the stamp loop.  The cadence groups
                // share them: with kSeg the block runs for the secondary and the first group.
                const double P = A.P.at(i), e = A.ecc.at(i), argp = A.argp.at(i);
                const double rhost = A.rhost.at(i);
                const double a_rs = A.a.at(i) / (rhost * kRsun);          // likelihoods.py:343 / :409
                const double inc = A.inc.at(i) * (kPi / 180.0);            // :344 / :410
                const double cfr = A.cfr.at(i);
                const double F_comp = cfr / (1.0 - cfr);
                double k_pri, k_sec = 0.0, d1, d2, F_EB;
                int two_stage;
                if (!A.eb) {
                    k_pri = A.body.at(i) * kRearth / (rhost * kRsun);      // :340
                    two_stage = 0;
                    d1 = 0.0;
                    d2 = A.companion_is_host ? 1.0 / F_comp : F_comp / 1.0;   // :352-357
                } else {
                    const double reb = A.body.at(i);
                    const double fr = A.ebfr.at(i);
                    F_EB = fr / (1.0 - fr);
                    k_pri = reb / rhost;
                    if (!A.scalar_rule) {
                        if ((k_pri - 1.0) < 1e-6) k_pri *= 0.999;          // :405-406 (no abs: every k <= 1)
                        k_sec = rhost / reb;                               // :417-418
                        if ((k_sec - 1.0) < 1e-6) k_sec *= 0.999;
                    } else {
                        if (fabs(k_pri - 1.0) < 1e-6) k_pri *= 0.999;      // :121-123
                        k_sec = 1.0 / k_pri;                               // :137
                    }
                    two_stage = 1;
                    if (A.companion_is_host) {                              // :427-432
                        d1 = F_EB / F_comp;
                        d2 = 1.0 / (F_comp + F_EB);
                    } else {                                                // :433-438
                        d1 = F_EB / 1.0;
                        d2 = F_comp / (1.0 + F_EB);
                    }
                }
                const double k = primary ? k_pri : k_sec;
                // w = (90 - argp) pi/180, + 180 deg for the secondary          :345 / :419
                const double w_rad = primary ? (90.0 - argp) * (kPi / 180.0)
                                             : (90.0 - argp + 180.0) * (kPi / 180.0);
                Orbit o;
                orbit_setup(o, A.tab, k, P, a_rs, inc, e, w_rad);
                Limb L;
                limb_setup(L, A.u1.at(i), A.u2.at(i), k);
                double skip_beyond;
                if constexpr (!kSeg) {
                    exptime = primary ? A.lc.exptime : 0.0;
                    if (primary) {
                        // time stamps that can be in transit
                        jlo = 0;
                        jhi = npts;
                        Window win;
                        if (transit_window(o, A.tab, a_rs, P, A.lc, win)) {
                            double half = 0.5 * A.lc.exptime;
                            const double* tp = VS.time;
                            jlo = lower_bound(tp, npts, win.t_lo - half);
                            jhi = lower_bound(tp, npts, win.t_hi + half);
                            if (jhi < jlo) jhi = jlo;
                        }
                    } else {
                        jlo = 0;
                        jhi = 25;
                    }
                    // centre probe (see max_projected_speed): only worth it with supersampling
                    probe = primary && ns > 1 && !o.table_clamped;
                    skip_beyond =
                        1.0 + k + max_projected_speed(o, a_rs) * (0.5 * exptime) + 1e-9;
                } else if (primary) {
                    // one window for every group: the image check uses the largest exposure
                    Window win;
                    sg.have_win = transit_window(o, A.tab, a_rs, P, A.lc, win);
                    sg.t_lo = win.t_lo;
                    sg.t_hi = win.t_hi;
                }
                if constexpr (kSeg) sg.speed = max_projected_speed(o, a_rs);
                __syncwarp();
                if (lane == 0) {
                    wd.o = o;
                    wd.L = L;
                    if constexpr (!kSeg) {
                        wd.skip_beyond = skip_beyond;
                        // table_clamped orbits (e >= 0.95) always take the generic path
                        wd.half_ma = o.table_clamped
                                         ? 1e30 : o.n_rate * (0.5 * exptime) * (1.0 + 1e-9) + 1e-12;
                    }
                    wd.d1 = d1;
                    wd.d2 = d2;
                    wd.two_stage = two_stage;
                }
                __syncwarp();
            }
            if constexpr (kSeg) {
                // ---- the group's stamp range, probe radius, sub-exposure half-width and offsets
                jlo = sg.g0;
                jhi = sg.g1;
                const double half = 0.5 * exptime;
                if (primary && sg.have_win) {
                    if (sg.t_hi + half < A.cad.tmin[grp] || sg.t_lo - half > A.cad.tmax[grp]) {
                        jhi = jlo;
                    } else {
                        const double* tp = VS.time;
                        jlo = sg.g0 + lower_bound(tp + sg.g0, sg.g1 - sg.g0, sg.t_lo - half);
                        jhi = sg.g0 + lower_bound(tp + sg.g0, sg.g1 - sg.g0, sg.t_hi + half);
                        if (jhi < jlo) jhi = jlo;
                    }
                }
                const bool clamped = vd.o.table_clamped;
                probe = primary && ns > 1 && !clamped;
                toff_tab = ns < kToffTable;
                __syncwarp();   // every lane is done with the previous group's record and offsets
                if (lane == 0) {
                    wd.skip_beyond = 1.0 + vd.o.k + sg.speed * half + 1e-9;
                    wd.half_ma = clamped ? 1e30 : vd.o.n_rate * half * (1.0 + 1e-9) + 1e-12;
                }
                if (primary && toff_tab) {
                    const double inv = 1.0 / ns;
                    for (int is = lane; is <= ns; is += 32)
                        S.toff[warp][is] = is ? exptime * ((is - 0.5) * inv - 0.5) : 0.0;
                }
                __syncwarp();
            }
            if (probe) {
                // Trim the window: stamps at its two ends whose whole exposure is out of transit
                // (centre probe) have model == 1 exactly and go to the prefix sums.  Lanes 0-15
                // walk in from the front, lanes 16-31 from the back, 16 stamps a side per step.
#pragma unroll 1
                for (;;) {
                    const bool back = lane >= 16;
                    const int j = back ? jhi - 1 - (lane - 16) : jlo + lane;
                    bool keep = false;
                    if (j >= jlo && j < jhi) {
                        const double* tp = VS.time;
                        keep = !(fabs(z_at(vd.o, A.tab, tp[j])) > vd.skip_beyond);
                    }
                    const unsigned b = __ballot_sync(0xffffffffu, keep);
                    const unsigned bf = b & 0xffffu, bb = b >> 16;
                    jlo += bf ? (__ffs(bf) - 1) : 16;
                    jhi -= bb ? (__ffs(bb) - 1) : 16;
                    if (jlo >= jhi) {
                        jhi = jlo = (jlo < (kSeg ? sg.g1 : npts) ? jlo : (kSeg ? sg.g1 : npts));
                        break;
                    }
                    if (bf && bb) break;
                }
            }
            if (primary && A.model_out) {   // outside the window the model is exactly 1
                double* row = A.model_out + (size_t)w * npts;
                for (int j = (kSeg ? sg.g0 : 0) + lane; j < (kSeg ? sg.g1 : npts); j += 32)
                    if (j < jlo || j >= jhi) row[A.perm[j]] = 1.0;
            }
            // per lane: the pass's chi^2 (with kSeg sg.red, which runs on over the groups) or, on
            // the secondary pass, its minimum
            double red = primary && !kSeg ? 0.0 : INFINITY;
            // lane <-> time stamp, serial over sub-exposures.  Full rounds take 16 stamps from
            // the front of the window and 16 from its back: ingress and egress mirror each
            // other, so the two halves of the warp are in the same occultation case (limb or
            // interior) at the same time instead of one half waiting for the other.  The
            // remainder (< 32 stamps, in the middle) forms the last round, where 2 (<= 16 stamps)
            // or 4 (<= 8) lanes share one stamp's sub-exposures.
            const int n_full = (jhi - jlo) >> 5;
            const int rem = (jhi - jlo) - 32 * n_full;
#pragma unroll 1
            for (int r = 0; r < n_full + (rem > 0 ? 1 : 0); ++r) {
                int gsh = 0, j, sub = 0;
                bool have = true;
                bool mirror = false;
                if (r < n_full) {
                    mirror = lane >= 16;
                    j = mirror ? jhi - 16 * r - 1 - (lane - 16) : jlo + 16 * r + lane;
                } else {
                    gsh = (primary && ns >= 4) ? (rem <= 8 ? 2 : (rem <= 16 ? 1 : 0)) : 0;
                    j = jlo + 16 * n_full + (lane >> gsh);
                    sub = lane & ((1 << gsh) - 1);
                    have = (lane >> gsh) < rem;
                }
                double acc = 0.0;
                if (have) {
                    double t;
                    if (primary) {
                        const double* tp = VS.time;
                        t = tp[j];
                    } else {
                        t = (j == 24) ? 0.05 : -0.05 + j * ((0.05 - -0.05) / 24.0);
                    }
                    // this lane's sub-exposures: is_lo .. is_hi of 1 .. ns
                    const int is_lo = 1 + ((sub * ns) >> gsh), is_hi = ((sub + 1) * ns) >> gsh;
                    // the centre of the exposure: generic orbit evaluation; the sub-exposures
                    // are expanded around it (tri_model.cuh, z_sub)
                    StampOrbit so;
                    bool fast;
                    const double zc = stamp_centre(vd.o, A.tab, t, vd.half_ma, so, fast);
                    if (probe && fabs(zc) > vd.skip_beyond) {
                        // the whole exposure is out of transit: model == 1
                        acc = (double)(is_hi - is_lo + 1);
                        if (kCount) n_skip += (sub == 0);
                    } else {
#pragma unroll 1
                        for (int is = is_lo; is <= is_hi; ++is) {
                            // sub-exposure offset exptime ((is - 1/2)/ns - 1/2), tabulated per
                            // block (kSeg: per warp and group; the back half of a paired round
                            // runs its sub-exposures backwards in time, the mirror image of the
                            // front half)
                            const int iso = mirror ? ns + 1 - is : is;
                            double toff = 0.0;
                            if (primary)
                                toff = toff_tab ? S.toff[kSeg ? warp : 0][iso]
                                                : exptime * ((iso - 0.5) / ns - 0.5);
                            const double z = fast ? z_sub(vd.o, A.tab, so, toff)
                                                  : z_at(vd.o, A.tab, t + toff);
                            int cls = 0;   // work class of SURVEY.md 8(d): 1 interior, 2 limb-crossing
                            const double k = vd.o.k;
                            acc += (z > 1.0 + k) ? 1.0 : occult_quad(z, k, vd.L, cls);
                            if (kCount) {
                                n_interior += (unsigned)(primary && cls == 1);
                                n_limb += (unsigned)(primary && cls == 2);
                            }
                        }
                    }
                }
                if (gsh) {   // (warp-uniform) the lanes of a stamp pool their sub-exposure sums
                    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
                    if (gsh == 2) acc += __shfl_xor_sync(0xffffffffu, acc, 2);
                }
                if (have && sub == 0) {
                    double m = acc / ns;
                    if (primary) {
                        if (vd.two_stage) m = (m + vd.d1) / (1.0 + vd.d1);
                        const double d2 = vd.d2;
                        const double md = (m + d2) / (1.0 + d2);
                        if (A.model_out) A.model_out[(size_t)w * npts + A.perm[j]] = md;
                        const double* fp = VS.flux;
                        const double rr = fp[j] - md;
                        double& sum = kSeg ? sg.red : red;
                        sum = fma(A.lc.weight ? rr * __ldg(A.lc.weight + j) : rr, rr, sum);
                    } else {
                        red = fmin(red, m);
                    }
                }
            }
            if (!primary) {
                double sec = warp_min(red);
                const double cfr = A.cfr.at(i), fr = A.ebfr.at(i);
                const double F_comp = cfr / (1.0 - cfr), F_EB = fr / (1.0 - fr);
                if (A.companion_is_host) sec = (sec + F_comp / F_EB) / (1.0 + F_comp / F_EB);
                else sec = (sec + 1.0 / F_EB) / (1.0 + 1.0 / F_EB);
                const double d2 = vd.d2;
                const double sd = 1.0 - (sec + d2) / (1.0 + d2);
                if (A.secdepth_out && lane == 0) A.secdepth_out[w] = sd;
                cut = !twin && !(sd < 1.5 * A.lc.sigma);                 // :535-538
                if (cut) break;
            } else if constexpr (kSeg) {
                const double* pre = VS.prefix;
                sg.pre_chi += (pre[jlo] - pre[sg.g0]) + (pre[sg.g1] - pre[jhi]);
                sg.n_win += jhi - jlo;
            } else {
                chi = warp_sum(red);
            }
        }
        double* outp = (twin && A.out_twin) ? A.out_twin : A.out;
        double val;
        if (cut) {
            val = A.raw ? INFINITY : -INFINITY;
        } else {
            if constexpr (kSeg) {
                chi = warp_sum(sg.red) + sg.pre_chi;
            } else {
                const double* pre = VS.prefix;
                chi += (pre[jlo] - pre[0]) + (pre[npts] - pre[jhi]);
            }
            const double sigma = A.lc.sigma;
            const double half_chi2 = A.lc.weight ? 0.5 * chi              // weights carry 1/sigma_j^2
                                                 : 0.5 * (chi / (sigma * sigma));   // likelihoods.py:486
            val = A.raw ? half_chi2 : S.lnorm - half_chi2;
        }
        if (kCount && A.counters) {
            unsigned long long c_skip = n_skip, c_int = n_interior, c_limb = n_limb;
            for (int o = 16; o > 0; o >>= 1) {
                c_skip += __shfl_xor_sync(0xffffffffu, c_skip, o);
                c_int += __shfl_xor_sync(0xffffffffu, c_int, o);
                c_limb += __shfl_xor_sync(0xffffffffu, c_limb, o);
            }
            if (lane == 0 && !cut) {
                S.cnt[warp][0] += (unsigned long long)(kSeg ? sg.n_win : jhi - jlo);
                S.cnt[warp][1] += (unsigned long long)(kSeg ? sg.n_win : jhi - jlo) - c_skip;
                S.cnt[warp][2] += c_int;
                S.cnt[warp][3] += c_limb;
            }
        }
        if (lane == 0) {
            outp[i] = val;
            if (A.cval) A.cval[slot] = val;
            if (A.lse_partials) {
                // the evidence epilogue: ln-weight = lnL + lnprior of this draw
                double x = val;
                if (A.lnprior.p) x += A.lnprior.at(i);
                lse_push(S.lse[warp][twin], x);
                if (A.hist16 && isfinite(val))
                    atomicAdd(A.hist16 + twin * kTopkBins + (int)(topk_key(val) >> 48), 1u);
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (A.lse_partials) {
            for (int b = 0; b < 2; ++b) {
                LsePartial a = S.lse[0][b];
                for (int wv = 1; wv < kLnlWarps; ++wv) lse_merge(a, S.lse[wv][b]);
                A.lse_partials[(size_t)b * gridDim.x + blockIdx.x] = a;
            }
        }
        if (kCount && A.counters) {
            for (int c = 0; c < 4; ++c) {
                unsigned long long v = 0;
                for (int wv = 0; wv < kLnlWarps; ++wv) v += S.cnt[wv][c];
                if (v) atomicAdd(A.counters + c, v);
            }
        }
    }
}

// ---- evidence + best draws: one block per scenario branch --------------------------------------
// (1) merges the per-block (max, scaled-sum) records of lnl_kernel in block order;
// (2) selects the best draws (reference marginal_likelihoods.py:152-153: the head of
//     (-lnL).argsort()) among the work items of the call.  The order is that of a stable sort
//     by (-lnL, index): a radix select on the composite (key of lnL, complemented index), which
//     has no ties.  The first two digits come for free from the 16-bit histogram lnl_kernel
//     filled; one pass over the work items then appends everything above the K-th value's
//     bucket to the output and parks the bucket's own entries in shared memory, where the
//     remaining digits are resolved (in global memory when the bucket does not fit: many equal
//     values).  NaN and -inf never qualify.
struct TopkState {
    unsigned long long n_finite;       // finite entries
    unsigned long long n_out;          // entries written to the output
};

struct FinalizeArgs {
    const LsePartial* partials;   // [branches][n_partials]
    int n_partials;
    LsePartial* lse_out;          // [branches]
    const int64_t* items;         // (draw index << 1) | branch, dense at the front and at the back
    const double* cval;           // lnL per work item, same slots
    int64_t cap;                  // capacity of items / cval
    const unsigned long long* count_dev;   // [0] items at the front, [3] at the back
    unsigned int* hist16;         // [branches][kTopkBins]; left zeroed for the next call
    int64_t top_cap[2];
    int64_t* top_idx[2];
    double* top_val[2];
    TopkState* st;                // [branches]
};

constexpr int kFinThreads = 1024;
constexpr int kFinCand = 2048;     // bucket entries that fit in shared memory
constexpr int kIdxBits = 40;       // draw indices below 2^40

struct Composite {   // what the selection orders by: (key of lnL, complemented index), descending
    unsigned long long hi, lo;
};

__device__ __forceinline__ unsigned comp_digit(const Composite& c, int d) {
    // digits 0..7: key bytes from the top; 8..12: the 40 index bits
    return d < 8 ? (unsigned)((c.hi >> (56 - 8 * d)) & 0xffu)
                 : (unsigned)((c.lo >> (kIdxBits - 8 - 8 * (d - 8))) & 0xffu);
}

__device__ __forceinline__ bool comp_match(const Composite& c, const Composite& prefix,
                                           const Composite& mask) {
    return (c.hi & mask.hi) == prefix.hi && (c.lo & mask.lo) == prefix.lo;
}

__device__ __forceinline__ Composite make_comp(double v, int64_t idx) {
    return Composite{topk_key(v), (~(unsigned long long)idx) & ((1ull << kIdxBits) - 1ull)};
}

__global__ void __launch_bounds__(kFinThreads) finalize_kernel(FinalizeArgs F) {
    const int br = blockIdx.x;
    const int tid = threadIdx.x;
    __shared__ LsePartial sh_lse[kFinThreads / 32];
    __shared__ unsigned int hist[256];
    __shared__ unsigned long long sh_u64[kFinThreads / 32];
    __shared__ unsigned long long cand_hi[kFinCand];
    __shared__ unsigned long long cand_lo[kFinCand];
    __shared__ unsigned int sh_bucket, sh_ncand, sh_nout, sh_digit;
    __shared__ unsigned long long sh_above, sh_need, sh_nfinite;

    // ---- (1) evidence: merge the blocks' records in block order (fixed tree)
    {
        LsePartial a{-INFINITY, 0.0, 0, 0};
        const LsePartial* p = F.partials + (size_t)br * F.n_partials;
        // contiguous chunk per thread keeps the block order
        const int per = (F.n_partials + kFinThreads - 1) / kFinThreads;
        for (int q = tid * per; q < (tid + 1) * per && q < F.n_partials; ++q) lse_merge(a, p[q]);
        // warp tree, then warp 0 over the warps: lower lanes / warps first
        for (int o = 1; o < 32; o <<= 1) {
            LsePartial b;
            b.m = __shfl_down_sync(0xffffffffu, a.m, o);
            b.s = __shfl_down_sync(0xffffffffu, a.s, o);
            b.n_finite = __shfl_down_sync(0xffffffffu, a.n_finite, o);
            b.n_posinf = __shfl_down_sync(0xffffffffu, a.n_posinf, o);
            if ((tid & 31) + o < 32) lse_merge(a, b);
        }
        if ((tid & 31) == 0) sh_lse[tid >> 5] = a;
        __syncthreads();
        if (tid == 0) {
            LsePartial r = sh_lse[0];
            for (int wv = 1; wv < kFinThreads / 32; ++wv) lse_merge(r, sh_lse[wv]);
            F.lse_out[br] = r;
        }
    }

    // ---- (2) best draws
    unsigned int* h16 = F.hist16 + (size_t)br * kTopkBins;
    constexpr int kPer = kTopkBins / kFinThreads;   // bins per thread: [tid*kPer, (tid+1)*kPer)
    unsigned long long c_t = 0;
    {
        const uint4* h4 = reinterpret_cast<const uint4*>(h16 + tid * kPer);
#pragma unroll 4
        for (int q = 0; q < kPer / 4; ++q) {
            uint4 v = h4[q];
            c_t += (unsigned long long)v.x + v.y + v.z + v.w;
        }
    }
    // entries in higher bins than this thread's: suffix sums over lanes, then over warps
    unsigned long long suf = c_t;
    for (int o = 1; o < 32; o <<= 1) {
        unsigned long long v = __shfl_down_sync(0xffffffffu, suf, o);
        if ((tid & 31) + o < 32) suf += v;
    }
    if ((tid & 31) == 0) sh_u64[tid >> 5] = suf;   // total of the warp
    __syncthreads();
    unsigned long long above_t = suf - c_t;
    unsigned long long total = 0;
    for (int wv = 0; wv < kFinThreads / 32; ++wv) {
        if (wv > (tid >> 5)) above_t += sh_u64[wv];
        total += sh_u64[wv];
    }
    const unsigned long long K = total < (unsigned long long)(F.top_cap[br] > 0 ? F.top_cap[br] : 0)
                                     ? total : (unsigned long long)(F.top_cap[br] > 0 ? F.top_cap[br] : 0);
    if (tid == 0) { sh_nfinite = total; sh_ncand = 0; sh_nout = 0; sh_bucket = 0; sh_above = 0; sh_need = 0; }
    __syncthreads();
    if (K > 0 && above_t < K && K <= above_t + c_t) {   // exactly one thread
        unsigned long long above = above_t;
        for (int q = kPer - 1; q >= 0; --q) {
            const unsigned long long c = h16[tid * kPer + q];
            if (above + c >= K) {
                sh_bucket = (unsigned)(tid * kPer + q);
                sh_above = above;
                sh_need = K - above;
                break;
            }
            above += c;
        }
    }
    __syncthreads();
    {   // leave the histogram clean for the next call
        uint4* h4 = reinterpret_cast<uint4*>(h16 + tid * kPer);
#pragma unroll 4
        for (int q = 0; q < kPer / 4; ++q) h4[q] = make_uint4(0u, 0u, 0u, 0u);
    }
    if (K == 0) {
        if (tid == 0) { F.st[br].n_finite = sh_nfinite; F.st[br].n_out = 0; }
        return;
    }
    const unsigned bucket = sh_bucket;
    const unsigned long long need = sh_need;          // entries wanted from the bucket (>= 1)
    const int64_t n_front = (int64_t)F.count_dev[0], n_back = (int64_t)F.count_dev[3];
    const int64_t n_items = n_front + n_back;
    int64_t* out_idx = F.top_idx[br];
    double* out_val = F.top_val[br];
    const int64_t top_cap = F.top_cap[br];
    const bool two = gridDim.x > 1;
    // one pass over the work items: above the bucket -> output; in the bucket -> candidates
    // (four independent loads in flight per thread: the pass is L2-latency bound)
    for (int64_t base = tid; base < n_items; base += 4 * kFinThreads) {
        int64_t item[4];
        double val[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t e = base + (int64_t)u * kFinThreads;
            item[u] = -1;
            val[u] = 0.0;
            if (e < n_items) {
                const int64_t slot = e < n_front ? e : F.cap - 1 - (e - n_front);
                item[u] = F.items[slot];
                val[u] = F.cval[slot];
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (item[u] < 0) continue;
            if (two && (int)(item[u] & 1) != br) continue;
            const double v = val[u];
            if (!isfinite(v)) continue;
            const unsigned bin = (unsigned)(topk_key(v) >> 48);
            if (bin > bucket) {
                unsigned pos = atomicAdd(&sh_nout, 1u);
                if ((int64_t)pos < top_cap) { out_idx[pos] = item[u] >> 1; out_val[pos] = v; }
            } else if (bin == bucket) {
                unsigned pos = atomicAdd(&sh_ncand, 1u);
                if (pos < (unsigned)kFinCand) {
                    Composite c = make_comp(v, item[u] >> 1);
                    cand_hi[pos] = c.hi;
                    cand_lo[pos] = c.lo;
                }
            }
        }
    }
    __syncthreads();
    const unsigned n_cand = sh_ncand;
    const bool in_smem = n_cand <= (unsigned)kFinCand;
    // radix select of the `need`-th largest composite among the bucket's entries: digits 2..12
    Composite prefix{(unsigned long long)bucket << 48, 0ull}, mask{0xffffull << 48, 0ull};
    unsigned long long k_rem = need;
    unsigned long long n_match = n_cand;     // entries matching the prefix so far
#pragma unroll 1
    for (int d = 2; d < 13 && n_match > k_rem; ++d) {
        if (tid < 256) hist[tid] = 0;
        __syncthreads();
        if (in_smem) {
            for (unsigned e = tid; e < n_cand; e += kFinThreads) {
                Composite c{cand_hi[e], cand_lo[e]};
                if (comp_match(c, prefix, mask)) atomicAdd(&hist[comp_digit(c, d)], 1u);
            }
        } else {
            for (int64_t e = tid; e < n_items; e += kFinThreads) {
                const int64_t slot = e < n_front ? e : F.cap - 1 - (e - n_front);
                const int64_t item = F.items[slot];
                if (two && (int)(item & 1) != br) continue;
                const double v = F.cval[slot];
                if (!isfinite(v)) continue;
                Composite c = make_comp(v, item >> 1);
                if (comp_match(c, prefix, mask)) atomicAdd(&hist[comp_digit(c, d)], 1u);
            }
        }
        __syncthreads();
        if (tid == 0) {
            unsigned long long above = 0;
            unsigned dg = 0, cnt = 0;
            for (int b = 255; b >= 0; --b) {
                cnt = hist[b];
                if (above + cnt >= k_rem && cnt > 0) { dg = (unsigned)b; break; }
                above += cnt;
            }
            sh_digit = dg;
            sh_above = above;
            sh_need = cnt;
        }
        __syncthreads();
        const unsigned dg = sh_digit;
        if (d < 8) {
            prefix.hi |= (unsigned long long)dg << (56 - 8 * d);
            mask.hi |= 0xffull << (56 - 8 * d);
        } else {
            prefix.lo |= (unsigned long long)dg << (kIdxBits - 8 - 8 * (d - 8));
            mask.lo |= 0xffull << (kIdxBits - 8 - 8 * (d - 8));
        }
        k_rem -= sh_above;
        n_match = sh_need;
        __syncthreads();
    }
    // every entry matching (prefix, mask) is wanted now (n_match <= k_rem; composites are
    // distinct, so the digits run out with n_match == k_rem == 1 at the latest), plus the
    // bucket's entries above it
    auto wanted = [&](const Composite& c) {
        if ((c.hi & mask.hi) != prefix.hi) return (c.hi & mask.hi) > prefix.hi;
        if ((c.lo & mask.lo) != prefix.lo) return (c.lo & mask.lo) > prefix.lo;
        return true;
    };
    if (in_smem) {
        for (unsigned e = tid; e < n_cand; e += kFinThreads) {
            Composite c{cand_hi[e], cand_lo[e]};
            if (!wanted(c)) continue;
            unsigned pos = atomicAdd(&sh_nout, 1u);
            if ((int64_t)pos >= top_cap) continue;
            unsigned long long u = c.hi;
            u = (u >> 63) ? (u & 0x7fffffffffffffffull) : ~u;   // inverse of topk_key
            out_idx[pos] = (int64_t)((~c.lo) & ((1ull << kIdxBits) - 1ull));
            out_val[pos] = __longlong_as_double((long long)u);
        }
    } else {
        for (int64_t e = tid; e < n_items; e += kFinThreads) {
            const int64_t slot = e < n_front ? e : F.cap - 1 - (e - n_front);
            const int64_t item = F.items[slot];
            if (two && (int)(item & 1) != br) continue;
            const double v = F.cval[slot];
            if (!isfinite(v)) continue;
            Composite c = make_comp(v, item >> 1);
            if ((unsigned)(c.hi >> 48) != bucket || !wanted(c)) continue;
            unsigned pos = atomicAdd(&sh_nout, 1u);
            if ((int64_t)pos < top_cap) { out_idx[pos] = item >> 1; out_val[pos] = v; }
        }
    }
    __syncthreads();
    if (tid == 0) {
        F.st[br].n_finite = sh_nfinite;
        F.st[br].n_out = sh_nout < (unsigned long long)top_cap ? sh_nout : (unsigned long long)top_cap;
    }
}

// ---- second moment of the weights (tri_set_moments) ---------------------------------------------
// s2[b] = sum over the finite ln-weights x of branch b of exp(2 (x - m_b)), with m_b the branch's
// maximum from finalize_kernel and x formed exactly as lnl_kernel's epilogue forms it (lnL +
// lnprior), so that every term is <= 1.  Reads the per-draw lnL arrays in draw order: block k
// sums a contiguous range, the last block to finish merges the block sums in block order, so the
// result does not depend on scheduling.
constexpr int kMomThreads = 256;

struct MomentsArgs {
    const double* lnl[2];         // per-draw lnL of branch 0 / 1 (-inf where not evaluated)
    Col lnprior;                  // ptr nullptr: none
    int64_t N;
    int branches;
    const LsePartial* lse;        // [branches] evidence records of finalize_kernel
    double* partials;             // [2][gridDim.x]
    unsigned int* done;           // block counter, 0 between launches
    double* s2_out;               // [branches]
};

__device__ __forceinline__ double block_sum_mom(double v, double* sh) {
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = kMomThreads / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    double r = sh[0];
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(kMomThreads) moments_kernel(MomentsArgs M) {
    __shared__ double sh[kMomThreads];
    __shared__ bool last;
    const int64_t per = (M.N + gridDim.x - 1) / gridDim.x;
    const int64_t lo = (int64_t)blockIdx.x * per;
    const int64_t hi = lo + per < M.N ? lo + per : M.N;
    for (int b = 0; b < M.branches; ++b) {
        const double m = M.lse[b].m;
        const double* lnl = b ? M.lnl[1] : M.lnl[0];   // (constant indices: no stack copy)
        double acc = 0.0;
        if (isfinite(m)) {
            for (int64_t i = lo + threadIdx.x; i < hi; i += kMomThreads) {
                double x = lnl[i];
                if (M.lnprior.p) x += M.lnprior.at(i);
                if (isfinite(x)) {
                    const double t = exp(x - m);
                    acc += t * t;
                }
            }
        }
        acc = block_sum_mom(acc, sh);
        if (threadIdx.x == 0) M.partials[(size_t)b * gridDim.x + blockIdx.x] = acc;
    }
    __threadfence();
    if (threadIdx.x == 0) last = atomicAdd(M.done, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    const int nb = (int)gridDim.x;
    const int chunk = (nb + kMomThreads - 1) / kMomThreads;
    for (int b = 0; b < M.branches; ++b) {
        double acc = 0.0;
        for (int q = threadIdx.x * chunk; q < (int)(threadIdx.x + 1) * chunk && q < nb; ++q)
            acc += __ldcg(M.partials + (size_t)b * nb + q);
        acc = block_sum_mom(acc, sh);
        if (threadIdx.x == 0) M.s2_out[b] = acc;
    }
    if (threadIdx.x == 0) *M.done = 0u;
}

// ---- posterior samples: systematic importance resampling (tri_set_posterior) -------------------
// Weights w_i = exp(x_i - m) with x_i = lnL_i + lnprior_i formed as lnl_kernel's epilogue forms it
// and m the branch's maximum from finalize_kernel (0 where x_i is not finite).  C_i is the
// inclusive prefix sum of w in draw order, T = C_{N-1}, u_k = (U + k) * (T / K) for k < K, and
// sample k is draw min{i : C_i > u_k}; positions at or above T go to the last draw at which C
// increases (the last draw of positive weight, unless rounding absorbed its weight).
//
// The draws are cut into tiles of kPostTile = 256 threads x 16 contiguous draws, independent of
// the SM count.  Inside a tile every sum is a serial chain: over a thread's 16 draws, over the 32
// thread totals of a warp, over the 8 warp totals; posterior_sums_kernel chains the tile totals in
// tile order.  So the last prefix a thread computes is, bit for bit, the start the next thread
// (or tile) computes, and the intervals [C_{i-1}, C_i) tile [0, T) with neither gap nor overlap:
// posterior_select_kernel writes every idx[k] exactly once, without atomics.
constexpr int kPostThreads = 256;
constexpr int kPostPer = 16;
constexpr int64_t kPostTile = (int64_t)kPostThreads * kPostPer;

struct PosteriorArgs {
    const double* lnl[2];         // per-draw lnL of branch 0 / 1 (-inf where not evaluated)
    Col lnprior;                  // ptr nullptr: none
    int64_t N;
    int64_t tiles;                // ceil(N / kPostTile) = gridDim.x
    const LsePartial* lse;        // [branches] evidence records of finalize_kernel
    double* tile_sum;             // [2][tiles]
    double* tile_off;             // [2][tiles + 1]: exclusive offsets, then T
    unsigned int* done;           // [2] block counters, 0 between launches
    double* total;                // [branches] T (+inf: a weight is +inf; 0: none finite)
    int64_t* idx[2];              // [K] sample -> draw, per branch
    int64_t K;
    unsigned long long seed, stream;
};

__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// U in [0, 1): _numerics.posterior_uniform(seed, stream, salt), bit for bit
__device__ __forceinline__ double posterior_uniform(unsigned long long seed,
                                                    unsigned long long stream,
                                                    unsigned long long salt) {
    unsigned long long h = splitmix64(seed);
    h = splitmix64(h ^ stream);
    h = splitmix64(h ^ salt);
    return (double)(h >> 11) * 0x1.0p-53;
}

// This thread's 16 inclusive prefix sums l[] (serial, from 0) and its start in the tile,
// start = Wb + E (E: serial chain of the warp's earlier thread totals, Wb: of the block's earlier
// warp totals); the tile-local C of draw j is start-sum Wb + (E + l[j]).  Returns the tile total.
__device__ __forceinline__ double post_tile_scan(const PosteriorArgs& P, int b, int64_t tile,
                                                 double m, bool live, double (&l)[kPostPer],
                                                 double& wb, double& e, double* sh_warp) {
    const double* lnl = b ? P.lnl[1] : P.lnl[0];   // (constant indices: no stack copy)
    const int64_t base = tile * kPostTile + (int64_t)threadIdx.x * kPostPer;
    double acc = 0.0;
#pragma unroll
    for (int j = 0; j < kPostPer; ++j) {
        const int64_t i = base + j;
        double w = 0.0;
        if (live && i < P.N) {
            double x = lnl[i];
            if (P.lnprior.p) x += P.lnprior.at(i);
            if (isfinite(x)) w = exp(x - m);
        }
        acc += w;
        l[j] = acc;
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double chain = 0.0;
    e = 0.0;
    for (int q = 0; q < 32; ++q) {
        const double t = __shfl_sync(0xffffffffu, acc, q);
        if (q == lane) e = chain;
        chain += t;
    }
    if (lane == 0) sh_warp[warp] = chain;
    __syncthreads();
    double tot = 0.0;
    wb = 0.0;
    for (int q = 0; q < kPostThreads / 32; ++q) {
        if (q == warp) wb = tot;
        tot += sh_warp[q];
    }
    __syncthreads();
    return tot;
}

__device__ __forceinline__ bool post_empty(const LsePartial& r) {
    return r.n_posinf > 0 || r.n_finite == 0;
}

// grid (tiles, branches): tile totals; the last block of a branch chains them into the offsets
// and T, then resets its counter.  The block stages the totals in shared memory, 256 at a time,
// so that the serial chain of thread 0 does not wait on one L2 load per tile.
__global__ void __launch_bounds__(kPostThreads) posterior_sums_kernel(PosteriorArgs P) {
    __shared__ double sh_warp[kPostThreads / 32];
    __shared__ double sh_tot[kPostThreads];
    __shared__ bool last;
    const int b = blockIdx.y;
    const LsePartial r = P.lse[b];
    double l[kPostPer], wb, e;
    const double tot = post_tile_scan(P, b, blockIdx.x, r.m, !post_empty(r), l, wb, e, sh_warp);
    if (threadIdx.x == 0) P.tile_sum[(size_t)b * P.tiles + blockIdx.x] = tot;
    __threadfence();
    if (threadIdx.x == 0) last = atomicAdd(P.done + b, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;   // (uniform over the block)
    __threadfence();
    const double* ts = P.tile_sum + (size_t)b * P.tiles;
    double* off = P.tile_off + (size_t)b * (P.tiles + 1);
    double o = 0.0;   // (thread 0's)
    for (int64_t base = 0; base < P.tiles; base += kPostThreads) {
        const int64_t t = base + threadIdx.x;
        sh_tot[threadIdx.x] = t < P.tiles ? __ldcg(ts + t) : 0.0;
        __syncthreads();
        if (threadIdx.x == 0) {
            const int n = (int)(P.tiles - base < kPostThreads ? P.tiles - base : kPostThreads);
            for (int q = 0; q < n; ++q) {
                off[base + q] = o;
                o += sh_tot[q];
            }
        }
        __syncthreads();
    }
    if (threadIdx.x != 0) return;
    off[P.tiles] = o;
    P.total[b] = r.n_posinf > 0 ? INFINITY : r.n_finite == 0 ? 0.0 : o;
    P.done[b] = 0u;
}

// number of k in [0, K) with (U + k) * step < c (u_k is non-decreasing in k)
__device__ __forceinline__ int64_t post_count(double c, double U, double step, int64_t K) {
    const double g = floor(c / step - U);
    int64_t k = g > 0.0 ? (g < (double)K ? (int64_t)g : K) : 0;
    while (k < K && (U + (double)k) * step < c) ++k;
    while (k > 0 && (U + (double)(k - 1)) * step >= c) --k;
    return k;
}

// grid (tiles, branches): each draw writes the samples whose u_k falls in [C_{i-1}, C_i)
__global__ void __launch_bounds__(kPostThreads) posterior_select_kernel(PosteriorArgs P) {
    __shared__ double sh_warp[kPostThreads / 32];
    const int b = blockIdx.y;
    const double T = P.total[b];
    if (!(T > 0.0) || !isfinite(T)) return;   // empty posterior (uniform over the block)
    double l[kPostPer], wb, e;
    post_tile_scan(P, b, blockIdx.x, P.lse[b].m, true, l, wb, e, sh_warp);
    const double o = P.tile_off[(size_t)b * (P.tiles + 1) + blockIdx.x];
    const double U = posterior_uniform(P.seed, P.stream, (unsigned long long)b);
    const double step = T / (double)P.K;
    int64_t* idx = b ? P.idx[1] : P.idx[0];
    const int64_t base = (int64_t)blockIdx.x * kPostTile + (int64_t)threadIdx.x * kPostPer;
    double lo = o + (wb + e);
#pragma unroll
    for (int j = 0; j < kPostPer; ++j) {
        const double hi = o + (wb + (e + l[j]));
        if (hi > lo) {
            const int64_t k1 = hi == T ? P.K : post_count(hi, U, step, P.K);
            for (int64_t k = post_count(lo, U, step, P.K); k < k1; ++k) idx[k] = base + j;
        }
        lo = hi;
    }
}

// ---- standalone log-mean-exp of an array (tri_log_mean_exp, _numerics.py:12-51) ----------------
constexpr int kLseThreads = 256;

// one partial per block over a contiguous slice: deterministic for a given grid
__global__ void __launch_bounds__(kLseThreads)
lse_partial_kernel(const double* lnl, Col lnprior, int64_t N, LsePartial* partials) {
    __shared__ LsePartial sh[kLseThreads];
    int64_t per_block = (N + gridDim.x - 1) / gridDim.x;
    int64_t lo = blockIdx.x * per_block;
    int64_t hi = lo + per_block < N ? lo + per_block : N;
    LsePartial a{-INFINITY, 0.0, 0, 0};
    for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        double x = lnl[i];
        if (lnprior.p) x += lnprior.at(i);
        lse_push(a, x);
    }
    sh[threadIdx.x] = a;
    __syncthreads();
    for (int o = kLseThreads / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) lse_merge(sh[threadIdx.x], sh[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) partials[blockIdx.x] = sh[0];
}

// merges up to a few thousand partials with one block (fixed tree: deterministic)
__global__ void __launch_bounds__(kLseThreads)
lse_final_kernel(const LsePartial* partials, int n, LsePartial* out) {
    __shared__ LsePartial sh[kLseThreads];
    LsePartial a{-INFINITY, 0.0, 0, 0};
    const int per = (n + kLseThreads - 1) / kLseThreads;
    for (int q = threadIdx.x * per; q < (int)(threadIdx.x + 1) * per && q < n; ++q)
        lse_merge(a, partials[q]);
    sh[threadIdx.x] = a;
    __syncthreads();
    for (int o = kLseThreads / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) lse_merge(sh[threadIdx.x], sh[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = sh[0];
}

// ---- FITPACK B-spline evaluation (device sampler: stellar relations, funcs.py:54-140) ----------
// y[i] = s(x[i]) for the spline (t[n], c[n], degree k <= 5) with extrapolation from the end
// intervals (splev ext=0): interval search + de Boor's recurrence (fpbspl), one thread per value.
constexpr int kSplevMaxKnots = 512;

template <int K>
__global__ void __launch_bounds__(256) splev_kernel(const double* __restrict__ t,
                                                     const double* __restrict__ c, int n,
                                                     const double* x, double* y, int64_t N) {
    constexpr int k = K;
    __shared__ double st[kSplevMaxKnots], sc[kSplevMaxKnots];
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
        st[j] = t[j];
        sc[j] = c[j];
    }
    __syncthreads();
    const int lmin = k, lmax = n - k - 2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N;
         i += (int64_t)gridDim.x * blockDim.x) {
        const double xv = x[i];
        // l = (number of knots <= x) - 1, clamped to the interior intervals
        int lo = 0, hi = n;
        while (lo < hi) {
            int mid = (lo + hi) >> 1;
            if (st[mid] <= xv) lo = mid + 1; else hi = mid;
        }
        int l = min(max(lo - 1, lmin), lmax);
        double h[K + 1], hh[K > 0 ? K : 1];
        h[0] = 1.0;
#pragma unroll
        for (int j = 1; j <= k; ++j) {
#pragma unroll
            for (int q = 0; q < j; ++q) hh[q] = h[q];
            h[0] = 0.0;
#pragma unroll
            for (int q = 0; q < j; ++q) {
                const double ti = st[l + q + 1], tj = st[l + q + 1 - j];
                const double f = hh[q] / (ti - tj);
                h[q] = h[q] + f * (ti - xv);
                h[q + 1] = f * (xv - tj);
            }
        }
        double sp = 0.0;
#pragma unroll
        for (int j = 0; j <= k; ++j) sp += sc[l - k + j] * h[j];
        y[i] = sp;
    }
}

// ---- FP64 issue-rate probe (roofline denominator measured on the box) -----------------------
__global__ void dfma_peak_kernel(double* out, int iters) {
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3;
    double a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double x = 1.0000001, y = 1e-9;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, x, y); a1 = fma(a1, x, y); a2 = fma(a2, x, y); a3 = fma(a3, x, y);
        a4 = fma(a4, x, y); a5 = fma(a5, x, y); a6 = fma(a6, x, y); a7 = fma(a7, x, y);
    }
    out[blockIdx.x * (size_t)blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

}  // namespace tri
