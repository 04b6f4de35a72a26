// Device sampler (opt-in mode, triceratops_b200.set_sampler("device")): ONE fused kernel per
// scenario draws the prior samples with a counter-based generator and applies every transform
// of the host path -- inverse-CDF samplers (reference priors.py:16-383), stellar and flux
// relations (funcs.py:54-140), limb-darkening look-ups (marginal_likelihoods.py:945-972,
// :1913-1924), companion / background priors with the contrast-curve interpolation
// (priors.py:580-1005, marginal_likelihoods.py:478-509, :1466-1492, :2147-2201) -- and writes the
// engine's SoA columns straight into HBM.  Nothing of it touches the host; the columns go to
// tri_submit_*_dev by pointer.
//
// The deviates are Philox4x32-10 streams keyed by (seed, scenario stream, draw index), not
// numpy's Mersenne Twister: results are statistically, not bitwise, equivalent to the host
// sampler (tests/test_device_sampler.py: two-sample KS per column, evidences within Monte-Carlo
// scatter).  The deterministic transforms are the formulas of priors.py / funcs.py.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/triceratops_b200.h"
#include "tri_model.cuh"

namespace tri {

// ---- Philox4x32-10 -----------------------------------------------------------------------------
struct Philox {
    uint32_t key[2];
    uint32_t ctr[4];
    uint32_t out[4];
    int have;   // unread words in out
    __device__ Philox(uint64_t seed, uint64_t stream, uint64_t index) {
        key[0] = (uint32_t)seed;
        key[1] = (uint32_t)(seed >> 32);
        ctr[0] = (uint32_t)index;
        ctr[1] = (uint32_t)(index >> 32);
        ctr[2] = (uint32_t)stream;
        ctr[3] = 0;          // block counter of this (stream, index)
        have = 0;
    }
    __device__ void refill() {
        uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
        uint32_t k0 = key[0], k1 = key[1];
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
            const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
            const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
            c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
        ctr[3] += 1;
        have = 4;
    }
    __device__ uint32_t next32() {
        if (have == 0) refill();
        return out[4 - have--];
    }
    // uniform on [0, 1) with 53 random bits (the construction numpy uses for its doubles)
    __device__ double uniform() {
        const uint32_t a = next32() >> 5, b = next32() >> 6;
        return (a * 67108864.0 + b) * (1.0 / 9007199254740992.0);
    }
    __device__ double normal() {   // Box-Muller, one deviate per call
        const double u1 = 1.0 - uniform(), u2 = uniform();
        return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
    }
    // Gamma(shape, 1), Marsaglia & Tsang (2000); shape < 1 through Gamma(shape + 1) U^(1/shape)
    __device__ double gamma(double shape) {
        double boost = 1.0;
        if (shape < 1.0) {
            boost = pow(1.0 - uniform(), 1.0 / shape);
            shape += 1.0;
        }
        const double d = shape - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
        for (;;) {
            double x, v;
            do {
                x = normal();
                v = 1.0 + c * x;
            } while (v <= 0.0);
            v = v * v * v;
            const double u = 1.0 - uniform();
            if (u < 1.0 - 0.0331 * (x * x) * (x * x)) return boost * d * v;
            if (log(u) < 0.5 * x * x + d * (1.0 - v + log(v))) return boost * d * v;
        }
    }
};

// ---- transforms ----------------------------------------------------------------------------------
// broken power law, inverse CDF (priors._piecewise_powerlaw; constants precomputed on the host)
__device__ __forceinline__ double pl_inverse(const tri_powerlaw& L, double x) {
    if (L.nseg <= 0) return L.constant;
    int k = 0;
    while (k < L.nseg - 1 && x > L.norm * L.cum[k]) ++k;
    double u = x / L.norm;
    for (int j = 0; j < k; ++j) u -= L.integrals[j];
    const double p1 = L.powers[k] + 1.0;
    return pow(fmax(u * p1 / L.amps[k] + L.epow[k], 1e-300), 1.0 / p1);
}

// FITPACK B-spline value with extrapolation (splev ext=0), as splev_kernel
__device__ double spline_at(const tri_spline& S, double xv) {
    const double* __restrict__ t = S.t;
    const double* __restrict__ c = S.c;
    const int n = S.n, k = S.k;
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(t + mid) <= xv) lo = mid + 1; else hi = mid;
    }
    const int l = min(max(lo - 1, k), n - k - 2);
    double h[6], hh[5];
    h[0] = 1.0;
    for (int j = 1; j <= k; ++j) {
        for (int q = 0; q < j; ++q) hh[q] = h[q];
        h[0] = 0.0;
        for (int q = 0; q < j; ++q) {
            const double ti = __ldg(t + l + q + 1), tj = __ldg(t + l + q + 1 - j);
            const double f = hh[q] / (ti - tj);
            h[q] = h[q] + f * (ti - xv);
            h[q + 1] = f * (xv - tj);
        }
    }
    double sp = 0.0;
    for (int j = 0; j <= k; ++j) sp += __ldg(c + l - k + j) * h[j];
    return sp;
}

// piecewise-linear interpolation with end clamping over (xp, fp), plain bisection (see
// device_sampler.py on numpy.interp and non-monotonic contrast curves)
__device__ double interp_at(const double* __restrict__ xp, const double* __restrict__ fp, int n,
                            double x) {
    if (n == 1) return __ldg(fp);
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (x < __ldg(xp + mid)) hi = mid; else lo = mid + 1;
    }
    const int j = min(max(lo - 1, 0), n - 2);
    if (x >= __ldg(xp + n - 1)) return __ldg(fp + n - 1);
    if (x <= __ldg(xp)) return __ldg(fp);
    const double x0 = __ldg(xp + j), x1 = __ldg(xp + j + 1);
    const double f0 = __ldg(fp + j), f1 = __ldg(fp + j + 1);
    return (f1 - f0) / (x1 - x0) * (x - x0) + f0;
}

// stellar_relations (funcs.py:54-79): cubic-spline mass -> (radius, Teff) with caps and floors
__device__ __forceinline__ void star_of_mass(const tri_sampler_args& A, double m, double max_R,
                                             double max_T, double& R, double& T) {
    const bool hot = m > 0.63;
    R = spline_at(hot ? A.hot_R : A.cool_R, m);
    T = spline_at(hot ? A.hot_T : A.cool_T, m);
    R = fmax(fmin(R, max_R), 0.1);
    T = fmax(fmin(T, max_T), 2800.0);
}

// F(m) / (F(m) + F(M_s)) in the TESS band or in the contrast-curve band (funcs.py:121-140)
__device__ __forceinline__ double flux_ratio(const tri_sampler_args& A, double m, bool cc_band) {
    const double f = pow(10.0, spline_at(cc_band ? A.flux_cc : A.flux_tess, m));
    return f / (f + (cc_band ? A.f_target_cc : A.f_target_tess));
}

// lnprior_bound_TP / lnprior_bound_EB (priors.py:580-1005): companion-rate prior from the
// period distribution of binaries inside the separation the contrast curve leaves unseen
__device__ double bound_prior(const tri_sampler_args& A, double delta_mag_abs) {
    const tri_bound_prior& B = A.bound;
    const double seps = B.d_pc * interp_at(A.cc_con, A.cc_sep, A.cc_n, delta_mag_abs);
    const double au_cm = 14959787070000.0;
    const double x = seps * au_cm;
    const double max_P = sqrt((4.0 * kPi * kPi) / (kG * B.M_eff * kMsun) * (x * x * x)) / 86400.0;
    const double lp = log10(max_P);
    const double t2p = 0.5 * (lp - 1.0) * (2.0 * B.f1 + B.slope * (lp - 1.0));
    const double t3p = 0.5 * B.alpha * (lp * lp - 5.4 * lp + 6.8) + B.f2 * (lp - 2.0);
    const double t4p = B.alpha * B.dlogP * (lp - 3.4) + B.f2 * (lp - 3.4)
                     + B.slope2 * (0.238095 * lp * lp - 0.952381 * lp + 0.485714);
    const double t5p = B.f3 * (3.33333 - 17.3566 * exp(-0.3 * lp));
    double f;
    if (B.first_decade) {
        if (lp >= 8.0) f = B.t2 + B.t3 + B.t4 + B.t5;
        else if (lp >= 5.5) f = B.t2 + B.t3 + B.t4 + t5p;
        else if (lp >= 3.4) f = B.t2 + B.t3 + t4p;
        else if (lp >= 2.0) f = B.t2 + t3p;
        else if (lp >= 1.0) f = t2p;
        else f = 0.0;
    } else {
        if (lp >= 8.0) f = B.t4 + B.t5;
        else if (lp >= 5.5) f = B.t4 + t5p;
        else if (lp >= 3.4) f = t4p;
        else f = 0.0;
    }
    if (B.M_act >= 1.0) return log(f);
    return log(fmax(0.65 * f + 0.35 * f * B.M_act, 0.0));
}

// clipping of marginal_likelihoods.py:488-489
__device__ __forceinline__ double clip_prior(double lnprior, double delta_mag) {
    lnprior = fmin(lnprior, 0.0);
    return delta_mag > 0.0 ? -INFINITY : lnprior;
}

// ---- importance proposal (tri_sampler_args.prop) --------------------------------------------------
// One tuned dimension (slot) maps the uniform u its inverse CDF would receive to the coordinate v
// it receives instead.  Off the prior branch of the defensive mixture, v = H^-1(u) with H the
// piecewise-linear CDF of the slot's binned density h (knots C[0..B], ln h[0..B-1]); on it, v = u.
// Either way s gains ln h of v's bin -- the bin the search found, not one recomputed from v,
// which rounding can put on a bin edge.  Identity tables (C_b = b / B, h = 1, B a power of two)
// give v = u exactly on both branches and s = 0.
struct Proposal {
    const double* tab;   // NULL: the prior, nothing is changed
    int B;
    bool mix;            // off the prior branch
    double s;            // sum over the tuned slots of ln h(v)
    double* coords;      // optional: v of each slot, column-major [TRI_PROP_SLOTS][n]
    int64_t n, i;
};

__device__ __forceinline__ double propose(Proposal& Q, int slot, double u) {
    if (Q.tab == nullptr) {
        if (Q.coords) Q.coords[slot * Q.n + Q.i] = u;
        return u;
    }
    const int B = Q.B;
    const double* __restrict__ C = Q.tab + (size_t)slot * (2 * B + 1);
    const double* __restrict__ lnh = C + B + 1;
    double v;
    int b;
    if (Q.mix) {
        int lo = 0, hi = B - 1;          // largest b with C[b] <= u
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (__ldg(C + mid) <= u) lo = mid; else hi = mid - 1;
        }
        b = lo;
        const double l = __ldg(lnh + b);
        v = ((double)b + (u - __ldg(C + b)) / (exp(l) / (double)B)) / (double)B;
        v = fmin(v, 0x1.fffffffffffffp-1);
        Q.s += l;
    } else {
        v = u;
        b = min((int)(v * (double)B), B - 1);
        Q.s += __ldg(lnh + b);
    }
    if (Q.coords) Q.coords[slot * Q.n + Q.i] = v;
    return v;
}

// ---- the kernel ----------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sampler_kernel(tri_sampler_args A) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < A.n;
         i += (int64_t)gridDim.x * blockDim.x) {
        Philox rng(A.seed, A.stream, (uint64_t)(A.index0 + i));
        Proposal Q;
        Q.tab = A.prop;
        Q.B = A.prop_bins;
        Q.s = 0.0;
        Q.mix = false;
        Q.coords = A.o_coords;
        Q.n = A.n;
        Q.i = i;
        if (A.prop) {
            // the mixture's coin comes from a counter block of its own: the draw's main stream
            // is consumed exactly as without a proposal
            Philox coin(A.seed, A.stream, (uint64_t)(A.index0 + i));
            coin.ctr[3] = 0x80000000u;
            Q.mix = !(coin.uniform() < A.prop_alpha);
        }
        const double P = A.P_lo == A.P_hi
                             ? A.P_lo
                             : A.P_lo + (A.P_hi - A.P_lo) * propose(Q, 0, rng.uniform());

        // ---- the star that hosts the event, and the star that dilutes it
        double M_host = A.M_s, R_host = A.R_s, T_host = A.Teff, u1 = A.u1, u2 = A.u2;
        double cfr = 0.0, lnprior = 0.0, m_comp = 0.0;
        bool ok = true;
        int64_t idx = 0;
        if (A.diluter == 1) {            // unresolved bound companion (P*, S*)
            const double q_comp = A.molusc_q ? A.molusc_q[i]
                                              : pl_inverse(A.qc_pl, propose(Q, 1, rng.uniform()));
            ok = q_comp != 0.0;          // MOLUSC padding (marginal_likelihoods.py:464, :534)
            m_comp = q_comp * A.M_s;
            cfr = ok ? flux_ratio(A, m_comp, false) : 0.0;
            if (A.host == 1 && ok) {     // the companion hosts the event (S*)
                M_host = m_comp;
                star_of_mass(A, m_comp, A.R_s, A.Teff, R_host, T_host);
                const double logg = log10(kG * (m_comp * kMsun) / ((R_host * kRsun) * (R_host * kRsun)));
                const double rg = fmin(fmax(rint(logg / 0.5) * 0.5, 3.5), 5.0);
                const double rT = fmin(fmax(rint(T_host / 250.0) * 250.0, 3500.0), A.Teff_cap);
                const int it = (int)((rT - 3500.0) / 250.0), ig = (int)rint((rg - 3.5) / 0.5);
                if (it > 26) {           // node beyond the grid: the reference raises (:1181)
                    atomicExch(A.err_flag, 1);
                    u1 = u2 = NAN;
                } else {
                    u1 = __ldg(A.ldc_u1 + it * 4 + ig);
                    u2 = __ldg(A.ldc_u2 + it * 4 + ig);
                }
            }
        } else if (A.diluter == 2) {     // chance-aligned background star (D*, B*)
            idx = (int64_t)(propose(Q, 1, rng.uniform()) * (double)A.idx_hi);
            if (idx >= A.idx_hi) idx = A.idx_hi - 1;
            cfr = __ldg(A.bg_fr_tess + idx);
            if (A.host == 2) {           // the background star hosts the event (B*)
                M_host = __ldg(A.bg_mass + idx);
                R_host = __ldg(A.bg_radius + idx);
                T_host = __ldg(A.bg_teff + idx);
                u1 = __ldg(A.bg_u1 + idx);
                u2 = __ldg(A.bg_u2 + idx);
                ok = __ldg(A.bg_logg + idx) >= 3.5 && T_host <= 10000.0;   // :1981-1986
            }
        }

        // ---- the transiting / eclipsing body
        double body, ebfr = 0.0, q = 0.0, mtot, inc, ecc, argp, m_eb = 0.0;
        if (A.kind == 0) {
            const double x = propose(Q, 2, rng.uniform());
            body = A.flatpriors ? x / (1.0 / 19.5) + 0.5
                                : pl_inverse(M_host > 0.45 ? A.rp_hi : A.rp_lo, x);
            inc = acos(1.0 - propose(Q, 3, rng.uniform())) * (180.0 / kPi);
            const double ga = rng.gamma(0.867), gb = rng.gamma(3.030);
            ecc = ga / (ga + gb);
            argp = propose(Q, 5, rng.uniform()) * 360.0;
            mtot = M_host;
        } else {
            inc = acos(1.0 - propose(Q, 3, rng.uniform())) * (180.0 / kPi);
            q = pl_inverse(A.q_pl, propose(Q, 2, rng.uniform()));
            ecc = pow(propose(Q, 4, rng.uniform()), 1.0 / A.ecc_expo);
            argp = propose(Q, 5, rng.uniform()) * 360.0;
            m_eb = q * M_host;
            double T_eb;
            star_of_mass(A, m_eb, R_host, T_host, body, T_eb);
            ebfr = flux_ratio(A, m_eb, false);
            if (A.host == 2) {           // EB behind the target: flux ratio rescaled from "bound
                                         // at the target's distance" to the star's brightness
                ebfr *= cfr / flux_ratio(A, M_host, false);              // :2147-2159
            }
            mtot = M_host + m_eb;
        }

        // ---- companion / background prior
        if (A.prior_mode == 1) {         // bound companion
            double term, dmag;
            const bool band = A.use_cc != 0;
            if (A.host == 1 && A.kind == 1) {          // SEB: companion + its EB (:1202-1205)
                const double fc = band ? flux_ratio(A, m_comp, true) : cfr;
                const double fe = band ? flux_ratio(A, m_eb, true) : ebfr;
                term = fc / (1.0 - fc) + fe / (1.0 - fe);
            } else {
                const double fc = band ? flux_ratio(A, m_comp, true) : cfr;
                term = fc / (1.0 - fc);
            }
            dmag = 2.5 * log10(term);
            lnprior = ok ? clip_prior(bound_prior(A, fabs(dmag)), dmag) : 0.0;
        } else if (A.prior_mode == 2) {  // background star
            double dmag;
            if (A.host == 2 && A.kind == 1) {          // BEB: star + its EB (:2187-2201)
                double fc = cfr, fe = ebfr;
                if (A.use_cc) {
                    fc = __ldg(A.bg_fr_cc + idx);
                    fe = flux_ratio(A, m_eb, A.beb_cc_band != 0)
                       * (fc / flux_ratio(A, M_host, A.beb_cc_band != 0));
                }
                dmag = 2.5 * log10(fc / (1.0 - fc) + fe / (1.0 - fe));
            } else {
                dmag = A.use_cc ? __ldg(A.bg_dmag_cc + idx) : 2.5 * log10(cfr / (1.0 - cfr));
            }
            const double lp = A.use_cc
                ? log((double)A.n_comp / 0.1 * (1.0 / 3600.0) * (1.0 / 3600.0)
                      * pow(interp_at(A.cc_con, A.cc_sep, A.cc_n, fabs(dmag)), 2.0))
                : A.bg_const_prior;
            lnprior = clip_prior(lp, dmag);
        }
        // importance weight of the proposal: lnprior - ln q(v), q = alpha + (1 - alpha) e^s
        // (exactly 0 for s = 0), after the clipping, which is part of the prior
        if (A.prop) lnprior -= log1p((1.0 - A.prop_alpha) * expm1(Q.s));

        A.o_body[i] = body;
        A.o_P[i] = P;
        A.o_inc[i] = inc;
        A.o_ecc[i] = ecc;
        A.o_argp[i] = argp;
        A.o_mtot[i] = mtot;
        if (A.o_ebfr) A.o_ebfr[i] = ebfr;
        if (A.o_q) A.o_q[i] = q;
        if (A.o_rhost) A.o_rhost[i] = R_host;
        if (A.o_u1) A.o_u1[i] = u1;
        if (A.o_u2) A.o_u2[i] = u2;
        if (A.o_cfr) A.o_cfr[i] = cfr;
        if (A.o_lnprior) A.o_lnprior[i] = lnprior;
        if (A.o_mask) A.o_mask[i] = ok ? 1 : 0;
        if (A.o_mhost) A.o_mhost[i] = M_host;
        if (A.o_meb) A.o_meb[i] = m_eb;
    }
}

}  // namespace tri
