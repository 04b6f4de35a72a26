/*
 * triceratops_b200 -- C ABI of the B200 (sm_100a) marginal-likelihood engine.
 *
 * The reference (stevengiacalone/triceratops) is pure Python and has no FFI; its seams for this
 * path are ordinary Python functions.  Each entry point below names the reference interface it
 * stands in for (paths relative to the reference's triceratops/ package).  The Python host layer
 * (triceratops_b200/_cabi.py) binds these with ctypes; INTEGRATION.md shows the stub a reference
 * maintainer would add.
 *
 * Conventions: every function returns 0 on success and a negative TRI_E* code on failure, with
 * text available from tri_last_error().  One process drives one GPU (one context per process);
 * calls are serialised by the caller.  The caller owns every buffer it passes; the library never
 * keeps a host pointer after return.  All floating-point data is IEEE float64.
 */
#ifndef TRICERATOPS_B200_H
#define TRICERATOPS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRI_OK 0
#define TRI_ECUDA (-1)      /* CUDA runtime error                                   */
#define TRI_EINVAL (-2)     /* bad argument (NULL, negative size, NaN light curve)  */
#define TRI_ESTATE (-3)     /* tri_init / tri_set_lightcurve not called             */
#define TRI_ENODEVICE (-4)  /* no CUDA device: there is no CPU fallback             */

#define TRI_MAX_INFLIGHT 4  /* evaluations that may be queued before one is waited for */

/* A per-draw column: stride 1 = array of N values, stride 0 = one value used for every draw
 * (the reference broadcasts scalars with np.full(N, x), e.g. marginal_likelihoods.py:125-128). */
typedef struct {
    const double* ptr;
    int64_t stride;
} tri_col;

/* Inputs of one TP-type scenario (lnZ_TTP/PTP/STP/DTP/BTP, marginal_likelihoods.py:39, :386,
 * :869, :1379, :1840): the UNMASKED prior draws.  Geometry, masks, light curves, chi^2, the
 * companion prior and the log-mean-exp all run on the GPU. */
typedef struct {
    int64_t N;
    tri_col rp;       /* planet radius [R_earth]                       sample_rp            */
    tri_col P_orb;    /* orbital period [d]                                                  */
    tri_col inc;      /* inclination [deg]                             sample_inc           */
    tri_col ecc;      /* eccentricity                                  sample_ecc           */
    tri_col argp;     /* argument of periastron [deg]                  sample_w             */
    tri_col mtot;     /* mass in Kepler's law [M_sun] (M_s, masses_comp, masses_comp[idxs])  */
    tri_col rhost;    /* host-star radius [R_sun]                                            */
    tri_col u1, u2;   /* quadratic limb-darkening coefficients of the host                  */
    tri_col cfr;      /* companion_fluxratio                                                 */
    tri_col lnprior;  /* lnprior_companion, ptr NULL = none (lnZ_TTP)                        */
    const uint8_t* extra_mask; /* optional AND-term of the mask (qs_comp != 0, logg/Teff cuts) */
    int32_t companion_is_host;
} tri_tp_args;

/* Inputs of one EB-type scenario (lnZ_TEB/PEB/SEB/DEB/BEB, marginal_likelihoods.py:175, :589,
 * :1080, :1571, :2038).  One set of draws yields two results: q < 0.95 at period P ("EB") and
 * q >= 0.95 at period 2P ("EBx2P"). */
typedef struct {
    int64_t N;
    tri_col reb;      /* EB radius [R_sun]            stellar_relations                     */
    tri_col ebfr;     /* EB_fluxratio                                                         */
    tri_col q;        /* mass ratio                   sample_q                               */
    tri_col P_orb, inc, ecc, argp;
    tri_col mtot;     /* M_host + M_EB [M_sun]                                                */
    tri_col rhost, u1, u2, cfr, lnprior;
    const uint8_t* extra_mask;
    int32_t companion_is_host;
    int32_t scalar_loop;  /* 1: the semantics of the reference's parallel=False loops
                           * (marginal_likelihoods.py:313-339, likelihoods.py:121-123, :137):
                           * a draw whose period-P transit probability exceeds 1 is skipped in
                           * BOTH branches, the primary radius ratio is scaled by 0.999 only when
                           * |k - 1| < 1e-6, and the secondary uses 1/k.  0: the vectorised
                           * branch (parallel=True).  TP-type scenarios do not differ. */
} tri_eb_args;

/* Output of one scenario branch.  lnZ = m + ln(s) - ln(N) (-inf if no finite entry, +inf if any
 * entry is +inf: _numerics.py:12-51); (m, s) are exposed so that ranks holding disjoint slices
 * of the draws can be combined with one collective.  (m, s) are accumulated per block of the
 * persistent light-curve kernel in the order its warps pick up the draws: the last bits of lnZ
 * may differ between two runs on the same input (|dlnZ| ~ 1e-15); per-draw lnL never does. */
typedef struct {
    double lnZ;
    double m, s;          /* max of the finite ln-weights and sum of exp(lnw - m)            */
    int64_t n_finite;     /* finite ln-weights                                                */
    int64_t n_posinf;     /* +inf ln-weights                                                  */
    int64_t n_pass;       /* draws that survived the geometric mask of this branch           */
    int64_t n_stamps;     /* time stamps whose sub-exposures were evaluated  } work counters  */
    int64_t n_interior;   /* evaluated model points, occultor inside the disc } of the roofline */
    int64_t n_limb;       /* evaluated model points, occultor on the limb    } model: 0 unless */
                          /*                                       tri_set_counting(1) is on  */
    double* lnL_out;      /* optional [N]: per-draw lnL (no prior), -inf where masked         */
    uint8_t* mask_out;    /* optional [N]: the geometric mask                                 */
    /* best draws, i.e. the head of (-lnL).argsort() (marginal_likelihoods.py:152-153), selected
     * on the GPU: up to top_cap entries with finite lnL, best first, ties by ascending index.
     * Leave top_cap = 0 to skip.  (Device-pointer calls return them unsorted.)                */
    int64_t top_cap;      /* in: capacity of top_idx / top_lnL                                */
    int64_t n_top;        /* out: entries written (= min(top_cap, n_evaluated))               */
    int64_t n_evaluated;  /* out: draws with a finite lnL                                     */
    int64_t* top_idx;     /* out [top_cap]: draw indices                                      */
    double* top_lnL;      /* out [top_cap]: their lnL                                         */
} tri_result;

/* Bind this process to one GPU, create the stream, build and upload the orbit table.  */
int tri_init(int device);
int tri_shutdown(void);
const char* tri_last_error(void);

/* Upload the (renormalised, NaN-free) folded light curve: what every lnZ_* receives as
 * (time, flux, sigma, exptime, nsamples) -- triceratops.py:738-740, marginal_likelihoods.py:39-43. */
int tri_set_lightcurve(const double* time, const double* flux, int64_t npts, double sigma,
                       double exptime, int32_t nsamples);

/* The same with one error per time stamp (an extension: the reference takes a scalar,
 * triceratops.py:674, funcs.py:176).  chi^2 = sum_j (flux_j - model_j)^2 / flux_err_j^2; the
 * scalar that the reference's formulas need -- the Gaussian constant -ln(sigma), applied once
 * per light curve (marginal_likelihoods.py:130), and the secondary-depth cut 1.5 sigma
 * (likelihoods.py:535) -- is sigma = mean(flux_err), what callers of the reference pass today.
 * Constant errors give the scalar call's results (to rounding: the weights enter the sums). */
int tri_set_lightcurve_err(const double* time, const double* flux, const double* flux_err,
                           int64_t npts, double exptime, int32_t nsamples);

/* Mixed cadence (an extension: the reference passes one exposure time and one supersampling
 * count, pytransit's QuadraticModel.set_data takes one per light curve): exptime[j] and
 * nsamples[j] per time stamp.  The stamps are grouped by their distinct (exptime, nsamples)
 * pairs, compared exactly; each group is modelled with its own exposure and sample count, and
 * chi^2 is the sum over all stamps.  flux_err NULL: the scalar `sigma` as in tri_set_lightcurve,
 * else one error per stamp as in tri_set_lightcurve_err (`sigma` is ignored).  The Gaussian
 * constant, the secondary-eclipse pass and its depth cut do not depend on the cadence.  One
 * distinct pair gives exactly the device state of the scalar calls.  TRI_EINVAL for an exptime
 * that is not finite or < 0, nsamples < 1, or more than TRI_MAX_CADENCES distinct pairs. */
#define TRI_MAX_CADENCES 8
int tri_set_lightcurve_cadence(const double* time, const double* flux, const double* flux_err,
                               double sigma, const double* exptime, const int32_t* nsamples,
                               int64_t npts);

/* L2 seam, host buffers: replaces the body of lnZ_* between the prior draws and _log_mean_exp. */
int tri_eval_tp(const tri_tp_args* args, tri_result* out);
int tri_eval_eb(const tri_eb_args* args, tri_result out[2]); /* [0]=EB, [1]=EBx2P */

/* Same with every pointer (columns, extra_mask, lnL_out, mask_out) in DEVICE memory; work is
 * queued on `stream` (a cudaStream_t; NULL = the CUDA default stream, so that the work is ordered
 * after the kernels that produced the columns there) and the call returns after
 * the small result record has been read back. */
int tri_eval_tp_dev(const tri_tp_args* args, tri_result* out, void* stream);
int tri_eval_eb_dev(const tri_eb_args* args, tri_result out[2], void* stream);

/* Asynchronous forms of the four calls above (which are submit + wait).  tri_submit_* queues the
 * column copies (on a copy stream of the library) and the kernels, and returns a ticket without
 * waiting for the GPU, so that the caller can prepare the next scenario's draws -- or submit
 * it -- while this one runs: the copies of one call overlap the kernels of the one before, the
 * way consecutive lnZ_* calls of calc_probs (triceratops.py:750-1440) are independent of each
 * other.  `want` is the record tri_eval_* would receive (optional output pointers, top_cap);
 * tri_wait(ticket, out) blocks until that evaluation is complete and fills out[0] (TP-type) or
 * out[0..1] (EB-type).  Every buffer named by `args` and `want` must stay valid and unmodified
 * until tri_wait returns; entries of top_idx / top_lnL beyond n_top are unspecified.  At most
 * TRI_MAX_INFLIGHT tickets may be outstanding (TRI_ESTATE otherwise); tickets may be waited for
 * in any order, once.  tri_set_lightcurve first lets outstanding evaluations finish. */
int tri_submit_tp(const tri_tp_args* args, const tri_result* want, int64_t* ticket);
int tri_submit_eb(const tri_eb_args* args, const tri_result want[2], int64_t* ticket);
int tri_submit_tp_dev(const tri_tp_args* args, const tri_result* want, void* stream,
                      int64_t* ticket);
int tri_submit_eb_dev(const tri_eb_args* args, const tri_result want[2], void* stream,
                      int64_t* ticket);
int tri_wait(int64_t ticket, tri_result* out);

/* L1 seam, host buffers: lnL_TP_p (likelihoods.py:443-487), lnL_EB_p (:490-539) and
 * lnL_EB_twin_p (:542-587) on already-masked draws.  out[n] = +0.5 chi^2 (+inf where the
 * secondary-depth cut fires, twin == 0 only), exactly what the reference functions return. */
int tri_lnl_tp(int64_t n, const double* R_p, const double* P_orb, const double* inc,
               const double* a, const double* R_s, const double* u1, const double* u2,
               const double* ecc, const double* argp, const double* companion_fluxratio,
               int32_t companion_is_host, double* out);
int tri_lnl_eb(int64_t n, const double* R_EB, const double* EB_fluxratio, const double* P_orb,
               const double* inc, const double* a, const double* R_s, const double* u1,
               const double* u2, const double* ecc, const double* argp,
               const double* companion_fluxratio, int32_t companion_is_host, int32_t twin,
               double* out);

/* Model light curves on the time stamps of the current light curve (whose flux and sigma are
 * then irrelevant): simulate_TP_transit_p (likelihoods.py:302-358) and simulate_EB_transit_p
 * (:361-439).  flux_out is [n][npts] row-major in the caller's stamp order, after dilution;
 * secdepth_out (optional) is [n].  scalar_rule = 1 applies the radius-ratio rules of the scalar
 * simulate_EB_transit (:121-123, :137: |k-1| < 1e-6 and secondary k = 1/k) instead of the
 * vectorised ones (:406, :417-418).  Meant for handfuls of draws (best-fit curves, plot_fits):
 * n * npts is limited to 2^28. */
int tri_simulate_tp(int64_t n, const double* R_p, const double* P_orb, const double* inc,
                    const double* a, const double* R_s, const double* u1, const double* u2,
                    const double* ecc, const double* argp, const double* companion_fluxratio,
                    int32_t companion_is_host, double* flux_out);
int tri_simulate_eb(int64_t n, const double* R_EB, const double* EB_fluxratio,
                    const double* P_orb, const double* inc, const double* a, const double* R_s,
                    const double* u1, const double* u2, const double* ecc, const double* argp,
                    const double* companion_fluxratio, int32_t companion_is_host,
                    int32_t scalar_rule, double* flux_out, double* secdepth_out);

/* Per-draw lnL of branch 0/1 of the most recent tri_eval_* call, copied to a host buffer of N
 * doubles (the array stays on the device until the next call). */
int tri_fetch_lnl(int32_t branch, double* out, int64_t N);

/* _log_mean_exp (_numerics.py:12-51) of a host array on the GPU; fills lnZ, m, s, n_*. */
int tri_log_mean_exp(const double* logw, int64_t n, tri_result* out);

/* Device time [ms] of the kernels of the most recent eval/lnl call, from CUDA events on the
 * stream they ran on: geometry, light-curve/chi^2 (with the fused evidence epilogue), the
 * finalize kernel (merge of the block records + best-draw selection; with tri_set_moments on,
 * also the moments kernel; with tri_set_posterior K > 0, also the two resampling kernels), and
 * their launch count (3 per evaluation, 4 with moments, 2 more with posterior samples). */
int tri_last_timing(double* geometry_ms, double* lnl_ms, double* lse_ms, int32_t* launches);

/* Device-side prior sampler support (opt-in mode, triceratops_b200.set_sampler("device")):
 * FITPACK B-spline evaluation y[i] = s(x[i]) for the stellar relations of funcs.py:54-140
 * (scipy splev, ext=0: the end intervals extrapolate).  t[n] knots and c[n] coefficients of a
 * degree-k spline (1 <= k <= 5, n <= 512); every pointer is a DEVICE pointer; x and y may alias.
 * Queued on `stream` (NULL = the CUDA default stream); does not wait for the GPU. */
int tri_dev_splev(const double* t, const double* c, int32_t n, int32_t k, const double* x,
                  double* y, int64_t N, void* stream);

/* ---- device sampler (opt-in): one fused kernel per scenario draws the prior samples in HBM and
 * applies the transforms of priors.py:16-383 / :580-1005, funcs.py:54-140 and the limb-darkening
 * look-ups of marginal_likelihoods.py, writing the columns tri_submit_*_dev takes.  Every pointer
 * below is a DEVICE pointer; the small tables are uploaded once by the Python layer. */
typedef struct {           /* broken power law, inverse CDF (priors.py:54-111) */
    int32_t nseg;          /* 0: not a draw, `constant` is returned */
    double constant;
    double powers[3], amps[3], integrals[3], cum[3], epow[3];   /* epow[k] = edges[k]^(p_k + 1) */
    double norm;
} tri_powerlaw;

typedef struct {           /* FITPACK spline (t, c, k) as scipy stores it */
    const double* t;
    const double* c;
    int32_t n, k;
} tri_spline;

typedef struct {           /* constants of lnprior_bound_TP / lnprior_bound_EB (priors.py:580-1005) */
    double d_pc;           /* 1000 / plx */
    double M_eff, M_act;   /* max(M_s, 1) and M_s */
    double f1, f2, f3, alpha, dlogP, slope, slope2, t2, t3, t4, t5;
    int32_t first_decade;  /* 1: lnprior_bound_EB, 0: lnprior_bound_TP */
} tri_bound_prior;

typedef struct {
    int64_t n;             /* draws to make (this rank's share) */
    int64_t index0;        /* global index of the first one: the random stream of a draw depends
                            * on (seed, stream, global index) only, whatever the sharding */
    uint64_t seed, stream;
    int32_t kind;          /* 0 TP-type, 1 EB-type */
    int32_t host;          /* event on: 0 the target, 1 its bound companion (S*), 2 a background
                            * star (B*) */
    int32_t diluter;       /* other star in the aperture: 0 none, 1 bound companion (P*, S*),
                            * 2 background star (D*, B*) */
    int32_t flatpriors;
    double P_lo, P_hi;     /* period range [d]; equal: fixed period */
    double ecc_expo;       /* binaries: eccentricity power-law exponent (priors.py:150-154) */
    double M_s, R_s, Teff, u1, u2;                  /* the target star */
    tri_powerlaw rp_hi, rp_lo, q_pl, qc_pl;         /* sample_rp (two mass regimes), sample_q,
                                                     * sample_q_companion */
    tri_spline hot_R, cool_R, hot_T, cool_T;        /* stellar_relations (funcs.py:54-79) */
    tri_spline flux_tess, flux_cc;                  /* flux_relation in the TESS band and in the
                                                     * contrast-curve band (funcs.py:121-140) */
    double f_target_tess, f_target_cc;              /* flux_relation(M_s) in those bands */
    const double *ldc_u1, *ldc_u2;                  /* [27][4] limb darkening at the target's Z
                                                     * over (Teff, logg) nodes (:945-972) */
    double Teff_cap;
    int32_t prior_mode;    /* 0 none, 1 bound companion, 2 background star */
    int32_t use_cc;        /* a contrast curve was given */
    int32_t beb_cc_band;   /* BEB with a contrast curve in J/H/K: flux_cc is that band */
    int32_t cc_n;
    const double *cc_sep, *cc_con;                  /* contrast curve (or the 2.2" / 1.0 default) */
    tri_bound_prior bound;
    double bg_const_prior;                          /* background prior without a contrast curve */
    const double* molusc_q;                         /* optional [n]: companion mass ratios */
    int64_t n_comp, idx_hi;                         /* TRILEGAL stars; randint upper bound */
    const double *bg_mass, *bg_radius, *bg_logg, *bg_teff, *bg_u1, *bg_u2;
    const double *bg_fr_tess, *bg_dmag_cc, *bg_fr_cc;
    /* outputs [n] (NULL: not wanted) */
    double *o_body, *o_ebfr, *o_q, *o_P, *o_inc, *o_ecc, *o_argp, *o_mtot, *o_rhost, *o_u1, *o_u2,
           *o_cfr, *o_lnprior, *o_mhost, *o_meb;
    uint8_t* o_mask;
    int32_t* err_flag;     /* set to 1 if a limb-darkening node lies beyond the grid */
    /* importance proposal (appended: the offsets above are unchanged).  Each tuned prior
     * dimension ("slot": 0 P when P_lo < P_hi, 1 the diluter's uniform -- q_comp or the TRILEGAL
     * index, not MOLUSC rows --, 2 R_p (TP) or q (EB), 3 inc, 4 ecc (EB only), 5 argp) is drawn
     * as its prior transform of v instead of the uniform u.  A coin c from a counter block of its
     * own picks the branch of the defensive mixture q(v) = alpha + (1 - alpha) prod_d h_d(v_d):
     * c < alpha, v = u (a prior draw); otherwise v = H_d^-1(u), H_d the piecewise-linear CDF of
     * h_d.  The kernel adds -ln q(v) = -log1p((1 - alpha) expm1(s)), s = sum_d ln h_d(v_d), to
     * o_lnprior (after the prior's clipping; a scenario without a companion prior then writes
     * one).  Identity tables (C_b = b / B, ln h = 0) give the columns of prop = NULL bit for bit
     * and a delta of exactly 0. */
    const double* prop;    /* NULL: the prior.  Else per slot, 2 B + 1 doubles: the knots
                            * C[0..B] of H (C[0] = 0, C[B] = 1), then ln h[0..B-1] */
    int32_t prop_bins;     /* B, a power of two */
    double prop_alpha;     /* alpha in (0, 1] */
    double* o_coords;      /* optional [TRI_PROP_SLOTS][n]: the v each slot used (the raw
                            * uniform without a proposal), NaN for slots the scenario does not
                            * draw */
} tri_sampler_args;
#define TRI_PROP_SLOTS 6

/* Queue the sampler kernel on `stream` (NULL = the CUDA default stream); does not wait. */
int tri_dev_sample(const tri_sampler_args* args, void* stream);

/* Measured FP64 FMA issue rate of this GPU [DFMA/s] (roofline denominator). */
int tri_fp64_peak(double* dfma_per_s);

/* Work accounting (off by default): when on, evaluations also count the work classes of the
 * roofline model -- n_stamps, n_interior, n_limb of tri_result -- in the hot loop (about 1.5 %
 * slower); when off those three fields are 0.  bench.py turns it on for one untimed pass. */
int tri_set_counting(int32_t on);

/* Second moment of the importance weights (off by default; captured per submission, like
 * tri_set_counting).  When on, every evaluation also runs one short kernel after the evidence
 * merge that sums s2 = sum over the finite ln-weights x of exp(2 (x - m)) per branch, with x =
 * lnL + lnprior formed as for lnZ and m the branch's record.  From (N, m, s, s2) follow the
 * standard error of lnZ and the effective sample size (triceratops_b200._numerics). */
int tri_set_moments(int32_t on);

/* s2 of branch 0 (and 1 for an EB-type call) of the evaluation most recently returned by
 * tri_eval_* / tri_eval_*_dev / tri_wait; NaN where moments were off for it (and for s2[1] of a
 * TP-type call).  A submission keeps its s2 until it is waited for. */
int tri_last_moments(double s2[2]);

/* Posterior samples by systematic importance resampling (off by default).  With K > 0 every
 * evaluation submitted afterwards also draws K samples from the N prior draws of each branch,
 * with weights w_i = exp(x_i - m), x_i = lnL_i + lnprior_i formed as for lnZ and m the branch's
 * record (0 where x_i is not finite): with C the prefix sums of w in draw order and T = C_{N-1},
 * sample k (k < K) is draw min{i : C_i > (U + k) T / K}, positions at or above T going to the
 * last draw at which C increases.  U in [0, 1) is a hash of (seed, stream, branch)
 * (triceratops_b200._numerics.posterior_uniform).  Two more kernels run per evaluation, after
 * the evidence merge (and the moments kernel); their results do not depend on scheduling or on
 * the SM count.  K, seed and stream are captured per submission.  Growing K beyond what any
 * earlier call set lets the evaluations in flight finish first, then grows the per-slot index
 * buffers (no evaluation allocates them).  TRI_EINVAL for K < 0 or K > TRI_MAX_POSTERIOR. */
#define TRI_MAX_POSTERIOR (1 << 20)
int tri_set_posterior(int64_t K, uint64_t seed, uint64_t stream);

/* Posterior sample indices (ascending, local to the call's draws) of branch `branch` of the
 * evaluation most recently returned by tri_eval_* / tri_eval_*_dev / tri_wait, copied to
 * idx[0..*n).  *n = K, or 0 when posterior samples were off for it or the posterior is empty (a
 * weight is +inf, or no weight is finite); *total = T, the sum of the weights relative to the
 * branch's m (NaN when off, +inf or 0 when empty).  A submission keeps its samples until it is
 * waited for.  TRI_EINVAL for a branch the evaluation does not have, or cap < K. */
int tri_last_posterior(int32_t branch, int64_t* idx, int64_t cap, int64_t* n, double* total);

/* sizeof() of the ABI structs, in the order tri_col, tri_tp_args, tri_eb_args, tri_result,
 * tri_powerlaw, tri_spline, tri_bound_prior, tri_sampler_args (the first n of them), so that a
 * binding can verify its own layouts.  Needs no device. */
int tri_struct_sizes(int64_t* out, int32_t n);

/* SM count of the bound device. */
int tri_sm_count(int32_t* n);

#ifdef __cplusplus
}
#endif
#endif
