"""The ten `lnZ_*` scenario functions of TRICERATOPS on the B200 engine.

Drop-in for triceratops/marginal_likelihoods.py of the reference: same names, same positional
and keyword arguments, same return dictionaries (keys M_s, R_s, u1, u2, P_orb, inc, b, R_p, ecc,
argp, M_EB, R_EB, fluxratio_EB, fluxratio_comp: the 100 best draws, best first; plus lnZ).
EB-type functions return (res, res_twin).

Division of labour:
  host (this file)  prior draws from numpy's global RNG in the reference's exact call order, so
                    that a given np.random.seed produces the reference's arrays; stellar
                    relations, flux ratios, companion priors, limb-darkening look-ups.
  GPU (csrc/)       Kepler's-law geometry, transit-probability / collision / inclination masks,
                    supersampled quadratic-limb-darkened light curve, secondary-eclipse cut,
                    chi^2, + companion prior, log-mean-exp.  Draws are sent UNMASKED.

`parallel` selects the SEMANTICS, as in the reference, not the execution (always the GPU):
parallel=True is the vectorised branch (lnL_TP_p / lnL_EB_p / lnL_EB_twin_p); parallel=False
(the reference's default, triceratops.py:676) is its scalar loop, which differs for EB-type
scenarios -- radius-ratio rules |k - 1| < 1e-6 and secondary 1/k (likelihoods.py:121-123, :137
vs :406, :417-418), and a draw whose period-P transit probability exceeds 1 is skipped in both
branches (marginal_likelihoods.py:316-319) -- and is reproduced by the engine's scalar_loop flag.
TP-type scenarios give the same numbers either way.
"""
import functools
import sys

import numpy as np
from pandas import read_csv

from . import _blocks, _dispatch, _fastrng
from . import _hostpar
from ._numerics import mc_error
from ._constants import G, Msun, Rsun, pi
from ._ldc import grid_for
from .funcs import (file_to_contrast_curve, flux_relation, stellar_relations, trilegal_results)
from .priors import (lnprior_background, lnprior_bound_EB, lnprior_bound_TP, sample_ecc,
                     sample_inc, sample_q, sample_q_companion, sample_rp, sample_w)

np.seterr(divide='ignore')

_SAMPLER = {"mode": "host"}


def _sampler_mode():
    return _SAMPLER["mode"]


def _device_sampler_twin(fn):
    """In device-sampler mode the call goes, arguments unchanged, to the device_sampler function
    of the same name (which takes the same parameters in the same order)."""
    @functools.wraps(fn)
    def call(*args, **kwargs):
        if _sampler_mode() == "device":
            from . import device_sampler
            return getattr(device_sampler, fn.__name__)(*args, **kwargs)
        ds = sys.modules.get(__package__ + ".device_sampler")
        if ds is not None and ds._prop["proposal"] is not None:
            raise ValueError("importance proposals draw on the device sampler only "
                             "(set_sampler('device'))")
        return fn(*args, **kwargs)
    return call


N_SAMPLES = 100
RESULT_KEYS = ('M_s', 'R_s', 'u1', 'u2', 'P_orb', 'inc', 'b', 'R_p', 'ecc', 'argp', 'M_EB', 'R_EB',
               'fluxratio_EB', 'fluxratio_comp')

__all__ = ["lnZ_TTP", "lnZ_TEB", "lnZ_PTP", "lnZ_PEB", "lnZ_STP", "lnZ_SEB", "lnZ_DTP",
           "lnZ_DEB", "lnZ_BTP", "lnZ_BEB",
           "lnZ_NTP_unknown", "lnZ_NEB_unknown", "lnZ_NTP_evolved", "lnZ_NEB_evolved"]


# ------------------------------------------------------------------------------ shared pieces
def _periods(P_orb, N):
    """Fixed period or uniform draws over a range (marginal_likelihoods.py:67-72).  Returns
    (per-draw array, or a float that the engine broadcasts; mean period for sample_ecc)."""
    if type(P_orb) not in [float, int]:
        P = _fastrng.uniform(P_orb[0], P_orb[-1], N)
        return P, np.mean(P)
    # np.mean(np.full(N, P)) is what the reference hands to sample_ecc; it can differ from P in
    # the last bits, which only matters at the P <= 10 switch: take the same route there, and
    # spare the generator-holding thread two 8 MB passes everywhere else
    if abs(float(P_orb) - 10.0) < 1e-6:
        return float(P_orb), np.mean(np.full(N, P_orb))
    return float(P_orb), float(P_orb)


def _take(x, idx):
    """x[idx] for per-draw arrays, np.full for broadcast scalars."""
    if np.ndim(x) == 0:
        return np.full(len(idx), x)
    return _hostpar.take(x, idx)       # (large float64 gathers run without the GIL)


def _logg(M, R):
    return np.log10(G * (M * Msun) / (R * Rsun) ** 2)


def result_table(n_zeros, twin, M_s, R_s, u1, u2, P, mtot, inc, ecc, argp, R_p=None, M_EB=None,
                 R_EB=None, fluxratio_EB=None, fluxratio_comp=None):
    """The reference's result dictionary (marginal_likelihoods.py:155-171, keys RESULT_KEYS)
    from the rows of the best draws: the twin branch reports the doubled period, a and the
    impact parameter b follow from the orbit, and a column the scenario does not have is
    n_zeros zeros."""
    P_orb = 2 * P if twin else P
    a = ((G * mtot * Msun) / (4 * pi ** 2) * (P_orb * 86400) ** 2) ** (1 / 3)
    r = a * (1 - ecc ** 2) / (1 + ecc * np.sin(argp * np.pi / 180))
    b = r * np.cos(inc * pi / 180) / (R_s * Rsun)
    given = dict(M_s=M_s, R_s=R_s, u1=u1, u2=u2, P_orb=P_orb, inc=inc, b=b, R_p=R_p, ecc=ecc,
                 argp=argp, M_EB=M_EB, R_EB=R_EB, fluxratio_EB=fluxratio_EB,
                 fluxratio_comp=fluxratio_comp)
    return {k: np.zeros(n_zeros) if given[k] is None else given[k] for k in RESULT_KEYS}


def _draw_ecc(N, planet, P_mean):
    """sample_ecc(np.random.rand(N), planet, P_orb) of the reference (priors.py:134-155): the
    uniform deviates are drawn and ignored, the eccentricities come from scipy.stats on numpy's
    global generator -- Beta(0.867, 3.03) for planets, a power law for binaries."""
    _fastrng.skip(N)
    if planet:
        return _fastrng.beta_rvs(0.867, 3.030, N, pinned=True)
    # scipy.stats.powerlaw.rvs(a, size=N) is pow(uniform deviates, 1/a): only the deviates are
    # taken here, while the generator is held; _ecc_binary() maps them later, chunk by chunk
    return _fastrng.rand(N, pinned=True)


def _prepare(kind, block, N, arrays, **ckw):
    """Outputs of a scenario's element-wise preparation: csrc/host_blocks.c (one GIL-free call,
    the same values bit for bit) when usable, else `block` chunk by chunk in Python threads."""
    res = _blocks.run(kind, N, **ckw)
    if res is None:
        cc = ckw.get("contrast_curve_file")
        if cc is not None and not _blocks.order_free(file_to_contrast_curve(cc)[1]):
            # numpy.interp on this table depends on the order of the queries: all N in one
            # call, as the reference makes it
            return block(*arrays)
        res = _hostpar.pmap_block(block, N, *arrays)
    return res


def _ecc_binary(x, P_mean):
    """In place: the binaries' eccentricities from the deviates _draw_ecc(N, False, .) drew."""
    np.power(x, 1.0 / (0.2 if P_mean <= 10 else 0.6), out=x)


class _PlanetDraws:
    """The deviates of a planet draw, taken from numpy's generator in the reference's order
    (rp, inc, ecc, argp; the eccentricity sampler draws from the generator itself).  The
    inverse-CDF transforms are applied by finish(), which a scenario calls after it has handed
    the generator on (_dispatch.rng_done): they are deterministic."""

    def __init__(self, N, P_mean):
        self.x_rp = _fastrng.rand(N)
        self.x_inc = _fastrng.rand(N)
        self.eccs = _draw_ecc(N, True, P_mean)
        self.x_w = _fastrng.rand(N)

    @staticmethod
    def transform(x_rp, x_inc, x_w, host_masses, flatpriors):
        """(rps, incs, argps) of a chunk of deviates; host_masses per draw or one value."""
        if np.ndim(host_masses) == 0:
            host_masses = np.full(len(x_rp), host_masses)
        return sample_rp(x_rp, host_masses, flatpriors), sample_inc(x_inc), sample_w(x_w)

    def finish(self, host_masses, flatpriors):
        def block(x_rp, x_inc, x_w, m):
            return self.transform(x_rp, x_inc, x_w, m, flatpriors)
        N = len(self.x_rp)
        arrays = (self.x_rp, self.x_inc, self.x_w, host_masses)
        if np.ndim(host_masses) == 0:
            rps, incs, argps = _prepare("TTP", block, N, arrays, M_s=host_masses, R_s=0.0,
                                        Teff=0.0, x_rp=self.x_rp, x_inc=self.x_inc,
                                        x_w=self.x_w, flatpriors=flatpriors)
        else:
            rps, incs, argps = _hostpar.pmap_block(block, N, *arrays)
        return rps, incs, self.eccs, argps


def _draw_planet(N, host_masses, flatpriors, P_mean):
    return _PlanetDraws(N, P_mean).finish(host_masses, flatpriors)


class _BinaryDraws:
    """Same for a stellar companion: inc, q, ecc, argp."""

    def __init__(self, N, P_mean):
        self.P_mean = P_mean
        self.x_inc = _fastrng.rand(N)
        self.x_q = _fastrng.rand(N)
        self.eccs = _draw_ecc(N, False, P_mean)      # deviates until transform() has run
        self.x_w = _fastrng.rand(N)

    def transform(self, x_inc, x_q, x_e, x_w, M_s):
        """(incs, qs, argps) of a chunk of deviates; the chunk of self.eccs becomes
        eccentricities in place."""
        _ecc_binary(x_e, self.P_mean)
        return sample_inc(x_inc), sample_q(x_q, M_s), sample_w(x_w)

    def finish(self, M_s):
        incs, qs, argps = _hostpar.pmap_block(
            lambda x_inc, x_q, x_e, x_w: self.transform(x_inc, x_q, x_e, x_w, M_s),
            len(self.x_inc), self.x_inc, self.x_q, self.eccs, self.x_w)
        return incs, qs, self.eccs, argps


class _CompanionDraw:
    """Mass ratios of bound companions: one uniform draw (transformed later) or, with a MOLUSC
    table, no draw at all (e.g. :455-464)."""

    def __init__(self, N, molusc_file):
        self.N, self.molusc_file = N, molusc_file
        self.x = _fastrng.rand(N) if molusc_file is None else None

    def finish(self, M_s):
        if self.molusc_file is None:
            return sample_q_companion(self.x, M_s)
        q = molusc_q(M_s, self.molusc_file)
        # zero-padded to N draws; a table with more than N rows raises, as in the reference
        return np.pad(q, (0, self.N - len(q)))

    def column(self, M_s):
        """What a scenario's block gets per draw: the deviates (the block applies `transform`)
        or, with a MOLUSC table, the mass ratios themselves."""
        return self.x if self.molusc_file is None else self.finish(M_s)

    def transform(self, col, M_s):
        return sample_q_companion(col, M_s) if self.molusc_file is None else col


def molusc_q(M_s, molusc_file):
    """Mass ratios of the bound companions a MOLUSC table lists with a(1 - e) > 10 AU, raised to
    at least 0.1 / M_s (e.g. :455-464)."""
    df = read_csv(molusc_file)
    sma = df["semi-major axis(AU)"].values
    e = df["eccentricity"].values
    # copy: pandas >= 3 hands out read-only views (the reference assigns into .values)
    q = np.array(df[sma * (1 - e) > 10]["mass ratio"].values, dtype=float)
    q[q < 0.1 / M_s] = 0.1 / M_s
    return q


def _fluxratio(masses, M_s, filt="TESS"):
    f = flux_relation(masses, filt)
    return f / (f + flux_relation(np.array([M_s]), filt))


def _clip_prior(lnprior, delta_mags):
    lnprior[lnprior > 0.0] = 0.0
    lnprior[delta_mags > 0.0] = -np.inf
    return lnprior


def _bound_prior(prior_fn, M_s, plx, N, molusc_file, contrast_curve_file, fr_tess, fr_cc_fn):
    """Companion prior of the P*/S* scenarios (e.g. :478-509).  fr_tess: flux-ratio term in the
    TESS band; fr_cc_fn(): the same term in the contrast-curve band (evaluated lazily)."""
    if molusc_file is not None:
        return np.zeros(N)
    if contrast_curve_file is None:
        delta_mags = 2.5 * np.log10(fr_tess)
        lnprior = prior_fn(M_s, plx, np.abs(delta_mags), np.array([2.2]), np.array([1.0]))
    else:
        delta_mags = 2.5 * np.log10(fr_cc_fn())
        separations, contrasts = file_to_contrast_curve(contrast_curve_file)
        lnprior = prior_fn(M_s, plx, np.abs(delta_mags), separations, contrasts)
    return _clip_prior(lnprior, delta_mags)


class _Background:
    """TRILEGAL population behind the target (e.g. :1452-1461)."""

    def __init__(self, trilegal_fname, Tmag, Jmag, Hmag, Kmag):
        (self.Tmags, self.masses, self.loggs, self.Teffs, self.Zs, Jm, Hm, Km) = \
            trilegal_results(trilegal_fname, Tmag)
        self.delta = {"T": Tmag - self.Tmags, "J": Jmag - Jm, "H": Hmag - Hm, "K": Kmag - Km}
        self.fluxratios = 10 ** (self.delta["T"] / 2.5) / (1 + 10 ** (self.delta["T"] / 2.5))
        self.N_comp = self.Tmags.shape[0]

    def band(self, filt):
        return self.delta[filt] if filt in ("J", "H", "K") else self.delta["T"]

    def fluxratios_in(self, filt):
        d = self.band(filt)
        return 10 ** (d / 2.5) / (1 + 10 ** (d / 2.5))

    def radii(self):
        return np.sqrt(G * self.masses * Msun / 10 ** self.loggs) / Rsun


def _background_prior(bg, N, contrast_curve_file, dmag_tess, dmag_cc):
    """Chance-alignment prior of the D*/B* scenarios (e.g. :1466-1492)."""
    if contrast_curve_file is None:
        lnprior = np.full(N, np.log((bg.N_comp / 0.1) * (1 / 3600) ** 2 * 2.2 ** 2))
        return _clip_prior(lnprior, dmag_tess)
    separations, contrasts = file_to_contrast_curve(contrast_curve_file)
    lnprior = lnprior_background(bg.N_comp, np.abs(dmag_cc), separations, contrasts)
    return _clip_prior(lnprior, dmag_cc)


class ScenarioResult(dict):
    """The reference's result dictionary (same keys) with diagnostics as attributes: n_pass
    (draws surviving the geometric mask) and n_evaluated (draws with a finite lnL; when it is
    below 100 the tail of the best-draw table holds draws of zero weight in arbitrary order, as
    in the reference).  Inside `triceratops_b200.mc_errors()` also the Monte-Carlo error of
    lnZ: N (draws), s2 (second moment of the weights, _numerics), lnZ_err (standard error of
    lnZ) and ess (effective sample size); None otherwise."""
    n_pass = 0
    n_evaluated = 0
    N = None
    s2 = None
    lnZ_err = None
    ess = None
    # (m, s, s2, n_finite, n_posinf) of the branch and (lnL, draw index) of the table's finite
    # rows: what calc_probs merges when it refines a scenario with more draws
    record = None
    top = None
    # inside `triceratops_b200.posterior_samples(K)`: the K posterior samples as a table (the
    # keys of RESULT_KEYS plus `draw`, the global draw index; 0 rows when the posterior is
    # empty) and their total weight relative to exp(record[0]); None otherwise
    posterior = None
    post_total = None
    # inside `triceratops_b200.record_coords()` (device sampler, with posterior samples): the
    # samples' coordinates in the sampler's unit cube, [K, 6] (NaN in slots the scenario does
    # not draw); None otherwise
    post_coords = None

    def set_moments(self, N, record, top):
        """Attach the branch's evidence record; the error fields when it carries s2."""
        self.N, self.record, self.top = int(N), tuple(record), top
        if record[2] is not None:
            self.s2 = float(record[2])
            self.lnZ_err, self.ess, _ = mc_error(N, record[0], record[1], record[2], record[3],
                                                 record[4])


def branch_result(br, table, posterior=None):
    """ScenarioResult of a merged branch (_dispatch.Branch) with the best-draw table `table` and,
    with posterior samples, their rows `posterior` (dicts of RESULT_KEYS columns; by default the
    rows that travelled with the samples, br.post_rows)."""
    out = ScenarioResult(table, lnZ=br.lnZ)
    out.n_pass, out.n_evaluated = br.n_pass, br.n_evaluated
    out.set_moments(br.N, br.record, (br.vals, np.asarray(br.idx)[:len(br.vals)]))
    if br.post_idx is not None:
        if posterior is None:
            posterior = {k: br.post_rows[:, i] for i, k in enumerate(RESULT_KEYS)}
        out.posterior = dict(posterior, draw=br.post_idx)
        out.post_total = br.post_total
    return out


def _result(br, twin, M_host, R_host, u1, u2, P, mtot, incs, eccs, argps, cfr, **body):
    """ScenarioResult of one branch: rows br.idx (and br.post_idx) of the scenario's columns;
    `body` holds the per-draw columns of the transiting body (R_p, or M_EB, R_EB and
    fluxratio_EB)."""
    def table(idx, n_zeros):
        return result_table(
            n_zeros, twin, _take(M_host, idx), _take(R_host, idx), _take(u1, idx),
            _take(u2, idx), _take(P, idx), _take(mtot, idx), incs[idx], eccs[idx], argps[idx],
            fluxratio_comp=_take(cfr, idx) if np.ndim(cfr) else None,
            **{k: v[idx] for k, v in body.items()})
    p = br.post_idx
    return branch_result(br, table(br.idx, N_SAMPLES), None if p is None else table(p, len(p)))


def _run_tp(N, M_host, R_host, u1, u2, P, mtot, rps, incs, eccs, argps, cfr, lnprior,
            extra_mask, companion_is_host):
    pb = _dispatch.submit_tp(N, rps, P, incs, eccs, argps, mtot, R_host, u1, u2, cfr,
                             lnprior=lnprior, extra_mask=extra_mask,
                             companion_is_host=companion_is_host)
    return _dispatch.deliver(lambda: _result(pb.finish(), False, M_host, R_host, u1, u2, P, mtot,
                                             incs, eccs, argps, cfr, R_p=rps), pb.prepare)


def _run_eb(N, M_host, R_host, u1, u2, P, mtot, incs, qs, eccs, argps, masses, radii,
            fluxratios, cfr, lnprior, extra_mask, companion_is_host, scalar_loop=False):
    pb = _dispatch.submit_eb(N, radii, fluxratios, qs, P, incs, eccs, argps, mtot, R_host,
                             u1, u2, cfr, lnprior=lnprior, extra_mask=extra_mask,
                             companion_is_host=companion_is_host, scalar_loop=scalar_loop)
    common = (M_host, R_host, u1, u2, P, mtot, incs, eccs, argps, cfr)
    body = dict(M_EB=masses, R_EB=radii, fluxratio_EB=fluxratios)
    return (_dispatch.deliver(lambda: _result(pb.finish()[0], False, *common, **body),
                              pb.prepare),
            _dispatch.deliver(lambda: _result(pb.finish()[1], True, *common, **body),
                              pb.prepare))


# ------------------------------------------------------------------- target-star scenarios
@_device_sampler_twin
def lnZ_TTP(time: np.ndarray, flux: np.ndarray, sigma: float,
            P_orb: float, M_s: float, R_s: float, Teff: float,
            Z: float, N: int = 1000000, parallel: bool = False,
            mission: str = "TESS", flatpriors: bool = False,
            exptime: float = 0.00139, nsamples: int = 20):
    """Transiting planet on the target star (marginal_likelihoods.py:39-172).  Also used for a
    nearby star (NTP) by calc_probs."""
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    u1, u2 = grid_for(mission).nearest(Z, Teff, _logg(M_s, R_s))
    draws = _PlanetDraws(N, P_mean)
    _dispatch.rng_done()
    rps, incs, eccs, argps = draws.finish(M_s, flatpriors)
    return _run_tp(N, M_s, R_s, u1, u2, P, M_s, rps, incs, eccs, argps, 0.0, None, None, False)


def _draw_binary(N, M_s, P_mean):
    return _BinaryDraws(N, P_mean).finish(M_s)


@_device_sampler_twin
def lnZ_TEB(time: np.ndarray, flux: np.ndarray, sigma: float,
            P_orb: float, M_s: float, R_s: float, Teff: float,
            Z: float, N: int = 1000000, parallel: bool = False,
            mission: str = "TESS", flatpriors: bool = False,
            exptime: float = 0.00139, nsamples: int = 20):
    """Eclipsing binary on the target star, periods P and 2P (marginal_likelihoods.py:175-383).
    Also used for a nearby star (NEB, NEBx2P) by calc_probs."""
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    u1, u2 = grid_for(mission).nearest(Z, Teff, _logg(M_s, R_s))
    draws = _BinaryDraws(N, P_mean)
    _dispatch.rng_done()

    def block(x_inc, x_q, x_e, x_w):
        incs, qs, argps = draws.transform(x_inc, x_q, x_e, x_w, M_s)
        masses = qs * M_s
        radii, _ = stellar_relations(masses, np.full(len(qs), R_s), np.full(len(qs), Teff))
        return incs, qs, argps, masses, radii, _fluxratio(masses, M_s), M_s + masses

    incs, qs, argps, masses, radii, fluxratios, mtot = _prepare(
        "TEB", block, N, (draws.x_inc, draws.x_q, draws.eccs, draws.x_w), M_s=M_s, R_s=R_s,
        Teff=Teff, x_inc=draws.x_inc, x_q=draws.x_q, x_e=draws.eccs, x_w=draws.x_w,
        P_mean=P_mean)
    return _run_eb(N, M_s, R_s, u1, u2, P, mtot, incs, qs, draws.eccs, argps, masses, radii,
                   fluxratios, 0.0, None, None, False, scalar_loop=not parallel)


# ---------------------------------------------------------------- bound-companion scenarios
@_device_sampler_twin
def lnZ_PTP(time: np.ndarray, flux: np.ndarray, sigma: float,
            P_orb: float, M_s: float, R_s: float, Teff: float,
            Z: float, plx: float, contrast_curve_file: str = None,
            filt: str = "TESS",
            N: int = 1000000, parallel: bool = False,
            mission: str = "TESS", flatpriors: bool = False,
            exptime: float = 0.00139, nsamples: int = 20,
            molusc_file: str = None):
    """Planet on the target, diluted by an unresolved bound companion (:386-586)."""
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    u1, u2 = grid_for(mission).nearest(Z, Teff, _logg(M_s, R_s))
    # all draws first, in the reference's order (q_comp, rp, inc, ecc, argp); what follows is
    # deterministic and may overlap the next scenario's draws
    comp, draws = _CompanionDraw(N, molusc_file), _PlanetDraws(N, P_mean)
    _dispatch.rng_done()

    def block(c_comp, x_rp, x_inc, x_w):
        qs_comp = comp.transform(c_comp, M_s)
        rps, incs, argps = draws.transform(x_rp, x_inc, x_w, M_s, flatpriors)
        masses_comp = qs_comp * M_s
        fluxratios_comp = _fluxratio(masses_comp, M_s)

        def cc_term():
            fr = _fluxratio(masses_comp, M_s, filt)
            return fr / (1 - fr)

        lnprior = _bound_prior(lnprior_bound_TP, M_s, plx, len(qs_comp), molusc_file,
                               contrast_curve_file, fluxratios_comp / (1 - fluxratios_comp),
                               cc_term)
        return rps, incs, argps, fluxratios_comp, lnprior, qs_comp != 0.0

    c_comp = comp.column(M_s)
    rps, incs, argps, fluxratios_comp, lnprior, extra = _prepare(
        "PTP", block, N, (c_comp, draws.x_rp, draws.x_inc, draws.x_w), M_s=M_s, R_s=R_s,
        Teff=Teff, c_comp=c_comp, x_rp=draws.x_rp, x_inc=draws.x_inc, x_w=draws.x_w,
        flatpriors=flatpriors, molusc=molusc_file is not None, filt=filt,
        contrast_curve_file=contrast_curve_file, plx=plx, bound_kind="TP")
    return _run_tp(N, M_s, R_s, u1, u2, P, M_s, rps, incs, draws.eccs, argps, fluxratios_comp,
                   lnprior, extra, False)


@_device_sampler_twin
def lnZ_PEB(time: np.ndarray, flux: np.ndarray, sigma: float,
            P_orb: float, M_s: float, R_s: float, Teff: float,
            Z: float, plx: float, contrast_curve_file: str = None,
            filt: str = "TESS",
            N: int = 1000000, parallel: bool = False,
            mission: str = "TESS", flatpriors: bool = False,
            exptime: float = 0.00139, nsamples: int = 20,
            molusc_file: str = None):
    """EB on the target, diluted by an unresolved bound companion (:589-866)."""
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    u1, u2 = grid_for(mission).nearest(Z, Teff, _logg(M_s, R_s))
    draws, comp = _BinaryDraws(N, P_mean), _CompanionDraw(N, molusc_file)
    _dispatch.rng_done()

    def block(c_comp, x_inc, x_q, x_e, x_w):
        qs_comp = comp.transform(c_comp, M_s)
        incs, qs, argps = draws.transform(x_inc, x_q, x_e, x_w, M_s)
        masses = qs * M_s
        radii, _ = stellar_relations(masses, np.full(len(qs), R_s), np.full(len(qs), Teff))
        fluxratios = _fluxratio(masses, M_s)
        masses_comp = qs_comp * M_s
        fluxratios_comp = _fluxratio(masses_comp, M_s)

        def cc_term():
            fr = _fluxratio(masses_comp, M_s, filt)
            return fr / (1 - fr)

        lnprior = _bound_prior(lnprior_bound_EB, M_s, plx, len(qs), molusc_file,
                               contrast_curve_file, fluxratios_comp / (1 - fluxratios_comp),
                               cc_term)
        return (incs, qs, argps, masses, radii, fluxratios, M_s + masses, fluxratios_comp,
                lnprior, qs_comp != 0.0)

    c_comp = comp.column(M_s)
    (incs, qs, argps, masses, radii, fluxratios, mtot, fluxratios_comp, lnprior,
     extra) = _prepare(
        "PEB", block, N, (c_comp, draws.x_inc, draws.x_q, draws.eccs, draws.x_w), M_s=M_s,
        R_s=R_s, Teff=Teff, c_comp=c_comp, x_inc=draws.x_inc, x_q=draws.x_q, x_e=draws.eccs,
        x_w=draws.x_w, P_mean=P_mean, molusc=molusc_file is not None, filt=filt,
        contrast_curve_file=contrast_curve_file, plx=plx, bound_kind="EB")
    return _run_eb(N, M_s, R_s, u1, u2, P, mtot, incs, qs, draws.eccs, argps, masses, radii,
                   fluxratios, fluxratios_comp, lnprior, extra, False,
                   scalar_loop=not parallel)


def _companion_stars(N, M_s, R_s, Teff, Z, mission, qs_comp, Teff_cap):
    """Properties of the drawn bound companions when THEY host the event (:927-972)."""
    masses_comp = qs_comp * M_s
    radii_comp, Teffs_comp = stellar_relations(masses_comp, np.full(len(qs_comp), R_s),
                                               np.full(len(qs_comp), Teff))
    loggs_comp = np.log10(G * (masses_comp * Msun) / (radii_comp * Rsun) ** 2)
    fluxratios_comp = _fluxratio(masses_comp, M_s)
    u1s, u2s = grid_for(mission).at_Z_rounded(Z, Teffs_comp, loggs_comp, Teff_cap)
    return masses_comp, radii_comp, Teffs_comp, fluxratios_comp, u1s, u2s


@_device_sampler_twin
def lnZ_STP(time: np.ndarray, flux: np.ndarray, sigma: float,
            P_orb: float, M_s: float, R_s: float, Teff: float, Z: float,
            plx: float, contrast_curve_file: str = None,
            filt: str = "TESS",
            N: int = 1000000, parallel: bool = False,
            mission: str = "TESS", flatpriors: bool = False,
            exptime: float = 0.00139, nsamples: int = 20,
            molusc_file: str = None):
    """Planet on an unresolved bound companion of the target (:869-1077)."""
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    # draws first (q_comp, then the planet around a host of mass q_comp M_s), see lnZ_PTP
    comp, draws = _CompanionDraw(N, molusc_file), _PlanetDraws(N, P_mean)
    _dispatch.rng_done()

    def block(c_comp, x_rp, x_inc, x_w):
        qs_comp = comp.transform(c_comp, M_s)
        rps, incs, argps = draws.transform(x_rp, x_inc, x_w, qs_comp * M_s, flatpriors)
        (masses_comp, radii_comp, _, fluxratios_comp, u1s, u2s) = _companion_stars(
            len(qs_comp), M_s, R_s, Teff, Z, mission, qs_comp, 10000)

        def cc_term():
            fr = _fluxratio(masses_comp, M_s, filt)
            return fr / (1 - fr)

        lnprior = _bound_prior(lnprior_bound_TP, M_s, plx, len(qs_comp), molusc_file,
                               contrast_curve_file, fluxratios_comp / (1 - fluxratios_comp),
                               cc_term)
        return (rps, incs, argps, masses_comp, radii_comp, fluxratios_comp, u1s, u2s, lnprior,
                qs_comp != 0.0)

    c_comp = comp.column(M_s)
    (rps, incs, argps, masses_comp, radii_comp, fluxratios_comp, u1s, u2s, lnprior,
     extra) = _prepare(
        "STP", block, N, (c_comp, draws.x_rp, draws.x_inc, draws.x_w), M_s=M_s, R_s=R_s,
        Teff=Teff, c_comp=c_comp, x_rp=draws.x_rp, x_inc=draws.x_inc, x_w=draws.x_w,
        flatpriors=flatpriors, molusc=molusc_file is not None, filt=filt,
        contrast_curve_file=contrast_curve_file, plx=plx, bound_kind="TP",
        ldc_grid=grid_for(mission), Z=Z, ldc_cap=10000)
    return _run_tp(N, masses_comp, radii_comp, u1s, u2s, P, masses_comp, rps, incs, draws.eccs,
                   argps, fluxratios_comp, lnprior, extra, True)


@_device_sampler_twin
def lnZ_SEB(time: np.ndarray, flux: np.ndarray, sigma: float,
            P_orb: float, M_s: float, R_s: float, Teff: float,
            Z: float, plx: float, contrast_curve_file: str = None,
            filt: str = "TESS",
            N: int = 1000000, parallel: bool = False,
            mission: str = "TESS", flatpriors: bool = False,
            exptime: float = 0.00139, nsamples: int = 20,
            molusc_file: str = None):
    """EB on an unresolved bound companion of the target (:1080-1376)."""
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    draws, comp = _BinaryDraws(N, P_mean), _CompanionDraw(N, molusc_file)
    _dispatch.rng_done()

    def block(c_comp, x_inc, x_q, x_e, x_w):
        qs_comp = comp.transform(c_comp, M_s)
        incs, qs, argps = draws.transform(x_inc, x_q, x_e, x_w, M_s)
        # Teff clamp of 13000 K (grid stops at 10000 K) as in the reference, :1181
        (masses_comp, radii_comp, Teffs_comp, fluxratios_comp, u1s, u2s) = _companion_stars(
            len(qs), M_s, R_s, Teff, Z, mission, qs_comp, 13000)
        masses = qs * masses_comp
        radii, _ = stellar_relations(masses, radii_comp, Teffs_comp)
        fluxratios = _fluxratio(masses, M_s)

        def cc_term():
            fr = _fluxratio(masses, M_s, filt)
            fr_comp = _fluxratio(masses_comp, M_s, filt)
            return (fr_comp / (1 - fr_comp)) + (fr / (1 - fr))

        lnprior = _bound_prior(lnprior_bound_EB, M_s, plx, len(qs), molusc_file,
                               contrast_curve_file,
                               (fluxratios_comp / (1 - fluxratios_comp))
                               + (fluxratios / (1 - fluxratios)), cc_term)
        return (incs, qs, argps, masses_comp, radii_comp, u1s, u2s, masses_comp + masses, masses,
                radii, fluxratios, fluxratios_comp, lnprior, qs_comp != 0.0)

    c_comp = comp.column(M_s)
    (incs, qs, argps, masses_comp, radii_comp, u1s, u2s, mtot, masses, radii, fluxratios,
     fluxratios_comp, lnprior, extra) = _prepare(
        "SEB", block, N, (c_comp, draws.x_inc, draws.x_q, draws.eccs, draws.x_w), M_s=M_s,
        R_s=R_s, Teff=Teff, c_comp=c_comp, x_inc=draws.x_inc, x_q=draws.x_q, x_e=draws.eccs,
        x_w=draws.x_w, P_mean=P_mean, molusc=molusc_file is not None, filt=filt,
        contrast_curve_file=contrast_curve_file, plx=plx, bound_kind="EB",
        ldc_grid=grid_for(mission), Z=Z, ldc_cap=13000)
    return _run_eb(N, masses_comp, radii_comp, u1s, u2s, P, mtot, incs, qs, draws.eccs,
                   argps, masses, radii, fluxratios, fluxratios_comp, lnprior, extra,
                   True, scalar_loop=not parallel)


# --------------------------------------------------------------------- background scenarios
@_device_sampler_twin
def lnZ_DTP(time: np.ndarray, flux: np.ndarray, sigma: float,
            P_orb: float, M_s: float, R_s: float, Teff: float,
            Z: float, Tmag: float, Jmag: float, Hmag: float,
            Kmag: float, trilegal_fname: str,
            contrast_curve_file: str = None, filt: str = "TESS",
            N: int = 1000000, parallel: bool = False,
            mission: str = "TESS", flatpriors: bool = False,
            exptime: float = 0.00139, nsamples: int = 20):
    """Planet on the target, diluted by a chance-aligned background star (:1379-1568)."""
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    u1, u2 = grid_for(mission).nearest(Z, Teff, _logg(M_s, R_s))
    bg = _Background(trilegal_fname, Tmag, Jmag, Hmag, Kmag)
    idxs = _fastrng.randint(0, bg.N_comp - 1, N)     # upper bound N_comp-1, as :1463
    draws = _PlanetDraws(N, P_mean)
    _dispatch.rng_done()
    band = bg.band(filt)

    def block(idxs, x_rp, x_inc, x_w):
        rps, incs, argps = draws.transform(x_rp, x_inc, x_w, M_s, flatpriors)
        cfr = _take(bg.fluxratios, idxs)
        lnprior = _background_prior(bg, len(idxs), contrast_curve_file,
                                    2.5 * np.log10(cfr / (1 - cfr)), _take(band, idxs))
        return rps, incs, argps, cfr, lnprior

    rps, incs, argps, cfr, lnprior = _prepare(
        "DTP", block, N, (idxs, draws.x_rp, draws.x_inc, draws.x_w), M_s=M_s, R_s=R_s,
        Teff=Teff, idxs=idxs, x_rp=draws.x_rp, x_inc=draws.x_inc, x_w=draws.x_w,
        flatpriors=flatpriors, contrast_curve_file=contrast_curve_file, N_comp=bg.N_comp,
        population=_blocks.Population(None, None, None, None, bg.fluxratios, band, None, None,
                                      None, None))
    return _run_tp(N, M_s, R_s, u1, u2, P, M_s, rps, incs, draws.eccs, argps, cfr, lnprior,
                   None, False)


@_device_sampler_twin
def lnZ_DEB(time: np.ndarray, flux: np.ndarray, sigma: float,
            P_orb: float, M_s: float, R_s: float, Teff: float,
            Z: float, Tmag: float, Jmag: float, Hmag: float,
            Kmag: float, trilegal_fname: str,
            contrast_curve_file: str = None, filt: str = "TESS",
            N: int = 1000000, parallel: bool = False,
            mission: str = "TESS", flatpriors: bool = False,
            exptime: float = 0.00139, nsamples: int = 20):
    """EB on the target, diluted by a chance-aligned background star (:1571-1837)."""
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    u1, u2 = grid_for(mission).nearest(Z, Teff, _logg(M_s, R_s))
    draws = _BinaryDraws(N, P_mean)
    bg = _Background(trilegal_fname, Tmag, Jmag, Hmag, Kmag)
    idxs = _fastrng.randint(0, bg.N_comp - 1, N)     # :1672
    _dispatch.rng_done()
    band = bg.band(filt)

    def block(idxs, x_inc, x_q, x_e, x_w):
        incs, qs, argps = draws.transform(x_inc, x_q, x_e, x_w, M_s)
        masses = qs * M_s
        radii, _ = stellar_relations(masses, np.full(len(qs), R_s), np.full(len(qs), Teff))
        fluxratios = _fluxratio(masses, M_s)
        cfr = _take(bg.fluxratios, idxs)
        lnprior = _background_prior(bg, len(idxs), contrast_curve_file,
                                    2.5 * np.log10(cfr / (1 - cfr)), _take(band, idxs))
        return incs, qs, argps, masses, radii, fluxratios, M_s + masses, cfr, lnprior

    incs, qs, argps, masses, radii, fluxratios, mtot, cfr, lnprior = _prepare(
        "DEB", block, N, (idxs, draws.x_inc, draws.x_q, draws.eccs, draws.x_w), M_s=M_s,
        R_s=R_s, Teff=Teff, idxs=idxs, x_inc=draws.x_inc, x_q=draws.x_q, x_e=draws.eccs,
        x_w=draws.x_w, P_mean=P_mean, contrast_curve_file=contrast_curve_file,
        N_comp=bg.N_comp,
        population=_blocks.Population(None, None, None, None, bg.fluxratios, band, None, None,
                                      None, None))
    return _run_eb(N, M_s, R_s, u1, u2, P, mtot, incs, qs, draws.eccs, argps, masses, radii,
                   fluxratios, cfr, lnprior, None, False, scalar_loop=not parallel)


@_device_sampler_twin
def lnZ_BTP(time: np.ndarray, flux: np.ndarray, sigma: float,
            P_orb: float, M_s: float, R_s: float, Teff: float,
            Tmag: float, Jmag: float, Hmag: float, Kmag: float,
            trilegal_fname: str,
            contrast_curve_file: str = None, filt: str = "TESS",
            N: int = 1000000, parallel: bool = False,
            mission: str = "TESS", flatpriors: bool = False,
            exptime: float = 0.00139, nsamples: int = 20):
    """Planet on a chance-aligned background star (:1840-2035)."""
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    bg = _Background(trilegal_fname, Tmag, Jmag, Hmag, Kmag)
    idxs = _fastrng.randint(0, bg.N_comp, N)         # :1926
    draws = _PlanetDraws(N, P_mean)
    _dispatch.rng_done()
    radii_comp = bg.radii()
    u1s_comp, u2s_comp = grid_for(mission).nearest_each(bg.Teffs, bg.loggs, bg.Zs)
    band = bg.band(filt)

    def block(idxs, x_rp, x_inc, x_w):
        host_masses = _take(bg.masses, idxs)
        rps, incs, argps = draws.transform(x_rp, x_inc, x_w, host_masses, flatpriors)
        cfr = _take(bg.fluxratios, idxs)
        lnprior = _background_prior(bg, len(idxs), contrast_curve_file,
                                    2.5 * np.log10(cfr / (1 - cfr)), _take(band, idxs))
        extra = (_take(bg.loggs, idxs) >= 3.5) & (_take(bg.Teffs, idxs) <= 10000)
        return (host_masses, rps, incs, argps, cfr, lnprior, _take(radii_comp, idxs),
                _take(u1s_comp, idxs), _take(u2s_comp, idxs), extra)

    (host_masses, rps, incs, argps, cfr, lnprior, host_radii, u1s, u2s, extra) = _prepare(
        "BTP", block, N, (idxs, draws.x_rp, draws.x_inc, draws.x_w), M_s=M_s, R_s=R_s,
        Teff=Teff, idxs=idxs, x_rp=draws.x_rp, x_inc=draws.x_inc, x_w=draws.x_w,
        flatpriors=flatpriors, contrast_curve_file=contrast_curve_file, N_comp=bg.N_comp,
        population=_blocks.Population(bg.masses, radii_comp, bg.Teffs, bg.loggs, bg.fluxratios,
                                      band, None, None, u1s_comp, u2s_comp))
    return _run_tp(N, host_masses, host_radii, u1s, u2s, P, host_masses, rps, incs, draws.eccs,
                   argps, cfr, lnprior, extra, True)


@_device_sampler_twin
def lnZ_BEB(time: np.ndarray, flux: np.ndarray, sigma: float,
            P_orb: float, M_s: float, R_s: float, Teff: float,
            Tmag: float, Jmag: float, Hmag: float, Kmag: float,
            trilegal_fname: str,
            contrast_curve_file: str = None, filt: str = "TESS",
            N: int = 1000000, parallel: bool = False,
            mission: str = "TESS", flatpriors: bool = False,
            exptime: float = 0.00139, nsamples: int = 20):
    """EB on a chance-aligned background star (:2038-2362)."""
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    x_inc, x_q = _fastrng.rand(N), _fastrng.rand(N)
    _fastrng.skip(N)                                  # q_comp: drawn and never used, as :2089
    eccs = _draw_ecc(N, False, P_mean)
    x_w = _fastrng.rand(N)
    bg = _Background(trilegal_fname, Tmag, Jmag, Hmag, Kmag)
    idxs = _fastrng.randint(0, bg.N_comp, N)         # :2139
    _dispatch.rng_done()
    radii_comp = bg.radii()
    u1s_comp, u2s_comp = grid_for(mission).nearest_each(bg.Teffs, bg.loggs, bg.Zs)
    # "TESS" and "Vis" share one flux relation and use the TESS-band magnitudes
    cc_band = filt if filt in ("J", "H", "K") else "TESS"
    band_fluxratios = {b: bg.fluxratios_in(b) for b in ("TESS", cc_band)}

    def block(idxs, x_inc, x_q, x_e, x_w):
        _ecc_binary(x_e, P_mean)
        incs, qs, argps = sample_inc(x_inc), sample_q(x_q, M_s), sample_w(x_w)
        host_masses = _take(bg.masses, idxs)
        host_radii = _take(radii_comp, idxs)
        cfr = _take(bg.fluxratios, idxs)
        masses = qs * host_masses
        radii, _ = stellar_relations(masses, host_radii, _take(bg.Teffs, idxs))

        def distance_corrected(band):
            # EB flux ratio scaled from "bound at the target's distance" to the background
            # star's actual brightness (:2147-2182)
            cfr_band = _take(band_fluxratios[band], idxs)
            bound = _fluxratio(host_masses, M_s, band)
            return _fluxratio(masses, M_s, band) * (cfr_band / bound), cfr_band

        fluxratios, _ = distance_corrected("TESS")
        if contrast_curve_file is None:
            dmag = 2.5 * np.log10((cfr / (1 - cfr)) + (fluxratios / (1 - fluxratios)))
            lnprior = _background_prior(bg, len(idxs), None, dmag, None)
        else:
            fr_cc, cfr_cc = distance_corrected(cc_band)
            dmag = 2.5 * np.log10((cfr_cc / (1 - cfr_cc)) + (fr_cc / (1 - fr_cc)))
            lnprior = _background_prior(bg, len(idxs), contrast_curve_file, None, dmag)
        extra = (_take(bg.loggs, idxs) >= 3.5) & (_take(bg.Teffs, idxs) <= 10000)
        return (incs, qs, argps, host_masses, host_radii, _take(u1s_comp, idxs),
                _take(u2s_comp, idxs), host_masses + masses, masses, radii, fluxratios, cfr,
                lnprior, extra)

    (incs, qs, argps, host_masses, host_radii, u1s, u2s, mtot, masses, radii, fluxratios, cfr,
     lnprior, extra) = _prepare(
        "BEB", block, N, (idxs, x_inc, x_q, eccs, x_w), M_s=M_s, R_s=R_s, Teff=Teff, idxs=idxs,
        x_inc=x_inc, x_q=x_q, x_e=eccs, x_w=x_w, P_mean=P_mean, filt=filt,
        contrast_curve_file=contrast_curve_file, N_comp=bg.N_comp,
        population=_blocks.Population(bg.masses, radii_comp, bg.Teffs, bg.loggs, bg.fluxratios,
                                      None, band_fluxratios["TESS"], band_fluxratios[cc_band],
                                      u1s_comp, u2s_comp))
    return _run_eb(N, host_masses, host_radii, u1s, u2s, P, mtot, incs, qs, eccs, argps, masses,
                   radii, fluxratios, cfr, lnprior, extra, True, scalar_loop=not parallel)


# ------------------------------------------------- nearby stars of unknown / evolved nature
# The reference defines these four but never calls them (marginal_likelihoods.py:2365-3178);
# they reuse the same two kernels.


class _PossibleHosts:
    """TRILEGAL stars within one magnitude of a nearby star of unknown properties (:2402-2415)."""

    def __init__(self, trilegal_fname, Tmag, mission):
        (Tmags, masses, loggs, Teffs, Zs, _, _, _) = trilegal_results(trilegal_fname, Tmag)
        near = (Tmag - 1 < Tmags) & (Tmags < Tmag + 1)
        self.masses, self.loggs, self.Teffs, self.Zs = (masses[near], loggs[near], Teffs[near],
                                                        Zs[near])
        self.radii = np.sqrt(G * self.masses * Msun / 10 ** self.loggs) / Rsun
        self.n = int(near.sum())
        self.u1s, self.u2s = grid_for(mission).nearest_each(self.Teffs, self.loggs, self.Zs)


def _no_hosts(with_b):
    # what the reference returns when no TRILEGAL star is similar enough (:2438-2454, :2648-2665)
    res = {k: 0 for k in RESULT_KEYS if with_b or k != 'b'}
    res['lnZ'] = -np.inf
    return res


def lnZ_NTP_unknown(time: np.ndarray, flux: np.ndarray, sigma: float,
                    P_orb: float, Tmag: float, trilegal_fname: str,
                    N: int = 1000000, parallel: bool = False,
                    mission: str = "TESS", flatpriors: bool = False,
                    exptime: float = 0.00139, nsamples: int = 20):
    """Planet on a nearby star of unknown properties, host drawn from the TRILEGAL stars of
    similar brightness (marginal_likelihoods.py:2365-2551)."""
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    hosts = _PossibleHosts(trilegal_fname, Tmag, mission)
    if hosts.n == 0:
        return _no_hosts(with_b=False)
    idxs = _fastrng.randint(0, hosts.n, N)
    host_masses = _take(hosts.masses, idxs)
    rps, incs, eccs, argps = _draw_planet(N, host_masses, flatpriors, P_mean)
    extra = (_take(hosts.loggs, idxs) >= 3.5) & (_take(hosts.Teffs, idxs) <= 10000)
    return _run_tp(N, host_masses, _take(hosts.radii, idxs), _take(hosts.u1s, idxs), _take(hosts.u2s, idxs), P,
                   host_masses, rps, incs, eccs, argps, 0.0, None, extra, False)


def lnZ_NEB_unknown(time: np.ndarray, flux: np.ndarray, sigma: float,
                    P_orb: float, Tmag: float, trilegal_fname: str,
                    N: int = 1000000, parallel: bool = False,
                    mission: str = "TESS", flatpriors: bool = False,
                    exptime: float = 0.00139, nsamples: int = 20):
    """EB on a nearby star of unknown properties (marginal_likelihoods.py:2554-2829)."""
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    incs, qs, eccs, argps = _draw_binary(N, 1.0, P_mean)       # sample_q with M_s = 1.0, :2593
    hosts = _PossibleHosts(trilegal_fname, Tmag, mission)
    if hosts.n == 0:
        return _no_hosts(with_b=True)                           # a single dict, as :2665
    idxs = _fastrng.randint(0, hosts.n, N)
    host_masses, host_radii = _take(hosts.masses, idxs), _take(hosts.radii, idxs)
    masses = qs * host_masses
    radii, _ = stellar_relations(masses, host_radii, _take(hosts.Teffs, idxs))
    f = flux_relation(masses)
    fluxratios = f / (f + flux_relation(host_masses))
    extra = (_take(hosts.loggs, idxs) >= 3.5) & (_take(hosts.Teffs, idxs) <= 10000)
    return _run_eb(N, host_masses, host_radii, _take(hosts.u1s, idxs), _take(hosts.u2s, idxs), P,
                   host_masses + masses, incs, qs, eccs, argps, masses, radii, fluxratios, 0.0,
                   None, extra, False, scalar_loop=not parallel)


def _subgiant_mass(R_s):
    # M_s = (10**logg)*(R_s*Rsun)**2 / G / Msun with logg = 3.0     (:2877-2878)
    logg = 3.0
    return logg, (10 ** logg) * (R_s * Rsun) ** 2 / G / Msun


def lnZ_NTP_evolved(time: np.ndarray, flux: np.ndarray, sigma: float,
                    P_orb: float, R_s: float, Teff: float, Z: float,
                    N: int = 1000000, parallel: bool = False,
                    mission: str = "TESS", flatpriors: bool = False,
                    exptime: float = 0.00139, nsamples: int = 20):
    """Planet on a nearby subgiant (logg = 3) of radius R_s (marginal_likelihoods.py:2832-2966)."""
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    logg, M_s = _subgiant_mass(R_s)
    u1, u2 = grid_for(mission).nearest(Z, Teff, logg)
    rps, incs, eccs, argps = _draw_planet(N, np.full(N, M_s), flatpriors, P_mean)
    return _run_tp(N, M_s, R_s, u1, u2, P, M_s, rps, incs, eccs, argps, 0.0, None, None, False)


def lnZ_NEB_evolved(time: np.ndarray, flux: np.ndarray, sigma: float,
                    P_orb: float, R_s: float, Teff: float, Z: float,
                    N: int = 1000000, parallel: bool = False,
                    mission: str = "TESS", flatpriors: bool = False,
                    exptime: float = 0.00139, nsamples: int = 20):
    """EB on a nearby subgiant (marginal_likelihoods.py:2969-3178).

    Reference quirk kept: the q >= 0.95 branch models a twin of radius R_s (it passes the scalar
    R_s as R_EB, :3100, and uses 2 R_s in Ptra_twin, :3052) while reporting R_EB = R_s; the two
    branches therefore see different companion radii and are evaluated in two engine calls.
    """
    N = int(N)
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    P, P_mean = _periods(P_orb, N)
    logg, M_s = _subgiant_mass(R_s)
    u1, u2 = grid_for(mission).nearest(Z, Teff, logg)
    incs, qs, eccs, argps = _draw_binary(N, 1.0, P_mean)
    masses = qs * M_s
    radii, _ = stellar_relations(masses, np.full(N, R_s), np.full(N, Teff))
    fluxratios = _fluxratio(masses, M_s)
    common = (N, M_s, R_s, u1, u2, P, M_s + masses, incs, qs, eccs, argps, masses)
    res, _ = _run_eb(*common, radii, fluxratios, 0.0, None, None, False, scalar_loop=not parallel)
    _, res_twin = _run_eb(*common, np.full(N, float(R_s)), fluxratios, 0.0, None, None, False, scalar_loop=not parallel)
    return res, res_twin
