"""`target.calc_probs(...)`: the caller of the marginal-likelihood path, as a drop-in.

Mirrors the reference's triceratops/triceratops.py:673-1485 (calc_probs) with the same signature,
scenario table layout (15 target-star rows + 3 per nearby star with tdepth > 0), attributes
(`probs`, `lnZ`, `FPP`, `NFPP`, `FPP_degenerate`, `star_num`, `u1`, `u2`, `fluxratio_EB`,
`fluxratio_comp`) and warnings.

`calc_depths` (triceratops.py:559-671), which produces the `fluxratio` / `tdepth` columns
calc_probs reads, is included as host numpy.  The rest of the reference's `target` class --
TIC/Gaia/TessCut queries in __init__, plotting, star-table bookkeeping -- is outside this
package's scope (SURVEY.md section 2 rows 8-10): there is no network here, so a `target` is built
from a stars table the caller already has (the reference's `target.stars` DataFrame, e.g. saved
from an online session), optionally its `pix_coords`, and a saved TRILEGAL file.
"""
import collections
import contextlib
import functools
import sys
import warnings

import numpy as np
from pandas import DataFrame, concat
from scipy.special import ndtr

from . import _bufpool, _dispatch
from ._numerics import (_normalize_probabilities, mc_error, merge_posteriors,
                        probability_errors)
from .funcs import renorm_flux
from .marginal_likelihoods import (RESULT_KEYS, ScenarioResult, lnZ_BEB, lnZ_BTP, lnZ_DEB,
                                   lnZ_DTP, lnZ_PEB, lnZ_PTP, lnZ_SEB, lnZ_STP, lnZ_TEB, lnZ_TTP)

_STAR_COLUMNS = ("ID", "Tmag", "Jmag", "Hmag", "Kmag", "ra", "dec", "mass", "rad", "Teff", "plx",
                 "fluxratio", "tdepth")

# scenario rows whose results may still be in flight while the next scenario is being drawn
_PIPELINE_DEPTH = 3

# (drop_scenario key, first row, star_num, scenario names) in the reference's order
# (triceratops.py:784-1332)
_TARGET_SCENARIOS = (
    ("TP", 0, 1, ("TP",)),
    ("EB", 1, 1, ("EB", "EBx2P")),
    ("PTP", 3, 1, ("PTP",)),
    ("PEB", 4, 1, ("PEB", "PEBx2P")),
    ("STP", 6, 2, ("STP",)),
    ("SEB", 7, 2, ("SEB", "SEBx2P")),
    ("DTP", 9, 1, ("DTP",)),
    ("DEB", 10, 1, ("DEB", "DEBx2P")),
    ("BTP", 12, 2, ("BTP",)),
    ("BEB", 13, 2, ("BEB", "BEBx2P")),
)


class target:
    def __init__(self, ID: int, sectors=None, search_radius: int = 10, mission: str = "TESS",
                 lightkurve_cache_dir=None, trilegal_fname=None, ra: float = None,
                 dec: float = None, verify_ssl: bool = True, stars: DataFrame = None,
                 pix_coords=None):
        """Offline constructor: same leading arguments as the reference (triceratops.py:42-45)
        plus `stars`, the table the reference would have assembled from TIC (one row per star,
        target first, columns ID, Tmag, Jmag, Hmag, Kmag, ra, dec, mass, rad, Teff, plx,
        fluxratio, tdepth).  `pix_coords` (optional, one [n_stars, 2] array of pixel positions
        per sector, the reference's `target.pix_coords`) enables `calc_depths`."""
        if mission != "TESS" and mission != "Kepler" and mission != "K2":
            raise ValueError("Introduced invalid mission: " + mission)
        if stars is None:
            raise NotImplementedError(
                "catalogue queries are outside triceratops_b200 (no network): pass the stars "
                "table as target(..., stars=DataFrame)")
        stars = stars.copy()
        if pix_coords is not None:
            for c in ("fluxratio", "tdepth"):       # filled by calc_depths
                if c not in stars.columns:
                    stars[c] = 0.0
        missing = [c for c in _STAR_COLUMNS if c not in stars.columns]
        if missing:
            raise ValueError("stars table lacks columns: " + ", ".join(missing))
        self.pix_coords = None if pix_coords is None else [np.asarray(p, float)
                                                           for p in pix_coords]
        self.ID = ID
        self.mission = mission
        self.sectors = sectors
        self.search_radius = search_radius
        self.N_pix = 2 * search_radius + 2
        self.stars = stars.reset_index(drop=True)
        self.trilegal_fname = trilegal_fname
        self.trilegal_url = None

    def calc_depths(self, tdepth: float, all_ap_pixels=None):
        """Flux ratio of every star inside the photometric aperture(s) and the transit depth
        each would need to cause the observed one (reference triceratops.py:559-671): circular
        Gaussian PSF of 0.75 px integrated analytically over each aperture pixel, averaged over
        apertures.  Fills stars["fluxratio"] and stars["tdepth"], the inputs of calc_probs."""
        if self.pix_coords is None:
            raise RuntimeError("calc_depths needs pix_coords (pass them to target())")
        if all_ap_pixels is None:
            print("No apertures provided, assuming 5x5 centered on target.")
            all_ap_pixels = []
            for pc in self.pix_coords:
                c = np.round(pc[0])
                all_ap_pixels.append(np.array([
                    np.repeat(np.arange(c[0] - 2, c[0] + 3, 1), 5),
                    np.tile(np.arange(c[1] - 2, c[1] + 3, 1), 5)]).T)
        sigma = 0.75
        Tmag = self.stars.Tmag.values
        A = 10 ** ((np.min(Tmag) - Tmag) / 2.5)        # flux relative to the brightest star
        ratios = np.zeros([len(all_ap_pixels), len(self.stars)])
        for k, pixels in enumerate(all_ap_pixels):
            pixels = np.array(pixels)
            mu = self.pix_coords[k]
            # separable pixel-box integral: [stars, pixels]
            gx = (ndtr((pixels[None, :, 0] + 0.5 - mu[:, None, 0]) / sigma)
                  - ndtr((pixels[None, :, 0] - 0.5 - mu[:, None, 0]) / sigma))
            gy = (ndtr((pixels[None, :, 1] + 0.5 - mu[:, None, 1]) / sigma)
                  - ndtr((pixels[None, :, 1] - 0.5 - mu[:, None, 1]) / sigma))
            rel = np.array([A[i] * np.sum(gx[i] * gy[i]) for i in range(len(A))])
            ratios[k, :] = rel / np.sum(rel)
        flux_ratios = np.mean(ratios, axis=0)
        self.stars["fluxratio"] = flux_ratios
        tdepths = np.zeros(len(self.stars))
        nz = flux_ratios != 0
        tdepths[nz] = 1 - (flux_ratios[nz] - tdepth) / flux_ratios[nz]
        tdepths[tdepths > 1] = 0
        self.stars["tdepth"] = tdepths
        hosts = self.stars[self.stars["tdepth"] > 0]
        for i, ID in enumerate(hosts["ID"].values):
            need = ["mass", "rad", "Teff"] + (["plx"] if i == 0 else [])
            if any(np.isnan(hosts[c].values[i]) for c in need):
                print("WARNING: " + str(ID) + " is missing stellar properties"
                      + (" required for validation." if i == 0
                         else "; Solar values will be assumed."))
        return

    def calc_probs(self, time: np.ndarray, flux_0: np.ndarray,
                   flux_err_0: float, P_orb,
                   contrast_curve_file: str = None, filt: str = "TESS",
                   N: int = 1000000, parallel: bool = False,
                   drop_scenario: list = [],
                   verbose: int = 1, flatpriors: bool = False,
                   exptime: float = 0.00139, nsamples: int = 20,
                   molusc_file: str = None, mc_errors: bool = False,
                   fpp_err_target: float = None, N_max: int = None,
                   posterior_samples: int = None, posterior_seed: int = 0):
        """Relative probability of every scenario, FPP and NFPP (triceratops.py:673-1485).

        Extensions of the reference's arguments: `flux_err_0` may hold one error per time stamp
        (chi^2 is then weighted per point; the Gaussian constant and the secondary-depth cut use
        their mean), and `exptime` and `nsamples` may each hold one value per time stamp, for a
        light curve that mixes cadences (e.g. 30-min and 200-s TESS FFIs with 2-min target
        pixels).  The stamps are then modelled in groups of equal (exptime, nsamples), at most
        TRI_MAX_CADENCES = 8 of them, each with its own integration time and supersampling.
        Per-stamp arrays lose the rows whose time or flux is NaN, like time and flux.

        Monte-Carlo error bars (not in the reference; lnZ, probs, FPP and NFPP are the same
        bits with and without them): `mc_errors=True` also sets `lnZ_err`, `ess` and `N_draws`
        (per row), `FPP_err` and `NFPP_err` (delta method over the rows' evidences, see
        _numerics.probability_errors) and adds a `prob_err` column to `probs`; without it these
        attributes are None.  `fpp_err_target` (implies mc_errors) then refines: after each
        round, the scenario calls that carry the largest shares of Var(FPP) -- from the top,
        until they add up to at least half of it -- get as many new draws as they have so far,
        at most `N_max` in all per call (default 16 N); the new draws merge with the old ones
        as one more disjoint slice.  Rounds stop when FPP_err <= fpp_err_target or no
        contributing call can grow.  Host sampler: the new draws continue numpy's global
        generator; device sampler: each round is a new scenario call (a fresh Philox stream).
        Refinement needs all draws on this process (no draw sharding over a process group).

        Posterior samples (not in the reference): `posterior_samples=K` draws K samples from the
        posterior of every scenario row by systematic importance resampling of its prior draws
        (weights exp(lnL + lnprior), on the GPU) and sets `self.posterior`, a long-format
        DataFrame: one block of K rows per scenario row whose posterior is not empty, with the
        columns ID, scenario, row (of `probs`), draw (the prior draw's index) and the parameter
        columns of `probs` plus u1, u2, fluxratio_EB and fluxratio_comp.  Without it
        `self.posterior` is None.  The samples depend on `posterior_seed` and the row (and on
        the round under fpp_err_target, whose rounds merge their samples); lnZ, probs, FPP,
        NFPP, the best-draw tables and numpy's generator are the same bits with and without
        them.  At an effective sample size of a few, the K samples hold few distinct draws."""
        post_K = None
        if posterior_samples is not None:
            post_K = _dispatch.check_posterior_K(posterior_samples)
            if isinstance(posterior_seed, bool) or not isinstance(posterior_seed,
                                                                  (int, np.integer)):
                raise ValueError("posterior_seed must be an integer")
        if fpp_err_target is not None:
            if not (np.isfinite(fpp_err_target) and fpp_err_target > 0):
                raise ValueError("fpp_err_target must be positive and finite")
            mc_errors = True
            if N_max is None:
                N_max = 16 * int(N)
            if _dispatch._dist() is not None:
                raise ValueError("fpp_err_target refines scenarios on one process: it cannot be "
                                 "combined with draws sharded over a process group (vet whole "
                                 "targets per rank instead, batch.vet_many)")
        if N_max is not None and int(N_max) < int(N):
            raise ValueError("N_max (%d) must be >= N (%d)" % (int(N_max), int(N)))
        n_in = np.size(time)
        keep = ~np.isnan(time) & ~np.isnan(flux_0)
        time = time[keep]
        flux_0 = flux_0[keep]
        if np.ndim(flux_err_0) != 0:
            # an error per time stamp (an extension of the reference's scalar flux_err_0, see
            # tri_set_lightcurve_err): chi^2 is weighted per point, the scalar formulas use the mean
            flux_err_0 = np.asarray(flux_err_0, dtype=float)[keep]
        if np.ndim(exptime) != 0 or np.ndim(nsamples) != 0:
            # per-stamp cadence (tri_set_lightcurve_cadence)
            cad = []
            for name, x in (("exptime", exptime), ("nsamples", nsamples)):
                if np.ndim(x) != 0:
                    x = np.asarray(x)
                    if x.shape != (n_in,):
                        raise ValueError("%s has shape %s; the light curve has %d time stamps"
                                         % (name, x.shape, n_in))
                    x = x[keep]
                cad.append(x)
            exptime, nsamples = cad
        filtered = self.stars[self.stars["tdepth"] > 0]
        n_rows = 3 * len(filtered) + 12
        targets = np.zeros(n_rows, dtype=np.dtype("i8"))
        star_num = np.zeros(n_rows, dtype=np.dtype("i8"))
        scenarios = np.zeros(n_rows, dtype=np.dtype("U6"))
        best = {k: np.zeros(n_rows) for k in RESULT_KEYS}
        lnZ = np.zeros(n_rows)
        row_results = [None] * n_rows      # (mc_errors) the resolved result of every row
        calls = []                         # (mc_errors) (rows, make(n_draws)) per scenario call

        # Results are read a few scenarios after they were requested: the GPU works on one
        # scenario while the host draws the priors of the next (_dispatch.deferring), and with
        # numpy's draws (host sampler) the scenario functions run in a few threads chained so
        # that the global generator is still consumed in the reference's order
        # (_dispatch.ScenarioChain).
        waiting = collections.deque()      # (rows, pending scenario call)
        held = []                          # (rows, results) waiting for the group's exchange
        from . import marginal_likelihoods as _ml
        host_sampler = _ml._sampler_mode() == "host"
        threads = _dispatch.scenario_threads(_dispatch._dist() is not None) if host_sampler else 1
        eng = _dispatch.get_engine()   # created here, not by whichever scenario thread comes first
        chain = _dispatch.ScenarioChain(threads)
        # Under a process group (one process per GPU) the evidence records and best-draw
        # candidates of ALL rows are exchanged with one all-gather at the end; with numpy's
        # draws rank 0 alone runs the scenario functions and scatters every engine call's
        # columns, the other ranks evaluate their slices (_dispatch.CallGroup).
        group = _dispatch.open_group(scatter=host_sampler)

        def fill(rows, parts):
            for j, res in zip(rows, parts):
                res = _dispatch.resolve(res)
                for k in RESULT_KEYS:
                    best[k][j] = res[k][0]
                lnZ[j] = res["lnZ"]
                row_results[j] = res

        def settle(keep):
            while len(waiting) > keep:
                rows, call = waiting.popleft()
                out = call.result()
                parts = out if isinstance(out, tuple) else (out,)
                if group is None:
                    fill(rows, parts)
                else:   # the local half now (frees the engine's slot), the rest after the exchange
                    for res in parts:
                        _dispatch.prepare(res)
                    held.append((rows, parts))

        def launch(row, ID, num, names, fn):
            """Start one lnZ_* call (one or two table rows) and read older results."""
            rows = [row + k for k in range(len(names))]
            for j, name in zip(rows, names):
                targets[j], star_num[j], scenarios[j] = ID, num, name
            if fn is None:
                for j in rows:
                    lnZ[j] = -np.inf
                return
            calls.append((rows, fn))
            waiting.append((rows, chain.run(functools.partial(_in_stream, fn, rows[0], N))))
            settle(_PIPELINE_DEPTH)

        def say(msg):
            if verbose == 1:
                print(msg)

        if self.trilegal_fname is None:
            raise RuntimeError("no saved TRILEGAL table: pass trilegal_fname to target(); "
                               "the online query of the reference is out of scope")
        trilegal_fname = self.trilegal_fname

        follower = group is not None and group.scatter and not group.is_root
        ok = False
        # the thread that holds numpy's generator hands the GIL back and forth with the
        # scenario threads ~150 times per call: a short switch interval keeps those hand-overs
        # from costing 5 ms each
        switch_interval = sys.getswitchinterval()
        sys.setswitchinterval(_dispatch.gil_switch_interval())
        _bufpool.note_call()       # (page-locked column buffers from a process's second call on)
        moments = _dispatch.mc_errors() if mc_errors else contextlib.nullcontext()
        post = (lambda: _dispatch.posterior_samples(post_K, posterior_seed)) if post_K else \
            contextlib.nullcontext
        try:
            with moments, post(), _dispatch.deferring():
                for i, ID in enumerate(filtered["ID"].values if not follower else ()):
                    star = {c: filtered[c].values[i] for c in _STAR_COLUMNS}
                    flux, flux_err = renorm_flux(flux_0, flux_err_0, star["fluxratio"])
                    M_s, R_s, Teff, plx = star["mass"], star["rad"], star["Teff"], star["plx"]
                    mags = (star["Tmag"], star["Jmag"], star["Hmag"], star["Kmag"])
                    Z = 0.0
                    lc = (time, flux, flux_err, P_orb)
                    tail = dict(parallel=parallel, mission=self.mission, flatpriors=flatpriors,
                                exptime=exptime, nsamples=nsamples)

                    if i == 0:
                        if np.isnan(M_s) or np.isnan(R_s) or np.isnan(Teff) or np.isnan(plx):
                            print("Insufficient information to validate " + str(ID)
                                  + ". Please ensure a stellar mass (in M_Sun), radius (in R_Sun), "
                                  + "Teff (in K), and plx (in mas) are provided in the .stars dataframe.")
                            break
                        # (bound now: the loop variables change under the threads)
                        runners = {
                            "TP": _bind(lnZ_TTP, *lc, M_s, R_s, Teff, Z, **tail),
                            "EB": _bind(lnZ_TEB, *lc, M_s, R_s, Teff, Z, **tail),
                            "PTP": _bind(lnZ_PTP, *lc, M_s, R_s, Teff, Z, plx, contrast_curve_file,
                                         filt, **tail, molusc_file=molusc_file),
                            "PEB": _bind(lnZ_PEB, *lc, M_s, R_s, Teff, Z, plx, contrast_curve_file,
                                         filt, **tail, molusc_file=molusc_file),
                            "STP": _bind(lnZ_STP, *lc, M_s, R_s, Teff, Z, plx, contrast_curve_file,
                                         filt, **tail, molusc_file=molusc_file),
                            "SEB": _bind(lnZ_SEB, *lc, M_s, R_s, Teff, Z, plx, contrast_curve_file,
                                         filt, **tail, molusc_file=molusc_file),
                            "DTP": _bind(lnZ_DTP, *lc, M_s, R_s, Teff, Z, *mags, trilegal_fname,
                                         contrast_curve_file, filt, **tail),
                            "DEB": _bind(lnZ_DEB, *lc, M_s, R_s, Teff, Z, *mags, trilegal_fname,
                                         contrast_curve_file, filt, **tail),
                            "BTP": _bind(lnZ_BTP, *lc, M_s, R_s, Teff, *mags, trilegal_fname,
                                         contrast_curve_file, filt, **tail),
                            "BEB": _bind(lnZ_BEB, *lc, M_s, R_s, Teff, *mags, trilegal_fname,
                                         contrast_curve_file, filt, **tail),
                        }
                        for key, row, num, names in _TARGET_SCENARIOS:
                            if len(names) == 1:
                                say("Calculating " + names[0] + " scenario probability for "
                                    + str(ID) + ".")
                            else:
                                say("Calculating " + names[0] + " and " + names[1]
                                    + " scenario probabilities for " + str(ID) + ".")
                            launch(row, ID, num, names,
                                   None if key in drop_scenario else runners[key])
                    else:
                        # nearby star: unknown properties default to solar (triceratops.py:1345-1350)
                        if np.isnan(Teff):
                            Teff = 5777
                        if np.isnan(M_s):
                            M_s = 1.0
                        if np.isnan(R_s):
                            R_s = 1.0
                        say("Calculating NTP, NEB, and NEB2xP scenario probabilities for "
                            + str(ID) + ".")
                        row = 15 + 3 * (i - 1)
                        launch(row, ID, 1, ("NTP",),
                               _bind(lnZ_TTP, *lc, M_s, R_s, Teff, Z, **tail))
                        launch(row + 1, ID, 1, ("NEB", "NEBx2P"),
                               _bind(lnZ_TEB, *lc, M_s, R_s, Teff, Z, **tail))
                settle(0)
                ok = True
        finally:
            chain.close()
            sys.setswitchinterval(switch_interval)
            try:
                if group is not None and group.scatter and group.is_root:
                    group.finish_root(error=not ok)
            finally:
                if not ok:
                    _dispatch.close_group()
        err = None
        posterior = None
        try:
            if follower:
                with _dispatch.mc_errors() if mc_errors else contextlib.nullcontext():
                    targets, star_num, scenarios, best, lnZ, err, posterior = group.follow(eng)
            elif group is not None:
                group.exchange()
                for rows, parts in held:
                    fill(rows, parts)
                if mc_errors:
                    err = _refine(calls, row_results, lnZ, best, None, None)
                if post_K:
                    posterior = _posterior_frame(targets, scenarios, row_results)
                if group.scatter:
                    group.publish((targets, star_num, scenarios, best, lnZ, err, posterior))
        finally:
            self.collectives = None if group is None else {
                "record_exchanges": group.collectives, "scatters": group.scatters}
            _dispatch.close_group()

        if mc_errors and group is None:
            with _dispatch.mc_errors(), post():
                err = _refine(calls, row_results, lnZ, best, fpp_err_target, N_max,
                              (post_K, posterior_seed) if post_K else None)
        if post_K and group is None:
            posterior = _posterior_frame(targets, scenarios, row_results)
        self.posterior = posterior
        relative_probs, status = _normalize_probabilities(lnZ)
        if status == 'anomaly':
            warnings.warn(
                "Unexpected NaN or +inf in scenario log-evidences. This indicates a numerical "
                "anomaly unrelated to geometric exclusions. Inspect self.lnZ for diagnostics.",
                RuntimeWarning, stacklevel=2)
            self.FPP_degenerate = True
        elif status == 'all_neginf':
            warnings.warn(
                "All scenario log-evidences are -inf: every MC draw was geometrically invalid. "
                "FPP=1.0 reflects a failed computation, not a confident false positive. "
                "Inspect self.lnZ for diagnostics.",
                RuntimeWarning, stacklevel=2)
            self.FPP_degenerate = True
        else:
            self.FPP_degenerate = False

        self.probs = DataFrame({
            "ID": targets, "scenario": scenarios,
            "M_s": best["M_s"], "R_s": best["R_s"], "P_orb": best["P_orb"], "inc": best["inc"],
            "b": best["b"], "ecc": best["ecc"], "w": best["argp"], "R_p": best["R_p"],
            "M_EB": best["M_EB"], "R_EB": best["R_EB"], "prob": relative_probs,
        })
        self.lnZ = lnZ
        self.star_num = star_num
        self.u1 = best["u1"]
        self.u2 = best["u2"]
        self.fluxratio_EB = best["fluxratio_EB"]
        self.fluxratio_comp = best["fluxratio_comp"]
        prob = self.probs.prob
        self.FPP = 1 - (prob[0] + prob[3] + prob[9])
        self.NFPP = np.sum(prob[15:]) if len(prob) > 15 else 0.0
        self.lnZ_err = self.ess = self.N_draws = self.FPP_err = self.NFPP_err = None
        if err is not None:
            self.lnZ_err, self.ess, self.N_draws = err["lnZ_err"], err["ess"], err["N"]
            self.FPP_err, self.NFPP_err = err["FPP_err"], err["NFPP_err"]
            self.probs["prob_err"] = err["prob_err"]
        return


_POSTERIOR_COLUMNS = (("M_s", "M_s"), ("R_s", "R_s"), ("P_orb", "P_orb"), ("inc", "inc"),
                      ("b", "b"), ("ecc", "ecc"), ("w", "argp"), ("R_p", "R_p"),
                      ("M_EB", "M_EB"), ("R_EB", "R_EB"), ("u1", "u1"), ("u2", "u2"),
                      ("fluxratio_EB", "fluxratio_EB"), ("fluxratio_comp", "fluxratio_comp"))


def _posterior_frame(targets, scenarios, row_results):
    """calc_probs' `posterior`: the rows' posterior tables stacked in row order."""
    blocks = []
    for j, res in enumerate(row_results):
        tab = None if res is None else res.posterior
        if tab is None or not len(tab["draw"]):
            continue
        n = len(tab["draw"])
        cols = {"ID": np.full(n, targets[j]), "scenario": np.full(n, scenarios[j]),
                "row": np.full(n, j), "draw": np.asarray(tab["draw"], dtype=np.int64)}
        cols.update({name: np.asarray(tab[key]) for name, key in _POSTERIOR_COLUMNS})
        blocks.append(DataFrame(cols))
    if not blocks:
        return DataFrame(columns=["ID", "scenario", "row", "draw"]
                         + [name for name, _ in _POSTERIOR_COLUMNS])
    return concat(blocks, ignore_index=True)


def _in_stream(make, stream, n):
    """One scenario call of n draws whose posterior samples use `stream`."""
    with _dispatch.call_stream(stream):
        return make(n)


def _bind(fn, *args, **kw):
    """One scenario call as a function of its number of draws: fn(*args, N=n, **kw)."""
    def make(n):
        return fn(*args, N=n, **kw)
    return make


def _row_errors(calls, lnZ):
    """Per-row (lnZ_err, ess, N) and the delta-method errors of the rows' probabilities, FPP and
    NFPP from the current result of every scenario call (`calls`: dicts with rows, N, cur)."""
    n = len(lnZ)
    lnZ_err, ess, r = np.full(n, np.nan), np.zeros(n), np.zeros(n)
    N_draws = np.zeros(n, dtype=np.int64)
    for c in calls:
        for j, res in zip(c["rows"], c["cur"]):
            N_draws[j] = c["N"]
            if res.s2 is None:        # (an engine without the moment pass)
                r[j] = np.nan
                continue
            lnZ_err[j], ess[j], r[j] = mc_error(c["N"], res.record[0], res.record[1],
                                                res.record[2], res.record[3], res.record[4])
    prob_err, fpp_err, nfpp_err, contrib = probability_errors(
        lnZ, r, [c["rows"] for c in calls], [c["N"] for c in calls])
    return dict(lnZ_err=lnZ_err, ess=ess, N=N_draws, prob_err=prob_err, FPP_err=fpp_err,
                NFPP_err=nfpp_err), contrib


def _merge_round(old, new, offset, post=None):
    """One branch's result over the draws of `old` followed by `new` (drawn after them: its
    indices start at `offset`), merged like the records of two ranks (_dispatch._merge_records):
    lnZ over all draws, the best-draw table the top 100 of both, each row from the round that
    drew it."""
    N = old.N + new.N
    allrec = np.stack([
        _dispatch.record_row(r.record[0], r.record[1], r.record[3], r.record[4], r.n_pass,
                             r.n_evaluated, r.record[2], np.asarray(r.top[1]) + off, r.top[0])
        for r, off in ((old, 0), (new, offset))])
    br = _dispatch._merge_records(allrec, 0, N, N)
    where = {}
    for src, off in ((new, offset), (old, 0)):
        for pos, i in enumerate(np.asarray(src.top[1])[:len(src.top[0])]):
            where.setdefault(int(i) + off, (src, pos))
    k = len(br.vals)
    picks = [where[int(i)] for i in br.idx[:k]]
    # rows of zero weight (fewer than 100 finite draws in all): old's padding rows
    picks += [(old, pos) for pos in range(k, len(old[RESULT_KEYS[0]]))]
    out = ScenarioResult({key: np.array([src[key][pos] for src, pos in picks])
                          for key in RESULT_KEYS}, lnZ=br.lnZ)
    out.n_pass, out.n_evaluated = br.n_pass, br.n_evaluated
    out.set_moments(N, (br.m, br.s, br.s2, br.n_finite, br.n_posinf),
                    (br.vals, br.idx[:k]))
    if post is not None and old.posterior is not None and new.posterior is not None:
        # post = (K, seed, stream of the new round, branch): merged like two slices of draws
        tabs = (old.posterior, {**new.posterior, "draw": new.posterior["draw"] + offset})
        idx, _, W = merge_posteriors(
            [(r.record[0], r.post_total, t["draw"]) for r, t in zip((old, new), tabs)], *post)
        draws = np.concatenate([t["draw"] for t in tabs])
        pos = np.searchsorted(draws, idx)
        out.posterior = {key: np.concatenate([np.asarray(t[key]) for t in tabs])[pos]
                         for key in tabs[0] if key != "draw"}
        out.posterior["draw"] = idx
        out.post_total = W
    return out


def _refine(calls, row_results, lnZ, best, target, N_max, post=None):
    """Error bars of calc_probs; with `target`, refinement rounds until FPP_err <= target or no
    call that contributes to Var(FPP) can grow (N_max draws per call).  Updates lnZ and best in
    place for the refined rows; returns the error fields."""
    state = [dict(rows=rows, make=make, N=int(row_results[rows[0]].N),
                  cur=[row_results[j] for j in rows]) for rows, make in calls]
    err, contrib = _row_errors(state, lnZ)
    rnd = 0
    while target is not None and np.isfinite(err["FPP_err"]) and err["FPP_err"] > target:
        total, acc, picked = contrib.sum(), 0.0, []
        for ci in np.argsort(-contrib, kind="stable"):
            if not contrib[ci] > 0 or acc >= 0.5 * total:
                break
            if state[ci]["N"] < N_max:
                picked.append(ci)
                acc += contrib[ci]
        if not picked:
            break
        rnd += 1
        for ci in picked:
            c = state[ci]
            n_new = min(c["N"], N_max - c["N"])
            stream = c["rows"][0] + (rnd << 32)     # (round 0 used the row itself)
            out = _in_stream(c["make"], stream, n_new)
            parts = out if isinstance(out, tuple) else (out,)
            c["cur"] = [_merge_round(old, new, c["N"],
                                     None if post is None else (*post, stream, b))
                        for b, (old, new) in enumerate(zip(c["cur"], parts))]
            c["N"] += n_new
            for j, res in zip(c["rows"], c["cur"]):
                lnZ[j] = res["lnZ"]
                for k in RESULT_KEYS:
                    best[k][j] = res[k][0]
        err, contrib = _row_errors(state, lnZ)
    return err
