"""The ten `lnZ_*` scenarios with the prior draws generated on the device (opt-in).

Same scenario definitions as `marginal_likelihoods.py` (reference
marginal_likelihoods.py:39-2362) -- same priors, same derived quantities, same wiring into the
two evaluation kernels -- but every per-draw column is produced in HBM by ONE fused kernel per
scenario (`csrc/tri_sampler.cuh`, `tri_dev_sample`): a Philox stream per draw, the inverse-CDF
samplers, the stellar / flux relations, the limb-darkening look-ups and the companion /
background priors.  The columns go to `tri_submit_*_dev` by pointer on the same stream; the host
touches only scalars, the small look-up tables (uploaded once per process and cached) and the
100-row result tables.

It CANNOT be bit-identical to the reference: the deviates are Philox streams, not numpy's
Mersenne Twister, so results agree with the host-sampler mode only statistically (same
distributions, evidences equal within Monte-Carlo error; tests/test_device_sampler.py).  The
default therefore stays the host sampler.  One documented difference in the transforms:
contrast curves are interpolated by plain bisection, whereas `numpy.interp` on a NON-monotonic
curve (the TOI-465 example is one) returns query-order-dependent values that no parallel
evaluation can reproduce.

Enable with `triceratops_b200.set_sampler("device", seed=...)`.  A draw's random stream depends
on (seed, scenario call number, GLOBAL draw index) only: under a process group every rank makes
its own N/G draws and the union is the same sample whatever the number of ranks; an unseeded run
agrees on one seed first (rank 0's entropy).
"""
import contextlib
import ctypes
import functools
import math
import os

import numpy as np
import torch

from . import _cabi, _dispatch, _numerics, funcs, priors
from . import marginal_likelihoods as ml
from ._cabi import tri_bound_prior, tri_powerlaw, tri_sampler_args, tri_spline
from ._ldc import grid_for
from .funcs import file_to_contrast_curve

N_SAMPLES = 100
F64 = torch.float64
_state = {"seed": None, "calls": 0}
_cache = {}


def seed(value):
    _state["seed"] = value
    _state["calls"] = 0


# ------------------------------------------------------------------------------- proposals
class Proposal:
    """An importance proposal of one scenario call: per slot of tri_sampler_args.prop the
    knots of H_d and ln h_d (`tables`, [TRI_PROP_SLOTS, 2 B + 1]; _numerics.fit_proposal), the
    mixture weight `alpha` of the prior, and the tables' copy on each device they were used on."""

    def __init__(self, tables, alpha=_numerics.PROP_ALPHA):
        tables = np.ascontiguousarray(tables, dtype=np.float64)
        B = (tables.shape[1] - 1) // 2
        if (tables.shape != (_cabi.TRI_PROP_SLOTS, 2 * B + 1) or B < 1 or B & (B - 1)
                or not np.all(np.isfinite(tables))):
            raise ValueError("proposal tables must be finite, [%d, 2 B + 1] with B a power of two"
                             % _cabi.TRI_PROP_SLOTS)
        if not 0.0 < float(alpha) <= 1.0:
            raise ValueError("alpha must be in (0, 1]")
        self.tables, self.bins, self.alpha = tables, B, float(alpha)
        self._dev = {}

    @classmethod
    def identity(cls, B=_numerics.PROP_BINS, alpha=_numerics.PROP_ALPHA):
        """The prior as a proposal: the columns of a call without one, bit for bit."""
        return cls(_numerics.identity_tables(B), alpha)

    def device_tables(self, dev):
        key = str(dev)
        if key not in self._dev:      # (a stream-ordered copy on the current stream)
            self._dev[key] = _t(self.tables, dev)
        return self._dev[key]


_prop = {"proposal": None, "record": 0}


@contextlib.contextmanager
def importance_proposal(p):
    """Device-sampler lnZ_* calls made inside draw from Proposal `p` (None: the prior)."""
    if p is not None and not isinstance(p, Proposal):
        raise ValueError("importance_proposal takes a device_sampler.Proposal or None")
    prev, _prop["proposal"] = _prop["proposal"], p
    try:
        yield
    finally:
        _prop["proposal"] = prev


@contextlib.contextmanager
def record_coords():
    """Device-sampler lnZ_* calls made inside that also draw posterior samples set
    ScenarioResult.post_coords, the samples' proposal coordinates ([K, TRI_PROP_SLOTS])."""
    _prop["record"] += 1
    try:
        yield
    finally:
        _prop["record"] -= 1


def _device():
    return torch.device("cuda", _dispatch.get_engine().device)


def _t(x, dev):
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), dtype=F64, device=dev)


def _cached(key, make):
    if key not in _cache:
        _cache[key] = make()
    return _cache[key]


# ------------------------------------------------------------------------------- descriptors
def _powerlaw(spec):
    """tri_powerlaw of a priors law (edges, powers, amps) for the kernel's inverse CDF; None:
    every draw is 1.0."""
    L = tri_powerlaw()
    if spec is None:
        L.nseg, L.constant = 0, 1.0
        return L
    edges, powers, amps = spec
    integrals, cum, L.norm = priors.powerlaw_tables(edges, powers, amps)
    L.nseg = len(powers)
    for k in range(L.nseg):
        L.powers[k], L.amps[k], L.integrals[k], L.cum[k] = powers[k], amps[k], integrals[k], cum[k]
        L.epow[k] = edges[k] ** (powers[k] + 1)
    return L


def _spline(spl, dev):
    t, c = _cached(("spline", id(spl), str(dev)),
                   lambda: (_t(spl._eval_args[0], dev), _t(spl._eval_args[1], dev)))
    S = tri_spline()
    S.t, S.c, S.n, S.k = t.data_ptr(), c.data_ptr(), t.numel(), int(spl._eval_args[2])
    return S


def _bound_prior(M_s, plx, first_decade):
    """tri_bound_prior of lnprior_bound_TP (first_decade False) / lnprior_bound_EB (True)."""
    K = priors.bound_constants(M_s, plx)
    return tri_bound_prior(
        d_pc=K["d"], M_eff=K["M_s"], first_decade=int(first_decade),
        **{n: K[n] for n in ("M_act", "f1", "f2", "f3", "alpha", "dlogP", "slope", "slope2", "t2",
                             "t3", "t4", "t5")})


def _ldc_tables(mission, Z, dev):
    return _cached(("ldc", mission, float(Z), str(dev)),
                   lambda: tuple(_t(tab, dev) for tab in grid_for(mission).dense_table(Z)))


def _contrast(contrast_curve_file, dev):
    if contrast_curve_file is None:      # the reference's 2.2 arcsec default (e.g. :478-487)
        return _cached(("cc", None, str(dev)), lambda: (_t([2.2], dev), _t([1.0], dev)))

    def make():
        s_, c_ = file_to_contrast_curve(contrast_curve_file)
        return _t(s_, dev), _t(c_, dev)
    return _cached(("cc", contrast_curve_file, os.path.getmtime(contrast_curve_file), str(dev)),
                   make)


class _Background:
    """marginal_likelihoods._Background (the TRILEGAL population behind the target), resident
    on the device."""

    def __init__(self, trilegal_fname, Tmag, Jmag, Hmag, Kmag, mission, dev):
        pop = ml._Background(trilegal_fname, Tmag, Jmag, Hmag, Kmag)
        self.N_comp = int(pop.N_comp)
        self.mass, self.logg = _t(pop.masses, dev), _t(pop.loggs, dev)
        self.teff = _t(pop.Teffs, dev)
        self.radius = _t(pop.radii(), dev)
        u1, u2 = grid_for(mission).nearest_each(pop.Teffs, pop.loggs, pop.Zs)
        self.u1, self.u2 = _t(u1, dev), _t(u2, dev)
        self.dmag = {b: _t(pop.band(b), dev) for b in "TJHK"}
        self.fr = {b: _t(pop.fluxratios_in(b), dev) for b in "TJHK"}


def _background(trilegal_fname, mags, mission, dev):
    key = ("bg", trilegal_fname, os.path.getmtime(trilegal_fname), tuple(float(m) for m in mags),
           mission, str(dev))
    return _cached(key, lambda: _Background(trilegal_fname, *mags, mission, dev))


def _band(filt):
    return filt if filt in ("J", "H", "K") else "T"


def _molusc(N, lo, hi, M_s, molusc_file, dev):
    # padded to the TOTAL draw count, this rank takes its slice (as the host sampler does)
    q = ml.molusc_q(M_s, molusc_file)[:N]
    return _t(np.pad(q, (0, N - len(q)))[lo:hi], dev)


# ------------------------------------------------------------------------------- one scenario
_OUT = ("body", "ebfr", "q", "P", "inc", "ecc", "argp", "mtot", "rhost", "u1", "u2", "cfr",
        "lnprior", "mhost", "meb")


def _sample(time, flux, sigma, exptime, nsamples, N, kind, host, diluter, P_orb, M_s, R_s, Teff,
            u12, flatpriors, mission, Z=0.0, Teff_cap=10000.0, prior=None, plx=np.nan,
            contrast_curve_file=None, filt="TESS", molusc_file=None, bg=None, idx_hi=0,
            beb=False):
    """Launch the sampler kernel of one scenario; returns (engine, device, n_local, columns)."""
    eng = _dispatch.get_engine()
    _dispatch.use_lightcurve(time, flux, sigma, exptime, nsamples)
    dev = _device()
    lo, hi = _dispatch.shard_bounds(N)
    n = hi - lo
    d = _dispatch._dist()
    if _state["seed"] is None:
        box = [int.from_bytes(os.urandom(7), "little")]
        if d is not None:        # one base seed for all ranks (rank 0's entropy)
            d.broadcast_object_list(box, src=0)
        _state["seed"] = box[0]
    A = tri_sampler_args()
    A.n, A.index0 = n, lo
    A.seed, A.stream = int(_state["seed"]) & (2 ** 64 - 1), _state["calls"]
    _state["calls"] += 1
    A.kind, A.host, A.diluter, A.flatpriors = kind, host, diluter, int(bool(flatpriors))
    if type(P_orb) not in [float, int]:
        A.P_lo, A.P_hi = float(P_orb[0]), float(P_orb[-1])
        P_mean = 0.5 * (A.P_lo + A.P_hi)
    else:
        A.P_lo = A.P_hi = P_mean = float(P_orb)
    A.ecc_expo = 0.2 if P_mean <= 10 else 0.6
    A.M_s, A.R_s, A.Teff = float(M_s), float(R_s), float(Teff)
    A.u1, A.u2 = (float(u12[0]), float(u12[1])) if u12 is not None else (math.nan, math.nan)
    A.rp_hi, A.rp_lo = (_powerlaw(spec) for spec in priors.rp_specs())
    A.q_pl = _powerlaw(priors.mass_ratio_spec(M_s, *priors.Q_LAW))
    A.qc_pl = _powerlaw(priors.mass_ratio_spec(M_s, *priors.Q_COMPANION_LAW))
    keep = []
    A.hot_R, A.cool_R = _spline(funcs._hot_R, dev), _spline(funcs._cool_R, dev)
    A.hot_T, A.cool_T = _spline(funcs._hot_T, dev), _spline(funcs._cool_T, dev)
    cc_band = _band(filt) if beb else filt
    cc_filt = {"T": "TESS"}.get(cc_band, cc_band)
    A.flux_tess = _spline(funcs._FLUX_SPLINES["TESS"], dev)
    A.flux_cc = _spline(funcs._FLUX_SPLINES[cc_filt], dev)
    A.f_target_tess = float(funcs.flux_relation(np.array([M_s]), "TESS")[0])
    A.f_target_cc = float(funcs.flux_relation(np.array([M_s]), cc_filt)[0])
    A.Teff_cap = float(Teff_cap)
    err = None
    if host == 1:
        t1, t2 = _ldc_tables(mission, Z, dev)
        A.ldc_u1, A.ldc_u2 = t1.data_ptr(), t2.data_ptr()
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        A.err_flag = err.data_ptr()
    A.use_cc = int(contrast_curve_file is not None)
    A.beb_cc_band = int(beb and cc_band in ("J", "H", "K"))
    A.prior_mode = 0
    if prior in ("bound_TP", "bound_EB") and molusc_file is None:
        A.prior_mode = 1
        A.bound = _bound_prior(M_s, plx, prior == "bound_EB")
    elif prior == "background":
        A.prior_mode = 2
    if A.prior_mode:
        sep, con = _contrast(contrast_curve_file, dev)
        A.cc_sep, A.cc_con, A.cc_n = sep.data_ptr(), con.data_ptr(), sep.numel()
    if molusc_file is not None and diluter == 1:
        mq = _molusc(N, lo, hi, M_s, molusc_file, dev)
        keep.append(mq)
        A.molusc_q = mq.data_ptr()
    if bg is not None:
        A.n_comp, A.idx_hi = bg.N_comp, int(idx_hi)
        A.bg_const_prior = math.log((bg.N_comp / 0.1) * (1 / 3600) ** 2 * 2.2 ** 2)
        A.bg_mass, A.bg_radius = bg.mass.data_ptr(), bg.radius.data_ptr()
        A.bg_logg, A.bg_teff = bg.logg.data_ptr(), bg.teff.data_ptr()
        A.bg_u1, A.bg_u2 = bg.u1.data_ptr(), bg.u2.data_ptr()
        A.bg_fr_tess = bg.fr["T"].data_ptr()
        band = _band(filt)
        A.bg_dmag_cc = bg.dmag[band].data_ptr()
        A.bg_fr_cc = bg.fr[band].data_ptr()
    # outputs: only the columns that are per-draw in this scenario (and P, which is cheap; a
    # fixed period reaches the engine as a scalar)
    want = {"body", "P", "inc", "ecc", "argp", "mtot"}
    if kind == 1:
        want |= {"ebfr", "q", "meb"}
    if host != 0:
        want |= {"rhost", "u1", "u2", "mhost"}
    if diluter != 0:
        want |= {"cfr"}
    prop = _prop["proposal"]
    if A.prior_mode or prop is not None:
        want |= {"lnprior"}
    cols = {k: torch.empty(max(n, 1), dtype=F64, device=dev)[:n] for k in _OUT if k in want}
    for k, v in cols.items():
        setattr(A, "o_" + k, v.data_ptr())
    if prop is not None:
        tab = prop.device_tables(dev)
        keep.append(tab)
        A.prop, A.prop_bins, A.prop_alpha = tab.data_ptr(), prop.bins, prop.alpha
    coords = None
    if _prop["record"] and _dispatch._post is not None:
        # the coordinates of the posterior samples (slots the scenario does not draw stay NaN)
        coords = torch.full((_cabi.TRI_PROP_SLOTS, max(n, 1)), math.nan, dtype=F64, device=dev)
        A.o_coords = coords.data_ptr()
    mask = None
    if (diluter == 1) or host == 2:
        mask = torch.empty(max(n, 1), dtype=torch.uint8, device=dev)[:n]
        A.o_mask = mask.data_ptr()
    stream = torch.cuda.current_stream(dev).cuda_stream
    _cabi.check(eng.lib.tri_dev_sample(ctypes.byref(A), ctypes.c_void_p(stream)))
    if err is not None and Teff_cap > 10000:   # (a read-back: only where the error can fire)
        if int(err.item()):
            # the reference's `.item()` raises for nodes beyond the grid (Teff clamp 13000, :1181)
            raise ValueError("can only convert an array of size 1 to a Python scalar")
    cols["mask"] = mask
    cols["_keep"] = keep
    cols["_coords"] = coords
    return eng, dev, n, cols, A.P_lo if A.P_lo == A.P_hi else cols["P"]


# ------------------------------------------------------------------------------- result tables
def _take_rows(columns, idx, dev):
    """Rows `idx` of every column (device tensors or scalars) as numpy arrays, with a single
    device-to-host copy for all tensor columns."""
    n = len(idx)
    tens = [k for k, v in columns.items() if torch.is_tensor(v)]
    out = {}
    if tens and n:
        block = torch.stack([columns[k][idx].to(F64) for k in tens]).cpu().numpy()
        out = {k: block[i] for i, k in enumerate(tens)}
    for k, v in columns.items():
        if k not in out and v is not None:
            out[k] = np.zeros(n) if torch.is_tensor(v) else np.full(n, float(v))
    return out


def _table(res, eng, N, dev, twin, M_host, R_host, u1, u2, P, mtot, incs, eccs, argps, cfr,
           rps=None, masses=None, radii=None, fluxratios=None, post=None, branch=0, coords=None):
    """This rank's record of one branch: its best local draws with their rows, and with
    posterior samples (post = (K, seed, stream) of the call) those with theirs, registered for
    the merge across ranks; returns the merge as a function (_finished)."""
    cols = dict(M_s=M_host, R_s=R_host, u1=u1, u2=u2, P=P, mtot=mtot, inc=incs, ecc=eccs,
                argp=argps, R_p=rps, M_EB=masses, R_EB=radii, fluxratio_EB=fluxratios,
                fluxratio_comp=cfr if torch.is_tensor(cfr) else None)

    def rows(idx):
        tab = ml.result_table(len(idx), twin, **_take_rows(cols, idx, dev))
        return np.stack([tab[k] for k in ml.RESULT_KEYS], axis=1)
    lo = _dispatch.shard_bounds(N)[0]
    idx, vals, n_eval = _dispatch._local_best(res, eng, False)
    fin = np.isfinite(vals)
    idx, vals = np.asarray(idx, dtype=np.int64)[fin], np.asarray(vals)[fin]
    tail = pcoords = None
    if post is not None and res.post_idx is not None:
        pidx = np.asarray(res.post_idx, dtype=np.int64)
        tidx = torch.as_tensor(pidx, device=dev)
        tail = (post[0], res.post_total, pidx + lo, rows(tidx))
        if coords is not None and _dispatch._dist() is None:
            # gathered on the device by posterior index, one copy (as _take_rows)
            pcoords = coords[:, tidx].T.contiguous().cpu().numpy() if len(pidx) else \
                np.zeros((0, _cabi.TRI_PROP_SLOTS))
    rec = _dispatch.pack_slice(res.m, res.s, res.n_finite, res.n_posinf, res.n_pass, n_eval,
                               getattr(res, "s2", None), idx + lo, vals,
                               rows(torch.as_tensor(idx, device=dev)), tail)
    group = _dispatch._group if _dispatch._dist() is not None else None
    key = None if group is None else group.add(rec)
    return functools.partial(_finished, rec, group, key, res.lnZ, N, post, branch, pcoords)


def _finished(rec, group, key, lnZ, N, post, branch, pcoords):
    br = _dispatch.merge_slices(_dispatch.gather_slices(rec, group, key), N,
                                len(ml.RESULT_KEYS), lnZ, post, branch)
    rows = br.rows
    if len(rows) < N_SAMPLES:
        # zero-weight padding: the last row repeated, so that the table always has N_SAMPLES rows
        pad = rows[-1:] if len(rows) else np.zeros((1, rows.shape[1]))
        rows = np.concatenate([rows, np.repeat(pad, N_SAMPLES - len(rows), axis=0)])
    out = ml.branch_result(br, {k: rows[:, i].copy() for i, k in enumerate(ml.RESULT_KEYS)})
    out.post_coords = pcoords
    return out


def _run(sampled, N, M_s, R_s, u12, is_host, scalar_loop=False):
    """Submit the evaluation of a sampled scenario and return its deferred result(s)."""
    eng, dev, n, c, P = sampled
    M_host = c.get("mhost", M_s)
    R_host = c.get("rhost", R_s)
    u1 = c.get("u1", u12[0] if u12 is not None else None)
    u2 = c.get("u2", u12[1] if u12 is not None else None)
    cfr = c.get("cfr", 0.0)
    common = dict(P_orb=P, inc=c["inc"], ecc=c["ecc"], argp=c["argp"], mtot=c["mtot"],
                  rhost=R_host, u1=u1, u2=u2, cfr=cfr, lnprior=c.get("lnprior"))
    post = _dispatch._next_post()
    if "ebfr" not in c:
        p = _dispatch._submit(eng, "tp_tensors", n, dict(rp=c["body"], **common), c["mask"],
                              is_host, N_SAMPLES, post=post)
        state = []

        def prepare():
            if not state:
                state.append(_table(p.result(), eng, N, dev, False, M_host, R_host, u1, u2, P,
                                    c["mtot"], c["inc"], c["ecc"], c["argp"], cfr,
                                    rps=c["body"], post=post, coords=c["_coords"]))

        def table():
            prepare()
            return state[0]()
        return _dispatch.deliver(table, prepare)
    kw = {"scalar_loop": True} if scalar_loop else {}
    p = _dispatch._submit(eng, "eb_tensors", n,
                          dict(reb=c["body"], ebfr=c["ebfr"], q=c["q"], **common), c["mask"],
                          is_host, N_SAMPLES, post=post, **kw)
    args = (M_host, R_host, u1, u2, P, c["mtot"], c["inc"], c["ecc"], c["argp"], cfr)
    tkw = dict(masses=c["meb"], radii=c["body"], fluxratios=c["ebfr"], post=post,
               coords=c["_coords"])
    state, done = [], {}

    def prepare():   # both branches at the first request, in a fixed order
        if not state:
            r0, r1 = p.result()
            state.append(_table(r0, eng, N, dev, False, *args, **tkw))
            state.append(_table(r1, eng, N, dev, True, *args, **tkw, branch=1))

    def table(b):
        prepare()
        if not done:   # (collectives inside when no CallGroup is open: fixed order)
            done[0], done[1] = state[0](), state[1]()
        return done[b]
    return (_dispatch.deliver(lambda: table(0), prepare),
            _dispatch.deliver(lambda: table(1), prepare))


# ------------------------------------------------------------------------------- scenarios
def lnZ_TTP(time, flux, sigma, P_orb, M_s, R_s, Teff, Z, N=1000000, parallel=False,
            mission="TESS", flatpriors=False, exptime=0.00139, nsamples=20):
    u12 = grid_for(mission).nearest(Z, Teff, ml._logg(M_s, R_s))
    s = _sample(time, flux, sigma, exptime, nsamples, int(N), 0, 0, 0, P_orb, M_s, R_s, Teff, u12,
                flatpriors, mission)
    return _run(s, int(N), M_s, R_s, u12, False)


def lnZ_TEB(time, flux, sigma, P_orb, M_s, R_s, Teff, Z, N=1000000, parallel=False,
            mission="TESS", flatpriors=False, exptime=0.00139, nsamples=20):
    u12 = grid_for(mission).nearest(Z, Teff, ml._logg(M_s, R_s))
    s = _sample(time, flux, sigma, exptime, nsamples, int(N), 1, 0, 0, P_orb, M_s, R_s, Teff, u12,
                flatpriors, mission)
    return _run(s, int(N), M_s, R_s, u12, False, scalar_loop=not parallel)


def _bound(kind, host, prior, Teff_cap, time, flux, sigma, P_orb, M_s, R_s, Teff, Z, plx,
           contrast_curve_file, filt, N, parallel, mission, flatpriors, exptime, nsamples,
           molusc_file):
    u12 = None if host == 1 else grid_for(mission).nearest(Z, Teff, ml._logg(M_s, R_s))
    s = _sample(time, flux, sigma, exptime, nsamples, int(N), kind, host, 1, P_orb, M_s, R_s,
                Teff, u12, flatpriors, mission, Z=Z, Teff_cap=Teff_cap, prior=prior, plx=plx,
                contrast_curve_file=contrast_curve_file, filt=filt, molusc_file=molusc_file)
    return _run(s, int(N), M_s, R_s, u12, host == 1, scalar_loop=(kind == 1 and not parallel))


def lnZ_PTP(time, flux, sigma, P_orb, M_s, R_s, Teff, Z, plx, contrast_curve_file=None,
            filt="TESS", N=1000000, parallel=False, mission="TESS", flatpriors=False,
            exptime=0.00139, nsamples=20, molusc_file=None):
    return _bound(0, 0, "bound_TP", 10000, time, flux, sigma, P_orb, M_s, R_s, Teff, Z, plx,
                  contrast_curve_file, filt, N, parallel, mission, flatpriors, exptime, nsamples,
                  molusc_file)


def lnZ_PEB(time, flux, sigma, P_orb, M_s, R_s, Teff, Z, plx, contrast_curve_file=None,
            filt="TESS", N=1000000, parallel=False, mission="TESS", flatpriors=False,
            exptime=0.00139, nsamples=20, molusc_file=None):
    return _bound(1, 0, "bound_EB", 10000, time, flux, sigma, P_orb, M_s, R_s, Teff, Z, plx,
                  contrast_curve_file, filt, N, parallel, mission, flatpriors, exptime, nsamples,
                  molusc_file)


def lnZ_STP(time, flux, sigma, P_orb, M_s, R_s, Teff, Z, plx, contrast_curve_file=None,
            filt="TESS", N=1000000, parallel=False, mission="TESS", flatpriors=False,
            exptime=0.00139, nsamples=20, molusc_file=None):
    return _bound(0, 1, "bound_TP", 10000, time, flux, sigma, P_orb, M_s, R_s, Teff, Z, plx,
                  contrast_curve_file, filt, N, parallel, mission, flatpriors, exptime, nsamples,
                  molusc_file)


def lnZ_SEB(time, flux, sigma, P_orb, M_s, R_s, Teff, Z, plx, contrast_curve_file=None,
            filt="TESS", N=1000000, parallel=False, mission="TESS", flatpriors=False,
            exptime=0.00139, nsamples=20, molusc_file=None):
    # Teff clamp of 13000 K (grid stops at 10000 K) as in the reference, :1181
    return _bound(1, 1, "bound_EB", 13000, time, flux, sigma, P_orb, M_s, R_s, Teff, Z, plx,
                  contrast_curve_file, filt, N, parallel, mission, flatpriors, exptime, nsamples,
                  molusc_file)


def _behind(kind, host, time, flux, sigma, P_orb, M_s, R_s, Teff, Z, mags, trilegal_fname,
            contrast_curve_file, filt, N, parallel, mission, flatpriors, exptime, nsamples):
    dev = _device()
    bg = _background(trilegal_fname, mags, mission, dev)
    u12 = None if host == 2 else grid_for(mission).nearest(Z, Teff, ml._logg(M_s, R_s))
    # randint upper bound N_comp - 1 in D*, N_comp in B* (:1463, :1672 vs :1926, :2139)
    idx_hi = bg.N_comp if host == 2 else bg.N_comp - 1
    s = _sample(time, flux, sigma, exptime, nsamples, int(N), kind, host, 2, P_orb, M_s, R_s,
                Teff, u12, flatpriors, mission, prior="background",
                contrast_curve_file=contrast_curve_file, filt=filt, bg=bg, idx_hi=idx_hi,
                beb=(kind == 1 and host == 2))
    return _run(s, int(N), M_s, R_s, u12, host == 2, scalar_loop=(kind == 1 and not parallel))


def lnZ_DTP(time, flux, sigma, P_orb, M_s, R_s, Teff, Z, Tmag, Jmag, Hmag, Kmag, trilegal_fname,
            contrast_curve_file=None, filt="TESS", N=1000000, parallel=False, mission="TESS",
            flatpriors=False, exptime=0.00139, nsamples=20):
    return _behind(0, 0, time, flux, sigma, P_orb, M_s, R_s, Teff, Z, (Tmag, Jmag, Hmag, Kmag),
                   trilegal_fname, contrast_curve_file, filt, N, parallel, mission, flatpriors,
                   exptime, nsamples)


def lnZ_DEB(time, flux, sigma, P_orb, M_s, R_s, Teff, Z, Tmag, Jmag, Hmag, Kmag, trilegal_fname,
            contrast_curve_file=None, filt="TESS", N=1000000, parallel=False, mission="TESS",
            flatpriors=False, exptime=0.00139, nsamples=20):
    return _behind(1, 0, time, flux, sigma, P_orb, M_s, R_s, Teff, Z, (Tmag, Jmag, Hmag, Kmag),
                   trilegal_fname, contrast_curve_file, filt, N, parallel, mission, flatpriors,
                   exptime, nsamples)


def lnZ_BTP(time, flux, sigma, P_orb, M_s, R_s, Teff, Tmag, Jmag, Hmag, Kmag, trilegal_fname,
            contrast_curve_file=None, filt="TESS", N=1000000, parallel=False, mission="TESS",
            flatpriors=False, exptime=0.00139, nsamples=20):
    return _behind(0, 2, time, flux, sigma, P_orb, M_s, R_s, Teff, 0.0, (Tmag, Jmag, Hmag, Kmag),
                   trilegal_fname, contrast_curve_file, filt, N, parallel, mission, flatpriors,
                   exptime, nsamples)


def lnZ_BEB(time, flux, sigma, P_orb, M_s, R_s, Teff, Tmag, Jmag, Hmag, Kmag, trilegal_fname,
            contrast_curve_file=None, filt="TESS", N=1000000, parallel=False, mission="TESS",
            flatpriors=False, exptime=0.00139, nsamples=20):
    return _behind(1, 2, time, flux, sigma, P_orb, M_s, R_s, Teff, 0.0, (Tmag, Jmag, Hmag, Kmag),
                   trilegal_fname, contrast_curve_file, filt, N, parallel, mission, flatpriors,
                   exptime, nsamples)
