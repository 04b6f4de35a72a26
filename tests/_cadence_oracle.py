"""Test helper: the CPU oracle engine (oracle/engine_port.py) extended to light curves with one
exposure time and one supersampling count per stamp, and to per-point errors.

The stamps are split into their cadence groups (triceratops_b200.engine.cadence_columns) and the
oracle evaluates each group with its own (exptime, nsamples): 0.5 chi^2 is the sum over the
groups, a +inf from the secondary-depth cut (the same for every group: the secondary pass does
not depend on the light curve) stays +inf, and simulated rows are scattered back into the
caller's stamp order.  With per-point errors chi^2 is weighted per stamp, computed from the
oracle's model light curves; the Gaussian constant and the depth cut use the mean error.
A light curve with one cadence and a scalar error is the plain OracleEngine.
"""
import numpy as np

from oracle import coracle
from oracle.engine_port import OracleEngine, _full, _lse_record, _Res, eb_masks, ln2pi, tp_mask
from triceratops_b200.engine import cadence_columns


def cadence_groups(exptime, nsamples, npts):
    """[(stamp indices, exptime, nsamples)] of each distinct pair, pairs in ascending order."""
    e, n = cadence_columns(exptime, nsamples, npts)
    if np.ndim(e) == 0:
        return [(np.arange(npts), float(e), int(n))]
    pairs = sorted(set(zip(e.tolist(), n.tolist())))
    return [(np.flatnonzero((e == pe) & (n == pn)), pe, pn) for pe, pn in pairs]


class CadenceOracleEngine(OracleEngine):

    def set_lightcurve(self, time, flux, sigma, exptime, nsamples):
        t, f = np.asarray(time, float), np.asarray(flux, float)
        self.err = None if np.ndim(sigma) == 0 else np.asarray(sigma, float)
        s = float(sigma) if self.err is None else float(self.err.mean())
        self.groups = cadence_groups(exptime, nsamples, t.size)
        self.full = (t, f, s)
        _, e0, n0 = self.groups[0]
        self.lc = (t, f, s, e0, n0)

    def _use(self, g):
        """Make group g the oracle's (single-cadence) light curve."""
        idx, e, n = self.groups[g]
        t, f, s = self.full
        self.lc = (t[idx], f[idx], s, e, n)
        return idx

    def _plain(self):
        return self.err is None and len(self.groups) == 1

    # ---- +0.5 chi^2 per draw (the lnL_*_p seam)
    def lnl_tp(self, R_p, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr, companion_is_host):
        if self._plain():
            return super().lnl_tp(R_p, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr,
                                  companion_is_host)
        if self.err is not None:
            model = self.simulate_tp(self.full[0].size, R_p, P_orb, inc, a, R_s, u1, u2, ecc, argp,
                                     cfr, companion_is_host)
            return self._weighted(model)
        out = 0.0
        for g in range(len(self.groups)):
            self._use(g)
            out = out + super().lnl_tp(R_p, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr,
                                       companion_is_host)
        return out

    def lnl_eb(self, R_EB, EB_fluxratio, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr,
               companion_is_host, twin, scalar_rule=False):
        if self._plain() and not scalar_rule:
            return super().lnl_eb(R_EB, EB_fluxratio, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr,
                                  companion_is_host, twin)
        if self.err is not None:
            model, sec = self.simulate_eb(self.full[0].size, R_EB, EB_fluxratio, P_orb, inc, a,
                                          R_s, u1, u2, ecc, argp, cfr, companion_is_host,
                                          scalar_rule)
            out = self._weighted(model)
            if not twin:
                out[~(sec < 1.5 * self.full[2])] = np.inf
            return out
        fn = coracle.lnL_EB_twin_p if twin else coracle.lnL_EB_p
        out = 0.0
        for g in range(len(self.groups)):
            self._use(g)
            t, f, s, e, n = self.lc
            out = out + fn(t, f, s, R_EB, EB_fluxratio, P_orb, inc, a, R_s, u1, u2, ecc, argp,
                           cfr, companion_is_host, e, n, scalar_rule=scalar_rule)
        return out

    def _weighted(self, model):
        f = self.full[1]
        return 0.5 * np.sum((f[None, :] - model) ** 2 / self.err[None, :] ** 2, axis=1)

    # ---- the L2 seam: masks as OracleEngine, lnL from the group sums
    def eval_tp(self, N, rp, P_orb, inc, ecc, argp, mtot, rhost, u1, u2, cfr, lnprior=None,
                extra_mask=None, companion_is_host=False, want_lnL=True, want_mask=False,
                n_best=0):
        if self._plain():
            return super().eval_tp(N, rp, P_orb, inc, ecc, argp, mtot, rhost, u1, u2, cfr,
                                   lnprior, extra_mask, companion_is_host)
        s = self.full[2]
        rp, P, inc, ecc, argp, mtot, rhost, u1, u2, cfr = [
            _full(x, N) for x in (rp, P_orb, inc, ecc, argp, mtot, rhost, u1, u2, cfr)]
        mask, a = tp_mask(N, rp, P, inc, ecc, argp, mtot, rhost, extra_mask)
        lnL = np.full(N, -np.inf)
        if mask.any():
            m = mask
            lnL[m] = -0.5 * ln2pi - np.log(s) - self.lnl_tp(
                rp[m], P[m], inc[m], a[m], rhost[m], u1[m], u2[m], ecc[m], argp[m], cfr[m],
                companion_is_host)
        res = _Res()
        res.N, res.lnL, res.mask, res.n_pass, res.n_stamps = N, lnL, mask, int(mask.sum()), 0
        return _lse_record(lnL if lnprior is None else lnL + _full(lnprior, N), N, res)

    def eval_eb(self, N, reb, ebfr, q, P_orb, inc, ecc, argp, mtot, rhost, u1, u2, cfr,
                lnprior=None, extra_mask=None, companion_is_host=False, want_lnL=True,
                want_mask=False, n_best=0, scalar_loop=False):
        if self._plain():
            return super().eval_eb(N, reb, ebfr, q, P_orb, inc, ecc, argp, mtot, rhost, u1, u2,
                                   cfr, lnprior, extra_mask, companion_is_host,
                                   scalar_loop=scalar_loop)
        s = self.full[2]
        reb, ebfr, q, P, inc, ecc, argp, mtot, rhost, u1, u2, cfr = [
            _full(x, N) for x in (reb, ebfr, q, P_orb, inc, ecc, argp, mtot, rhost, u1, u2, cfr)]
        out = []
        masks = eb_masks(N, reb, q, P, inc, ecc, argp, mtot, rhost, extra_mask, scalar_loop)
        for twin in (False, True):
            Pk = 2 * P if twin else P
            mask, a = masks[int(twin)]
            lnL = np.full(N, -np.inf)
            if mask.any():
                m = mask
                lnL[m] = -0.5 * ln2pi - np.log(s) - self.lnl_eb(
                    reb[m], ebfr[m], Pk[m], inc[m], a[m], rhost[m], u1[m], u2[m], ecc[m],
                    argp[m], cfr[m], companion_is_host, twin, scalar_rule=scalar_loop)
            res = _Res()
            res.N, res.lnL, res.mask, res.n_pass, res.n_stamps = N, lnL, mask, int(mask.sum()), 0
            out.append(_lse_record(lnL if lnprior is None else lnL + _full(lnprior, N), N, res))
        return tuple(out)

    # ---- simulate seam: each group's rows scattered back into stamp order
    def simulate_tp(self, npts, *args):
        if len(self.groups) == 1:
            return super().simulate_tp(npts, *args)
        out = np.empty((np.size(args[0]), npts))
        for g in range(len(self.groups)):
            idx = self._use(g)
            out[:, idx] = super().simulate_tp(idx.size, *args)
        return out

    def simulate_eb(self, npts, *args, **kw):
        if len(self.groups) == 1:
            return super().simulate_eb(npts, *args, **kw)
        out = np.empty((np.size(args[0]), npts))
        for g in range(len(self.groups)):
            idx = self._use(g)
            out[:, idx], sec = super().simulate_eb(idx.size, *args, **kw)
        return out, sec


def install():
    """Route triceratops_b200's host layer to a fresh CadenceOracleEngine."""
    from oracle.engine_port import install as _install
    return _install(CadenceOracleEngine())


def mixed_lightcurve(t, f, seed=0):
    """A two-cadence light curve: the folded curve (t, f) as 2-min stamps (exptime 0.00139 d,
    20 samples) plus its copy binned to 30 min (0.02083 d, 20 samples), shuffled so that the
    input is not grouped.  Returns (time, flux, exptime, nsamples)."""
    width = 0.02083
    b = np.floor((t - t.min()) / width).astype(np.int64)
    _, inv, cnt = np.unique(b, return_inverse=True, return_counts=True)
    tb = np.bincount(inv, weights=t) / cnt
    fb = np.bincount(inv, weights=f) / cnt
    time = np.concatenate([t, tb])
    flux = np.concatenate([f, fb])
    exptime = np.concatenate([np.full(t.size, 0.00139), np.full(tb.size, width)])
    nsamples = np.full(time.size, 20, dtype=np.int32)
    p = np.random.default_rng(seed).permutation(time.size)
    return time[p], flux[p], exptime[p], nsamples[p]
