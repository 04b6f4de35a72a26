"""Test helper: the CPU oracle engine (oracle/engine_port.py) with the moment pass of
tri_set_moments -- each result also carries s2 = sum exp(2 (lnw - m)) over its finite
ln-weights lnw = lnL + lnprior, computed from its own per-draw values.  The oracle itself is
unchanged.  `draws` keeps every branch's per-draw lnw (oldest first), `calls` every
evaluation's (key, [lnw per branch]); the key tells the scenario calls of calc_probs apart
(kind, light curve, whether a prior is applied)."""
import numpy as np

from oracle.engine_port import OracleEngine, _full, install  # noqa: F401
from triceratops_b200._numerics import lse_moments


class MomentsOracleEngine(OracleEngine):
    def __init__(self):
        self._moments = False
        self.draws = []
        self.calls = []

    def set_moments(self, on):
        self._moments = bool(on)

    def _attach(self, res, lnprior, N):
        lnw = res.lnL if lnprior is None else res.lnL + _full(lnprior, N)
        self.draws.append(lnw)
        res.s2 = lse_moments(lnw)[2] if self._moments else None
        return res

    def eval_tp(self, N, rp, P_orb, inc, ecc, argp, mtot, rhost, u1, u2, cfr, lnprior=None,
                extra_mask=None, companion_is_host=False, want_lnL=True, want_mask=False,
                n_best=0):
        res = super().eval_tp(N, rp, P_orb, inc, ecc, argp, mtot, rhost, u1, u2, cfr, lnprior,
                              extra_mask, companion_is_host)
        res = self._attach(res, lnprior, N)
        self.calls.append((self._key("tp", lnprior), [self.draws[-1]]))
        return res

    def eval_eb(self, N, reb, ebfr, q, P_orb, inc, ecc, argp, mtot, rhost, u1, u2, cfr,
                lnprior=None, extra_mask=None, companion_is_host=False, want_lnL=True,
                want_mask=False, n_best=0, scalar_loop=False):
        out = super().eval_eb(N, reb, ebfr, q, P_orb, inc, ecc, argp, mtot, rhost, u1, u2, cfr,
                              lnprior, extra_mask, companion_is_host, scalar_loop=scalar_loop)
        out = tuple(self._attach(r, lnprior, N) for r in out)
        self.calls.append((self._key("eb", lnprior), self.draws[-2:]))
        return out

    def _key(self, kind, lnprior):
        return kind, hash(self.lc[1].tobytes()), lnprior is None
