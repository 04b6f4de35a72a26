"""Host-side handle of the GPU engine: one process <-> one B200.

Wraps the C ABI (include/triceratops_b200.h) for numpy callers.  Device selection follows the
one-process-per-GPU launch convention (LOCAL_RANK), and results of ranks that hold disjoint
slices of the prior draws are merged with `combine_lse` (SURVEY.md section 8e).
"""
import ctypes
import functools
import math
import os
import threading

import numpy as np

from . import _cabi
from ._cabi import tri_col, tri_eb_args, tri_result, tri_tp_args

_engine = None
_engine_lock = threading.Lock()


def get_engine(device=None):
    """Process-wide engine bound to `device` (default: LOCAL_RANK or 0).  Safe to call from
    several threads: the first caller creates it (CUDA context, orbit table), the others wait."""
    global _engine
    if _engine is None:
        with _engine_lock:
            if _engine is None:
                _engine = Engine(device)
    if device is not None and device != _engine.device:
        raise RuntimeError("engine already bound to device %d" % _engine.device)
    return _engine


def cadence_columns(exptime, nsamples, npts):
    """Check the cadence of a light curve of `npts` stamps: `exptime` and `nsamples` are each a
    scalar or one value per stamp.  Returns (exptime, nsamples) as a float and an int when they
    hold one (exptime, nsamples) pair, else as a float64 and an int32 array of npts values (at
    most TRI_MAX_CADENCES distinct pairs, compared exactly).  Raises ValueError."""
    e = np.asarray(exptime)
    n = np.asarray(nsamples)
    for name, x in (("exptime", e), ("nsamples", n)):
        if x.ndim > 1 or (x.ndim == 1 and x.size != npts):
            raise ValueError("%s has shape %s; the light curve has %d time stamps"
                             % (name, x.shape, npts))
        if x.dtype.kind not in "biuf":
            raise ValueError("%s must be numeric" % name)
    e = np.broadcast_to(e.astype(np.float64), (npts,))
    if not np.all(np.isfinite(e)) or np.any(e < 0):
        raise ValueError("exptime must be finite and >= 0 at every stamp")
    if n.dtype.kind == "f" and not np.all(np.isfinite(n) & (n == np.floor(n))):
        raise ValueError("nsamples must be integral")
    if np.any(n < 1) or np.any(n > np.iinfo(np.int32).max):
        raise ValueError("nsamples must be >= 1 at every stamp")
    n = np.broadcast_to(n.astype(np.int32), (npts,))
    pairs = np.unique(np.stack([e, n.astype(np.float64)]), axis=1)
    if pairs.shape[1] > _cabi.TRI_MAX_CADENCES:
        raise ValueError("%d distinct (exptime, nsamples) pairs, at most %d are supported: round "
                         "the exposure times to their cadences"
                         % (pairs.shape[1], _cabi.TRI_MAX_CADENCES))
    if pairs.shape[1] == 1:
        return float(e[0]), int(n[0])
    return np.ascontiguousarray(e), np.ascontiguousarray(n)


class BranchResult:
    """One scenario branch: lnZ pieces + optional per-draw arrays."""
    __slots__ = ("lnZ", "m", "s", "n_finite", "n_posinf", "n_pass", "n_stamps", "n_interior",
                 "n_limb", "lnL", "mask", "N", "top_idx", "top_lnL", "n_evaluated", "branch",
                 "s2", "post_idx", "post_total")

    def __init__(self, r, N, lnL, mask, top=None, branch=0):
        self.lnZ, self.m, self.s = r.lnZ, r.m, r.s
        self.n_finite, self.n_posinf = r.n_finite, r.n_posinf
        self.n_pass, self.n_stamps = r.n_pass, r.n_stamps
        self.n_interior, self.n_limb = r.n_interior, r.n_limb
        self.lnL, self.mask, self.N = lnL, mask, N
        self.branch = branch
        self.s2 = None       # second moment of the weights (Engine.set_moments), set on wait
        # posterior samples (Engine.set_posterior), set on wait: int64 [K] draw indices in
        # ascending order ([0] when the posterior is empty) and T, the sum of the weights
        # relative to exp(m); None when off
        self.post_idx = self.post_total = None
        if top is not None:
            self.top_idx, self.top_lnL = top[0][:r.n_top], top[1][:r.n_top]
            self.n_evaluated = r.n_evaluated
        else:
            self.top_idx = self.top_lnL = None
            self.n_evaluated = None


def _locked(method):
    """The library is not re-entrant: every call into it (and the engine's own bookkeeping) is
    serialised, so that scenario functions running in different threads can share the engine."""
    @functools.wraps(method)
    def wrapper(self, *args, **kw):
        with self._lock:
            return method(self, *args, **kw)
    return wrapper


class Pending:
    """An evaluation queued with tri_submit_* and not necessarily finished.  `result()` waits
    for it (once) and returns what the synchronous call returns."""

    def __init__(self, engine, ticket, rr, n_branches, keep, build, n_best):
        self._engine, self._ticket, self._rr, self._nb = engine, ticket, rr, n_branches
        self._keep, self._build, self._n_best = keep, build, n_best
        self._moments = engine._moments     # (tri_set_moments is captured per submission)
        self._post_K = engine._post_K       # (and so is tri_set_posterior)
        self._out = None

    def done(self):
        return self._out is not None

    def result(self):
        with self._engine._lock:
            return self._result()

    def _result(self):
        if self._out is None:
            eng = self._engine
            try:
                _cabi.check(eng.lib.tri_wait(ctypes.c_int64(self._ticket), self._rr))
            finally:
                # the library has released the slot whether or not the wait succeeded: a failed
                # evaluation must not stay at the head of the queue (every later submit would
                # wait for its dead ticket again)
                if self in eng._inflight:
                    eng._inflight.remove(self)
            out = self._build(self._rr)
            if self._moments:
                s2 = (ctypes.c_double * 2)()
                _cabi.check(eng.lib.tri_last_moments(s2))
                for b, br in enumerate(out):
                    br.s2 = s2[b]
            if self._post_K > 0:
                for b, br in enumerate(out):
                    idx = np.empty(self._post_K, dtype=np.int64)
                    n, T = ctypes.c_int64(), ctypes.c_double()
                    _cabi.check(eng.lib.tri_last_posterior(
                        b, idx.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), idx.size,
                        ctypes.byref(n), ctypes.byref(T)))
                    br.post_idx, br.post_total = idx[:n.value], T.value
            # fewer finite draws than the table has rows: the caller pads the table from the
            # full lnL array, which is only reachable until the next evaluation completes
            for b, br in enumerate(out):
                if (self._n_best > 0 and br.lnL is None and br.N > 0
                        and br.n_evaluated is not None and br.n_evaluated < self._n_best):
                    br.lnL = eng.fetch_lnl(b, br.N)
            self._keep = None
            self._out = out[0] if self._nb == 1 else tuple(out)
        return self._out


_U64 = (1 << 64) - 1


def combine_lse(parts, N_total):
    """lnZ from per-rank (m, s, n_finite, n_posinf) records over disjoint slices of N_total draws.

    m = max_r m_r ; S = sum_r s_r exp(m_r - m) ; lnZ = m + ln S - ln N_total, with the
    reference's edge semantics (_numerics.py:46-51): any +inf -> +inf, nothing finite -> -inf.
    """
    if any(p[3] > 0 for p in parts):
        return math.inf
    fin = [p for p in parts if p[2] > 0]
    if not fin:
        return -math.inf
    m = max(p[0] for p in fin)
    S = sum(p[1] * math.exp(p[0] - m) for p in fin)
    return m + math.log(S) - math.log(N_total)


def combine_moments(parts):
    """Merged (m, s, s2, n_finite, n_posinf) of (m, s, s2, n_finite, n_posinf) records over
    disjoint slices of draws (ranks, or rounds of refinement): s and s2 are rescaled to the
    common maximum, s by exp(m_r - m) and s2 by exp(2 (m_r - m)).  lnZ itself is combine_lse's."""
    n_fin = sum(int(p[3]) for p in parts)
    n_pinf = sum(int(p[4]) for p in parts)
    fin = [p for p in parts if p[3] > 0]
    if not fin:
        return -math.inf, 0.0, 0.0, n_fin, n_pinf
    m = max(p[0] for p in fin)
    s = sum(p[1] * math.exp(p[0] - m) for p in fin)
    s2 = sum(p[2] * math.exp(2.0 * (p[0] - m)) for p in fin)
    return m, s, s2, n_fin, n_pinf


class Engine:
    def __init__(self, device=None):
        self.lib = _cabi.load()
        self._lock = threading.RLock()
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        self.device = int(device)
        _cabi.check(self.lib.tri_init(self.device))
        self._lc_key = None
        self._keep = []
        self._inflight = []      # Pendings not waited for yet, oldest first
        self._side_streams = None
        self._side_turn = 0
        self._moments = False
        self._post_K, self._post_seed = 0, 0

    @_locked
    def _make_room(self):
        """The library holds TRI_MAX_INFLIGHT evaluations: wait for the oldest when full."""
        while len(self._inflight) >= _cabi.TRI_MAX_INFLIGHT:
            self._inflight[0]._result()

    @_locked
    def drain(self):
        """Wait for everything in flight (results stay available from their Pendings)."""
        while self._inflight:
            self._inflight[0]._result()

    # ------------------------------------------------------------------ light curve
    @_locked
    def set_lightcurve(self, time, flux, sigma, exptime, nsamples):
        """Make (time, flux, sigma, exptime, nsamples) the current light curve.  sigma: a scalar
        or one error per stamp (tri_set_lightcurve_err); exptime and nsamples: scalars or one
        value per stamp, for a light curve that mixes cadences (tri_set_lightcurve_cadence, see
        cadence_columns).  Per-stamp cadences that hold one pair are the scalar call."""
        time = _cabi.f64(time)
        flux = _cabi.f64(flux)
        if time.shape != flux.shape or time.ndim != 1:
            raise ValueError("time and flux must be 1-D arrays of equal length")
        if np.ndim(exptime) != 0 or np.ndim(nsamples) != 0:
            exptime, nsamples = cadence_columns(exptime, nsamples, time.size)
        if np.ndim(exptime) != 0:   # several cadences (tri_set_lightcurve_cadence)
            err = None
            if np.ndim(sigma) != 0:
                err = _cabi.f64(sigma)
                if err.shape != time.shape:
                    raise ValueError("per-point errors must have the shape of time")
            key = (time.tobytes(), flux.tobytes(),
                   err.tobytes() if err is not None else np.float64(sigma).tobytes(),
                   exptime.tobytes(), nsamples.tobytes())
            if key == self._lc_key:
                return
            _cabi.check(self.lib.tri_set_lightcurve_cadence(
                _cabi.dptr(time), _cabi.dptr(flux), _cabi.dptr(err) if err is not None else None,
                float(sigma) if err is None else 0.0, _cabi.dptr(exptime),
                nsamples.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), time.size))
        elif np.ndim(sigma) == 0:
            key = (time.tobytes(), flux.tobytes(), float(sigma), float(exptime), int(nsamples))
            if key == self._lc_key:
                return
            _cabi.check(self.lib.tri_set_lightcurve(_cabi.dptr(time), _cabi.dptr(flux),
                                                    time.size, float(sigma), float(exptime),
                                                    int(nsamples)))
        else:   # one error per stamp (tri_set_lightcurve_err)
            err = _cabi.f64(sigma)
            if err.shape != time.shape:
                raise ValueError("per-point errors must have the shape of time")
            key = (time.tobytes(), flux.tobytes(), err.tobytes(), float(exptime), int(nsamples))
            if key == self._lc_key:
                return
            _cabi.check(self.lib.tri_set_lightcurve_err(_cabi.dptr(time), _cabi.dptr(flux),
                                                        _cabi.dptr(err), time.size,
                                                        float(exptime), int(nsamples)))
        self._lc_key = key

    # ------------------------------------------------------------------ helpers
    def _col(self, x, N):
        """numpy array of N values (stride 1) or scalar (stride 0) -> tri_col (keeps a ref)."""
        if x is None:
            return tri_col(None, 0)
        a = np.asarray(x, dtype=np.float64)
        if a.ndim == 0 or (a.size == 1 and N != 1):
            a = np.ascontiguousarray(a.reshape(1))
            stride = 0
        else:
            a = np.ascontiguousarray(a)
            if a.shape != (N,):
                raise ValueError("column has shape %s, expected (%d,)" % (a.shape, N))
            stride = 1
        self._keep.append(a)
        return tri_col(a.ctypes.data, stride)

    def _mask(self, m, N):
        if m is None:
            return None
        a = np.asarray(m)
        if a.dtype == np.bool_ and a.flags.c_contiguous:
            a = a.view(np.uint8)                       # (same bytes, no copy)
        else:
            a = np.ascontiguousarray(a.astype(np.uint8))
        if a.shape != (N,):
            raise ValueError("extra_mask has shape %s, expected (%d,)" % (a.shape, N))
        self._keep.append(a)
        return a.ctypes.data

    def _result(self, N, want_lnL, want_mask, n_best=0):
        r = tri_result()
        lnL = np.empty(N) if want_lnL else None
        mask = np.empty(N, dtype=np.uint8) if want_mask else None
        r.lnL_out = lnL.ctypes.data if want_lnL else None
        r.mask_out = mask.ctypes.data if want_mask else None
        top = None
        if n_best > 0:
            top = (np.zeros(n_best, dtype=np.int64), np.full(n_best, -np.inf))
            r.top_cap = n_best
            r.top_idx, r.top_lnL = top[0].ctypes.data, top[1].ctypes.data
        return r, lnL, mask, top

    @_locked
    def fetch_lnl(self, branch, N):
        """Per-draw lnL of the most recent eval_tp / eval_eb call (kept on the device)."""
        out = np.empty(int(N))
        _cabi.check(self.lib.tri_fetch_lnl(int(branch), _cabi.dptr(out), int(N)))
        return out

    # ------------------------------------------------------------------ L2 seam
    def eval_tp(self, *args, **kw):
        return self.submit_tp(*args, **kw).result()

    def eval_eb(self, *args, **kw):
        return self.submit_eb(*args, **kw).result()

    @_locked
    def submit_tp(self, N, rp, P_orb, inc, ecc, argp, mtot, rhost, u1, u2, cfr, lnprior=None,
                  extra_mask=None, companion_is_host=False, want_lnL=True, want_mask=False,
                  n_best=0, lightcurve=None, post_stream=0):
        """Queue a TP-type evaluation (tri_submit_tp) and return its Pending: the column copies
        overlap the kernels of the call submitted before.  `eval_tp` is submit + result().
        `lightcurve` = (time, flux, sigma, exptime, nsamples) makes that the current light
        curve in the same critical section (callers in several threads).  `post_stream`: the
        stream of the posterior samples' U (set_posterior)."""
        N = int(N)
        if lightcurve is not None:
            self.set_lightcurve(*lightcurve)
        self._make_room()
        self._keep = []
        a = tri_tp_args()
        a.N = N
        for name, val in (("rp", rp), ("P_orb", P_orb), ("inc", inc), ("ecc", ecc),
                          ("argp", argp), ("mtot", mtot), ("rhost", rhost), ("u1", u1),
                          ("u2", u2), ("cfr", cfr), ("lnprior", lnprior)):
            setattr(a, name, self._col(val, N))
        a.extra_mask = self._mask(extra_mask, N)
        a.companion_is_host = int(bool(companion_is_host))
        r, lnL, mask, top = self._result(N, want_lnL, want_mask, n_best)
        rr = (tri_result * 1)(r)
        ticket = ctypes.c_int64()
        self._arm_posterior(post_stream)
        _cabi.check(self.lib.tri_submit_tp(ctypes.byref(a), rr, ctypes.byref(ticket)))
        keep, self._keep = self._keep + [a, lnL, mask, top], []

        def build(rr):
            return [BranchResult(rr[0], N, lnL, mask.astype(bool) if mask is not None else None,
                                 top, 0)]
        p = Pending(self, ticket.value, rr, 1, keep, build, n_best)
        self._inflight.append(p)
        return p

    @_locked
    def submit_eb(self, N, reb, ebfr, q, P_orb, inc, ecc, argp, mtot, rhost, u1, u2, cfr,
                  lnprior=None, extra_mask=None, companion_is_host=False, want_lnL=True,
                  want_mask=False, n_best=0, lightcurve=None, scalar_loop=False, post_stream=0):
        """EB-type counterpart of submit_tp.  scalar_loop=True evaluates with the semantics of
        the reference's parallel=False loops (see tri_eb_args.scalar_loop)."""
        N = int(N)
        if lightcurve is not None:
            self.set_lightcurve(*lightcurve)
        self._make_room()
        self._keep = []
        a = tri_eb_args()
        a.N = N
        for name, val in (("reb", reb), ("ebfr", ebfr), ("q", q), ("P_orb", P_orb), ("inc", inc),
                          ("ecc", ecc), ("argp", argp), ("mtot", mtot), ("rhost", rhost),
                          ("u1", u1), ("u2", u2), ("cfr", cfr), ("lnprior", lnprior)):
            setattr(a, name, self._col(val, N))
        a.extra_mask = self._mask(extra_mask, N)
        a.companion_is_host = int(bool(companion_is_host))
        a.scalar_loop = int(bool(scalar_loop))
        rr = (tri_result * 2)()
        outs = []
        for b in range(2):
            r, lnL, mask, top = self._result(N, want_lnL, want_mask, n_best)
            rr[b] = r
            outs.append((lnL, mask, top))
        ticket = ctypes.c_int64()
        self._arm_posterior(post_stream)
        _cabi.check(self.lib.tri_submit_eb(ctypes.byref(a), rr, ctypes.byref(ticket)))
        keep, self._keep = self._keep + [a, outs], []

        def build(rr):
            return [BranchResult(rr[b], N, outs[b][0],
                                 outs[b][1].astype(bool) if outs[b][1] is not None else None,
                                 outs[b][2], b)
                    for b in range(2)]
        p = Pending(self, ticket.value, rr, 2, keep, build, n_best)
        self._inflight.append(p)
        return p

    # ------------------------------------------------------------------ L2 seam, device columns
    def _tensor_col(self, x, N, keep):
        """torch CUDA float64 tensor of N values (stride 1) or scalar (stride 0) -> tri_col."""
        import torch
        if x is None:
            return tri_col(None, 0)
        if torch.is_tensor(x) and x.ndim == 1 and x.numel() == N and N != 1:
            t = x.contiguous()
            if t.dtype != torch.float64:
                t = t.double()
            stride = 1
        else:
            t = torch.as_tensor(x, dtype=torch.float64, device=self._torch_device()).reshape(-1)
            if t.numel() != 1 and t.numel() != N:
                raise ValueError("column has %d values, expected %d" % (t.numel(), N))
            t = t.to(self._torch_device()).contiguous()
            stride = 0 if t.numel() == 1 and N != 1 else 1
        keep.append(t)
        return tri_col(t.data_ptr(), stride)

    def _torch_device(self):
        import torch
        return torch.device("cuda", self.device)

    def _tensor_result(self, N, n_best, keep):
        import torch
        r = tri_result()
        ti = torch.zeros(max(n_best, 1), dtype=torch.int64, device=self._torch_device())
        tv = torch.full((max(n_best, 1),), -math.inf, dtype=torch.float64,
                        device=self._torch_device())
        keep += [ti, tv]
        r.top_cap = n_best
        r.top_idx, r.top_lnL = ti.data_ptr(), tv.data_ptr()
        return r, ti, tv

    @staticmethod
    def _sorted_top(r, ti, tv):
        """Device-pointer calls return the candidates unsorted: best first, ties by index."""
        k = int(r.n_top)
        idx = ti[:k].cpu().numpy()
        val = tv[:k].cpu().numpy()
        order = np.lexsort((idx, -val))
        return idx[order], val[order]

    @_locked
    def _submit_tensors(self, kind, N, cols, extra_mask, companion_is_host, n_best,
                        lightcurve=None, scalar_loop=False, post_stream=0):
        import torch
        N = int(N)
        if lightcurve is not None:
            self.set_lightcurve(*lightcurve)
        self._make_room()
        keep = []
        a = tri_tp_args() if kind == "tp" else tri_eb_args()
        a.N = N
        for name, val in cols.items():
            setattr(a, name, self._tensor_col(val, N, keep))
        if extra_mask is not None:
            m = extra_mask.to(torch.uint8).contiguous()
            keep.append(m)
            a.extra_mask = m.data_ptr()
        a.companion_is_host = int(bool(companion_is_host))
        if kind == "eb":
            a.scalar_loop = int(bool(scalar_loop))
        nb = 1 if kind == "tp" else 2
        rr = (tri_result * nb)()
        tops = []
        for b in range(nb):
            rr[b], ti, tv = self._tensor_result(N, n_best, keep)
            tops.append((ti, tv))
        # The evaluation runs on one of two side streams, ordered after what torch's current
        # stream has queued so far (the kernels that produced the columns): the sampler kernels
        # of the next scenario then overlap this evaluation's tail instead of queueing behind it.
        # The columns stay referenced by the Pending until the evaluation has completed.
        cur = torch.cuda.current_stream(self._torch_device())
        if self._side_streams is None:
            self._side_streams = [torch.cuda.Stream(self._torch_device()) for _ in range(2)]
        side = self._side_streams[self._side_turn]
        self._side_turn ^= 1
        side.wait_stream(cur)
        stream = side.cuda_stream
        fn = self.lib.tri_submit_tp_dev if kind == "tp" else self.lib.tri_submit_eb_dev
        ticket = ctypes.c_int64()
        self._arm_posterior(post_stream)
        _cabi.check(fn(ctypes.byref(a), rr, ctypes.c_void_p(stream), ctypes.byref(ticket)))
        keep.append(a)

        def build(rr):
            return [BranchResult(rr[b], N, None, None, self._sorted_top(rr[b], *tops[b]), b)
                    for b in range(nb)]
        p = Pending(self, ticket.value, rr, nb, keep, build, 0)
        self._inflight.append(p)
        return p

    def submit_tp_tensors(self, N, cols, extra_mask=None, companion_is_host=False, n_best=100,
                          lightcurve=None, post_stream=0):
        """tri_submit_tp_dev on torch CUDA tensors (columns: rp, P_orb, inc, ecc, argp, mtot,
        rhost, u1, u2, cfr, lnprior; tensors of N values or scalars), queued on torch's current
        stream behind the kernels that produce them.  Returns a Pending."""
        return self._submit_tensors("tp", N, cols, extra_mask, companion_is_host, n_best,
                                    lightcurve, post_stream=post_stream)

    def submit_eb_tensors(self, N, cols, extra_mask=None, companion_is_host=False, n_best=100,
                          lightcurve=None, scalar_loop=False, post_stream=0):
        return self._submit_tensors("eb", N, cols, extra_mask, companion_is_host, n_best,
                                    lightcurve, scalar_loop, post_stream)

    def eval_tp_tensors(self, *args, **kw):
        return self.submit_tp_tensors(*args, **kw).result()

    def eval_eb_tensors(self, *args, **kw):
        return self.submit_eb_tensors(*args, **kw).result()

    # ------------------------------------------------------------------ L1 seam
    @_locked
    def lnl_tp(self, R_p, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr, companion_is_host):
        n = int(np.size(R_p))
        cols = [self._full(x, n) for x in (R_p, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr)]
        out = np.empty(n)
        _cabi.check(self.lib.tri_lnl_tp(n, *[_cabi.dptr(c) for c in cols],
                                        int(bool(companion_is_host)), _cabi.dptr(out)))
        return out

    @_locked
    def lnl_eb(self, R_EB, EB_fluxratio, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr,
               companion_is_host, twin):
        n = int(np.size(R_EB))
        cols = [self._full(x, n) for x in (R_EB, EB_fluxratio, P_orb, inc, a, R_s, u1, u2, ecc,
                                           argp, cfr)]
        out = np.empty(n)
        _cabi.check(self.lib.tri_lnl_eb(n, *[_cabi.dptr(c) for c in cols],
                                        int(bool(companion_is_host)), int(bool(twin)),
                                        _cabi.dptr(out)))
        return out

    # ------------------------------------------------------------------ simulate seam
    @_locked
    def simulate_tp(self, npts, R_p, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr,
                    companion_is_host):
        n = int(np.size(R_p))
        cols = [self._full(x, n) for x in (R_p, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr)]
        out = np.empty((n, int(npts)))
        if n:
            _cabi.check(self.lib.tri_simulate_tp(n, *[_cabi.dptr(c) for c in cols],
                                                 int(bool(companion_is_host)), _cabi.dptr(out)))
        return out

    @_locked
    def simulate_eb(self, npts, R_EB, EB_fluxratio, P_orb, inc, a, R_s, u1, u2, ecc, argp, cfr,
                    companion_is_host, scalar_rule=False):
        n = int(np.size(R_EB))
        cols = [self._full(x, n) for x in (R_EB, EB_fluxratio, P_orb, inc, a, R_s, u1, u2, ecc,
                                           argp, cfr)]
        out = np.empty((n, int(npts)))
        sec = np.empty(n)
        if n:
            _cabi.check(self.lib.tri_simulate_eb(n, *[_cabi.dptr(c) for c in cols],
                                                 int(bool(companion_is_host)),
                                                 int(bool(scalar_rule)), _cabi.dptr(out),
                                                 _cabi.dptr(sec)))
        return out, sec

    @staticmethod
    def _full(x, n):
        a = np.asarray(x, dtype=np.float64)
        if a.ndim == 0:
            a = np.full(n, float(a))
        a = np.ascontiguousarray(a)
        if a.shape != (n,):
            raise ValueError("array has shape %s, expected (%d,)" % (a.shape, n))
        return a

    # ------------------------------------------------------------------ misc
    @_locked
    def log_mean_exp(self, logw):
        logw = _cabi.f64(logw)
        r = tri_result()
        _cabi.check(self.lib.tri_log_mean_exp(_cabi.dptr(logw), logw.size, ctypes.byref(r)))
        return r.lnZ, (r.m, r.s, r.n_finite, r.n_posinf)

    @_locked
    def last_timing(self):
        g, l, s = ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
        n = ctypes.c_int32()
        _cabi.check(self.lib.tri_last_timing(ctypes.byref(g), ctypes.byref(l), ctypes.byref(s),
                                             ctypes.byref(n)))
        return {"geometry_ms": g.value, "lnl_ms": l.value, "lse_ms": s.value,
                "launches": n.value}

    @_locked
    def set_counting(self, on):
        """Work counters of the roofline model (n_stamps, n_interior, n_limb) on / off."""
        _cabi.check(self.lib.tri_set_counting(int(bool(on))))

    @_locked
    def set_moments(self, on):
        """Second moment of the weights per branch (tri_set_moments): BranchResult.s2 of the
        evaluations submitted while it is on, None otherwise."""
        _cabi.check(self.lib.tri_set_moments(int(bool(on))))
        self._moments = bool(on)

    @_locked
    def set_posterior(self, K, seed=0):
        """K posterior samples per branch of every evaluation submitted while K > 0
        (tri_set_posterior): BranchResult.post_idx / post_total.  The third part of the hash
        that gives U, the stream, is passed with each submission (`post_stream`)."""
        K, seed = int(K), int(seed) & _U64
        _cabi.check(self.lib.tri_set_posterior(K, seed, 0))
        self._post_K, self._post_seed = K, seed

    def _arm_posterior(self, post_stream):
        """Hand the submission's stream to tri_set_posterior (lock held, K > 0 only)."""
        if self._post_K > 0:
            _cabi.check(self.lib.tri_set_posterior(self._post_K, self._post_seed,
                                                   int(post_stream) & _U64))

    @_locked
    def fp64_peak(self):
        v = ctypes.c_double()
        _cabi.check(self.lib.tri_fp64_peak(ctypes.byref(v)))
        return v.value

    @_locked
    def sm_count(self):
        n = ctypes.c_int32()
        _cabi.check(self.lib.tri_sm_count(ctypes.byref(n)))
        return n.value
