"""Glue between the lnZ_* host functions and the GPU engine: sharding of the prior draws over
ranks (one process per GPU), the single small collective that merges the per-rank
(max, scaled-sum) records and best-draw candidates, and selection of the 100 best draws
(reference marginal_likelihoods.py:152-154).

Sharding follows SURVEY.md section 8e: rank r evaluates the contiguous slice
[r*N/G, (r+1)*N/G) of every scenario's draws and contributes one record per scenario branch
(pack_slice): the evidence header, its 100 best (lnL, global index) candidates -- with their
rows where only this rank holds them (device sampler) -- and with posterior samples their
indices (and rows); no per-draw data is exchanged.  merge_slices merges the records of the
ranks, and likewise those of the rounds of fpp_err_target refinement (triceratops._merge_round).

  * a single lnZ_* call under a process group: every rank makes the same host draws (same
    seed) and the records are merged with one all-gather per call;
  * `target.calc_probs` (CallGroup): the records of ALL scenario rows travel in ONE all-gather
    at the end of the call.  With numpy's draws (host sampler) rank 0 alone runs the scenario
    functions -- the generator is sequential, repeating it on every rank would only divide
    the host's cores -- and scatters each engine call's columns to the ranks (pinned host ->
    device -> NCCL scatter over NVLink); the other ranks evaluate what they receive.
"""
import contextlib
import threading

import numpy as np

from . import _cabi, _numerics
from . import engine as _engine_mod

N_BEST = 100

def get_engine():
    """The process-wide CUDA engine.  There is no other engine in the product: the CPU tests
    and bench.py's recorder / CPU arm stand in for it by patching this name from outside."""
    return _engine_mod.get_engine()


_sharding = True


class no_sharding:
    """Context manager: evaluate every draw on this rank even inside a process group (used when
    whole targets, not draws, are distributed over the ranks -- batch.vet_many)."""

    def __enter__(self):
        global _sharding
        self._prev, _sharding = _sharding, False

    def __exit__(self, *exc):
        global _sharding
        _sharding = self._prev


def _dist():
    if not _sharding:
        return None
    try:
        import torch.distributed as dist
    except Exception:  # pragma: no cover
        return None
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist
    return None


def shard_bounds(N, rank=None, world=None):
    """Contiguous slice of the N draws owned by `rank`."""
    d = _dist()
    if rank is None:
        rank = d.get_rank() if d else 0
    if world is None:
        world = d.get_world_size() if d else 1
    return (rank * N) // world, ((rank + 1) * N) // world


def _slice(x, lo, hi):
    if x is None or np.ndim(x) == 0:
        return x
    return x[lo:hi]


def _mask_slice(m, lo, hi):
    """AND-term of the mask for this rank; None when it excludes nothing (saves the upload)."""
    if m is None:
        return None
    m = m[lo:hi]
    return None if m.all() else m


def best_indices(lnL, n_best=N_BEST):
    """First n_best entries of (-lnL).argsort() (marginal_likelihoods.py:152-153) without a
    full sort when enough finite entries exist."""
    n = lnL.size
    if n <= 4 * n_best:
        return (-lnL).argsort()[:n_best]
    neg = -lnL
    cand = np.argpartition(neg, n_best)[:n_best]
    vals = neg[cand]
    if not np.all(np.isfinite(vals)):
        # fewer than n_best finite draws: the reference's order among the -inf entries is that
        # of numpy's sort on the full array
        return neg.argsort()[:n_best]
    order = np.lexsort((cand, vals))
    return cand[order][:n_best]


# ---- Monte-Carlo error bars (tri_set_moments) ----------------------------------------------------
_moments = 0      # > 0 inside mc_errors(): engine calls also return s2 (process-wide)


@contextlib.contextmanager
def mc_errors():
    """Inside this context the engine also sums the second moment of the weights of every
    scenario branch, and the lnZ_* results carry N, s2, lnZ_err and ess (ScenarioResult)."""
    global _moments
    _moments += 1
    try:
        yield
    finally:
        _moments -= 1


def _sync_moments(eng):
    """Switch the engine's moment pass to what the caller's context asks for (engines without
    one -- test stand-ins -- are left alone while moments are off)."""
    want = _moments > 0
    if want or getattr(eng, "_moments", False):
        eng.set_moments(want)


# ---- posterior samples (tri_set_posterior) ------------------------------------------------------
_post = None      # [K, seed, next stream] inside posterior_samples() (process-wide)
_post_lock = threading.Lock()


def check_posterior_K(K):
    """K as an int, or ValueError: an integer in [1, TRI_MAX_POSTERIOR]."""
    if isinstance(K, bool) or not isinstance(K, (int, np.integer)):
        raise ValueError("posterior_samples must be an integer, got %r" % (K,))
    if not 1 <= int(K) <= _cabi.TRI_MAX_POSTERIOR:
        raise ValueError("posterior_samples must be in [1, %d], got %d"
                         % (_cabi.TRI_MAX_POSTERIOR, int(K)))
    return int(K)


@contextlib.contextmanager
def posterior_samples(K, seed=0):
    """Inside this context every scenario evaluation also draws K posterior samples per branch
    (systematic importance resampling on the GPU).  Each engine call takes the next stream of a
    per-context counter, unless the caller names it (call_stream)."""
    global _post
    K = check_posterior_K(K)
    prev, _post = _post, [K, int(seed), 0]
    try:
        yield
    finally:
        _post = prev


@contextlib.contextmanager
def call_stream(stream):
    """The stream of the posterior samples of the engine calls this thread makes inside."""
    prev = getattr(_tls, "post_stream", None)
    _tls.post_stream = int(stream)
    try:
        yield
    finally:
        _tls.post_stream = prev


def _next_post():
    """(K, seed, stream) of the engine call being submitted, None when posterior samples are
    off."""
    if _post is None:
        return None
    s = getattr(_tls, "post_stream", None)
    if s is None:
        with _post_lock:
            s = _post[2]
            _post[2] += 1
    return _post[0], _post[1], s


def _post_kw(eng, post):
    """Switch the engine's posterior samples to `post` (engines without them -- test
    stand-ins -- are left alone while they are off); the submission's keyword."""
    if post is not None or getattr(eng, "_post_K", 0):
        eng.set_posterior(post[0] if post else 0, post[1] if post else 0)
    return {} if post is None else {"post_stream": post[2]}


class Branch:
    """One scenario branch merged over its slices of draws (merge_slices): lnZ over all N draws;
    record = (m, s, s2, n_finite, n_posinf) (s2 None without moments); the finite best-draw
    candidates, best first: global draw indices `idx`, lnL `vals` and, where their rows travelled
    with them, `rows` [k, R]; with posterior samples, their global draw indices `post_idx`
    (ascending), rows `post_rows` and total weight `post_total` relative to exp(record[0]), else
    None."""
    __slots__ = ("lnZ", "N", "record", "n_pass", "n_evaluated", "idx", "vals", "rows",
                 "post_idx", "post_rows", "post_total")


def _local_best(res, eng, single_rank):
    """(indices, lnL values, number of draws with finite lnL) of this rank's best draws.

    The CUDA engine selects them on the device (no per-draw read-back), best first, ties in
    index order.  With fewer than N_BEST finite draws the reference pads its table with
    zero-weight draws in the order numpy's argsort happens to give the -inf entries; a single
    rank reproduces that by fetching the array (single_rank=True)."""
    top_idx = getattr(res, "top_idx", None)
    if top_idx is not None:
        if single_rank and res.n_evaluated < N_BEST and res.N > 0:
            # (the engine fetched the array when the evaluation completed)
            lnL = res.lnL if res.lnL is not None else eng.fetch_lnl(res.branch, res.N)
            idx = best_indices(lnL)
            return idx, lnL[idx], int(res.n_evaluated)
        return top_idx, res.top_lnL, int(res.n_evaluated)
    if res.lnL is None or not res.lnL.size:
        return np.zeros(0, dtype=np.int64), np.zeros(0), 0
    idx = best_indices(res.lnL)
    return idx, res.lnL[idx], int(np.isfinite(res.lnL).sum())


def _allgather(mat, d):
    """numpy [rows, cols] of every rank -> [world, rows, cols] (one collective)."""
    import torch
    world = d.get_world_size()
    dev = "cuda" if d.get_backend() == "nccl" else "cpu"
    mine = torch.from_numpy(np.ascontiguousarray(mat, dtype=np.float64).reshape(-1)).to(dev)
    allrec = torch.empty(world * mine.numel(), dtype=torch.float64, device=dev)
    d.all_gather_into_tensor(allrec, mine)
    return allrec.cpu().numpy().reshape((world,) + tuple(np.shape(mat)))


def gather_records(records, N_total):
    """Global evidences from this rank's (m, s, n_finite, n_posinf) records of several scenario
    branches over disjoint slices of N_total draws each: ONE all-gather for all of them."""
    d = _dist()
    if d is None:
        return [_engine_mod.combine_lse([r], N_total) for r in records]
    allrec = _allgather(np.asarray(records, dtype=np.float64).reshape(len(records), 4), d)
    return [_engine_mod.combine_lse([tuple(allrec[r, j]) for r in range(allrec.shape[0])],
                                    N_total) for j in range(len(records))]


# ---- the record of a branch over one slice of draws, and the merge of slices -------------------
H = 7   # header: m, s, n_finite, n_posinf, n_pass, n_evaluated, s2


def pack_slice(m, s, n_finite, n_posinf, n_pass, n_eval, s2, idx, vals, rows=None, post=None):
    """A branch over one slice of draws (a rank's, or a round's of refinement) as one float64
    row: the header (s2 None -> NaN); the N_BEST finite candidates' lnL values, then their
    GLOBAL draw indices (NaN past them); with `rows` ([candidates, R]) their N_BEST x R rows;
    with posterior samples, post = (K, T, global indices[, rows]) appends T, K indices and K x R
    rows (NaN where the posterior is empty).  R = 0 where the rows can be looked up by index
    after the merge (host sampler); R = len(RESULT_KEYS) where they live only where they were
    drawn (device sampler) or in an earlier round (refinement)."""
    R = 0 if rows is None else np.shape(rows)[1]
    P = H + N_BEST * (2 + R)
    K = 0 if post is None else post[0]
    rec = np.full(P + (0 if post is None else 1 + K * (1 + R)), np.nan)
    rec[:H] = (m, s, n_finite, n_posinf, n_pass, n_eval, np.nan if s2 is None else s2)
    vals = np.asarray(vals)
    fin = np.isfinite(vals)
    k = int(fin.sum())
    rec[H:H + k] = vals[fin]
    rec[H + N_BEST:H + N_BEST + k] = np.asarray(idx)[fin]
    if R:
        rec[H + 2 * N_BEST:H + 2 * N_BEST + k * R] = np.asarray(rows)[fin].ravel()
    if post is not None:
        n = len(post[2])
        rec[P] = post[1]
        rec[P + 1:P + 1 + n] = post[2]
        if R:
            rec[P + 1 + K:P + 1 + K + n * R] = np.asarray(post[3]).ravel()
    return rec


def merge_slices(allrec, N, R=0, lnZ=None, post=None, branch=0):
    """Branch of [slices, width] records (pack_slice, slices in draw order) over N draws in all.
    lnZ and the record merge with combine_lse / combine_moments; one slice keeps the engine's
    numbers: `lnZ` and its header as they are.  The candidates are the finite ones ordered by
    (lnL descending, global index ascending), cut to N_BEST, with their rows where R > 0.  With
    post = (K, seed, stream) of the call and the records' tails, the posterior samples merge with
    merge_posteriors, each taking its row along.  No padding: the callers fill their tables."""
    br = Branch()
    hd = allrec[:, :H].tolist()
    br.N, br.n_pass, br.n_evaluated = N, int(sum(r[4] for r in hd)), int(sum(r[5] for r in hd))
    if len(hd) == 1:
        br.lnZ = lnZ
        m, s, n_fin, n_pinf, _, _, s2 = hd[0]
    else:
        br.lnZ = _engine_mod.combine_lse([(r[0], r[1], int(r[2]), int(r[3])) for r in hd], N)
        m, s, s2, n_fin, n_pinf = _engine_mod.combine_moments(
            [(r[0], r[1], r[6], r[2], r[3]) for r in hd])
    br.record = (m, s, None if any(np.isnan(r[6]) for r in hd) else s2, int(n_fin), int(n_pinf))
    P = H + N_BEST * (2 + R)
    vals = allrec[:, H:H + N_BEST].ravel()
    gidx = allrec[:, H + N_BEST:H + 2 * N_BEST].ravel()
    ok = ~np.isnan(gidx)
    vals, gidx = vals[ok], gidx[ok].astype(np.int64)
    order = np.lexsort((gidx, -vals))[:N_BEST]
    br.vals, br.idx, br.rows = vals[order], gidx[order], None
    if R:
        br.rows = allrec[:, H + 2 * N_BEST:P].reshape(-1, R)[ok][order]
    br.post_idx = br.post_rows = br.post_total = None
    if post is not None and allrec.shape[1] > P:
        K = post[0]
        parts, rows = [], []
        for r in allrec:
            t = r[P + 1:P + 1 + K]
            n = int((~np.isnan(t)).sum())
            parts.append((r[0], r[P], t[:n].astype(np.int64)))
            rows.append(r[P + 1 + K:P + 1 + K + n * R].reshape(n, R))
        br.post_idx, _, br.post_total = _numerics.merge_posteriors(parts, K, *post[1:], branch)
        if R:   # (the slices' samples are disjoint and ascending)
            pos = np.searchsorted(np.concatenate([p[2] for p in parts]), br.post_idx)
            br.post_rows = np.concatenate(rows)[pos]
    return br


def gather_slices(rec, group=None, key=None):
    """[ranks, width] records of one branch: this rank's alone without a process group, the
    rows of `key` after the CallGroup's exchange, else those of an all-gather of its own."""
    d = _dist()
    if d is None:
        return rec[None, :]
    if group is not None:
        return group.rows(key)
    return _allgather(rec[None, :], d)[:, 0, :]


def _host_record(res, lo, eng, post):
    """This rank's record of one branch of the host sampler (R = 0: _result looks the rows up by
    index); post = (K, seed, stream) of the call or None."""
    idx, vals, n_eval = _local_best(res, eng, False)
    tail = None
    if post is not None and getattr(res, "post_idx", None) is not None:
        tail = (post[0], res.post_total, np.asarray(res.post_idx, dtype=np.int64) + lo)
    return pack_slice(res.m, res.s, res.n_finite, res.n_posinf, res.n_pass, n_eval,
                      getattr(res, "s2", None), np.asarray(idx) + lo, vals, post=tail)


def _host_branch(allrec, res, N, eng, post, branch):
    """Merged Branch of the host sampler with idx holding the table's min(N_BEST, N) draws.  The
    rows past the finite candidates carry zero weight: on one rank they come in the order of
    the reference's argsort over the whole lnL array; across ranks every rank appends the lowest
    draw indices not yet listed, so that all ranks build the same table."""
    br = merge_slices(allrec, N, lnZ=res.lnZ, post=post, branch=branch)
    if len(allrec) == 1:
        br.idx = _local_best(res, eng, True)[0]
        return br
    idx, want = br.idx, min(N_BEST, N)
    if idx.size < want:
        taken = set(idx.tolist())
        extra = [i for i in range(min(N, want + idx.size)) if i not in taken][:want - idx.size]
        br.idx = np.concatenate([idx, np.asarray(extra, dtype=np.int64)])
    return br


# ---- one exchange per calc_probs ----------------------------------------------------------------
_group = None     # the CallGroup of the calc_probs call in progress (process-wide)


class CallGroup:
    """A `target.calc_probs` call under a process group.  Every scenario branch registers its
    local record under a key that is the same on all ranks; `exchange()` moves all of them
    with ONE all-gather.  scatter=True (host sampler): rank 0 runs the scenario functions and
    hands each engine call's columns to the ranks (`scatter_submit`), the others `follow()`."""

    def __init__(self, d, scatter):
        self.d, self.scatter = d, bool(scatter)
        self.world, self.rank = d.get_world_size(), d.get_rank()
        self.is_root = self.rank == 0
        self.lock = threading.RLock()
        self.records, self.all = {}, None
        self.auto = self.seq = 0
        self.lc_key = None
        self.collectives = 0          # exchanges of records (the contract: one per call)
        self.scatters = 0             # engine calls whose columns were distributed
        self.device = "cuda" if d.get_backend() == "nccl" else "cpu"

    # -- records
    def add(self, rec, key=None):
        with self.lock:
            if key is None:
                key = ("a", self.auto)
                self.auto += 1
            self.records[key] = np.asarray(rec, dtype=np.float64)
        return key

    def exchange(self):
        keys = sorted(self.records)
        width = max([self.records[k].size for k in keys] + [1])
        mat = np.full((max(len(keys), 1), width), np.nan)
        for i, k in enumerate(keys):
            mat[i, :self.records[k].size] = self.records[k]
        allrec = _allgather(mat, self.d)
        self.collectives += 1
        self.all = {k: allrec[:, i, :self.records[k].size] for i, k in enumerate(keys)}

    def rows(self, key):
        if self.all is None:
            raise RuntimeError("CallGroup.exchange() has not run yet")
        return self.all[key]

    # -- rank 0 draws, everybody evaluates
    def _bcast(self, obj=None):
        box = [obj]
        self.d.broadcast_object_list(box, src=0)
        return box[0]

    def _evaluate(self, eng, hdr, mine, lc):
        """Submit this rank's slice of one engine call (device / CPU tensors)."""
        n = hdr["bounds"][self.rank + 1] - hdr["bounds"][self.rank]
        cols = {k: mine[j, :n] for j, k in enumerate(hdr["arrays"])}
        cols.update(hdr["scalars"])
        cols.update({k: None for k in hdr["absent"]})
        mask = (mine[len(hdr["arrays"]), :n] != 0) if hdr["has_mask"] else None
        name = hdr["kind"] + "_tensors"
        kw = dict(extra_mask=mask, companion_is_host=hdr["is_host"], n_best=N_BEST)
        if hdr["scalar_loop"]:
            kw["scalar_loop"] = True
        _sync_moments(eng)
        kw.update(_post_kw(eng, hdr["post"]))
        fn = getattr(eng, "submit_" + name, None)
        if fn is not None:
            return fn(n, cols, lightcurve=lc, **kw)
        with _fallback_lock:     # stand-in engines (CPU tests): one call at a time
            if lc is not None:
                eng.set_lightcurve(*lc)
            return _Done(getattr(eng, "eval_" + name)(n, cols, **kw))

    def scatter_submit(self, eng, kind, N, cols, extra_mask, is_host, scalar_loop=False,
                       post=None):
        """Rank 0: announce one engine call, scatter its per-draw columns, evaluate the own
        slice.  Returns (pending, lo, seq)."""
        import torch
        lc = current_lightcurve()
        arrays = [k for k, v in cols.items()
                  if v is not None and np.ndim(v) == 1 and np.size(v) == N and N != 1]
        scalars = {k: float(np.asarray(v, dtype=np.float64).reshape(-1)[0])
                   for k, v in cols.items() if v is not None and k not in arrays}
        absent = [k for k, v in cols.items() if v is None]
        bounds = [(r * N) // self.world for r in range(self.world + 1)]
        chunk = max(max(bounds[r + 1] - bounds[r] for r in range(self.world)), 1)
        ncol = len(arrays) + (extra_mask is not None)
        with self.lock:
            seq = self.seq
            self.seq += 1
            # (bytes: exptime and nsamples may be arrays, one value per stamp)
            key = None if lc is None else (
                np.asarray(lc[0]).tobytes(), np.asarray(lc[1]).tobytes(),
                np.asarray(lc[2], dtype=np.float64).tobytes(),
                np.asarray(lc[3], dtype=np.float64).tobytes(), np.asarray(lc[4]).tobytes())
            send_lc = lc if key != self.lc_key else None
            self.lc_key = key
            hdr = dict(op="call", seq=seq, kind=kind, N=N, arrays=arrays, scalars=scalars,
                       absent=absent, has_mask=extra_mask is not None, is_host=bool(is_host),
                       scalar_loop=bool(scalar_loop), bounds=bounds, chunk=chunk, ncol=ncol, lc=send_lc,
                       post=post)
            self._bcast(hdr)
            pin = self.device == "cuda"
            buf = torch.zeros((self.world, max(ncol, 1), chunk), dtype=torch.float64,
                              pin_memory=pin)
            view = buf.numpy()
            for j, k in enumerate(arrays):
                col = np.asarray(cols[k], dtype=np.float64)
                for r in range(self.world):
                    view[r, j, :bounds[r + 1] - bounds[r]] = col[bounds[r]:bounds[r + 1]]
            if extra_mask is not None:
                m = np.asarray(extra_mask)
                for r in range(self.world):
                    view[r, ncol - 1, :bounds[r + 1] - bounds[r]] = m[bounds[r]:bounds[r + 1]]
            dev = buf.to(self.device, non_blocking=True) if pin else buf
            mine = torch.empty((max(ncol, 1), chunk), dtype=torch.float64, device=self.device)
            self.d.scatter(mine, scatter_list=list(dev.unbind(0)), src=0)
            self.scatters += 1
            pending = self._evaluate(eng, hdr, mine, lc)
        return pending, bounds[0], seq

    def finish_root(self, error=False):
        """Rank 0, after its last engine call: release the followers."""
        with self.lock:
            self._bcast(dict(op="end", error=bool(error)))

    def follow(self, eng):
        """Ranks other than 0: evaluate the slices rank 0 sends until it says `end`, register the
        records; returns after the exchange with rank 0's result payload."""
        import torch
        held, lc = [], None
        while True:
            hdr = self._bcast()
            if hdr["op"] == "end":
                if hdr["error"]:
                    raise RuntimeError("calc_probs failed on rank 0")
                break
            if hdr["lc"] is not None:
                lc = hdr["lc"]
            mine = torch.empty((max(hdr["ncol"], 1), hdr["chunk"]), dtype=torch.float64,
                               device=self.device)
            self.d.scatter(mine, scatter_list=None, src=0)
            self.scatters += 1
            held.append((hdr, self._evaluate(eng, hdr, mine, lc)))
        for hdr, pending in held:
            res = pending.result()
            lo = hdr["bounds"][self.rank]
            for b, r in enumerate(res if isinstance(res, tuple) else (res,)):
                self.add(_host_record(r, lo, eng, hdr["post"]), ("s", hdr["seq"], b))
        self.exchange()
        return self._bcast()

    def publish(self, payload):
        """Rank 0 -> everybody: the finished result tables of the call."""
        with self.lock:
            return self._bcast(payload)


def open_group(scatter):
    """Start the CallGroup of a calc_probs call (None without a process group)."""
    global _group
    d = _dist()
    _group = CallGroup(d, scatter) if d is not None else None
    return _group


def close_group():
    global _group
    _group = None


# ---- the light curve of the scenario being prepared (per thread) --------------------------------
_tls = threading.local()
_fallback_lock = threading.Lock()


def use_lightcurve(time, flux, sigma, exptime, nsamples):
    """What every lnZ_* does first: name the light curve its draws will be evaluated against.
    It becomes the engine's current light curve together with the submission (scenario functions
    may run in different threads; the engine has one current light curve)."""
    _tls.lightcurve = (time, flux, sigma, exptime, nsamples)


def current_lightcurve():
    return getattr(_tls, "lightcurve", None)


def rng_done():
    """Called by an lnZ_* function after its last draw from numpy's global generator: the next
    scenario may start drawing while this one finishes its deterministic work."""
    ev = getattr(_tls, "rng_event", None)
    if ev is not None:
        ev.set()


# ---- submit / finish ----------------------------------------------------------------------------
class _Done:
    """Pending-like wrapper of an already computed result (engines without a submit API)."""

    def __init__(self, out):
        self._out = out

    def result(self):
        return self._out


def _submit(eng, name, *args, post=None, **kw):
    lc = current_lightcurve()
    _sync_moments(eng)
    kw.update(_post_kw(eng, post))
    fn = getattr(eng, "submit_" + name, None)
    if fn is not None:
        return fn(*args, lightcurve=lc, **kw)
    with _fallback_lock:     # engines without a submit API (test stand-ins): one call at a time
        if lc is not None:
            eng.set_lightcurve(*lc)
        return _Done(getattr(eng, "eval_" + name)(*args, **kw))


class PendingBranches:
    """A scenario evaluation in flight on this rank.  `prepare()` waits for the local result and
    packs this rank's records (inside a CallGroup, registered for its exchange); `finish()`
    returns the globally merged Branch (TP-type) or the (EB, EBx2P) pair -- right away with its
    own collective for a single lnZ_* call, after the group's one exchange inside calc_probs.
    Both are idempotent."""

    def __init__(self, pending, lo, N, eng, seq=None, post=None):
        self._pending, self._lo, self._N, self._eng = pending, lo, N, eng
        self._post = post
        self._seq, self._group = seq, _group
        self._res = self._out = None
        self._lock = threading.Lock()

    def prepare(self):
        with self._lock:
            if self._res is None:
                res = self._pending.result()
                self._res = res if isinstance(res, tuple) else (res,)
                self._tuple = isinstance(res, tuple)
                self._pending = None
                self._recs = [_host_record(r, self._lo, self._eng, self._post)
                              for r in self._res]
                g = self._group
                self._keys = [None if g is None else
                              g.add(rec, None if self._seq is None else ("s", self._seq, b))
                              for b, rec in enumerate(self._recs)]

    def finish(self):
        self.prepare()
        with self._lock:
            if self._out is None:
                out = [_host_branch(gather_slices(rec, self._group, key), r, self._N, self._eng,
                                    self._post, b)
                       for b, (rec, key, r) in enumerate(zip(self._recs, self._keys, self._res))]
                self._out = tuple(out) if self._tuple else out[0]
        return self._out


def _submit_sharded(kind, N, cols, extra_mask, companion_is_host, scalar_loop=False):
    eng = get_engine()
    g = _group
    post = _next_post()
    if g is not None and g.scatter:
        # calc_probs under a process group, numpy draws: this is rank 0 (the others follow)
        pending, lo, seq = g.scatter_submit(eng, kind, N, cols, extra_mask, companion_is_host,
                                            scalar_loop, post)
        return PendingBranches(pending, lo, N, eng, seq, post)
    lo, hi = shard_bounds(N)
    sl = {k: _slice(v, lo, hi) for k, v in cols.items()}
    lnprior = sl.pop("lnprior")
    kw = {"scalar_loop": True} if scalar_loop else {}
    p = _submit(eng, kind, hi - lo, *sl.values(), lnprior=lnprior,
                extra_mask=_mask_slice(extra_mask, lo, hi),
                companion_is_host=companion_is_host, want_lnL=False, n_best=N_BEST, post=post,
                **kw)
    return PendingBranches(p, lo, N, eng, post=post)


def submit_tp(N, rp, P_orb, inc, ecc, argp, mtot, rhost, u1, u2, cfr, lnprior=None,
              extra_mask=None, companion_is_host=False):
    cols = dict(rp=rp, P_orb=P_orb, inc=inc, ecc=ecc, argp=argp, mtot=mtot, rhost=rhost, u1=u1,
                u2=u2, cfr=cfr, lnprior=lnprior)
    return _submit_sharded("tp", N, cols, extra_mask, companion_is_host)


def submit_eb(N, reb, ebfr, q, P_orb, inc, ecc, argp, mtot, rhost, u1, u2, cfr, lnprior=None,
              extra_mask=None, companion_is_host=False, scalar_loop=False):
    cols = dict(reb=reb, ebfr=ebfr, q=q, P_orb=P_orb, inc=inc, ecc=ecc, argp=argp, mtot=mtot,
                rhost=rhost, u1=u1, u2=u2, cfr=cfr, lnprior=lnprior)
    return _submit_sharded("eb", N, cols, extra_mask, companion_is_host, scalar_loop)


def run_tp(*args, **kw):
    return submit_tp(*args, **kw).finish()


def run_eb(*args, **kw):
    return submit_eb(*args, **kw).finish()


# ---- deferred delivery: calc_probs overlaps one scenario's GPU work with the next one's draws ----
_deferring = False


class Deferred:
    """A scenario result whose evaluation may still be running; `resolve()` returns the
    reference's result dictionary (and caches it).  `prepare()` is its local half: wait for
    this rank's evaluation and register its records with the call's CallGroup, so that
    calc_probs can exchange all rows at once before resolving any of them."""

    def __init__(self, make, prepare=None):
        self._make, self._prepare, self._out = make, prepare, None

    def prepare(self):
        if self._prepare is not None:
            self._prepare()
            self._prepare = None

    def resolve(self):
        if self._make is not None:
            self.prepare()
            self._out = self._make()
            self._make = None
        return self._out


@contextlib.contextmanager
def deferring():
    """Inside this context the lnZ_* functions return `Deferred` results instead of waiting for
    the GPU (calc_probs resolves them a few scenarios later, in order).  Everywhere else they
    return finished dictionaries, like the reference."""
    global _deferring
    saved, _deferring = _deferring, True
    try:
        yield
    finally:
        _deferring = saved


class ScenarioChain:
    """Runs scenario functions in a few threads while keeping numpy's global generator strictly
    sequential: scenario k+1 starts when scenario k has made its last draw (`rng_done()`, or its
    return), so its draws follow in the reference's order while k's deterministic preparation
    (stellar relations, priors, flux ratios, submission) still runs."""

    def __init__(self, n_threads):
        from concurrent.futures import ThreadPoolExecutor
        self._pool = ThreadPoolExecutor(n_threads) if n_threads > 1 else None
        self._last = None

    def run(self, fn):
        """Start fn() after the previous scenario's draws; returns an object with .result()."""
        if self._pool is None:
            return _Done(fn())
        prev, mine = self._last, threading.Event()
        self._last = mine
        deferring_now = _deferring

        def task():
            if prev is not None:
                prev.wait()
            _tls.rng_event = mine
            try:
                return fn()
            finally:
                _tls.rng_event = None
                mine.set()
        assert deferring_now, "scenario threads are used inside deferring() only"
        return self._pool.submit(task)

    def close(self):
        if self._pool is not None:
            self._pool.shutdown(wait=True)


def deliver(make, prepare=None):
    return Deferred(make, prepare) if _deferring else make()


def resolve(res):
    return res.resolve() if isinstance(res, Deferred) else res


def prepare(res):
    if isinstance(res, Deferred):
        res.prepare()


def scenario_threads(scattering=False):
    """Threads calc_probs uses for the host-side preparation of consecutive scenarios
    (TRI_B200_SCENARIO_THREADS; 1 = everything in the calling thread, the default -- 2 when
    rank 0 also packs and scatters every scenario's columns to the other ranks of a process
    group, which is worth overlapping with the next scenario's draws: 0.28 s vs 0.39 s per call
    on 2 GPUs).

    While a scenario's preparation took 0.1-0.3 s of single-threaded numpy, running it beside the
    next scenario's draws paid (4 threads, rounds 1-2).  Now that both the generator helpers and
    the preparation blocks are short multi-threaded C calls, overlapping them only makes them
    compete for memory bandwidth and cores: on the 16-core GPU box the public call takes 0.209 s
    with 1 thread, 0.247 s with 2, 0.280 s with 4 (the GPU work overlaps either way: submissions
    are asynchronous)."""
    import os
    default = 2 if scattering else 1
    try:
        return max(1, int(os.environ.get("TRI_B200_SCENARIO_THREADS", str(default))))
    except ValueError:
        return default


def gil_switch_interval():
    """Interpreter switch interval [s] while calc_probs runs its scenario threads
    (TRI_B200_SWITCH_INTERVAL, default 0.2 ms; Python's own default is 5 ms)."""
    import os
    try:
        return max(1e-5, float(os.environ.get("TRI_B200_SWITCH_INTERVAL", "0.0002")))
    except ValueError:
        return 0.0002
