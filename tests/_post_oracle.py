"""Test helper: the moments oracle engine (tests/_mc_oracle.py) with the posterior samples of
tri_set_posterior, drawn by a numpy mirror of the GPU's systematic resampler from each
evaluation's own per-draw ln-weights.  The oracle itself is unchanged.  `posts` keeps (stream,
[post_idx per branch]) of every evaluation made with posterior samples on."""
import numpy as np

from _mc_oracle import MomentsOracleEngine, install  # noqa: F401
from triceratops_b200._numerics import posterior_uniform


def prefix_sums(lnw):
    """C = cumsum(exp(lnw - m)) over the finite ln-weights (0 elsewhere), accumulated in
    extended precision and rounded once: a reference for the GPU's prefix sums, whose serial
    chains are at most 16 + 32 + 8 + N / 4096 additions long, where a float64 cumsum over N
    draws drifts by up to N rounding errors."""
    fin = np.isfinite(lnw)
    m = lnw[fin].max()
    w = np.where(fin, np.exp(np.where(fin, lnw, m) - m), 0.0)
    return np.cumsum(w.astype(np.longdouble)).astype(np.float64)


def resample(lnw, K, U):
    """(indices, T) of K systematic samples of ln-weights lnw: sample k is min{i : C_i > (U +
    k) T / K} with C = prefix_sums(lnw); positions at or above T go to the last draw at which
    C increases.  Empty for a +inf weight or no finite weight (T = inf / 0)."""
    lnw = np.asarray(lnw, dtype=float)
    empty = np.zeros(0, dtype=np.int64)
    if np.isposinf(lnw).any():
        return empty, np.inf
    if not np.isfinite(lnw).any():
        return empty, 0.0
    C = prefix_sums(lnw)
    T = float(C[-1])
    u = (U + np.arange(K, dtype=np.float64)) * (T / K)
    idx = np.searchsorted(C, u, side="right")
    grew = np.flatnonzero(np.diff(np.concatenate([[0.0], C])) > 0)
    idx[idx >= C.size] = grew[-1]
    return idx.astype(np.int64), T


class PosteriorOracleEngine(MomentsOracleEngine):
    def __init__(self):
        super().__init__()
        self._post_K, self._post_seed = 0, 0
        self.posts = []

    def set_posterior(self, K, seed=0):
        self._post_K, self._post_seed = int(K), int(seed)

    def _post(self, results, stream):
        if self._post_K == 0:
            return
        for b, (res, lnw) in enumerate(zip(results, self.draws[-len(results):])):
            res.post_idx, res.post_total = resample(
                lnw, self._post_K, posterior_uniform(self._post_seed, stream, b))
        self.posts.append((stream, [r.post_idx for r in results]))

    def eval_tp(self, *args, post_stream=None, **kw):
        res = super().eval_tp(*args, **kw)
        res.post_idx = res.post_total = None
        self._post((res,), self._stream if post_stream is None else post_stream)
        return res

    def eval_eb(self, *args, post_stream=None, **kw):
        out = super().eval_eb(*args, **kw)
        for r in out:
            r.post_idx = r.post_total = None
        self._post(out, self._stream if post_stream is None else post_stream)
        return out

    # (the tensor entry points of the device sampler and of a process group)
    _stream = 0

    def eval_tp_tensors(self, *args, post_stream=0, **kw):
        self._stream = post_stream
        return super().eval_tp_tensors(*args, **kw)

    def eval_eb_tensors(self, *args, post_stream=0, **kw):
        self._stream = post_stream
        return super().eval_eb_tensors(*args, **kw)
