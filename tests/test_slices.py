"""The record of a scenario branch over one slice of draws and the merge of such records
(_dispatch.pack_slice / merge_slices), in pure numpy: ln-weights with -inf entries and exact
ties, split into 1 to 4 contiguous slices, packed without rows (R = 0, host sampler) and with
rows (R = 3, rows a known function of the global draw index), merged, and checked against the
whole array."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from _post_oracle import resample  # noqa: E402
from triceratops_b200 import _dispatch  # noqa: E402
from triceratops_b200 import _numerics as nx  # noqa: E402

N, K, SEED, STREAM = 1501, 64, 9, 4


def _lnw():
    rng = np.random.default_rng(17)
    x = np.round(rng.normal(-3.0, 1.0, N) * 4) / 4      # (quarter steps: many exact ties)
    x[rng.random(N) < 0.4] = -np.inf
    return x


def _rows(gidx):
    g = np.asarray(gidx, dtype=np.float64)
    return np.stack([g, 0.5 * g + 1, np.sin(g)], axis=1)


def _slices(lnw, world):
    """Per slice (lo, record fields, local posterior (T, global indices)), packed with R = 0
    and with R = 3."""
    out = []
    for r in range(world):
        lo, hi = (r * N) // world, ((r + 1) * N) // world
        x = lnw[lo:hi]
        m, s, s2, n_fin, n_pinf = nx.lse_moments(x)
        fin = np.flatnonzero(np.isfinite(x))
        top = fin[np.lexsort((fin, -x[fin]))][:_dispatch.N_BEST]
        pidx, T = resample(x, K, nx.posterior_uniform(SEED, STREAM + r, 0))
        hdr = (m, s, n_fin, n_pinf, hi - lo, n_fin, s2, top + lo, x[top])
        recs = [_dispatch.pack_slice(*hdr, post=(K, T, pidx + lo)),
                _dispatch.pack_slice(*hdr, rows=_rows(top + lo),
                                     post=(K, T, pidx + lo, _rows(pidx + lo)))]
        out.append((lo, (m, T, pidx + lo), recs))
    return out


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_merged_slices_equal_the_whole_array(world):
    lnw = _lnw()
    sl = _slices(lnw, world)
    whole = nx._log_mean_exp(lnw, N_total=N)
    m, s, s2, n_fin, n_pinf = nx.lse_moments(lnw)
    fin = np.flatnonzero(np.isfinite(lnw))
    top = fin[np.lexsort((fin, -lnw[fin]))][:_dispatch.N_BEST]
    assert len(np.unique(lnw[top])) < len(top)              # ties inside the table
    want_idx, _, want_W = nx.merge_posteriors([p for _, p, _ in sl], K, SEED, STREAM, 1)
    merged = []
    for R in (0, 3):
        allrec = np.stack([recs[R > 0] for _, _, recs in sl])
        # (one slice: lnZ is the engine's number, handed in as it is)
        br = _dispatch.merge_slices(allrec, N, R, lnZ=whole if world == 1 else None,
                                    post=(K, SEED, STREAM), branch=1)
        assert br.N == N and br.n_pass == N and br.n_evaluated == n_fin
        assert br.lnZ == pytest.approx(whole, rel=0, abs=1e-12)
        assert br.record[0] == m and br.record[3:] == (n_fin, n_pinf)
        assert br.record[1] == pytest.approx(s, rel=1e-12)
        assert br.record[2] == pytest.approx(s2, rel=1e-12)
        assert np.array_equal(br.idx, top) and np.array_equal(br.vals, lnw[top])
        assert np.array_equal(br.post_idx, want_idx) and br.post_total == want_W
        assert np.all(np.isfinite(lnw[br.post_idx]))
        if R:
            assert np.array_equal(br.rows, _rows(br.idx))
            assert np.array_equal(br.post_rows, _rows(br.post_idx))
        else:
            assert br.rows is None and br.post_rows is None
        merged.append(br)
    assert np.array_equal(merged[0].idx, merged[1].idx)


def test_slices_without_finite_draws_or_posterior():
    lnw = np.full(300, -np.inf)
    lnw[250] = -1.0
    recs = []
    for lo, hi in ((0, 150), (150, 300)):
        x = lnw[lo:hi]
        m, s, s2, n_fin, n_pinf = nx.lse_moments(x)
        fin = np.flatnonzero(np.isfinite(x))
        recs.append(_dispatch.pack_slice(m, s, n_fin, n_pinf, hi - lo, n_fin, None, fin + lo,
                                         x[fin], rows=_rows(fin + lo)))
    br = _dispatch.merge_slices(np.stack(recs), 300, 3, post=(K, SEED, STREAM))
    assert br.lnZ == pytest.approx(-1.0 - np.log(300), abs=1e-12)
    assert br.record[2] is None                     # no moments: s2 stays None
    assert np.array_equal(br.idx, [250]) and np.array_equal(br.rows, _rows([250]))
    assert br.post_idx is None and br.post_total is None
