"""Posterior samples on the GPU (tri_set_posterior, posterior_sums_kernel and
posterior_select_kernel): the indices of every branch against a host mirror built from the
fetched per-draw lnL and lnprior, the engine with posterior samples off as before, indices per
ticket with submissions in flight, shards merged with merge_posteriors, the largest K, the
posterior mean against the importance-weighted mean, and calc_probs on both samplers."""
import numpy as np
import pytest

from conftest import draw_eb_columns, draw_tp_columns
from _post_oracle import prefix_sums, resample
from triceratops_b200 import _cabi
from triceratops_b200 import _numerics as nx

pytestmark = pytest.mark.gpu


def _prior(N, seed):
    rng = np.random.default_rng(seed)
    p = rng.normal(-4.0, 1.5, N)
    p[rng.random(N) < 0.1] = -np.inf
    return p


def _lnw(res, lnprior):
    return res.lnL if lnprior is None else res.lnL + np.broadcast_to(lnprior, res.lnL.shape)


def _check(res, lnw, K, seed, stream, b):
    """GPU indices against the host mirror: equal except where u_k lies within 1e-12 T of a
    host-computed boundary C_i; copy counts floor or ceil of K w_i / T.  T agrees with the
    extended-precision reference to 1e-12: the kernels' serial chains (16 + 32 + 8 + N / 4096
    additions, at most 2.8e-13 T of rounding at N = 1e7) stay well inside it."""
    U = nx.posterior_uniform(seed, stream, b)
    want, T_h = resample(lnw, K, U)
    if want.size == 0:
        assert res.post_idx.size == 0 and res.post_total == T_h
        return 0
    assert res.post_total == pytest.approx(T_h, rel=1e-12)
    got = res.post_idx
    assert got.dtype == np.int64 and got.size == K and np.all(np.diff(got) >= 0)
    fin = np.isfinite(lnw)
    w = np.where(fin, np.exp(np.where(fin, lnw, 0.0) - res.m), 0.0)
    C = prefix_sums(lnw)
    T = res.post_total
    bad = np.flatnonzero(got != want)
    if bad.size:
        u = (U + bad.astype(np.float64)) * (T / K)
        j = np.clip(np.searchsorted(C, u), 1, C.size - 1)
        near = np.minimum(np.abs(C[j] - u), np.abs(C[j - 1] - u))
        assert np.all(near <= 1e-12 * T), bad[:10]
    counts = np.bincount(got, minlength=lnw.size)
    exp = K * w / T
    assert np.all(counts >= np.floor(exp * (1 - 1e-9))) and np.all(counts <= np.ceil(exp + 1e-6))
    assert np.all(counts[w == 0] == 0)
    return bad.size


@pytest.fixture()
def post_on(gpu_engine, toi465_lc):
    t, f, s = toi465_lc
    gpu_engine.set_lightcurve(t, f, 10 * s, 0.00139, 20)
    gpu_engine.set_posterior(4096, seed=21)
    yield gpu_engine
    gpu_engine.set_posterior(0)


@pytest.mark.parametrize("prior", [None, "scalar", "per-draw"])
def test_indices_match_the_host_mirror_tp(post_on, prior):
    eng, N = post_on, 200_000
    lnprior = {None: None, "scalar": -3.0, "per-draw": _prior(N, 1)}[prior]
    res = eng.eval_tp(N, **draw_tp_columns(N, 11), lnprior=lnprior, want_lnL=True, n_best=100,
                      post_stream=5)
    assert res.n_finite > 0
    _check(res, _lnw(res, lnprior), 4096, 21, 5, 0)


@pytest.mark.parametrize("scalar_loop", [False, True])
@pytest.mark.parametrize("prior", [None, "per-draw"])
def test_indices_match_the_host_mirror_eb(post_on, scalar_loop, prior):
    eng, N = post_on, 200_000
    lnprior = None if prior is None else _prior(N, 2)
    out = eng.eval_eb(N, **draw_eb_columns(N, 12), lnprior=lnprior, want_lnL=True, n_best=100,
                      scalar_loop=scalar_loop, post_stream=9)
    for b, res in enumerate(out):
        _check(res, _lnw(res, lnprior), 4096, 21, 9, b)


def test_indices_on_the_device_pointer_path(post_on):
    import torch
    eng, N = post_on, 150_000
    dev = torch.device("cuda", eng.device)
    cols = draw_tp_columns(N, 13)
    lnprior = _prior(N, 3)
    host = eng.eval_tp(N, **cols, lnprior=lnprior, want_lnL=True, n_best=100, post_stream=2)
    tcols = {k: torch.as_tensor(v, dtype=torch.float64, device=dev) for k, v in cols.items()}
    tcols["lnprior"] = torch.as_tensor(lnprior, device=dev)
    res = eng.eval_tp_tensors(N, tcols, n_best=100, post_stream=2)
    _check(res, _lnw(host, lnprior), 4096, 21, 2, 0)
    ecols = draw_eb_columns(N, 14)
    hb = eng.eval_eb(N, **ecols, want_lnL=True, n_best=100, post_stream=3)
    tb = eng.eval_eb_tensors(N, {k: torch.as_tensor(v, dtype=torch.float64, device=dev)
                                 for k, v in ecols.items()}, n_best=100, post_stream=3)
    for b, (h, d) in enumerate(zip(hb, tb)):
        _check(d, _lnw(h, None), 4096, 21, 3, b)


def test_posterior_off_is_the_parent_path(gpu_engine, toi465_lc):
    eng, N = gpu_engine, 100_000
    t, f, s = toi465_lc
    eng.set_lightcurve(t, f, s, 0.00139, 20)
    cols = draw_eb_columns(N, 15)
    off = eng.eval_eb(N, **cols, n_best=100, want_lnL=False)
    assert eng.last_timing()["launches"] == 3
    assert all(r.post_idx is None for r in off)
    eng.set_posterior(1000, seed=1)
    try:
        on = eng.eval_eb(N, **cols, n_best=100, want_lnL=False)
        assert eng.last_timing()["launches"] == 5
        again = eng.eval_eb(N, **cols, n_best=100, want_lnL=False)
        eng.set_moments(True)
        both = eng.eval_eb(N, **cols, n_best=100, want_lnL=False)
        assert eng.last_timing()["launches"] == 6
        eng.set_posterior(0)
        eng.eval_eb(N, **cols, n_best=100, want_lnL=False)
        assert eng.last_timing()["launches"] == 4
    finally:
        eng.set_moments(False)
        eng.set_posterior(0)
    for a, b, c, d in zip(off, on, again, both):
        assert a.lnZ == b.lnZ and a.m == b.m and a.s == b.s
        np.testing.assert_array_equal(a.top_idx, b.top_idx)
        np.testing.assert_array_equal(a.top_lnL, b.top_lnL)
        # fixed tiles and summation order: the same bits run to run
        np.testing.assert_array_equal(b.post_idx, c.post_idx)
        np.testing.assert_array_equal(b.post_idx, d.post_idx)
        assert b.post_total == c.post_total == d.post_total


def test_each_ticket_keeps_its_own_indices(gpu_engine, toi465_lc):
    eng, N = gpu_engine, 80_000
    t, f, s = toi465_lc
    eng.set_lightcurve(t, f, 10 * s, 0.00139, 20)
    cols = [draw_tp_columns(N, 20 + k) for k in range(4)]
    Ks = [300, 0, 5000, 77]
    lnws, pend = [], []
    try:
        for c in cols:
            eng.set_posterior(0)
            lnws.append(eng.eval_tp(N, **c, want_lnL=True).lnL)
        for k, c in enumerate(cols):
            eng.set_posterior(Ks[k], seed=3)
            pend.append(eng.submit_tp(N, **c, want_lnL=False, n_best=100, post_stream=40 + k))
    finally:
        eng.set_posterior(0)
    for k in (3, 0, 2, 1):      # out of order
        r = pend[k].result()
        if Ks[k]:
            _check(r, lnws[k], Ks[k], 3, 40 + k, 0)
        else:
            assert r.post_idx is None


def test_bad_arguments_are_refused(gpu_engine, toi465_lc):
    import ctypes
    lib = gpu_engine.lib
    assert lib.tri_set_posterior(-1, 0, 0) == _cabi.TRI_EINVAL
    assert lib.tri_set_posterior(_cabi.TRI_MAX_POSTERIOR + 1, 0, 0) == _cabi.TRI_EINVAL
    t, f, s = toi465_lc
    gpu_engine.set_lightcurve(t, f, 10 * s, 0.00139, 20)
    gpu_engine.set_posterior(50)
    try:
        gpu_engine.eval_tp(20_000, **draw_tp_columns(20_000, 5), want_lnL=False)
    finally:
        gpu_engine.set_posterior(0)
    idx = (ctypes.c_int64 * 50)()
    n, T = ctypes.c_int64(), ctypes.c_double()
    assert lib.tri_last_posterior(1, idx, 50, ctypes.byref(n), ctypes.byref(T)) == \
        _cabi.TRI_EINVAL
    assert lib.tri_last_posterior(0, idx, 49, ctypes.byref(n), ctypes.byref(T)) == \
        _cabi.TRI_EINVAL
    assert lib.tri_last_posterior(0, idx, 50, ctypes.byref(n), ctypes.byref(T)) == 0
    assert n.value == 50


def test_merged_shards_hold_the_bounds(post_on):
    eng, N, K = post_on, 240_000, 4096
    cols = draw_tp_columns(N, 30)
    lnprior = _prior(N, 4)
    parts, lnw = [], []
    bounds = (0, 80_000, 200_000, N)
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        c = {k: v[lo:hi] if np.ndim(v) else v for k, v in cols.items()}
        r = eng.eval_tp(hi - lo, **c, lnprior=lnprior[lo:hi], want_lnL=True, post_stream=6)
        parts.append((r.m, r.post_total, r.post_idx + lo))
        lnw.append(_lnw(r, lnprior[lo:hi]))
    idx, m, W = nx.merge_posteriors(parts, K, 21, 6)
    assert idx.size == K and np.all(np.diff(idx) >= 0)
    Wr = np.array([T * np.exp(mm - m) for mm, T, _ in parts])
    c = np.histogram(idx, bins=bounds)[0]
    assert np.all(c >= np.floor(K * Wr / W)) and np.all(c <= np.ceil(K * Wr / W))
    lnw = np.concatenate(lnw)
    assert np.all(np.isfinite(lnw[idx]))


def test_largest_K_at_ten_million_draws(gpu_engine, toi465_lc):
    eng, N, K = gpu_engine, 10_000_000, _cabi.TRI_MAX_POSTERIOR
    t, f, s = toi465_lc
    eng.set_lightcurve(t, f, 10 * s, 0.00139, 20)
    eng.set_posterior(K, seed=8)
    try:
        res = eng.eval_tp(N, **draw_tp_columns(N, 31), want_lnL=True, post_stream=1)
    finally:
        eng.set_posterior(0)
    _check(res, res.lnL, K, 8, 1, 0)


def test_posterior_mean_matches_the_weighted_mean(post_on):
    """The mean of R_p over the K samples against the importance-weighted mean over all draws,
    within 5 standard errors of a sample of min(K, ess) independent draws."""
    eng, N, K = post_on, 400_000, 4096
    cols = draw_tp_columns(N, 32)
    res = eng.eval_tp(N, **cols, want_lnL=True, post_stream=11)
    w = np.where(np.isfinite(res.lnL), np.exp(res.lnL - res.m), 0.0)
    rp = np.broadcast_to(cols["rp"], (N,))
    mean = np.sum(w * rp) / w.sum()
    sd = np.sqrt(np.sum(w * (rp - mean) ** 2) / w.sum())
    ess = w.sum() ** 2 / np.sum(w * w)
    got = rp[res.post_idx].mean()
    assert abs(got - mean) <= 5 * sd / np.sqrt(min(K, ess)) + 1e-12


@pytest.mark.parametrize("sampler", ["host", "device"])
def test_calc_probs_posterior(gpu_engine, sampler):
    """Config-2 inputs at N = 1e5: lnZ unchanged (to the rounding of the light-curve kernel's
    block merge) with posterior samples on, the posterior table's shape, and -- host sampler,
    whose TP call is seen with its columns -- the posterior mean of R_p in the TP row against
    the importance-weighted mean from the per-draw lnL of that call, within 5 standard errors
    of min(K, ess) independent draws."""
    from _workloads import lightcurve, make_target, run_calc_probs
    from triceratops_b200 import set_sampler
    K = 1000
    lc = lightcurve(2)
    seen = {}
    submit_tp = gpu_engine.submit_tp

    def spy(N, rp, *args, post_stream=0, **kw):
        if post_stream == 0 and gpu_engine._post_K:     # (row 0: the TP call)
            kw["want_lnL"] = True
            p = submit_tp(N, rp, *args, post_stream=post_stream, **kw)
            seen.update(rp=np.broadcast_to(rp, (N,)).copy(), lnprior=kw.get("lnprior"), p=p)
            return p
        return submit_tp(N, rp, *args, post_stream=post_stream, **kw)
    try:
        set_sampler(sampler, seed=7)
        base = run_calc_probs(make_target(2), 2, lc, 100_000, 7)
        set_sampler(sampler, seed=7)      # (the device sampler's streams start again)
        gpu_engine.submit_tp = spy
        tgt = run_calc_probs(make_target(2), 2, lc, 100_000, 7, posterior_samples=K,
                             posterior_seed=3)
    finally:
        gpu_engine.__dict__.pop("submit_tp", None)
        set_sampler("host")
    assert base.posterior is None
    np.testing.assert_allclose(tgt.lnZ, base.lnZ, rtol=0, atol=1e-9)
    P = tgt.posterior
    rows = [j for j in range(len(tgt.lnZ)) if np.isfinite(tgt.lnZ[j])]
    assert sorted(set(P.row)) == rows
    for j, blk in P.groupby("row"):
        assert len(blk) == K and np.all(np.diff(blk.draw.values) >= 0)
        assert blk.draw.max() < 100_000
    tp = P[P.row == 0]
    assert (tp.scenario == "TP").all() and np.all(tp.R_p > 0)
    if sampler == "host":
        res = seen["p"].result()
        lnw = _lnw(res, seen["lnprior"])
        np.testing.assert_array_equal(tp.R_p.values, seen["rp"][tp.draw.values])
        fin = np.isfinite(lnw)
        w = np.where(fin, np.exp(np.where(fin, lnw, 0.0) - res.m), 0.0)
        mean = np.sum(w * seen["rp"]) / w.sum()
        sd = np.sqrt(np.sum(w * (seen["rp"] - mean) ** 2) / w.sum())
        ess = w.sum() ** 2 / np.sum(w * w)
        assert abs(tp.R_p.mean() - mean) <= 5 * sd / np.sqrt(min(K, ess)) + 1e-12
