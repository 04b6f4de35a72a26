"""Adaptive importance sampling on the CPU: the proposal tables (_numerics.fit_proposal and the
numpy mirror of the sampler kernel's inverse CDF and ln q), the reflected KDE on hand-built
posteriors, the allocation of an EB-type call's two branches, the whole pilot -> fit -> final
schedule on a toy likelihood with a known evidence, and calc_probs(proposal=...) validation."""
import numpy as np
import pytest
from scipy.special import ndtr

from triceratops_b200 import _numerics as nx

B, ALPHA, D = nx.PROP_BINS, nx.PROP_ALPHA, nx.PROP_SLOTS


def _fitted(seed=0, K=4096):
    rng = np.random.default_rng(seed)
    c = np.full((K, D), np.nan)
    c[:, 2] = np.clip(rng.normal(0.3, 0.05, K), 0, 0.999)
    c[:, 3] = rng.beta(0.5, 20.0, K)          # piled up at 0: the reflection matters
    c[:, 5] = rng.random(K)
    return nx.fit_proposal(c, [2, 3, 5])


# ---- tables ------------------------------------------------------------------------------------
def test_identity_tables_are_exact():
    tab = nx.identity_tables()
    assert tab.shape == (D, 2 * B + 1)
    assert np.array_equal(tab[:, :B + 1], np.tile(np.arange(B + 1) / B, (D, 1)))
    assert np.all(tab[:, B + 1:] == 0.0)
    u = np.random.default_rng(1).random(100_000)
    u[:4] = [0.0, 1.0 - 2 ** -53, 0.5, 3.0 / B]        # edges and the largest uniform
    for mix in (False, True):
        v, b = nx.proposal_inverse(tab[0], u, mix)
        assert np.array_equal(v, u)
        assert np.array_equal(b, np.minimum((u * B).astype(int), B - 1))
    assert np.all(nx.proposal_lnq(tab, np.tile(u[:, None], (1, D)), range(D)) == 0.0)


def test_fitted_table_invariants():
    tab = _fitted()
    for d in range(D):
        C, lnh = tab[d, :B + 1], tab[d, B + 1:]
        h = np.exp(lnh)
        assert C[0] == 0.0 and C[-1] == 1.0
        assert np.all(np.diff(C) > 0)
        assert np.all(h > 0) and np.all(np.isfinite(lnh))
        assert abs(np.sum(h) / B - 1.0) <= 1e-15
        np.testing.assert_allclose(np.diff(C), h / B, rtol=1e-12, atol=2e-15)   # (ulp of C near 1)
    for d in (0, 1, 4):                       # slots not fitted stay the prior
        assert np.array_equal(tab[d], nx.identity_tables()[d])
    # ln q >= ln alpha for any s (h -> 0 at the extremes)
    v = np.random.default_rng(2).random((50_000, D))
    assert np.all(nx.proposal_lnq(tab, v, [2, 3, 5]) >= np.log(ALPHA) - 1e-15)
    s = np.array([-1e3, -50.0, -1.0, 0.0, 1.0, 30.0])
    assert np.all(np.log1p((1 - ALPHA) * np.expm1(s)) >= np.log(ALPHA) - 1e-15)


def test_inverse_cdf_mirror_round_trips():
    tab = _fitted(3)
    u = np.random.default_rng(4).random(200_000)
    for d in (2, 3, 5):
        C, h = tab[d, :B + 1], np.exp(tab[d, B + 1:])
        v, b = nx.proposal_inverse(tab[d], u, True)
        assert np.all((v >= 0) & (v < 1))
        assert np.all(v >= b / B - 1e-15) and np.all(v <= (b + 1) / B + 1e-15)
        # H(v) = C_b + h_b (v - b / B) returns u
        np.testing.assert_allclose(C[b] + h[b] * (v - b / B), u, rtol=0, atol=1e-15)
        # and the bin found is floor(v B) except on an edge that rounding reached
        fl = np.minimum((v * B).astype(int), B - 1)
        assert np.mean(fl != b) < 1e-4
    # the prior branch keeps u and takes ln h at floor(u B)
    v, b = nx.proposal_inverse(tab[3], u, False)
    assert np.array_equal(v, u) and np.array_equal(b, np.minimum((u * B).astype(int), B - 1))


def test_mirror_samples_the_mixture_marginal():
    from scipy.stats import kstest
    tab = _fitted(5)
    rng = np.random.default_rng(6)
    n = 100_000
    mix = ~(rng.random(n) < ALPHA)
    v, _ = nx.proposal_inverse(tab[2], rng.random(n), mix)
    C = tab[2, :B + 1]
    h = np.exp(tab[2, B + 1:])

    def cdf(x):
        b = np.minimum((np.asarray(x) * B).astype(int), B - 1)
        return ALPHA * x + (1 - ALPHA) * (C[b] + h[b] * (x - b / B))
    assert kstest(v, cdf).pvalue > 1e-3


# ---- KDE ---------------------------------------------------------------------------------------
def _reflected_kde_exact(x, w, bw):
    e = np.arange(B + 1) / B
    m = sum(np.diff(ndtr((e[:, None] - c[None, :]) / bw) @ w) for c in (x, -x, 2 - x))
    return m * B / m.sum()


def test_kde_weights_distinct_draws_by_multiplicity():
    x = np.array([0.2, 0.2, 0.2, 0.6])        # a resample: 0.2 three times
    c = np.full((4, D), np.nan)
    c[:, 2] = x
    tab = nx.fit_proposal(c, [2])
    xs, w = np.array([0.2, 0.6]), np.array([0.75, 0.25])
    mu = np.sum(w * xs)
    bw = max(np.sqrt(np.sum(w * (xs - mu) ** 2)) * 2 ** -0.2, 8 / B)   # n = 2 distinct draws
    h = np.exp(tab[2, B + 1:])
    np.testing.assert_allclose(h, _reflected_kde_exact(xs, w, bw), rtol=0, atol=2e-2 * h.max())
    # the multiplicity counts: the unweighted KDE of the two draws is a different density
    flat = _reflected_kde_exact(xs, np.array([0.5, 0.5]),
                                max(np.std(xs) * 2 ** -0.2, 8 / B))
    assert np.abs(h - flat).max() > 0.2 * h.max()
    assert h[int(0.2 * B)] > 2 * h[int(0.6 * B)]


def test_kde_single_distinct_draw_uses_the_floor_bandwidth():
    c = np.full((4096, D), np.nan)
    c[:, 3] = 0.001                           # one draw, next to the reflecting edge
    tab = nx.fit_proposal(c, [3])
    h = np.exp(tab[3, B + 1:])
    want = _reflected_kde_exact(np.array([0.001]), np.array([1.0]), 8 / B)
    np.testing.assert_allclose(h, want, rtol=0, atol=2e-2 * h.max())
    assert np.argmax(h) == 0 and h.min() > 0
    # reflection: no mass lost below 0, the density at 0 is about twice a free Gaussian's peak
    assert h[0] > 1.5 * (B / (8 * np.sqrt(2 * np.pi))) * 0.9


@pytest.mark.parametrize("coords", ["none", "empty", "inf-total", "nan"])
def test_empty_posteriors_give_identity_tables(coords):
    ident = nx.identity_tables()
    if coords == "none":
        got = nx.fit_proposal(np.zeros((0, D)), [2, 3])
    elif coords == "nan":
        got = nx.fit_proposal(np.full((10, D), np.nan), [2, 3])
    elif coords == "empty":
        rows = nx.pooled_posterior([(-np.inf, 0.0, np.zeros((0, D)))], 4096, 0, 0)
        got = nx.fit_proposal(rows, [2, 3])
    else:
        rows = nx.pooled_posterior([(0.0, np.inf, np.full((4, D), 0.5)),
                                    (0.0, 1.0, np.full((4, D), 0.4))], 4, 0, 0)
        assert rows.shape == (0, D)
        got = nx.fit_proposal(rows, [2, 3])
    assert np.array_equal(got, ident)


def test_eb_branches_pooled_by_evidence():
    """Two branches of weights W_a, W_b: the pooled K rows hold floor or ceil of K W_a / W of
    branch a's rows (in their order, thinned systematically), the rest of b's."""
    K = 1000
    a = np.full((K, D), 0.25)
    b = np.full((K, D), 0.75)
    a[:, 0] = np.arange(K)
    b[:, 0] = np.arange(K) + K
    for (ma, Ta, mb, Tb) in [(0.0, 3.0, 0.0, 1.0), (-2.0, 5.0, 0.5, 0.2), (1.0, 1.0, 1.0, 0.0)]:
        rows = nx.pooled_posterior([(ma, Ta, a), (mb, Tb, b)], K, 7, 3)
        Wa, Wb = Ta * np.exp(ma - max(ma, mb)), Tb * np.exp(mb - max(ma, mb))
        na = int((rows[:, 2] == 0.25).sum())
        assert rows.shape == (K, D)
        assert np.floor(K * Wa / (Wa + Wb)) <= na <= np.ceil(K * Wa / (Wa + Wb))
        assert np.all(np.diff(rows[:na, 0]) >= 0) and np.all(rows[na:, 0] >= K)
    # one branch empty: the other alone; a single TP-type branch is returned as is
    rows = nx.pooled_posterior([(-np.inf, 0.0, np.zeros((0, D))), (0.0, 2.0, b)], K, 0, 0)
    assert np.array_equal(rows, b)
    assert np.array_equal(nx.pooled_posterior([(0.0, 2.0, a)], K, 0, 0), a)
    # the allocation over many streams is unbiased
    share = np.mean([(nx.pooled_posterior([(0.0, 1.0, a), (0.0, 2.0, b)], 7, 1, s)[:, 2] == 0.25)
                     .mean() for s in range(3000)])
    assert share == pytest.approx(1 / 3, abs=0.01)


# ---- the schedule on a toy likelihood ------------------------------------------------------------
MU = np.array([0.3, 0.55, 0.7, 0.45])
SIG = 0.06
SLOTS = [1, 2, 3, 5]


def _lnL(v):
    return -0.5 * np.sum(((v[:, SLOTS] - MU) / SIG) ** 2, axis=1)


Z_TRUE = float(np.prod(SIG * np.sqrt(2 * np.pi) * (ndtr((1 - MU) / SIG) - ndtr(-MU / SIG))))


def _draw(rng, n, tabs):
    """n draws of the kernel's mixture in numpy: (v [n, D], ln weight)."""
    u = rng.random((n, D))
    if tabs is None:
        return u, _lnL(u)
    mix = ~(rng.random(n) < ALPHA)
    v = np.full((n, D), np.nan)
    bins = np.zeros((n, D), dtype=np.int64)
    for d in SLOTS:
        v[:, d], bins[:, d] = nx.proposal_inverse(tabs[d], u[:, d], mix)
    return v, _lnL(v) - nx.proposal_lnq(tabs, v, SLOTS, bins=bins)


def _systematic(lnw, K, rng):
    w = np.exp(lnw - lnw.max())
    C = np.cumsum(w)
    return np.minimum(np.searchsorted(C, (rng.random() + np.arange(K)) * C[-1] / K, "right"),
                      lnw.size - 1)


def _adaptive(seed, N, N_pilot, stages=2, K=4096):
    rng = np.random.default_rng(seed)
    tabs = None
    for _ in range(stages):
        v, lnw = _draw(rng, N_pilot, tabs)
        tabs = nx.fit_proposal(v[_systematic(lnw, K, rng)], SLOTS)
    _, lnw = _draw(rng, N, tabs)
    return np.exp(lnw).mean()


def test_schedule_is_unbiased_and_beats_prior_sampling():
    N, N_pilot = 80_000, 10_000
    # the prior pilot sees tens of hits
    _, lnw = _draw(np.random.default_rng(0), N_pilot, None)
    w = np.exp(lnw)
    assert 10 <= w.sum() ** 2 / np.sum(w * w) <= 100
    za = np.array([_adaptive(s, N, N_pilot) for s in range(200)])
    zp = np.array([np.exp(_draw(np.random.default_rng(10_000 + s), N + 2 * N_pilot, None)[1])
                   .mean() for s in range(200)])
    for z in (za, zp):
        assert abs(z.mean() - Z_TRUE) <= 4 * z.std(ddof=1) / np.sqrt(z.size)
    assert za.std(ddof=1) * 10 <= zp.std(ddof=1)


def test_a_misplaced_proposal_costs_at_most_one_over_alpha():
    """Tables fitted where the likelihood is not: E_q[w^2] <= E_p[L^2] / alpha, and the
    estimate stays unbiased."""
    rng = np.random.default_rng(11)
    far = np.full((4096, D), np.nan)
    far[:, SLOTS] = np.clip(rng.normal(0.95, 0.02, (4096, len(SLOTS))), 0, 0.999)
    tabs = nx.fit_proposal(far, SLOTS)
    EL2 = float(np.prod(SIG * np.sqrt(np.pi) * (ndtr(np.sqrt(2) * (1 - MU) / SIG)
                                                 - ndtr(-np.sqrt(2) * MU / SIG))))
    w2, zs = [], []
    for s in range(200):
        _, lnw = _draw(np.random.default_rng(s), 20_000, tabs)
        w = np.exp(lnw)
        w2.append(np.mean(w * w))
        zs.append(w.mean())
    w2, zs = np.array(w2), np.array(zs)
    assert w2.mean() <= EL2 / ALPHA * (1 + 4 * w2.std(ddof=1) / np.sqrt(w2.size) / w2.mean())
    # the variance of the estimate within the bound (up to the scatter of 200 replicas)
    assert zs.var(ddof=1) <= (EL2 / ALPHA - Z_TRUE ** 2) / 20_000 * 1.5
    assert abs(zs.mean() - Z_TRUE) <= 4 * zs.std(ddof=1) / np.sqrt(zs.size)


# ---- calc_probs validation ------------------------------------------------------------------------
@pytest.fixture()
def recorder():
    from _workloads import Recorder, patched_engine
    rec = Recorder()
    with patched_engine(rec):
        yield rec


def _calc(toi465_lc, **kw):
    from _workloads import make_target, run_calc_probs
    return run_calc_probs(make_target(2), 2, toi465_lc, 20_000, 1, **kw)


def test_calc_probs_rejects_an_unknown_proposal(recorder, toi465_lc):
    with pytest.raises(ValueError, match="'prior' or 'adaptive'"):
        _calc(toi465_lc, proposal="adaptve")
    assert recorder.calls == []


def test_calc_probs_adaptive_rejects_the_host_sampler(recorder, toi465_lc):
    from triceratops_b200 import set_sampler
    set_sampler("host")
    with pytest.raises(ValueError, match="device sampler only"):
        _calc(toi465_lc, proposal="adaptive")
    assert recorder.calls == []


def test_calc_probs_adaptive_rejects_refinement(recorder, toi465_lc):
    from triceratops_b200 import set_sampler
    set_sampler("device", seed=1)
    try:
        with pytest.raises(ValueError, match="fpp_err_target"):
            _calc(toi465_lc, proposal="adaptive", fpp_err_target=0.01)
    finally:
        set_sampler("host")
    assert recorder.calls == []


def test_calc_probs_adaptive_rejects_sharded_draws(recorder, toi465_lc, monkeypatch):
    from triceratops_b200 import _dispatch, set_sampler
    monkeypatch.setattr(_dispatch, "_dist", lambda: object())
    set_sampler("device", seed=1)
    try:
        with pytest.raises(ValueError, match="process group"):
            _calc(toi465_lc, proposal="adaptive")
    finally:
        set_sampler("host")
    assert recorder.calls == []


def test_host_sampler_rejects_a_proposal(toi465_lc):
    from triceratops_b200 import device_sampler, importance_proposal, set_sampler
    from triceratops_b200.marginal_likelihoods import lnZ_TTP
    set_sampler("host")
    t, f, s = toi465_lc
    with importance_proposal(device_sampler.Proposal.identity()):
        with pytest.raises(ValueError, match="device sampler only"):
            lnZ_TTP(t, f, s, 3.8, 0.8, 0.8, 5000.0, 0.0, N=10)
    with pytest.raises(ValueError):
        device_sampler.Proposal(np.zeros((D, 2 * 1000 + 1)))     # B not a power of two
