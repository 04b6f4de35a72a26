"""Adaptive importance sampling on the GPU (tri_sampler_args.prop, device_sampler.Proposal,
calc_probs(proposal="adaptive")): identity tables reproduce the prior columns bit for bit, a
fitted proposal's columns follow the numpy mirror of the kernel, the recorded coordinates follow
the mixture's marginals, and on config-2 inputs with inflated flux errors the adaptive evidences,
FPP and posterior means agree with prior sampling within Monte-Carlo error."""
import numpy as np
import pytest
import torch

import _workloads as wl
from triceratops_b200 import _numerics as nx
from triceratops_b200 import device_sampler as ds
from triceratops_b200 import (importance_proposal, posterior_samples, record_coords,
                              set_sampler)

pytestmark = pytest.mark.gpu

B, ALPHA = nx.PROP_BINS, nx.PROP_ALPHA
S = wl.TOI465
CC = wl.os.path.join(wl.GOLD, "TOI465_01_contrastcurve.csv")
TRI = wl.os.path.join(wl.GOLD, "trilegal_synth.csv")


def _scenario(name, lc, N, P=None):
    from triceratops_b200 import marginal_likelihoods as ml
    t, f, s = lc
    P = S["P"] if P is None else P
    mags = (S["T"], S["J"], S["H"], S["K"])
    tail = dict(N=N, parallel=True)
    if name in ("TTP", "TEB"):
        return getattr(ml, "lnZ_" + name)(t, f, s, P, S["M"], S["R"], S["Teff"], 0.0, **tail)
    if name in ("PTP", "SEB"):
        return getattr(ml, "lnZ_" + name)(t, f, s, P, S["M"], S["R"], S["Teff"], 0.0, S["plx"],
                                          CC, "K", **tail)
    if name == "DTP":
        return ml.lnZ_DTP(t, f, s, P, S["M"], S["R"], S["Teff"], 0.0, *mags, TRI, CC, "K", **tail)
    return ml.lnZ_BEB(t, f, s, P, S["M"], S["R"], S["Teff"], *mags, TRI, CC, "K", **tail)


def _columns(name, lc, N, seed, P=None, prop=None, post=None):
    """(result(s), columns of the sampler kernel as numpy) of one scenario call."""
    seen = []
    orig = ds._run

    def spy(sampled, *a, **k):
        seen.append({k_: v.cpu().numpy() for k_, v in sampled[3].items() if torch.is_tensor(v)})
        return orig(sampled, *a, **k)
    set_sampler("device", seed=seed)
    ds._run = spy
    try:
        with importance_proposal(prop):
            if post:
                with posterior_samples(post, seed=3), record_coords():
                    res = _scenario(name, lc, N, P)
            else:
                res = _scenario(name, lc, N, P)
    finally:
        ds._run = orig
        set_sampler("host")
    return res, seen[0]


@pytest.fixture(scope="module")
def lc10(toi465_lc):
    t, f, s = toi465_lc
    return t, f, 10 * s


@pytest.mark.parametrize("name,P", [("TTP", None), ("TTP", (3.7, 3.9)), ("TEB", None),
                                    ("PTP", None), ("SEB", None), ("DTP", None), ("BEB", None)])
def test_identity_tables_reproduce_the_prior(gpu_engine, lc10, name, P):
    N = 200_000
    base, cb = _columns(name, lc10, N, 5, P)
    got, cg = _columns(name, lc10, N, 5, P, prop=ds.Proposal.identity())
    for k, v in cb.items():
        assert np.array_equal(v, cg[k], equal_nan=True), k
    lnp = cg["lnprior"]                 # written with a proposal; delta exactly 0
    assert np.array_equal(lnp, cb["lnprior"] if "lnprior" in cb else np.zeros(N),
                          equal_nan=True)
    for a, b in zip(base if isinstance(base, tuple) else (base,),
                    got if isinstance(got, tuple) else (got,)):
        # (the light-curve kernel's block merge may round the last bits differently per run)
        assert a["lnZ"] == pytest.approx(b["lnZ"], rel=1e-13, abs=1e-13)
        assert a.n_pass == b.n_pass


def _fit(name, lc, seed, P=None):
    res, _ = _columns(name, lc, 100_000, seed, P, post=4096)
    parts = res if isinstance(res, tuple) else (res,)
    rows = nx.pooled_posterior([(r.record[0], r.post_total, r.post_coords) for r in parts],
                               4096, 3, 0)
    slots = [d for d in range(6) if rows.shape[0] and np.all(np.isfinite(rows[:, d]))]
    assert rows.shape[0] > 0 and len(slots) >= 3
    return ds.Proposal(nx.fit_proposal(rows, slots)), slots


def _off_edges(v):
    x = v * B
    return np.abs(x - np.rint(x)) > 1e-9


@pytest.mark.parametrize("name,P", [("TTP", (3.7, 3.9)), ("TEB", None)])
def test_fitted_proposal_follows_the_mirror(gpu_engine, lc10, name, P):
    from scipy.stats import kstest
    prop, slots = _fit(name, lc10, 8, P)
    assert 0 in slots or P is None
    N = 200_000
    res, c = _columns(name, lc10, N, 9, P, prop=prop, post=64)
    v = c["_coords"][:, :N].T                 # [N, 6]
    assert np.all(np.isfinite(v[:, slots])) and np.all(np.isnan(np.delete(v, slots, axis=1)))
    # lnprior: no prior in these scenarios, so it is -ln q(v) alone
    ok = np.all(_off_edges(v[:, slots]), axis=1)
    assert ok.mean() > 0.999
    want = -nx.proposal_lnq(prop.tables, v[ok], slots)
    # (to 1e-15 of |ln q|, which reaches ~10: libdevice's and numpy's log1p / expm1, and the
    # order of the sum s, may differ in the last bit)
    np.testing.assert_allclose(c["lnprior"][ok], want, rtol=1e-15, atol=1e-15)
    assert np.all(c["lnprior"] <= -np.log(ALPHA) + 1e-15)
    # the parameter columns are the prior transforms of v
    np.testing.assert_allclose(c["argp"], 360.0 * v[:, 5], rtol=1e-14, atol=0)
    np.testing.assert_allclose(c["inc"], np.degrees(np.arccos(1.0 - v[:, 3])), rtol=1e-14,
                               atol=1e-14)
    if P is not None:
        np.testing.assert_allclose(c["P"], P[0] + (P[1] - P[0]) * v[:, 0], rtol=1e-14, atol=0)
    if name == "TEB":
        np.testing.assert_allclose(c["ecc"], v[:, 4] ** (1.0 / 0.2), rtol=1e-14, atol=1e-300)
    # each slot follows its marginal under the mixture, alpha v + (1 - alpha) H(v)
    for d in slots:
        C, h = prop.tables[d, :B + 1], np.exp(prop.tables[d, B + 1:])

        def cdf(x):
            b = np.minimum((np.asarray(x) * B).astype(np.int64), B - 1)
            return ALPHA * x + (1 - ALPHA) * (C[b] + h[b] * (x - b / B))
        assert kstest(v[:50_000, d], cdf).pvalue > 1e-4, d
    # unbiased: lnZ within the errors of a prior run of the same size
    for r in (res if isinstance(res, tuple) else (res,)):
        assert np.isfinite(r["lnZ"])


def _run(mode, N, seed, lc, **kw):
    set_sampler("device", seed=seed)
    try:
        return wl.run_calc_probs(wl.make_target(2), 2, lc, N, 1, mc_errors=True,
                                 proposal=mode, **kw)
    finally:
        set_sampler("host")


@pytest.fixture(scope="module")
def lc30(toi465_lc):
    t, f, s = toi465_lc
    return t, f, 30 * s


@pytest.fixture(scope="module")
def arms(gpu_engine, lc30):
    K = 4096
    return (_run("prior", 1_000_000, 21, lc30, posterior_samples=K, posterior_seed=2),
            _run("adaptive", 1_000_000, 22, lc30, posterior_samples=K, posterior_seed=2))


def test_adaptive_agrees_with_prior_sampling(arms):
    p, a = arms
    assert p.N_pilot is None and a.N_pilot == 125_000
    fin = np.isfinite(p.lnZ) & np.isfinite(a.lnZ)
    assert np.array_equal(fin, np.isfinite(p.lnZ))
    err = np.sqrt(a.lnZ_err[fin] ** 2 + p.lnZ_err[fin] ** 2)
    assert np.all(np.abs(a.lnZ[fin] - p.lnZ[fin]) <= 4 * err), (a.lnZ - p.lnZ, err)
    assert abs(a.FPP - p.FPP) <= 4 * np.hypot(a.FPP_err, p.FPP_err)
    assert np.all(a.N_draws[fin] == 1_000_000)
    ratio = a.ess[fin] / p.ess[fin]
    assert np.median(ratio) > 1, ratio


def test_adaptive_posterior_means_agree(arms):
    p, a = arms
    for j in np.flatnonzero(np.isfinite(p.lnZ) & (p.ess > 50)):
        bp, ba = p.posterior[p.posterior.row == j], a.posterior[a.posterior.row == j]
        assert len(bp) == len(ba) == 4096
        for col in ("inc", "w"):
            sd = max(bp[col].std(), ba[col].std(), 1e-12)
            n_p, n_a = min(4096, p.ess[j]), min(4096, a.ess[j])
            tol = 5 * sd * np.sqrt(1 / n_p + 1 / n_a)
            assert abs(bp[col].mean() - ba[col].mean()) <= tol, (j, col)


def test_adaptive_is_deterministic_and_composes(gpu_engine, lc30):
    a = _run("adaptive", 200_000, 5, lc30, posterior_samples=500, posterior_seed=1)
    b = _run("adaptive", 200_000, 5, lc30, posterior_samples=500, posterior_seed=1)
    np.testing.assert_allclose(a.lnZ, b.lnZ, rtol=1e-12, atol=0)
    cols = [c for c in a.probs.columns if c not in ("prob", "prob_err")]
    assert a.probs[cols].equals(b.probs[cols])          # the final round's best draws
    assert a.posterior.equals(b.posterior)              # and its posterior samples
    # composition: the final round's errors and posterior, N_pilot = max(N // 8, 10 000)
    assert a.N_pilot == 25_000 and np.all(a.N_draws[np.isfinite(a.lnZ)] == 200_000)
    fin = np.isfinite(a.lnZ)
    assert np.all(np.isfinite(a.lnZ_err[fin])) and np.all(a.ess[fin] > 0)
    assert np.isfinite(a.FPP_err)
    assert sorted(set(a.posterior.row)) == list(np.flatnonzero(fin))
    assert a.posterior.draw.max() < 200_000
    # without posterior samples: the same evidences, no posterior table
    c = _run("adaptive", 200_000, 5, lc30, posterior_seed=1)     # (the pilots resample with it)
    assert c.posterior is None
    np.testing.assert_allclose(c.lnZ, a.lnZ, rtol=1e-12, atol=0)
