"""The moment pass on the GPU (tri_set_moments, moments_kernel): s2 of every branch against a
host recomputation from the per-draw lnL, the engine with moments off as before, s2 per ticket
with submissions in flight, shards, the calibration of lnZ_err, and calc_probs refinement."""
import os

import numpy as np
import pytest

from conftest import TOI465, draw_eb_columns, draw_tp_columns
from triceratops_b200.engine import combine_moments

pytestmark = pytest.mark.gpu


def _host_s2(res, lnprior):
    lnw = res.lnL if lnprior is None else res.lnL + np.broadcast_to(lnprior, res.lnL.shape)
    fin = np.isfinite(lnw)
    return float(np.sum(np.exp(2.0 * (lnw[fin] - res.m))))


def _prior(N, seed):
    """A per-draw prior like the contrast-curve scenarios' (some draws excluded)."""
    rng = np.random.default_rng(seed)
    p = rng.normal(-4.0, 1.5, N)
    p[rng.random(N) < 0.1] = -np.inf
    return p


@pytest.fixture()
def moments_on(gpu_engine, toi465_lc):
    t, f, s = toi465_lc
    gpu_engine.set_lightcurve(t, f, s, 0.00139, 20)
    gpu_engine.set_moments(True)
    yield gpu_engine
    gpu_engine.set_moments(False)


@pytest.mark.parametrize("prior", [None, "scalar", "per-draw"])
def test_s2_matches_the_host_recomputation_tp(moments_on, prior):
    eng, N = moments_on, 200_000
    lnprior = {None: None, "scalar": -3.0, "per-draw": _prior(N, 1)}[prior]
    res = eng.eval_tp(N, **draw_tp_columns(N, 11), lnprior=lnprior, want_lnL=True, n_best=100)
    assert res.n_finite > 0
    assert res.s2 == pytest.approx(_host_s2(res, lnprior), rel=1e-12)
    assert 1.0 <= res.s2 <= res.s


@pytest.mark.parametrize("scalar_loop", [False, True])
@pytest.mark.parametrize("prior", [None, "per-draw"])
def test_s2_matches_the_host_recomputation_eb(moments_on, scalar_loop, prior):
    eng, N = moments_on, 200_000
    lnprior = None if prior is None else _prior(N, 2)
    out = eng.eval_eb(N, **draw_eb_columns(N, 12), lnprior=lnprior, want_lnL=True, n_best=100,
                      scalar_loop=scalar_loop)
    for res in out:
        if res.n_finite:
            assert res.s2 == pytest.approx(_host_s2(res, lnprior), rel=1e-12)
        else:
            assert res.s2 == 0.0


def test_s2_on_the_device_pointer_path(moments_on):
    import torch
    eng, N = moments_on, 150_000
    dev = torch.device("cuda", eng.device)
    cols = draw_tp_columns(N, 13)
    lnprior = _prior(N, 3)
    host = eng.eval_tp(N, **cols, lnprior=lnprior, want_lnL=True, n_best=100)
    tcols = {k: torch.as_tensor(v, dtype=torch.float64, device=dev) for k, v in cols.items()}
    tcols["lnprior"] = torch.as_tensor(lnprior, device=dev)
    res = eng.eval_tp_tensors(N, tcols, n_best=100)
    assert res.lnZ == host.lnZ
    assert res.s2 == pytest.approx(_host_s2(host, lnprior), rel=1e-12)
    ecols = draw_eb_columns(N, 14)
    hb = eng.eval_eb(N, **ecols, want_lnL=True, n_best=100)
    tb = eng.eval_eb_tensors(N, {k: torch.as_tensor(v, dtype=torch.float64, device=dev)
                                 for k, v in ecols.items()}, n_best=100)
    for h, d in zip(hb, tb):
        assert d.s2 == pytest.approx(_host_s2(h, None), rel=1e-12)


def test_moments_off_is_the_parent_path(gpu_engine, toi465_lc):
    eng, N = gpu_engine, 100_000
    t, f, s = toi465_lc
    eng.set_lightcurve(t, f, s, 0.00139, 20)
    cols = draw_eb_columns(N, 15)
    off = eng.eval_eb(N, **cols, n_best=100, want_lnL=False)
    assert eng.last_timing()["launches"] == 3
    assert all(r.s2 is None for r in off)
    eng.set_moments(True)
    try:
        on = eng.eval_eb(N, **cols, n_best=100, want_lnL=False)
        assert eng.last_timing()["launches"] == 4
        again = eng.eval_eb(N, **cols, n_best=100, want_lnL=False)
    finally:
        eng.set_moments(False)
    for a, b, c in zip(off, on, again):
        assert a.lnZ == b.lnZ and a.m == b.m and a.s == b.s
        np.testing.assert_array_equal(a.top_idx, b.top_idx)
        np.testing.assert_array_equal(a.top_lnL, b.top_lnL)
        assert b.s2 == c.s2        # fixed reduction order: the same bits run to run


def test_each_ticket_keeps_its_own_s2(gpu_engine, toi465_lc):
    eng, N = gpu_engine, 80_000
    t, f, s = toi465_lc
    eng.set_lightcurve(t, f, s, 0.00139, 20)
    cols = [draw_tp_columns(N, 20 + k) for k in range(4)]
    want = []
    eng.set_moments(True)
    try:
        for c in cols:
            r = eng.eval_tp(N, **c, want_lnL=True)
            want.append(_host_s2(r, None))
        pend = []
        for k, c in enumerate(cols):
            eng.set_moments(k % 2 == 0)
            pend.append(eng.submit_tp(N, **c, want_lnL=False, n_best=100))
    finally:
        eng.set_moments(False)
    for k in (3, 0, 2, 1):      # out of order
        r = pend[k].result()
        if k % 2 == 0:
            assert r.s2 == pytest.approx(want[k], rel=1e-12)
        else:
            assert r.s2 is None


def test_shard_combined_s2_equals_the_whole(moments_on):
    eng, N = moments_on, 240_000
    cols = draw_tp_columns(N, 30)
    lnprior = _prior(N, 4)
    whole = eng.eval_tp(N, **cols, lnprior=lnprior, want_lnL=False)
    parts = []
    for lo, hi in ((0, 80_000), (80_000, 200_000), (200_000, N)):
        c = {k: v[lo:hi] if np.ndim(v) else v for k, v in cols.items()}
        r = eng.eval_tp(hi - lo, **c, lnprior=lnprior[lo:hi], want_lnL=False)
        parts.append((r.m, r.s, r.s2, r.n_finite, r.n_posinf))
    m, s, s2, nf, npi = combine_moments(parts)
    assert m == whole.m and nf == whole.n_finite
    assert s2 == pytest.approx(whole.s2, rel=1e-12)


def test_lnZ_err_is_calibrated(gpu_engine, toi465_lc):
    """64 seeds at N = 1e5: the spread of lnZ over seeds against the reported lnZ_err.  The
    flux errors are inflated 30-fold so that the effective sample size is in the hundreds to
    thousands, where the delta method holds; with the real errors a handful of draws carry the
    evidence (ess of a few) and the sample variance of the weights underestimates the spread
    (DESIGN.md section 4e)."""
    import triceratops_b200
    from triceratops_b200 import marginal_likelihoods as ml
    t, f, s = toi465_lc
    args = (t, f, 30 * s, TOI465["P"], TOI465["M"], TOI465["R"], TOI465["Teff"], 0.0)
    for name in ("lnZ_TTP", "lnZ_TEB"):
        lnZ, err, ess = [], [], []
        with triceratops_b200.mc_errors():
            for seed in range(64):
                np.random.seed(1000 + seed)
                res = getattr(ml, name)(*args, N=100_000, parallel=True)
                res = res[0] if isinstance(res, tuple) else res
                lnZ.append(res["lnZ"])
                err.append(res.lnZ_err)
                ess.append(res.ess)
        assert np.median(ess) > 100
        ratio = np.std(lnZ, ddof=1) / np.median(err)
        assert 0.75 <= ratio <= 1.33, (name, ratio)


@pytest.mark.parametrize("sampler", ["host", "device"])
def test_refinement_reaches_the_target(gpu_engine, sampler):
    from _workloads import lightcurve, make_target, run_calc_probs
    from triceratops_b200 import set_sampler
    lc = lightcurve(2)
    set_sampler(sampler, seed=7)
    try:
        base = run_calc_probs(make_target(2), 2, lc, 100_000, 7, mc_errors=True)
        tgt = run_calc_probs(make_target(2), 2, lc, 100_000, 7, fpp_err_target=0.02)
        assert tgt.FPP_err <= 0.02
        # a target below the first round's error: rounds run, within N_max = 16 N
        tight = base.FPP_err / 4
        ref = run_calc_probs(make_target(2), 2, lc, 100_000, 7, fpp_err_target=tight)
        assert 100_000 < ref.N_draws.max() <= 1_600_000
        assert ref.FPP_err <= tight or ref.N_draws.max() == 1_600_000
        if sampler == "host":
            again = run_calc_probs(make_target(2), 2, lc, 100_000, 7, fpp_err_target=tight)
            # the same draws and rounds; FPP_err to rounding (the light-curve kernel's evidence
            # sums merge its blocks in the order they finish)
            assert np.array_equal(again.N_draws, ref.N_draws)
            np.testing.assert_allclose(again.lnZ, ref.lnZ, rtol=0, atol=1e-12)
            assert again.FPP_err == pytest.approx(ref.FPP_err, rel=1e-9)
    finally:
        set_sampler("host")
