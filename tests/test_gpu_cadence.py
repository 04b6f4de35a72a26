"""Mixed-cadence light curves on the GPU (tri_set_lightcurve_cadence, lnl_seg_kernel): constant
cadence arrays are the scalar call, chi^2 is additive over cadence groups on the lnL_*_p seam,
the L2 seam agrees with the per-group oracle (tests/_cadence_oracle.py), simulated rows come
back in the caller's order, the C ABI rejects bad cadences, and calc_probs runs on a mixed
curve with both samplers."""
import ctypes
import os

import numpy as np
import pytest

from _cadence_oracle import CadenceOracleEngine, cadence_groups, mixed_lightcurve
from conftest import GOLD, TOI465, draw_eb_columns, draw_tp_columns

pytestmark = pytest.mark.gpu

SCALAR = (0.00139, 20)


@pytest.fixture(scope="module")
def mixed_lc(toi465_lc):
    t, f, s = toi465_lc
    return mixed_lightcurve(t, f) + (s,)


def _restore(eng, lc):
    t, f, s = lc
    eng.set_lightcurve(t, f, s, *SCALAR)


@pytest.mark.parametrize("pointwise", [False, True])
def test_constant_cadence_arrays_are_the_scalar_call(gpu_engine, toi465_lc, pointwise):
    t, f, s = toi465_lc
    sig = s * np.random.default_rng(1).uniform(0.5, 2.0, t.size) if pointwise else s
    N = 20000
    tp, eb = draw_tp_columns(N, 21), draw_eb_columns(N, 22)
    out = []
    try:
        for e, n in (SCALAR, (np.full(t.size, SCALAR[0]), np.full(t.size, SCALAR[1]))):
            gpu_engine.set_lightcurve(t, f, sig, e, n)
            out.append((gpu_engine.eval_tp(N, **tp, want_mask=True),
                        gpu_engine.eval_eb(N, **eb, want_mask=True)))
    finally:
        _restore(gpu_engine, toi465_lc)
    (a, (a0, a1)), (b, (b0, b1)) = out
    for x, y in ((a, b), (a0, b0), (a1, b1)):
        assert np.array_equal(x.mask, y.mask)
        assert np.array_equal(x.lnL, y.lnL)
        assert abs(x.lnZ - y.lnZ) <= 1e-12 * max(1.0, abs(x.lnZ))


def _additivity_lc(t, f):
    """2-min stamps (ns 20); their 30-min binned copy with ns 80 (>= 64: the offset formula
    instead of the table); and 40 stamps at 1.0-1.2 d after mid-transit, outside every window
    of a P = 3.84 d orbit (200-s exposures, ns 5)."""
    time, flux, exptime, nsamples = mixed_lightcurve(t, f, seed=5)
    nsamples = np.where(exptime > 0.01, 80, nsamples).astype(np.int32)
    far = np.linspace(1.0, 1.2, 40)
    time = np.r_[time, far]
    flux = np.r_[flux, 1.0 + 1e-4 * np.sin(far * 50)]
    exptime = np.r_[exptime, np.full(far.size, 200 / 86400)]
    nsamples = np.r_[nsamples, np.full(far.size, 5, dtype=np.int32)]
    return time, flux, exptime, nsamples


def test_chi2_is_additive_over_cadence_groups(gpu_engine, toi465_lc):
    from oracle.engine_port import eb_masks, tp_mask
    from triceratops_b200 import likelihoods as lk
    t, f, s = toi465_lc
    time, flux, exptime, nsamples = _additivity_lc(t, f)
    groups = cadence_groups(exptime, nsamples, time.size)
    assert len(groups) == 3 and max(g[2] for g in groups) >= 64
    N = 6000
    c = draw_tp_columns(N, 31)
    mask, a = tp_mask(N, c["rp"], c["P_orb"], c["inc"], c["ecc"], c["argp"], c["mtot"], c["rhost"])
    m = np.flatnonzero(mask)
    tp_args = (c["rp"][m], c["P_orb"], c["inc"][m], a[m], c["rhost"], c["u1"], c["u2"],
               c["ecc"][m], c["argp"][m], c["cfr"])
    e = draw_eb_columns(N, 32)
    (mk, ak), (mt, at) = eb_masks(N, e["reb"], e["q"], e["P_orb"], e["inc"], e["ecc"], e["argp"],
                                  e["mtot"], e["rhost"])

    def eb_args(mm, aa, P):
        k = np.flatnonzero(mm)
        return (e["reb"][k], e["ebfr"][k], P, e["inc"][k], aa[k], e["rhost"], e["u1"], e["u2"],
                e["ecc"][k], e["argp"][k], e["cfr"])
    calls = [(lk.lnL_TP_p, tp_args), (lk.lnL_EB_p, eb_args(mk, ak, e["P_orb"])),
             (lk.lnL_EB_twin_p, eb_args(mt, at, 2 * e["P_orb"]))]
    try:
        for fn, args in calls:
            assert args[0].size > 20
            mixed = fn(time, flux, s, *args, exptime=exptime, nsamples=nsamples)
            parts = [fn(time[idx], flux[idx], s, *args, exptime=ge, nsamples=gn)
                     for idx, ge, gn in groups]
            total = sum(parts)
            fin = np.isfinite(total)
            assert np.array_equal(np.isfinite(mixed), fin), fn.__name__
            assert np.array_equal(np.isposinf(mixed), np.isposinf(total)), fn.__name__
            np.testing.assert_allclose(mixed[fin], total[fin], rtol=1e-12, err_msg=fn.__name__)
        # the far group is out of transit for every draw: its chi^2 is that of model == 1
        far = [g for g in groups if g[1] == 200 / 86400][0][0]
        want = 0.5 * np.sum((flux[far] - 1.0) ** 2) / s ** 2
        got = lk.lnL_TP_p(time[far], flux[far], s, *tp_args, exptime=200 / 86400, nsamples=5)
        np.testing.assert_allclose(got, want, rtol=1e-12)
    finally:
        _restore(gpu_engine, toi465_lc)


@pytest.mark.parametrize("is_host", [False, True])
def test_l2_seam_matches_the_per_group_oracle(gpu_engine, mixed_lc, toi465_lc, is_host):
    time, flux, exptime, nsamples, s = mixed_lc
    ora = CadenceOracleEngine()
    ora.set_lightcurve(time, flux, s, exptime, nsamples)
    N = 20000
    tp = draw_tp_columns(N, 41)
    tp["cfr"] = 0.1 if is_host else 0.0
    eb = draw_eb_columns(N, 42)
    eb["cfr"] = 0.1 if is_host else 0.0
    gpu_engine.set_lightcurve(time, flux, s, exptime, nsamples)
    try:
        pairs = [(gpu_engine.eval_tp(N, **tp, companion_is_host=is_host, want_mask=True),
                  ora.eval_tp(N, **tp, companion_is_host=is_host))]
        for loop in (False, True):
            g = gpu_engine.eval_eb(N, **eb, companion_is_host=is_host, want_mask=True,
                                   scalar_loop=loop)
            o = ora.eval_eb(N, **eb, companion_is_host=is_host, scalar_loop=loop)
            pairs += list(zip(g, o))
    finally:
        _restore(gpu_engine, toi465_lc)
    for g, o in pairs:
        assert np.array_equal(g.mask, o.mask)
        fin = np.isfinite(o.lnL)
        assert np.array_equal(np.isfinite(g.lnL), fin)
        np.testing.assert_allclose(g.lnL[fin], o.lnL[fin], rtol=1e-9)
        assert abs(g.lnZ - o.lnZ) < 1e-6 or g.lnZ == o.lnZ


def test_simulate_rows_in_caller_order(gpu_engine, mixed_lc, toi465_lc):
    from oracle.engine_port import eb_masks, tp_mask
    from triceratops_b200 import likelihoods as lk
    time, flux, exptime, nsamples, s = mixed_lc
    groups = cadence_groups(exptime, nsamples, time.size)
    N = 3000
    c = draw_tp_columns(N, 51)
    mask, a = tp_mask(N, c["rp"], c["P_orb"], c["inc"], c["ecc"], c["argp"], c["mtot"], c["rhost"])
    m = np.flatnonzero(mask)[:200]
    targs = (c["rp"][m], c["P_orb"], c["inc"][m], a[m], c["rhost"], c["u1"], c["u2"],
             c["ecc"][m], c["argp"][m], np.full(m.size, 0.05))
    e = draw_eb_columns(N, 52)
    (mk, ak), _ = eb_masks(N, e["reb"], e["q"], e["P_orb"], e["inc"], e["ecc"], e["argp"],
                           e["mtot"], e["rhost"])
    k = np.flatnonzero(mk)[:200]
    eargs = (e["reb"][k], e["ebfr"][k], e["P_orb"], e["inc"][k], ak[k], e["rhost"], e["u1"],
             e["u2"], e["ecc"][k], e["argp"][k], np.full(k.size, 0.05))
    try:
        rows = lk.simulate_TP_transit_p(time, *targs, exptime=exptime, nsamples=nsamples)
        erows, esec = lk.simulate_EB_transit_p(time, *eargs, exptime=exptime, nsamples=nsamples)
        want = np.empty_like(rows)
        ewant = np.empty_like(erows)
        for idx, ge, gn in groups:
            want[:, idx] = lk.simulate_TP_transit_p(time[idx], *targs, exptime=ge, nsamples=gn)
            ewant[:, idx], sec = lk.simulate_EB_transit_p(time[idx], *eargs, exptime=ge,
                                                          nsamples=gn)
            # (the secondary pass is the same for every group; the two kernels may round it
            # differently)
            np.testing.assert_allclose(np.asarray(sec), np.asarray(esec), rtol=1e-13, atol=1e-15)
    finally:
        _restore(gpu_engine, toi465_lc)
    assert np.any(rows < 1 - 1e-4) and np.any(erows < 1 - 1e-4)
    np.testing.assert_allclose(rows, want, rtol=1e-13, atol=0)
    np.testing.assert_allclose(erows, ewant, rtol=1e-13, atol=0)


def test_c_abi_rejects_bad_cadences(gpu_engine, toi465_lc):
    from triceratops_b200 import _cabi
    t, f, s = toi465_lc
    n = t.size
    lib = gpu_engine.lib
    tt, ff = _cabi.f64(t), _cabi.f64(f)
    i32 = ctypes.POINTER(ctypes.c_int32)
    good_e = np.full(n, 0.00139)
    good_n = np.full(n, 20, dtype=np.int32)
    bad = []
    for j, v in ((0, np.nan), (1, -0.001)):
        e = good_e.copy()
        e[j] = v
        bad.append((e, good_n))
    nz = good_n.copy()
    nz[3] = 0
    bad.append((good_e, nz))
    bad.append((0.001 * (1 + np.arange(n) % 9), good_n))
    try:
        for e, ns in bad:
            e = _cabi.f64(e)
            ns = np.ascontiguousarray(ns, dtype=np.int32)
            rc = lib.tri_set_lightcurve_cadence(_cabi.dptr(tt), _cabi.dptr(ff), None, s,
                                                _cabi.dptr(e), ns.ctypes.data_as(i32), n)
            assert rc == _cabi.TRI_EINVAL
            assert lib.tri_last_error().decode()
        e8 = _cabi.f64(0.001 * (1 + np.arange(n) % 8))
        assert lib.tri_set_lightcurve_cadence(_cabi.dptr(tt), _cabi.dptr(ff), None, s,
                                              _cabi.dptr(e8), good_n.ctypes.data_as(i32),
                                              n) == _cabi.TRI_OK
    finally:
        gpu_engine._lc_key = None
        _restore(gpu_engine, toi465_lc)


def _calc_probs(time, flux, err, exptime, nsamples, N, seed):
    from triceratops_b200 import synthetic as synth
    from triceratops_b200.triceratops import target
    stars = synth.stars_table(9, TOI465["T"], TOI465["J"], TOI465["H"], TOI465["K"], TOI465["M"],
                              TOI465["R"], TOI465["Teff"], TOI465["plx"], n_neighbours=0)
    tgt = target(9, stars=stars, trilegal_fname=os.path.join(GOLD, "trilegal_synth.csv"))
    np.random.seed(seed)
    tgt.calc_probs(time, flux, err, TOI465["P"], N=N, parallel=True, verbose=0,
                   exptime=exptime, nsamples=nsamples,
                   drop_scenario=["PTP", "PEB", "STP", "SEB", "DEB", "BTP", "BEB"])
    return tgt


def test_calc_probs_on_a_mixed_curve(gpu_engine, mixed_lc, toi465_lc):
    import _cadence_oracle
    from oracle.engine_port import uninstall
    import triceratops_b200
    time, flux, exptime, nsamples, s = mixed_lc
    N = 100_000
    gpu = _calc_probs(time, flux, s, exptime, nsamples, N, 7)
    _cadence_oracle.install()
    try:
        ora = _calc_probs(time, flux, s, exptime, nsamples, N, 7)
    finally:
        uninstall()
    fin = np.isfinite(ora.lnZ)
    assert fin.sum() >= 3 and np.array_equal(np.isfinite(gpu.lnZ), fin)
    np.testing.assert_allclose(gpu.lnZ[fin], ora.lnZ[fin], rtol=0, atol=1e-6)
    np.testing.assert_allclose(gpu.probs.prob.values, ora.probs.prob.values, rtol=0, atol=1e-6)
    # the device sampler: a finite table on the mixed curve; constant arrays = the scalar call
    t, f, _ = toi465_lc
    try:
        triceratops_b200.set_sampler("device", seed=9)
        dev = _calc_probs(time, flux, s, exptime, nsamples, N, 7)
        assert np.isfinite(dev.lnZ).sum() >= 3 and np.isfinite(dev.FPP)
        out = []
        for e, n in (SCALAR, (np.full(t.size, SCALAR[0]), np.full(t.size, SCALAR[1]))):
            triceratops_b200.set_sampler("device", seed=10)
            out.append(_calc_probs(t, f, s, e, n, N, 7))
    finally:
        triceratops_b200.set_sampler("host")
        _restore(gpu_engine, toi465_lc)
    np.testing.assert_array_equal(out[0].lnZ, out[1].lnZ)
    np.testing.assert_array_equal(out[0].probs.prob.values, out[1].probs.prob.values)
