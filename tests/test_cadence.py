"""Mixed-cadence light curves on the CPU: validation of per-stamp exposure times and sample
counts, the per-group oracle (tests/_cadence_oracle.py), calc_probs end to end on it, and the
two-rank scatter path over gloo with a mixed light curve."""
import os
import pickle
import socket
import subprocess
import sys
import threading

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from _cadence_oracle import CadenceOracleEngine, cadence_groups, mixed_lightcurve  # noqa: E402
from conftest import TOI465, draw_eb_columns, draw_tp_columns, load_lc  # noqa: E402


@pytest.fixture()
def cadence_oracle():
    import _cadence_oracle
    from oracle.engine_port import uninstall
    eng = _cadence_oracle.install()
    yield eng
    uninstall()


@pytest.fixture(scope="module")
def mixed_lc(toi465_lc):
    t, f, s = toi465_lc
    return mixed_lightcurve(t, f) + (s,)


def _engine_without_device():
    """Engine.set_lightcurve on an engine whose library is never reached: validation must fail
    before any call into it."""
    from triceratops_b200.engine import Engine
    eng = object.__new__(Engine)
    eng._lock = threading.RLock()
    eng.lib = None
    eng._lc_key = None
    return eng


BAD_CADENCES = [
    ("length", np.full(9, 0.00139), 20),
    ("length", 0.00139, np.full(11, 20)),
    ("nan", np.r_[np.full(9, 0.00139), np.nan], 20),
    ("negative", np.r_[np.full(9, 0.00139), -0.001], 20),
    ("infinite", np.r_[np.full(9, 0.00139), np.inf], 20),
    ("zero samples", 0.00139, np.r_[np.full(9, 20), 0]),
    ("non-integer samples", 0.00139, np.r_[np.full(9, 20.0), 2.5]),
    ("nine cadences", 0.001 * (1 + np.arange(10) % 9), 20),
]


@pytest.mark.parametrize("what,exptime,nsamples", BAD_CADENCES, ids=[b[0] for b in BAD_CADENCES])
def test_bad_cadences_raise_before_the_engine(what, exptime, nsamples):
    from triceratops_b200.engine import cadence_columns
    t = np.linspace(-0.1, 0.1, 10)
    with pytest.raises(ValueError):
        cadence_columns(exptime, nsamples, t.size)
    with pytest.raises(ValueError):
        _engine_without_device().set_lightcurve(t, np.ones(10), 1e-3, exptime, nsamples)
    with pytest.raises(ValueError):
        CadenceOracleEngine().set_lightcurve(t, np.ones(10), 1e-3, exptime, nsamples)


def test_cadence_columns_collapse_and_keep():
    from triceratops_b200.engine import cadence_columns
    e, n = cadence_columns(np.full(5, 0.02), np.full(5, 7.0), 5)
    assert (e, n) == (0.02, 7) and type(e) is float and type(n) is int
    e, n = cadence_columns(0.001 * (1 + np.arange(16) % 8), 20, 16)   # eight cadences: accepted
    assert e.dtype == np.float64 and n.dtype == np.int32 and n.shape == (16,)
    groups = cadence_groups(np.r_[0.02, 0.001, 0.02, 0.0], np.r_[20, 20, 20, 1], 4)
    assert [(list(i), e, n) for i, e, n in groups] == [([3], 0.0, 1), ([1], 0.001, 20),
                                                       ([0, 2], 0.02, 20)]


def test_constant_cadence_arrays_equal_the_scalar_call(toi465_lc):
    t, f, s = toi465_lc
    N = 3000
    tp, eb = draw_tp_columns(N, 11), draw_eb_columns(N, 12)
    out = []
    for e, n in ((0.00139, 20), (np.full(t.size, 0.00139), np.full(t.size, 20))):
        eng = CadenceOracleEngine()
        eng.set_lightcurve(t, f, s, e, n)
        out.append((eng.eval_tp(N, **tp), eng.eval_eb(N, **eb)))
    (a, (a0, a1)), (b, (b0, b1)) = out
    for x, y in ((a, b), (a0, b0), (a1, b1)):
        assert np.array_equal(x.mask, y.mask)
        assert np.array_equal(x.lnL, y.lnL)
        assert x.lnZ == y.lnZ


def test_mixed_chi2_is_the_sum_of_the_groups(mixed_lc):
    from oracle.engine_port import OracleEngine
    time, flux, exptime, nsamples, s = mixed_lc
    N = 3000
    tp, eb = draw_tp_columns(N, 13), draw_eb_columns(N, 14)
    eng = CadenceOracleEngine()
    eng.set_lightcurve(time, flux, s, exptime, nsamples)
    mixed_tp = eng.eval_tp(N, **tp)
    mixed_eb = eng.eval_eb(N, **eb)
    const = -0.5 * np.log(2 * np.pi) - np.log(s)
    parts_tp, parts_eb = 0.0, [0.0, 0.0]
    groups = cadence_groups(exptime, nsamples, time.size)
    assert len(groups) == 2
    for idx, e, n in groups:
        one = OracleEngine()
        one.set_lightcurve(time[idx], flux[idx], s, e, n)
        r = one.eval_tp(N, **tp)
        parts_tp = parts_tp + (const - r.lnL)
        for b, rb in enumerate(one.eval_eb(N, **eb)):
            parts_eb[b] = parts_eb[b] + (const - rb.lnL)
    for res, half in ((mixed_tp, parts_tp), (mixed_eb[0], parts_eb[0]),
                      (mixed_eb[1], parts_eb[1])):
        fin = np.isfinite(res.lnL)
        assert fin.sum() > (100 if res is mixed_tp else 0)
        assert np.array_equal(fin, np.isfinite(half))
        np.testing.assert_allclose(const - res.lnL[fin], half[fin], rtol=1e-13)


def _three_groups(t, f):
    """2-min stamps (ns 20), their 30-min binned copy (ns 20) and one unbinned stamp (ns 1)."""
    time, flux, exptime, nsamples = mixed_lightcurve(t, f, seed=3)
    time = np.r_[time, 0.0005]
    flux = np.r_[flux, 0.999]
    exptime = np.r_[exptime, 0.0]
    nsamples = np.r_[nsamples, 1]
    return time, flux, exptime, nsamples


def _calc_probs(t, f, err, exptime, nsamples, N=301, seed=77):
    from triceratops_b200 import synthetic as synth
    from triceratops_b200.triceratops import target
    stars = synth.stars_table(9, TOI465["T"], TOI465["J"], TOI465["H"], TOI465["K"], TOI465["M"],
                              TOI465["R"], TOI465["Teff"], TOI465["plx"], n_neighbours=0)
    tgt = target(9, stars=stars, trilegal_fname=os.path.join(ROOT, "tests", "golden",
                                                              "trilegal_synth.csv"))
    np.random.seed(seed)
    tgt.calc_probs(t, f, err, TOI465["P"], N=N, parallel=True, verbose=0,
                   exptime=exptime, nsamples=nsamples,
                   drop_scenario=["PTP", "PEB", "STP", "SEB", "DEB", "BTP", "BEB"])
    return tgt


def test_calc_probs_three_cadences_on_the_oracle(cadence_oracle, toi465_lc):
    t, f, s = toi465_lc
    time, flux, exptime, nsamples = _three_groups(t, f)
    assert len(cadence_groups(exptime, nsamples, time.size)) == 3
    for err in (s, s * np.random.default_rng(2).uniform(0.5, 2.0, time.size)):
        tgt = _calc_probs(time, flux, err, exptime, nsamples)
        assert np.isfinite(tgt.lnZ).sum() >= 3
        assert np.isfinite(tgt.FPP) and abs(tgt.probs.prob.sum() - 1.0) < 1e-9
        # the cadence differs from today's workaround: the forced single cadence moves lnZ
        forced = _calc_probs(time, flux, err, 0.00139, 20)
        fin = np.isfinite(tgt.lnZ)
        assert np.max(np.abs(tgt.lnZ[fin] - forced.lnZ[fin])) > 1e-6


class _Recorder(CadenceOracleEngine):
    def set_lightcurve(self, time, flux, sigma, exptime, nsamples):
        self.seen = (np.asarray(time), np.asarray(flux), exptime, nsamples)
        super().set_lightcurve(time, flux, sigma, exptime, nsamples)


def test_calc_probs_drops_nan_rows_from_the_cadence(toi465_lc):
    from oracle.engine_port import install, uninstall
    t, f, s = toi465_lc
    time, flux, exptime, nsamples = _three_groups(t, f)
    time, flux = time.copy(), flux.copy()
    time[5] = np.nan
    flux[17] = np.nan
    eng = install(_Recorder())
    try:
        _calc_probs(time, flux, s, exptime, nsamples, N=50)
        keep = np.ones(time.size, bool)
        keep[[5, 17]] = False
        rt, rf, re, rn = eng.seen
        assert np.array_equal(rt, time[keep])
        assert np.array_equal(re, exptime[keep]) and np.array_equal(rn, nsamples[keep])
        with pytest.raises(ValueError):
            _calc_probs(time, flux, s, exptime[:-1], nsamples, N=50)
        with pytest.raises(ValueError):
            _calc_probs(time, flux, s, exptime, nsamples[:-1], N=50)
    finally:
        uninstall()


# ---- two ranks over gloo, scatter mode (the pattern of test_dist_gloo.py) --------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(out_path):
    """One rank: calc_probs with a mixed light curve; rank 0 draws and scatters."""
    import torch.distributed as dist
    dist.init_process_group("gloo")
    import _cadence_oracle
    _cadence_oracle.install()
    t, f, s = load_lc("TOI465_01_lightcurve.csv")
    time, flux, exptime, nsamples = mixed_lightcurve(t, f)
    tgt = _calc_probs(time, flux, s, exptime, nsamples)
    with open(out_path + ".%d" % dist.get_rank(), "wb") as fh:
        pickle.dump(dict(lnZ=tgt.lnZ.copy(), prob=tgt.probs.prob.values.copy(),
                         R_p=tgt.probs.R_p.values.copy(), FPP=float(tgt.FPP),
                         collectives=tgt.collectives), fh)
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_equal_one_with_mixed_cadence(tmp_path, cadence_oracle, mixed_lc):
    out = str(tmp_path / "res.pkl")
    port = _free_port()
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE="2",
                   MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), OMP_NUM_THREADS="2")
        procs.append(subprocess.Popen([sys.executable, os.path.abspath(__file__), out], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    logs = [p.communicate(timeout=600)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    res = [pickle.load(open(out + ".%d" % r, "rb")) for r in range(2)]
    time, flux, exptime, nsamples, s = mixed_lc
    one = _calc_probs(time, flux, s, exptime, nsamples)
    assert np.isfinite(one.lnZ).sum() >= 3
    for r in res:
        np.testing.assert_allclose(r["lnZ"], one.lnZ, rtol=0, atol=1e-9)
        np.testing.assert_allclose(r["prob"], one.probs.prob.values, rtol=0, atol=1e-9)
        np.testing.assert_allclose(r["R_p"], one.probs.R_p.values, rtol=1e-12)
        assert abs(r["FPP"] - one.FPP) < 1e-9
        assert r["collectives"]["scatters"] == 3


if __name__ == "__main__":
    _worker(sys.argv[1])
