"""Monte-Carlo error bars of lnZ, the scenario probabilities, FPP and NFPP, and refinement of
calc_probs toward a requested FPP precision, on the CPU: the statistics of _numerics on
synthetic ln-weights, calc_probs on the moments oracle (tests/_mc_oracle.py), and a two-rank
gloo run."""
import math
import os
import pickle
import socket
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from conftest import TOI465, load_lc  # noqa: E402
from triceratops_b200 import _numerics as nx  # noqa: E402
from triceratops_b200.engine import combine_lse, combine_moments  # noqa: E402


def _lnw(seed, N=5000, frac=0.3):
    rng = np.random.default_rng(seed)
    x = rng.normal(-3.0, 2.0, N)
    x[rng.random(N) > frac] = -np.inf
    return x


# ---- statistics ------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["spread", "one finite", "with -inf"])
def test_lnZ_err_and_ess_equal_the_standard_error_of_the_mean(case):
    if case == "spread":
        x = np.random.default_rng(1).normal(0.0, 1.5, 2000)
    elif case == "one finite":
        x = np.full(10, -np.inf)
        x[4] = -7.0
    else:
        x = _lnw(2)
    N = x.size
    rec = nx.lse_moments(x)
    err, ess, r = nx.mc_error(N, *rec)
    w = np.exp(x)
    sem = np.std(w, ddof=1) / np.sqrt(N)
    assert err == pytest.approx(sem / np.mean(w), rel=1e-9)
    assert ess == pytest.approx(w.sum() ** 2 / (w * w).sum(), rel=1e-12)
    assert r == pytest.approx(err ** 2, rel=1e-12)


def test_edge_cases():
    x = np.array([0.0, np.inf, -1.0])
    assert math.isnan(nx.mc_error(3, *nx.lse_moments(x))[0])
    none = nx.lse_moments(np.full(5, -np.inf))
    err, ess, r = nx.mc_error(5, *none)
    assert math.isnan(err) and ess == 0.0 and r == 0.0
    # a row without finite weights carries no variance
    lnZ = np.r_[-1.0, -np.inf, -2.0, -0.5, np.full(8, -3.0)]
    r = np.r_[0.01, 0.0, 0.02, 0.03, np.full(8, 0.01)]
    calls = [[0], [1, 2], [3]] + [[j] for j in range(4, 12)]
    pe, fe, ne, contrib = nx.probability_errors(lnZ, r, calls, [100] * len(calls))
    assert pe[1] == 0.0 and np.isfinite(fe) and ne == 0.0 and contrib[1] >= 0


def test_shard_and_round_combined_s2_equals_the_whole():
    x = _lnw(3, N=9000)
    whole = nx.lse_moments(x)
    for cuts in ([3000, 6000], [1, 8999], [4500]):
        parts = [nx.lse_moments(p) for p in np.split(x, cuts)]
        m, s, s2, nf, npi = combine_moments(parts)
        assert (m, nf, npi) == (whole[0], whole[3], whole[4])
        assert s == pytest.approx(whole[1], rel=1e-13)
        assert s2 == pytest.approx(whole[2], rel=1e-13)
        lnZ = combine_lse([(p[0], p[1], p[3], p[4]) for p in parts], x.size)
        assert lnZ == pytest.approx(nx._log_mean_exp(x, N_total=x.size), abs=1e-12)


def test_delta_method_gradient_matches_finite_differences():
    rng = np.random.default_rng(4)
    Z = rng.uniform(0.1, 2.0, 20)
    for R in ([0, 3, 9], [5], list(range(15, 20))):
        g = nx.sum_gradient(Z, R)
        for j in range(Z.size):
            h = 1e-6 * Z[j]
            zp, zm = Z.copy(), Z.copy()
            zp[j] += h
            zm[j] -= h
            fd = (zp[R].sum() / zp.sum() - zm[R].sum() / zm.sum()) / (2 * h)
            assert g[j] == pytest.approx(fd, rel=1e-6, abs=1e-9)


def test_eb_covariance_matches_its_definition():
    # two branches of one call: the same draws, disjoint masks
    rng = np.random.default_rng(5)
    N = 4000
    x = rng.normal(-2.0, 1.0, N)
    twin = rng.random(N) < 0.3
    wa = np.where(~twin, np.exp(x), 0.0)
    wb = np.where(twin, np.exp(x), 0.0)
    Za, Zb = wa.mean(), wb.mean()
    direct = np.cov(wa, wb, ddof=1)[0, 1] / N
    lnZ = np.log([Za, Zb])
    ra = nx.mc_error(N, *nx.lse_moments(np.log(wa)))[2]
    rb = nx.mc_error(N, *nx.lse_moments(np.log(wb)))[2]
    Z, V = nx.evidence_covariance(lnZ, np.array([ra, rb]), [[0, 1]], [N])
    scale = math.exp(lnZ.max())
    assert V[0, 1] * scale ** 2 == pytest.approx(direct, rel=1e-9)
    assert V[0, 0] * scale ** 2 == pytest.approx(np.var(wa, ddof=1) / N, rel=1e-9)


def test_fpp_err_agrees_with_a_bootstrap():
    rng = np.random.default_rng(6)
    N, n_rows = 20000, 18
    calls = [[0], [1, 2], [3], [4, 5], [6], [7, 8], [9], [10, 11], [12], [13, 14], [15],
             [16, 17]]
    lnw = {}
    for rows in calls:
        x = rng.normal(rng.uniform(-6, -2), 1.2, N)
        x[rng.random(N) < 0.5] = -np.inf
        if len(rows) == 2:
            twin = rng.random(N) < 0.4
            lnw[rows[0]] = np.where(twin, -np.inf, x)
            lnw[rows[1]] = np.where(twin, x, -np.inf)
        else:
            lnw[rows[0]] = x

    def fpp(idx_by_call):
        lnZ = np.empty(n_rows)
        for rows, idx in zip(calls, idx_by_call):
            for j in rows:
                lnZ[j] = nx._log_mean_exp(lnw[j][idx], N_total=N)
        p = np.exp(lnZ - np.logaddexp.reduce(lnZ))
        return 1 - (p[0] + p[3] + p[9]), lnZ

    ident = [np.arange(N)] * len(calls)
    _, lnZ = fpp(ident)
    r = np.array([nx.mc_error(N, *nx.lse_moments(lnw[j]))[2] for j in range(n_rows)])
    _, fpp_err, _, contrib = nx.probability_errors(lnZ, r, calls, [N] * len(calls))
    assert contrib.sum() == pytest.approx(fpp_err ** 2, rel=1e-12)
    boot = [fpp([rng.integers(0, N, N) for _ in calls])[0] for _ in range(2000)]
    assert fpp_err == pytest.approx(np.std(boot, ddof=1), rel=0.10)


# ---- calc_probs on the moments oracle -------------------------------------------------------
_DROP = ["PTP", "PEB", "STP", "SEB", "DTP", "DEB", "BTP"]


@pytest.fixture()
def mc_oracle():
    import _mc_oracle
    from oracle.engine_port import uninstall
    eng = _mc_oracle.install(_mc_oracle.MomentsOracleEngine())
    yield eng
    uninstall()


def _target(n_neighbours=1):
    from triceratops_b200 import synthetic as synth
    from triceratops_b200.triceratops import target
    stars = synth.stars_table(9, TOI465["T"], TOI465["J"], TOI465["H"], TOI465["K"], TOI465["M"],
                              TOI465["R"], TOI465["Teff"], TOI465["plx"],
                              n_neighbours=n_neighbours)
    return target(9, stars=stars, trilegal_fname=os.path.join(ROOT, "tests", "golden",
                                                              "trilegal_synth.csv"))


def _calc_probs(lc, N=300, seed=11, **kw):
    """calc_probs with the flux errors inflated tenfold: at N = 300 the rows' evidences are
    then of comparable size (FPP about 0.7 +- 0.17), not one row taking all the probability."""
    t, f, s = lc
    tgt = _target()
    np.random.seed(seed)
    tgt.calc_probs(t, f, 10 * s, TOI465["P"], N=N, parallel=True, verbose=0,
                   drop_scenario=_DROP, **kw)
    return tgt


def test_mc_errors_leave_the_results_bit_identical(mc_oracle, toi465_lc):
    plain = _calc_probs(toi465_lc)
    assert plain.FPP_err is None and plain.lnZ_err is None and "prob_err" not in plain.probs
    err = _calc_probs(toi465_lc, mc_errors=True)
    assert np.array_equal(plain.lnZ, err.lnZ)
    assert np.array_equal(plain.probs.prob.values, err.probs.prob.values)
    assert plain.FPP == err.FPP and plain.NFPP == err.NFPP
    assert np.array_equal(plain.probs.R_p.values, err.probs.R_p.values)
    assert np.isfinite(err.FPP_err) and err.FPP_err > 0 and np.isfinite(err.NFPP_err)
    ran = np.isfinite(err.lnZ)
    assert np.all(np.isfinite(err.lnZ_err[ran])) and np.all(err.N_draws[ran] == 300)
    assert np.all(err.N_draws[~np.isfinite(err.lnZ) & (err.N_draws == 0)] == 0)
    assert np.all(err.probs.prob_err.values >= 0)
    # the row errors agree with the per-draw ln-weights of the oracle
    lnw = mc_oracle.draws[-1]       # the last call: the nearby star's NEB pair, branch NEBx2P
    e, ess, _ = nx.mc_error(300, *nx.lse_moments(lnw))
    if np.isfinite(err.lnZ[-1]):
        assert err.lnZ_err[-1] == pytest.approx(e, rel=1e-12)
        assert err.ess[-1] == pytest.approx(ess, rel=1e-12)


def test_loose_target_runs_no_extra_round(mc_oracle, toi465_lc):
    ref = _calc_probs(toi465_lc, mc_errors=True)
    n0 = len(mc_oracle.draws)
    mc_oracle.draws.clear()
    tgt = _calc_probs(toi465_lc, fpp_err_target=1.0)
    assert len(mc_oracle.draws) == n0
    assert np.all(tgt.N_draws[tgt.N_draws > 0] == 300)
    assert np.array_equal(tgt.lnZ, ref.lnZ) and tgt.FPP_err == ref.FPP_err


def test_tight_target_refines_and_merges_the_rounds(mc_oracle, toi465_lc):
    tgt0 = _calc_probs(toi465_lc, mc_errors=True)
    mc_oracle.calls.clear()
    tgt = _calc_probs(toi465_lc, fpp_err_target=1e-9, N_max=1200)
    assert tgt.N_draws.max() == 1200
    assert set(np.unique(tgt.N_draws)) <= {0, 300, 600, 1200}
    # round 0 is the plain call: the generator was consumed the same way up to there
    assert np.array_equal(tgt.lnZ[tgt.N_draws == 300], tgt0.lnZ[tgt.N_draws == 300])
    # per-draw ln-weights of every evaluation, grouped by scenario call: round 0 first; the
    # calls of this table in row order: TP, EB (2 rows), BEB (2), NTP, NEB (2)
    rows_of_call = [[0], [1, 2], [13, 14], [15], [16, 17]]
    by_key = {}
    for key, lnw in mc_oracle.calls:
        by_key.setdefault(key, []).append(lnw)
    assert len(by_key) == len(rows_of_call)
    rounds = dict(zip(map(tuple, rows_of_call), by_key.values()))
    for rows, parts in rounds.items():
        for b, j in enumerate(rows):
            cat = np.concatenate([p[b] for p in parts])
            assert cat.size == tgt.N_draws[j]
            want = nx._log_mean_exp(cat, N_total=cat.size)
            if np.isfinite(want):
                assert tgt.lnZ[j] == pytest.approx(want, abs=1e-12)
            else:
                assert tgt.lnZ[j] == want


def test_refined_table_is_the_top_of_the_union(mc_oracle, toi465_lc):
    from triceratops_b200 import marginal_likelihoods as ml
    from triceratops_b200.triceratops import _merge_round
    t, f, s = toi465_lc
    from triceratops_b200 import _dispatch
    _dispatch.use_lightcurve(t, f, s, 0.00139, 20)
    with _dispatch.mc_errors():
        np.random.seed(3)
        a = ml.lnZ_TTP(t, f, s, TOI465["P"], TOI465["M"], TOI465["R"], TOI465["Teff"], 0.0,
                       N=400, parallel=True)
        b = ml.lnZ_TTP(t, f, s, TOI465["P"], TOI465["M"], TOI465["R"], TOI465["Teff"], 0.0,
                       N=400, parallel=True)
        np.random.seed(3)
        np.random.rand(0)
    lnw = np.concatenate(mc_oracle.draws[-2:])
    merged = _merge_round(a, b, 400)
    fin = np.flatnonzero(np.isfinite(lnw))
    top = fin[np.lexsort((fin, -lnw[fin]))][:100]
    assert np.array_equal(merged.top[1], top)
    both = {k: np.concatenate([a[k][:len(a.top[0])], b[k][:len(b.top[0])]])
            for k in ml.RESULT_KEYS}
    src = {int(i): p for p, i in enumerate(np.r_[a.top[1], np.asarray(b.top[1]) + 400])}
    for k in ml.RESULT_KEYS:
        assert np.array_equal(merged[k][:top.size], both[k][[src[int(i)] for i in top]])
    assert merged.N == 800
    assert merged["lnZ"] == pytest.approx(nx._log_mean_exp(lnw, N_total=800), abs=1e-12)


@pytest.mark.parametrize("kw", [dict(fpp_err_target=0.0), dict(fpp_err_target=-1.0),
                                dict(fpp_err_target=float("nan")),
                                dict(fpp_err_target=float("inf")),
                                dict(mc_errors=True, N_max=100),
                                dict(fpp_err_target=0.01, N_max=299)])
def test_invalid_refinement_arguments_raise_before_any_draw(mc_oracle, toi465_lc, kw):
    mc_oracle.draws.clear()
    with pytest.raises(ValueError):
        _calc_probs(toi465_lc, **kw)
    assert mc_oracle.draws == []


# ---- two ranks over gloo (the pattern of test_dist_gloo.py) ----------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(out_path, sampler):
    import torch.distributed as dist
    dist.init_process_group("gloo")
    import _mc_oracle
    from triceratops_b200 import set_sampler
    _mc_oracle.install(_mc_oracle.MomentsOracleEngine())
    lc = load_lc("TOI465_01_lightcurve.csv")
    set_sampler(sampler, seed=5)
    tgt = _calc_probs(lc, mc_errors=True)
    raised = False
    try:
        _calc_probs(lc, fpp_err_target=0.01)
    except ValueError:
        raised = True
    with open(out_path + ".%d" % dist.get_rank(), "wb") as fh:
        pickle.dump(dict(lnZ=tgt.lnZ.copy(), lnZ_err=tgt.lnZ_err.copy(), FPP_err=tgt.FPP_err,
                         NFPP_err=tgt.NFPP_err, prob_err=tgt.probs.prob_err.values.copy(),
                         collectives=tgt.collectives, raised=raised), fh)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("sampler", ["host"])
def test_two_ranks_give_the_error_bars_of_one(tmp_path, mc_oracle, toi465_lc, sampler):
    from triceratops_b200 import set_sampler
    out = str(tmp_path / "res.pkl")
    port = _free_port()
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE="2",
                   MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), OMP_NUM_THREADS="2")
        procs.append(subprocess.Popen([sys.executable, os.path.abspath(__file__), out, sampler],
                                      env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    logs = [p.communicate(timeout=600)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    res = [pickle.load(open(out + ".%d" % r, "rb")) for r in range(2)]
    set_sampler(sampler, seed=5)
    try:
        one = _calc_probs(toi465_lc, mc_errors=True)
    finally:
        set_sampler("host")
    for r in res:
        assert r["raised"]
        assert r["collectives"]["record_exchanges"] == 1
        fin = np.isfinite(one.lnZ_err)
        assert np.array_equal(np.isfinite(r["lnZ_err"]), fin)
        if sampler == "host":
            # the same draws split over two ranks: the records merge to the same numbers
            np.testing.assert_allclose(r["lnZ_err"][fin], one.lnZ_err[fin], rtol=1e-9)
            assert r["FPP_err"] == pytest.approx(one.FPP_err, rel=1e-9)
            np.testing.assert_allclose(r["prob_err"], one.probs.prob_err.values, rtol=1e-9,
                                       atol=1e-15)
        assert np.isfinite(r["FPP_err"])
    assert np.array_equal(res[0]["lnZ_err"], res[1]["lnZ_err"], equal_nan=True)
    assert res[0]["FPP_err"] == res[1]["FPP_err"]


if __name__ == "__main__":
    _worker(sys.argv[1], sys.argv[2])
