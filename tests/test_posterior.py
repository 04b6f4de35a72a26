"""Posterior samples by systematic importance resampling, on the CPU: the uniform of
_numerics.posterior_uniform, the numpy mirror of the GPU resampler (tests/_post_oracle.py),
merge_posteriors, calc_probs(posterior_samples=K) on the posterior oracle, and a two-rank gloo
run."""
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


def _lnw(seed, N=3000, frac=0.3):
    rng = np.random.default_rng(seed)
    x = rng.normal(-3.0, 2.0, N)
    x[rng.random(N) > frac] = -np.inf
    return x


def _weights(lnw):
    fin = np.isfinite(lnw)
    return np.where(fin, np.exp(np.where(fin, lnw, 0.0) - lnw[fin].max()), 0.0)


# ---- the uniform and the resampler -----------------------------------------------------------
def test_posterior_uniform_is_deterministic_and_in_unit_interval():
    us = [nx.posterior_uniform(s, t, b) for s in range(20) for t in range(20) for b in range(3)]
    assert us == [nx.posterior_uniform(s, t, b) for s in range(20) for t in range(20)
                  for b in range(3)]
    assert all(0.0 <= u < 1.0 for u in us)
    assert len(set(us)) == len(us)
    assert nx.posterior_uniform(2 ** 64 - 1, 2 ** 63, 5) < 1.0
    # a known value: the kernel mirrors these bits
    h = nx._splitmix64(nx._splitmix64(nx._splitmix64(7) ^ 3) ^ 1)
    assert nx.posterior_uniform(7, 3, 1) == (h >> 11) / 2.0 ** 53


@pytest.mark.parametrize("K", [1, 7, 1000, 4096])
def test_resampler_copy_counts_are_floor_or_ceil(K):
    from _post_oracle import resample
    lnw = _lnw(K)
    w = _weights(lnw)
    idx, T = resample(lnw, K, nx.posterior_uniform(1, K, 0))
    assert idx.size == K and np.all(np.diff(idx) >= 0)
    assert T == pytest.approx(w.sum(), rel=1e-12)
    counts = np.bincount(idx, minlength=lnw.size)
    want = K * w / T
    assert np.all(counts >= np.floor(want - 1e-9)) and np.all(counts <= np.ceil(want + 1e-9))
    assert np.all(counts[w == 0] == 0)


def test_resampler_empty_posteriors():
    from _post_oracle import resample
    idx, T = resample(np.r_[0.0, np.inf, -1.0], 10, 0.5)
    assert idx.size == 0 and T == np.inf
    idx, T = resample(np.full(5, -np.inf), 10, 0.5)
    assert idx.size == 0 and T == 0.0
    idx, T = resample(np.r_[np.nan, -np.inf, 2.0, np.nan], 5, 0.99)
    assert np.array_equal(idx, np.full(5, 2))


# ---- merging slices ------------------------------------------------------------------------
def _slices(lnw, cuts, K, seed, stream):
    from _post_oracle import resample
    parts, lo = [], 0
    for hi in list(cuts) + [lnw.size]:
        x = lnw[lo:hi]
        idx, T = resample(x, K, nx.posterior_uniform(seed, stream, 0))
        m = x[np.isfinite(x)].max() if np.isfinite(x).any() else -np.inf
        parts.append((m, T, idx + lo))
        lo = hi
    return parts


def test_merge_of_one_slice_is_the_identity():
    parts = _slices(_lnw(3), [], 500, 1, 2)
    idx, m, W = nx.merge_posteriors(parts, 500, 1, 2)
    assert np.array_equal(idx, parts[0][2]) and W == parts[0][1]


def test_merge_allocates_floor_or_ceil_per_slice():
    lnw = _lnw(4, N=4000)
    K = 999
    for stream in range(20):
        parts = _slices(lnw, [700, 2100, 3000], K, 9, stream)
        idx, m, W = nx.merge_posteriors(parts, K, 9, stream)
        assert idx.size == K and np.all(np.diff(idx) >= 0)
        Wr = np.array([T * np.exp(mm - m) for mm, T, _ in parts])
        assert W == pytest.approx(Wr.sum(), rel=1e-12)
        c = np.histogram(idx, bins=[0, 700, 2100, 3000, 4000])[0]
        want = K * Wr / W
        assert np.all(c >= np.floor(want - 1e-9)) and np.all(c <= np.ceil(want + 1e-9))
        for r, (_, _, pidx) in enumerate(parts):   # samples come from the slice's own
            assert np.isin(idx[(idx >= [0, 700, 2100, 3000][r])
                               & (idx < [700, 2100, 3000, 4000][r])], pidx).all()


def test_merge_is_unbiased():
    lnw = _lnw(5, N=40, frac=0.8)
    w = _weights(lnw)
    K, reps = 16, 2500
    counts = np.zeros((reps, lnw.size))
    for s in range(reps):
        parts = _slices(lnw, [13, 25], K, s, 77)
        idx, _, _ = nx.merge_posteriors(parts, K, s, 77)
        counts[s] = np.bincount(idx, minlength=lnw.size)
    mean, sd = counts.mean(0), counts.std(0, ddof=1)
    want = K * w / w.sum()
    se = np.maximum(sd, 1e-3) / np.sqrt(reps)
    assert np.all(np.abs(mean - want) <= 4 * se + 1e-12)


def test_merge_edge_cases():
    a = (0.0, 3.0, np.arange(4))
    assert nx.merge_posteriors([a, (1.0, np.inf, np.zeros(0, np.int64))], 4, 0, 0)[0].size == 0
    idx, _, W = nx.merge_posteriors([(-np.inf, 0.0, np.zeros(0, np.int64))] * 2, 4, 0, 0)
    assert idx.size == 0 and W == 0.0
    assert nx.merge_posteriors([a, (0.0, 1.0, None)], 4, 0, 0)[0] is None
    # an empty slice takes no samples, the other one keeps all of them
    idx, _, _ = nx.merge_posteriors([(-np.inf, 0.0, np.zeros(0, np.int64)), a], 4, 0, 0)
    assert np.array_equal(idx, np.arange(4))


# ---- calc_probs on the posterior oracle -----------------------------------------------------
_DROP = ["PTP", "PEB", "STP", "SEB", "DTP", "DEB", "BTP"]


@pytest.fixture()
def post_oracle():
    import _post_oracle
    from oracle.engine_port import uninstall
    eng = _post_oracle.install(_post_oracle.PosteriorOracleEngine())
    yield eng
    uninstall()


def _target():
    from triceratops_b200 import synthetic as synth
    from triceratops_b200.triceratops import target
    stars = synth.stars_table(9, TOI465["T"], TOI465["J"], TOI465["H"], TOI465["K"], TOI465["M"],
                              TOI465["R"], TOI465["Teff"], TOI465["plx"], n_neighbours=1)
    return target(9, stars=stars, trilegal_fname=os.path.join(ROOT, "tests", "golden",
                                                              "trilegal_synth.csv"))


def _calc_probs(lc, N=300, seed=11, **kw):
    t, f, s = lc
    tgt = _target()
    np.random.seed(seed)
    tgt.calc_probs(t, f, 10 * s, TOI465["P"], N=N, parallel=True, verbose=0,
                   drop_scenario=_DROP, **kw)
    tgt.rng_state = np.random.get_state()
    return tgt


def _same_state(a, b):
    return a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2:] == b[2:]


def test_posterior_leaves_the_results_bit_identical(post_oracle, toi465_lc):
    plain = _calc_probs(toi465_lc)
    assert plain.posterior is None
    post = _calc_probs(toi465_lc, posterior_samples=200, posterior_seed=4)
    assert np.array_equal(plain.lnZ, post.lnZ)
    assert plain.FPP == post.FPP and plain.NFPP == post.NFPP
    assert plain.probs.equals(post.probs)
    for k in ("u1", "u2", "fluxratio_EB", "fluxratio_comp"):
        assert np.array_equal(getattr(plain, k), getattr(post, k))
    assert _same_state(plain.rng_state, post.rng_state)
    P = post.posterior
    assert list(P.columns[:4]) == ["ID", "scenario", "row", "draw"]
    assert set(["M_s", "R_s", "P_orb", "inc", "b", "ecc", "w", "R_p", "M_EB", "R_EB", "u1",
                "u2", "fluxratio_EB", "fluxratio_comp"]) <= set(P.columns)
    # one block of K rows per row with a non-empty posterior, ascending draws within a block
    for j, blk in P.groupby("row"):
        assert len(blk) == 200 and np.all(np.diff(blk.draw.values) >= 0)
        assert (blk.scenario == post.probs.scenario[j]).all()
    assert set(P.row) == {j for j in range(len(post.lnZ)) if np.isfinite(post.lnZ[j])}


def test_posterior_rows_are_the_draws_of_the_scenario(post_oracle, toi465_lc):
    """Each posterior row equals the scenario's own columns at `draw`: the same lnZ_* call
    made directly gives its best-draw table from the same columns, and its rows at the
    posterior draws must match."""
    from triceratops_b200 import _dispatch, posterior_samples
    from triceratops_b200 import marginal_likelihoods as ml
    from _post_oracle import resample
    t, f, s = toi465_lc
    s = 10 * s
    _dispatch.use_lightcurve(t, f, s, 0.00139, 20)
    np.random.seed(3)
    with posterior_samples(300, seed=8):
        tp = ml.lnZ_TTP(t, f, s, TOI465["P"], TOI465["M"], TOI465["R"], TOI465["Teff"], 0.0,
                        N=500, parallel=True)
        eb, ebx2 = ml.lnZ_TEB(t, f, s, TOI465["P"], TOI465["M"], TOI465["R"], TOI465["Teff"],
                              0.0, N=500, parallel=True)
    lnw_tp, lnw_eb, lnw_x2 = post_oracle.draws[-3:]
    for res, lnw, stream, b in ((tp, lnw_tp, 0, 0), (eb, lnw_eb, 1, 0), (ebx2, lnw_x2, 1, 1)):
        idx, T = resample(lnw, 300, nx.posterior_uniform(8, stream, b))
        assert np.array_equal(res.posterior["draw"], idx) and res.post_total == T
    # rows: the best-draw table holds rows of the same columns; every posterior sample that
    # is one of its draws carries that draw's row in every key
    hits = 0
    for res in (tp, eb, ebx2):
        assert len(res.posterior["draw"]) == (300 if np.isfinite(res["lnZ"]) else 0)
        where = {int(i): p for p, i in enumerate(res.top[1])}
        for q, d in enumerate(res.posterior["draw"]):
            if int(d) in where:
                hits += 1
                for k in ml.RESULT_KEYS:
                    assert res.posterior[k][q] == res[k][where[int(d)]], k
    assert hits > 0


def test_another_seed_gives_another_sample(post_oracle, toi465_lc):
    a = _calc_probs(toi465_lc, posterior_samples=100, posterior_seed=1)
    b = _calc_probs(toi465_lc, posterior_samples=100, posterior_seed=1)
    c = _calc_probs(toi465_lc, posterior_samples=100, posterior_seed=2)
    assert a.posterior.equals(b.posterior)
    assert not np.array_equal(a.posterior.draw.values, c.posterior.draw.values)
    assert np.array_equal(a.lnZ, c.lnZ)


def test_refinement_merges_the_posteriors(post_oracle, toi465_lc):
    from _post_oracle import resample
    post_oracle.posts.clear()
    tgt = _calc_probs(toi465_lc, fpp_err_target=1e-9, N_max=1200, posterior_samples=150)
    ref = _calc_probs(toi465_lc, fpp_err_target=1e-9, N_max=1200)
    assert np.array_equal(tgt.lnZ, ref.lnZ) and tgt.FPP_err == ref.FPP_err
    assert tgt.probs.equals(ref.probs)
    rows_of_call = [[0], [1, 2], [13, 14], [15], [16, 17]]
    by_key = {}
    for key, lnw in post_oracle.calls:
        by_key.setdefault(key, []).append(lnw)
    by_key = list(by_key.values())[:len(rows_of_call)]
    refined = 0
    for rows, parts in zip(rows_of_call, by_key):
        for b, j in enumerate(rows):
            blk = tgt.posterior[tgt.posterior.row == j]
            if not np.isfinite(tgt.lnZ[j]):
                assert len(blk) == 0
                continue
            assert len(blk) == 150 and blk.draw.max() < tgt.N_draws[j]
            if len(parts) > 1 and tgt.N_draws[j] > 300:
                refined += 1
                # the merged sample covers the later rounds' draws too, and only draws of
                # positive weight
                lnw = np.concatenate([p[b] for p in parts])[:tgt.N_draws[j]]
                assert np.all(np.isfinite(lnw[blk.draw.values]))
            else:
                idx, _ = resample(parts[0][b], 150, nx.posterior_uniform(0, rows[0], b))
                assert np.array_equal(blk.draw.values, idx)
    assert refined > 0


@pytest.mark.parametrize("kw", [dict(posterior_samples=0), dict(posterior_samples=-3),
                                dict(posterior_samples=2.5), dict(posterior_samples="10"),
                                dict(posterior_samples=True),
                                dict(posterior_samples=(1 << 20) + 1),
                                dict(posterior_samples=10, posterior_seed=1.5)])
def test_invalid_posterior_arguments_raise_before_any_draw(post_oracle, toi465_lc, kw):
    post_oracle.draws.clear()
    state = np.random.get_state()
    with pytest.raises(ValueError):
        _target().calc_probs(*toi465_lc, TOI465["P"], N=300, verbose=0, drop_scenario=_DROP,
                             **kw)
    assert post_oracle.draws == []
    assert _same_state(state, np.random.get_state())


# ---- two ranks over gloo --------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(out_path):
    import torch.distributed as dist
    dist.init_process_group("gloo")
    import _post_oracle
    _post_oracle.install(_post_oracle.PosteriorOracleEngine())
    lc = load_lc("TOI465_01_lightcurve.csv")
    tgt = _calc_probs(lc, posterior_samples=120, posterior_seed=6)
    with open(out_path + ".%d" % dist.get_rank(), "wb") as fh:
        pickle.dump(dict(lnZ=tgt.lnZ.copy(), posterior=tgt.posterior,
                         collectives=tgt.collectives), fh)
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_hold_the_same_posterior(tmp_path, post_oracle, toi465_lc):
    out = str(tmp_path / "res.pkl")
    port = _free_port()
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE="2",
                   MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), OMP_NUM_THREADS="2")
        procs.append(subprocess.Popen([sys.executable, os.path.abspath(__file__), out],
                                      env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    logs = [p.communicate(timeout=600)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    res = [pickle.load(open(out + ".%d" % r, "rb")) for r in range(2)]
    one = _calc_probs(toi465_lc, posterior_samples=120, posterior_seed=6)
    for r in res:
        assert r["collectives"]["record_exchanges"] == 1
        np.testing.assert_allclose(r["lnZ"], one.lnZ, rtol=1e-12)
        P = r["posterior"]
        assert set(P.row) == set(one.posterior.row)
        for j, blk in P.groupby("row"):
            assert len(blk) == 120 and np.all(np.diff(blk.draw.values) >= 0)
            assert blk.draw.max() < 300
    assert res[0]["posterior"].equals(res[1]["posterior"])


if __name__ == "__main__":
    _worker(sys.argv[1])
