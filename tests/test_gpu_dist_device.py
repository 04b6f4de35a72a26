"""The device sampler on two ranks: two gloo processes share one GPU, each draws and evaluates
its own contiguous half of every scenario's draws, and calc_probs merges the halves with its one
exchange of records.  A draw's Philox stream depends on its global index only, so the union of
the halves is the one-process sample: evidences, error bars and the best-draw tables must equal
the one-process run."""
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

N = 200_001           # odd on purpose: ragged halves
SEED = 41
K = 500
_TABLE = ("M_s", "R_s", "P_orb", "inc", "b", "ecc", "w", "R_p", "M_EB", "R_EB")


def _run():
    from _workloads import lightcurve, make_target, run_calc_probs
    from triceratops_b200 import set_sampler
    set_sampler("device", seed=SEED)
    try:
        tgt = run_calc_probs(make_target(2), 2, lightcurve(2), N, 7, mc_errors=True,
                             posterior_samples=K, posterior_seed=3)
    finally:
        set_sampler("host")
    return dict(lnZ=tgt.lnZ.copy(), lnZ_err=tgt.lnZ_err.copy(), FPP=tgt.FPP, NFPP=tgt.NFPP,
                FPP_err=tgt.FPP_err, table={c: tgt.probs[c].values.copy() for c in _TABLE},
                u1=np.array(tgt.u1), u2=np.array(tgt.u2),
                fluxratio_EB=np.array(tgt.fluxratio_EB),
                fluxratio_comp=np.array(tgt.fluxratio_comp),
                post_row=tgt.posterior.row.values.copy(),
                post_draw=tgt.posterior.draw.values.copy(), collectives=tgt.collectives)


def _worker(out_path):
    import torch.distributed as dist
    dist.init_process_group("gloo")
    res = _run()
    with open(out_path + ".%d" % dist.get_rank(), "wb") as fh:
        pickle.dump(res, fh)
    dist.barrier()
    dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.gpu
def test_two_ranks_equal_one(tmp_path, gpu_engine):
    out = str(tmp_path / "res.pkl")
    port = _free_port()
    procs = []
    for rank in range(2):
        # both processes on the one GPU of the test (LOCAL_RANK picks the engine's device)
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK="0", WORLD_SIZE="2",
                   MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), OMP_NUM_THREADS="2")
        procs.append(subprocess.Popen([sys.executable, os.path.abspath(__file__), out],
                                      env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    try:
        logs = [p.communicate(timeout=900)[0].decode() for p in procs]
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
                p.wait()
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    res = [pickle.load(open(out + ".%d" % r, "rb")) for r in range(2)]
    try:
        one = _run()
    finally:     # (calc_probs leaves the engine's switches as its last call set them)
        gpu_engine.set_moments(False)
        gpu_engine.set_posterior(0)

    a, b = res
    for key in ("lnZ", "lnZ_err", "u1", "u2", "fluxratio_EB", "fluxratio_comp", "post_row",
                "post_draw"):
        assert np.array_equal(a[key], b[key], equal_nan=True), key
    for c in _TABLE:
        assert np.array_equal(a["table"][c], b["table"][c], equal_nan=True), c
    assert (a["FPP"], a["NFPP"], a["FPP_err"]) == (b["FPP"], b["NFPP"], b["FPP_err"])

    assert one["collectives"] is None
    fin = np.isfinite(one["lnZ"])
    assert fin.sum() >= 3
    for r in res:
        assert r["collectives"]["record_exchanges"] == 1
        assert np.array_equal(np.isfinite(r["lnZ"]), fin)
        np.testing.assert_allclose(r["lnZ"][fin], one["lnZ"][fin], rtol=0, atol=1e-9)
        efin = np.isfinite(one["lnZ_err"])
        assert np.array_equal(np.isfinite(r["lnZ_err"]), efin)
        np.testing.assert_allclose(r["lnZ_err"][efin], one["lnZ_err"][efin], rtol=0, atol=1e-9)
        # the best draw of every row with a finite evidence: the same draw, the same bits
        for c in _TABLE:
            assert np.array_equal(r["table"][c][fin], one["table"][c][fin], equal_nan=True), c
        for key in ("u1", "u2", "fluxratio_EB", "fluxratio_comp"):
            assert np.array_equal(r[key][fin], one[key][fin], equal_nan=True), key
        assert len(r["post_draw"]) and np.all((0 <= r["post_draw"]) & (r["post_draw"] < N))
        assert sorted(set(r["post_row"])) == sorted(set(one["post_row"]))


if __name__ == "__main__":
    _worker(sys.argv[1])
