"""The four submission entry points, tri_submit_tp / tri_submit_eb (host buffers) and
tri_submit_tp_dev / tri_submit_eb_dev (device pointers), run the same checks: host and device
columns give the same answers, bad arguments are rejected before anything is queued and leak no
slot, an N = 0 call takes the moment and posterior switches of its submission, and the launch
count follows the switches."""
import ctypes
import math

import numpy as np
import pytest

from conftest import draw_eb_columns, draw_tp_columns
from triceratops_b200 import _cabi
from triceratops_b200._cabi import tri_col, tri_eb_args, tri_result, tri_tp_args

pytestmark = pytest.mark.gpu

KINDS = ("tp", "eb")
PATHS = ("host", "dev")


@pytest.fixture()
def eng(gpu_engine, toi465_lc):
    t, f, s = toi465_lc
    gpu_engine.set_lightcurve(t, f, s, 0.00139, 20)
    yield gpu_engine
    gpu_engine.set_moments(False)
    gpu_engine.set_posterior(0)


def _columns(kind, N, seed):
    return draw_tp_columns(N, seed) if kind == "tp" else draw_eb_columns(N, seed)


def _tensors(eng, cols):
    import torch
    dev = torch.device("cuda", eng.device)
    return {k: torch.as_tensor(v, dtype=torch.float64, device=dev) for k, v in cols.items()}


def _eval(eng, kind, path, N, cols, **kw):
    """One evaluation through the entry point of (kind, path); a list of its branches."""
    if path == "host":
        fn = eng.eval_tp if kind == "tp" else eng.eval_eb
        out = fn(N, **cols, n_best=100, want_lnL=False, **kw)
    else:
        fn = eng.eval_tp_tensors if kind == "tp" else eng.eval_eb_tensors
        out = fn(N, _tensors(eng, cols), n_best=100, **kw)
    return [out] if kind == "tp" else list(out)


@pytest.mark.parametrize("kind,scalar_loop", [("tp", False), ("eb", False), ("eb", True)])
def test_host_and_device_pointer_calls_agree(eng, kind, scalar_loop):
    import torch
    N = 100_000
    cols = _columns(kind, N, 31)
    rng = np.random.default_rng(32)
    cols["lnprior"] = rng.normal(-4.0, 1.5, N)
    mask = rng.random(N) < 0.9
    kw = {"scalar_loop": scalar_loop} if kind == "eb" else {}
    host = _eval(eng, kind, "host", N, cols, extra_mask=mask, **kw)
    dmask = torch.as_tensor(mask, device=torch.device("cuda", eng.device))
    dev = _eval(eng, kind, "dev", N, cols, extra_mask=dmask, **kw)
    for h, d in zip(host, dev):
        assert h.n_finite > 0
        # the evidence's scaled sum is merged in the order the blocks took their draws, so its
        # last bits may differ between two runs (tri_result in include/triceratops_b200.h)
        assert d.lnZ == pytest.approx(h.lnZ, rel=1e-14) and d.s == pytest.approx(h.s, rel=1e-14)
        assert (d.m, d.n_finite, d.n_pass, d.n_evaluated) == (h.m, h.n_finite, h.n_pass,
                                                              h.n_evaluated)
        np.testing.assert_array_equal(d.top_idx, h.top_idx)
        np.testing.assert_array_equal(d.top_lnL, h.top_lnL)


def _raw_args(eng, kind, path, N, keep):
    """ctypes arguments of one (kind, path) call over N draws, buffers referenced by `keep`."""
    cols = _columns(kind, N, 41)
    a = tri_tp_args() if kind == "tp" else tri_eb_args()
    a.N = N
    for name, val in cols.items():
        arr = np.array(np.broadcast_to(np.asarray(val, float), (N,)))
        if path == "dev":
            arr = _tensors(eng, {name: arr})[name]
            ptr = arr.data_ptr()
        else:
            ptr = arr.ctypes.data
        keep.append(arr)
        setattr(a, name, tri_col(ptr, 1))
    want = (tri_result * (1 if kind == "tp" else 2))()
    return a, want


def _submit_raw(eng, kind, path, a, want, ticket):
    import torch
    fn = getattr(eng.lib, "tri_submit_%s%s" % (kind, "_dev" if path == "dev" else ""))
    tk = ctypes.byref(ticket) if ticket is not None else None
    if path == "dev":
        stream = torch.cuda.current_stream(torch.device("cuda", eng.device)).cuda_stream
        return fn(ctypes.byref(a), want, ctypes.c_void_p(stream), tk)
    return fn(ctypes.byref(a), want, tk)


def test_bad_arguments_are_rejected_and_leak_no_slot(eng):
    eng.drain()
    N, keep = 4000, []
    calls = [(k, p) + _raw_args(eng, k, p, N, keep) for k in KINDS for p in PATHS]
    tk = ctypes.c_int64()
    for kind, path, a, want in calls:
        required = "q" if kind == "eb" else "rp"   # (q: a column only EB-type calls have)
        for field, bad in ((required, tri_col(None, 1)), ("inc", tri_col(a.inc.ptr, 2))):
            good = tri_col(getattr(a, field).ptr, getattr(a, field).stride)   # (not a view)
            setattr(a, field, bad)
            assert _submit_raw(eng, kind, path, a, want, tk) == _cabi.TRI_EINVAL, (kind, path)
            setattr(a, field, good)
        a.N = -1
        assert _submit_raw(eng, kind, path, a, want, tk) == _cabi.TRI_EINVAL, (kind, path)
        a.N = N
        assert _submit_raw(eng, kind, path, a, want, None) == _cabi.TRI_EINVAL, (kind, path)
    # every slot is still free: a full ring of submissions goes through
    tickets = []
    for i in range(_cabi.TRI_MAX_INFLIGHT):
        kind, path, a, want = calls[i % len(calls)]
        t = ctypes.c_int64()
        _cabi.check(_submit_raw(eng, kind, path, a, want, t))
        tickets.append((t, want))
    kind, path, a, want = calls[0]
    assert _submit_raw(eng, kind, path, a, (tri_result * 2)(), tk) == _cabi.TRI_ESTATE
    for t, want in tickets:
        _cabi.check(eng.lib.tri_wait(t, want))
        assert want[0].n_finite > 0


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("kind", KINDS)
def test_empty_call_takes_the_switches_of_its_submission(eng, kind, path):
    # (one value per column: an empty tensor's data pointer is NULL)
    cols = {k: float(np.ravel(v)[0]) for k, v in _columns(kind, 1, 51).items()}
    eng.set_moments(True)
    eng.set_posterior(64, seed=3)
    for res in _eval(eng, kind, path, 0, cols):
        assert res.lnZ == -math.inf
        assert (res.n_finite, res.n_posinf, res.n_pass, res.n_stamps, res.n_interior,
                res.n_limb, res.n_evaluated) == (0,) * 7
        assert res.top_idx.size == 0
        assert res.s2 == 0.0
        assert res.post_idx.size == 0 and res.post_total == 0.0
    eng.set_moments(False)
    eng.set_posterior(0)
    out = _eval(eng, kind, path, 0, cols)
    s2 = (ctypes.c_double * 2)()
    _cabi.check(eng.lib.tri_last_moments(s2))
    for b, res in enumerate(out):
        assert res.lnZ == -math.inf and res.s2 is None and res.post_idx is None
        assert math.isnan(s2[b])


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("kind", KINDS)
def test_launch_count_follows_the_switches(eng, kind, path):
    N = 20_000
    cols = _columns(kind, N, 61)
    for moments, post_K, launches in ((False, 0, 3), (True, 0, 4), (False, 256, 5),
                                      (True, 256, 6)):
        eng.set_moments(moments)
        eng.set_posterior(post_K, seed=4)
        out = _eval(eng, kind, path, N, cols)
        assert eng.last_timing()["launches"] == launches, (moments, post_K)
        for res in out:
            assert (res.s2 is not None) == moments
            assert (res.post_idx is not None) == (post_K > 0)
