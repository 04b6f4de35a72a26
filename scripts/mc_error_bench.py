"""Cost and quality of the Monte-Carlo error bars (DESIGN.md section 4e).  Three measurements
in one run, with the card's name and power limit read in the same run:

  (a) moment-pass cost: the 18-row TOI-465.01 table (bench.py config 2, N = 1e6 draws per
      scenario), recorded once from `target.calc_probs`' host side and replayed from HBM with
      moments off and on, the arms alternated; CUDA events around every step of 12 engine calls.
  (b) refinement: `calc_probs` on TOI-465.01 (config 2 inputs) at N = 1e5 with
      fpp_err_target = 0.01, host and device sampler: wall time, draws per row, achieved FPP_err;
      then again with a target of a quarter of that run's FPP_err, so that rounds run.
  (c) calibration: 32 seeds of calc_probs(mc_errors=True) at N = 1e5 (host sampler): the
      empirical standard deviation of FPP against the mean reported FPP_err; once with the
      curve's flux errors, once with them inflated 30-fold.
Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        return out.splitlines()[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def moment_cost(eng, draws, steps, warmup, seed):
    import torch
    import _workloads as wl
    lc = wl.lightcurve(2)
    calls, _ = wl.record_calls(2, draws, seed, lc)
    dev = torch.device("cuda", eng.device)
    work = []
    for c in calls:
        cols = {k: (torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64)).to(dev)
                    if np.size(v) > 1 else v)
                for k, v in c["cols"].items() if v is not None}
        mask = (torch.from_numpy(np.asarray(c["extra_mask"], bool)).to(dev)
                if c["extra_mask"] is not None else None)
        work.append((c, cols, mask))

    def step(on):
        eng.set_moments(on)
        pend = []
        for c, cols, mask in work:
            sub = eng.submit_tp_tensors if c["kind"] == "tp" else eng.submit_eb_tensors
            pend.append(sub(c["N"], cols, extra_mask=mask, companion_is_host=c["is_host"],
                            n_best=100, lightcurve=c["lc"]))
        out = []
        for p in pend:
            r = p.result()
            out += [(x.lnZ, x.s2) for x in (r if isinstance(r, tuple) else (r,))]
        return out

    for _ in range(warmup):
        for on in (False, True):
            step(on)
    ms = {False: [], True: []}
    last = {}
    for _ in range(steps):
        for on in (False, True):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            last[on] = step(on)
            e1.record()
            e1.synchronize()
            ms[on].append(e0.elapsed_time(e1))
    eng.set_moments(False)
    same = all(a[0] == b[0] for a, b in zip(last[False], last[True]))
    out = {"workload": "config 2, 18 rows, N = %d" % draws, "steps": steps, "warmup": warmup,
           "lnZ_identical": bool(same)}
    for on, name in ((False, "off"), (True, "on")):
        m = np.asarray(ms[on])
        out[name] = {"ms_mean": float(m.mean()), "ms_min": float(m.min()),
                     "ms_max": float(m.max())}
    out["on_over_off"] = out["on"]["ms_mean"] / out["off"]["ms_mean"]
    return out


def refinement(target_err, draws):
    import _workloads as wl
    from triceratops_b200 import set_sampler
    lc = wl.lightcurve(2)
    out = {}
    for sampler in ("host", "device"):
        set_sampler(sampler, seed=7)
        try:
            wl.run_calc_probs(wl.make_target(2), 2, lc, draws, 7, mc_errors=True)   # warm-up
            t0 = time.perf_counter()
            tgt = wl.run_calc_probs(wl.make_target(2), 2, lc, draws, 7,
                                    fpp_err_target=target_err)
            wall = time.perf_counter() - t0
            # a target below the first round's error, so that refinement rounds run
            tight = float(tgt.FPP_err) / 4
            t0 = time.perf_counter()
            ref = wl.run_calc_probs(wl.make_target(2), 2, lc, draws, 7, fpp_err_target=tight)
            wall_tight = time.perf_counter() - t0
        finally:
            set_sampler("host")
        out[sampler] = {"target": target_err, "wall_s": wall, "FPP": float(tgt.FPP),
                        "FPP_err": float(tgt.FPP_err),
                        "N_draws": [int(n) for n in tgt.N_draws],
                        "tight": {"target": tight, "wall_s": wall_tight, "FPP": float(ref.FPP),
                                  "FPP_err": float(ref.FPP_err),
                                  "N_draws": [int(n) for n in ref.N_draws]}}
    return out


def calibration(n_seeds, draws, err_scale=1.0):
    import _workloads as wl
    t, f, s = wl.lightcurve(2)
    lc = (t, f, err_scale * s)
    fpp, err = [], []
    for seed in range(n_seeds):
        tgt = wl.run_calc_probs(wl.make_target(2), 2, lc, draws, 100 + seed, mc_errors=True)
        fpp.append(float(tgt.FPP))
        err.append(float(tgt.FPP_err))
    return {"seeds": n_seeds, "N": draws, "flux_err_scale": err_scale, "FPP_mean": float(np.mean(fpp)),
            "FPP_std_empirical": float(np.std(fpp, ddof=1)),
            "FPP_err_mean_reported": float(np.mean(err)),
            "FPP_err_median_reported": float(np.median(err))}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--draws", type=int, default=1_000_000, help="N of measurement (a)")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--refine-draws", type=int, default=100_000)
    ap.add_argument("--target", type=float, default=0.01)
    ap.add_argument("--seeds", type=int, default=32)
    ap.add_argument("--only", choices=("a", "b", "c"), default=None)
    args = ap.parse_args()
    from triceratops_b200.engine import get_engine
    eng = get_engine()
    res = {"card": _card()}
    if args.only in (None, "a"):
        res["a_moment_cost"] = moment_cost(eng, args.draws, args.steps, args.warmup, args.seed)
    if args.only in (None, "b"):
        res["b_refinement"] = refinement(args.target, args.refine_draws)
    if args.only in (None, "c"):
        res["c_calibration"] = calibration(args.seeds, args.refine_draws)
        # the same with the flux errors inflated 30-fold: effective sample sizes in the
        # hundreds, where the delta method is expected to hold
        res["c_calibration_err_x30"] = calibration(args.seeds, args.refine_draws, 30.0)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
