"""Mixed-cadence throughput on the headline workload (DESIGN.md section 4d).

The 18-row TOI-465.01 table (bench.py config 2: 858-stamp folded curve, N = 1e6 draws per
scenario) is recorded once from `target.calc_probs`' host side (tests/_workloads.py).  Each
engine call's light curve then gets a second cadence group: the same folded curve binned to
30 min, exptime 0.02083 d, nsamples 20 (tests/_cadence_oracle.mixed_lightcurve).  Two arms are
timed alternately in one process, inputs resident in HBM, CUDA events around every step of
12 engine calls (18 rows):

  mixed   the two-group light curve on the segmented kernel (lnl_seg_kernel)
  forced  the same stamps forced to one cadence (0.00139 d, 20): today's workaround

model_points_per_s = 18 * N * sum_g(npts_g * nsamples_g) / step time.  This counts sub-exposure
evaluations the model asks for; it is NOT bench.py's samples*points/s (18 * N * npts / time).
Prints one JSON line; the card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

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


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--draws", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=5, help="timed steps per arm")
    ap.add_argument("--warmup", type=int, default=1, help="untimed steps per arm")
    ap.add_argument("--seed", type=int, default=2024)
    args = ap.parse_args()
    import torch
    import _workloads as wl
    from _cadence_oracle import mixed_lightcurve
    from triceratops_b200.engine import get_engine

    lc = wl.lightcurve(2)
    calls, _ = wl.record_calls(2, args.draws, args.seed, lc)
    eng = get_engine()
    dev = torch.device("cuda", eng.device)
    work = []
    for c in calls:
        cols = {k: (torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64)).to(dev)
                    if np.size(v) > 1 else v)
                for k, v in c["cols"].items() if v is not None}
        mask = (torch.from_numpy(np.asarray(c["extra_mask"], bool)).to(dev)
                if c["extra_mask"] is not None else None)
        t, f, s = c["lc"][:3]
        time, flux, exptime, nsamples = mixed_lightcurve(t, f)
        arms = {"mixed": (time, flux, s, exptime, nsamples),
                "forced": (time, flux, s, 0.00139, 20)}
        work.append((c, cols, mask, arms))
    t0, f0 = lc[:2]
    time, _, exptime, nsamples = mixed_lightcurve(t0, f0)
    pts = {"mixed": int(np.sum(nsamples.astype(np.int64))),   # sum_g npts_g * ns_g
           "forced": int(time.size * 20)}
    n_groups = len(set(zip(exptime.tolist(), nsamples.tolist())))

    def step(arm):
        pend = []
        for c, cols, mask, arms in work:
            sub = eng.submit_tp_tensors if c["kind"] == "tp" else eng.submit_eb_tensors
            pend.append(sub(c["N"], cols, extra_mask=mask, companion_is_host=c["is_host"],
                            n_best=100, lightcurve=arms[arm]))
        out = []
        for p in pend:
            r = p.result()
            out += [x.lnZ for x in (r if isinstance(r, tuple) else (r,))]
        return out

    for _ in range(args.warmup):
        for arm in ("mixed", "forced"):
            step(arm)
    ms = {"mixed": [], "forced": []}
    lnZ = {}
    for _ in range(args.steps):
        for arm in ("mixed", "forced"):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            lnZ[arm] = step(arm)
            e1.record()
            e1.synchronize()
            ms[arm].append(e0.elapsed_time(e1))
    res = {"card": _card(), "workload": "config 2 (18 rows, N = %d) + 30-min binned copy"
           % args.draws, "stamps": int(time.size), "cadence_groups": n_groups,
           "steps": args.steps, "warmup": args.warmup}
    for arm in ("mixed", "forced"):
        m = np.asarray(ms[arm])
        res[arm] = {"ms_per_step_mean": float(m.mean()), "ms_per_step_min": float(m.min()),
                    "ms_per_step_max": float(m.max()),
                    "model_points_per_s": 18 * args.draws * pts[arm] / (m.mean() * 1e-3),
                    "model_points_per_draw": pts[arm],
                    "finite_lnZ": int(np.isfinite(lnZ[arm]).sum())}
    res["mixed_over_forced_ms"] = res["mixed"]["ms_per_step_mean"] / res["forced"]["ms_per_step_mean"]
    print(json.dumps(res))


if __name__ == "__main__":
    main()
