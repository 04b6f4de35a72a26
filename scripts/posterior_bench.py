"""Cost of the posterior samples (DESIGN.md section 4f), with the card's name and power limit
read in the same run: the 18-row TOI-465.01 table (bench.py config 2, N = 1e6 draws per
scenario), recorded once from `target.calc_probs`' host side and replayed from HBM with
posterior samples off, K = 1000 and K = 65536, the arms alternated; CUDA events around every
step.  Then one profiled step per arm (torch.profiler, CUDA activities) gives the own time of
posterior_sums_kernel and posterior_select_kernel.  Prints one JSON line.
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
    ap = argparse.ArgumentParser()
    ap.add_argument("--draws", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    import torch
    import _workloads as wl
    from triceratops_b200.engine import get_engine
    if not torch.cuda.is_available():
        raise SystemExit("posterior_bench.py measures on the GPU: no CUDA device")
    eng = get_engine()
    lc = wl.lightcurve(2)
    calls, _ = wl.record_calls(2, args.draws, args.seed, lc)
    dev = torch.device("cuda", eng.device)
    work = []
    for c in calls:
        cols = {k: (torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64)).to(dev)
                    if np.size(v) > 1 else v)
                for k, v in c["cols"].items() if v is not None}
        mask = (torch.from_numpy(np.asarray(c["extra_mask"], bool)).to(dev)
                if c["extra_mask"] is not None else None)
        work.append((c, cols, mask))

    def step(K):
        eng.set_posterior(K, seed=1)
        pend = []
        for i, (c, cols, mask) in enumerate(work):
            sub = eng.submit_tp_tensors if c["kind"] == "tp" else eng.submit_eb_tensors
            pend.append(sub(c["N"], cols, extra_mask=mask, companion_is_host=c["is_host"],
                            n_best=100, lightcurve=c["lc"], post_stream=i))
        out = []
        for p in pend:
            r = p.result()
            out += [(x.lnZ, x.post_idx) for x in (r if isinstance(r, tuple) else (r,))]
        return out

    arms = (0, 1000, 65536)
    for _ in range(args.warmup):
        for K in arms:
            step(K)
    ms = {K: [] for K in arms}
    last = {}
    for _ in range(args.steps):
        for K in arms:
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            last[K] = step(K)
            e1.record()
            e1.synchronize()
            ms[K].append(e0.elapsed_time(e1))
    kern = {}
    from torch.profiler import ProfilerActivity, profile
    for K in arms[1:]:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step(K)
            torch.cuda.synchronize()
        tot = {}
        for ev in prof.key_averages():
            if "posterior_" in ev.key:
                name = "sums" if "sums" in ev.key else "select"
                tot[name] = tot.get(name, 0.0) + ev.self_device_time_total / 1000.0
        kern[str(K)] = tot
    eng.set_posterior(0)
    same = all(a[0] == b[0] for K in arms[1:] for a, b in zip(last[0], last[K]))
    out = {"card": _card(), "workload": "config 2, 18 rows, N = %d, inputs in HBM" % args.draws,
           "steps": args.steps, "warmup": args.warmup, "lnZ_identical": bool(same),
           "kernel_ms_per_step": kern}
    for K in arms:
        m = np.asarray(ms[K])
        out["K=%d" % K] = {"ms_mean": float(m.mean()), "ms_min": float(m.min()),
                           "ms_max": float(m.max())}
    for K in arms[1:]:
        out["K=%d_over_off" % K] = out["K=%d" % K]["ms_mean"] / out["K=0"]["ms_mean"]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
