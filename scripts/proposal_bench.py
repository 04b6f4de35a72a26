"""Adaptive importance sampling against prior sampling (DESIGN.md section 4g), with the card's
name and power limit read in the same run, on the config-2 inputs (TOI-465.01, 18 rows, device
sampler, mc_errors on):

  (a) per row: ess, lnZ_err and the survivors of the geometric mask of the final round, and the
      GPU time of one whole calc_probs (CUDA events; adaptive includes its pilots), for
      proposal="prior" and "adaptive" at the same N;
  (b) the spread of FPP over --seeds seeds for both arms at roughly equal GPU time (the prior
      arm gets N_prior = N * t_adaptive / t_prior draws, from the times of (a)), with the real
      flux errors and with them inflated 30x;
  (c) one pilot stage against two (the module constant _STAGES), at the same N.

Prints one JSON line; --out also writes it to a file.
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
    ap.add_argument("--seeds", type=int, default=16)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import _workloads as wl
    from triceratops_b200 import set_sampler
    from triceratops_b200 import triceratops as tr
    from triceratops_b200.engine import get_engine
    if not torch.cuda.is_available():
        raise SystemExit("proposal_bench.py measures on the GPU: no CUDA device")
    get_engine()
    t, f, s = wl.lightcurve(2)
    tgt = wl.make_target(2)

    def run(mode, N, seed, inflate=1.0):
        set_sampler("device", seed=seed)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        wl.run_calc_probs(tgt, 2, (t, f, inflate * s), N, 1, mc_errors=True, proposal=mode)
        e1.record()
        e1.synchronize()
        set_sampler("host")
        return tgt.FPP, tgt.FPP_err, tgt.lnZ.copy(), tgt.ess.copy(), tgt.lnZ_err.copy(), \
            e0.elapsed_time(e1)

    def survivors(mode, N, seed, inflate=1.0):
        """n_pass of every row of the final round (one more run, same seed)."""
        from triceratops_b200 import device_sampler as ds
        seen = []
        orig = ds._finished

        def spy(ex):
            out = orig(ex)
            seen.append(out.n_pass)
            return out
        ds._finished = spy
        try:
            run(mode, N, seed, inflate)
        finally:
            ds._finished = orig
        return seen[-18:]

    out = {"card": _card(), "workload": "config 2 (TOI-465.01, 18 rows, device sampler, "
           "mc_errors), N = %d per call" % args.draws, "note": "times: CUDA events around one "
           "whole calc_probs, host work included"}
    for mode in ("prior", "adaptive"):       # warm-up (module loads, tables, allocator)
        run(mode, args.draws, 99)
    # (a) per row, both flux-error levels
    times = {}
    for inflate in (1.0, 30.0):
        key = "errors_x%d" % inflate
        rows = {}
        for mode in ("prior", "adaptive"):
            ms = []
            for rep in range(3):
                fpp, fe, lnZ, ess, lerr, dt = run(mode, args.draws, 1 + rep, inflate)
                ms.append(dt)
            rows[mode] = dict(ms_per_calc_probs=ms, FPP=fpp, FPP_err=fe,
                              lnZ=lnZ.tolist(), ess=ess.tolist(), lnZ_err=lerr.tolist(),
                              n_pass=survivors(mode, args.draws, 1, inflate))
            times[(inflate, mode)] = float(np.median(ms))
        r_ess = np.array(rows["adaptive"]["ess"]) / np.maximum(np.array(rows["prior"]["ess"]),
                                                                1e-300)
        fin = np.isfinite(rows["prior"]["lnZ"])
        rows["median_ess_ratio_equal_N"] = float(np.median(r_ess[fin]))
        rows["median_ess_per_gpu_second_ratio"] = float(
            np.median(r_ess[fin]) * times[(inflate, "prior")] / times[(inflate, "adaptive")])
        out["a_" + key] = rows
    # (b) FPP spread over seeds at about equal GPU time
    for inflate in (1.0, 30.0):
        key = "errors_x%d" % inflate
        N_prior = int(round(args.draws * times[(inflate, "adaptive")]
                            / times[(inflate, "prior")] / 1000.0)) * 1000
        res = {}
        for mode, N in (("prior", N_prior), ("adaptive", args.draws)):
            fpps, ms = [], []
            for sd in range(args.seeds):
                fpp, _, _, _, _, dt = run(mode, N, 1000 + sd, inflate)
                fpps.append(fpp)
                ms.append(dt)
            res[mode] = dict(N=N, FPP=fpps, FPP_mean=float(np.mean(fpps)),
                             FPP_std=float(np.std(fpps, ddof=1)), ms_median=float(np.median(ms)))
        out["b_" + key] = res
    # (c) one pilot stage against two, at the same N, inflated errors (ess in the hundreds)
    res = {}
    for stages in (1, 2):
        tr._STAGES = stages
        fpps, ess, ms = [], [], []
        for sd in range(args.seeds // 2):
            fpp, _, lnZ, e, _, dt = run("adaptive", args.draws, 2000 + sd, 30.0)
            fpps.append(fpp)
            ess.append(e[np.isfinite(lnZ)])
            ms.append(dt)
        res["stages=%d" % stages] = dict(
            FPP_std=float(np.std(fpps, ddof=1)), median_ess=float(np.median(np.stack(ess))),
            ms_median=float(np.median(ms)))
    tr._STAGES = 2
    out["c_stages_errors_x30"] = res
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
