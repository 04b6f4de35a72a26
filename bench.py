#!/usr/bin/env python
"""bench.py -- headline benchmark of the marginal-likelihood path (BASELINE.json):
calc_probs samples*points/sec, 18 scenarios, N = 1e6 prior draws per scenario.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--config 2|3|4] [--draws N] [--scaling weak|strong] [--dump-outputs DIR]

One "step" is one pass of the hot path over one batch of synthetic input: the 12 engine calls
(6 TP-type, 6 EB-type) that a full 18-row `target.calc_probs` makes -- 15 target-star rows + NTP,
NEB, NEBx2P of one nearby star.  --config selects BASELINE.json's configuration (default 2 =
configs[1], the one the metric is quoted on: TOI-465.01, 858 stamps; 3 = Kepler-10b with 29.4-min
exposures; 4 = the 20 000-stamp synthetic light curve, N = 1e7).  Contrast curve
TOI465_01_contrastcurve.csv, synthetic stars table and synthetic TRILEGAL population (no
MAST/Gaia/TRILEGAL offline).  The prior draws are made on the host by the package's own lnZ_*
code (numpy seed), exactly as `calc_probs` makes them.

  value    : 18 * N * npts / t, inputs already resident in HBM, through tri_eval_*_dev on the
             torch stream, timed with CUDA events (max over ranks).
  e2e      : the same metric through the PUBLIC call, `target.calc_probs(...)`: host prior draws
             (numpy generator, the reference's order), transforms, host->device copies, kernels,
             result tables.  `e2e.engine` is the C-ABI-only part of it (tri_submit_* / tri_wait
             on pinned host columns, draws already made).
  roofline : FP64-issue roofline of the dominant kernel (lnl_kernel), see DESIGN.md.
  parity   : the north_star gates evaluated on the timed inputs, outside the timed region
             (tests/_parity.py): masks of all N draws, lnL of a seeded subset against the C
             oracle, device lnZ against the host log-mean-exp, probabilities.
  cpu_baseline / --impl reference: the same public call routed to the oracle port (C
             restatement + numpy masks, all host cores) on a bounded number of draws.

--steps K times K steps in every GPU leg (value, e2e.engine, e2e, e2e.device_sampler).

--dump-outputs DIR: after the timed steps, rank 0 writes what its last timed step returned as
float64 DIR/<name>.npy (a few kB in all), so that two builds can be compared output for output on
the same seeded inputs:
  lnZ, records, top_lnL, top_idx   the `value` leg: per scenario branch (engine-call order, TP
             one branch, EB two) the evidence, its (m, s, n_finite, n_posinf, n_pass) record and
             the 100 best draws (sorted best first, ties by index; NaN / -1 past n_top)
  e2e_lnZ, e2e_prob, e2e_best, e2e_fpp_nfpp   the `e2e` leg (calc_probs): the 18 rows' lnZ and
             probabilities, their best-draw table (columns E2E_BEST_COLUMNS) and (FPP, NFPP);
             absent with --kernel-only

N > 1 (torchrun, one rank per GPU): --scaling weak (default): every rank evaluates its own N
draws per scenario (different seed per rank); --scaling strong: N draws in total, sharded.  One
NCCL all-gather per step merges the per-scenario (max, scaled-sum) records (the package's own
`_dispatch.gather_records`).
"""
import argparse
import collections
import contextlib
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

N_ROWS = 18            # scenario rows of the configuration
N_BEST = 100           # best draws returned per row (marginal_likelihoods.py:152)
SEED = 2026
METRIC = "calc_probs samples*points/sec (18 scenarios, N=1e6)"
E2E_BEST_COLUMNS = ("M_s", "R_s", "P_orb", "inc", "b", "ecc", "w", "R_p", "M_EB", "R_EB")
DUMP_LIMIT_BYTES = 64 << 20

# FP64 issue slots per model point (DESIGN.md "Roofline", frozen from SURVEY.md 8d)
SLOTS_ORBIT, SLOTS_INTERIOR, SLOTS_LIMB, SLOTS_STAMP = 90, 367, 489, 4


# ------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); smax.append(float(p[2])); power.append(float(p[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # the median over samples taken while the GPU was busy (power above the idle floor)
        busy = [c for c, w in zip(sm, power) if w > 0.5 * max(power)] or sm
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(smax)),
                "power_w_max": float(max(power)), "samples": len(sm),
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------- helpers
@contextlib.contextmanager
def _stdout_to_stderr():
    """Keep stdout for the one JSON line: anything libraries print meanwhile goes to stderr."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        yield
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)


def _pinned_like(torch, a):
    t = torch.empty(a.shape, dtype=torch.float64 if a.dtype != np.uint8 else torch.uint8,
                    pin_memory=True)
    out = t.numpy()
    out[...] = a
    return t, out


def _host_threads():
    from triceratops_b200 import _hostpar
    return int(_hostpar.N_THREADS)


def _host_preparation():
    """Which code turns the prior deviates into engine columns in the e2e leg."""
    from triceratops_b200 import _blocks, _fastrng
    return {"draws": "csrc/host_rng.c (numpy's MT19937 stream, bit-identical)"
            if _fastrng._load() is not None else "numpy",
            "transforms": "csrc/host_blocks.c (numpy's statements in C, bit-identical)"
            if _blocks.available() else "numpy in threads"}


def _cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def _host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def _profiled(key):
    """Numbers that only a profiler can give (ncu capture summarised under profiles/)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", name)))
            if key in d:
                return d[key], name
        except Exception:
            continue
    return None, None


def _measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def _value_outputs(dev_calls, dev_tops, lnZ):
    """What the value leg's last step returned, per scenario branch (see --dump-outputs)."""
    rows = [r for _, _, res in dev_calls for r in res]
    top_lnL = np.full((len(rows), N_BEST), np.nan)
    top_idx = np.full((len(rows), N_BEST), -1.0)
    for j, (r, (di, dv)) in enumerate(zip(rows, dev_tops)):
        idx, val = di.cpu().numpy()[:r.n_top], dv.cpu().numpy()[:r.n_top]
        order = np.lexsort((idx, -val))     # device-pointer calls return them unsorted
        top_idx[j, :r.n_top], top_lnL[j, :r.n_top] = idx[order], val[order]
    return {"lnZ": np.asarray(lnZ, np.float64),
            "records": np.array([[r.m, r.s, r.n_finite, r.n_posinf, r.n_pass] for r in rows],
                                np.float64),
            "top_lnL": top_lnL, "top_idx": top_idx}


def _dump_outputs(out_dir, arrays):
    arrays = {k: np.asarray(v, np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, "dump of %d bytes exceeds 64 MB" % total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _slice_call(c, lo, hi):
    """The draws [lo, hi) of a recorded engine call."""
    def sl(x):
        return x if x is None or np.ndim(x) == 0 or np.size(x) == 1 else np.asarray(x)[lo:hi]
    return dict(c, N=hi - lo, cols={k: sl(v) for k, v in c["cols"].items()},
                extra_mask=None if c["extra_mask"] is None else np.asarray(c["extra_mask"])[lo:hi])


# ------------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    import _workloads
    from triceratops_b200 import _cabi, _dispatch
    from triceratops_b200._cabi import tri_col, tri_eb_args, tri_result, tri_tp_args
    from triceratops_b200.engine import get_engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        raise SystemExit("--gpus %d needs torchrun (one rank per GPU)" % args.gpus)
    torch.cuda.set_device(local)
    config = args.config
    label, star, default_draws, mission, exptime = _workloads.CONFIGS[config]
    N_arg = args.draws or default_draws
    eng = get_engine(local)
    lib = eng.lib
    lc = _workloads.lightcurve(config, model=_workloads.engine_model)
    npts = lc[0].size

    # host draws first, while no process group exists (calc_probs' host code shards the draws
    # over ranks when one does).  weak: N draws per scenario per GPU, a different seed per rank;
    # strong: N draws per scenario in total, every rank keeps its contiguous slice.
    strong = args.scaling == "strong" and world > 1
    if strong:
        calls, host_prep_s = _workloads.record_calls(config, N_arg, SEED, lc)
        lo, hi = (rank * N_arg) // world, ((rank + 1) * N_arg) // world
        calls = [_slice_call(c, lo, hi) for c in calls]
        N, N_total = hi - lo, N_arg
    else:
        calls, host_prep_s = _workloads.record_calls(config, N_arg, SEED + rank, lc)
        N, N_total = N_arg, N_arg * world
    if world > 1:
        with _stdout_to_stderr():      # NCCL announces its version on stdout
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
    units_per_step = N_ROWS * N_total * npts            # samples x points, all ranks

    # ---- device-resident copies (value path) and pinned host copies (engine-level e2e)
    keep = []
    dev_calls, host_calls = [], []
    dev_tops = []                       # (top_idx, top_lnL) device buffers, one per branch
    h2d_bytes = d2h_bytes = 0
    # the engine-level leg keeps a second, page-locked copy of every column: skipped when that
    # would pin more than 4 GB of host memory (N = 1e7)
    col_bytes = sum(np.size(v) * 8 for c in calls for v in c["cols"].values()
                    if v is not None and np.size(v) > 1)
    engine_leg = col_bytes <= (4 << 30)
    for c in calls:
        struct = tri_tp_args if c["kind"] == "tp" else tri_eb_args
        da, ha = struct(), struct()
        da.N = ha.N = c["N"]
        da.companion_is_host = ha.companion_is_host = int(c["is_host"])
        for name, val in c["cols"].items():
            if val is None:
                setattr(da, name, tri_col(None, 0)); setattr(ha, name, tri_col(None, 0))
                continue
            a = np.ascontiguousarray(np.asarray(val, dtype=np.float64).reshape(-1))
            stride = 0 if a.size == 1 and c["N"] != 1 else 1
            d = torch.from_numpy(a).cuda()
            keep.append(d)
            setattr(da, name, tri_col(d.data_ptr(), stride))
            if engine_leg:
                pt, pa = _pinned_like(torch, a)
                keep.append(pt)
                setattr(ha, name, tri_col(pa.ctypes.data, stride))
            h2d_bytes += a.nbytes
        if c["extra_mask"] is not None:
            m = np.ascontiguousarray(np.asarray(c["extra_mask"]).astype(np.uint8))
            d = torch.from_numpy(m).cuda()
            keep.append(d)
            da.extra_mask = d.data_ptr()
            if engine_leg:
                pt, pa = _pinned_like(torch, m)
                keep.append(pt)
                ha.extra_mask = pa.ctypes.data
            h2d_bytes += m.nbytes
        nb = 1 if c["kind"] == "tp" else 2
        dres, hres = (tri_result * nb)(), (tri_result * nb)()
        for b in range(nb):
            # what the production host layer asks for: the 100 best draws (selected on the
            # device) and the evidence record; the per-draw lnL stays in HBM
            di = torch.empty(N_BEST, dtype=torch.int64, device="cuda")
            dv = torch.empty(N_BEST, dtype=torch.float64, device="cuda")
            pi_ = torch.empty(N_BEST, dtype=torch.int64, pin_memory=True)
            pv = torch.empty(N_BEST, dtype=torch.float64, pin_memory=True)
            keep += [di, dv, pi_, pv]
            dev_tops.append((di, dv))
            dres[b].top_cap = hres[b].top_cap = N_BEST
            dres[b].top_idx, dres[b].top_lnL = di.data_ptr(), dv.data_ptr()
            hres[b].top_idx, hres[b].top_lnL = pi_.numpy().ctypes.data, pv.numpy().ctypes.data
            d2h_bytes += N_BEST * 16 + ctypes.sizeof(tri_result)
        dev_calls.append((c, da, dres))
        host_calls.append((c, ha, hres))

    stream = torch.cuda.current_stream().cuda_stream
    stat = dict(lnl_ms=0.0, geom_ms=0.0, tail_ms=0.0, launches=0, lnl_calls=0)
    work = dict(n_pass=0, n_stamps=0, n_interior=0, n_limb=0)
    g_ms, l_ms, s_ms = ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
    nl = ctypes.c_int32()

    def merge(records):
        """Local (m, s, n_finite, n_posinf) records of the step -> global evidences: ONE
        collective (the package's own all-gather of the packed records)."""
        return _dispatch.gather_records(records, N_total)

    def device_step(collect, count):
        records = []
        for c, a, res in dev_calls:
            eng.set_lightcurve(*c["lc"])        # cached: re-uploaded only when it changes
            fn = lib.tri_eval_tp_dev if c["kind"] == "tp" else lib.tri_eval_eb_dev
            _cabi.check(fn(ctypes.byref(a), res, stream))
            for b in range(len(res)):
                records.append((res[b].m, res[b].s, res[b].n_finite, res[b].n_posinf))
            if collect:
                _cabi.check(lib.tri_last_timing(ctypes.byref(g_ms), ctypes.byref(l_ms),
                                                ctypes.byref(s_ms), ctypes.byref(nl)))
                stat["geom_ms"] += g_ms.value; stat["lnl_ms"] += l_ms.value
                stat["tail_ms"] += s_ms.value; stat["launches"] += nl.value
                stat["lnl_calls"] += 1
            if count:
                work["n_pass"] += sum(res[b].n_pass for b in range(len(res)))
                work["n_stamps"] += res[0].n_stamps
                work["n_interior"] += res[0].n_interior
                work["n_limb"] += res[0].n_limb
        return merge(records)

    def engine_step():
        """The library's submit/wait form on pinned host columns: while one scenario's kernels
        run, the next one's columns are copied in (up to TRI_MAX_INFLIGHT calls queued)."""
        inflight = collections.deque()

        def wait_oldest():
            ticket, res = inflight.popleft()
            _cabi.check(lib.tri_wait(ctypes.c_int64(ticket), res))
        for c, a, res in host_calls:
            eng.set_lightcurve(*c["lc"])
            if len(inflight) == _cabi.TRI_MAX_INFLIGHT:
                wait_oldest()
            ticket = ctypes.c_int64()
            fn = lib.tri_submit_tp if c["kind"] == "tp" else lib.tri_submit_eb
            _cabi.check(fn(ctypes.byref(a), res, ctypes.byref(ticket)))
            inflight.append((ticket.value, res))
        while inflight:
            wait_oldest()
        records = []
        for c, a, res in host_calls:
            for b in range(len(res)):
                records.append((res[b].m, res[b].s, res[b].n_finite, res[b].n_posinf))
        return merge(records)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- FP64 issue peak of this GPU, measured before the timed region
    fp64_peak = eng.fp64_peak()

    # ---- value: inputs resident in HBM
    for _ in range(args.warmup):
        lnZ = device_step(False, False)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        lnZ = device_step(True, False)
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    # before the counting pass below overwrites the results of the last timed step
    outputs = _value_outputs(dev_calls, dev_tops, lnZ) if args.dump_outputs else None

    if args.kernel_only:
        if rank == 0:
            if outputs is not None:
                _dump_outputs(args.dump_outputs, outputs)
            print(json.dumps({"lib": os.environ.get("TRI_B200_LIB", "default"),
                              "config": config, "ms_per_step": ms_total / args.steps,
                              "lnl_ms_per_step": stat["lnl_ms"] / args.steps,
                              "geom_ms_per_step": stat["geom_ms"] / args.steps,
                              "tail_ms_per_step": stat["tail_ms"] / args.steps,
                              "launches_per_step": stat["launches"] / args.steps,
                              "clocks": clocks, "lnZ_check": [float(x) for x in lnZ[:6]]}))
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- work counts of the roofline model: one untimed pass with the counting kernel
    eng.set_counting(True)
    device_step(False, True)
    eng.set_counting(False)

    # ---- engine-level e2e: pinned host columns through tri_submit_* / tri_wait
    engine_s = None
    if engine_leg:
        for _ in range(max(1, min(args.warmup, 2))):
            engine_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            lnZ_e2e = engine_step()
        torch.cuda.synchronize()
        engine_s = max_over_ranks(time.perf_counter() - t0)
        assert np.allclose(lnZ, lnZ_e2e, rtol=0, atol=1e-9, equal_nan=True), "paths disagree"

    # ---- e2e: the public call.  target.calc_probs with numpy's draws (parity mode), N_total
    # draws per scenario, sharded over the ranks by the package itself
    import triceratops_b200

    def public_call(sampler_mode, n_calls, n_warm):
        tgt = _workloads.make_target(config)
        walls = []
        triceratops_b200.set_sampler(sampler_mode, seed=SEED)
        try:
            for k in range(n_warm + n_calls):
                barrier()
                t0 = time.perf_counter()
                _workloads.run_calc_probs(tgt, config, lc, N_total, SEED)
                torch.cuda.synchronize()
                walls.append(max_over_ranks(time.perf_counter() - t0))
        finally:
            triceratops_b200.set_sampler("host")
        return walls, tgt

    n_warm = 2 if N_total <= 2_000_000 else 1
    walls, tgt = public_call("host", args.steps, n_warm)
    e2e_s = float(np.mean(walls[n_warm:]))
    probs_gpu = np.asarray(tgt.probs.prob.values, float)
    lnZ_rows = np.asarray(tgt.lnZ, float)
    fpp, nfpp = float(tgt.FPP), float(tgt.NFPP)
    if outputs is not None:
        outputs.update(e2e_lnZ=lnZ_rows, e2e_prob=probs_gpu, e2e_fpp_nfpp=[fpp, nfpp],
                       e2e_best=tgt.probs[list(E2E_BEST_COLUMNS)].to_numpy(np.float64))
    dwalls, dtgt = public_call("device", args.steps, 1)
    dev_s = float(np.mean(dwalls[1:]))

    # ---- roofline of lnl_kernel (per launch, averaged over the timed launches)
    ns = calls[0]["lc"][4]
    pts_all = work["n_pass"] * npts * ns                    # what the reference evaluates
    # what the kernel evaluated: stamps inside a transit window that the centre probe kept
    # (the probes themselves, one orbit evaluation per window stamp, are not counted)
    pts_exec = work["n_stamps"] * ns
    W_alg = (pts_all * SLOTS_ORBIT + work["n_interior"] * SLOTS_INTERIOR
             + work["n_limb"] * SLOTS_LIMB + work["n_pass"] * npts * (SLOTS_STAMP + ns))
    W_exec = (pts_exec * SLOTS_ORBIT + work["n_interior"] * SLOTS_INTERIOR
              + work["n_limb"] * SLOTS_LIMB + work["n_stamps"] * (SLOTS_STAMP + ns))
    lnl_s_per_step = stat["lnl_ms"] * 1e-3 / args.steps     # this rank's launches of one step
    achieved = 2.0 * W_alg / lnl_s_per_step / 1e12          # TFLOP/s, DFMA = 2 flop
    peak = 2.0 * fp64_peak / 1e12
    pipe, pipe_src = _profiled("ncu_fp64_pipe_busy_pct")
    traffic, traffic_src = _profiled("traffic_bytes_per_launch")
    roofline = {
        "bound": "fp64", "kernel": "lnl_kernel", "unit": "TFLOP/s",
        "achieved": achieved, "peak": peak, "frac": achieved / peak,
        "frac_meaning": "contract W: SURVEY 8(d) slot count of the REFERENCE algorithm's work "
                        "(every model point it evaluates) / time / measured DFMA peak; can "
                        "exceed 1 because the kernel proves most points to be exactly 1 and "
                        "skips them",
        "peak_source": "measured here: DFMA-chain kernel (tri_fp64_peak); nominal 37.2",
        "executed": 2.0 * W_exec / lnl_s_per_step / 1e12,
        "frac_executed": 2.0 * W_exec / lnl_s_per_step / 1e12 / peak,
        "frac_hw": None if pipe is None else pipe / 100.0,
        "frac_hw_source": None if pipe is None else
        "profiles/%s: ncu sm__inst_executed_pipe_fp64 (%% of peak), config 2" % pipe_src,
        "ms_per_launch": stat["lnl_ms"] / max(stat["lnl_calls"], 1),
        "share_of_step": stat["lnl_ms"] / ms_total,
        "model_points_per_s": pts_all / lnl_s_per_step,
        "model_points_executed_per_s": pts_exec / lnl_s_per_step,
        "slots_per_point": {"orbit": SLOTS_ORBIT, "interior": SLOTS_INTERIOR,
                            "limb": SLOTS_LIMB, "per_stamp": SLOTS_STAMP},
        "work": {"draws_surviving_masks": work["n_pass"], "stamps_evaluated": work["n_stamps"],
                 "points_interior": work["n_interior"], "points_limb": work["n_limb"],
                 "points_reference_evaluates": pts_all},
        "param_stream_GBs": h2d_bytes * args.steps / (ms_total * 1e-3) / 1e9,
        "hbm_peak_GBs": _measured_peaks().get("hbm_gbs"),
        "traffic": traffic,
        "traffic_source": None if traffic is None else
        "profiles/%s (dram bytes read+write per launch, ncu --set full)" % traffic_src,
    }

    value = units_per_step * args.steps / (ms_total * 1e-3)
    out = {
        "metric": METRIC,
        "value": value, "unit": "samples*points/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "%s; N=%d draws per scenario%s" % (
                       label, N_total if strong else N, " in total" if strong else " per GPU"),
                   "baseline_config": config,
                   "draws_per_scenario_per_gpu": N, "draws_per_scenario_total": N_total,
                   "npts": int(npts), "nsamples": int(ns), "exptime_d": exptime,
                   "engine_calls_per_step": len(calls),
                   "l2": "inputs larger than L2: %.0f MB of draw columns per step"
                         % (h2d_bytes / 1e6),
                   "parallelism": "draws sharded, dp%d" % world},
        "e2e": {"value": N_ROWS * N_total * npts / e2e_s, "unit": "samples*points/s",
                "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h_bytes),
                "ms_per_step": e2e_s * 1e3, "steps": args.steps, "all_walls_s": walls,
                "api": "target.calc_probs(time, flux, sigma, P_orb, contrast_curve_file, filt, "
                       "N=%d, parallel=True): numpy prior draws in the reference's order "
                       "(sequential generator), transforms, pinned staging + H2D, kernels, "
                       "best-draw tables, probabilities" % N_total,
                "FPP": fpp, "NFPP": nfpp,
                "engine": None if engine_s is None else {
                    "value": units_per_step * args.steps / engine_s,
                    "ms_per_step": engine_s * 1e3 / args.steps,
                    "api": "tri_submit_tp/eb + tri_wait on pinned host columns (draws already "
                           "made), up to %d calls in flight" % _cabi.TRI_MAX_INFLIGHT},
                "device_sampler": {"value": N_ROWS * N_total * npts / dev_s,
                                   "ms_per_step": dev_s * 1e3, "steps": args.steps,
                                   "FPP": float(dtgt.FPP), "NFPP": float(dtgt.NFPP),
                                   "note": "opt-in mode: prior draws generated on the GPU "
                                           "(statistically equivalent, not numpy's stream)"}},
        "gpu_launches": int(stat["launches"]),
        "roofline": roofline,
        "clocks": clocks,
        "host_prior_draws_s": host_prep_s,
        "host": {"cores": _host_cores(), "cpu": _cpu_model(),
                 "threads": _host_threads(), "preparation": _host_preparation()},
        "lnZ_check": [float(x) for x in lnZ[:3]],
    }

    # ---- parity gates on the timed inputs (outside every timed region)
    if not args.no_parity:
        import _parity
        n_sub = args.parity_draws
        gates = [_parity.check_call(eng, c, n_sub=n_sub, seed=k) for k, c in enumerate(calls)]
        g = _parity.merge(gates)
        # probabilities: the public call's rows against the normalisation of host-side
        # log-mean-exps of the per-draw lnL the device returned for the same draws (rank 0 of a
        # weak run holds different draws than calc_probs(N_total): N == N_total only at 1 GPU)
        g["prob_max_abs"] = None
        if world == 1:
            g["prob_max_abs"] = _probability_gate(eng, config, lc, N_total, probs_gpu, lnZ_rows)
        g["draws_checked_per_call"] = n_sub
        g["gates"] = {"masks": "bit-exact, all N draws", "lnL_rel": 1e-9, "lnZ_abs": 1e-6,
                      "prob_abs": 1e-6}
        g["ok"] = bool(g["masks_equal"] and g["inf_equal"] and g["top_equal"]
                       and g["lnL_max_rel"] <= 1e-9 and g["lnZ_max_abs"] <= 1e-6
                       and (g["prob_max_abs"] is None or g["prob_max_abs"] <= 1e-6))
        out["parity"] = max_parity(g, world, dist)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_leg(config, lc, args.cpu_draws, steps=1, warmup=0)
    if rank == 0:
        if outputs is not None:
            _dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def max_parity(g, world, dist):
    """Worst case over ranks of the parity gates (each rank checked its own draws)."""
    if world == 1:
        return g
    import torch
    v = torch.tensor([g["lnL_max_rel"], g["lnZ_max_abs"], 0.0 if g["ok"] else 1.0],
                     dtype=torch.float64, device="cuda")
    dist.all_reduce(v, op=dist.ReduceOp.MAX)
    g["lnL_max_rel"], g["lnZ_max_abs"] = float(v[0]), float(v[1])
    g["ok"] = bool(v[2].item() == 0.0)
    return g


def _probability_gate(eng, config, lc, N, probs_gpu, lnZ_rows):
    """|probabilities of the public call - probabilities from host-side evidences|: the same
    seed is drawn again (recorder), every engine call is evaluated with per-draw output, and
    each row's lnZ is recomputed on the host from the device's lnL (+ prior)."""
    import _workloads
    from triceratops_b200._numerics import _normalize_probabilities
    calls, _ = _workloads.record_calls(config, N, SEED, lc)
    # the recorder may see the calls in a different order than calc_probs' rows (scenario
    # threads), so rows are matched by value: every row of the public call must have a partner
    # among the host-side evidences
    host = []
    for c in calls:
        eng.set_lightcurve(*c["lc"])
        kw = dict(c["cols"], extra_mask=c["extra_mask"], companion_is_host=c["is_host"],
                  want_lnL=True)
        res = eng.eval_tp(c["N"], **kw) if c["kind"] == "tp" else eng.eval_eb(c["N"], **kw)
        for r in ((res,) if c["kind"] == "tp" else res):
            lnw = r.lnL if c["cols"].get("lnprior") is None else r.lnL + c["cols"]["lnprior"]
            fin = np.isfinite(lnw)
            if not fin.any():
                host.append(-np.inf)
                continue
            m = lnw[fin].max()
            host.append(float(m + np.log(np.exp(lnw[fin] - m).sum()) - np.log(c["N"])))
    host = np.array(host)
    rows = np.array(lnZ_rows, float)
    matched = []
    for v in rows:
        if np.isfinite(v):
            j = int(np.argmin(np.where(np.isfinite(host), np.abs(host - v), np.inf)))
        else:
            j = int(np.flatnonzero(~np.isfinite(host))[0])
        matched.append(host[j])
    p_host, _ = _normalize_probabilities(np.array(matched))
    return float(np.max(np.abs(p_host - probs_gpu)))


# ------------------------------------------------------------------------------- CPU legs
def cpu_leg(config, lc, n_draws, steps, warmup):
    """The public call on the host cores: `target.calc_probs(N=n_draws)` with the engine
    replaced by the oracle port (numpy masks + the C restatement of likelihoods.py, OpenMP over
    draws, every core of the box).  Host prior draws included, as in the GPU arm's e2e."""
    import _workloads
    from oracle import coracle
    from oracle.engine_port import OracleEngine
    cores = _host_cores()
    coracle.set_num_threads(cores)      # torchrun exports OMP_NUM_THREADS=1: not for this arm
    coracle.orbit_table()
    ora = OracleEngine()
    tgt = _workloads.make_target(config)
    npts = lc[0].size

    def step():
        with _workloads.patched_engine(ora):
            _workloads.run_calc_probs(tgt, config, lc, n_draws, SEED)

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return {"value": N_ROWS * n_draws * npts * steps / dt, "unit": "samples*points/s",
            "cores": coracle.num_threads(), "cpu": _cpu_model(), "kind": "port",
            "seconds": dt, "ms_per_step": dt * 1e3 / steps,
            "FPP": float(tgt.FPP),
            "sample": "target.calc_probs(N=%d) per step -- host prior draws + all 18 scenario "
                      "rows through oracle/engine_port.py (numpy masks + C restatement of "
                      "likelihoods.py, OpenMP over draws); throughput-normalised, the GPU arm "
                      "runs the configuration's full N" % n_draws}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import _workloads
    config = args.config
    label = _workloads.CONFIGS[config][0]
    lc = _workloads.lightcurve(config)      # (config 4: the oracle's own model makes the curve)
    leg = cpu_leg(config, lc, args.cpu_draws, steps=args.steps, warmup=min(args.warmup, 1))
    out = {
        "impl": "reference",
        "metric": METRIC,
        "value": leg["value"], "unit": "samples*points/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": leg["ms_per_step"],
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "%s; bounded sample of %d draws per scenario per step on the host "
                               "CPU" % (label, args.cpu_draws),
                   "baseline_config": config,
                   "note": "the reference cannot be installed here (pytransit==2.2, astropy "
                           "absent, no network): CPU arm = oracle port of its algorithm behind "
                           "the same public call"},
        "cpu_baseline": {k: leg[k] for k in ("value", "unit", "cores", "cpu", "kind", "sample")},
        "e2e": {"value": leg["value"], "unit": "samples*points/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "host": {"cores": _host_cores(), "cpu": _cpu_model()},
        "gpu_launches": 0,
    }
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4],
                    help="BASELINE.json configuration (2 = configs[1], the headline)")
    ap.add_argument("--draws", type=int, default=0,
                    help="prior draws per scenario (per GPU when weak; default: the config's)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--cpu-draws", type=int, default=20000,
                    help="draws per scenario in the bounded CPU sample (both CPU legs)")
    ap.add_argument("--parity-draws", type=int, default=1500,
                    help="surviving draws per engine-call branch checked against the oracle")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--kernel-only", action="store_true",
                    help="A/B runs: the device-resident leg only")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU legs' outputs: --impl ours only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
