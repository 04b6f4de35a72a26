"""Batch vetting of many targets (BASELINE config 5: sweeps of hundreds of TOIs).

One `calc_probs` is dominated by its host side -- numpy's sequential RNG and the Python glue take
~2 s at N = 1e6 while the GPU work takes ~0.2 s -- so a sweep is scheduled TOI-major: whole
targets are handed to worker processes, several per GPU (each worker owns a CUDA context on its
GPU; their kernels time-slice, their host work runs in parallel on the host cores).  No
collective is needed: targets are independent.  Within torchrun the same function splits the
job list over ranks instead (`jobs[rank::world]`).

A job is a dict with the arguments of `target(...)` and `calc_probs(...)`:
    {"ID": 123, "stars": DataFrame, "trilegal_fname": "...", "time": t, "flux": f,
     "flux_err": sigma, "P_orb": 3.2, "seed": 7, "calc_probs": {"N": 1_000_000, ...},
     "sampler": "host" | "device"}
"sampler" picks where the prior draws are made for that job (`set_sampler`): "host" (default)
reproduces the reference's numpy streams for the job's seed; "device" draws in HBM, which removes
most of the host work and makes the sweep GPU-bound.
The result per job is {"ID", "FPP", "NFPP", "FPP_degenerate", "lnZ", "probs" (DataFrame as dict),
"wall_s"}.
"""
import multiprocessing as mp
import os
import queue
import time as _time

import numpy as np


def run_job(job):
    """One target through the drop-in `target.calc_probs` on this process's engine."""
    from .triceratops import target
    from . import set_sampler
    t0 = _time.perf_counter()
    tgt = target(job["ID"], stars=job["stars"], trilegal_fname=job.get("trilegal_fname"),
                 mission=job.get("mission", "TESS"))
    if job.get("seed") is not None:
        np.random.seed(job["seed"])
    kw = dict(parallel=True, verbose=0)
    kw.update(job.get("calc_probs", {}))
    sampler = job.get("sampler", "host")
    try:
        set_sampler(sampler, seed=job.get("seed"))
        tgt.calc_probs(np.asarray(job["time"], float), np.asarray(job["flux"], float),
                       job["flux_err"], job["P_orb"], **kw)
    finally:
        set_sampler("host")
    out = {"ID": job["ID"], "FPP": float(tgt.FPP), "NFPP": float(tgt.NFPP),
           "FPP_degenerate": bool(tgt.FPP_degenerate), "lnZ": np.asarray(tgt.lnZ),
           "probs": tgt.probs.to_dict(orient="list"), "wall_s": _time.perf_counter() - t0}
    if tgt.FPP_err is not None:    # (calc_probs with mc_errors / fpp_err_target)
        out["FPP_err"], out["NFPP_err"] = float(tgt.FPP_err), float(tgt.NFPP_err)
    return out


def _worker(worker_id, n_gpus, jobs, out_q, n_workers=None):
    os.environ["LOCAL_RANK"] = str(worker_id % max(n_gpus, 1))
    # the workers share the host: an equal part of the cores each for the generator helpers and
    # the preparation blocks (measured on the 16-core GPU box, numpy draws: 4 workers x 4 threads
    # 3.7 TOIs/s, 16 x 1 2.3, 1 x 16 2.3), one numpy/BLAS thread
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        cores = os.cpu_count() or 1
    share = max(1, cores // max(1, n_workers or cores))
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    os.environ.setdefault("TRI_B200_HOST_THREADS", str(share))
    os.environ.setdefault("TRI_B200_SCENARIO_THREADS", "1")
    try:
        for idx, job in jobs:
            out_q.put((idx, run_job(job), None))
    except Exception as exc:  # pragma: no cover - reported to the parent
        out_q.put((-1, None, "worker %d: %r" % (worker_id, exc)))
    out_q.put((None, None, None))


def vet_many(jobs, n_gpus=None, workers_per_gpu=4):
    """Run `jobs` TOI-major and return their results in job order.

    Under torchrun (WORLD_SIZE > 1) this rank processes jobs[rank::world] in-process and returns
    only those (callers gather if they need to).  Otherwise `n_gpus * workers_per_gpu` worker
    processes are spawned (n_gpus defaults to the visible CUDA devices)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        rank = int(os.environ.get("RANK", "0"))
        from . import _dispatch
        results = []
        with _dispatch.no_sharding():
            for job in jobs[rank::world]:
                results.append(run_job(job))
        return results
    if n_gpus is None:
        import torch
        n_gpus = torch.cuda.device_count()
    if n_gpus < 1:
        raise RuntimeError("vet_many needs at least one CUDA device (no CPU fallback)")
    n_workers = max(1, min(n_gpus * workers_per_gpu, len(jobs)))
    ctx = mp.get_context("spawn")
    out_q = ctx.Queue()
    procs = []
    for w in range(n_workers):
        share = [(i, jobs[i]) for i in range(w, len(jobs), n_workers)]
        p = ctx.Process(target=_worker, args=(w, n_gpus, share, out_q, n_workers))
        p.start()
        procs.append(p)
    results = [None] * len(jobs)
    done = 0
    error = None
    while done < n_workers and error is None:
        try:
            idx, res, err = out_q.get(timeout=5.0)
        except queue.Empty:
            # a worker that died (killed, crashed in native code) never reports: do not wait
            dead = [p for p in procs if p.exitcode not in (None, 0)]
            if dead:
                error = "worker process exited with code %s" % dead[0].exitcode
            continue
        if err is not None:
            error = err
        elif idx is None:
            done += 1
        else:
            results[idx] = res
    if error:
        for p in procs:
            if p.is_alive():
                p.terminate()
    for p in procs:
        p.join()
    if error:
        raise RuntimeError(error)
    return results
