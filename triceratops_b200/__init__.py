"""triceratops_b200: B200 (sm_100a) engine for the marginal-likelihood path of TRICERATOPS.

Drop-in for `target.calc_probs(...)` and the ten `lnZ_*` functions of the reference
(stevengiacalone/triceratops, triceratops/marginal_likelihoods.py): the host code stays in Python
and mirrors the reference signatures; geometry, light curves, chi^2 and the log-mean-exp run in
hand-written CUDA kernels behind a C ABI (include/triceratops_b200.h).  No CPU fallback.

    import triceratops_b200
    triceratops_b200.patch()          # an installed reference now runs this path on the GPU
"""
import importlib

__version__ = "0.1.0"

LNZ_NAMES = ("lnZ_TTP", "lnZ_TEB", "lnZ_PTP", "lnZ_PEB", "lnZ_STP", "lnZ_SEB", "lnZ_DTP",
             "lnZ_DEB", "lnZ_BTP", "lnZ_BEB")
LNL_NAMES = ("lnL_TP_p", "lnL_EB_p", "lnL_EB_twin_p")

_saved = []


def patch(level="lnZ", package="triceratops"):
    """Route an installed reference package through the GPU engine.

    level="lnZ": replace the ten scenario functions.  `calc_probs` resolves them from the globals
                 of `<package>.triceratops` (star import, triceratops.py:30), so they are set there
                 and in `<package>.marginal_likelihoods`.
    level="lnL": keep the reference's own lnZ_* host code and replace only the three per-draw
                 likelihood functions it calls (`from .likelihoods import *`,
                 marginal_likelihoods.py:6); requires parallel=True.
    Returns the list of (module, name) pairs that were replaced; undo with unpatch().
    """
    from . import likelihoods, marginal_likelihoods
    ml = importlib.import_module(package + ".marginal_likelihoods")
    mods = [ml]
    try:
        mods.append(importlib.import_module(package + ".triceratops"))
    except Exception:  # the class module needs the catalogue stack; the functions do not
        pass
    if level == "lnZ":
        names, source = LNZ_NAMES, marginal_likelihoods
    elif level == "lnL":
        names, source = LNL_NAMES, likelihoods
    else:
        raise ValueError("level must be 'lnZ' or 'lnL'")
    done = []
    for mod in mods:
        for name in names:
            if hasattr(mod, name):
                _saved.append((mod, name, getattr(mod, name)))
                setattr(mod, name, getattr(source, name))
                done.append((mod.__name__, name))
    return done


def unpatch():
    """Restore everything patch() replaced."""
    while _saved:
        mod, name, fn = _saved.pop()
        setattr(mod, name, fn)


def mc_errors():
    """Context manager: lnZ_* calls made inside it also return the Monte-Carlo error of their
    evidence -- attributes N, s2, lnZ_err and ess of each result (marginal_likelihoods.
    ScenarioResult).  The GPU then runs one extra short kernel per evaluation; lnZ and the
    best-draw tables are the same bits as without it.  calc_probs(mc_errors=True) uses it."""
    from . import _dispatch
    return _dispatch.mc_errors()


def posterior_samples(K, seed=0):
    """Context manager: lnZ_* calls made inside it also draw K posterior samples of every
    scenario branch, by systematic importance resampling of its prior draws on the GPU with
    weights exp(lnL + lnprior).  Each result's `posterior` then holds them as a table (the
    result keys plus `draw`, the global draw index), `post_total` their total weight.  lnZ,
    the best-draw tables and numpy's generator are the same as without it.  Each call takes
    the next stream of a counter that starts at 0 in each context; `seed` and the stream fix
    the samples.  calc_probs(posterior_samples=K) uses it."""
    from . import _dispatch
    return _dispatch.posterior_samples(K, seed)


def importance_proposal(p):
    """Context manager: device-sampler lnZ_* calls made inside it draw their tuned prior
    dimensions from `p`, a device_sampler.Proposal (the defensive mixture of the prior and a
    fitted product of binned marginals, _numerics.fit_proposal), and weight each draw by
    L prior / q: lnZ stays an unbiased evidence.  Outside it nothing changes.  A host-sampler
    lnZ_* call inside it raises ValueError.  calc_probs(proposal="adaptive") uses it."""
    from . import device_sampler
    return device_sampler.importance_proposal(p)


def record_coords():
    """Context manager: device-sampler lnZ_* calls made inside it that also draw posterior
    samples (posterior_samples) set each result's `post_coords`, the samples' coordinates in
    the sampler's unit cube ([K, 6], one column per slot of tri_sampler_args.prop, NaN where
    the scenario does not draw that slot): what a proposal is fitted to."""
    from . import device_sampler
    return device_sampler.record_coords()


def set_sampler(mode="host", seed=None):
    """Where the prior draws are made.

    "host" (default): numpy's global RNG in the reference's call order -- a given np.random.seed
        reproduces the reference's draws bit for bit (the parity mode).
    "device": draws are generated in HBM by one fused kernel per scenario (Philox streams,
        csrc/tri_sampler.cuh) and never visit the host; statistically equivalent results, a
        calc_probs at N = 1e6 in the time of its GPU work (device_sampler.py).  `seed` makes the
        device streams reproducible.
    """
    from . import marginal_likelihoods
    if mode not in ("host", "device"):
        raise ValueError("mode must be 'host' or 'device'")
    marginal_likelihoods._SAMPLER["mode"] = mode
    if mode == "device":
        from . import device_sampler
        device_sampler.seed(seed)
