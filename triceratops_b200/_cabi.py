"""ctypes binding of include/triceratops_b200.h (the drop-in boundary of the engine).

There is no CPU fallback: loading fails loudly if the CUDA library has not been built, and
every call raises if no GPU is usable.
"""
import ctypes
import os

import numpy as np

from . import _build

c_double_p = ctypes.POINTER(ctypes.c_double)
c_uint8_p = ctypes.POINTER(ctypes.c_uint8)

TRI_OK, TRI_ECUDA, TRI_EINVAL, TRI_ESTATE, TRI_ENODEVICE = 0, -1, -2, -3, -4
TRI_MAX_INFLIGHT = 4     # include/triceratops_b200.h
TRI_MAX_CADENCES = 8     # include/triceratops_b200.h
TRI_MAX_POSTERIOR = 1 << 20   # include/triceratops_b200.h


class TriError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("triceratops_b200 error %d: %s" % (code, msg))
        self.code = code


class tri_col(ctypes.Structure):
    _fields_ = [("ptr", ctypes.c_void_p), ("stride", ctypes.c_int64)]


class tri_tp_args(ctypes.Structure):
    _fields_ = ([("N", ctypes.c_int64)]
                + [(n, tri_col) for n in ("rp", "P_orb", "inc", "ecc", "argp", "mtot", "rhost",
                                          "u1", "u2", "cfr", "lnprior")]
                + [("extra_mask", ctypes.c_void_p), ("companion_is_host", ctypes.c_int32)])


class tri_eb_args(ctypes.Structure):
    _fields_ = ([("N", ctypes.c_int64)]
                + [(n, tri_col) for n in ("reb", "ebfr", "q", "P_orb", "inc", "ecc", "argp",
                                          "mtot", "rhost", "u1", "u2", "cfr", "lnprior")]
                + [("extra_mask", ctypes.c_void_p), ("companion_is_host", ctypes.c_int32),
                   ("scalar_loop", ctypes.c_int32)])


class tri_result(ctypes.Structure):
    _fields_ = [("lnZ", ctypes.c_double), ("m", ctypes.c_double), ("s", ctypes.c_double),
                ("n_finite", ctypes.c_int64), ("n_posinf", ctypes.c_int64),
                ("n_pass", ctypes.c_int64), ("n_stamps", ctypes.c_int64),
                ("n_interior", ctypes.c_int64), ("n_limb", ctypes.c_int64),
                ("lnL_out", ctypes.c_void_p), ("mask_out", ctypes.c_void_p),
                ("top_cap", ctypes.c_int64), ("n_top", ctypes.c_int64),
                ("n_evaluated", ctypes.c_int64),
                ("top_idx", ctypes.c_void_p), ("top_lnL", ctypes.c_void_p)]


class tri_powerlaw(ctypes.Structure):
    _fields_ = [("nseg", ctypes.c_int32), ("constant", ctypes.c_double),
                ("powers", ctypes.c_double * 3), ("amps", ctypes.c_double * 3),
                ("integrals", ctypes.c_double * 3), ("cum", ctypes.c_double * 3),
                ("epow", ctypes.c_double * 3), ("norm", ctypes.c_double)]


class tri_spline(ctypes.Structure):
    _fields_ = [("t", ctypes.c_void_p), ("c", ctypes.c_void_p), ("n", ctypes.c_int32),
                ("k", ctypes.c_int32)]


class tri_bound_prior(ctypes.Structure):
    _fields_ = ([(n, ctypes.c_double) for n in ("d_pc", "M_eff", "M_act", "f1", "f2", "f3",
                                                "alpha", "dlogP", "slope", "slope2", "t2", "t3",
                                                "t4", "t5")]
                + [("first_decade", ctypes.c_int32)])


class tri_sampler_args(ctypes.Structure):
    _fields_ = (
        [("n", ctypes.c_int64), ("index0", ctypes.c_int64), ("seed", ctypes.c_uint64),
         ("stream", ctypes.c_uint64), ("kind", ctypes.c_int32), ("host", ctypes.c_int32),
         ("diluter", ctypes.c_int32), ("flatpriors", ctypes.c_int32)]
        + [(n, ctypes.c_double) for n in ("P_lo", "P_hi", "ecc_expo", "M_s", "R_s", "Teff", "u1",
                                          "u2")]
        + [(n, tri_powerlaw) for n in ("rp_hi", "rp_lo", "q_pl", "qc_pl")]
        + [(n, tri_spline) for n in ("hot_R", "cool_R", "hot_T", "cool_T", "flux_tess",
                                     "flux_cc")]
        + [("f_target_tess", ctypes.c_double), ("f_target_cc", ctypes.c_double),
           ("ldc_u1", ctypes.c_void_p), ("ldc_u2", ctypes.c_void_p), ("Teff_cap", ctypes.c_double),
           ("prior_mode", ctypes.c_int32), ("use_cc", ctypes.c_int32),
           ("beb_cc_band", ctypes.c_int32), ("cc_n", ctypes.c_int32),
           ("cc_sep", ctypes.c_void_p), ("cc_con", ctypes.c_void_p), ("bound", tri_bound_prior),
           ("bg_const_prior", ctypes.c_double), ("molusc_q", ctypes.c_void_p),
           ("n_comp", ctypes.c_int64), ("idx_hi", ctypes.c_int64)]
        + [(n, ctypes.c_void_p) for n in ("bg_mass", "bg_radius", "bg_logg", "bg_teff", "bg_u1",
                                          "bg_u2", "bg_fr_tess", "bg_dmag_cc", "bg_fr_cc")]
        + [("o_" + n, ctypes.c_void_p) for n in ("body", "ebfr", "q", "P", "inc", "ecc", "argp",
                                                 "mtot", "rhost", "u1", "u2", "cfr", "lnprior",
                                                 "mhost", "meb")]
        + [("o_mask", ctypes.c_void_p), ("err_flag", ctypes.c_void_p)])


# every symbol include/triceratops_b200.h declares
EXPORTS = ("tri_init", "tri_shutdown", "tri_last_error", "tri_set_lightcurve", "tri_eval_tp",
           "tri_eval_eb", "tri_eval_tp_dev", "tri_eval_eb_dev", "tri_lnl_tp", "tri_lnl_eb",
           "tri_simulate_tp", "tri_simulate_eb",
           "tri_fetch_lnl", "tri_log_mean_exp", "tri_last_timing", "tri_fp64_peak", "tri_sm_count",
           "tri_submit_tp", "tri_submit_eb", "tri_submit_tp_dev", "tri_submit_eb_dev", "tri_wait",
           "tri_dev_splev", "tri_set_counting", "tri_set_lightcurve_err", "tri_dev_sample",
           "tri_struct_sizes", "tri_set_lightcurve_cadence", "tri_set_moments",
           "tri_last_moments", "tri_set_posterior", "tri_last_posterior")

_lib = None


def library_path():
    # TRI_B200_LIB lets developers A/B a differently tuned build of the same sources
    return os.environ.get("TRI_B200_LIB", _build.SO_PATH)


def load():
    """Load the CUDA library (raises if it is missing -- build it with __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise ImportError(
            "CUDA extension %s is missing; run `python -c 'import __graft_entry__ as g; "
            "g.build()'` (needs nvcc). triceratops_b200 has no CPU fallback." % path)
    L = ctypes.CDLL(path)
    for name in EXPORTS:
        getattr(L, name)  # AttributeError if the header and the library disagree
    L.tri_last_error.restype = ctypes.c_char_p
    L.tri_init.argtypes = [ctypes.c_int]
    L.tri_set_lightcurve.argtypes = [c_double_p, c_double_p, ctypes.c_int64, ctypes.c_double,
                                     ctypes.c_double, ctypes.c_int32]
    L.tri_set_lightcurve_err.argtypes = [c_double_p, c_double_p, c_double_p, ctypes.c_int64,
                                         ctypes.c_double, ctypes.c_int32]
    L.tri_set_lightcurve_cadence.argtypes = [c_double_p, c_double_p, c_double_p, ctypes.c_double,
                                             c_double_p, ctypes.POINTER(ctypes.c_int32),
                                             ctypes.c_int64]
    L.tri_eval_tp.argtypes = [ctypes.POINTER(tri_tp_args), ctypes.POINTER(tri_result)]
    L.tri_eval_eb.argtypes = [ctypes.POINTER(tri_eb_args), ctypes.POINTER(tri_result)]
    L.tri_eval_tp_dev.argtypes = [ctypes.POINTER(tri_tp_args), ctypes.POINTER(tri_result),
                                  ctypes.c_void_p]
    L.tri_eval_eb_dev.argtypes = [ctypes.POINTER(tri_eb_args), ctypes.POINTER(tri_result),
                                  ctypes.c_void_p]
    c_i64_p = ctypes.POINTER(ctypes.c_int64)
    L.tri_submit_tp.argtypes = [ctypes.POINTER(tri_tp_args), ctypes.POINTER(tri_result), c_i64_p]
    L.tri_submit_eb.argtypes = [ctypes.POINTER(tri_eb_args), ctypes.POINTER(tri_result), c_i64_p]
    L.tri_submit_tp_dev.argtypes = [ctypes.POINTER(tri_tp_args), ctypes.POINTER(tri_result),
                                    ctypes.c_void_p, c_i64_p]
    L.tri_submit_eb_dev.argtypes = [ctypes.POINTER(tri_eb_args), ctypes.POINTER(tri_result),
                                    ctypes.c_void_p, c_i64_p]
    L.tri_wait.argtypes = [ctypes.c_int64, ctypes.POINTER(tri_result)]
    L.tri_dev_splev.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32,
                                ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]
    L.tri_lnl_tp.argtypes = [ctypes.c_int64] + [c_double_p] * 10 + [ctypes.c_int32, c_double_p]
    L.tri_lnl_eb.argtypes = ([ctypes.c_int64] + [c_double_p] * 11
                             + [ctypes.c_int32, ctypes.c_int32, c_double_p])
    L.tri_simulate_tp.argtypes = [ctypes.c_int64] + [c_double_p] * 10 + [ctypes.c_int32,
                                                                        c_double_p]
    L.tri_simulate_eb.argtypes = ([ctypes.c_int64] + [c_double_p] * 11
                                  + [ctypes.c_int32, ctypes.c_int32, c_double_p, c_double_p])
    L.tri_fetch_lnl.argtypes = [ctypes.c_int32, c_double_p, ctypes.c_int64]
    L.tri_log_mean_exp.argtypes = [c_double_p, ctypes.c_int64, ctypes.POINTER(tri_result)]
    L.tri_last_timing.argtypes = [c_double_p, c_double_p, c_double_p,
                                  ctypes.POINTER(ctypes.c_int32)]
    L.tri_fp64_peak.argtypes = [c_double_p]
    L.tri_set_counting.argtypes = [ctypes.c_int32]
    L.tri_set_moments.argtypes = [ctypes.c_int32]
    L.tri_last_moments.argtypes = [c_double_p]
    L.tri_set_posterior.argtypes = [ctypes.c_int64, ctypes.c_uint64, ctypes.c_uint64]
    L.tri_last_posterior.argtypes = [ctypes.c_int32, ctypes.POINTER(ctypes.c_int64),
                                     ctypes.c_int64, ctypes.POINTER(ctypes.c_int64), c_double_p]
    L.tri_dev_sample.argtypes = [ctypes.POINTER(tri_sampler_args), ctypes.c_void_p]
    L.tri_struct_sizes.argtypes = [ctypes.POINTER(ctypes.c_int64), ctypes.c_int32]
    L.tri_sm_count.argtypes = [ctypes.POINTER(ctypes.c_int32)]
    _lib = L
    return L


def check(rc):
    if rc != TRI_OK:
        raise TriError(rc, load().tri_last_error().decode("utf-8", "replace"))


def dptr(a):
    return a.ctypes.data_as(c_double_p)


def f64(x):
    """C-contiguous float64 view/copy (what the ABI requires of every column)."""
    return np.ascontiguousarray(x, dtype=np.float64)
