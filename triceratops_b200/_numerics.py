"""Host-side numerics of the path: the reference's `_log_mean_exp` and
`_normalize_probabilities` contracts (triceratops/_numerics.py:12-76).

`_log_mean_exp` is what the GPU's fused log-sum-exp implements per scenario (and what
`engine.combine_lse` implements across ranks); this host version exists for the 18-element
normalisation, for small inputs, and as the definition the kernel is tested against.
"""
import numpy as np
from scipy.special import logsumexp as _logsumexp


def _log_mean_exp(logw: np.ndarray, *, N_total: int) -> float:
    """log(mean(exp(logw))) with -inf/NaN entries weighing zero but counting in N_total.

    Mirrors _numerics.py:12-51: raises ValueError when N_total != logw.size, returns +inf if
    any entry is +inf and -inf if no entry is finite.
    """
    logw = np.asarray(logw)
    if N_total != logw.size:
        raise ValueError(
            f"N_total ({N_total}) must equal len(logw) ({logw.size}). "
            "Passing len(lnL[finite]) instead of len(lnL) would silently "
            "overestimate evidence for scenarios with geometric exclusions."
        )
    if np.isposinf(logw).any():
        return np.inf
    keep = np.isfinite(logw)
    if not keep.any():
        return -np.inf
    return float(_logsumexp(logw[keep]) - np.log(N_total))


def _normalize_probabilities(lnZ: np.ndarray):
    """(probs, status) with status in {'ok', 'all_neginf', 'anomaly'} (_numerics.py:54-76)."""
    lnZ = np.asarray(lnZ, dtype=float)
    if np.isnan(lnZ).any() or np.isposinf(lnZ).any():
        return np.zeros(len(lnZ)), 'anomaly'
    if np.isneginf(lnZ).all():
        return np.zeros(len(lnZ)), 'all_neginf'
    return np.exp(lnZ - _logsumexp(lnZ)), 'ok'


# ---- Monte-Carlo error of the evidences ---------------------------------------------------------
# Each lnZ is the log-mean-exp of N ln-weights lnw = lnL + lnprior.  With m = max finite lnw,
# s = sum exp(lnw - m) and s2 = sum exp(2 (lnw - m)) over the finite entries:
#   ess = s^2 / s2                          (effective sample size)
#   r   = (N s2 / s^2 - 1) / (N - 1)        (unbiased sample variance of the weights / N, over Z^2)
#   lnZ_err = sqrt(r)                       (delta method: sd(Z) / Z)

def lse_moments(logw):
    """(m, s, s2, n_finite, n_posinf) of an array of ln-weights: the record the GPU keeps per
    branch, with the second moment of tri_set_moments."""
    logw = np.asarray(logw, dtype=float)
    n_posinf = int(np.isposinf(logw).sum())
    fin = logw[np.isfinite(logw)]
    if not fin.size:
        return -np.inf, 0.0, 0.0, 0, n_posinf
    m = float(fin.max())
    t = np.exp(fin - m)
    return m, float(t.sum()), float((t * t).sum()), int(fin.size), n_posinf


def mc_error(N, m, s, s2, n_finite, n_posinf):
    """(lnZ_err, ess, r) of one branch of N draws from its (m, s, s2) record.  lnZ_err is NaN
    when a weight is +inf, when nothing is finite (lnZ = -inf: the row then carries no variance,
    r = 0) and for N < 2."""
    if n_posinf > 0:
        return np.nan, np.nan, np.nan
    if n_finite == 0 or not s > 0:
        return np.nan, 0.0, 0.0
    ess = s * s / s2
    if N < 2:
        return np.nan, ess, np.nan
    r = max((N * s2 / (s * s) - 1.0) / (N - 1), 0.0)
    return float(np.sqrt(r)), float(ess), float(r)


def evidence_covariance(lnZ, r, calls, N_calls):
    """Covariance of the scaled evidences Z_j = exp(lnZ_j - max lnZ) of the scenario rows.
    `calls`: the rows of each scenario call (one row, or the two branches of an EB-type call,
    which share their draws with disjoint masks); `N_calls`: the draws of each call.  Rows of
    different calls are independent: Var(Z_j) = r_j Z_j^2; the branches a, b of one call have
    Cov = -Z_a Z_b / (N - 1).  Returns (Z, V)."""
    lnZ = np.asarray(lnZ, dtype=float)
    Z = np.exp(lnZ - np.max(lnZ))
    V = np.zeros((lnZ.size, lnZ.size))
    for rows, N in zip(calls, N_calls):
        for a in rows:
            if Z[a] > 0:
                V[a, a] = r[a] * Z[a] ** 2
        if len(rows) == 2 and N > 1:
            a, b = rows
            V[a, b] = V[b, a] = -Z[a] * Z[b] / (N - 1)
    return Z, V


def sum_gradient(Z, R):
    """Gradient over Z of F_R = sum_{i in R} Z_i / sum_j Z_j: (1{j in R} - F_R) / T."""
    T = Z.sum()
    ind = np.zeros(Z.size)
    ind[list(R)] = 1.0
    return (ind - Z[list(R)].sum() / T) / T


def probability_errors(lnZ, r, calls, N_calls, fpp_rows=(0, 3, 9), nfpp_from=15):
    """Delta-method errors of the scenario probabilities, FPP and NFPP.

    Returns (prob_err [rows], FPP_err, NFPP_err, var_fpp_by_call [calls]); the last one is the
    additive contribution of each call to Var(FPP) (calls are independent).  All NaN when the
    probabilities are not defined (a NaN or +inf lnZ, or every lnZ -inf) or an error is NaN."""
    lnZ = np.asarray(lnZ, dtype=float)
    r = np.asarray(r, dtype=float)
    n = lnZ.size
    nan = (np.full(n, np.nan), np.nan, np.nan, np.full(len(calls), np.nan))
    if np.isnan(lnZ).any() or np.isposinf(lnZ).any() or np.isneginf(lnZ).all():
        return nan
    Z, V = evidence_covariance(lnZ, r, calls, N_calls)
    if np.isnan(V).any():
        return nan
    prob_err = np.empty(n)
    for i in range(n):
        g = sum_gradient(Z, (i,))
        prob_err[i] = np.sqrt(max(g @ V @ g, 0.0))
    g = sum_gradient(Z, fpp_rows)
    contrib = np.array([g[rows] @ V[np.ix_(rows, rows)] @ g[rows] for rows in calls])
    fpp_err = float(np.sqrt(max(contrib.sum(), 0.0)))
    nfpp_err = 0.0
    if n > nfpp_from:
        g = sum_gradient(Z, range(nfpp_from, n))
        nfpp_err = float(np.sqrt(max(g @ V @ g, 0.0)))
    return prob_err, fpp_err, nfpp_err, contrib


# ---- posterior samples: systematic importance resampling ----------------------------------------
# For one slice of draws, sample k < K is draw min{i : C_i > (U + k) T / K}, with C the prefix sums
# of w_i = exp(lnw_i - m) in draw order and T = C_{N-1} (tri_set_posterior).  U in [0, 1) is a
# hash of (seed, stream, salt), so that no state is taken from numpy's global generator.  Salts:
# 2 j + branch, with j = 0 for the GPU's own resampling of a slice, j = 1 for the allocation of
# merge_posteriors and j = 2 + r for its thinning of slice r.
_M64 = (1 << 64) - 1


def _splitmix64(x):
    x = (x + 0x9E3779B97F4A7C15) & _M64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & _M64
    return x ^ (x >> 31)


def posterior_uniform(seed, stream, salt):
    """U in [0, 1) from (seed, stream, salt): three splitmix64 steps, the top 53 bits times
    2^-53.  posterior_select_kernel computes the same bits."""
    h = _splitmix64(int(seed) & _M64)
    h = _splitmix64(h ^ (int(stream) & _M64))
    h = _splitmix64(h ^ (int(salt) & _M64))
    return (h >> 11) * 2.0 ** -53


def _systematic_counts(U, W, K, edges):
    """Number of positions (U + k) W / K, k < K, below each of the non-decreasing `edges`."""
    step = W / K
    u = (U + np.arange(K, dtype=np.float64)) * step
    return np.searchsorted(u, np.asarray(edges, dtype=np.float64), side="left")


def merge_posteriors(parts, K, seed, stream, branch=0):
    """Merge the K-sample posteriors of disjoint slices of draws, in slice order (ranks in rank
    order, or rounds of refinement).  parts: (m_r, T_r, idx_r) per slice -- the slice's record
    maximum, its sum of weights relative to exp(m_r), its K sample indices (global, ascending;
    None when the slice had posterior samples off).

    With m = max m_r and W_r = T_r exp(m_r - m), slice r gets c_r of the K merged samples, the
    number of positions (U_0 + k) W / K in [sum_{r'<r} W_r', sum_{r'<=r} W_r') (so c_r is
    floor or ceil of K W_r / W), and contributes its samples at positions floor((j + U_r) K /
    c_r), j < c_r.  Each draw then has K w_i / W expected copies, as from one slice of all the
    draws; a sharded run gives the same distribution as one rank, not the same bits.  One slice
    is returned unchanged.  Returns (idx, m, W): empty idx when a T_r is +inf or no weight is
    finite, None when a slice had samples off."""
    K = int(K)
    if any(p[2] is None for p in parts):
        return None, np.nan, np.nan
    if any(np.isposinf(p[1]) for p in parts):
        return np.zeros(0, dtype=np.int64), np.nan, np.inf
    live = [p for p in parts if p[1] > 0 and len(p[2])]
    if not live:
        return np.zeros(0, dtype=np.int64), -np.inf, 0.0
    m = max(p[0] for p in live)
    if len(parts) == 1:
        return np.asarray(parts[0][2], dtype=np.int64), m, float(parts[0][1])
    Wr = np.array([p[1] * np.exp(p[0] - m) if (p[1] > 0 and len(p[2])) else 0.0
                   for p in parts])
    cum = np.cumsum(Wr)
    W = float(cum[-1])
    ends = _systematic_counts(posterior_uniform(seed, stream, 2 + branch), W, K, cum)
    # (positions that rounding left at or above W: the last slice of positive weight)
    ends[int(np.flatnonzero(Wr > 0)[-1]):] = K
    c = np.diff(np.concatenate([[0], ends]))
    out = []
    for r, (p, cr) in enumerate(zip(parts, c)):
        if cr == 0:
            continue
        idx = np.asarray(p[2], dtype=np.int64)
        if cr >= len(idx):
            out.append(idx)
            continue
        U = posterior_uniform(seed, stream, 2 * (2 + r) + branch)
        pos = np.floor((np.arange(cr) + U) * (len(idx) / cr)).astype(np.int64)
        out.append(idx[np.minimum(pos, len(idx) - 1)])
    return np.concatenate(out), m, W
