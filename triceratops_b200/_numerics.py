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


# ---- adaptive importance sampling: proposal tables ----------------------------------------------
# The device sampler draws each tuned prior dimension ("slot", tri_sampler_args.prop) as its
# inverse prior CDF of a coordinate v in [0, 1).  A proposal replaces the uniform v of each slot
# d by a piecewise-constant density h_d on B equal bins inside the defensive mixture
# q(v) = alpha + (1 - alpha) prod_d h_d(v_d); the importance weight of a draw is then L pi / q(v),
# and q >= alpha bounds it by L pi / alpha.  Tables per slot: the B + 1 knots C of h's
# piecewise-linear CDF (C_0 = 0, C_B = 1), then B values of ln h.
PROP_SLOTS = 6
PROP_BINS = 1024          # B
PROP_ALPHA = 0.1          # weight of the prior in the mixture
_BELOW_ONE = np.nextafter(1.0, 0.0)
_KDE_FLOOR = 1e-6         # share of a flat density in each fitted h: every bin stays positive


def identity_tables(B=PROP_BINS):
    """Tables of the prior for every slot: C_b = b / B, ln h = 0 (exact for a power-of-two B)."""
    one = np.concatenate([np.arange(B + 1, dtype=np.float64) / B, np.zeros(B)])
    return np.tile(one, (PROP_SLOTS, 1))


def _slot_table(h):
    """(2 B + 1) table of a density h over B bins (h > 0, mean 1)."""
    B = h.size
    C = np.concatenate([[0.0], np.cumsum(h / B)])
    C[-1] = 1.0
    return np.concatenate([C, np.log(h)])


def _kde_bins(x, w, B):
    """Gaussian KDE of points x in [0, 1] with weights w (sum 1), reflected at 0 and 1, as a
    density on B equal bins (mean 1).  Bandwidth: Scott's rule over the distinct points,
    sigma n^(-1/5), at least 8 bins.  The points are placed at the centres of 4 B sub-bins (at
    most 1/64 of the bandwidth away) so that the bin masses are one convolution."""
    from scipy.signal import fftconvolve
    from scipy.special import ndtr
    n = x.size
    mu = float(np.sum(w * x))
    sd = float(np.sqrt(max(np.sum(w * (x - mu) ** 2), 0.0)))
    bw = max(sd * n ** -0.2, 8.0 / B)
    R = 4 * B
    hist = np.bincount(np.minimum((x * R).astype(np.int64), R - 1), weights=w, minlength=R)
    ext = np.concatenate([hist[::-1], hist, hist[::-1]])    # mirror images at 0 and 1
    # CDF at edge b / B: sum_k ext[k] Phi((4 b + R - k - 1/2) / (R bw)), a full convolution
    g = ndtr((np.arange(-2 * R, 2 * R + 1) - 0.5) / (R * bw))
    F = fftconvolve(ext, g)[3 * R + 4 * np.arange(B + 1)]
    mass = np.maximum(np.diff(F), 0.0)
    h = mass * (B / mass.sum())
    h = (1.0 - _KDE_FLOOR) * h + _KDE_FLOOR
    return h * (B / h.sum())


def fit_proposal(coords, slots, B=PROP_BINS, alpha=PROP_ALPHA):
    """Proposal tables ([PROP_SLOTS, 2 B + 1]) fitted to K resampled posterior rows `coords`
    ([K, PROP_SLOTS], the v of each slot; rows of a systematic resample repeat draws).  The
    distinct rows are weighted by their multiplicity; each slot in `slots` gets the binned
    reflected-KDE density of its coordinates, every other slot the identity table.  An empty
    posterior (no rows, or rows that are not finite in a fitted slot) gives identity tables.
    `alpha` enters only the kernel's mixture (kept here for the signature of the schedule)."""
    del alpha
    tab = identity_tables(B)
    coords = np.asarray(coords, dtype=np.float64).reshape(-1, PROP_SLOTS)
    slots = [int(d) for d in slots]
    if not coords.shape[0] or not slots or not np.all(np.isfinite(coords[:, slots])):
        return tab
    rows, counts = np.unique(coords[:, slots], axis=0, return_counts=True)
    w = counts / counts.sum()
    for j, d in enumerate(slots):
        tab[d] = _slot_table(_kde_bins(np.clip(rows[:, j], 0.0, 1.0), w, B))
    return tab


def proposal_inverse(tab, u, mix):
    """Numpy mirror of the kernel's map of one slot: (v, b) for uniforms u; `mix` True off the
    prior branch of the mixture (v = H^-1(u)), False on it (v = u)."""
    tab = np.asarray(tab, dtype=np.float64)
    B = (tab.size - 1) // 2
    C, lnh = tab[:B + 1], tab[B + 1:]
    u = np.asarray(u, dtype=np.float64)
    mix = np.broadcast_to(np.asarray(mix, dtype=bool), u.shape)
    b_mix = np.clip(np.searchsorted(C, u, side="right") - 1, 0, B - 1)
    v_mix = np.minimum((b_mix + (u - C[b_mix]) / (np.exp(lnh[b_mix]) / B)) / B, _BELOW_ONE)
    b_pri = np.minimum((u * B).astype(np.int64), B - 1)
    return np.where(mix, v_mix, u), np.where(mix, b_mix, b_pri)


def proposal_lnq(tabs, v, slots, alpha=PROP_ALPHA, bins=None):
    """ln q(v) of the mixture for coordinates v ([n, PROP_SLOTS]) over the tuned `slots`: s = sum
    of ln h_d at the bin of v_d (floor(v_d B), or the given `bins` [n, PROP_SLOTS]), ln q =
    log1p((1 - alpha) expm1(s)); what the kernel subtracts from lnprior."""
    tabs = np.asarray(tabs, dtype=np.float64)
    B = (tabs.shape[1] - 1) // 2
    v = np.atleast_2d(np.asarray(v, dtype=np.float64))
    s = np.zeros(v.shape[0])
    for d in slots:
        b = (np.minimum((v[:, d] * B).astype(np.int64), B - 1) if bins is None
             else np.asarray(bins)[:, d])
        s = s + tabs[d, B + 1 + b]
    return np.log1p((1.0 - alpha) * np.expm1(s))


def pooled_posterior(branches, K, seed, stream):
    """The K posterior rows of one scenario call for fitting its proposal: for an EB-type call,
    the mixture of its two branches' posteriors (disjoint masks over the same draws), with the
    K rows allocated between them by evidence (merge_posteriors, the branches as two slices).
    branches: (m, T, coords [K_b, PROP_SLOTS]) per branch.  Returns [k, PROP_SLOTS] rows (k = 0
    when the posterior is empty or a weight is +inf)."""
    if len(branches) == 1:
        m, T, c = branches[0]
        if not (np.isfinite(T) and T > 0) or c is None:
            return np.zeros((0, PROP_SLOTS))
        return np.asarray(c, dtype=np.float64).reshape(-1, PROP_SLOTS)
    if any(c is None for _, _, c in branches):
        return np.zeros((0, PROP_SLOTS))
    parts, rows, off = [], [], 0
    for m, T, c in branches:
        c = np.asarray(c, dtype=np.float64).reshape(-1, PROP_SLOTS)
        parts.append((m, T, off + np.arange(len(c), dtype=np.int64)))
        rows.append(c)
        off += len(c)
    idx, _, W = merge_posteriors(parts, K, seed, stream)
    if idx is None or not len(idx) or not np.isfinite(W):
        return np.zeros((0, PROP_SLOTS))
    return np.concatenate(rows)[idx]
