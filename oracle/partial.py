"""
NumPy restatement of the partial-correlation stage (``fcd_corr_partial``, csrc/fcd_corr_partial.cu).

Per subject s: the cleaned, centred residual rows of ``clean.residuals`` over the kept frames, the unusable-row
rule of ``clean.subject_r``; the N_s usable rows scaled to unit variance with the 1/n_s normalisation give
X (n_s x N_s).  Ledoit-Wolf as ``sklearn.covariance.ledoit_wolf(X, assume_centered=True)`` (restated here),
or a fixed shrinkage; P = ``numpy.linalg.inv`` of the shrunk matrix, r_nm = -P_nm / sqrt(P_nn P_mm), then
the clip / arctanh and edge layout of ``clean.corr_clean``.  An unusable region's edges are 0, or NaN with
``mark_missing``.
"""
import numpy as np

from . import clean as OC
from . import iar_oracle as O


def ledoit_wolf(X, shrinkage=None):
    """X (n, p) centred samples -> (Sigma, delta): Sigma = (1 - delta) R + delta mu I with R = X^T X / n,
    mu = tr R / p and delta the Ledoit-Wolf estimate (sklearn's ledoit_wolf_shrinkage), or ``shrinkage``."""
    (n, p) = X.shape
    R = X.T @ X / n
    mu = np.trace(R) / p
    if shrinkage is None:
        d2 = np.sum((R - mu * np.eye(p)) ** 2) / p
        x4 = np.sum(np.sum(X * X, axis=1) ** 2)                # sum_t |x_t|^4
        b2 = min(d2, (x4 / n - np.sum(R * R)) / (n * p))
        shrinkage = b2 / d2 if b2 > 0 else 0.0
    return (1.0 - shrinkage) * R + shrinkage * mu * np.eye(p), shrinkage


def unit_rows(x, keep, g=None):
    """(N, n_s) usable rows scaled to unit variance (zero rows for unusable regions), and the (N,) unusable
    flags; x (N, T), keep (T,) bool, g (T, K) or None.  The rows and the rule of ``clean.subject_r``."""
    xk = np.asarray(x, dtype=np.float32)[:, keep].astype(np.float64)
    gk = None if g is None else np.asarray(g, dtype=np.float64)[keep]
    finite = np.isfinite(xk).all(axis=1)
    xk = np.where(finite[:, None], xk, 0.0)
    (e, ssc) = OC.residuals(xk, gk)
    sse = np.sum(e * e, axis=1)
    bad = ~finite | ~(sse > OC.UNUSABLE_REL * ssc)
    z = np.where(bad[:, None], 0.0, e / np.sqrt(np.where(bad, 1.0, sse))[:, None])
    return z * np.sqrt(xk.shape[1]), bad


def subject_partial(x, keep, g=None, shrinkage=None):
    """(N, N) partial correlations of one subject (0 on an unusable region's edges, 1 on the diagonal), the
    unusable flags and delta."""
    (z, bad) = unit_rows(x, keep, g)
    use = ~bad
    N = z.shape[0]
    r = np.eye(N)
    if use.sum() == 0:
        return r, bad, 0.0
    (sigma, delta) = ledoit_wolf(z[use].T, shrinkage)
    P = np.linalg.inv(sigma)
    d = np.sqrt(np.diag(P))
    r[np.ix_(use, use)] = -P / np.outer(d, d)
    np.fill_diagonal(r, 1.0)
    return r, bad, delta


def corr_partial(ts, keep, confounds=None, fisher=True, mark_missing=False, shrinkage=None):
    """ts (S, N, T) (zero-padded), keep (S, T) bool, confounds (S, T, K) or None, shrinkage None (Ledoit-Wolf)
    or a float -> ((C, S) float64 in util edge order, (S,) delta)."""
    (S, N, _) = ts.shape
    (n, m) = O.edge_pairs(N)
    out = np.empty((len(n), S), dtype=np.float64)
    deltas = np.empty(S)
    lim = 1.0 - 2.0 ** -53
    for s in range(S):
        (r, bad, deltas[s]) = subject_partial(ts[s], np.asarray(keep[s], dtype=bool),
                                              None if confounds is None else confounds[s], shrinkage)
        v = np.clip(r[n, m], -1.0, 1.0)
        out[:, s] = np.arctanh(np.clip(v, -lim, lim)) if fisher else v
        if mark_missing:
            out[bad[n] | bad[m], s] = np.nan
    return out, deltas
