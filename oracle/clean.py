"""
NumPy restatement of the cleaned correlation stage (``fcd_corr_fisherz_clean``, csrc/fcd_corr_clean.cu).

Per subject s: the kept frames (t < T_s and the sample mask keeps t) in fp64, ``lstsq`` of every region on
[1, G_s] over those frames, the residual rows, ``numpy.corrcoef`` of the residuals, then the clip / arctanh
of ``iar_oracle.corr_fisherz``.  A region row with a non-finite kept sample, or whose residual sum of
squares is at most 2^-40 of its centred sum of squares, is unusable: r = 0 on its edges, or NaN with
``mark_missing`` (the convention of ``missing.corr_fisherz_masked``).  Samples and confounds of frames that
are not kept are never used.
"""
import numpy as np

from . import iar_oracle as O

UNUSABLE_REL = 2.0 ** -40


def residuals(x, g):
    """x (N, n) fp64 rows over the kept frames, g (n, K) confounds or None -> (N, n) residuals of x after
    least squares on [1, g], and the (N,) centred sums of squares."""
    n = x.shape[1]
    xc = x - x.mean(axis=1, keepdims=True)
    A = np.ones((n, 1)) if g is None or g.shape[1] == 0 else np.hstack([np.ones((n, 1)), g])
    # regressing the centred rows gives the residuals of x itself (the constant is a column of A), and a
    # row that is constant over the kept frames an exactly zero residual
    coef = np.linalg.lstsq(A, xc.T, rcond=None)[0]
    e = xc - (A @ coef).T
    return e, np.sum(xc * xc, axis=1)


def subject_r(x, keep, g=None):
    """(N, N) correlations of one subject over its kept frames, and the (N,) unusable-row flags.
    x (N, T) samples, keep (T,) bool, g (T, K) confounds or None."""
    xk = np.asarray(x, dtype=np.float32)[:, keep].astype(np.float64)
    gk = None if g is None else np.asarray(g, dtype=np.float64)[keep]
    finite = np.isfinite(xk).all(axis=1)
    xk = np.where(finite[:, None], xk, 0.0)
    (e, ssc) = residuals(xk, gk)
    sse = np.sum(e * e, axis=1)
    bad = ~finite | ~(sse > UNUSABLE_REL * ssc)
    z = np.where(bad[:, None], 0.0, e / np.sqrt(np.where(bad, 1.0, sse))[:, None])
    return z @ z.T, bad


def corr_clean(ts, keep, confounds=None, fisher=True, mark_missing=False):
    """ts (S, N, T) (zero-padded), keep (S, T) bool (False beyond each subject's length), confounds
    (S, T, K) or None -> (C, S) float64 in util edge order."""
    (S, N, _) = ts.shape
    (n, m) = O.edge_pairs(N)
    out = np.empty((len(n), S), dtype=np.float64)
    lim = 1.0 - 2.0 ** -53
    for s in range(S):
        (r, bad) = subject_r(ts[s], np.asarray(keep[s], dtype=bool), None if confounds is None else confounds[s])
        v = np.clip(r[n, m], -1.0, 1.0)
        out[:, s] = np.arctanh(np.clip(v, -lim, lim)) if fisher else v
        if mark_missing:
            out[bad[n] | bad[m], s] = np.nan
    return out


def partial_corr_precision(x, keep, g=None):
    """Independent formulation for the tests: the partial correlation of every pair of regions given the
    confounds (and a constant) over the kept frames, from the precision matrix of the joint covariance of
    (x_n, x_m, G): -P_nm / sqrt(P_nn P_mm), computed one pair at a time.  x (N, T), keep (T,), g (T, K)."""
    xk = np.asarray(x, dtype=np.float64)[:, keep]
    gk = np.zeros((xk.shape[1], 0)) if g is None else np.asarray(g, dtype=np.float64)[keep]
    N = xk.shape[0]
    r = np.eye(N)
    for a in range(N):
        for b in range(a):
            P = np.linalg.inv(np.cov(np.vstack([xk[a], xk[b], gk.T])))
            r[a, b] = r[b, a] = -P[0, 1] / np.sqrt(P[0, 0] * P[1, 1])
    return r
