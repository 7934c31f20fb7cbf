"""
NumPy restatement of the partial-correlation stage (``fcd_corr_partial``, csrc/fcd_corr_partial.cu).

Per subject s: the cleaned, centred residual rows of ``clean.residuals`` over the kept frames, the unusable-row
rule of ``clean.subject_r``; the N_s usable rows scaled to unit variance with the 1/n_s normalisation give
X (n_s x N_s).  Ledoit-Wolf as ``sklearn.covariance.ledoit_wolf(X, assume_centered=True)`` (restated here),
or a fixed shrinkage; P = ``numpy.linalg.inv`` of the shrunk matrix, r_nm = -P_nm / sqrt(P_nn P_mm), then
the clip / arctanh and edge layout of ``clean.corr_clean``.  An unusable region's edges are 0, or NaN with
``mark_missing``.

``subject_partial_ld`` restates one subject in ``np.longdouble`` (a 64-bit mantissa on x86-64) for the
precision tests: the yardstick both the kernel and the fp64 oracle are measured against.
"""
import numpy as np

from . import clean as OC
from . import iar_oracle as O

LD = np.longdouble
RANK_TOL = 1e-10                                # confound_basis_kernel's drop rule (kRankTol)


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


# ------------------------------------------------------------------ extended-precision reference
def confound_basis_ld(gk):
    """(n, r) orthonormal basis of the centred confound columns gk (n, K) over the kept frames, longdouble:
    modified Gram-Schmidt run twice (the second pass restores orthogonality at any conditioning).  A column
    whose norm after projection is <= RANK_TOL of its raw norm (pass 1) or <= RANK_TOL (pass 2) is dropped,
    the rule of confound_basis_kernel; the projection does not depend on the basis otherwise."""
    g = np.asarray(gk, dtype=LD)
    raw = np.sqrt(np.sum(g * g, axis=0))
    q = g - g.mean(axis=0)
    live = np.ones(q.shape[1], dtype=bool)
    for ref in (raw, np.ones_like(raw)):
        for j in range(q.shape[1]):
            if not live[j]:
                continue
            nrm = np.sqrt(q[:, j] @ q[:, j])
            if not nrm > RANK_TOL * ref[j]:
                live[j] = False
                continue
            q[:, j] /= nrm
            rest = live.copy()
            rest[:j + 1] = False
            q[:, rest] -= np.outer(q[:, j], q[:, j] @ q[:, rest])
    return q[:, live]


def unit_rows_ld(x, keep, g=None):
    """(N, n_s) longdouble rows of unit norm over the kept frames (zero rows for unusable regions) and the
    (N,) unusable flags: centred, cleared of the confounds by the projection on ``confound_basis_ld``, the
    unusable-row rule of ``clean.subject_r``.  x (N, T) float32 samples, keep (T,) bool, g (T, K) or None."""
    xk = np.asarray(x, dtype=np.float32)[:, keep].astype(LD)
    finite = np.isfinite(xk).all(axis=1)
    xk = np.where(finite[:, None], xk, LD(0))
    xc = xk - np.sum(xk, axis=1, keepdims=True) / LD(xk.shape[1])
    ssc = np.sum(xc * xc, axis=1)
    e = xc
    if g is not None and g.shape[1]:
        q = confound_basis_ld(np.asarray(g, dtype=np.float64)[keep])
        e = xc - (xc @ q) @ q.T
    sse = np.sum(e * e, axis=1)
    bad = ~finite | ~(sse > LD(OC.UNUSABLE_REL) * ssc)
    z = np.where(bad[:, None], LD(0), e / np.sqrt(np.where(bad, LD(1), sse))[:, None])
    return z, bad


def ledoit_wolf_ld(z, shrinkage=None):
    """z (p, n) unit-norm rows -> (Sigma, delta) in longdouble, ``ledoit_wolf`` on X = sqrt(n) z^T: R = z z^T,
    sum_t |x_t|^4 / n = n sum_t w_t^2 with w_t = sum_i z_it^2."""
    (p, n) = z.shape
    R = z @ z.T
    mu = np.trace(R) / LD(p)
    eye = np.eye(p, dtype=LD)
    if shrinkage is None:
        d2 = np.sum((R - mu * eye) ** 2) / LD(p)
        w = np.sum(z * z, axis=0)
        b2 = min(d2, (LD(n) * np.sum(w * w) - np.sum(R * R)) / (LD(n) * LD(p)))
        delta = b2 / d2 if b2 > 0 else LD(0)
    else:
        delta = LD(shrinkage)
    return (LD(1) - delta) * R + delta * mu * eye, delta


def sweep_ld(A, nb=64):
    """(-A^-1, pivots) of a symmetric A by the sweep operator in natural pivot order, nb pivots a block (each
    block swept one pivot at a time, then a rank-nb update of the rest), in longdouble.  pivots[k] is the
    k-th Schur-complement diagonal (= L_kk^2 of a Cholesky factor).  At the first pivot <= 0 the sweep stops:
    the inverse is None and the later pivots NaN."""
    A = np.array(A, dtype=LD)
    N = A.shape[0]
    piv = np.full(N, np.nan, dtype=LD)
    for k0 in range(0, N, nb):
        K = slice(k0, min(k0 + nb, N))
        D = A[K, K].copy()
        for p in range(D.shape[0]):
            d = D[p, p]
            piv[k0 + p] = d
            if not d > 0:
                return None, piv
            c = D[:, p] / d
            D -= np.outer(D[:, p], c)
            D[:, p] = c
            D[p, :] = c
            D[p, p] = -LD(1) / d
        B = A[:, K].copy()                      # panel A_IK, rows of K zero
        B[K] = 0
        W = -B @ D                              # A_IK D^-1 (D holds -D^-1)
        A -= W @ B.T
        A[:, K] = W
        A[K, :] = W.T
        A[K, K] = D
    return A, piv


def subject_partial_ld(x, keep, g=None, shrinkage=None):
    """One subject in longdouble from the same float32 samples: (r, bad, delta, pivots, kappa).  r (N, N)
    longdouble partial correlations (0 on an unusable region's edges, 1 on the diagonal, NaN when a pivot is
    <= 0), the (N,) unusable flags, delta, the sweep pivots of Sigma over the usable regions in natural order,
    and kappa_2(Sigma) (fp64 eigenvalues of Sigma and of its longdouble inverse)."""
    (z, bad) = unit_rows_ld(x, keep, g)
    use = ~bad
    N = z.shape[0]
    r = np.eye(N, dtype=LD)
    if use.sum() == 0:
        return r, bad, LD(0), np.zeros(0, dtype=LD), 1.0
    (sigma, delta) = ledoit_wolf_ld(z[use], shrinkage)
    (mP, piv) = sweep_ld(sigma)
    if mP is None:
        r[np.ix_(use, use)] = np.nan
        np.fill_diagonal(r, 1.0)
        return r, bad, delta, piv, np.inf
    d = np.sqrt(-np.diag(mP))
    r[np.ix_(use, use)] = mP / np.outer(d, d)
    np.fill_diagonal(r, 1.0)
    kappa = float(np.linalg.eigvalsh(sigma.astype(np.float64))[-1] * np.linalg.eigvalsh(
        (-mP).astype(np.float64))[-1])
    return r, bad, delta, piv, kappa


# The accuracy standard of the partial path, per subject: the kernel's error against subject_partial_ld is at
# most F_R times that of the fp64 oracle (numpy.linalg.inv) against the same reference, or F_R * ERR_FLOOR
# when the oracle's error is below the floor; delta the same with F_DELTA.
F_R = 12.0                      # largest ratio measured on a B200: 10.6 (DESIGN.md, partial correlations)
F_DELTA = 4.0                   # largest measured: 2.4
ERR_FLOOR = 4 * 2.0 ** -53


def references(x, keep, g=None, shrinkage=None):
    """Both references of one subject: ``subject_partial_ld`` and the fp64 ``subject_partial`` (NaN where
    numpy.linalg.inv finds Sigma singular), as a dict."""
    keep = np.asarray(keep, dtype=bool)
    (r, bad, delta, piv, kappa) = subject_partial_ld(x, keep, g, shrinkage)
    try:
        (r64, bad64, delta64) = subject_partial(x, keep, g, shrinkage)
    except np.linalg.LinAlgError:                      # singular in fp64: a case the kernel must flag
        (r64, bad64, delta64) = (np.full(r.shape, np.nan), bad, np.nan)
    return dict(r=r, bad=bad, delta=delta, piv=piv, kappa=kappa, r64=r64, bad64=bad64, delta64=delta64,
                min_piv=float(np.nanmin(piv.astype(np.float64))) if piv.size else np.inf)


def accuracy(col, delta, ref):
    """col (C,) partial r of one subject in edge order (no Fisher z), delta its shrinkage, ref ``references``
    -> dict of err_gpu / err_np / ratio (max |r - r_ld| over the edges of two usable regions) and the same
    for delta (derr_gpu, derr_np, dratio)."""
    N = ref["bad"].shape[0]
    (n, m) = O.edge_pairs(N)
    use = ~ref["bad"][n] & ~ref["bad"][m]
    ld = ref["r"][n, m][use]

    def err(v):
        return float(np.max(np.abs(np.asarray(v, dtype=LD) - ld))) if use.any() else 0.0

    out = dict(kappa=ref["kappa"], err_gpu=err(col[use]), err_np=err(ref["r64"][n, m][use]),
               derr_gpu=float(abs(LD(delta) - ref["delta"])), derr_np=float(abs(LD(ref["delta64"]) - ref["delta"])))
    out["ratio"] = out["err_gpu"] / max(out["err_np"], ERR_FLOOR)
    out["dratio"] = out["derr_gpu"] / max(out["derr_np"], ERR_FLOOR)
    return out
