"""CPU: the partial-correlation oracle (oracle/partial.py) against sklearn's Ledoit-Wolf and against residual
correlations, its unusable-region rule, and the host checks of corr.correlations(kind="partial") that run
before any device work."""
import numpy as np
import numpy.testing as nptest
import pytest

from oracle import iar_oracle as O
from oracle import partial as OP
from fcdiff_b200 import corr


def series(N, T, K, seed):
    rng = np.random.RandomState(seed)
    g = rng.standard_normal((T, K))
    x = rng.standard_normal((N, N)) @ rng.standard_normal((N, T)) + rng.standard_normal((N, K)) @ g.T
    return (x + rng.uniform(-5, 5, (N, 1))).astype(np.float32), g


@pytest.mark.parametrize("n,p", [(200, 40), (50, 3), (30, 60), (1200, 25)])
def test_ledoit_wolf_is_sklearn(n, p):
    cov = pytest.importorskip("sklearn.covariance")
    rng = np.random.RandomState(n + p)
    X = rng.standard_normal((n, p)) @ (np.eye(p) + 0.3 * rng.standard_normal((p, p)))
    X -= X.mean(axis=0)
    X /= np.sqrt((X * X).mean(axis=0))
    (sig, delta) = OP.ledoit_wolf(X)
    (sig_sk, delta_sk) = cov.ledoit_wolf(X, assume_centered=True)
    assert abs(delta - delta_sk) <= 1e-14
    nptest.assert_allclose(sig, sig_sk, rtol=0, atol=1e-14)


@pytest.mark.parametrize("K", [0, 2, 5])
def test_unshrunk_is_residual_correlation(K):
    (N, T) = (9, 80)
    (x, g) = series(N, T, K, 20 + K)
    keep = np.random.RandomState(K).rand(T) > 0.2
    (r, bad, delta) = OP.subject_partial(x, keep, g if K else None, shrinkage=0.0)
    assert not bad.any() and delta == 0.0
    xk = x[:, keep].astype(np.float64)
    n = xk.shape[1]
    assert n > N + K + 1
    base = np.hstack([np.ones((n, 1)), g[keep]]) if K else np.ones((n, 1))
    for a in range(N):
        for b in range(a):
            A = np.hstack([base, np.delete(xk, [a, b], axis=0).T])
            ea = xk[a] - A @ np.linalg.lstsq(A, xk[a], rcond=None)[0]
            eb = xk[b] - A @ np.linalg.lstsq(A, xk[b], rcond=None)[0]
            assert abs(r[a, b] - ea @ eb / np.sqrt((ea @ ea) * (eb @ eb))) <= 1e-11


@pytest.mark.parametrize("how", ["nan", "constant", "confound"])
def test_unusable_region_is_left_out(how):
    (N, T, K) = (8, 60, 2)
    (x, g) = series(N, T, K, 5)
    keep = np.ones(T, dtype=bool)
    keep[[3, 17]] = False
    if how == "nan":
        x[4, 10] = np.nan
    elif how == "constant":
        x[4] = np.float32(2.5)
    else:
        x[4] = (3.0 * g[:, 1] - 1.0).astype(np.float32)
    (r, bad, delta) = OP.subject_partial(x, keep, g)
    assert bad.tolist() == [n == 4 for n in range(N)]
    use = ~bad
    (r_sub, bad_sub, delta_sub) = OP.subject_partial(x[use], keep, g)
    assert not bad_sub.any() and abs(delta - delta_sub) <= 1e-14         # lstsq rounds by the batch of rows
    nptest.assert_allclose(r[np.ix_(use, use)], r_sub, rtol=0, atol=1e-13)
    assert (r[4, use] == 0).all()
    (out, _) = OP.corr_partial(x[None], keep[None], g[None], mark_missing=True)
    (n, m) = O.edge_pairs(N)
    assert np.isnan(out[(n == 4) | (m == 4), 0]).all() and np.isfinite(out[(n != 4) & (m != 4), 0]).all()


def test_full_shrinkage_gives_zero():
    (x, _) = series(6, 40, 0, 1)
    (r, _, delta) = OP.subject_partial(x, np.ones(40, bool), shrinkage=1.0)
    assert delta == 1.0
    assert (r[~np.eye(6, dtype=bool)] == 0).all()


# ------------------------------------------------------------------ host checks (no device needed)
def test_unknown_kind_raises():
    ts = np.zeros((2, 4, 30), np.float32)
    with pytest.raises(ValueError, match="kind"):
        corr.correlations(ts, kind="tangent")
    with pytest.raises(ValueError, match="kind"):
        corr.check_kind("precision", "ledoit-wolf")


@pytest.mark.parametrize("bad", [-0.1, 1.5, float("nan"), "oas"])
def test_shrinkage_outside_unit_interval_raises(bad):
    with pytest.raises(ValueError, match="shrinkage"):
        corr.correlations(np.zeros((2, 4, 30), np.float32), kind="partial", shrinkage=bad)


def test_return_shrinkage_needs_partial():
    with pytest.raises(ValueError, match="return_shrinkage"):
        corr.correlations(np.zeros((2, 4, 30), np.float32), return_shrinkage=True)


@pytest.mark.parametrize("K", [0, 3])
def test_unshrunk_singular_subject_raises(K):
    (S, N, T) = (3, 20, 40)
    ts = np.random.RandomState(0).standard_normal((S, N, T)).astype(np.float32)
    keep = np.ones((S, T), bool)
    keep[1, N + K + 1:] = False                     # n_1 = N + K + 1: still fine
    keep[2, N + K:] = False                         # n_2 = N + K: singular
    g = np.random.RandomState(1).standard_normal((S, T, K)) if K else None
    with pytest.raises(ValueError, match="subject 2 keeps %d frames" % (N + K)):
        corr.correlations(ts, kind="partial", shrinkage=0.0, sample_mask=keep, confounds=g)
    lists = [ts[s][:, :N + K] for s in range(S)]    # ragged: every subject singular
    with pytest.raises(ValueError, match="subject 0"):
        corr.correlations(lists, kind="partial", shrinkage=0.0,
                          confounds=None if g is None else [g[s][:N + K] for s in range(S)])


# ------------------------------------------------------------------ the longdouble reference
def factor_series(N, T, K, seed):
    """Planted 8-factor series with confound components: well conditioned (kappa ~ 10 under Ledoit-Wolf)."""
    rng = np.random.RandomState(seed)
    a = np.where(rng.rand(N) < 0.5, 0.55, -0.27)
    f = rng.standard_normal((8, T))
    g = rng.standard_normal((T, K))
    x = np.sqrt(1 - a * a)[:, None] * rng.standard_normal((N, T)) + a[:, None] * f[np.arange(N) % 8]
    x += 0.5 * rng.standard_normal((N, K)) @ g.T + rng.uniform(-5, 5, (N, 1))
    return x.astype(np.float32), g


@pytest.mark.parametrize("N,T,K,shrinkage", [(40, 300, 0, None), (70, 200, 3, None), (65, 500, 2, 0.0),
                                             (30, 20, 1, None)])
def test_longdouble_reference_is_the_fp64_oracle_when_well_conditioned(N, T, K, shrinkage):
    (x, g) = factor_series(N, T, K, N + K)
    keep = np.random.RandomState(T).rand(T) > 0.15
    (r, bad, delta, piv, kappa) = OP.subject_partial_ld(x, keep, g if K else None, shrinkage)
    (r64, bad64, delta64) = OP.subject_partial(x, keep, g if K else None, shrinkage)
    assert kappa < 100 and (bad == bad64).all() and not bad.any()
    assert np.abs(r.astype(np.float64) - r64).max() <= 1e-14
    assert abs(float(delta) - delta64) <= 1e-14
    assert piv.dtype == np.longdouble and (piv > 0).all()


def test_longdouble_reference_closed_forms():
    # N = 2: Sigma = [[1, (1 - delta) rho], [(1 - delta) rho, 1]], so r = (1 - delta) rho, rho the Pearson
    # correlation of the cleaned rows
    LD = np.longdouble
    (x, g) = factor_series(2, 90, 2, 3)
    x[1] += 2 * x[0]                                    # strongly correlated: delta < 1
    keep = np.ones(90, bool)
    keep[::7] = False
    (r, _, delta, _, _) = OP.subject_partial_ld(x, keep, g)
    assert 0 < delta < 1
    (z, _) = OP.unit_rows_ld(x, keep, g)
    rho = np.sum(z[0] * z[1]) / np.sqrt(np.sum(z[0] * z[0]) * np.sum(z[1] * z[1]))
    assert abs(r[0, 1] - (1 - delta) * rho) <= 1e-17
    # N = 3: the three-variable formula r_ab.c = (s_ab - s_ac s_bc) / sqrt((1 - s_ac^2)(1 - s_bc^2)) on the
    # shrunk Sigma with its diagonal scaled to 1
    (x, _) = factor_series(3, 60, 0, 4)
    x[2] += x[0] - x[1]
    keep = np.ones(60, bool)
    (r, _, delta, _, _) = OP.subject_partial_ld(x, keep)
    xc = x.astype(LD) - np.sum(x.astype(LD), axis=1, keepdims=True) / LD(60)
    R = (xc @ xc.T) / np.sqrt(np.outer(np.sum(xc * xc, axis=1), np.sum(xc * xc, axis=1)))
    sig = (1 - delta) * R + delta * np.trace(R) / 3 * np.eye(3, dtype=LD)
    s = sig / np.sqrt(np.outer(np.diag(sig), np.diag(sig)))
    for (a, b, c) in ((0, 1, 2), (0, 2, 1), (1, 2, 0)):
        want = (s[a, b] - s[a, c] * s[b, c]) / np.sqrt((1 - s[a, c] ** 2) * (1 - s[b, c] ** 2))
        assert abs(r[a, b] - want) <= 1e-17 and r[a, b] == r[b, a]


def test_longdouble_pivots_are_the_squared_cholesky_diagonal():
    LD = np.longdouble
    (x, _) = factor_series(150, 170, 0, 9)             # three sweep blocks, the last partial
    (z, _) = OP.unit_rows_ld(x, np.ones(170, bool))
    (sigma, _) = OP.ledoit_wolf_ld(z, 0.0)
    (mP, piv) = OP.sweep_ld(sigma)
    L = np.zeros_like(sigma)
    for j in range(150):                                # left-looking Cholesky, column by column
        d = sigma[j, j] - np.sum(L[j, :j] * L[j, :j])
        L[j, j] = np.sqrt(d)
        L[j + 1:, j] = (sigma[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
    assert np.abs(piv / np.diag(L) ** 2 - 1).max() <= 1e-15
    assert piv.min() < 0.1                               # n_s = N + 20: small pivots late in the chain
    assert np.abs((-mP).astype(np.float64) @ sigma.astype(np.float64) - np.eye(150)).max() <= 1e-9
    # a singular matrix stops at its first pivot <= 0
    z[5] = z[2]
    (sigma, _) = OP.ledoit_wolf_ld(z, 0.0)
    (mP, piv) = OP.sweep_ld(sigma)
    assert mP is None and abs(piv[5]) <= 1e-17 and np.isnan(piv[6:].astype(np.float64)).all()
