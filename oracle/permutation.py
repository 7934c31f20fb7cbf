"""
TEST INFRASTRUCTURE ONLY -- NumPy restatements of the Westfall-Young step-down max-T
p-values (``fcdiff_b200.sweep.maxt_pvalues``, csrc/fcd_permutation.cu) and a sampler
with anomalous regions planted at chosen places.

T is (R1, K): row 0 the observed statistics, rows 1.. those of relabelled data
(exchangeable under H0).  Within a family of columns F, one-sided (large values
are evidence against H0):

    p[k]      = #{r : T[r,k] >= T[0,k]} / R1
    p_fwer    step-down max-T (Westfall & Young 1993, algorithm 4.1): columns in
              descending order of the observed value, successive maxima over the
              columns not yet passed, then monotone enforcement.

``maxt_pvalues_literal`` is that algorithm written as loops; ``maxt_pvalues`` the
vectorised restatement the kernel implements: with sigma ordering F ascending by
(T[0,k], k), count_sd[j] = #{r : max_{i <= j} T[r,sigma(i)] >= T[0,sigma(j)]} and
p_fwer[sigma(j)] = max_{i >= j} count_sd[i] / R1.
"""
import numpy as np

from . import iar_oracle as O


def _families(K, families):
    return [(0, K)] if families is None else [(int(a), int(b)) for (a, b) in families]


def maxt_pvalues_literal(T, families=None):
    """(p, p_fwer) (K,) float64 from the descending-order step-down, as loops."""
    T = np.asarray(T, dtype=np.float64)
    (R1, K) = T.shape
    p = np.full(K, np.nan)                      # NaN outside every family
    p_fwer = np.full(K, np.nan)
    for (k0, k1) in _families(K, families):
        cols = list(range(k0, k1))
        for k in cols:
            n = 0
            for r in range(R1):
                if T[r, k] >= T[0, k]:
                    n += 1
            p[k] = n / R1
        # descending observed value; ties in column order (any tie order gives the same p_fwer)
        desc = sorted(cols, key=lambda k: -T[0, k])
        m = len(desc)
        count = [0] * m
        u = [-np.inf] * R1                      # successive maxima from the least significant column up
        for j in range(m - 1, -1, -1):
            k = desc[j]
            for r in range(R1):
                u[r] = max(u[r], T[r, k])
            count[j] = sum(1 for r in range(R1) if u[r] >= T[0, k])
        prev = 0.0
        for j in range(m):
            prev = max(prev, count[j] / R1)
            p_fwer[desc[j]] = prev
    return p, p_fwer


def maxt_pvalues(T, families=None):
    """(p, p_fwer) (K,) float64 from the prefix-max restatement (vectorised)."""
    T = np.asarray(T, dtype=np.float64)
    (R1, K) = T.shape
    p = np.full(K, np.nan)                      # NaN outside every family
    p_fwer = np.full(K, np.nan)
    for (k0, k1) in _families(K, families):
        X = T[:, k0:k1]
        obs = X[0]
        sigma = np.lexsort((np.arange(k1 - k0), obs))
        pm = np.maximum.accumulate(X[:, sigma], axis=1)
        count_sd = (pm >= obs[sigma]).sum(axis=0)
        count_unc = (X >= obs).sum(axis=0)
        p[k0:k1] = count_unc / R1
        p_fwer[k0 + sigma] = np.maximum.accumulate(count_sd[::-1])[::-1] / R1
    return p, p_fwer


def sample_planted(th, N, H, U, pi_region, rng):
    """``iar_oracle.sample`` with a per-region P(region anomalous): pi_region (N,).  With pi_region constant at
    th.pi it draws the same numbers in the same order and returns O.sample's arrays bit for bit."""
    pi_region = np.asarray(pi_region, dtype=np.float64).reshape(N)
    C = O.N_to_C(N)
    n, m = O.edge_pairs(N)
    r = rng.binomial(1, np.broadcast_to(pi_region[:, None], (N, U)), (N, U)) > 0
    both = r[n] & r[m]
    neither = ~r[n] & ~r[m]
    coin = rng.binomial(1, th.eta, (C, U)) > 0
    t = np.where(both, True, np.where(neither, False, coin))
    f = rng.multinomial(1, th.gamma, C) > 0
    e = th.epsilon
    fk = np.argmax(f, axis=1)
    p_keep = np.where(t, e, 1 - e)
    u1 = rng.uniform(size=(C, U))
    u2 = rng.uniform(size=(C, U))
    keep = u1 < p_keep
    other = (fk[:, None] + 1 + (u2 < 0.5)) % 3
    ftk = np.where(keep, fk[:, None], other)
    f_tilde = np.zeros((C, U, 3), dtype=bool)
    np.put_along_axis(f_tilde, ftk[:, :, None], True, axis=2)
    b = rng.normal(th.mu[fk][:, None], th.sigma[fk][:, None], (C, H)).clip(-1, 1)
    b_tilde = rng.normal(th.mu[ftk], th.sigma[ftk]).clip(-1, 1)
    return r, t, f, f_tilde, b, b_tilde
