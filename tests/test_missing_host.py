"""CPU: missing entries marginalised (``missing="marginalize"``).  The masked oracle (oracle/missing.py) against
brute-force enumeration over the observed entries only, the consequences of the marginalisation that can be
stated exactly (prior posteriors where nothing is observed, a missing control column is a dropped one), and the
argument checks of the fit, which run before any device work."""
import itertools

import numpy as np
import numpy.testing as nptest
import pytest
import scipy.special
import scipy.stats

from oracle import connections as OC
from oracle import iar_oracle as O
from oracle import missing as OM
from oracle import patients as OP


def _draw(N, H, U, seed, frac=0.2):
    """A draw of the model with a share ``frac`` of the entries of b and bt set to NaN (missing at random)."""
    rng = np.random.RandomState(seed)
    (_, _, _, _, b, bt) = O.sample(O.Theta(), N, H, U, rng)
    b = np.where(rng.uniform(size=b.shape) < frac, np.nan, b)
    bt = np.where(rng.uniform(size=bt.shape) < frac, np.nan, bt)
    return b, bt


def _one_hot_lq_F(C, seed):
    f = np.random.RandomState(seed).randint(0, 3, C)
    lq = np.full((C, 1, 3), -np.inf)
    lq[np.arange(C), 0, f] = 0.0
    return lq


def _brute_force(th, lq_F, x):
    """(log evidence (S,), log posterior over R (2^N, S), R): sum over all 2^N region configurations of
    p(R) prod over the OBSERVED entries of sum_k q_F[c,k] M_{k,l_c(R)}(x_c), with the densities of
    scipy.stats.norm and the missing entries dropped from the product."""
    C = x.shape[0]
    N = int(O.C_to_N(C))
    q_F = np.exp(lq_F)[:, 0, :]
    (n, m) = O.edge_pairs(N)
    R = np.array(list(itertools.product((0, 1), repeat=N)))
    lj = np.zeros((R.shape[0], x.shape[1]))
    for s in range(x.shape[1]):
        obs = np.flatnonzero(~np.isnan(x[:, s]))
        dens = np.stack([scipy.stats.norm.pdf(x[obs, s], th.mu[j], th.sigma[j]) for j in range(3)], axis=-1)
        for r in range(R.shape[0]):
            l = np.where(R[r, n[obs]] == R[r, m[obs]], R[r, n[obs]], 2)
            e = np.array([O.eval_M_eps(th.eta, th.epsilon, int(v)) for v in l])
            M = np.zeros(obs.size)
            for k in range(3):
                Mk = e * dens[:, k] + (1 - e) * 0.5 * (dens.sum(axis=1) - dens[:, k])
                M += q_F[obs, k] * Mk
            lj[r, s] = np.sum(np.where(R[r] == 1, np.log(th.pi), np.log(1 - th.pi))) + np.sum(np.log(M))
    ev = scipy.special.logsumexp(lj, axis=0)
    return ev, lj - ev, R


@pytest.mark.parametrize("N", [5, 6])
@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
def test_masked_oracle_equals_enumeration_over_the_observed_entries(N, lookup):
    """With q_F one-hot, the exact log-evidence of a patient minus the masked oracle's bound l_P is
    KL(q_R || p(R | x)), both over the observed entries only (the bound after the sweeps, for any q_R)."""
    th = O.Theta()
    C = N * (N - 1) // 2
    (_, x) = _draw(N, 2, 7, seed=N, frac=0.3)
    x[:, 0] = np.nan                                   # a subject with nothing observed
    x[[0, 1, 2], 1] = np.nan                           # a subject with region 0 and 1 partly missing
    lq_F = _one_hot_lq_F(C, N)
    (lq_R, terms) = OM.score_patients_masked(th, lq_F, x, edge_lookup=lookup, sweeps=6)
    (fe, _) = OP.free_energies(th, N, terms)
    (ev, lpost, R) = _brute_force(th, lq_F, x)
    lq = np.stack([lq_R[np.arange(N), :, R[r]].sum(axis=0) for r in range(R.shape[0])])
    kl = np.sum(np.exp(lq) * (lq - lpost), axis=0)
    nptest.assert_allclose(ev - (-fe), kl, atol=1e-10)
    assert np.all(kl > -1e-12)
    nptest.assert_allclose(ev[0], 0.0, atol=1e-12)     # nothing observed: the evidence is 1
    # and l_C over the observed entries
    lpc = [np.nansum(np.log(scipy.stats.norm.pdf(x[:, s], th.mu[np.argmax(lq_F[:, 0], 1)],
                                                 th.sigma[np.argmax(lq_F[:, 0], 1)]))) for s in range(x.shape[1])]
    nptest.assert_allclose(OM.control_loglik_masked(th, lq_F, x), lpc, rtol=1e-12, atol=1e-12)


def test_masked_caches_are_the_marginalised_densities():
    th = O.Theta()
    (b, bt) = _draw(6, 5, 7, seed=1)
    (lp, p, lM) = OM.update_lps_masked(b, bt, th)
    (lp0, p0, lM0) = O.update_lps(np.nan_to_num(b), np.nan_to_num(bt), th)
    nptest.assert_array_equal(lp[np.isnan(b)], 0.0)
    nptest.assert_array_equal(p[np.isnan(bt)], 1.0)
    nptest.assert_allclose(lM[np.isnan(bt)], 0.0, atol=1e-15)
    nptest.assert_array_equal(lp[~np.isnan(b)], lp0[~np.isnan(b)])
    nptest.assert_array_equal(lM[~np.isnan(bt)], lM0[~np.isnan(bt)])


def test_an_edge_missing_in_every_subject_keeps_the_prior_template():
    th = O.Theta()
    (b, bt) = _draw(7, 6, 8, seed=2)
    (b[4], bt[4]) = (np.nan, np.nan)
    (lp, p, lM) = OM.update_lps_masked(b, bt, th)
    (_, lq_R) = O.init_lps(7, 8)
    lq_R = np.log(np.random.RandomState(0).dirichlet([1, 1], size=(7, 8)))
    lq_F = O.update_lq_F(th.gamma, lp, lM, lq_R)
    nptest.assert_allclose(np.exp(lq_F[4, 0]), th.gamma, rtol=1e-14)
    out = OM.run_masked(b, bt, O.Theta(), max_iters=3, rel_tol=-1.0)
    assert np.all(np.isfinite(out["energy"]))


def test_a_region_with_all_edges_missing_keeps_the_prior_region_posterior():
    """Symmetric lookup: region n of patient u sees only its own edges, so with all of them missing q_R[n,u]
    is the prior (1 - pi, pi) after a sweep."""
    th = O.Theta()
    N = 7
    (b, bt) = _draw(N, 6, 8, seed=3, frac=0.0)
    (n, m) = O.edge_pairs(N)
    bt[(n == 2) | (m == 2), 5] = np.nan
    (lp, p, lM) = OM.update_lps_masked(b, bt, th)
    lq_F = O.update_lq_F(th.gamma, lp, lM, O.init_lps(N, 8)[1])
    lq_R = O.update_lq_R(np.array([1 - th.pi, th.pi]), lq_F, lM, O.init_lps(N, 8)[1], "symmetric")
    nptest.assert_allclose(np.exp(lq_R[2, 5]), [1 - th.pi, th.pi], rtol=1e-13)


def test_a_missing_control_column_is_a_dropped_control():
    (b, bt) = _draw(6, 7, 9, seed=4, frac=0.1)
    b2 = b.copy()
    b2[:, 3] = np.nan
    full = OM.run_masked(b2, bt, O.Theta(), max_iters=3, rel_tol=-1.0, polish=True)
    drop = OM.run_masked(np.delete(b, 3, axis=1), bt, O.Theta(), max_iters=3, rel_tol=-1.0, polish=True)
    nptest.assert_allclose(full["energy"], drop["energy"], rtol=1e-12)
    nptest.assert_allclose(full["lq_F"], drop["lq_F"], rtol=1e-10, atol=1e-12)
    nptest.assert_allclose(full["lq_R"], drop["lq_R"], rtol=1e-10, atol=1e-12)


def test_connection_posteriors_of_missing_entries_are_the_prior():
    """A missing element: P(T = 1) = w_1 + eta w_2, and F~ keeps the template state k with probability eps_l,
    i.e. the limit of the closed forms of oracle/connections.py at p = (1/3, 1/3, 1/3).  Observed elements are
    those of the unmasked oracle."""
    th = O.Theta()
    (_, bt) = _draw(6, 2, 9, seed=5, frac=0.3)
    lq_F = np.log(np.random.RandomState(1).dirichlet([1, 1, 1], size=(15, 1)))
    lq_R = np.log(np.random.RandomState(2).dirichlet([1, 1], size=(6, 9)))
    (qT, qFt) = OM.connection_posteriors_masked(th, lq_F, lq_R, bt)
    miss = np.isnan(bt)
    # oracle/connections.py evaluated at a correlation whose three densities are equal gives the prior
    th_flat = O.Theta()
    (th_flat.mu, th_flat.sigma) = (np.zeros(3), np.ones(3))
    (qT_flat, qFt_flat) = OC.connection_posteriors(th_flat, lq_F, lq_R, np.zeros(bt.shape))
    nptest.assert_allclose(qT[miss], qT_flat[miss], rtol=1e-13)
    nptest.assert_allclose(qFt[miss], qFt_flat[miss], rtol=1e-13)
    (qT0, qFt0) = OC.connection_posteriors(th, lq_F, lq_R, np.nan_to_num(bt))
    nptest.assert_array_equal(qT[~miss], qT0[~miss])
    nptest.assert_array_equal(qFt[~miss], qFt0[~miss])


def test_corr_oracle_marks_regions_without_a_time_series():
    rng = np.random.RandomState(0)
    ts = rng.normal(size=(3, 6, 40)).astype(np.float32)
    ts[0, 2, 5] = np.nan
    ts[1, 4, :] = 1.5
    ts[2, 0, 7] = np.inf
    out = OM.corr_fisherz_masked(ts)
    with np.errstate(invalid="ignore", divide="ignore"):
        ref = O.corr_fisherz(ts)
    (n, m) = O.edge_pairs(6)
    for (s, r) in ((0, 2), (1, 4), (2, 0)):
        hit = (n == r) | (m == r)
        assert np.all(np.isnan(out[hit, s]))
        nptest.assert_array_equal(out[~hit, s], ref[~hit, s])


# ------------------------------------------------------------------ argument checks (no device needed)
def _fit(N=5, H=4, U=3, missing="marginalize"):
    import fcdiff_b200 as fcdiff
    fit = fcdiff.fit.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    fit.missing = missing
    C = N * (N - 1) // 2
    (fit.b, fit.bt) = (np.zeros((C, H)), np.zeros((C, U)))
    return fit


def test_default_mode_rejects_nan_and_masked_mode_accepts_it():
    import fcdiff_b200 as fcdiff
    assert fcdiff.fit.UnsharedRegionFit().missing == "reject"
    fit = _fit(missing="reject")
    x = np.zeros((10, 2))
    x[3, 1] = np.nan
    fit._lq_F = np.full((10, 1, 3), -np.log(3))
    with pytest.raises(ValueError):
        fit.score_controls(x)
    with pytest.raises(ValueError):
        fit.classify_subjects(x, prior_patient=0.5)
    fit.missing = "marginalize"
    fit._check_finite(x, "x", allow_nan=fit._masked())          # accepted: the check is host-side


@pytest.mark.parametrize("missing", ["reject", "marginalize"])
@pytest.mark.parametrize("v", [np.inf, -np.inf])
def test_inf_is_rejected_in_both_modes(missing, v):
    fit = _fit(missing=missing)
    fit._lq_F = np.full((10, 1, 3), -np.log(3))
    x = np.zeros((10, 2))
    x[3, 1] = v
    with pytest.raises(ValueError):
        fit.score_controls(x)
    with pytest.raises(ValueError):
        fit.classify_subjects(x, prior_patient=0.5)
    if missing == "marginalize":
        with pytest.raises(ValueError):
            fit.score_patients(x)
        fit.bt = x.copy()
        with pytest.raises(ValueError, match="finite"):
            fit._ensure_inputs()


def test_masked_mode_rejects_what_it_does_not_cover():
    fit = _fit()
    fit.update_mu_sigma = True
    with pytest.raises(ValueError, match="update_mu_sigma"):
        fit.run()
    fit = _fit()
    fit.shards = object()
    with pytest.raises(ValueError, match="shards"):
        fit.run()
    fit = _fit()
    fit._lM = np.zeros((10, 3, 3, 3))
    with pytest.raises(ValueError, match="_lM"):
        fit._update_lq_F()
    fit = _fit()
    fit._lp_B_g_F = np.zeros((10, 4, 3))
    with pytest.raises(ValueError, match="_lp_B_g_F"):
        fit._eval_energy()
    fit = _fit(missing="nan")
    with pytest.raises(ValueError, match="missing"):
        fit.run()
