"""CPU: the NumPy oracle of the two-group read-outs (oracle/subjects.py) against the oracle's energy terms and
exact enumeration, the cross-validation folds, and the argument checks of ``UnsharedRegionFit.score_controls`` /
``classify_subjects``, which raise before any device work."""
import numpy as np
import numpy.testing as nptest
import pytest
import scipy.special

from oracle import iar_oracle as O
from oracle import patients as OP
from oracle import subjects as OS
from oracle.make_golden import golden_inputs


@pytest.mark.parametrize("N,H,U", [(10, 20, 20), (90, 50, 50)])
def test_control_loglik_sums_to_E_lp_B_g_F(N, H, U):
    (b, bt) = golden_inputs(N, H, U)
    th = O.Theta()
    out = O.run(b, bt, th, max_iters=2, rel_tol=-1.0)
    (lp_B_g_F, _, _) = O.update_lps(b, bt, th)
    got = OS.control_loglik(th, out["lq_F"], b)
    assert got.shape == (H,)
    nptest.assert_allclose(got.sum(), O.eval_E_lp_B_g_F(np.exp(out["lq_F"]), lp_B_g_F), rtol=1e-13)


def one_hot_lq_F(f):
    """log of a one-hot q_F (C, 1, 3) with exp(lq_F) exactly 0 off the template state."""
    return np.where(f, 0.0, -1000.0)[:, None, :]


@pytest.mark.parametrize("N", [5, 6])
@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
def test_bound_gap_is_the_kl_of_q_R(N, lookup):
    """One-hot q_F: exact log-evidence - l_P = KL(q_R || p(R | x)) for any mean-field q_R, here the q_R of three
    sweeps from the uniform start; and l_C is the exact control log-likelihood."""
    th = O.Theta(pi=0.2, eta=0.4)
    (_, _, f, _, b, bt) = O.sample(th, N, 7, 9, np.random.RandomState(N))
    lq_F = one_hot_lq_F(f)
    (lq_R, _) = OP.score_patients(th, lq_F, bt, None, lookup, sweeps=3)
    (log_odds, control, elbo) = OS.classify(th, lq_F, bt, 0.3, lq_R)
    exact = OS.exact_log_evidence_patient(th, lq_F, bt)
    kl = OS.kl_qR(lq_R, th, lq_F, bt)
    assert np.all(kl >= -1e-12) and np.any(kl > 1e-6)
    nptest.assert_allclose(exact - elbo, kl, rtol=0, atol=1e-10)
    nptest.assert_allclose(log_odds, elbo - control + np.log(0.3 / 0.7), rtol=1e-15, atol=1e-12)
    for x in (b, bt):
        nptest.assert_allclose(OS.control_loglik(th, lq_F, x), OS.exact_log_evidence_control(th, lq_F, x),
                               rtol=1e-14)
    (R, lpost) = OS.exact_posterior_R(th, lq_F, bt)
    assert R.shape == (2 ** N, N)
    nptest.assert_allclose(np.exp(lpost).sum(axis=0), 1.0, rtol=1e-13)


def test_exact_posterior_probabilities_are_calibrated():
    """Over subjects drawn from the two-group mixture with the true theta and F, the mean of the exact
    P(patient | x) is the prior rho (tower property); checked to three standard errors."""
    (N, S, rho) = (5, 4000, 0.3)
    th = O.Theta(pi=0.2, eta=0.4)
    rng = np.random.RandomState(5)
    n_pat = rng.binomial(S, rho)
    (_, _, f, _, b, bt) = O.sample(th, N, S - n_pat, n_pat, rng)
    lq_F = one_hot_lq_F(f)
    x = np.concatenate([b, bt], axis=1)
    log_odds = (OS.exact_log_evidence_patient(th, lq_F, x) - OS.exact_log_evidence_control(th, lq_F, x) +
                np.log(rho / (1 - rho)))
    p = scipy.special.expit(log_odds)
    se = p.std() / np.sqrt(S)
    assert abs(p.mean() - rho) < 3 * se, (p.mean(), rho, se)
    assert p[S - n_pat:].mean() > p[:S - n_pat].mean()


# ------------------------------------------------------------------ folds
def test_stratified_folds():
    from fcdiff_b200.sweep import stratified_folds
    labels = np.zeros(103, dtype=bool)
    labels[np.random.RandomState(1).permutation(103)[:41]] = True
    fold = stratified_folds(labels, 5, seed=3)
    assert fold.shape == (103,) and set(fold.tolist()) == set(range(5))       # a partition into five folds
    for cls in (False, True):
        counts = np.bincount(fold[labels == cls], minlength=5)
        assert counts.max() - counts.min() <= 1 and counts.sum() == (labels == cls).sum()
    sizes = np.bincount(fold, minlength=5)
    assert sizes.max() - sizes.min() <= 1
    nptest.assert_array_equal(fold, stratified_folds(labels, 5, seed=3))
    assert not np.array_equal(fold, stratified_folds(labels, 5, seed=4))
    with pytest.raises(ValueError):
        stratified_folds(labels, 1)
    with pytest.raises(ValueError):
        stratified_folds(np.arange(10) < 3, 5)


# ------------------------------------------------------------------ argument checks (no device needed)
def _fit(N=6, S=4):
    import fcdiff_b200 as fcdiff
    fit = fcdiff.fit.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    C = N * (N - 1) // 2
    fit._lq_F = np.full((C, 1, 3), -np.log(3))
    return fit, np.zeros((C, S))


def test_checks_reject_wrong_shapes():
    (fit, x) = _fit()
    for bad in (x[1:], x[:, 0], x[:, :0]):
        with pytest.raises(ValueError):
            fit.score_controls(bad)
        with pytest.raises(ValueError):
            fit.classify_subjects(bad, prior_patient=0.5)


def test_checks_reject_non_finite_input():
    (fit, x) = _fit()
    for v in (np.nan, np.inf):
        y = x.copy()
        y[2, 1] = v
        with pytest.raises(ValueError):
            fit.score_controls(y)
        with pytest.raises(ValueError):
            fit.classify_subjects(y, prior_patient=0.5)


def test_checks_on_the_prior():
    (fit, x) = _fit()
    for rho in (0.0, 1.0, -0.1, 1.5, np.nan):
        with pytest.raises(ValueError):
            fit.classify_subjects(x, prior_patient=rho)
    with pytest.raises(ValueError):                  # a fit assembled from theta and q_F has no cohort
        fit.classify_subjects(x)


def test_checks_reject_a_sharded_fit():
    (fit, x) = _fit()
    fit.shards = object()
    with pytest.raises(ValueError):
        fit.score_controls(x)
    with pytest.raises(ValueError):
        fit.classify_subjects(x, prior_patient=0.5)


def test_checks_reject_arrays_mode():
    (fit, x) = _fit()
    fit._lp_B_g_F = np.zeros((x.shape[0], 3, 3))
    with pytest.raises(ValueError):
        fit.score_controls(x)
    with pytest.raises(ValueError):
        fit.classify_subjects(x, prior_patient=0.5)
    (fit, x) = _fit()
    fit._lM = np.zeros((x.shape[0], x.shape[1], 3, 3))
    with pytest.raises(ValueError):
        fit.classify_subjects(x, prior_patient=0.5)


def test_score_controls_needs_controls():
    (fit, _) = _fit()
    with pytest.raises(ValueError):
        fit.score_controls()
