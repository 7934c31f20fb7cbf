"""CPU: the NumPy oracle of the connection posteriors (oracle/connections.py) against brute-force enumeration of
the generative model, its calibration at the truth, planted recovery, and the argument checks of
``UnsharedRegionFit.connection_posteriors``, which raise before any device work."""
import numpy as np
import pytest
from scipy.stats import rankdata

from oracle import connections as OC
from oracle import iar_oracle as O
from oracle import patients as OP

PAIRS = {0: (0, 0), 1: (1, 1), 2: (0, 1)}       # pair state l -> states of regions (1, 0) of the one edge of N = 2


def _one_edge(k, l, U):
    """lq_F one-hot on k and lq_R of N = 2 regions whose pair is in state l."""
    lq_F = np.full((1, 1, 3), -np.inf)
    lq_F[0, 0, k] = 0.0
    q_R = np.zeros((2, U, 2))
    (s1, s0) = PAIRS[l]
    q_R[1, :, s1] = 1.0
    q_R[0, :, s0] = 1.0
    with np.errstate(divide="ignore"):
        return lq_F, np.log(q_R)


@pytest.mark.parametrize("theta,tol", [
    (dict(), 1e-14),
    (dict(eta=1 - 1e-5, epsilon=1e-5), 2e-11),
    (dict(eta=1e-5, epsilon=1 - 1e-5), 2e-11),
    (dict(epsilon=1e-7), 2e-9)])
def test_oracle_equals_enumeration(theta, tol):
    """Measured largest differences: 5e-15 at the default theta, 9e-12 and 8e-12 with (eta, epsilon) on the
    optimiser's bounds, 3.7e-10 at epsilon = 1e-7.  The growth is the plane form a_l + b_l p_k, ill-conditioned
    at extreme epsilon where p_k is near 1, not an error in the formula."""
    th = O.Theta(**theta)
    x = np.linspace(-0.4, 0.5, 20)
    for k in range(3):
        for l in range(3):
            (lq_F, lq_R) = _one_edge(k, l, x.size)
            (q_T, q_Ft) = OC.connection_posteriors(th, lq_F, lq_R, x[None, :])
            (e_T, e_F) = OC.exact_conditionals(th, x, k, l)
            np.testing.assert_allclose(q_T[0], e_T, rtol=0, atol=tol, err_msg="k=%d l=%d" % (k, l))
            np.testing.assert_allclose(q_Ft[0], e_F, rtol=0, atol=tol, err_msg="k=%d l=%d" % (k, l))


def _truth_draw():
    th = O.Theta(pi=0.1, eta=0.5)
    (r, t, f, f_tilde, b, bt) = O.sample(th, 20, 30, 2000, np.random.RandomState(7))
    with np.errstate(divide="ignore"):
        lq_F = np.log(f[:, None, :].astype(np.float64))
        lq_R = np.log(np.stack([~r, r], axis=-1).astype(np.float64))
    return th, t, f, f_tilde, lq_F, lq_R, bt


def test_calibration_at_the_truth():
    """q_F and q_R one-hot at the sampled truth, 380,000 connections: mean q_T 0.10033 against a sampled mean t of
    0.10026, mean P(F~ != F) 0.12407 against 0.12401 (the standard error of the mean of t is about 5e-4)."""
    (th, t, f, f_tilde, lq_F, lq_R, bt) = _truth_draw()
    (q_T, q_Ft) = OC.connection_posteriors(th, lq_F, lq_R, bt)
    assert np.abs(q_Ft.sum(axis=-1) - 1).max() <= 1e-13
    assert q_T.min() >= 0.0 and q_T.max() <= 1.0
    fk = np.argmax(f, axis=1)
    changed = 1.0 - np.take_along_axis(q_Ft, fk[:, None, None].repeat(bt.shape[1], 1), axis=2)[:, :, 0]
    assert abs(q_T.mean() - t.mean()) <= 2e-3
    assert abs(changed.mean() - (np.argmax(f_tilde, axis=-1) != fk[:, None]).mean()) <= 2e-3


def auc(score, label):
    """Area under the ROC curve (Mann-Whitney U over midranks)."""
    (s, y) = (np.ravel(score), np.ravel(label).astype(bool))
    rk = rankdata(s)
    (n1, n0) = (int(y.sum()), int((~y).sum()))
    return (rk[y].sum() - n1 * (n1 + 1) / 2.0) / (n1 * n0)


def planted_draw():
    """The draw of the planted recovery tests (here and in test_gpu_connections.py): 20 regions, 30 controls,
    120 patients with pi = 0.1, eta = 0.5; fitted on the first 60 patients, the other 60 held out."""
    return O.sample(O.Theta(pi=0.1, eta=0.5), 20, 30, 120, np.random.RandomState(12)), 60


def test_oracle_recovers_planted_connections():
    """A 10-iteration symmetric-lookup oracle fit on 60 patients, the held-out 60 scored with 50 sweeps.  Measured
    here: AUC of q_T against t 0.9974 (cohort) and 0.9967 (held out); argmax q_F~ against f~ 0.9976 and 0.9982."""
    ((r, t, f, f_tilde, b, bt), Ut) = planted_draw()
    th = O.Theta()
    out = O.run(b, bt[:, :Ut], th, max_iters=10, rel_tol=-1.0, edge_lookup="symmetric", polish=True)
    (lq_R_held, _) = OP.score_patients(th, out["lq_F"], bt[:, Ut:], None, "symmetric", sweeps=50)
    for (lq_R, cols) in ((out["lq_R"], slice(0, Ut)), (lq_R_held, slice(Ut, None))):
        (q_T, q_Ft) = OC.connection_posteriors(th, out["lq_F"], lq_R, bt[:, cols])
        assert auc(q_T, t[:, cols]) > 0.99
        assert (np.argmax(q_Ft, axis=-1) == np.argmax(f_tilde[:, cols], axis=-1)).mean() > 0.99
        assert np.abs(q_Ft.sum(axis=-1) - 1).max() <= 1e-13


# ------------------------------------------------------------------ argument checks (no device needed)
def _fit(N=6, U=4):
    import fcdiff_b200 as fcdiff
    fit = fcdiff.fit.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    C = N * (N - 1) // 2
    fit._lq_F = np.full((C, 1, 3), -np.log(3))
    fit._lq_R = np.full((N, U, 2), -np.log(2))
    fit.bt = np.zeros((C, U))
    return fit, np.zeros((C, U)), np.full((N, U, 2), -np.log(2))


def test_connection_posteriors_takes_bt_new_and_lq_R_together():
    (fit, bt, lq_R) = _fit()
    with pytest.raises(ValueError):
        fit.connection_posteriors(bt)
    with pytest.raises(ValueError):
        fit.connection_posteriors(lq_R=lq_R)


def test_connection_posteriors_rejects_wrong_shapes():
    (fit, bt, lq_R) = _fit()
    with pytest.raises(ValueError):
        fit.connection_posteriors(bt[1:], lq_R)
    with pytest.raises(ValueError):
        fit.connection_posteriors(bt[:, 0], lq_R)
    with pytest.raises(ValueError):
        fit.connection_posteriors(bt, lq_R[:, :3])
    with pytest.raises(ValueError):
        fit.connection_posteriors(bt, lq_R[1:])
    fit._lq_R = lq_R[:, :3]                     # the fit's own q_R does not match its patients
    with pytest.raises(ValueError):
        fit.connection_posteriors()


def test_connection_posteriors_rejects_a_sharded_fit():
    (fit, bt, lq_R) = _fit()
    fit.shards = object()
    with pytest.raises(ValueError):
        fit.connection_posteriors()
    with pytest.raises(ValueError):
        fit.connection_posteriors(bt, lq_R)


@pytest.mark.parametrize("name", ["_lM", "_lp_B_g_F", "_p_Bt_g_Ft"])
def test_connection_posteriors_rejects_arrays_mode(name):
    (fit, bt, lq_R) = _fit()
    setattr(fit, name, np.zeros(1))
    with pytest.raises(ValueError):
        fit.connection_posteriors(bt, lq_R)


def test_connection_posteriors_needs_a_model_q_F_q_R_and_patients():
    import fcdiff_b200 as fcdiff
    (fit, bt, lq_R) = _fit()
    fit.model = None
    with pytest.raises(ValueError):
        fit.connection_posteriors()
    fit = fcdiff.fit.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    with pytest.raises(ValueError):
        fit.connection_posteriors(bt, lq_R)
    fit._lq_F = np.full((bt.shape[0], 1, 3), -np.log(3))
    with pytest.raises(ValueError):               # no q_R
        fit.connection_posteriors()
    fit._lq_R = lq_R
    with pytest.raises(ValueError):               # no patients
        fit.connection_posteriors()


def test_connection_posteriors_is_reachable_through_the_alias():
    import fcdiff
    assert fcdiff.fit.ConnectionPosteriors._fields == ("q_T", "q_F_tilde", "expected_anomalous", "anomalous_rate")
    assert hasattr(fcdiff.fit.UnsharedRegionFit, "connection_posteriors")
