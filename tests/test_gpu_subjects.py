"""GPU: held-out control log-likelihoods, the two-group classifier and cross-validation
(``UnsharedRegionFit.score_controls`` / ``classify_subjects``, ``sweep.cross_validate``, csrc/fcd_patients.cu)
against the NumPy oracle (oracle/subjects.py), exact enumeration, the fit's own energy terms and
``score_patients``."""
import ctypes

import numpy as np
import numpy.testing as nptest
import pytest
import scipy.special
import scipy.stats
import torch

from oracle import iar_oracle as O
from oracle import subjects as OS
from oracle.make_golden import golden_inputs

pytestmark = pytest.mark.gpu

import fcdiff_b200 as fcdiff          # noqa: E402
from fcdiff_b200 import _dev, _lib, sweep    # noqa: E402

F = fcdiff.fit


@pytest.fixture(scope="module", autouse=True)
def _native_library_loaded():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    lib = _lib.load()
    n0 = lib.fcd_launch_count()
    yield
    assert lib.fcd_launch_count() > n0, "no kernel of libfcdiff_b200.so was launched"


def _run_fit(b, bt, iters, lookup="reference"):
    fit = F.UnsharedRegionFit()
    fit.b, fit.bt = b, bt
    fit.model = fcdiff.UnsharedRegionModel()
    fit.edge_lookup = lookup
    fit.max_iters = iters
    fit.rel_tol = -1.0
    fit.run()
    return fit


def _fit_at(th, lq_F, lookup):
    """A fit that holds only theta and q_F."""
    fit = F.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    (fit.model.pi, fit.model.eta, fit.model.epsilon) = (th.pi, th.eta, th.epsilon)
    (fit.model.gamma, fit.model.mu, fit.model.sigma) = (th.gamma.copy(), th.mu.copy(), th.sigma.copy())
    fit.edge_lookup = lookup
    fit._lq_F = lq_F
    return fit


def _theta_of(model):
    return O.Theta(pi=float(model.pi), eta=float(model.eta), gamma=np.array(model.gamma, dtype=np.float64),
                   epsilon=float(model.epsilon), mu=np.array(model.mu, dtype=np.float64),
                   sigma=np.array(model.sigma, dtype=np.float64))


_FITTED = {}


def _fitted_state(N):
    """theta and a peaked q_F of a fit on training data of N regions (cached per module)."""
    if N not in _FITTED:
        (_, _, _, _, b, bt) = O.sample(O.Theta(), N, 30, 40, np.random.RandomState(N + 7))
        fit = _run_fit(b, bt, 4)
        _FITTED[N] = (_theta_of(fit.model), fit._lq_F.copy())
    return _FITTED[N]


def _state(N, qF_kind):
    if qF_kind == "fitted":
        return _fitted_state(N)
    rng = np.random.RandomState(2 * N)
    return O.Theta(), np.log(rng.dirichlet([1, 1, 1], size=(N * (N - 1) // 2, 1)))


def _auc(score_pos, score_neg):
    """Mann-Whitney AUC: the probability that a positive outscores a negative (ties count half)."""
    s = np.concatenate([score_pos, score_neg])
    ranks = scipy.stats.rankdata(s)
    n1 = len(score_pos)
    return (ranks[:n1].sum() - n1 * (n1 + 1) / 2.0) / (n1 * len(score_neg))


# ------------------------------------------------------------------ score_controls against the oracle
@pytest.mark.parametrize("N", [10, 90])
@pytest.mark.parametrize("S", [1, 31, 45])
@pytest.mark.parametrize("qF_kind", ["random", "fitted"])
@pytest.mark.parametrize("where", ["host", "cuda"])
def test_score_controls_parity_with_oracle(N, S, qF_kind, where):
    """S < 32 takes several row blocks per warp; odd S pads the device columns (pitchS = S + 1)."""
    (th, lq_F) = _state(N, qF_kind)
    (_, _, _, _, b, _) = O.sample(O.Theta(), N, S, 1, np.random.RandomState(N + S))
    fit = _fit_at(th, lq_F, "reference")
    got = fit.score_controls(b if where == "host" else torch.from_numpy(b).cuda())
    assert got.shape == (S,) and got.dtype == np.float64
    nptest.assert_allclose(got, OS.control_loglik(th, lq_F, b), rtol=1e-12)


def test_sums_equal_the_fit_energy_term():
    """score_controls() of a fit's own controls adds up to K4's E_lp_B_g_F (from the control sums S1 / S2)."""
    (b, bt) = golden_inputs(90, 50, 50)
    fit = _run_fit(b, bt, 3)
    assert not fit.update_mu_sigma
    got = fit.score_controls()
    assert got.shape == (50,)
    nptest.assert_allclose(got.sum(), fit._energy_terms()[1], rtol=1e-11)
    nptest.assert_array_equal(got, fit.score_controls(b))


def test_sums_equal_the_fit_energy_term_in_replica_mode():
    (b, bt) = golden_inputs(90, 50, 50)
    corr = torch.from_numpy(np.concatenate([bt[:, :20], b, bt[:, 20:]], axis=1)).cuda()
    con = np.arange(20, 70)
    pat = np.concatenate([np.arange(20), np.arange(70, 100)])
    model = fcdiff.UnsharedRegionModel()
    fit = F.UnsharedRegionFit()
    fit.model = model
    fit.max_iters = 3
    fit.rel_tol = -1.0
    fit.set_shared_inputs(sweep.SharedPlanes(corr, model), con, pat)
    fit.run()
    got = fit.score_controls()
    nptest.assert_allclose(got.sum(), fit._energy_terms()[1], rtol=1e-11)
    nptest.assert_array_equal(got, fit.score_controls(b))


def test_batch_pitch_invariance_and_determinism():
    (th, lq_F) = _fitted_state(90)
    (_, _, _, _, b, _) = O.sample(O.Theta(), 90, 45, 1, np.random.RandomState(61))
    fit = _fit_at(th, lq_F, "reference")
    whole = fit.score_controls(b)
    nptest.assert_array_equal(whole, fit.score_controls(b))
    for s in (0, 17, 44):
        nptest.assert_array_equal(fit.score_controls(b[:, s:s + 1]), whole[s:s + 1])
    perm = np.random.RandomState(62).permutation(45)
    nptest.assert_array_equal(fit.score_controls(b[:, perm]), whole[perm])
    # any pitch: the columns at a pitch of 64
    lib = _lib.load()
    (C, S, pitchS) = (b.shape[0], 45, 64)
    X = _dev.zeros((C, pitchS))
    X[:, :S].copy_(torch.from_numpy(b))
    out = _dev.empty((S,))
    ws = _dev.empty((int(lib.fcd_control_terms_ws_bytes(C, S)) // 8,))
    th_c = fit._theta(use_snapshot=False)
    _lib.check(lib.fcd_control_terms(_dev.ptr(X), C, S, pitchS, _dev.ptr(fit._mF.get_dev()[1]), ctypes.byref(th_c),
                                     _dev.ptr(out), _dev.ptr(ws), 0, _dev.stream()), "fcd_control_terms")
    nptest.assert_array_equal(out.cpu().numpy(), whole)


# ------------------------------------------------------------------ classify_subjects
def test_classify_is_score_patients_plus_score_controls():
    (th, lq_F) = _fitted_state(90)
    (_, _, _, _, b, bt) = O.sample(O.Theta(), 90, 20, 25, np.random.RandomState(71))
    x = np.concatenate([b, bt], axis=1)
    fit = _fit_at(th, lq_F, "symmetric")
    c = fit.classify_subjects(x, prior_patient=0.3)
    s = fit.score_patients(x)
    nptest.assert_array_equal(c.lq_R, s.lq_R)
    assert (c.sweeps, c.max_change) == (s.sweeps, s.max_change)
    ctrl = fit.score_controls(x)
    nptest.assert_array_equal(c.control_loglik, ctrl)
    nptest.assert_array_equal(c.patient_elbo, -s.free_energy)
    nptest.assert_array_equal(c.log_odds, (-s.free_energy - ctrl) + scipy.special.logit(0.3))
    nptest.assert_array_equal(c.p_patient, scipy.special.expit(c.log_odds))
    c2 = fit.classify_subjects(torch.from_numpy(x).cuda(), prior_patient=0.8)
    shift = scipy.special.logit(0.8) - scipy.special.logit(0.3)
    nptest.assert_allclose(c2.log_odds - c.log_odds, shift, rtol=0, atol=1e-12 * np.abs(c.log_odds).max())
    nptest.assert_array_equal(c2.control_loglik, c.control_loglik)
    nptest.assert_array_equal(c2.patient_elbo, c.patient_elbo)


def test_log_odds_gap_is_the_kl_of_q_R():
    """N = 6, one-hot q_F (the template known): l_C is exact and l_P lies below the exact log-evidence of the
    patient model by KL(q_R || p(R | x)), so the GPU log-odds are below the exact ones by exactly that."""
    th = O.Theta(pi=0.2, eta=0.4)
    (_, _, f, _, b, bt) = O.sample(th, 6, 12, 20, np.random.RandomState(81))
    lq_F = np.where(f, 0.0, -1000.0)[:, None, :]
    x = np.concatenate([b, bt], axis=1)
    fit = _fit_at(th, lq_F, "symmetric")
    c = fit.classify_subjects(x, prior_patient=0.4)
    nptest.assert_allclose(c.control_loglik, OS.exact_log_evidence_control(th, lq_F, x), rtol=1e-12)
    exact = (OS.exact_log_evidence_patient(th, lq_F, x) - OS.exact_log_evidence_control(th, lq_F, x) +
             np.log(0.4 / 0.6))
    gap = exact - c.log_odds
    assert np.all(gap >= -1e-9), gap.min()
    nptest.assert_allclose(gap, OS.kl_qR(c.lq_R, th, lq_F, x), rtol=0, atol=1e-9)


def test_held_out_subjects_are_classified():
    """90 regions; a 10-iteration fit on 50 + 50 subjects, then 50 + 50 held-out subjects of the same draw
    (same template F) are classified at the default prior."""
    (_, _, _, _, b, bt) = O.sample(O.Theta(), 90, 100, 100, np.random.RandomState(91))
    fit = _run_fit(b[:, :50], bt[:, :50], 10, "symmetric")
    c = fit.classify_subjects(np.concatenate([b[:, 50:], bt[:, 50:]], axis=1))
    auc = _auc(c.log_odds[50:], c.log_odds[:50])
    acc = float(np.mean((c.p_patient > 0.5) == (np.arange(100) >= 50)))
    print("held-out AUC %.4f accuracy %.3f" % (auc, acc))
    assert auc >= 0.99, auc


@pytest.mark.parametrize("call", ["score_controls", "classify_subjects"])
def test_the_fit_is_untouched(call):
    (b, bt) = golden_inputs(90, 50, 50)
    (f1, f2) = (_run_fit(b, bt, 3), _run_fit(b, bt, 3))
    before = (f1.model.pi, f1.model.eta, f1.model.epsilon, f1.model.gamma.copy(), f1.model.mu.copy(),
              f1.model.sigma.copy(), f1._lq_F.copy(), f1._lq_R.copy(), list(f1.energy))
    inp = f1._in
    (_, _, _, _, x, _) = O.sample(O.Theta(), 90, 33, 1, np.random.RandomState(41))
    if call == "score_controls":
        f1.score_controls()
        f1.score_controls(x)
    else:
        f1.classify_subjects(x, max_sweeps=5)
    after = (f1.model.pi, f1.model.eta, f1.model.epsilon, f1.model.gamma, f1.model.mu, f1.model.sigma,
             f1._lq_F, f1._lq_R, f1.energy)
    for (u, v) in zip(before, after):
        nptest.assert_array_equal(u, v)
    assert f1._in is inp
    f1._update_lq_R()
    f2._update_lq_R()
    nptest.assert_array_equal(f1._lq_R, f2._lq_R)


# ------------------------------------------------------------------ cross-validation
def _cv_problem():
    (b, bt) = golden_inputs(90, 50, 50)
    perm = np.random.RandomState(101).permutation(100)
    corr = np.concatenate([b, bt], axis=1)[:, perm]
    labels = (np.arange(100) >= 50)[perm]
    return corr, labels


def test_cross_validate_matches_folds_fitted_by_hand():
    (corr, labels) = _cv_problem()
    opts = dict(max_iters=5, rel_tol=-1.0)
    cv = sweep.cross_validate(corr, labels, n_folds=5, seed=2, fit_options=opts, streams=1)
    fold = cv["fold"]
    nptest.assert_array_equal(fold, sweep.stratified_folds(labels, 5, 2))
    assert np.bincount(fold, minlength=5).sum() == 100 and len(cv["folds"]) == 5
    for name in ("log_odds", "p_patient", "control_loglik", "patient_elbo"):
        assert cv[name].shape == (100,) and np.all(np.isfinite(cv[name]))
    dev = _dev.device()
    corr_dev = torch.from_numpy(corr).to(dev)
    model = fcdiff.UnsharedRegionModel()
    shared = sweep.SharedPlanes(corr_dev, model)
    for i in range(5):
        train = fold != i
        fit = F.UnsharedRegionFit()
        fit.model = fcdiff.UnsharedRegionModel()
        (fit.max_iters, fit.rel_tol) = (5, -1.0)
        fit.set_shared_inputs(shared, np.flatnonzero(train & ~labels), np.flatnonzero(train & labels))
        fit.run()
        held = np.flatnonzero(fold == i)
        c = fit.classify_subjects(corr_dev.index_select(1, torch.from_numpy(held).to(dev)))
        for name in ("log_odds", "p_patient", "control_loglik", "patient_elbo"):
            nptest.assert_array_equal(cv[name][held], getattr(c, name))
        assert cv["folds"][i]["free_energy"] == fit.energy[-1]
        assert cv["folds"][i]["eta"] == fit.model.eta and cv["folds"][i]["epsilon"] == fit.model.epsilon
    cv2 = sweep.cross_validate(corr, labels, n_folds=5, seed=2, fit_options=opts, streams=2)
    for name in ("fold", "log_odds", "p_patient", "control_loglik", "patient_elbo"):
        nptest.assert_array_equal(cv2[name], cv[name])
    assert [f["free_energy"] for f in cv2["folds"]] == [f["free_energy"] for f in cv["folds"]]
