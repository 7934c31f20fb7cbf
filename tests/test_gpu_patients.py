"""GPU: scoring held-out patients with a fitted model (``UnsharedRegionFit.score_patients``,
csrc/fcd_patients.cu) against the package's own region step and energy terms, the NumPy oracle
(oracle/patients.py) and planted anomalies."""
import numpy as np
import numpy.testing as nptest
import pytest
import torch

from oracle import iar_oracle as O
from oracle import patients as OP
from oracle.make_golden import golden_inputs

pytestmark = pytest.mark.gpu

import fcdiff_b200 as fcdiff          # noqa: E402
from fcdiff_b200 import _dev, _lib    # noqa: E402

F = fcdiff.fit


@pytest.fixture(scope="module", autouse=True)
def _native_library_loaded():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    lib = _lib.load()
    n0 = lib.fcd_launch_count()
    yield
    assert lib.fcd_launch_count() > n0, "no kernel of libfcdiff_b200.so was launched"


def _run_fit(b, bt, iters, lookup):
    fit = F.UnsharedRegionFit()
    fit.b, fit.bt = b, bt
    fit.model = fcdiff.UnsharedRegionModel()
    fit.edge_lookup = lookup
    fit.max_iters = iters
    fit.rel_tol = -1.0
    fit.run()
    return fit


def _fit_at(th, lq_F, lookup):
    """A fit that holds only theta and q_F: enough to score patients."""
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


def _lM_of(th, bt):
    p = np.stack([O.norm_pdf(bt, th.mu[k], th.sigma[k]) for k in range(3)], axis=-1)
    return O.lM_from_p(p, th.eta, th.epsilon)


# ------------------------------------------------------------------ against the package's own steps
@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
def test_one_sweep_reproduces_update_lq_R(lookup):
    """Same planes, kernels and launch shape as `_update_lq_R`; only exp(lq_R) of the start is formed on the
    host here (the fit keeps the sweep kernel's own exponentials), so bits may differ in the last place."""
    (b, bt) = golden_inputs(90, 50, 50)
    (f1, f2) = (_run_fit(b, bt, 3, lookup), _run_fit(b, bt, 3, lookup))
    s = f1.score_patients(f1.bt, lq_R0=f1._lq_R, max_sweeps=1)
    f2._update_lq_R()
    assert s.sweeps == 1 and s.lq_R.shape == (90, 50, 2)
    nptest.assert_allclose(s.lq_R, f2._lq_R, rtol=0, atol=1e-13)


def test_terms_sum_to_the_whole_fit_terms():
    (b, bt) = golden_inputs(90, 50, 50)
    fit = _run_fit(b, bt, 3, "reference")
    (lq_R, t, sweeps, _) = fit._score_terms(fit.bt, fit._lq_R, 0, 1e-9)
    assert sweeps == 0
    nptest.assert_array_equal(lq_R, fit._lq_R)
    (q_F, q_R) = (np.exp(fit._lq_F), np.exp(fit._lq_R))
    fit._update_lps()                      # the arrays below at the model's theta
    nptest.assert_allclose(t[:, 0].sum(), F._eval_E_lM(q_F, q_R, fit._lM), rtol=1e-12)
    nptest.assert_allclose(t[:, 1].sum(), F._eval_E_lp_R(q_R, F._pi2(fit.model.pi)), rtol=1e-12)
    nptest.assert_allclose(t[:, 2].sum(), F._eval_E_lq_R(q_R, fit._lq_R), rtol=1e-12)
    s = fit.score_patients(fit.bt, lq_R0=fit._lq_R, max_sweeps=0)
    nptest.assert_array_equal(s.free_energy, (-t[:, 1] - t[:, 0]) + t[:, 2])
    assert np.isnan(s.max_change)


# ------------------------------------------------------------------ against the oracle
_FITTED = {}


def _fitted_state(N, lookup):
    """theta and a peaked q_F of a fit on training data of N regions (cached per module)."""
    if (N, lookup) not in _FITTED:
        (_, _, _, _, b, bt) = O.sample(O.Theta(), N, 30, 40, np.random.RandomState(N + 5))
        fit = _run_fit(b, bt, 4, lookup)
        _FITTED[(N, lookup)] = (_theta_of(fit.model), fit._lq_F.copy())
    return _FITTED[(N, lookup)]


def _check_vs_oracle(th, lq_F, bt, lookup, sweeps=3, lq_R0=None, rtol=(1e-9, 1e-10), atol=(1e-10, 1e-9)):
    fit = _fit_at(th, lq_F, lookup)
    (lq_R, t, k, _) = fit._score_terms(bt, lq_R0, sweeps, -1.0)
    assert k == sweeps
    (exp_R, _) = OP.score_patients(th, lq_F, bt, lq_R0, lookup, sweeps=sweeps)
    nptest.assert_allclose(lq_R, exp_R, rtol=rtol[0], atol=atol[0])
    # the four sums, at the posterior the GPU reached
    exp_t = OP.patient_terms(th, lq_F, lq_R, _lM_of(th, bt))
    nptest.assert_allclose(t, exp_t, rtol=rtol[1], atol=atol[1])
    s = fit.score_patients(bt, lq_R0, sweeps, -1.0)
    (fe, typ) = OP.free_energies(th, lq_R.shape[0], exp_t)
    nptest.assert_allclose(s.free_energy, fe, rtol=rtol[1], atol=atol[1])
    nptest.assert_allclose(s.free_energy_typical, typ, rtol=rtol[1], atol=atol[1])


@pytest.mark.parametrize("N,U", [(10, 1), (10, 45), (90, 1), (90, 45)])
@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
@pytest.mark.parametrize("qF_kind", ["random", "fitted"])
def test_parity_with_oracle(N, U, lookup, qF_kind):
    """N = 10 takes the stepwise sweep kernel, N = 90 the blocked one; U' = 1 and 45 (not a multiple of 32).
    Random q_F: every edge unpeaked (three planes, nine logarithms); fitted q_F: peaked edges (one plane)."""
    if qF_kind == "fitted":
        (th, lq_F) = _fitted_state(N, lookup)
    else:
        th = O.Theta()
        rng = np.random.RandomState(3 * N + U)
        lq_F = np.log(rng.dirichlet([1, 1, 1], size=(N * (N - 1) // 2, 1)))
    (_, _, _, _, _, bt) = O.sample(O.Theta(), N, 2, U, np.random.RandomState(N + U))
    _check_vs_oracle(th, lq_F, bt, lookup)


@pytest.mark.parametrize("N", [10, 90])
@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
@pytest.mark.parametrize("theta", ["bound", "safe"])
def test_parity_with_oracle_at_extreme_theta(N, lookup, theta):
    """(eta, epsilon) on the optimiser's bounds [1e-5, 1 - 1e-5]; and epsilon = 1e-7 <= 2^-19, where the
    lean logarithm does not apply and the SAFE kernel variants run.  There the responsibility planes limit the
    agreement: a_1 + b_1 p_k = a_1 (1 - p_k) + epsilon p_k, and where the true state's p_k is within ~1e-8 of 1
    the rounding of p_k (1e-16) is a relative error of ~5e-17 / epsilon in log M_k1 -- after three sweeps over
    89 edges per region ~5e-7 in lq_R (measured 4.5e-7), whichever kernel or NumPy code evaluates that form."""
    (th, lq_F) = _fitted_state(N, lookup)
    th = th.copy()
    if theta == "bound":
        (th.eta, th.epsilon) = (1 - 1e-5, 1e-5)
    else:
        th.epsilon = 1e-7
    (_, _, _, _, _, bt) = O.sample(O.Theta(), N, 2, 37, np.random.RandomState(N + 1))
    rng = np.random.RandomState(N)
    lq_R0 = np.log(rng.dirichlet([1, 1], size=(N, 37)))
    if theta == "safe":
        _check_vs_oracle(th, lq_F, bt, lookup, lq_R0=lq_R0, rtol=(1e-6, 1e-8), atol=(1e-6, 1e-6))
    else:
        _check_vs_oracle(th, lq_F, bt, lookup, lq_R0=lq_R0)


def test_qR_change_per_patient_maxima():
    lib = _lib.load()
    rng = np.random.RandomState(0)
    (N, U) = (90, 45)
    (a, b) = (rng.rand(N, U, 2), rng.rand(N, U, 2))
    b[:, 7] = a[:, 7]
    (da, db) = (_dev.upload(a), _dev.upload(b))
    (maxU, out) = (_dev.empty((U,)), _dev.zeros((1,)))
    _lib.check(lib.fcd_qR_change(_dev.ptr(da), _dev.ptr(db), N, U, _dev.ptr(maxU), _dev.ptr(out), _dev.stream()),
               "fcd_qR_change")
    exp = np.abs(b - a).max(axis=(0, 2))
    nptest.assert_array_equal(maxU.cpu().numpy(), exp)
    assert out.cpu().numpy()[0] == exp.max() and exp[7] == 0.0


# ------------------------------------------------------------------ properties of the scorer
def test_batch_invariance():
    (th, lq_F) = _fitted_state(90, "symmetric")
    (_, _, _, _, _, bt) = O.sample(O.Theta(), 90, 2, 45, np.random.RandomState(21))
    lq_R0 = np.log(np.random.RandomState(22).dirichlet([1, 1], size=(90, 45)))
    fit = _fit_at(th, lq_F, "symmetric")
    (A, B) = (slice(0, 13), slice(13, 45))
    (_, t_ab, _, _) = fit._score_terms(bt, lq_R0, 0, 1e-9)
    (_, t_a, _, _) = fit._score_terms(bt[:, A], lq_R0[:, A], 0, 1e-9)
    (_, t_b, _, _) = fit._score_terms(bt[:, B], lq_R0[:, B], 0, 1e-9)
    nptest.assert_array_equal(t_ab[A], t_a)
    nptest.assert_array_equal(t_ab[B], t_b)
    tol = 1e-9
    s_ab = fit.score_patients(bt, max_sweeps=1000, tol=tol)
    (s_a, s_b) = (fit.score_patients(bt[:, A], max_sweeps=1000, tol=tol),
                  fit.score_patients(bt[:, B], max_sweeps=1000, tol=tol))
    assert max(s_ab.sweeps, s_a.sweeps, s_b.sweeps) < 1000
    nptest.assert_allclose(np.exp(s_ab.lq_R[:, A]), np.exp(s_a.lq_R), rtol=0, atol=10 * tol)
    nptest.assert_allclose(np.exp(s_ab.lq_R[:, B]), np.exp(s_b.lq_R), rtol=0, atol=10 * tol)


def test_symmetric_sweeps_converge_monotonically():
    (th, lq_F) = _fitted_state(90, "symmetric")
    (_, _, _, _, _, bt) = O.sample(O.Theta(), 90, 2, 40, np.random.RandomState(31))
    fit = _fit_at(th, lq_F, "symmetric")
    fe = np.array([fit.score_patients(bt, max_sweeps=k, tol=-1.0).free_energy for k in range(1, 6)])
    assert np.all(np.diff(fe, axis=0) <= 1e-10 * np.abs(fe[1:])), np.diff(fe, axis=0).max()
    tol = 1e-9
    s = fit.score_patients(bt, max_sweeps=2000, tol=tol)
    assert s.sweeps < 2000 and s.max_change <= tol
    s2 = fit.score_patients(bt, lq_R0=s.lq_R, max_sweeps=1)
    assert s2.max_change <= tol
    nptest.assert_allclose(np.exp(s2.lq_R), np.exp(s.lq_R), rtol=0, atol=tol)


@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
def test_the_fit_is_untouched(lookup):
    (b, bt) = golden_inputs(90, 50, 50)
    (f1, f2) = (_run_fit(b, bt, 3, lookup), _run_fit(b, bt, 3, lookup))
    before = (f1.model.pi, f1.model.eta, f1.model.epsilon, f1.model.gamma.copy(), f1.model.mu.copy(),
              f1.model.sigma.copy(), f1._lq_F.copy(), f1._lq_R.copy(), list(f1.energy))
    (inp, WT, PsT, kcache, spec) = (f1._in, f1._in['WT'], f1._in['PsT'], f1._in['kcache'], f1._spec)
    (WT0, PsT0) = (WT.clone(), PsT.clone())
    (_, _, _, _, _, bt_new) = O.sample(O.Theta(), 90, 2, 33, np.random.RandomState(41))
    f1.score_patients(bt_new, max_sweeps=5)
    after = (f1.model.pi, f1.model.eta, f1.model.epsilon, f1.model.gamma, f1.model.mu, f1.model.sigma,
             f1._lq_F, f1._lq_R, f1.energy)
    for (x, y) in zip(before, after):
        nptest.assert_array_equal(x, y)
    assert f1._in is inp and inp['WT'] is WT and inp['PsT'] is PsT and inp['kcache'] is kcache and f1._spec is spec
    assert torch.equal(WT, WT0) and torch.equal(PsT, PsT0)
    f1._update_lq_R()
    f2._update_lq_R()
    nptest.assert_array_equal(f1._lq_R, f2._lq_R)


def test_planted_regions_of_held_out_patients_are_recovered():
    """A fit on 60 patients, then the 60 held-out ones (same draw) are scored with the symmetric lookup.
    Thresholds: the NumPy oracle reaches recall 0.992 and precision 1.0 at this seed and size
    (tests/test_patients_host.py); both must exceed 0.9 here."""
    th_true = O.Theta(pi=0.1, eta=0.5)
    (r, _, _, _, b, bt) = O.sample(th_true, 20, 30, 120, np.random.RandomState(12))
    Ut = 60
    fit = _run_fit(b, bt[:, :Ut], 10, "symmetric")
    s = fit.score_patients(bt[:, Ut:])
    assert s.sweeps < 50
    pred = s.lq_R[:, :, 1] > s.lq_R[:, :, 0]
    truth = r[:, Ut:]
    tp = float((pred & truth).sum())
    (rec, prec) = (tp / truth.sum(), tp / max(pred.sum(), 1))
    assert rec > 0.9 and prec > 0.9, (rec, prec)
    # a planted patient's typical-minus-actual free energy grows with its number of anomalous regions
    score = s.free_energy_typical - s.free_energy
    assert np.all(score >= -1e-9)
    none = truth.sum(axis=0) == 0
    if none.any() and (~none).any():
        assert score[~none].mean() > score[none].mean()


def test_determinism_and_device_input():
    (th, lq_F) = _fitted_state(90, "reference")
    (_, _, _, _, _, bt) = O.sample(O.Theta(), 90, 2, 45, np.random.RandomState(51))
    fit = _fit_at(th, lq_F, "reference")
    s1 = fit.score_patients(bt)
    s2 = fit.score_patients(bt)
    s3 = fit.score_patients(torch.from_numpy(bt).cuda())
    for s in (s2, s3):
        nptest.assert_array_equal(s.lq_R, s1.lq_R)
        nptest.assert_array_equal(s.free_energy, s1.free_energy)
        nptest.assert_array_equal(s.free_energy_typical, s1.free_energy_typical)
        assert (s.sweeps, s.max_change) == (s1.sweeps, s1.max_change)
