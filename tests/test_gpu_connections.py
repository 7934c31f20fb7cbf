"""GPU: posteriors of the anomalous connections and of the patients' connection states
(``UnsharedRegionFit.connection_posteriors``, csrc/fcd_patients.cu) against the NumPy oracle
(oracle/connections.py), for the fitted cohort and held-out patients, and against planted anomalies."""
import numpy as np
import numpy.testing as nptest
import pytest
import torch

from oracle import connections as OC
from oracle import iar_oracle as O
from oracle.make_golden import golden_inputs

pytestmark = pytest.mark.gpu

import fcdiff_b200 as fcdiff          # noqa: E402
from fcdiff_b200 import _lib, sweep   # noqa: E402

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


def _fit_at(th, lq_F):
    """A fit that holds only theta and q_F: enough to read out held-out patients."""
    fit = F.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    (fit.model.pi, fit.model.eta, fit.model.epsilon) = (th.pi, th.eta, th.epsilon)
    (fit.model.gamma, fit.model.mu, fit.model.sigma) = (th.gamma.copy(), th.mu.copy(), th.sigma.copy())
    fit.edge_lookup = "symmetric"
    fit._lq_F = lq_F
    return fit


def _theta_of(model):
    return O.Theta(pi=float(model.pi), eta=float(model.eta), gamma=np.array(model.gamma, dtype=np.float64),
                   epsilon=float(model.epsilon), mu=np.array(model.mu, dtype=np.float64),
                   sigma=np.array(model.sigma, dtype=np.float64))


def _check(got, exp_T, exp_Ft, atol=1e-12, rtol=1e-12):
    """Maps against the oracle (absolute), reductions against the oracle's sums (relative) and against the
    returned map (1e-12).  The reductions also get an absolute 1e-14: the kernel drops weights <= 2^-60, which
    moves a sum of a few thousand q_T by at most ~1e-15, the whole of a sum that is itself that small."""
    nptest.assert_allclose(got.q_T, exp_T, rtol=0, atol=atol)
    nptest.assert_allclose(got.q_F_tilde, exp_Ft, rtol=0, atol=atol)
    nptest.assert_allclose(got.expected_anomalous, exp_T.sum(axis=0), rtol=rtol, atol=1e-14)
    nptest.assert_allclose(got.anomalous_rate, exp_T.mean(axis=1), rtol=rtol, atol=1e-14)
    nptest.assert_allclose(got.expected_anomalous, got.q_T.sum(axis=0), rtol=1e-12, atol=1e-14)
    nptest.assert_allclose(got.anomalous_rate, got.q_T.mean(axis=1), rtol=1e-12, atol=1e-14)


def _check_maps_off(fit, with_maps, *args):
    """maps=False: no maps, reductions bit-identical to maps=True."""
    r = fit.connection_posteriors(*args, maps=False)
    assert r.q_T is None and r.q_F_tilde is None
    nptest.assert_array_equal(r.expected_anomalous, with_maps.expected_anomalous)
    nptest.assert_array_equal(r.anomalous_rate, with_maps.anomalous_rate)


# ------------------------------------------------------------------ held-out patients against the oracle
_FITTED = {}


def _fitted_state(N):
    """theta and a peaked q_F of a fit on training data of N regions (cached per module)."""
    if N not in _FITTED:
        (_, _, _, _, b, bt) = O.sample(O.Theta(), N, 30, 40, np.random.RandomState(N + 5))
        fit = _run_fit(b, bt, 4, "symmetric")
        _FITTED[N] = (_theta_of(fit.model), fit._lq_F.copy())
    return _FITTED[N]


def _case(N, U, qF_kind, qR_kind, seed=0):
    if qF_kind == "fitted":
        (th, lq_F) = _fitted_state(N)
    else:
        th = O.Theta()
        lq_F = np.log(np.random.RandomState(3 * N + U).dirichlet([1, 1, 1], size=(N * (N - 1) // 2, 1)))
    (_, _, _, _, _, bt) = O.sample(O.Theta(), N, 2, U, np.random.RandomState(N + U + seed))
    fit = _fit_at(th, lq_F)
    if qR_kind == "fitted":
        lq_R = fit.score_patients(bt).lq_R                 # peaked regions and undecided ones: mixed tiers
    else:
        lq_R = np.log(np.random.RandomState(N * U + 1).dirichlet([1, 1], size=(N, U)))
    return th, lq_F, bt, lq_R, fit


@pytest.mark.parametrize("N,U", [(10, 1), (10, 45), (90, 1), (90, 45)])
@pytest.mark.parametrize("qF_kind", ["random", "fitted"])
@pytest.mark.parametrize("qR_kind", ["random", "fitted"])
def test_parity_with_oracle(N, U, qF_kind, qR_kind):
    """Random q_F: every edge unpeaked (nine terms); fitted q_F: peaked edges (one or three terms).  Random q_R:
    every region undecided; fitted q_R: mostly peaked regions.  U' = 1 and 45 (not a multiple of 32)."""
    (th, lq_F, bt, lq_R, fit) = _case(N, U, qF_kind, qR_kind)
    (exp_T, exp_Ft) = OC.connection_posteriors(th, lq_F, lq_R, bt)
    got = fit.connection_posteriors(bt, lq_R)
    assert got.q_T.shape == (N * (N - 1) // 2, U) and got.q_F_tilde.shape == (N * (N - 1) // 2, U, 3)
    _check(got, exp_T, exp_Ft)
    _check_maps_off(fit, got, bt, lq_R)


@pytest.mark.parametrize("N", [10, 90])
@pytest.mark.parametrize("theta", ["bound_low_eps", "bound_high_eps", "tiny_eps"])
def test_parity_with_oracle_at_extreme_theta(N, theta):
    """(eta, epsilon) on the optimiser's bounds, and epsilon = 1e-7.  The plane form a_l + b_l p_k of the
    denominators is ill-conditioned at extreme epsilon where p_k is near 1: the rounding of p_k (1e-16) becomes
    a relative error of ~1e-16 / min(epsilon, 1 - epsilon), whichever kernel or NumPy code evaluates it (the
    limit of test_parity_with_oracle_at_extreme_theta in test_gpu_patients.py, and of the oracle against
    enumeration in test_connections_host.py).  Measured largest differences on a B200: on the bounds 4.5e-12
    (q_T) and 1.8e-11 (q_F~), checked at 1e-10; at epsilon = 1e-7 1.3e-15 (q_T) and 1.2e-9 (q_F~), checked at
    1e-8."""
    (th, lq_F) = _fitted_state(N)
    th = th.copy()
    if theta == "bound_low_eps":
        (th.eta, th.epsilon) = (1 - 1e-5, 1e-5)
    elif theta == "bound_high_eps":
        (th.eta, th.epsilon) = (1e-5, 1 - 1e-5)
    else:
        th.epsilon = 1e-7
    (_, _, _, _, _, bt) = O.sample(O.Theta(), N, 2, 37, np.random.RandomState(N + 1))
    lq_R = np.log(np.random.RandomState(N).dirichlet([1, 1], size=(N, 37)))
    fit = _fit_at(th, lq_F)
    (exp_T, exp_Ft) = OC.connection_posteriors(th, lq_F, lq_R, bt)
    got = fit.connection_posteriors(bt, lq_R)
    tol = 1e-8 if theta == "tiny_eps" else 1e-10
    _check(got, exp_T, exp_Ft, atol=tol, rtol=tol)
    _check_maps_off(fit, got, bt, lq_R)


# ------------------------------------------------------------------ the fitted cohort
@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
def test_fitted_cohort(lookup):
    """After run(): the fit's own planes, q_F and q_R; equal to the oracle at the fit's state, and to the
    held-out path given the fit's own columns (which forms exp(lq_R) on the host: last bits may differ)."""
    (b, bt) = golden_inputs(90, 50, 50)
    fit = _run_fit(b, bt, 3, lookup)
    got = fit.connection_posteriors()
    (exp_T, exp_Ft) = OC.connection_posteriors(_theta_of(fit.model), fit._lq_F, fit._lq_R, bt)
    _check(got, exp_T, exp_Ft)
    held = fit.connection_posteriors(fit.bt, fit._lq_R)
    for (x, y) in zip(got, held):
        nptest.assert_allclose(x, y, rtol=1e-13, atol=1e-13)
    _check_maps_off(fit, got)


def test_replica_mode_fit_equals_the_plain_fit():
    (N, H, U) = (30, 20, 24)
    (_, _, _, _, b, bt) = O.sample(O.Theta(pi=0.1, eta=0.5), N, H, U, np.random.RandomState(61))
    plain = _run_fit(b, bt, 3, "reference")
    sp = sweep.SharedPlanes(np.concatenate([b, bt], axis=1), fcdiff.UnsharedRegionModel())
    rep = F.UnsharedRegionFit()
    rep.model = fcdiff.UnsharedRegionModel()
    rep.set_shared_inputs(sp, np.arange(H), H + np.arange(U))
    (rep.max_iters, rep.rel_tol) = (3, -1.0)
    rep.run()
    got = rep.connection_posteriors()
    (exp_T, exp_Ft) = OC.connection_posteriors(_theta_of(rep.model), rep._lq_F, rep._lq_R, bt)
    _check(got, exp_T, exp_Ft)
    ref = plain.connection_posteriors()
    for (x, y) in zip(got, ref):
        nptest.assert_allclose(x, y, rtol=1e-9, atol=1e-9)


# ------------------------------------------------------------------ properties
def test_batch_invariance():
    """A patient's maps and expected count do not depend on which other patients are in the call."""
    (th, lq_F, bt, lq_R, fit) = _case(90, 45, "fitted", "fitted", seed=21)
    whole = fit.connection_posteriors(bt, lq_R)
    for cols in (slice(0, 13), slice(13, 45)):
        part = fit.connection_posteriors(bt[:, cols], lq_R[:, cols])
        nptest.assert_array_equal(part.q_T, whole.q_T[:, cols])
        nptest.assert_array_equal(part.q_F_tilde, whole.q_F_tilde[:, cols])
        nptest.assert_array_equal(part.expected_anomalous, whole.expected_anomalous[cols])


def test_determinism_and_device_input():
    (th, lq_F, bt, lq_R, fit) = _case(90, 45, "fitted", "fitted", seed=51)
    r1 = fit.connection_posteriors(bt, lq_R)
    r2 = fit.connection_posteriors(bt, lq_R)
    r3 = fit.connection_posteriors(torch.from_numpy(bt).cuda(), torch.from_numpy(lq_R).cuda())
    for r in (r2, r3):
        for (x, y) in zip(r, r1):
            nptest.assert_array_equal(x, y)


@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
def test_the_fit_is_untouched(lookup):
    (b, bt) = golden_inputs(90, 50, 50)
    (f1, f2) = (_run_fit(b, bt, 3, lookup), _run_fit(b, bt, 3, lookup))
    before = (f1.model.pi, f1.model.eta, f1.model.epsilon, f1.model.gamma.copy(), f1.model.mu.copy(),
              f1.model.sigma.copy(), f1._lq_F.copy(), f1._lq_R.copy(), list(f1.energy))
    (inp, WT, PsT, kcache, spec) = (f1._in, f1._in['WT'], f1._in['PsT'], f1._in['kcache'], f1._spec)
    (WT0, PsT0, P0) = (WT.clone(), PsT.clone(), inp['P'].clone())
    s = f1.score_patients(bt[:, :20])
    f1.connection_posteriors()
    f1.connection_posteriors(maps=False)
    f1.connection_posteriors(bt[:, :20], s.lq_R)
    after = (f1.model.pi, f1.model.eta, f1.model.epsilon, f1.model.gamma, f1.model.mu, f1.model.sigma,
             f1._lq_F, f1._lq_R, f1.energy)
    for (x, y) in zip(before, after):
        nptest.assert_array_equal(x, y)
    assert f1._in is inp and inp['WT'] is WT and inp['PsT'] is PsT and inp['kcache'] is kcache and f1._spec is spec
    assert torch.equal(WT, WT0) and torch.equal(PsT, PsT0) and torch.equal(inp['P'], P0)
    f1._update_lq_R()
    f2._update_lq_R()
    nptest.assert_array_equal(f1._lq_R, f2._lq_R)


def _auc(score, label):
    from scipy.stats import rankdata
    (s, y) = (np.ravel(score), np.ravel(label).astype(bool))
    rk = rankdata(s)
    (n1, n0) = (int(y.sum()), int((~y).sum()))
    return (rk[y].sum() - n1 * (n1 + 1) / 2.0) / (n1 * n0)


def test_planted_connections_are_recovered():
    """A 10-iteration symmetric-lookup fit on 60 patients (the draw of test_gpu_patients.py's recovery test),
    its own patients and the 60 held out.  The NumPy oracle reaches AUC 0.9974 / 0.9967 of q_T against the
    sampler's t and argmax accuracy 0.9976 / 0.9982 of q_F~ against f~ (tests/test_connections_host.py); all four
    must exceed 0.99 here."""
    (_, t, _, f_tilde, b, bt) = O.sample(O.Theta(pi=0.1, eta=0.5), 20, 30, 120, np.random.RandomState(12))
    Ut = 60
    fit = _run_fit(b, bt[:, :Ut], 10, "symmetric")
    s = fit.score_patients(bt[:, Ut:])
    for (r, cols) in ((fit.connection_posteriors(), slice(0, Ut)),
                      (fit.connection_posteriors(bt[:, Ut:], s.lq_R), slice(Ut, None))):
        (auc, acc) = (_auc(r.q_T, t[:, cols]), (np.argmax(r.q_F_tilde, axis=-1) ==
                                                np.argmax(f_tilde[:, cols], axis=-1)).mean())
        assert auc > 0.99 and acc > 0.99, (cols, auc, acc)
