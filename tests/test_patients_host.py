"""CPU: the NumPy oracle of held-out patient scoring (oracle/patients.py) against the oracle's own EM steps,
and the argument checks of ``UnsharedRegionFit.score_patients``, which raise before any device work."""
import numpy as np
import numpy.testing as nptest
import pytest

from oracle import iar_oracle as O
from oracle import patients as OP
from oracle.make_golden import golden_inputs

CONFIGS = {1: (10, 20, 20), 2: (90, 50, 50)}


def _training_state(N, H, U, iters=2, lookup="reference"):
    (b, bt) = golden_inputs(N, H, U)
    th = O.Theta()
    out = O.run(b, bt, th, max_iters=iters, rel_tol=-1.0, edge_lookup=lookup)
    return b, bt, th, out["lq_F"], out["lq_R"]


@pytest.mark.parametrize("cfg", [1, 2])
@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
def test_one_sweep_is_the_region_update(cfg, lookup):
    """One sweep from a training state is `update_lq_R` (fit.py:176-198) on the same columns."""
    (b, bt, th, lq_F, lq_R) = _training_state(*CONFIGS[cfg], lookup=lookup)
    (_, _, lM) = O.update_lps(b, bt, th)
    exp = O.update_lq_R(np.array([1 - th.pi, th.pi]), lq_F, lM, lq_R, lookup)
    (got, _) = OP.score_patients(th, lq_F, bt, lq_R, lookup, sweeps=1)
    nptest.assert_allclose(got, exp, rtol=1e-14, atol=1e-14)


@pytest.mark.parametrize("cfg", [1, 2])
def test_patient_terms_sum_to_the_whole_fit_terms(cfg):
    (b, bt, th, lq_F, lq_R) = _training_state(*CONFIGS[cfg])
    (_, _, lM) = O.update_lps(b, bt, th)
    t = OP.patient_terms(th, lq_F, lq_R, lM)
    (q_F, q_R) = (np.exp(lq_F), np.exp(lq_R))
    assert t.shape == (bt.shape[1], 4)
    nptest.assert_allclose(t[:, 0].sum(), O.eval_E_lM(q_F, q_R, lM), rtol=1e-12)
    nptest.assert_allclose(t[:, 1].sum(), O.eval_E_lp_R(q_R, np.array([1 - th.pi, th.pi])), rtol=1e-12)
    nptest.assert_allclose(t[:, 2].sum(), O.eval_E_lq_R(q_R, lq_R), rtol=1e-12)
    # the typical share: q_R all typical gives E_lM = sum q_F log M_k0, E_lp_R = N log(1 - pi), E_lq_R = 0
    N = lq_R.shape[0]
    lq_typ = np.zeros_like(lq_R)
    lq_typ[:, :, 1] = -np.inf
    with np.errstate(invalid="ignore"):
        t_typ = OP.patient_terms(th, lq_F, lq_typ, lM)
    nptest.assert_allclose(t_typ[:, 0], t[:, 3], rtol=1e-12)
    nptest.assert_allclose(t_typ[:, 1], N * np.log(1 - th.pi), rtol=1e-14)


@pytest.mark.parametrize("cfg", [1, 2])
def test_symmetric_sweeps_do_not_raise_the_free_energy(cfg):
    """With the symmetric lookup a sweep is exact coordinate ascent on each patient's share of the
    free energy: from the uniform start it never increases, patient by patient."""
    (b, bt, th, lq_F, _) = _training_state(*CONFIGS[cfg], lookup="symmetric")
    fe = []
    for k in range(0, 6):
        (_, t) = OP.score_patients(th, lq_F, bt, None, "symmetric", sweeps=k)
        fe.append(OP.free_energies(th, int(O.C_to_N(bt.shape[0])), t)[0])
    fe = np.array(fe)
    assert np.all(np.diff(fe, axis=0) <= 1e-9 * np.abs(fe[1:])), np.diff(fe, axis=0).max()
    assert np.all(fe[-1] < fe[0])


def planted_problem():
    """Planted anomalies for the recovery tests (here and in test_gpu_patients.py): 20 regions, 30 controls,
    120 patients drawn with pi = 0.1, eta = 0.5; the fit sees the first 60 patients, the other 60 are scored."""
    th_true = O.Theta(pi=0.1, eta=0.5)
    (r, _, _, _, b, bt) = O.sample(th_true, 20, 30, 120, np.random.RandomState(12))
    return r, b, bt, 60


def recall_precision(lq_R, r):
    pred = lq_R[:, :, 1] > lq_R[:, :, 0]
    tp = float((pred & r).sum())
    return tp / max(r.sum(), 1), tp / max(pred.sum(), 1)


def test_oracle_recovers_planted_regions_of_held_out_patients():
    """The oracle at the size and seed of the GPU recovery test: a 10-iteration fit on the training half,
    50 symmetric sweeps on the held-out half.  Recall 0.992 and precision 1.0 here (133 planted regions)."""
    (r, b, bt, Ut) = planted_problem()
    th = O.Theta()
    out = O.run(b, bt[:, :Ut], th, max_iters=10, rel_tol=-1.0, edge_lookup="symmetric", polish=True)
    (lq_R, _) = OP.score_patients(th, out["lq_F"], bt[:, Ut:], None, "symmetric", sweeps=50)
    (rec, prec) = recall_precision(lq_R, r[:, Ut:])
    assert rec >= 0.9 and prec >= 0.9, (rec, prec)


# ------------------------------------------------------------------ argument checks (no device needed)
def _fit(N=6, U=4):
    import fcdiff_b200 as fcdiff
    fit = fcdiff.fit.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    C = N * (N - 1) // 2
    fit._lq_F = np.full((C, 1, 3), -np.log(3))
    return fit, np.zeros((C, U))


def test_score_patients_rejects_a_wrong_edge_count():
    (fit, bt) = _fit()
    with pytest.raises(ValueError):
        fit.score_patients(bt[1:])
    with pytest.raises(ValueError):
        fit.score_patients(bt[:, 0])
    with pytest.raises(ValueError):
        fit.score_patients(bt, lq_R0=np.zeros((6, 3, 2)))


def test_score_patients_rejects_a_sharded_fit():
    (fit, bt) = _fit()
    fit.shards = object()
    with pytest.raises(ValueError):
        fit.score_patients(bt)


def test_score_patients_rejects_arrays_mode():
    (fit, bt) = _fit()
    fit._lM = np.zeros((bt.shape[0], bt.shape[1], 3, 3))
    with pytest.raises(ValueError):
        fit.score_patients(bt)


def test_score_patients_needs_a_model_and_q_F():
    import fcdiff_b200 as fcdiff
    (fit, bt) = _fit()
    fit.model = None
    with pytest.raises(ValueError):
        fit.score_patients(bt)
    fit = fcdiff.fit.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    with pytest.raises(ValueError):
        fit.score_patients(bt)
