"""GPU: missing entries marginalised (``UnsharedRegionFit.missing = "marginalize"``; csrc: fcd_resp_cache,
fcd_control_terms and fcd_materialize_lps with missing = 1, fcd_healthy_stats and the K2 / K4 launches with an S0
array, fcd_corr_mark_missing) against the default path on complete data (bit for bit) and the masked NumPy oracle
(oracle/missing.py) on data with NaN entries."""
import copy

import numpy as np
import numpy.testing as nptest
import pytest
import torch

from oracle import iar_oracle as O
from oracle import missing as OM
from oracle import patients as OP
from oracle.make_golden import golden_inputs

pytestmark = pytest.mark.gpu

import fcdiff_b200 as fcdiff          # noqa: E402
from fcdiff_b200 import _dev, _lib, corr, sweep    # noqa: E402

F = fcdiff.fit


@pytest.fixture(scope="module", autouse=True)
def _native_library_loaded():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    lib = _lib.load()
    n0 = lib.fcd_launch_count()
    yield
    assert lib.fcd_launch_count() > n0, "no kernel of libfcdiff_b200.so was launched"


def _fit(b, bt, missing="marginalize", iters=2, lookup="reference", solver="newton", model=None):
    fit = F.UnsharedRegionFit()
    (fit.b, fit.bt) = (b, bt)
    fit.model = copy.deepcopy(model) if model is not None else fcdiff.UnsharedRegionModel()
    fit.missing = missing
    fit.edge_lookup = lookup
    fit.theta_solver = solver
    fit.max_iters = iters
    fit.rel_tol = -1.0
    return fit


def _theta_of(model):
    return O.Theta(pi=float(model.pi), eta=float(model.eta), gamma=np.array(model.gamma, dtype=np.float64),
                   epsilon=float(model.epsilon), mu=np.array(model.mu, dtype=np.float64),
                   sigma=np.array(model.sigma, dtype=np.float64))


def _pattern(kind, b, bt, seed):
    """NaN patterns: missing at random (10 % / 40 %), whole-region dropout per subject, edges missing in every
    subject together with a subject with nothing observed."""
    rng = np.random.RandomState(seed)
    (b, bt) = (b.copy(), bt.copy())
    C = b.shape[0]
    N = int(O.C_to_N(C))
    (n, m) = O.edge_pairs(N)
    if kind.startswith("mcar"):
        frac = float(kind[4:]) / 100
        b[rng.uniform(size=b.shape) < frac] = np.nan
        bt[rng.uniform(size=bt.shape) < frac] = np.nan
    elif kind == "regions":
        for x in (b, bt):
            drop = rng.uniform(size=(N, x.shape[1])) < 0.2
            for s in range(x.shape[1]):
                x[drop[n, s] | drop[m, s], s] = np.nan
    elif kind == "edges_subject":
        cut = rng.choice(C, size=max(1, C // 10), replace=False)
        (b[cut], bt[cut]) = (np.nan, np.nan)
        (b[:, 1], bt[:, 2]) = (np.nan, np.nan)
    return b, bt


PATTERNS = ["mcar10", "mcar40", "regions", "edges_subject"]


# ------------------------------------------------------------------ the masked form on complete data
@pytest.mark.parametrize("N, H, U", [(90, 50, 50), (400, 500, 500)])
def test_marginalize_without_nan_is_bit_identical(N, H, U):
    (b, bt) = golden_inputs(N, H, U, seed=3)
    fits = {}
    for missing in ("reject", "marginalize"):
        fit = _fit(b, bt, missing=missing)
        fit.run()
        fits[missing] = fit
    (a, z) = (fits["reject"], fits["marginalize"])
    assert a.energy == z.energy
    nptest.assert_array_equal(a._lq_F, z._lq_F)
    nptest.assert_array_equal(a._lq_R, z._lq_R)
    assert (a.model.pi, a.model.eta, a.model.epsilon) == (z.model.pi, z.model.eta, z.model.epsilon)
    nptest.assert_array_equal(a.model.gamma, z.model.gamma)
    nptest.assert_array_equal(a._energy_terms(), z._energy_terms())
    if N > 100:
        return
    x = golden_inputs(N, 7, 9, seed=4)[1]
    (sa, sz) = (a.score_patients(x), z.score_patients(x))
    for (u, v) in zip(sa, sz):
        nptest.assert_array_equal(u, v)
    (ca, cz) = (a.connection_posteriors(), z.connection_posteriors())
    for (u, v) in zip(ca, cz):
        nptest.assert_array_equal(u, v)
    nptest.assert_array_equal(a.score_controls(), z.score_controls())
    (ka, kz) = (a.classify_subjects(x, 0.5), z.classify_subjects(x, 0.5))
    for (u, v) in zip(ka, kz):
        nptest.assert_array_equal(u, v)
    nptest.assert_array_equal(a._lp_B_g_F, z._lp_B_g_F)
    nptest.assert_array_equal(a._lM, z._lM)


# ------------------------------------------------------------------ full runs and single steps against the oracle
@pytest.mark.parametrize("kind", PATTERNS)
@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
@pytest.mark.parametrize("solver", ["newton", "lbfgsb"])
def test_full_run_matches_the_masked_oracle(kind, lookup, solver):
    (b, bt) = _pattern(kind, *golden_inputs(10, 20, 20, seed=0), seed=1)
    fit = _fit(b, bt, iters=4, lookup=lookup, solver=solver)
    fit.model.eta += 0.1
    fit.run()
    th = O.Theta()
    th.eta += 0.1
    out = OM.run_masked(b, bt, th, max_iters=4, rel_tol=-1.0, edge_lookup=lookup, polish=solver == "newton")
    nptest.assert_allclose(fit.energy, out["energy"], rtol=1e-6)
    nptest.assert_allclose([fit.model.pi, fit.model.eta, fit.model.epsilon], [th.pi, th.eta, th.epsilon], rtol=1e-6)
    nptest.assert_allclose(np.exp(fit._lq_F), np.exp(out["lq_F"]), rtol=1e-6, atol=1e-9)
    nptest.assert_allclose(np.exp(fit._lq_R), np.exp(out["lq_R"]), rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
def test_config2_run_matches_the_masked_oracle(lookup):
    (b, bt) = _pattern("regions", *golden_inputs(90, 50, 50, seed=0), seed=2)
    fit = _fit(b, bt, iters=3, lookup=lookup)
    fit.run()
    th = O.Theta()
    out = OM.run_masked(b, bt, th, max_iters=3, rel_tol=-1.0, edge_lookup=lookup, polish=True)
    nptest.assert_allclose(fit.energy, out["energy"], rtol=1e-6)
    nptest.assert_allclose([fit.model.pi, fit.model.eta, fit.model.epsilon], [th.pi, th.eta, th.epsilon], rtol=1e-6)
    nptest.assert_allclose(np.exp(fit._lq_R), np.exp(out["lq_R"]), rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize("kind", PATTERNS)
def test_single_steps_match_the_masked_oracle(kind):
    (N, H, U) = (10, 20, 20)
    (b, bt) = _pattern(kind, *golden_inputs(N, H, U, seed=5), seed=6)
    fit = _fit(b, bt)
    fit._init_lps(N, H, U)
    fit._update_lps()
    th = O.Theta()
    (lp, p, lM) = OM.update_lps_masked(b, bt, th)
    (lq_F, lq_R) = O.init_lps(N, U)
    for it in range(2):
        fit._update_lq_F()
        lq_F = O.update_lq_F(th.gamma, lp, lM, lq_R)
        nptest.assert_allclose(fit._lq_F, lq_F, rtol=1e-10, atol=1e-10)
        fit._update_lq_R()
        lq_R = O.update_lq_R(np.array([1 - th.pi, th.pi]), lq_F, lM, lq_R)
        nptest.assert_allclose(fit._lq_R, lq_R, rtol=1e-10, atol=1e-10)
        fit._update_pi()
        fit._update_gamma()
        (th.pi, th.gamma) = (O.update_pi(lq_R), O.update_gamma(lq_F))
        fit._update_lps()
        nptest.assert_allclose(fit._energy_terms(), O.eval_energy_terms(th, fit._lq_F, fit._lq_R, lp, lM),
                               rtol=1e-10, atol=1e-9)
        x = np.array([0.3, 0.2])
        (f, g) = fit._objective(x)
        (fo, go) = O.elm_objective_and_grad(p, np.exp(fit._lq_F), np.exp(fit._lq_R), x)
        nptest.assert_allclose(f, fo, rtol=1e-10)
        nptest.assert_allclose(g, go, rtol=5e-9)
    # the materialised caches hold the oracle's masked values
    nptest.assert_array_equal(fit._lp_B_g_F[np.isnan(b)], 0.0)
    nptest.assert_array_equal(fit._p_Bt_g_Ft[np.isnan(bt)], 1.0)
    nptest.assert_array_equal(fit._lM[np.isnan(bt)], 0.0)


# ------------------------------------------------------------------ read-outs
@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
def test_read_outs_match_the_masked_oracle(lookup):
    (b, bt) = _pattern("mcar10", *golden_inputs(12, 30, 30, seed=8), seed=9)
    fit = _fit(b, bt, iters=3, lookup=lookup)
    fit.run()
    th = _theta_of(fit.model)
    x = _pattern("regions", *golden_inputs(12, 6, 11, seed=10), seed=11)[1]
    x[:, 3] = np.nan
    s = fit.score_patients(x, max_sweeps=3, tol=0.0)
    (lq_R, terms) = OM.score_patients_masked(th, fit._lq_F, x, edge_lookup=lookup, sweeps=3)
    nptest.assert_allclose(s.lq_R, lq_R, rtol=1e-10, atol=1e-12)
    (fe, fe0) = OP.free_energies(th, 12, terms)
    # atol: subject 3 has nothing observed; its shares are 0 up to the rounding residue of the encoding (DESIGN §4)
    nptest.assert_allclose(s.free_energy, fe, rtol=1e-10, atol=1e-12)
    nptest.assert_allclose(s.free_energy_typical, fe0, rtol=1e-10, atol=1e-12)
    nptest.assert_allclose(np.exp(s.lq_R[:, 3]), np.tile([1 - th.pi, th.pi], (12, 1)), rtol=1e-12)
    cp = fit.connection_posteriors(x, s.lq_R)
    (qT, qFt) = OM.connection_posteriors_masked(th, fit._lq_F, s.lq_R, x)
    nptest.assert_allclose(cp.q_T, qT, rtol=1e-10, atol=1e-13)
    nptest.assert_allclose(cp.q_F_tilde, qFt, rtol=1e-10, atol=1e-13)
    own = fit.connection_posteriors()
    (qT, _) = OM.connection_posteriors_masked(th, fit._lq_F, fit._lq_R, bt)
    nptest.assert_allclose(own.q_T, qT, rtol=1e-10, atol=1e-13)
    nptest.assert_allclose(fit.score_controls(x), OM.control_loglik_masked(th, fit._lq_F, x), rtol=1e-12)
    nptest.assert_allclose(fit.score_controls(), OM.control_loglik_masked(th, fit._lq_F, b), rtol=1e-12)
    k = fit.classify_subjects(x, 0.3, max_sweeps=3, tol=0.0)
    (lo, con, elbo) = OM.classify_masked(th, fit._lq_F, x, 0.3, k.lq_R)
    nptest.assert_allclose(k.control_loglik, con, rtol=1e-12, atol=1e-12)
    nptest.assert_allclose(k.patient_elbo, elbo, rtol=1e-10, atol=1e-12)
    nptest.assert_allclose(k.log_odds, lo, rtol=1e-9, atol=1e-9)
    nptest.assert_allclose(k.log_odds[3], np.log(0.3 / 0.7), atol=1e-9)     # nothing observed: the prior
    with pytest.raises(ValueError):
        fit.update_mu_sigma = True
        fit.run()


def test_a_missing_control_column_is_a_dropped_control():
    (b, bt) = _pattern("mcar10", *golden_inputs(10, 20, 20, seed=12), seed=13)
    b2 = b.copy()
    b2[:, 4] = np.nan
    full = _fit(b2, bt, iters=3)
    full.run()
    drop = _fit(np.delete(b, 4, axis=1), bt, iters=3)
    drop.run()
    nptest.assert_allclose(full.energy, drop.energy, rtol=1e-12)
    nptest.assert_allclose(full._lq_R, drop._lq_R, rtol=1e-9, atol=1e-12)


# ------------------------------------------------------------------ replica modes
def test_masked_replicas_equal_masked_fits():
    (b, bt) = _pattern("regions", *golden_inputs(20, 24, 24, seed=14), seed=15)
    corr = np.concatenate([b, bt], axis=1)
    labels = np.arange(48) >= 24
    opts = dict(max_iters=3, rel_tol=-1.0, missing="marginalize")
    res = sweep.permutation_sweep(corr, labels, 2, seed=1, fit_options=opts, streams=1)
    dev = _dev.device()
    corr_dev = torch.from_numpy(corr).to(dev)
    shared = sweep.SharedPlanes(corr_dev, fcdiff.UnsharedRegionModel(), missing="marginalize")
    fit = _fit(None, None, iters=3)
    fit.set_shared_inputs(shared, torch.arange(24), torch.arange(24, 48))
    fit.run()
    assert res[0]["energy"] == fit.energy
    plain = _fit(b, bt, iters=3)
    plain.run()
    nptest.assert_allclose(res[0]["energy"], plain.energy, rtol=1e-12)
    with pytest.raises(ValueError):                  # planes of the other mode
        other = _fit(None, None, missing="reject")
        other.set_shared_inputs(shared, torch.arange(24), torch.arange(24, 48))
        other.run()
    cv = sweep.cross_validate(corr, labels, n_folds=4, seed=3, fit_options=opts, streams=1)
    fold = cv["fold"]
    for name in ("log_odds", "control_loglik", "patient_elbo"):
        assert np.all(np.isfinite(cv[name]))
    i = 2
    train = fold != i
    f2 = _fit(None, None, iters=3)
    f2.set_shared_inputs(shared, torch.from_numpy(np.flatnonzero(train & ~labels)),
                         torch.from_numpy(np.flatnonzero(train & labels)))
    f2.run()
    held = np.flatnonzero(fold == i)
    k = f2.classify_subjects(corr_dev[:, torch.from_numpy(held).to(dev)])
    nptest.assert_array_equal(cv["log_odds"][held], k.log_odds)


# ------------------------------------------------------------------ K1
def test_correlations_mark_regions_without_a_time_series():
    rng = np.random.RandomState(0)
    (S, N, T) = (5, 70, 300)
    ts = rng.normal(size=(S, N, T)).astype(np.float32)
    ts[0, 3, 17] = np.nan
    ts[1, 40, :] = 2.0
    ts[2, 69, 0] = np.inf
    ts[4, 0, :] = np.nan
    full = corr.correlations(ts)
    masked = corr.correlations(ts, missing=True)
    (n, m) = O.edge_pairs(N)
    flag = np.zeros(full.shape, dtype=bool)
    for (s, r) in ((0, 3), (1, 40), (2, 69), (4, 0)):
        flag[(n == r) | (m == r), s] = True
    nptest.assert_array_equal(np.isnan(masked), flag)
    nptest.assert_array_equal(masked[~flag], full[~flag])
    ref = OM.corr_fisherz_masked(ts)
    nptest.assert_array_equal(np.isnan(ref), flag)


# ------------------------------------------------------------------ recovery
def test_planted_regions_are_recovered_under_region_dropout():
    """20 % of the (region, patient) pairs dropped out: region recall and precision above 0.9 when the
    dropped entries are marginalised.  The same numbers under zero imputation (r = 0, what K1 writes for a
    zero-variance row) are printed for comparison, not asserted."""
    th = O.Theta()
    (N, H, U) = (40, 60, 60)
    (r, _, _, _, b, bt) = O.sample(th, N, H, U, np.random.RandomState(21))
    rng = np.random.RandomState(22)
    (n, m) = O.edge_pairs(N)
    drop = rng.uniform(size=(N, U)) < 0.2
    bt_nan = bt.copy()
    for u in range(U):
        bt_nan[drop[n, u] | drop[m, u], u] = np.nan
    scores = {}
    for (name, x, missing) in (("marginalize", bt_nan, "marginalize"), ("zero", np.nan_to_num(bt_nan), "reject")):
        fit = _fit(b, x, missing=missing, iters=10, lookup="symmetric")
        fit.run()
        keep = ~drop
        pred = fit.map_anomalous_regions()
        tp = np.sum(pred & r & keep)
        scores[name] = (tp / max(np.sum(r & keep), 1), tp / max(np.sum(pred & keep), 1))
    print("region recall / precision on observed pairs:", scores)
    assert scores["marginalize"][0] > 0.9 and scores["marginalize"][1] > 0.9
