"""GPU parity tests: the CUDA path (through the reference-shaped Python API and
the ctypes C-ABI underneath) against the golden vectors produced by the
reference's own step functions and against the CPU oracle on seeded inputs.

Tolerances (BASELINE.json north_star): MAP labels bit-exact away from ties;
posteriors, parameters and free energy within 1e-6 relative.  The step-level
checks below are much tighter (1e-9 .. 1e-12) because they compare single
steps in float64; only transcendental ulp differences and summation order
separate the two sides.
"""
import numpy as np
import numpy.testing as nptest
import pytest
import torch

from oracle import iar_oracle as O
from oracle.make_golden import golden_inputs

pytestmark = pytest.mark.gpu

import fcdiff_b200 as fcdiff          # noqa: E402
from fcdiff_b200 import _lib          # noqa: E402

F = fcdiff.fit


@pytest.fixture(scope="module", autouse=True)
def _native_library_loaded():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    lib = _lib.load()                 # raises if libfcdiff_b200.so is missing
    n0 = lib.fcd_launch_count()
    yield
    assert lib.fcd_launch_count() > n0, "no kernel of libfcdiff_b200.so was launched"


def ideal_model():
    m = fcdiff.UnsharedRegionModel()
    (m.pi, m.epsilon, m.eta) = (0.1, 0.01, 0.3)
    m.gamma = np.ones((3,)) / 3
    m.mu = np.array([-0.5, 0, 0.5])
    m.sigma = np.ones((3,)) * 0.05
    return m


# ------------------------------------------------------------------ arrays API vs the reference's unit vectors
def test_update_lps_materialised(unit_vectors):
    g = unit_vectors
    (N, C, H, U) = (4, 6, 7, 5)
    fit = F.UnsharedRegionFit()
    fit.b, fit.bt = g["lps_b"], g["lps_bt"]
    fit.model = ideal_model()
    fit._init_lps(N, H, U)
    fit._update_lps()
    # bit-equal in the reference's own test; here exp/log (and the host's log sigma)
    # differ from NumPy's by <= 2 ulp of the operands
    nptest.assert_allclose(fit._lp_B_g_F, g["lps_lp_B_g_F"], rtol=4e-16, atol=2e-15)
    finite = np.isfinite(g["lps_lM"])
    nptest.assert_allclose(fit._p_Bt_g_Ft, g["lps_p_Bt_g_Ft"], rtol=1e-15, atol=0)
    nptest.assert_allclose(fit._lM[finite], g["lps_lM"][finite], rtol=1e-14, atol=0)
    nptest.assert_array_equal(np.isfinite(fit._lM), finite)


def test_eval_M_all_kl(unit_vectors):
    g = unit_vectors
    (eta, eps) = g["M_eta_eps"]
    for k in range(3):
        for l in range(3):
            nptest.assert_array_equal(F._eval_M(g["M_p"], eta, eps, k, l), g["M_out"][:, :, k, l])


def test_update_lq_F_arrays(unit_vectors):
    g = unit_vectors
    fit = F.UnsharedRegionFit()
    fit._lq_R = np.log(g["lqF_q_R"])
    fit._lp_B_g_F = g["lqF_lp_B_g_F"]
    fit._lM = g["lqF_lM"]
    fit.model = fcdiff.UnsharedRegionModel()
    fit.model.gamma = g["lqF_gamma"]
    fit._update_lq_F()
    assert fit._lq_F.shape == (15, 1, 3)
    nptest.assert_allclose(fit._lq_F, g["lqF_out"], rtol=1e-12)


@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
def test_update_lq_R_arrays(unit_vectors, lookup):
    g = unit_vectors
    fit = F.UnsharedRegionFit()
    fit._lq_R = np.log(g["lqR_q_R"])
    fit._lq_F = np.log(g["lqR_q_F"])
    fit._lM = g["lqR_lM"]
    fit.model = fcdiff.UnsharedRegionModel()
    fit.model.pi = g["lqR_pi"]
    fit.edge_lookup = lookup
    fit._update_lq_R()
    assert fit._lq_R.shape == (6, 4, 2)
    if lookup == "reference":
        nptest.assert_allclose(fit._lq_R, g["lqR_out"], rtol=1e-12)
    else:
        exp = O.update_lq_R(g["lqR_pi"], np.log(g["lqR_q_F"]), g["lqR_lM"], np.log(g["lqR_q_R"]), "symmetric")
        nptest.assert_allclose(fit._lq_R, exp, rtol=1e-12)


def test_update_pi_gamma(unit_vectors):
    g = unit_vectors
    fit = F.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    fit._lq_R = np.log(g["lqR_q_R"])
    fit._update_pi()
    nptest.assert_allclose(fit.model.pi, g["pi_out"], rtol=1e-14)
    assert np.ndim(fit.model.pi) == 0
    fit2 = F.UnsharedRegionFit()
    fit2.model = fcdiff.UnsharedRegionModel()
    fit2._lq_F = np.log(g["lqR_q_F"])
    fit2._update_gamma()
    assert fit2.model.gamma.shape == (3,)
    nptest.assert_allclose(fit2.model.gamma, g["gamma_out"], rtol=1e-14)


def test_energy_terms_arrays(unit_vectors):
    g = unit_vectors
    (q_F, q_R, lM) = (g["lqR_q_F"], g["lqR_q_R"], g["lqR_lM"])
    nptest.assert_allclose(F._eval_E_lp_F(q_F, g["E_gamma"]), g["E_lp_F"], rtol=1e-13)
    nptest.assert_allclose(F._eval_E_lp_B_g_F(q_F, g["E_lpB"]), g["E_lp_B_g_F"], rtol=1e-13)
    nptest.assert_allclose(F._eval_E_lp_R(q_R, g["lqR_pi"]), g["E_lp_R"], rtol=1e-13)
    nptest.assert_allclose(F._eval_E_lM(q_F, q_R, lM), g["E_lM"], rtol=1e-13)
    nptest.assert_allclose(F._eval_E_lq_F(q_F, np.log(q_F)), g["E_lq_F"], rtol=1e-13)
    nptest.assert_allclose(F._eval_E_lq_R(q_R, np.log(q_R)), g["E_lq_R"], rtol=1e-13)


def test_derivatives_arrays(unit_vectors):
    g = unit_vectors
    (eta, eps) = g["d_eta_eps"]
    (q_F, q_R) = (g["lqR_q_F"], g["lqR_q_R"])
    nptest.assert_allclose(F._eval_dE_dh(q_R, q_F, g["d_norm"], g["d_mix"], eps), g["dE_dh"], rtol=1e-11)
    nptest.assert_allclose(F._eval_dE_de(q_R, q_F, g["d_norm"], g["d_mix"], eta), g["dE_de"], rtol=1e-11)
    for k in range(3):
        nptest.assert_allclose(F._eval_dlM_dh(g["d_norm"], g["d_mix"][:, :, k, 2], eps, k),
                               g["dlM_dh"][:, :, k], rtol=1e-14)
        for l in range(3):
            nptest.assert_allclose(F._eval_dlM_de(g["d_norm"], g["d_mix"][:, :, k, l], eta, k, l),
                                   g["dlM_de"][:, :, k, l], rtol=1e-14)


def test_q_R_w(unit_vectors):
    g = unit_vectors
    w = F._eval_q_R_w(g["lqR_q_R"], 3, 1)
    assert w.shape == (4, 3)
    nptest.assert_array_equal(w, g["qRw_out"])


def test_eval_energy_arrays_mode(unit_vectors):
    g = unit_vectors
    fit = F.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    fit.model.gamma = g["E_gamma"]
    fit.model.pi = g["lqR_pi"]
    fit._lq_F = np.log(g["lqR_q_F"])
    fit._lq_R = np.log(g["lqR_q_R"])
    fit._lp_B_g_F = g["E_lpB"]
    fit._lM = g["lqR_lM"]
    exp = -g["E_lp_F"] - g["E_lp_B_g_F"] - g["E_lp_R"] - g["E_lM"] + g["E_lq_F"] + g["E_lq_R"]
    nptest.assert_allclose(fit._eval_energy(), exp, rtol=1e-12)


# ------------------------------------------------------------------ fused path vs the reference trajectory
SOLVERS = ["newton", "lbfgsb"]


def _fit_for(b, bt, model=None, eta_shift=0.0, solver="lbfgsb"):
    """``solver``: "lbfgsb" = SciPy's L-BFGS-B with its default tolerances, the optimiser call the
    reference-generated golden trajectories were produced with; "newton" = the device-resident
    solver (the package default), which converges to the minimiser itself -- its oracle is
    ``O.run(..., polish=True)``."""
    fit = F.UnsharedRegionFit()
    fit.b, fit.bt = b, bt
    fit.model = model or fcdiff.UnsharedRegionModel()
    fit.model.eta += eta_shift
    fit.theta_solver = solver
    return fit


def test_cfg1_fused_iterations_without_optimiser(cfg1):
    g = cfg1
    fit = _fit_for(g["b"], g["bt"])
    fit._init_lps(10, 20, 20)
    fit._update_lps()
    for it in range(2):
        fit._update_lq_F()
        fit._update_lq_R()
        fit._update_pi()
        fit._update_gamma()
        nptest.assert_allclose(fit._lq_F, g["noopt_it%d_lq_F" % it], rtol=1e-9, atol=1e-10)
        nptest.assert_allclose(fit._lq_R, g["noopt_it%d_lq_R" % it], rtol=1e-9, atol=1e-10)
        nptest.assert_allclose(fit.model.pi, g["noopt_it%d_pi" % it], rtol=1e-11)
        nptest.assert_allclose(fit.model.gamma, g["noopt_it%d_gamma" % it], rtol=1e-11)
        nptest.assert_allclose(fit._energy_terms(), g["noopt_it%d_terms" % it], rtol=1e-10)
        nptest.assert_allclose(fit._eval_energy(), g["noopt_it%d_energy" % it], rtol=1e-10)
    for x, fg in zip(g["noopt_obj_pts"], g["noopt_obj_fg"]):
        (f, grad) = fit._objective(x)
        nptest.assert_allclose(f, fg[0], rtol=1e-10)
        # the gradient uses 1/M' = r(1 - u + u^2): truncation <= 9.3e-10 relative (fcd_math.cuh)
        nptest.assert_allclose(grad, fg[1:], rtol=5e-9)
        nptest.assert_allclose(fit._opt_fun(np.array(x)), fg[0], rtol=1e-10)


def _check_run(fit, g, final_only=False, tol_theta=1e-6, tol_q=1e-6):
    nptest.assert_allclose(fit.energy, g["energy"], rtol=1e-6)
    assert len(fit.energy) == len(g["energy"])
    nptest.assert_allclose([fit.model.pi, fit.model.eta, fit.model.epsilon],
                           [g["pi"][-1], g["eta"][-1], g["epsilon"][-1]], rtol=tol_theta)
    nptest.assert_allclose(fit.model.gamma, g["gamma"][-1], rtol=1e-6)
    lqF = g["lq_F_final"] if final_only else g["lq_F"][-1]
    lqR = g["lq_R_final"] if final_only else g["lq_R"][-1]
    nptest.assert_allclose(np.exp(fit._lq_F), np.exp(lqF), rtol=tol_q, atol=1e-300)
    nptest.assert_allclose(np.exp(fit._lq_R), np.exp(lqR), rtol=tol_q, atol=1e-300)
    # MAP labels bit-exact away from ties
    gap_F = np.sort(lqF, axis=2)
    clear = (gap_F[:, :, 2] - gap_F[:, :, 1]) > 1e-6
    nptest.assert_array_equal(np.argmax(fit._lq_F, axis=2)[clear], np.argmax(lqF, axis=2)[clear])
    clear_R = np.abs(lqR[:, :, 1] - lqR[:, :, 0]) > 1e-6
    nptest.assert_array_equal((fit._lq_R[:, :, 1] > fit._lq_R[:, :, 0])[clear_R],
                              (lqR[:, :, 1] > lqR[:, :, 0])[clear_R])
    assert clear.mean() > 0.99 and clear_R.mean() > 0.99


# The golden trajectories were produced by the reference's step functions with SciPy's L-BFGS-B at
# its DEFAULT tolerances, which stops 1e-7 .. 2e-6 (relative) short of the minimiser of the (eta,
# epsilon) sub-problem (measured with the oracle: tests/test_oracle_golden.py::test_polish_*).
# "lbfgsb" repeats that optimiser call iterate for iterate and is held to 1e-6 everywhere; "newton"
# converges to the minimiser itself, so against THESE files its theta / posteriors are held to the
# optimiser slack of the golden run (and to 1e-6 against the polished oracle, test_newton_*).
_GOLDEN_TOL = {"lbfgsb": dict(), "newton": dict(tol_theta=2e-5, tol_q=5e-4)}


@pytest.mark.parametrize("solver", SOLVERS)
def test_cfg1_full_run_matches_reference(cfg1, solver):
    g = cfg1
    fit = _fit_for(g["b"], g["bt"], eta_shift=0.1, solver=solver)
    fit.run()
    _check_run(fit, g, **_GOLDEN_TOL[solver])
    assert isinstance(fit.energy, list) and fit._lq_F.shape == (45, 1, 3) and fit._lq_R.shape == (10, 20, 2)


@pytest.mark.parametrize("solver", SOLVERS)
def test_cfg2_full_run_matches_reference(cfg2, solver):
    g = cfg2
    (b, bt) = golden_inputs(90, 50, 50)
    fit = _fit_for(b, bt, eta_shift=0.1, solver=solver)
    fit.run()
    _check_run(fit, g, final_only=True, **_GOLDEN_TOL[solver])


@pytest.mark.parametrize("N,H,U,iters", [(10, 20, 20, 6), (24, 9, 33, 4), (90, 50, 50, 3)])
@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
def test_newton_solver_full_run_vs_polished_oracle(N, H, U, iters, lookup):
    """The default (device-resident Newton) solver against the oracle whose (eta, epsilon) solve is
    polished to the minimiser: energies, parameters and posteriors at 1e-6, MAP labels exact away
    from ties; every solve must report convergence within a handful of evaluations."""
    (_, _, _, _, b, bt) = O.sample(O.Theta(), N, H, U, np.random.RandomState(N + 1))
    fit = _fit_for(b, bt, eta_shift=0.1, solver="newton")
    fit.edge_lookup = lookup
    fit.max_iters = iters
    fit.rel_tol = -1.0
    fit.run()
    tho = O.Theta()
    tho.eta += 0.1
    out = O.run(b, bt, tho, max_iters=iters, rel_tol=-1.0, edge_lookup=lookup, polish=True)
    nptest.assert_allclose(fit.energy, out["energy"], rtol=1e-6)
    nptest.assert_allclose([fit.model.pi, fit.model.eta, fit.model.epsilon], [tho.pi, tho.eta, tho.epsilon], rtol=1e-6)
    nptest.assert_allclose(fit.model.gamma, tho.gamma, rtol=1e-6)
    nptest.assert_allclose(np.exp(fit._lq_F), np.exp(out["lq_F"]), rtol=1e-6, atol=1e-300)
    nptest.assert_allclose(np.exp(fit._lq_R), np.exp(out["lq_R"]), rtol=1e-6, atol=1e-300)
    assert len(fit.solver_status) == iters
    assert all(done == 1 and nfev <= 12 for (done, nfev) in fit.solver_status), fit.solver_status


@pytest.mark.parametrize("N,H,U,iters", [(24, 9, 33, 5), (90, 50, 50, 4), (160, 40, 400, 10)])
def test_speculative_estep_is_bit_identical(N, H, U, iters):
    """`run()` enqueues the next iteration's E-step behind the device-resident (eta, epsilon) solve
    (fcd_estep_qF_coded with a solver state: theta read from the solver's state block on the device) and adopts it
    when nothing changed: the same fit with the feature off must give the same numbers bit for bit, the
    launches must actually be adopted, and a fit that stops leaves no stray result behind."""
    (_, _, _, _, b, bt) = O.sample(O.Theta(), N, H, U, np.random.RandomState(3 * N + 1))

    def run(spec, stop=None):
        fit = _fit_for(b, bt, eta_shift=0.1, solver="newton")
        fit.speculative_estep = spec
        fit.max_iters = iters if stop is None else stop
        fit.rel_tol = -1.0
        fit.run()
        return fit

    (f1, f0) = (run(True), run(False))
    assert f0.spec_stats == [0, 0]
    # the first iteration's E-step takes the uniform-start path and the last M-step launches none
    assert f1.spec_stats[1] <= f1.spec_stats[0] <= iters - 1, f1.spec_stats
    if N >= 160:           # (small problems keep the tiered forms -- no code plane, nothing to launch early -- or
        #                     need more evaluations than the first batch holds: the launch is dropped)
        assert f1.spec_stats[1] >= 1, (f1.spec_stats, f1.solver_status)
    assert f1.energy == f0.energy
    assert (f1.model.pi, f1.model.eta, f1.model.epsilon) == (f0.model.pi, f0.model.eta, f0.model.epsilon)
    nptest.assert_array_equal(f1._lq_F, f0._lq_F)
    nptest.assert_array_equal(f1._lq_R, f0._lq_R)
    # stepping by hand after run(): nothing speculative is pending, the step functions behave as before
    f1._update_lq_F()
    f0._update_lq_F()
    nptest.assert_array_equal(f1._lq_F, f0._lq_F)
    assert f1._spec is None


@pytest.mark.parametrize("N,H,U,iters,lookup", [(12, 9, 11, 3, "reference"), (33, 20, 70, 4, "symmetric"),
                                                 (90, 50, 50, 4, "reference"), (120, 30, 333, 5, "reference")])
def test_region_weights_from_edge_major_planes_vs_oracle(N, H, U, iters, lookup):
    """The region weights read the E-step's edge-major planes (fcd_region_weights_em: the dominant-state plane
    gathered by a transposing pass, unpeaked edges through strided reads).  The small problems keep unpeaked
    edges and undecided regions for several iterations, the odd sizes exercise the partial 32 x 32 tiles of the
    gather."""
    (_, _, _, _, b, bt) = O.sample(O.Theta(), N, H, U, np.random.RandomState(7 * N + U))
    fit = _fit_for(b, bt, eta_shift=0.1, solver="newton")
    fit.edge_lookup = lookup
    fit.max_iters = iters
    fit.rel_tol = -1.0
    fit.run()
    # against the oracle (polished optimiser = the device Newton solver's fixed point)
    tho = O.Theta()
    tho.eta += 0.1
    out = O.run(b, bt, tho, max_iters=iters, rel_tol=-1.0, edge_lookup=lookup, polish=True)
    nptest.assert_allclose(fit.energy, out["energy"], rtol=1e-6)
    nptest.assert_allclose(np.exp(fit._lq_R), np.exp(out["lq_R"]), rtol=1e-6, atol=1e-300)


def test_newton_solver_reaches_active_bounds_and_leaves_the_table_window():
    """Start points far from the minimiser: epsilon has to travel more than the factor 8 one pass of
    the solver may move it (the box that sizes the kernels' logarithm table), and a problem whose
    minimiser sits ON the reference's bound 1e-5 (patients drawn with epsilon = 0: no edge deviates
    from the template beyond the region effects)."""
    th_true = O.Theta()
    (_, _, _, _, b, bt) = O.sample(th_true, 20, 12, 40, np.random.RandomState(4))
    for (eta0, eps0) in ((0.6, 0.3), (0.02, 0.0004), (0.7, 0.002)):     # all in the basin of the minimiser with epsilon < 1/2
        model = fcdiff.UnsharedRegionModel()
        (model.eta, model.epsilon) = (eta0, eps0)
        fit = _fit_for(b, bt, model, solver="newton")
        fit.max_iters = 2
        fit.rel_tol = -1.0
        fit.run()
        tho = O.Theta(eta=eta0, epsilon=eps0)
        out = O.run(b, bt, tho, max_iters=2, rel_tol=-1.0, polish=True)
        nptest.assert_allclose([fit.model.eta, fit.model.epsilon], [tho.eta, tho.epsilon], rtol=1e-6)
        nptest.assert_allclose(fit.energy, out["energy"], rtol=1e-6)
    th0 = O.Theta(epsilon=1e-9, pi=0.0001)
    (_, _, _, _, b, bt) = O.sample(th0, 12, 10, 30, np.random.RandomState(8))
    fit = _fit_for(b, bt, solver="newton")
    fit.max_iters = 3
    fit.rel_tol = -1.0
    fit.run()
    tho = O.Theta()
    out = O.run(b, bt, tho, max_iters=3, rel_tol=-1.0, polish=True)
    nptest.assert_allclose(fit.energy, out["energy"], rtol=1e-6)
    nptest.assert_allclose(fit.model.epsilon, tho.epsilon, rtol=1e-6, atol=1e-12)
    assert tho.epsilon == 1e-5 and fit.model.epsilon == 1e-5          # both sit on the reference's lower bound
    nptest.assert_allclose(fit.model.eta, tho.eta, rtol=1e-5)


# ------------------------------------------------------------------ fused path vs the oracle on seeded inputs
def _oracle_state(b, bt, th, seed, peaked=False):
    """Random posteriors; ``peaked``: most of them one-hot to rounding (q = 1.0
    exactly, the rest ~1e-25 .. 1e-40), as they are after an EM iteration --
    this is what sends the kernels down their T1 / T2 tiers."""
    (C, H) = b.shape
    U = bt.shape[1]
    N = int(O.C_to_N(C))
    rng = np.random.RandomState(seed)
    q_R = rng.dirichlet([1, 1], size=(N, U))
    q_F = rng.dirichlet([1, 1, 1], size=(C, 1))
    if peaked:
        hot = rng.rand(N, U) < 0.9
        one = (rng.rand(N, U) < 0.15).astype(int)
        pk = np.full((N, U, 2), 1e-25)
        pk[np.arange(N)[:, None], np.arange(U)[None, :], one] = 1.0
        q_R[hot] = pk[hot]
        hotF = rng.rand(C) < 0.9
        kk = rng.randint(0, 3, size=C)
        pkF = np.full((C, 1, 3), 1e-30)
        pkF[np.arange(C), 0, kk] = 1.0
        pkF[np.arange(C), 0, (kk + 1) % 3] = 1e-40
        q_F[hotF] = pkF[hotF]
    return N, H, U, np.log(q_F), np.log(q_R)


@pytest.mark.parametrize("N,H,U", [(3, 1, 1), (4, 2, 3), (7, 5, 9), (10, 20, 20), (33, 17, 31), (40, 64, 128),
                                   (24, 8, 300),
                                   # N >= 64: the blocked sweep, and its fused form (weights formed in the far loop;
                                   # unpeaked edges -- peaked = False -- take its three-plane path)
                                   (70, 4, 9), (100, 3, 33)])
@pytest.mark.parametrize("lookup", ["reference", "symmetric"])
@pytest.mark.parametrize("peaked", [False, True])
def test_fused_steps_vs_oracle(N, H, U, lookup, peaked):
    th = O.Theta() if (N % 2) else O.Theta.ideal()
    (_, _, _, _, b, bt) = O.sample(th, N, H, U, np.random.RandomState(N))
    (N, H, U, lq_F, lq_R) = _oracle_state(b, bt, th, N + 1, peaked)
    (lpB, pBt, lM) = O.update_lps(b, bt, th)
    model = fcdiff.UnsharedRegionModel()
    (model.pi, model.eta, model.epsilon) = (th.pi, th.eta, th.epsilon)
    (model.gamma, model.mu, model.sigma) = (th.gamma.copy(), th.mu.copy(), th.sigma.copy())
    fit = _fit_for(b, bt, model)
    fit.edge_lookup = lookup
    fit._init_lps(N, H, U)
    fit._update_lps()
    fit._lq_R = lq_R
    fit._lq_F = lq_F
    # K4 at a random state
    terms = O.eval_energy_terms(th, lq_F, lq_R, lpB, lM)
    nptest.assert_allclose(fit._energy_terms(), terms, rtol=1e-10)
    # K2
    fit._update_lq_F()
    exp_F = O.update_lq_F(th.gamma, lpB, lM, lq_R)
    nptest.assert_allclose(fit._lq_F, exp_F, rtol=1e-9, atol=1e-10)
    nptest.assert_allclose(np.exp(fit._lq_F).sum(axis=2), 1.0, rtol=1e-12)
    # K2b: region weights + sweep over WT
    exp_R = O.update_lq_R(np.array([1 - th.pi, th.pi]), exp_F, lM, lq_R, lookup)
    fit._update_lq_R()
    nptest.assert_allclose(fit._lq_R, exp_R, rtol=1e-9, atol=1e-10)
    # K3a
    fit._update_pi()
    fit._update_gamma()
    nptest.assert_allclose(fit.model.pi, O.update_pi(exp_R), rtol=1e-10)
    nptest.assert_allclose(fit.model.gamma, O.update_gamma(exp_F), rtol=1e-10)
    # K3b objective + analytic gradient at interior and near-bound points
    # (both forms of the kernel: bucketed streams and tiered walk over the planes)
    for path in ("tiered", "streams", "auto"):
        fit.elm_path = path
        for x in ([0.3, 0.03], [0.7, 0.4], [1e-5, 1 - 1e-5], [1 - 1e-5, 1e-5]):
            (f, grad) = fit._objective(x)
            (fo, go) = O.elm_objective_and_grad(pBt, np.exp(exp_F), np.exp(exp_R), x)
            nptest.assert_allclose(f, fo, rtol=1e-10)
            nptest.assert_allclose(grad, go, rtol=1e-8, atol=1e-8 * max(1.0, np.abs(go).max()))
        assert fit._ctx['name'] == {"tiered": "K3b_elm_obj_grad", "streams": "K3b_elm_streams"}.get(path, fit._ctx['name'])
    # K3c sufficient statistics for mu / sigma
    mom = fit._state_moments()
    momo = O.state_moments(b, bt, th, np.exp(exp_F), np.exp(exp_R))
    nptest.assert_allclose(mom, momo, rtol=1e-9, atol=1e-9 * np.abs(momo).max())


@pytest.mark.parametrize("solver", SOLVERS)
def test_mu_sigma_update_vs_oracle_and_lowers_energy(solver):
    """mu / sigma re-estimation (disabled in the reference, fit.py:232-237): the
    GPU fit with ``update_mu_sigma`` follows the oracle's trajectory, and the
    generalised-EM step never raises the free energy."""
    th_true = O.Theta()
    (_, _, _, _, b, bt) = O.sample(th_true, 16, 30, 25, np.random.RandomState(11))
    model = fcdiff.UnsharedRegionModel()
    model.mu = np.array([-0.2, 0.02, 0.25])
    model.sigma = np.array([0.04, 0.05, 0.07])
    fit = _fit_for(b, bt, model, solver=solver)
    fit.update_mu_sigma = True
    fit.edge_lookup = "symmetric"    # a true coordinate descent (the reference's lookup quirk is not, SURVEY 0.3)
    fit.max_iters = 4
    fit.rel_tol = -1.0               # run all iterations
    fit.run()
    tho = O.Theta(mu=(-0.2, 0.02, 0.25), sigma=(0.04, 0.05, 0.07))
    out = O.run(b, bt, tho, max_iters=4, rel_tol=-1.0, update_mu_sigma=True, edge_lookup="symmetric",
                polish=(solver == "newton"))
    nptest.assert_allclose(fit.energy, out["energy"], rtol=1e-6)
    nptest.assert_allclose(fit.model.mu, tho.mu, rtol=1e-6, atol=1e-9)
    nptest.assert_allclose(fit.model.sigma, tho.sigma, rtol=1e-6)
    nptest.assert_allclose([fit.model.pi, fit.model.eta, fit.model.epsilon], [tho.pi, tho.eta, tho.epsilon], rtol=1e-6)
    assert np.all(np.diff(fit.energy) < 0)
    # the re-estimated parameters moved towards the generating ones
    assert np.abs(fit.model.mu - th_true.mu).max() < 0.02
    assert np.abs(fit.model.sigma - th_true.sigma).max() < 0.01


@pytest.mark.parametrize("solver", SOLVERS)
def test_full_run_symmetric_lookup_vs_oracle(solver):
    th = O.Theta()
    (_, _, _, _, b, bt) = O.sample(th, 14, 12, 15, np.random.RandomState(5))
    fit = _fit_for(b, bt, eta_shift=0.1, solver=solver)
    fit.edge_lookup = "symmetric"
    fit.max_iters = 5
    fit.run()
    tho = O.Theta()
    tho.eta += 0.1
    out = O.run(b, bt, tho, max_iters=5, edge_lookup="symmetric", polish=(solver == "newton"))
    nptest.assert_allclose(fit.energy, out["energy"], rtol=1e-6)
    nptest.assert_allclose(np.exp(fit._lq_F), np.exp(out["lq_F"]), rtol=1e-6, atol=1e-300)
    nptest.assert_allclose(np.exp(fit._lq_R), np.exp(out["lq_R"]), rtol=1e-6, atol=1e-300)
    nptest.assert_allclose([fit.model.pi, fit.model.eta, fit.model.epsilon], [tho.pi, tho.eta, tho.epsilon], rtol=1e-6)


def test_far_tail_inputs_stay_finite():
    """Fisher-z inputs can leave [-1, 1]; the reference's pdf underflows there
    (-inf / nan), the log-domain kernels must stay finite and agree with the
    oracle wherever the oracle is finite."""
    th = O.Theta()
    rng = np.random.RandomState(3)
    (N, H, U) = (6, 4, 8)
    b = rng.uniform(-1, 1, (15, H))
    bt = rng.uniform(-2.5, 2.5, (15, U))
    fit = _fit_for(b, bt)
    fit._init_lps(N, H, U)
    fit._update_lps()
    fit._update_lq_F()
    fit._update_lq_R()
    assert np.all(np.isfinite(fit._lq_F)) and np.all(np.isfinite(fit._lq_R))
    assert np.isfinite(fit._eval_energy())


def test_single_region_pair_rejected_in_reference_lookup():
    fit = _fit_for(np.zeros((1, 2)), np.zeros((1, 2)))
    fit._init_lps(2, 2, 2)
    fit._update_lps()
    fit._update_lq_F()
    with pytest.raises(_lib.FcdError, match="N < 3"):
        fit._update_lq_R()
    fit.edge_lookup = "symmetric"
    fit._update_lq_R()
    assert fit._lq_R.shape == (2, 2, 2)


# ------------------------------------------------------------------ size-independent properties at BASELINE sizes
def _device_problem(N, H, U, seed=0, planted=False):
    model = fcdiff.UnsharedRegionModel()
    model.rng = np.random.RandomState(seed)
    (r, t, f, ft, b, bt) = model.sample_device(N, H, U)
    if planted:
        return model, b, bt, f.cpu().numpy() > 0, r.cpu().numpy() > 0
    return model, b, bt


@pytest.mark.parametrize("solver,variant", [("newton", "polished"), ("lbfgsb", "lbfgsb")])
def test_config3_two_iterations_vs_oracle_golden(solver, variant):
    """The BENCHMARKED configuration (Schaefer-400 x 500 + 500) against the oracle: two full
    ``run()`` iterations from the uniform start.  The oracle takes ~20 minutes and 13 GB at this
    size, so its result is a committed fixture (oracle/make_golden_cfg3.py; inputs regenerated here
    bit-identically by the same NumPy sampler call): energies, theta, a fixed random sample of
    40,000 entries of each posterior at 1e-6, checksums, and the MAP labels of ALL 79,800 edges and
    200,000 (region, patient) pairs exact away from ties."""
    import os
    from oracle import make_golden_cfg3 as G
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cfg3_run2_%s.npz" % variant)
    assert os.path.isfile(path), "fixture missing: run oracle/make_golden_cfg3.py %s" % variant
    with np.load(path) as z:
        g = {k: z[k] for k in z.files}
    (b, bt) = G.inputs()
    assert b.shape == (79800, 500) and bt.shape == (79800, 500)
    fit = _fit_for(b, bt, eta_shift=0.1, solver=solver)
    fit.max_iters = G.ITERS
    fit.rel_tol = -1.0
    fit.run()
    nptest.assert_allclose(fit.energy, g["energy"], rtol=1e-6)
    nptest.assert_allclose([fit.model.pi, fit.model.eta, fit.model.epsilon],
                           [g["pi"][-1], g["eta"][-1], g["epsilon"][-1]], rtol=1e-6)
    nptest.assert_allclose(fit.model.gamma, g["gamma"][-1], rtol=1e-6)
    (lqF, lqR) = (fit._lq_F, fit._lq_R)
    got = G.summarise(lqF, lqR)
    nptest.assert_allclose(np.exp(got["lq_F_sample"]), np.exp(g["lq_F_sample"]), rtol=1e-6, atol=1e-300)
    nptest.assert_allclose(np.exp(got["lq_R_sample"]), np.exp(g["lq_R_sample"]), rtol=1e-6, atol=1e-300)
    nptest.assert_allclose(got["sum_qF"], g["sum_qF"], rtol=1e-9)
    nptest.assert_allclose(got["sum_qR"], g["sum_qR"], rtol=1e-9)
    nptest.assert_allclose([got["ent_F"], got["ent_R"]], [g["ent_F"], g["ent_R"]], rtol=1e-6, atol=1e-6)
    # MAP labels bit-exact away from ties (the fixture carries the oracle's own "clear" flags)
    clearF = np.unpackbits(g["gap_F"])[:79800].astype(bool)
    mapF = lambda a: (np.unpackbits(a)[:2 * 79800].reshape(-1, 2) * np.array([1, 2])).sum(axis=1)
    nptest.assert_array_equal(mapF(got["map_F"])[clearF], mapF(g["map_F"])[clearF])
    clearR = np.unpackbits(g["gap_R"])[:400 * 500].astype(bool)
    nptest.assert_array_equal(np.unpackbits(got["map_R"])[:400 * 500][clearR], np.unpackbits(g["map_R"])[:400 * 500][clearR])
    assert clearF.mean() > 0.99 and clearR.mean() > 0.99
    if solver == "newton":
        assert all(done == 1 for (done, _) in fit.solver_status), fit.solver_status


@pytest.mark.parametrize("N,H,U", [(400, 500, 500)])
def test_config3_invariants(N, H, U):
    """Schaefer-400 x 1000 subjects: shard additivity, determinism,
    normalisation, energy consistency -- no CPU oracle at this size."""
    import ctypes
    from fcdiff_b200 import _dev
    lib = _lib.load()
    (model, b_dev, bt_dev, f_true, r_true) = _device_problem(N, H, U, planted=True)
    C = N * (N - 1) // 2
    fit = F.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    fit.b = _dev.download(b_dev)
    fit.bt = _dev.download(bt_dev)
    fit.max_iters = 2
    fit.run()
    q_F = np.exp(fit._lq_F)
    q_R = np.exp(fit._lq_R)
    nptest.assert_allclose(q_F.sum(axis=2), 1.0, rtol=1e-12)
    nptest.assert_allclose(q_R.sum(axis=2), 1.0, rtol=1e-12)
    assert len(fit.energy) >= 2 and np.all(np.isfinite(fit.energy))
    # the fit lowers the free energy from the uniform start
    assert fit.energy[1] < fit.energy[0]
    # planted template recovered (b, bt were drawn from the default model by the device sampler): the MAP of q_F
    # equals the sampled f on > 99.5 % of the edges.  (The planted REGIONS are only recoverable with
    # edge_lookup="symmetric": test_fit_recovers_planted_template_and_regions.)
    assert (np.argmax(fit._lq_F[:, 0, :], axis=1) == np.argmax(f_true, axis=1)).mean() > 0.995
    # -- determinism: a second run is bit-identical
    fit2 = F.UnsharedRegionFit()
    fit2.model = fcdiff.UnsharedRegionModel()
    fit2.b, fit2.bt = fit.b, fit.bt
    fit2.max_iters = 2
    fit2.run()
    nptest.assert_array_equal(fit2._lq_F, fit._lq_F)
    nptest.assert_array_equal(fit2._lq_R, fit._lq_R)
    assert fit2.energy == fit.energy
    # -- shard additivity of K3b (objective, gradient, theta-free part): sum over 3 ragged edge shards == whole
    inp = fit._ensure_cache()
    (lqF, qF) = fit._mF.get_dev()
    (lqR, qR) = fit._mR.get_dev()
    (fstate, rstate) = (fit._mF.get_state(), fit._mR.get_state())
    th = fit._theta()
    ws = _dev.workspace()
    (P, pitch, pitchS) = (inp['P'], inp['pitchU'], rstate.shape[1])

    def elm(a, e, fst=None, rst=None, grad=1):
        fst = fstate if fst is None else fst
        rst = rstate if rst is None else rst
        out = _dev.empty((4,))
        _lib.check(lib.fcd_elm_obj_grad(
            _dev.ptr(P[0, a:]), C * pitch, e - a, U, pitch, _dev.ptr(qF[a * 3:]), _dev.ptr(fst[a:]), _dev.ptr(qR),
            _dev.ptr(rst), pitchS, N, _dev.ptr(inp['nm'][a:]), ctypes.byref(th), grad, _dev.ptr(out), _dev.ptr(ws),
            _dev.stream()))
        _lib.check(lib.fcd_elm_const(
            _dev.ptr(inp['L'][a:]), e - a, U, pitch, _dev.ptr(qF[a * 3:]), _dev.ptr(fst[a:]), _dev.ptr(qR),
            _dev.ptr(rst), pitchS, N, _dev.ptr(inp['nm'][a:]), _dev.ptr(out[3:]), _dev.ptr(ws), _dev.stream()))
        return _dev.download(out)

    w = elm(0, C)
    cuts = [0, 1234, 40001, C]
    parts = sum(elm(a, e) for (a, e) in zip(cuts[:-1], cuts[1:]))
    gtol = 1e-13 * abs(w[0])              # the gradient is a cancelling sum of terms of the objective's size
    nptest.assert_allclose(parts[[0, 3]], w[[0, 3]], rtol=1e-12)
    nptest.assert_allclose(parts[1:3], w[1:3], rtol=0, atol=gtol)
    # -- tiers: with every peak state forced to "not peaked" the kernels take the reference's
    #    nine-log form for every element; the tiered result must agree to rounding
    f_mixed = torch.full_like(fstate, 3)
    r_mixed = rstate.clone()
    r_mixed[r_mixed < 2] = 2
    assert float((fstate < 3).float().mean()) > 0.99 and float((rstate < 2).float().mean()) > 0.5
    for (fs_, rs_) in ((f_mixed, r_mixed), (fstate, r_mixed), (f_mixed, rstate)):
        v = elm(0, C, fs_, rs_)
        nptest.assert_allclose(v[[0, 3]], w[[0, 3]], rtol=1e-12)
        nptest.assert_allclose(v[1:3], w[1:3], rtol=0, atol=gtol)
    nptest.assert_allclose(elm(0, C, f_mixed, r_mixed, grad=0)[[0, 3]], w[[0, 3]], rtol=1e-12)
    # -- the energy from a reused K3b evaluation equals the energy from a fresh pass
    fit.reuse_evaluations = False
    e_fresh = fit._eval_energy()
    fit.reuse_evaluations = True
    nptest.assert_allclose(fit._eval_energy(), e_fresh, rtol=1e-13)
    nptest.assert_allclose(fit.energy[-1], e_fresh, rtol=1e-13)
    nptest.assert_allclose(fit._energy_terms()[3], w[0] + w[3], rtol=1e-12)
    # -- the bucketed-streams form of K3b equals the tiered walk over the planes
    res = {}
    for path in ("tiered", "streams"):
        fit.elm_path = path
        res[path] = fit._objective([th.eta, th.epsilon])
        assert fit._ctx['name'] == ("K3b_elm_streams" if path == "streams" else "K3b_elm_obj_grad")
    nptest.assert_allclose(res["streams"][0], res["tiered"][0], rtol=1e-13)
    nptest.assert_allclose(res["streams"][1], res["tiered"][1], rtol=0, atol=gtol)
    nptest.assert_allclose(-res["streams"][0], w[0] + w[3], rtol=1e-12)
    fit.elm_path = "auto"
    # -- K2 on a shard equals the slice of the whole; tiered K2 equals the all-deferred form
    (a, e) = (40001, C)

    def estep(a, e, rst):
        lq = _dev.empty(((e - a) * 3,))
        _lib.check(lib.fcd_estep_qF(_dev.ptr(inp['S1'][a:]), _dev.ptr(inp['S2'][a:]), None, H, _dev.ptr(P[0, a:]),
                                    C * pitch, e - a, U, pitch, _dev.ptr(qR), _dev.ptr(rst), pitchS, N, _dev.ptr(inp['nm'][a:]),
                                    ctypes.byref(th), _dev.ptr(lq), None, _dev.stream()))
        return _dev.download(lq)

    whole = estep(0, C, rstate)
    nptest.assert_array_equal(estep(a, e, rstate), whole[a * 3:])
    nptest.assert_allclose(estep(0, C, r_mixed), whole, rtol=1e-12, atol=1e-9)


@pytest.mark.parametrize("N,H,U", [(4, 2, 3), (10, 20, 20), (24, 8, 129), (33, 17, 300)])
def test_uniform_start_fast_path_equals_general_kernels_and_oracle(N, H, U):
    """The uniform start (fit.py:84-102): the row log-sums of csrc/fcd_uniform.cu (nine running products per
    row) must give the initial free energy and the first E-step of the general kernels (nine
    logarithms per element) and of the oracle."""
    th = O.Theta()
    (_, _, _, _, b, bt) = O.sample(th, N, H, U, np.random.RandomState(N))
    out = {}
    for fast in (True, False):
        fit = _fit_for(b, bt, eta_shift=0.1)
        fit.uniform_fast_path = fast
        fit._init_lps(N, H, U)
        fit._update_lps()
        e0 = fit._eval_energy()
        fit._update_lq_F()
        out[fast] = (e0, fit._lq_F.copy())
        if fast:
            assert 'rowsums' in fit._in
    nptest.assert_allclose(out[True][0], out[False][0], rtol=1e-12)
    nptest.assert_allclose(out[True][1], out[False][1], rtol=1e-10, atol=1e-10)
    tho = O.Theta()
    tho.eta += 0.1
    (lq_F, lq_R) = O.init_lps(N, U)
    (lpB, p, lM) = O.update_lps(b, bt, tho)
    nptest.assert_allclose(out[True][0], O.energy_from_terms(O.eval_energy_terms(tho, lq_F, lq_R, lpB, lM)), rtol=1e-10)
    nptest.assert_allclose(out[True][1], O.update_lq_F(tho.gamma, lpB, lM, lq_R), rtol=1e-9, atol=1e-10)


# ------------------------------------------------------------------ config 4 geometry: one edge shard vs the oracle
class _RowWindow(object):
    """Stands in for ``dist.EdgeShards`` on ONE process: this 'rank' owns the edge rows
    [c0, c0 + Cl) of a larger atlas and all patients; every exchange is the identity.  Lets the
    edge-local steps (K2, K3b, code pass) run through the product path on a slice of a problem
    whose full arrays the oracle cannot hold (config 4: 499,500 edges x 1000 + 1000)."""

    (rank, world) = (0, 1)

    def __init__(self, c0, Cl):
        (self.c0, self.Cl) = (c0, Cl)

    def key(self):
        return ("rows", self.c0, self.Cl)

    def ranges(self, C, U):
        return (self.c0, self.Cl, 0, U)

    def peer_window(self):
        return None

    def reduce_read(self, res, n=None, stream=None):
        return res.read(stream)

    def any_rank(self, flag):
        return bool(flag)

    def fix_replicated(self, host_vec, idxs):
        return host_vec

    def edge_buffer_len(self, C):
        return C * 3

    def allgather_edges(self, lqF, qF, C):
        pass


@pytest.mark.parametrize("c0,Cl", [(123456, 1536), (499500 - 700, 700)])
def test_config4_edge_shard_vs_oracle(c0, Cl):
    """BASELINE.json configs[3] (1000 regions = 499,500 edges, 1000 + 1000 subjects): the rows
    [c0, c0 + Cl) through the product path -- rows of 1000 patients (8 TMA segments, code pitch 1008 !=
    U), region indices up to 999, peaked and undecided posteriors -- against the oracle restricted
    to the same rows: K2 (both kernels), the K3b objective / gradient (tiered and coded form)."""
    (N, H, U) = (1000, 1000, 1000)
    C = N * (N - 1) // 2
    th = O.Theta()
    rng = np.random.RandomState(c0 % 1000)
    (n_all, m_all) = O.edge_pairs(N)
    (n, m) = (n_all[c0:c0 + Cl], m_all[c0:c0 + Cl])
    # rows drawn like model.sample: template state per edge, patients deviate with probability ~ epsilon
    fk = rng.choice(3, size=Cl, p=th.gamma)
    b = rng.normal(th.mu[fk][:, None], th.sigma[fk][:, None], (Cl, H)).clip(-1, 1)
    ftk = np.where(rng.rand(Cl, U) < 0.06, rng.choice(3, size=(Cl, U)), fk[:, None])
    bt = rng.normal(th.mu[ftk], th.sigma[ftk]).clip(-1, 1)
    # region posteriors as they are after an iteration: ~90 % decided (exactly one-hot), the rest undecided
    q_R = rng.dirichlet([1, 1], size=(N, U))
    hot = rng.rand(N, U) < 0.9
    one = (rng.rand(N, U) < 0.1).astype(int)
    pk = np.full((N, U, 2), 1e-25)
    pk[np.arange(N)[:, None], np.arange(U)[None, :], one] = 1.0
    q_R[hot] = pk[hot]
    lq_R = np.log(q_R)
    # ---- oracle on the rows (fit.py:157-174 with the rows' region pairs)
    (lpB, p, lM) = O.update_lps(b, bt, th)
    w = O.eval_q_R_w(q_R, n, m)
    lq = np.tile(np.log(th.gamma), (Cl, 1, 1))
    lq[:, 0, :] += np.sum(lpB, axis=1)
    lq[:, 0, :] += np.einsum("cul,cukl->ck", w, lM)
    import scipy.special
    exp_F = lq - scipy.special.logsumexp(lq, axis=2, keepdims=True)
    # ---- product path on the shard
    model = fcdiff.UnsharedRegionModel()
    fit = _fit_for(torch.from_numpy(b).cuda(), torch.from_numpy(bt).cuda(), model)
    fit.shards = _RowWindow(c0, Cl)
    fit.n_edges = C
    fit._init_lps(N, H, U)
    fit._update_lps()
    fit._lq_R = lq_R
    fit._update_lq_F()                                     # tiered K2 (no code pass yet)
    nptest.assert_allclose(fit._lq_F[c0:c0 + Cl], exp_F, rtol=1e-9, atol=1e-9)
    lqF_full = np.full((C, 1, 3), -np.log(3))
    lqF_full[c0:c0 + Cl] = exp_F
    q_F = np.exp(exp_F)
    for x in ([th.eta, th.epsilon], [0.55, 0.11]):
        (f, g0, g1) = O._elm_chunk(p, q_F, q_R, (n, m), x[0], x[1])
        for path in ("tiered", "streams"):
            fit._lq_F = lqF_full
            fit.elm_path = path
            (fv, gv) = fit._objective(np.array(x))
            assert fit._ctx['name'] == ("K3b_elm_streams" if path == "streams" else "K3b_elm_obj_grad")
            nptest.assert_allclose(fv, f, rtol=1e-11)
            nptest.assert_allclose(gv, [g0, g1], rtol=1e-7, atol=1e-9 * abs(f))
    # coded K2: the code plane of the last pass describes this q_R
    fit.elm_path = "streams"
    fit._lq_F = lqF_full
    fit._objective(np.array([th.eta, th.epsilon]))
    assert fit._in.get('code_verR') == fit._mR.version
    fit._update_lq_F()
    nptest.assert_allclose(fit._lq_F[c0:c0 + Cl], exp_F, rtol=1e-9, atol=1e-9)


# ------------------------------------------------------------------ kernel variants behind the C-ABI
def test_safe_variant_outside_log_table_range():
    """epsilon below 2^-19 leaves the log table's range: the host must pick the
    SAFE kernels (log()/division) and still match the oracle."""
    th = O.Theta()
    th.epsilon = 1e-7
    th.eta = 0.2
    (N, H, U) = (9, 6, 10)
    (_, _, _, _, b, bt) = O.sample(O.Theta(), N, H, U, np.random.RandomState(2))
    (N, H, U, lq_F, lq_R) = _oracle_state(b, bt, th, 3)
    (lpB, pBt, lM) = O.update_lps(b, bt, th)
    model = fcdiff.UnsharedRegionModel()
    (model.eta, model.epsilon) = (th.eta, th.epsilon)
    fit = _fit_for(b, bt, model)
    fit._init_lps(N, H, U)
    fit._update_lps()
    fit._lq_R, fit._lq_F = lq_R, lq_F
    nptest.assert_allclose(fit._energy_terms(), O.eval_energy_terms(th, lq_F, lq_R, lpB, lM), rtol=1e-10)
    fit._update_lq_F()
    exp_F = O.update_lq_F(th.gamma, lpB, lM, lq_R)
    nptest.assert_allclose(fit._lq_F, exp_F, rtol=1e-9, atol=1e-10)
    fit._update_lq_R()
    nptest.assert_allclose(fit._lq_R, O.update_lq_R(np.array([1 - th.pi, th.pi]), exp_F, lM, lq_R), rtol=1e-9, atol=1e-10)
    (f, grad) = fit._objective([th.eta, th.epsilon])
    (fo, go) = O.elm_objective_and_grad(pBt, np.exp(exp_F), np.exp(fit._lq_R), [th.eta, th.epsilon])
    nptest.assert_allclose(f, fo, rtol=1e-10)
    nptest.assert_allclose(grad, go, rtol=1e-7)


def test_misaligned_planes_are_rejected_by_the_c_abi():
    """The plane kernels use 128-bit loads: an odd pitch or an 8-byte-aligned
    plane must fail loudly (error code + message), not read garbage."""
    import ctypes
    from fcdiff_b200 import _dev
    lib = _lib.load()
    (N, H, U) = (12, 7, 13)
    C = N * (N - 1) // 2
    (_, _, _, _, b, bt) = O.sample(O.Theta(), N, H, U, np.random.RandomState(4))
    fit = _fit_for(b, bt)
    fit._init_lps(N, H, U)
    fit._update_lps()
    inp = fit._ensure_cache()
    assert inp['pitchU'] == U + 1                      # odd U is padded to an even pitch
    (_, qF) = fit._mF.get_dev()
    (_, qR) = fit._mR.get_dev()
    (fstate, rstate) = (fit._mF.get_state(), fit._mR.get_state())
    th = fit._theta()
    out = _dev.empty((3,))

    def call(P, pitch):
        return lib.fcd_elm_obj_grad(_dev.ptr(P), C * pitch, C, U, pitch, _dev.ptr(qF), _dev.ptr(fstate), _dev.ptr(qR),
                                    _dev.ptr(rstate), rstate.shape[1], N, _dev.ptr(inp['nm']), ctypes.byref(th), 1,
                                    _dev.ptr(out), _dev.ptr(_dev.workspace()), _dev.stream())

    assert call(inp['P'], inp['pitchU']) == 0
    assert call(inp['P'], U) != 0                      # odd pitch
    assert b"aligned" in lib.fcd_last_error()
    assert call(inp['P'].view(-1)[1:], inp['pitchU']) != 0      # 8-byte aligned base
    with pytest.raises(_lib.FcdError):
        _lib.check(call(inp['P'], U), "fcd_elm_obj_grad")


def test_evaluation_reuse_is_invalidated_by_assignments():
    th = O.Theta()
    (_, _, _, _, b, bt) = O.sample(th, 8, 5, 6, np.random.RandomState(7))
    fit = _fit_for(b, bt, eta_shift=0.1)
    fit.max_iters = 2
    fit.run()
    e1 = list(fit.energy)
    lqF1 = fit._lq_F.copy()
    assert fit._find_eval() is not None
    fit._lq_R = fit._lq_R.copy()                 # any assignment bumps the version
    assert fit._find_eval() is None
    fit2 = _fit_for(b, bt, eta_shift=0.1)
    fit2.max_iters = 2
    fit2.reuse_evaluations = False
    fit2.run()
    nptest.assert_allclose(e1, fit2.energy, rtol=1e-13)
    nptest.assert_allclose(lqF1, fit2._lq_F, rtol=1e-10, atol=1e-11)


# ------------------------------------------------------------------ recovery of planted structure (SURVEY 8f item 2)
@pytest.mark.parametrize("lookup", ["symmetric", "reference"])
def test_fit_recovers_planted_template_and_regions(lookup):
    """Data drawn from create_ideal_model() (test_fit.py:11-22) by the device
    sampler in util edge order; the fit started at the truth must recover the
    planted template f on nearly every edge and, with the mathematically
    consistent edge lookup, the planted anomalous regions r."""
    from fcdiff_b200 import _dev
    true_model = ideal_model()
    true_model.rng = np.random.RandomState(11)
    (N, H, U) = (60, 40, 50)
    (r, t, f, ft, b, bt) = true_model.sample(N, H, U)
    fit = _fit_for(b, bt, ideal_model())
    fit.edge_lookup = lookup
    fit.convergence_rule = "magnitude"
    fit.max_iters = 15
    fit.run()
    map_f = np.argmax(fit._lq_F[:, 0, :], axis=1)
    assert np.mean(map_f == np.argmax(f, axis=1)) > 0.995
    if lookup == "symmetric":
        map_r = fit._lq_R[:, :, 1] > fit._lq_R[:, :, 0]
        assert np.mean(map_r == r) > 0.97
        nptest.assert_allclose(fit.model.pi, r.mean(), atol=0.03)
        nptest.assert_allclose(fit.model.gamma, f.mean(axis=0), atol=0.02)
    assert np.all(np.isfinite(fit.energy))
