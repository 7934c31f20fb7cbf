"""GPU test of the series-model moments the evaluation kernels accumulate (csrc/fcd_solver.cuh):
a device-resident (eta, epsilon) solve, with the tiered evaluator (small problems) and with the
coded-plane evaluator, against the host build of the same solver driven with the moments
A_k, B_k restated in fp64 NumPy on the fit's own planes."""
import ctypes

import numpy as np
import numpy.testing as nptest
import pytest
import torch

from oracle import iar_oracle as O

pytestmark = pytest.mark.gpu

import fcdiff_b200 as fcdiff          # noqa: E402
from fcdiff_b200 import _lib          # noqa: E402
from test_solver_model_host import _moment_sums  # noqa: E402


@pytest.mark.parametrize("N,H,U,seed", [(24, 9, 33, 1), (90, 50, 50, 2), (160, 40, 60, 3)])
def test_device_solve_matches_the_host_model_solve(N, H, U, seed):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    lib = _lib.load()
    K = int(lib.fcd_solver_moments())
    (_, _, _, _, b, bt) = O.sample(O.Theta(), N, H, U, np.random.RandomState(seed))
    fit = fcdiff.fit.UnsharedRegionFit()
    fit.b, fit.bt = b, bt
    fit.model = fcdiff.UnsharedRegionModel()
    fit.model.eta += 0.1
    fit.theta_solver = "newton"
    fit._init_lps(N, H, U)
    fit._update_lps()
    fit._update_lq_F()
    fit._update_lq_R()
    x0 = (float(fit.model.eta), float(fit.model.epsilon))
    p = np.array(fit._p_Bt_g_Ft)
    (q_F, q_R) = (np.exp(fit._lq_F), np.exp(fit._lq_R))
    fit._update_theta()
    (done, nfev) = fit.solver_status[-1]
    assert done == 1

    S = p.sum(axis=2)
    (p3, L) = (p / S[:, :, None], np.log(S))
    st = _lib.SolverState()
    lo = 1e-5                                          # the reference's box (fit._update_theta_sub)
    assert lib.fcd_solver_init_host(ctypes.byref(st), x0[0], x0[1], _lib.d3([lo, lo]), _lib.d3([1 - lo, 1 - lo]),
                                    float(fit.solver_tol), 60) == 0
    while not st.done:
        s = _moment_sums(p3, L, q_F, q_R, st.x[0], st.x[1], K)
        assert lib.fcd_solver_step_host_moments(ctypes.byref(st), _lib.d3(list(s)), K) == 0
    assert st.done == 1
    # the same evaluations (the device sums differ from NumPy's in summation order only)
    assert abs(nfev - st.nfev) <= 1, (nfev, st.nfev)
    nptest.assert_allclose([fit.model.eta, fit.model.epsilon], [st.x[0], st.x[1]], rtol=1e-7)
    ref = O.minimize_eta_epsilon(lambda x: O.elm_objective_and_grad(p, q_F, q_R, x), x0, polish=True)
    nptest.assert_allclose([fit.model.eta, fit.model.epsilon], ref.x, rtol=1e-7)
