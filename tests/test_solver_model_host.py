"""
CPU tests of the series model of the (eta, epsilon) objective (csrc/fcd_solver.cuh): the
moments A_k, B_k are formed by NumPy from the oracle's planes, the model and its remainder
bounds are evaluated by the library's host build of the same code the evaluation kernels'
last CTA runs, and the one-evaluation solve is checked against the oracle's polished optimum.
"""
import ctypes

import numpy as np
import numpy.testing as nptest
import pytest

from oracle import iar_oracle as O
from fcdiff_b200 import _lib


def _moment_sums(p3, L, q_F, q_R, eta, eps, K):
    """Sums of csrc/fcd_solver.cuh with K moments per series: {obj, ge, G2, A_2, B_2, konst,
    A_3..A_K, B_3..B_K}, A_k = sum_{l<2} w (s_l g)^k, B_k = sum_{l=2} w g^k."""
    C = q_F.shape[0]
    (n, m) = O.edge_pairs(q_R.shape[0])
    w = O.eval_q_R_w(q_R, n[:C], m[:C])
    epsl = [1 - eps, eps, eta * eps + (1 - eta) * (1 - eps)]
    sl = [-1.0, 1.0, 2 * eta - 1]
    (obj, ge, konst) = (0.0, 0.0, 0.0)
    A = np.zeros(K + 1)
    B = np.zeros(K + 1)
    for k in range(3):
        D = 1.5 * p3[:, :, k] - 0.5
        for l in range(3):
            W = q_F[:, 0, k][:, None] * w[:, :, l]
            y = (1 - epsl[l]) / 2 + (epsl[l] - (1 - epsl[l]) / 2) * p3[:, :, k]
            g = D / y
            obj += np.sum(W * np.log(y))
            ge += sl[l] * np.sum(W * g)
            konst += np.sum(W * L)
            for j in range(1, K + 1):
                if l == 2:
                    B[j] += np.sum(W * g ** j)
                else:
                    A[j] += np.sum(W * (sl[l] * g) ** j)
    return np.concatenate([[obj, ge, B[1], A[2], B[2], konst], A[3:], B[3:]])


def _problem(N, H, U, seed, th=None):
    th = th or O.Theta()
    (_, _, _, _, b, bt) = O.sample(th, N, H, U, np.random.RandomState(seed))
    thf = O.Theta()
    (lq_F, lq_R) = O.init_lps(N, U)
    (lpB, p, lM) = O.update_lps(b, bt, thf)
    lq_F = O.update_lq_F(thf.gamma, lpB, lM, lq_R)
    lq_R = O.update_lq_R(np.array([1 - thf.pi, thf.pi]), lq_F, lM, lq_R)
    S = p.sum(axis=2)
    return p, p / S[:, :, None], np.log(S), np.exp(lq_F), np.exp(lq_R)


def _model(sums, K, x0, z):
    out = (ctypes.c_double * 4)()
    assert _lib.load().fcd_solver_model_host(_lib.d3(list(sums)), K, x0[0], x0[1], _lib.d3(list(z)), out) == 0
    return list(out)


def _solve(p, p3, L, q_F, q_R, x0, K, tol=2e-4, max_evals=60, lo=1e-5):
    lib = _lib.load()
    st = _lib.SolverState()
    assert lib.fcd_solver_init_host(ctypes.byref(st), x0[0], x0[1], _lib.d3([lo, lo]), _lib.d3([1 - lo, 1 - lo]),
                                    tol, max_evals) == 0
    while not st.done:
        s = _moment_sums(p3, L, q_F, q_R, st.x[0], st.x[1], K)
        assert lib.fcd_solver_step_host_moments(ctypes.byref(st), _lib.d3(list(s)), K) == 0
    return st


def test_device_moment_count_is_even_and_served_by_the_host_entry():
    K = int(_lib.load().fcd_solver_moments())
    assert K in (4, 6, 8)


@pytest.mark.parametrize("K", [2, 4, 6, 8])
@pytest.mark.parametrize("x0", [(0.6, 0.4), (0.3, 0.03), (0.7, 0.002), (0.2, 0.995)])
@pytest.mark.parametrize("rho", [0.02, 0.1, 0.25])
def test_series_model_is_within_its_remainder_bound(K, x0, rho):
    (p, p3, L, q_F, q_R) = _problem(10, 12, 14, 2)
    s = _moment_sums(p3, L, q_F, q_R, x0[0], x0[1], K)
    (eta, eps) = x0
    G01 = max(1 / eps, 1 / (1 - eps))
    e2 = eta * eps + (1 - eta) * (1 - eps)
    G2 = max(1 / e2, 1 / (1 - e2))
    for (se, sh) in ((1, 0), (-1, 0), (0, 1), (0, -1), (1, 1), (-1, 1)):
        # a move of relative size rho in eps (and in eps_2 through eta)
        ep = eps + se * 0.999 * rho / G01
        et = (e2 + sh * 0.999 * rho / G2 - (1 - ep)) / (2 * ep - 1)   # eps_2 = (1 - eps) + eta (2 eps - 1)
        z = (et, ep)
        (val, _, vb, r) = _model(s, K, x0, z)
        assert r <= rho * (1 + 1e-9)
        f = O.elm_objective_and_grad(p, q_F, q_R, list(z))[0]
        assert abs(val - f) <= vb * (1 + 1e-9) + 1e-12 * abs(f), (K, x0, rho, z, val, f, vb)


@pytest.mark.parametrize("N,H,U,seed", [(10, 20, 20, 0), (16, 8, 30, 3), (30, 20, 25, 5)])
def test_one_evaluation_solve_lands_on_the_polished_optimum(N, H, U, seed):
    (p, p3, L, q_F, q_R) = _problem(N, H, U, seed)
    f = lambda x: O.elm_objective_and_grad(p, q_F, q_R, x)
    ref = O.minimize_eta_epsilon(f, (0.6, 0.05), polish=True)
    # start a few percent away from the optimum: the model of one evaluation reaches it
    x0 = (ref.x[0] * 1.01, ref.x[1] * 0.99)
    st = _solve(p, p3, L, q_F, q_R, x0, 8)
    assert st.done == 1 and st.nfev == 1, (st.done, st.nfev)
    nptest.assert_allclose([st.x[0], st.x[1]], ref.x, rtol=1e-7)
    nptest.assert_allclose(st.f, ref.fun, rtol=1e-12)


@pytest.mark.parametrize("K", [4, 6, 8])
@pytest.mark.parametrize("x0", [(0.4, 0.03), (0.6, 0.3), (0.02, 0.0004), (0.7, 0.002)])
def test_model_solve_from_far_starts_finds_the_polished_optimum(K, x0):
    (p, p3, L, q_F, q_R) = _problem(16, 8, 30, 3)
    ref = O.minimize_eta_epsilon(lambda x: O.elm_objective_and_grad(p, q_F, q_R, x), x0, polish=True)
    st = _solve(p, p3, L, q_F, q_R, x0, K)
    assert st.done == 1 and st.nfev <= 14, (st.done, st.nfev)
    nptest.assert_allclose([st.x[0], st.x[1]], ref.x, rtol=1e-6)
    nptest.assert_allclose(st.f, ref.fun, rtol=1e-11)


def test_model_solve_stops_on_an_active_bound():
    (p, p3, L, q_F, q_R) = _problem(12, 10, 30, 8, O.Theta(epsilon=1e-9, pi=0.0001))
    ref = O.minimize_eta_epsilon(lambda x: O.elm_objective_and_grad(p, q_F, q_R, x), (0.3, 0.03), polish=True)
    st = _solve(p, p3, L, q_F, q_R, (0.3, 0.03), 6)
    assert st.done == 1
    nptest.assert_allclose([st.x[0], st.x[1]], ref.x, rtol=1e-6, atol=1e-12)
    nptest.assert_allclose(st.f, ref.fun, rtol=1e-10)


def test_trust_region_exit_evaluates_on_the_boundary():
    """The optimum lies 28 % (relative) above the start in epsilon: the first quadratic step stays
    inside the region, the model's iteration leaves it, the next evaluation is made on its
    boundary, and the solve ends on the model of a later evaluation."""
    (p, p3, L, q_F, q_R) = _problem(16, 8, 30, 3)
    ref = O.minimize_eta_epsilon(lambda x: O.elm_objective_and_grad(p, q_F, q_R, x), (0.6, 0.05), polish=True)
    lib = _lib.load()
    x0 = (ref.x[0], ref.x[1] * 0.78)
    st = _lib.SolverState()
    lib.fcd_solver_init_host(ctypes.byref(st), x0[0], x0[1], _lib.d3([1e-5, 1e-5]), _lib.d3([1 - 1e-5, 1 - 1e-5]),
                             2e-4, 60)
    s = _moment_sums(p3, L, q_F, q_R, x0[0], x0[1], 6)
    assert lib.fcd_solver_step_host_moments(ctypes.byref(st), _lib.d3(list(s)), 6) == 0
    assert st.done == 0 and st.nfev == 1
    nptest.assert_allclose(_model(s, 6, x0, (st.x[0], st.x[1]))[3], 0.25, rtol=1e-5)
    st2 = _solve(p, p3, L, q_F, q_R, x0, 6)
    assert st2.done == 1 and 2 <= st2.nfev <= 4, (st2.done, st2.nfev)
    nptest.assert_allclose([st2.x[0], st2.x[1]], ref.x, rtol=1e-7)
    nptest.assert_allclose(st2.f, ref.fun, rtol=1e-12)
