"""
TEST INFRASTRUCTURE ONLY -- NumPy restatement of the fit and its read-outs with
missing entries marginalised (``UnsharedRegionFit.missing = "marginalize"``),
built from the step functions of ``iar_oracle``, ``patients``, ``subjects`` and
``connections``, which are not edited.

A NaN correlation is an entry that was not observed.  Integrating it out of the
model gives it a density factor of 1 in every term:

* a patient entry: ``p_Bt_g_Ft[c,u,:] = (1, 1, 1)``, so that M_kl = eps_l +
  (1 - eps_l) = 1 for every (k, l) (fcdiff/fit.py:427-430) and lM = 0;
* a control entry: ``lp_B_g_F[c,h,:] = 0``.

The unmodified E-step, region sweep, (eta, epsilon) objective and energy terms
then run on these caches.  (The GPU stores a missing patient entry as the
planes p_k = 1/3, L = log 3: the same M_kl divided by sum_j N_j = 3.)
"""
import numpy as np

from . import connections as OC
from . import iar_oracle as O
from . import patients as OP
from . import subjects as OS


def update_lps_masked(b, bt, th):
    """``iar_oracle.update_lps`` (fcdiff/fit.py:104-122) with NaN entries of b / bt marginalised."""
    (mb, mbt) = (np.isnan(b), np.isnan(bt))
    (lp_B_g_F, p_Bt_g_Ft, _) = O.update_lps(np.where(mb, 0.0, b), np.where(mbt, 0.0, bt), th)
    lp_B_g_F[mb] = 0.0
    p_Bt_g_Ft[mbt] = 1.0
    return lp_B_g_F, p_Bt_g_Ft, O.lM_from_p(p_Bt_g_Ft, th.eta, th.epsilon)


def run_masked(b, bt, th, max_iters=10, rel_tol=1e-5, edge_lookup="reference", optimise=True, polish=False):
    """``iar_oracle.run`` (fcdiff/fit.py:56-82) on the caches of ``update_lps_masked``.  ``th`` is mutated like
    ``fit.model``.  Returns dict(lq_F, lq_R, energy)."""
    (C, _) = b.shape
    U = bt.shape[1]
    N = int(O.C_to_N(C))
    (lq_F, lq_R) = O.init_lps(N, U)
    (lp_B_g_F, p_Bt_g_Ft, lM) = update_lps_masked(b, bt, th)
    energy = [O.energy_from_terms(O.eval_energy_terms(th, lq_F, lq_R, lp_B_g_F, lM))]
    for i in range(1, max_iters + 1):
        (lq_F, lq_R, lM, e, _) = O.em_iteration(b, bt, th, lq_F, lq_R, lp_B_g_F, p_Bt_g_Ft, lM, edge_lookup, optimise,
                                                polish=polish)
        energy.append(e)
        if O.is_converged(energy, i, rel_tol):
            break
    return dict(lq_F=lq_F, lq_R=lq_R, energy=energy)


def lM_masked(th, x):
    """(C, S, 3, 3) log M of the columns of x with NaN entries marginalised (lM = 0)."""
    return update_lps_masked(np.zeros((x.shape[0], 1)), x, th)[2]


def score_patients_masked(th, lq_F, bt_new, lq_R0=None, edge_lookup="reference", sweeps=1):
    """``patients.score_patients`` with NaN entries of bt_new marginalised: (lq_R, patient_terms at lq_R)."""
    N = int(O.C_to_N(bt_new.shape[0]))
    lM = lM_masked(th, bt_new)
    W = O.eval_W(np.exp(lq_F), lM)
    lq_R = np.full((N, bt_new.shape[1], 2), -np.log(2)) if lq_R0 is None else np.array(lq_R0, dtype=np.float64)
    pi2 = np.array([1.0 - th.pi, th.pi])
    for _ in range(sweeps):
        lq_R = O.update_lq_R(pi2, lq_F, lM, lq_R, edge_lookup, W=W)
    return lq_R, OP.patient_terms(th, lq_F, lq_R, lM)


def control_loglik_masked(th, lq_F, x):
    """(S,) ``subjects.control_loglik`` over the observed entries of x."""
    miss = np.isnan(x)
    lp = OS._lp(th, np.where(miss, 0.0, x))
    lp[miss] = 0.0
    return np.einsum("ck,csk->s", np.exp(lq_F)[:, 0, :], lp)


def classify_masked(th, lq_F, x, prior, lq_R):
    """``subjects.classify`` with NaN entries of x marginalised: (log_odds, control_loglik, patient_elbo)."""
    N = lq_R.shape[0]
    (fe, _) = OP.free_energies(th, N, OP.patient_terms(th, lq_F, lq_R, lM_masked(th, x)))
    elbo = -fe
    control = control_loglik_masked(th, lq_F, x)
    return (elbo - control) + np.log(prior / (1.0 - prior)), control, elbo


def connection_posteriors_masked(th, lq_F, lq_R, bt):
    """``connections.connection_posteriors`` with NaN entries of bt marginalised.  A missing element keeps its
    prior: q_T = w_1 + eta w_2 and q_F~[j] = sum_k q_F[c,k] sum_l w_l (eps_l if j == k else (1 - eps_l) / 2)."""
    miss = np.isnan(bt)
    (q_T, q_Ft) = OC.connection_posteriors(th, lq_F, lq_R, np.where(miss, 0.0, bt))
    q_F = np.exp(lq_F)[:, 0, :]
    q_R = np.exp(lq_R)
    C = q_F.shape[0]
    (n, m) = O.edge_pairs(q_R.shape[0])
    w = O.eval_q_R_w(q_R, n[:C], m[:C])                                          # (C, U, 3)
    prior_T = w[:, :, 1] + th.eta * w[:, :, 2]
    prior_Ft = np.zeros(bt.shape + (3,))
    for l in range(3):
        e = O.eval_M_eps(th.eta, th.epsilon, l)
        for k in range(3):
            keep = np.full(3, (1 - e) / 2)
            keep[k] = e
            prior_Ft += (q_F[:, None, k] * w[:, :, l])[:, :, None] * keep
    q_T[miss] = prior_T[miss]
    q_Ft[miss] = prior_Ft[miss]
    return q_T, q_Ft


def corr_fisherz_masked(ts, fisher=True):
    """``iar_oracle.corr_fisherz`` with the regions of a subject that have a non-finite sample or zero variance
    marked as not observed: NaN on all their edges of that subject."""
    (S, N, _) = ts.shape
    x = np.asarray(ts, dtype=np.float32).astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        d = x - x.mean(axis=2, keepdims=True)
        bad = ~(np.sum(d * d, axis=2) > 0)                                       # (S, N); NaN compares False
        out = O.corr_fisherz(np.where(np.isfinite(x), x, 0.0), fisher)
    (n, m) = O.edge_pairs(N)
    for s in range(S):
        out[bad[s, n] | bad[s, m], s] = np.nan
    return out
