"""
TEST INFRASTRUCTURE ONLY -- NumPy restatement of the two-group read-outs of a
fitted model (``UnsharedRegionFit.score_controls`` / ``classify_subjects``),
built from ``iar_oracle`` and ``oracle.patients``, which stay as pinned.

With theta and q_F fixed, a new column x has
  as a control  l_C(x) = sum_c sum_k q_F[c,k] log N(x_c; mu_k, sigma_k), one
                control's share of E_lp_B_g_F (fcdiff/fit.py:461-472);
  as a patient  l_P(x) = -free_energy, the patient's share of the evidence bound
                (``patients.patient_terms``);
and log_odds = l_P - l_C + log(rho / (1 - rho)).

For small N the exact quantities are enumerated over all 2^N region
configurations R (l_c(R): 0 both regions of edge c typical, 1 both anomalous,
2 mixed; eps_0 = 1 - epsilon, so a patient without anomalous regions is not a
control):
  p(x | patient) = sum_R p(R) prod_c sum_k q_F[c,k] M_{k,l_c(R)}(x_c)
  p(x | control) = prod_c sum_k q_F[c,k] N(x_c; mu_k, sigma_k)
which are the exact likelihoods when q_F is one-hot (the template F known).
"""
import itertools

import numpy as np
import scipy.special

from . import iar_oracle as O
from . import patients as OP


def _lp(th, x):
    """(C, S, 3) log N(x; mu_k, sigma_k) (fit.py:111-114)."""
    return np.stack([O.norm_logpdf(x, th.mu[k], th.sigma[k]) for k in range(3)], axis=-1)


def _lM(th, x):
    p = np.stack([O.norm_pdf(x, th.mu[k], th.sigma[k]) for k in range(3)], axis=-1)    # fit.py:115
    return O.lM_from_p(p, th.eta, th.epsilon)


def control_loglik(th, lq_F, x):
    """(S,) l_C of the columns of x (C, S)."""
    return np.einsum("ck,csk->s", np.exp(lq_F)[:, 0, :], _lp(th, x))


def classify(th, lq_F, x, prior, lq_R):
    """(log_odds, control_loglik, patient_elbo) of the columns of x at the region posteriors lq_R (N, S, 2)."""
    N = lq_R.shape[0]
    (fe, _) = OP.free_energies(th, N, OP.patient_terms(th, lq_F, lq_R, _lM(th, x)))
    elbo = -fe
    control = control_loglik(th, lq_F, x)
    return (elbo - control) + np.log(prior / (1.0 - prior)), control, elbo


def _configs(N):
    """(2^N, N) 0/1 region configurations and (2^N, C) pair states l_c(R) in edge order."""
    if N > 8:
        raise ValueError("exact enumeration is for N <= 8 (got %d)" % N)
    R = np.array(list(itertools.product((0, 1), repeat=N)), dtype=np.int64)
    (n, m) = O.edge_pairs(N)
    L = np.where(R[:, n] == R[:, m], R[:, n], 2)
    return R, L


def _log_joint(th, lq_F, x):
    """(2^N, S) log p(R) + log prod_c sum_k q_F[c,k] M_{k,l_c(R)}(x_c), and the configurations R."""
    C = x.shape[0]
    N = int(O.C_to_N(C))
    (R, L) = _configs(N)
    G = scipy.special.logsumexp(_lM(th, x) + lq_F[:, 0, :][:, None, :, None], axis=2)      # (C, S, 3)
    lpR = np.where(R == 1, np.log(th.pi), np.log(1.0 - th.pi)).sum(axis=1)
    cs = np.arange(C)
    out = np.stack([lpR[r] + G[cs, :, L[r]].sum(axis=0) for r in range(R.shape[0])])
    return out, R


def exact_log_evidence_patient(th, lq_F, x):
    """(S,) log sum_R p(R) prod_c sum_k q_F[c,k] M_{k,l_c(R)}(x_c)."""
    return scipy.special.logsumexp(_log_joint(th, lq_F, x)[0], axis=0)


def exact_log_evidence_control(th, lq_F, x):
    """(S,) sum_c log sum_k q_F[c,k] N(x_c; mu_k, sigma_k)."""
    return scipy.special.logsumexp(_lp(th, x) + lq_F[:, 0, :][:, None, :], axis=2).sum(axis=0)


def exact_posterior_R(th, lq_F, x):
    """(R (2^N, N), log p(R | x) (2^N, S)) under the patient model."""
    (lj, R) = _log_joint(th, lq_F, x)
    return R, lj - scipy.special.logsumexp(lj, axis=0)


def kl_qR(lq_R, th, lq_F, x):
    """(S,) KL(q_R || p(R | x)) of the mean-field q_R(R) = prod_n q_R[n, s, R_n], lq_R (N, S, 2)."""
    (R, lpost) = exact_posterior_R(th, lq_F, x)
    N = lq_R.shape[0]
    lq = np.stack([lq_R[np.arange(N), :, R[r]].sum(axis=0) for r in range(R.shape[0])])       # (2^N, S)
    return np.sum(np.exp(lq) * (lq - lpost), axis=0)
