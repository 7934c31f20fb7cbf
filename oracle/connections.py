"""
TEST INFRASTRUCTURE ONLY -- NumPy restatement of the posteriors of the anomalous
connections T and the patients' connection states F~
(``UnsharedRegionFit.connection_posteriors``), built from the step functions of
``iar_oracle``, which are not edited.

The generative model (``iar_oracle.sample``, fcdiff/model.py:141-188): t = 0 if
both regions of the edge are typical, t = 1 if both are anomalous, t ~
Bernoulli(eta) for a mixed pair; F~ keeps the template state F = k with
probability 1 - epsilon if t = 0 and epsilon if t = 1, the two other states
share the rest equally; b~ ~ N(mu_F~, sigma_F~).  Given (F = k, pair state l,
b~), with the plane values p_j = N_j / sum N and eps_l of fit.py:433-444,
a_l = (1 - eps_l) / 2, b_l = eps_l - a_l:

    P(F~ = j | k, l, b~) = eps_l p_k / (a_l + b_l p_k)     (j = k)
                         = a_l p_j / (a_l + b_l p_k)       (j != k)
    P(T = 1  | k, l, b~) = 0 (l = 0), 1 (l = 1),
                           eta (eps p_k + (1 - eps)(1 - p_k) / 2) / (a_2 + b_2 p_k)   (l = 2)

The read-outs are their expectations under q_F[c,k] and the pair weights w_l
of the edge's own regions (fit.py:382-406).
"""
import numpy as np
import scipy.stats

from . import iar_oracle as O


def connection_posteriors(th, lq_F, lq_R, bt):
    """(q_T (C, U), q_F_tilde (C, U, 3)) for the patients of ``bt`` (C, U) with log-posteriors lq_F (C, 1, 3)
    and lq_R (N, U, 2)."""
    q_F = np.exp(lq_F)[:, 0, :]
    q_R = np.exp(lq_R)
    C = q_F.shape[0]
    (n, m) = O.edge_pairs(q_R.shape[0])
    w = O.eval_q_R_w(q_R, n[:C], m[:C])                                          # (C, U, 3)
    dens = np.stack([O.norm_pdf(bt, th.mu[k], th.sigma[k]) for k in range(3)], axis=-1)
    p = dens / dens.sum(axis=-1, keepdims=True)                                  # (C, U, 3)
    q_T = np.zeros(bt.shape)
    q_Ft = np.zeros(bt.shape + (3,))
    eps = th.epsilon
    for l in range(3):
        e = O.eval_M_eps(th.eta, th.epsilon, l)
        (a, b) = ((1 - e) / 2, e - (1 - e) / 2)
        for k in range(3):
            wt = q_F[:, None, k] * w[:, :, l]
            pk = p[:, :, k]
            den = a + b * pk
            post = a * p / den[:, :, None]
            post[:, :, k] = e * pk / den
            q_Ft += wt[:, :, None] * post
            if l == 1:
                q_T += wt
            elif l == 2:
                q_T += wt * (th.eta * (eps * pk + (1 - eps) * (1 - pk) / 2) / den)
    return q_T, q_Ft


def exact_conditionals(th, x, k, l):
    """Brute-force enumeration over (t, f~) of P(T = 1 | F = k, l, b~ = x) and P(F~ = . | k, l, x) (shape
    x.shape + (3,)) with scipy.stats.norm.pdf: the generative model without the plane form."""
    x = np.asarray(x, dtype=np.float64)
    p_t = {0: [1.0, 0.0], 1: [0.0, 1.0], 2: [1.0 - th.eta, th.eta]}[l]
    joint = np.zeros(x.shape + (2, 3))
    for t in range(2):
        keep = th.epsilon if t else 1.0 - th.epsilon
        for j in range(3):
            p_j = keep if j == k else (1.0 - keep) / 2
            joint[..., t, j] = p_t[t] * p_j * scipy.stats.norm.pdf(x, th.mu[j], th.sigma[j])
    joint /= joint.sum(axis=(-2, -1), keepdims=True)
    return joint[..., 1, :].sum(axis=-1), joint.sum(axis=-2)
