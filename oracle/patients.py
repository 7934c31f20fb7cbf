"""
TEST INFRASTRUCTURE ONLY -- NumPy restatement of held-out patient scoring
(``UnsharedRegionFit.score_patients``), built from the step functions of
``iar_oracle`` and kept beside them so that they stay as pinned.

With theta and q_F fixed, the free energy of fcdiff/fit.py:142-155 is a sum
over patient columns u: E_lp_R, E_lM and E_lq_R (fit.py:475-539) are sums over
u, and E_lp_F, E_lp_B_g_F, E_lq_F do not involve the patients.  The region
weights W = sum_k q_F log M_kl do not involve q_R (fit.py:187-194), so they are
formed once and the reference's region sweep (fit.py:176-198) is repeated on
the held-out columns.
"""
import numpy as np

from . import iar_oracle as O


def patient_terms(th, lq_F, lq_R, lM):
    """(U, 4): per patient u, E_lM,u (fit.py:489-511, pair weights of the edge's own regions), E_lp_R,u
    (fit.py:475-486), E_lq_R,u (fit.py:528-539) and sum_c sum_k q_F[c,k] log M_k0(c,u) (E_lM,u with every
    region typical)."""
    q_F = np.exp(lq_F)
    q_R = np.exp(lq_R)
    C = q_F.shape[0]
    (n, m) = O.edge_pairs(q_R.shape[0])
    w = O.eval_q_R_w(q_R, n[:C], m[:C])                                          # (C, U, 3)
    pi2 = np.array([1.0 - th.pi, th.pi])
    return np.stack([
        np.einsum("ck,cul,cukl->u", q_F[:, 0, :], w, lM),
        np.einsum("nus,s->u", q_R, np.log(pi2)),
        np.sum(q_R * lq_R, axis=(0, 2)),
        np.einsum("ck,cuk->u", q_F[:, 0, :], lM[:, :, :, 0])], axis=1)


def free_energies(th, N, terms):
    """(free_energy, free_energy_typical) per patient from ``patient_terms``: the patient's share of
    fit.py:148-155, and the same share with every region typical."""
    fe = -terms[:, 1]
    fe = fe - terms[:, 0]
    fe = fe + terms[:, 2]
    return fe, -N * np.log(1.0 - th.pi) - terms[:, 3]


def score_patients(th, lq_F, bt_new, lq_R0=None, edge_lookup="reference", sweeps=1):
    """``sweeps`` region sweeps of the columns of ``bt_new`` (C, U') from ``lq_R0`` (None: uniform, fit.py:97)
    with theta and q_F fixed.  Returns (lq_R, patient_terms at lq_R)."""
    C = bt_new.shape[0]
    N = int(O.C_to_N(C))
    p = np.stack([O.norm_pdf(bt_new, th.mu[k], th.sigma[k]) for k in range(3)], axis=-1)    # fit.py:115
    lM = O.lM_from_p(p, th.eta, th.epsilon)
    W = O.eval_W(np.exp(lq_F), lM)
    lq_R = np.full((N, bt_new.shape[1], 2), -np.log(2)) if lq_R0 is None else np.array(lq_R0, dtype=np.float64)
    pi2 = np.array([1.0 - th.pi, th.pi])
    for _ in range(sweeps):
        lq_R = O.update_lq_R(pi2, lq_F, lM, lq_R, edge_lookup, W=W)
    return lq_R, patient_terms(th, lq_F, lq_R, lM)
