"""GPU: the read-outs of a fitted model (``score_patients`` / ``_score_terms``, ``connection_posteriors``,
``score_controls``; csrc/fcd_patients.cu) at atlas scale, 257 to 1000 regions, against the NumPy oracles
(oracle/patients.py, connections.py, subjects.py, missing.py), against themselves across batch sizes and against
the fit's own K3b / K4 energy terms.

The three row kernels share one cell mapping: the C edge rows are cut into ``pt_row_blocks(C)`` blocks of at
least kPtMinRows rows and at most kPtMaxBlocks blocks, rows = ceil(C / nb); one thread evaluates one (row
block, patient) cell, and with fewer than 32 patients a warp takes 32 / lanesP row blocks side by side (lanesP:
U' rounded up to a power of two).  The N <= 90 tests of test_gpu_patients.py, test_gpu_connections.py and
test_gpu_subjects.py never leave the uncapped partition (rows = 16, one running product per cell, no empty
block).  The cases here reach every branch of that mapping; ``test_cases_reach_every_branch`` (no GPU) restates
the partition from the constants read out of the sources and fails if a retuned constant leaves a branch
unreached:

  capped partition, rows not a multiple of 16     N = 257 (rows 17), 400 (rows 39), 1000 (rows 244)
  empty trailing row blocks                        N = 257 (112 of 2048), N = 400 (1)
  the last of 2048 blocks holding edges            N = 1000 (32 rows)
  running products flushed inside a cell           fitted q_F at N = 400 (one flush), N = 1000 (ten)
  tail group of kCtRows = 8 in a capped partition  every N (17, 39, 244 are not multiples of 8)
  lanesP = 1, 2, 4, 8, 16, 32                      U' = 1, 2, 3, 5, 13, 17 / 33 / 40
  cluster form of the blocked sweep                N = 1000, U' = 2 and 5 (2 U' <= 148 SMs)

Error budget.  The FAST forms take the table logarithm (within 3e-13 absolute per term, fcd_math.cuh) and a
running product of n factors carries n 2^-53 relative, i.e. absolute in its logarithm: 24 x 1.1e-16 = 2.7e-15,
below one table logarithm.  A region's update sums N - 1 edges' weights, so one sweep moves its logit by at most
(N - 1) x 3e-13; the N = 90 tolerance on lq_R (atol 1e-10, about four times 89 x 3e-13) is scaled by
(N - 1) / 89 here: 4.5e-10 at N = 400, 1.1e-9 at N = 1000.  The per-patient sums add C terms each within
3e-13 of a term of magnitude >= ~1 (|log M| and L), so rtol 1e-10 holds with orders of magnitude to spare; the
maps (one division per term, no logarithm) and the control terms (no logarithm, sums of C terms in a fixed
order, against NumPy's pairwise sums) keep the 1e-12 of the small shapes.  The SAFE form (epsilon = 1e-7) is
limited by the plane form a_1 + b_1 p_k (test_gpu_patients.py: 4.5e-7 in lq_R after three sweeps over 89 edges
per region), scaled by (N - 1) / 89 as well.

Each case prints its largest absolute / relative deviations (run with -s).  Measured on an NVIDIA B200 at its
1000 W power limit, over all cases: lq_R 2.4e-11 (N = 1000; checked at 1.1e-9), SAFE form 1.7e-6 (checked at
4.5e-6); per-patient sums and free energies 6.2e-14 relative (1e-10); q_T 2.2e-15 and q_F~ 8.2e-15 absolute
(1e-12); expected counts 2.2e-13 relative (N = 1000; 1e-12); control terms 4.8e-14 relative (1e-12); the
cohort's sums against K3b / K4 4.0e-16 relative (1e-12 / 1e-11).  The file runs in about 45 s there."""
import ctypes
import os
import re

import numpy as np
import numpy.testing as nptest
import pytest
import torch

from oracle import connections as OC
from oracle import iar_oracle as O
from oracle import missing as OM
from oracle import patients as OP
from oracle import subjects as OS

import fcdiff_b200 as fcdiff          # noqa: E402
from fcdiff_b200 import _dev, _lib    # noqa: E402

F = fcdiff.fit
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "fcdiff_b200", "csrc")
B200_SMS = 148

# (N, U', edge lookup, q_F kind): the patient and connection cases
PATIENT_CASES = ([(400, U, "symmetric" if i % 2 == 0 else "reference", "fitted")
                  for (i, U) in enumerate((1, 2, 3, 5, 13, 17, 40))] +
                 [(257, 2, "reference", "fitted"), (257, 33, "symmetric", "fitted"),
                  (1000, 2, "symmetric", "fitted"), (1000, 5, "reference", "fitted"),
                  (400, 3, "symmetric", "random"), (257, 33, "reference", "random"), (1000, 2, "symmetric", "random")])
# (N, S, q_F kind): the control cases
CONTROL_CASES = ([(N, S, "fitted") for N in (257, 400, 1000) for S in (1, 2, 3, 5, 13, 33)] +
                 [(N, 5, "random") for N in (257, 400, 1000)])
MASKED_CONTROL_CASES = [(400, 5), (400, 33)]
BATCH_N = 400
BATCH_SIZES = (2, 3, 5, 13, 17, 40)
EMPTY_BLOCK_N = 257


# ------------------------------------------------------------------ the partition, restated (no GPU)
def _const(fname, name):
    with open(os.path.join(CSRC, fname)) as f:
        m = re.search(r"constexpr\s+\w+\s+%s\s*=\s*(\d+)\s*;" % name, f.read())
    assert m is not None, "%s not found in %s" % (name, fname)
    return int(m.group(1))


def _cluster_min_regions():
    with open(os.path.join(CSRC, "fcd_estep.cu")) as f:
        m = re.search(r"int T = N >= (\d+) \? 512", f.read())
    assert m is not None, "the sweep's launch-shape rule was not found in fcd_estep.cu"
    return int(m.group(1))


def _row_blocks(C, min_rows, max_blocks):
    """pt_row_blocks(C) and rows = ceil(C / nb) of fcd_patients.cu."""
    nb = max(min(-(-C // min_rows), max_blocks), 1)
    return nb, -(-C // nb)


def _lanes(U):
    lanesP = 1
    while lanesP < 32 and lanesP < U:
        lanesP *= 2
    return lanesP


def test_cases_reach_every_branch():
    """The case lists of this file reach every branch of the row partition and lane mapping, with the
    constants as the sources have them (a retuned constant fails here instead of leaving the GPU cases
    vacuous)."""
    (min_rows, max_blocks) = (_const("fcd_patients.cu", "kPtMinRows"), _const("fcd_patients.cu", "kPtMaxBlocks"))
    (prod_max, ct_rows) = (_const("fcd_math.cuh", "kProdMax"), _const("fcd_patients.cu", "kCtRows"))
    assert (min_rows, max_blocks, prod_max, ct_rows) == (16, 2048, 24, 8)     # the values the docstring quotes

    def part(N):
        C = N * (N - 1) // 2
        (nb, rows) = _row_blocks(C, min_rows, max_blocks)
        return dict(C=C, nb=nb, rows=rows, capped=-(-C // min_rows) > max_blocks,
                    empty=sum(1 for rb in range(nb) if rb * rows >= C), last_full=(nb - 1) * rows < C)

    pN = {N for (N, _, _, _) in PATIENT_CASES}
    cN = {N for (N, _, _) in CONTROL_CASES}
    for Ns in (pN, cN):
        # capped partition with rows not a multiple of the minimum
        assert any(part(N)["capped"] and part(N)["rows"] % min_rows != 0 for N in Ns)
        # at least one empty trailing block, and a capped partition whose last block holds edges
        assert any(part(N)["empty"] > 0 for N in Ns)
        assert any(part(N)["capped"] and part(N)["last_full"] for N in Ns)
    assert part(EMPTY_BLOCK_N)["empty"] > 0 and part(EMPTY_BLOCK_N)["capped"]
    # mid-row flushes of the running products: a cell of >= 2 kProdMax rows with a fitted (peaked) q_F
    assert any(part(N)["rows"] >= 2 * prod_max for (N, _, _, kind) in PATIENT_CASES if kind == "fitted")
    assert any(prod_max < part(N)["rows"] < 2 * prod_max for (N, _, _, kind) in PATIENT_CASES if kind == "fitted")
    # tail groups of kCtRows inside a capped partition, plain and masked
    assert any(part(N)["capped"] and part(N)["rows"] % ct_rows != 0 for N in cN)
    assert all(part(N)["capped"] and part(N)["rows"] % ct_rows != 0 for (N, _) in MASKED_CONTROL_CASES)
    # every lane packing, for patients, controls and the batch-invariance sizes
    every = {1, 2, 4, 8, 16, 32}
    assert {_lanes(U) for (_, U, _, _) in PATIENT_CASES} == every
    assert {_lanes(S) for (_, S, _) in CONTROL_CASES} == every
    assert {_lanes(U) for U in BATCH_SIZES + (1,)} == every
    assert part(BATCH_N)["capped"]
    # both edge lookups in a capped partition
    assert {lk for (N, _, lk, _) in PATIENT_CASES if part(N)["capped"]} == {"reference", "symmetric"}
    # the cluster form of the blocked sweep: >= 700 regions and two CTAs per patient within one wave
    nmin = _cluster_min_regions()
    assert any(N >= nmin and 2 * U <= B200_SMS for (N, U, _, _) in PATIENT_CASES)


# ------------------------------------------------------------------ GPU fixtures
@pytest.fixture(scope="module")
def native():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    lib = _lib.load()
    n0 = lib.fcd_launch_count()
    yield lib
    assert lib.fcd_launch_count() > n0, "no kernel of libfcdiff_b200.so was launched"


gpu = pytest.mark.gpu


def _run_fit(b, bt, iters, lookup):
    fit = F.UnsharedRegionFit()
    fit.b, fit.bt = b, bt
    fit.model = fcdiff.UnsharedRegionModel()
    fit.edge_lookup = lookup
    fit.max_iters = iters
    fit.rel_tol = -1.0
    fit.run()
    return fit


def _fit_at(th, lq_F, lookup, missing="reject"):
    """A fit that holds only theta and q_F: enough for the read-outs."""
    fit = F.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    (fit.model.pi, fit.model.eta, fit.model.epsilon) = (th.pi, th.eta, th.epsilon)
    (fit.model.gamma, fit.model.mu, fit.model.sigma) = (th.gamma.copy(), th.mu.copy(), th.sigma.copy())
    fit.edge_lookup = lookup
    fit.missing = missing
    fit._lq_F = lq_F
    return fit


def _theta_of(model):
    return O.Theta(pi=float(model.pi), eta=float(model.eta), gamma=np.array(model.gamma, dtype=np.float64),
                   epsilon=float(model.epsilon), mu=np.array(model.mu, dtype=np.float64),
                   sigma=np.array(model.sigma, dtype=np.float64))


_FITTED = {}


def _fitted_state(N, lookup):
    """theta and a peaked q_F of a 4-iteration fit on training data of N regions (cached per module)."""
    if (N, lookup) not in _FITTED:
        (_, _, _, _, b, bt) = O.sample(O.Theta(), N, 30, 40, np.random.RandomState(N + 5))
        fit = _run_fit(b, bt, 4, lookup)
        peaked = float((fit._mF.get_state()[:N * (N - 1) // 2] < 3).double().mean())
        print("fitted state N=%d %s: %.4f of the edges peaked" % (N, lookup, peaked))
        # the FAST running products only see peaked edges: a fit that leaves q_F undecided tests nothing of them
        assert peaked > 0.5, peaked
        _FITTED[(N, lookup)] = (_theta_of(fit.model), fit._lq_F.copy())
    return _FITTED[(N, lookup)]


def _state(N, lookup, kind):
    if kind == "fitted":
        return _fitted_state(N, lookup)
    rng = np.random.RandomState(3 * N + 1)
    return O.Theta(), np.log(rng.dirichlet([1, 1, 1], size=(N * (N - 1) // 2, 1)))


def _lM_of(th, bt):
    p = np.stack([O.norm_pdf(bt, th.mu[k], th.sigma[k]) for k in range(3)], axis=-1)
    return O.lM_from_p(p, th.eta, th.epsilon)


def _scale(N):
    """The N = 90 tolerances on lq_R scaled by the edges a region's update sums (module docstring)."""
    return max(1.0, (N - 1) / 89.0)


def _dev_of(got, exp):
    """(largest absolute, largest relative) deviation."""
    (got, exp) = (np.asarray(got, dtype=np.float64), np.asarray(exp, dtype=np.float64))
    d = np.abs(got - exp)
    return float(d.max()), float((d / np.maximum(np.abs(exp), 1e-300)).max())


def _report(tag, **pairs):
    print(tag + "  " + "  ".join("%s %.2e/%.2e" % ((k,) + _dev_of(*v)) for (k, v) in pairs.items()))


def _check_patients(th, lq_F, bt, lookup, lq_R0, sweeps, tag, rtol=(1e-9, 1e-10), atol=(1e-10, 1e-9),
                    missing="reject"):
    """_score_terms / score_patients against OP (OM for NaN entries), as test_gpu_patients._check_vs_oracle."""
    fit = _fit_at(th, lq_F, lookup, missing)
    (lq_R, t, k, _) = fit._score_terms(bt, lq_R0, sweeps, -1.0)
    assert k == sweeps
    if missing == "reject":
        (exp_R, _) = OP.score_patients(th, lq_F, bt, lq_R0, lookup, sweeps=sweeps)
        exp_t = OP.patient_terms(th, lq_F, lq_R, _lM_of(th, bt))
    else:
        (exp_R, _) = OM.score_patients_masked(th, lq_F, bt, lq_R0, lookup, sweeps=sweeps)
        exp_t = OP.patient_terms(th, lq_F, lq_R, OM.lM_masked(th, bt))
    s = fit.score_patients(bt, lq_R0, sweeps, -1.0)
    (fe, typ) = OP.free_energies(th, lq_R.shape[0], exp_t)
    qR = np.exp(lq_R)
    print("%s: %.3f of (region, patient) pairs peaked" % (tag, float(np.mean(np.max(qR, axis=2) == 1.0))))
    _report(tag, lq_R=(lq_R, exp_R), terms=(t, exp_t), fe=(s.free_energy, fe), fe_typ=(s.free_energy_typical, typ))
    nptest.assert_allclose(lq_R, exp_R, rtol=rtol[0], atol=atol[0])
    nptest.assert_allclose(t, exp_t, rtol=rtol[1], atol=atol[1])
    nptest.assert_array_equal(s.lq_R, lq_R)
    nptest.assert_allclose(s.free_energy, fe, rtol=rtol[1], atol=atol[1])
    nptest.assert_allclose(s.free_energy_typical, typ, rtol=rtol[1], atol=atol[1])
    return fit, lq_R


def _columns(N, U, seed):
    return O.sample(O.Theta(), N, 2, U, np.random.RandomState(seed))[5]


def _random_lq_R(N, U, seed):
    return np.log(np.random.RandomState(seed).dirichlet([1, 1], size=(N, U)))


# ------------------------------------------------------------------ score_patients against the oracle
@gpu
@pytest.mark.parametrize("N,U,lookup,qF_kind", PATIENT_CASES)
def test_score_patients_parity_with_oracle(native, N, U, lookup, qF_kind):
    """Three sweeps from a random lq_R0, then the four per-patient sums and the free energies.  Fitted q_F:
    peaked edges, running products of 39 (N = 400) or 244 (N = 1000) factors per cell flushed every kProdMax;
    random q_F: every edge unpeaked, nine terms from three planes."""
    (th, lq_F) = _state(N, lookup, qF_kind)
    bt = _columns(N, U, N + U)
    sc = _scale(N)
    _check_patients(th, lq_F, bt, lookup, _random_lq_R(N, U, N * U), 3, "patients N=%d U=%d %s %s"
                    % (N, U, lookup, qF_kind), atol=(1e-10 * sc, 1e-9))


@gpu
def test_score_patients_safe_form(native):
    """epsilon = 1e-7: outside the log table, the SAFE kernel variants (log() per term, no running product)
    at N = 400, U' = 13.  Tolerances of the N = 90 SAFE case scaled by (N - 1) / 89 (module docstring)."""
    (th, lq_F) = _fitted_state(400, "symmetric")
    th = th.copy()
    th.epsilon = 1e-7
    bt = _columns(400, 13, 4001)
    sc = _scale(400)
    _check_patients(th, lq_F, bt, "symmetric", _random_lq_R(400, 13, 4002), 3, "patients SAFE N=400 U=13",
                    rtol=(1e-6 * sc, 1e-8), atol=(1e-6 * sc, 1e-6))


@gpu
def test_score_patients_to_convergence(native):
    """Sweeps until the largest change of q_R is <= 1e-9 (qR_change_kernel on 400 regions and 5 patients),
    against the oracle run for the same number of sweeps; the reported change is the host's
    max |exp(lq_R) - exp(lq_R of the sweep before)| up to the rounding of the two exponentials.  The symmetric
    lookup: its sweep is exact coordinate ascent and converges; the reference lookup's need not (here it still
    changed q_R by 0.58 after 200 sweeps)."""
    (th, lq_F) = _fitted_state(400, "symmetric")
    bt = _columns(400, 5, 4011)
    fit = _fit_at(th, lq_F, "symmetric")
    tol = 1e-9
    s = fit.score_patients(bt, max_sweeps=200, tol=tol)
    assert 1 < s.sweeps < 200 and s.max_change <= tol, (s.sweeps, s.max_change)
    prev = fit.score_patients(bt, max_sweeps=s.sweeps - 1, tol=-1.0)
    change = np.abs(np.exp(s.lq_R) - np.exp(prev.lq_R)).max()
    (exp_R, exp_t) = OP.score_patients(th, lq_F, bt, None, "symmetric", sweeps=s.sweeps)
    print("converged in %d sweeps: change %.3e (host %.3e)" % (s.sweeps, s.max_change, change))
    _report("patients converged N=400 U=5", lq_R=(s.lq_R, exp_R))
    nptest.assert_allclose(s.max_change, change, rtol=0, atol=1e-15)
    nptest.assert_allclose(s.lq_R, exp_R, rtol=1e-9, atol=1e-10 * _scale(400))
    (fe, _) = OP.free_energies(th, 400, exp_t)
    nptest.assert_allclose(s.free_energy, fe, rtol=1e-10, atol=1e-9)


@gpu
def test_masked_score_patients(native):
    """NaN entries marginalised, N = 400, U' = 5, against OM.score_patients_masked: ~10 % missing entries, one
    patient with nothing observed."""
    (th, lq_F) = _fitted_state(400, "symmetric")
    bt = _columns(400, 5, 4021)
    rng = np.random.RandomState(4022)
    bt[rng.rand(*bt.shape) < 0.1] = np.nan
    bt[:, 2] = np.nan
    # atol of the terms: the patient with nothing observed has E_lM = 0 up to the encoding's rounding residue,
    # < 3e-13 per missing element (DESIGN.md section 4) and the same for every element: C x 3e-13 = 2.4e-8
    C = bt.shape[0]
    _check_patients(th, lq_F, bt, "symmetric", _random_lq_R(400, 5, 4023), 3, "patients masked N=400 U=5",
                    atol=(1e-10 * _scale(400), C * 3e-13), missing="marginalize")


# ------------------------------------------------------------------ connection_posteriors against the oracle
def _check_connections(got, exp_T, exp_Ft, tag, atol=1e-12, rtol=1e-12):
    """test_gpu_connections._check: maps absolute, reductions relative (+ 1e-14 for the dropped weights)."""
    _report(tag, q_T=(got.q_T, exp_T), q_Ft=(got.q_F_tilde, exp_Ft),
            expected=(got.expected_anomalous, exp_T.sum(axis=0)), rate=(got.anomalous_rate, exp_T.mean(axis=1)))
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


@gpu
@pytest.mark.parametrize("N,U,lookup,qF_kind", PATIENT_CASES)
def test_connection_posteriors_parity_with_oracle(native, N, U, lookup, qF_kind):
    """At the region posteriors of three sweeps (peaked regions beside undecided ones: one, three and nine
    terms per element), with maps and without."""
    (th, lq_F) = _state(N, lookup, qF_kind)
    bt = _columns(N, U, N + U + 1)
    fit = _fit_at(th, lq_F, lookup)
    lq_R = fit.score_patients(bt, _random_lq_R(N, U, N * U + 1), 3, -1.0).lq_R
    got = fit.connection_posteriors(bt, lq_R)
    (exp_T, exp_Ft) = OC.connection_posteriors(th, lq_F, lq_R, bt)
    _check_connections(got, exp_T, exp_Ft, "connections N=%d U=%d %s %s" % (N, U, lookup, qF_kind))
    _check_maps_off(fit, got, bt, lq_R)


# ------------------------------------------------------------------ score_controls against the oracle
@gpu
@pytest.mark.parametrize("N,S,qF_kind", CONTROL_CASES)
def test_score_controls_parity_with_oracle(native, N, S, qF_kind):
    """Row blocks of 17, 39 and 244 rows: tail groups of 1, 7 and 4 rows of kCtRows = 8."""
    (th, lq_F) = _state(N, "reference", qF_kind)
    x = O.sample(O.Theta(), N, S, 1, np.random.RandomState(N + S + 2))[4]
    got = _fit_at(th, lq_F, "reference").score_controls(x)
    exp = OS.control_loglik(th, lq_F, x)
    _report("controls N=%d S=%d %s" % (N, S, qF_kind), l_C=(got, exp))
    nptest.assert_allclose(got, exp, rtol=1e-12)


def _block_edges(N):
    """(nb, rows) of the partition of N regions."""
    return _row_blocks(N * (N - 1) // 2, 16, 2048)


@gpu
@pytest.mark.parametrize("N,S", MASKED_CONTROL_CASES)
def test_masked_score_controls(native, N, S):
    """~10 % NaN entries, one all-NaN column, and NaNs on the last row of a block and inside the tail group of
    8 rows (rows 32..38 of a 39-row block) of every subject."""
    (th, lq_F) = _fitted_state(N, "symmetric")
    x = O.sample(O.Theta(), N, S, 1, np.random.RandomState(N + S + 3))[4]
    rng = np.random.RandomState(N + S + 4)
    x[rng.rand(*x.shape) < 0.1] = np.nan
    (nb, rows) = _block_edges(N)
    C = x.shape[0]
    blocks = rng.choice(nb - 1, size=(40, S))
    for s in range(S):
        x[np.minimum(blocks[:, s] * rows + rows - 1, C - 1), s] = np.nan                 # last row of a block
        x[np.minimum(blocks[:, s] * rows + rows - 1 - (rows % 8) // 2, C - 1), s] = np.nan  # inside the tail
    x[:, S // 2] = np.nan
    got = _fit_at(th, lq_F, "symmetric", "marginalize").score_controls(x)
    exp = OM.control_loglik_masked(th, lq_F, x)
    _report("controls masked N=%d S=%d" % (N, S), l_C=(got, exp))
    assert got[S // 2] == 0.0
    nptest.assert_allclose(got, exp, rtol=1e-12)


# ------------------------------------------------------------------ batch invariance at N = 400
@gpu
def test_batch_invariance(native):
    """A subject's per-patient terms, q_T / q_F~ and expected count, and its control term, do not depend on how
    many subjects are scored with it, which they are, or where its lane falls: bit for bit, scored alone
    (lanesP = 1) and in calls of 2, 3, 5, 13, 17 and 40 subjects in a scrambled order (lanesP = 2 .. 32)."""
    (th, lq_F) = _fitted_state(BATCH_N, "symmetric")
    U = 40
    bt = _columns(BATCH_N, U, 4031)
    x = O.sample(O.Theta(), BATCH_N, U, 1, np.random.RandomState(4032))[4]
    fit = _fit_at(th, lq_F, "symmetric")
    lq_R = fit.score_patients(bt, _random_lq_R(BATCH_N, U, 4033), 3, -1.0).lq_R     # peaked and undecided
    (_, t_all, _, _) = fit._score_terms(bt, lq_R, 0, 1e-9)
    c_all = fit.connection_posteriors(bt, lq_R)
    l_all = fit.score_controls(x)
    batches = [np.array([u]) for u in (0, 21, 39)] + [(np.arange(k) * 7 + k) % U for k in BATCH_SIZES]
    for cols in batches:
        (_, t, _, _) = fit._score_terms(bt[:, cols], lq_R[:, cols], 0, 1e-9)
        nptest.assert_array_equal(t, t_all[cols])
        c = fit.connection_posteriors(bt[:, cols], lq_R[:, cols])
        nptest.assert_array_equal(c.q_T, c_all.q_T[:, cols])
        nptest.assert_array_equal(c.q_F_tilde, c_all.q_F_tilde[:, cols])
        nptest.assert_array_equal(c.expected_anomalous, c_all.expected_anomalous[cols])
        nptest.assert_array_equal(fit.score_controls(x[:, cols]), l_all[cols])


# ------------------------------------------------------------------ the fitted cohort against K3b / K4
@gpu
def test_cohort_sums_equal_the_fit_energy_terms(native):
    """A 3-iteration fit at N = 400 with H = 60 controls and U = 61 patients (pitchU = 62 on the fit's own
    planes).  The read-outs over the fit's own columns add up to the fit's E_lM (K3b), E_lp_R, E_lq_R and
    E_lp_B_g_F (K4), which are computed by different code; connection_posteriors() of the cohort equals the
    oracle at the fit's state.  The fused E_lM sums C U = 4.9e6 terms each within 3e-13 of a term of magnitude
    ~1: 1.5e-6 against |E_lM| ~ 1e6 at worst, inside rtol 1e-12."""
    (_, _, _, _, b, bt) = O.sample(O.Theta(), 400, 60, 61, np.random.RandomState(4041))
    fit = _run_fit(b, bt, 3, "symmetric")
    e = fit._energy_terms()                # E_lp_F, E_lp_B_g_F, E_lp_R, E_lM, E_lq_F, E_lq_R
    (_, t, sweeps, _) = fit._score_terms(fit.bt, fit._lq_R, 0, 1e-9)
    assert sweeps == 0
    ctrl = fit.score_controls()
    _report("cohort sums N=400", E_lM=(t[:, 0].sum(), e[3]), E_lp_R=(t[:, 1].sum(), e[2]),
            E_lq_R=(t[:, 2].sum(), e[5]), E_lp_B_g_F=(ctrl.sum(), e[1]))
    nptest.assert_allclose(t[:, 0].sum(), e[3], rtol=1e-12)
    nptest.assert_allclose(t[:, 1].sum(), e[2], rtol=1e-12)
    nptest.assert_allclose(t[:, 2].sum(), e[5], rtol=1e-12)
    nptest.assert_allclose(ctrl.sum(), e[1], rtol=1e-11)
    got = fit.connection_posteriors()
    (exp_T, exp_Ft) = OC.connection_posteriors(_theta_of(fit.model), fit._lq_F, fit._lq_R, bt)
    _check_connections(got, exp_T, exp_Ft, "connections cohort N=400 U=61")
    _check_maps_off(fit, got)


# ------------------------------------------------------------------ empty row blocks through the C-ABI
@gpu
def test_empty_row_blocks_write_zero_partials(native):
    """N = 257: 2048 blocks of 17 rows, the last 112 hold no edge.  Their workspace partials must be exactly
    +0.0 in all three row kernels (for fcd_patient_terms, log_pos(1.0) of the two empty running products is
    exactly 0), and every other partial finite; the workspaces start as NaN, so a partial not written shows.
    The launches' results equal the Python read-outs bit for bit."""
    lib = native
    N = EMPTY_BLOCK_N
    C = N * (N - 1) // 2
    (nb, rows) = _block_edges(N)
    empty = np.arange(nb) * rows >= C
    assert nb == 2048 and rows == 17 and int(empty.sum()) == 112
    (th, lq_F) = _fitted_state(N, "reference")
    fit = _fit_at(th, lq_F, "reference")
    U = 3
    bt = _columns(N, U, 2571)
    lq_R = fit.score_patients(bt, _random_lq_R(N, U, 2572), 3, -1.0).lq_R
    th_c = fit._theta(use_snapshot=False)
    pitchU = _dev.even(U)
    PL = fit._planes_of(bt, C, U, pitchU, th_c)
    (_, qF) = fit._mF.get_dev()
    fstate = fit._mF.get_state()
    (lqR, qR) = (_dev.upload(lq_R.reshape(-1)), _dev.upload(np.exp(lq_R).reshape(-1)))

    def nan_ws(nbytes):
        return torch.full((int(nbytes) // 8,), float("nan"), dtype=torch.float64, device=_dev.device())

    def check_parts(part, what):
        assert np.all(part[empty] == 0.0) and not np.any(np.signbit(part[empty])), what
        assert np.all(np.isfinite(part[~empty])), what

    ws = nan_ws(lib.fcd_patient_terms_ws_bytes(C, U))
    out4 = _dev.empty((U, 4))
    _lib.check(lib.fcd_patient_terms(_dev.ptr(PL), C * pitchU, _dev.ptr(PL[3]), C, U, pitchU, _dev.ptr(qF),
                                     _dev.ptr(fstate), _dev.ptr(qR), _dev.ptr(lqR), N, ctypes.byref(th_c),
                                     _dev.ptr(out4), _dev.ptr(ws), _dev.stream()), "fcd_patient_terms")
    check_parts(ws.cpu().numpy().reshape(nb, U, 2), "fcd_patient_terms")
    nptest.assert_array_equal(out4.cpu().numpy(), fit._score_terms(bt, lq_R, 0, 1e-9)[1])

    ref = fit.connection_posteriors(bt, lq_R)
    for maps in (True, False):
        ws = nan_ws(lib.fcd_connection_ws_bytes(C, U))
        (qT, qFt) = (_dev.empty((C, U)), _dev.empty((C, U, 3)) if maps else None)
        (expected, rate) = (_dev.empty((U,)), _dev.empty((C,)))
        _lib.check(lib.fcd_connection_posteriors(_dev.ptr(PL), C * pitchU, C, U, pitchU, _dev.ptr(qF),
                                                 _dev.ptr(fstate), _dev.ptr(qR), N, ctypes.byref(th_c), _dev.ptr(qT),
                                                 _dev.ptr(qFt), _dev.ptr(expected), _dev.ptr(rate), _dev.ptr(ws),
                                                 _dev.stream()), "fcd_connection_posteriors")
        check_parts(ws.cpu().numpy().reshape(nb, U), "fcd_connection_posteriors maps=%s" % maps)
        nptest.assert_array_equal(expected.cpu().numpy(), ref.expected_anomalous)
        nptest.assert_array_equal(rate.cpu().numpy(), ref.anomalous_rate)

    S = 5
    x = O.sample(O.Theta(), N, S, 1, np.random.RandomState(2573))[4]
    pitchS = _dev.even(S)
    X = fit._columns_on_device(x, C, S, pitchS)
    for missing in (0, 1):
        name = "fcd_control_terms missing=%d" % missing
        ws = nan_ws(lib.fcd_control_terms_ws_bytes(C, S))
        out = _dev.empty((S,))
        _lib.check(lib.fcd_control_terms(_dev.ptr(X), C, S, pitchS, _dev.ptr(qF), ctypes.byref(th_c), _dev.ptr(out),
                                         _dev.ptr(ws), missing, _dev.stream()), name)
        check_parts(ws.cpu().numpy().reshape(nb, S), name)
        nptest.assert_array_equal(out.cpu().numpy(), fit.score_controls(x))
