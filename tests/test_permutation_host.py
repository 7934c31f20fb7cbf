"""CPU: the max-T oracle (oracle/permutation.py) against the literal step-down, a hand-worked example, the
properties of the p-values, the planted sampler, and the argument checks of ``sweep.maxt_pvalues`` and
``sweep.permutation_inference``, which raise before the library is loaded."""
import numpy as np
import pytest

from oracle import iar_oracle as O
from oracle import permutation as OP


def _cases():
    rng = np.random.RandomState(11)
    out = []
    for _ in range(40):
        (R1, K) = (rng.randint(1, 12), rng.randint(1, 12))
        out.append(rng.randn(R1, K))
        out.append(rng.choice([-0.0, 0.0, 0.25, 0.5, 1.0], (R1, K)))
    out += [np.full((5, 4), 0.5), np.full((1, 6), -0.0), rng.randn(1, 7), rng.randn(9, 1),
            np.array([[0.0, -0.0, 0.0], [-0.0, 0.0, -0.0]])]
    return out


def test_vectorised_equals_literal():
    for T in _cases():
        (p, pf) = OP.maxt_pvalues(T)
        (pl, pfl) = OP.maxt_pvalues_literal(T)
        np.testing.assert_array_equal(p, pl)
        np.testing.assert_array_equal(pf, pfl)
        K = T.shape[1]
        if K >= 3:
            fams = [(0, 1), (1, K - 1)]             # the last column outside every family
            (p, pf) = OP.maxt_pvalues(T, fams)
            (pl, pfl) = OP.maxt_pvalues_literal(T, fams)
            np.testing.assert_array_equal(p, pl)
            np.testing.assert_array_equal(pf, pfl)
            assert np.isnan(p[-1]) and np.isnan(pf[-1])


def test_hand_worked_example():
    T = np.array([[0.5, 0.9, 0.2],
                  [0.1, 0.1, 0.7],
                  [0.6, 0.3, 0.1],
                  [0.2, 0.4, 0.0]])
    # uncorrected: column 0 is reached by rows 0 and 2, column 1 by row 0, column 2 by rows 0 and 1.
    # step-down, descending observed value (1, 0, 2): successive maxima over {2}: (.2, .7, .1, 0) -> 2 rows
    # reach .2; over {2, 0}: (.5, .7, .6, .2) -> 3 rows reach .5; over {2, 0, 1}: (.9, .7, .6, .4) -> 1 row
    # reaches .9; then monotone in descending order: .25, max(.25, .75), max(.75, .5).
    (p, pf) = OP.maxt_pvalues(T)
    np.testing.assert_array_equal(p, [0.5, 0.25, 0.5])
    np.testing.assert_array_equal(pf, [0.75, 0.25, 0.75])
    np.testing.assert_array_equal(OP.maxt_pvalues_literal(T)[1], pf)


def test_properties():
    for T in _cases():
        (R1, K) = T.shape
        (p, pf) = OP.maxt_pvalues(T)
        assert (p >= 1.0 / R1).all() and (p <= 1.0).all()
        assert (pf >= p).all()
        obs = T[0]
        for i in range(K):
            for j in range(K):
                if obs[i] == obs[j]:
                    assert pf[i] == pf[j]                   # ties: equal p_fwer
                elif obs[i] < obs[j]:
                    assert pf[i] >= pf[j]                   # non-increasing in the observed value


def test_single_row_gives_ones():
    (p, pf) = OP.maxt_pvalues(np.random.RandomState(0).randn(1, 5))
    np.testing.assert_array_equal(p, np.ones(5))
    np.testing.assert_array_equal(pf, np.ones(5))


def test_sample_planted_constant_pi_is_sample():
    th = O.Theta(pi=0.2)
    for (N, H, U, seed) in ((12, 9, 11, 0), (30, 40, 40, 5)):
        a = O.sample(th, N, H, U, np.random.RandomState(seed))
        b = OP.sample_planted(th, N, H, U, np.full(N, th.pi), np.random.RandomState(seed))
        for (x, y) in zip(a, b):
            assert x.dtype == y.dtype
            np.testing.assert_array_equal(x, y)


def test_sample_planted_plants():
    th = O.Theta()
    pi = np.full(30, 0.01)
    pi[[3, 17]] = 0.6
    r = OP.sample_planted(th, 30, 40, 400, pi, np.random.RandomState(1))[0]
    rate = r.mean(axis=1)
    assert rate[3] > 0.5 and rate[17] > 0.5
    assert np.delete(rate, [3, 17]).max() < 0.05


@pytest.fixture
def no_library(monkeypatch):
    """Any library load or device query fails loudly: the checks must come first."""
    from fcdiff_b200 import _dev, _lib

    def refuse(*a, **k):
        raise AssertionError("device work before the argument checks")
    monkeypatch.setattr(_lib, "load", refuse)
    monkeypatch.setattr(_dev, "device", refuse)


@pytest.mark.parametrize("stats,families,match", [
    (np.zeros((0, 3)), None, "at least one row"),
    (np.zeros((3, 0)), None, "at least one row"),
    (np.zeros(3), None, r"\(R1, K\)"),
    (np.array([[0.0, 1.0, np.nan], [0.0, np.nan, 1.0]]), None, "column 1"),
    (np.array([[0.0, np.inf, 0.0]]), None, "column 1"),
    (np.array([[0.0, 0.0, -np.inf]]), None, "column 2"),
    (np.zeros((2, 5)), [(0, 3), (2, 5)], "overlap"),
    (np.zeros((2, 5)), [(0, 6)], "range"),
    (np.zeros((2, 5)), [(-1, 2)], "range"),
    (np.zeros((2, 5)), [(3, 3)], "range"),
    (np.zeros((2, 5)), [], "no range"),
])
def test_maxt_pvalues_argument_errors(no_library, stats, families, match):
    from fcdiff_b200 import sweep
    with pytest.raises(ValueError, match=match):
        sweep.maxt_pvalues(stats, families)


def _inputs(N=6, S=10):
    C = N * (N - 1) // 2
    labels = np.zeros(S, dtype=bool)
    labels[S // 2:] = True
    return np.zeros((C, S)), labels


@pytest.mark.parametrize("change,match", [
    (dict(n_permutations=-1), "n_permutations"),
    (dict(labels=np.ones(10, dtype=bool)), "one control and one patient"),
    (dict(labels=np.zeros(10, dtype=bool)), "one control and one patient"),
    (dict(labels=np.arange(9) % 2 == 0), r"corr must be \(C, S\)"),
    (dict(corr=np.zeros((14, 10))), "triangular"),
    (dict(corr=np.zeros(10)), r"corr must be \(C, S\)"),
    (dict(rank=2, world=2), "rank 2 of world 2"),
    (dict(rank=0, world=0), "world 0"),
    (dict(rank=0, world=2), "process group"),
])
def test_permutation_inference_argument_errors(no_library, change, match):
    from fcdiff_b200 import sweep
    (corr, labels) = _inputs()
    kw = dict(corr=corr, labels=labels, n_permutations=3)
    kw.update(change)
    if "process group" in match:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            pytest.skip("a process group is active in this process")
    with pytest.raises(ValueError, match=match):
        sweep.permutation_inference(**kw)
