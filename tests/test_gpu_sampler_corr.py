"""GPU: the Philox sampler (K5) matched in distribution against the model
(moment and Kolmogorov-Smirnov tests, after test_fcdiff/test_model.py:15-245)
and the correlation stage (K1) against numpy.corrcoef + arctanh."""
import numpy as np
import numpy.testing as nptest
import pytest
import scipy.stats
import torch

from oracle import iar_oracle as O

pytestmark = pytest.mark.gpu

import fcdiff_b200 as fcdiff          # noqa: E402
from fcdiff_b200 import corr, _dev    # noqa: E402


def test_str():
    assert type(fcdiff.UnsharedRegionModel().__str__()) == str


def test_sample_shapes_dtypes():
    model = fcdiff.UnsharedRegionModel()
    (N, H, U, C) = (10, 5, 4, 45)
    (R, T, Fm, f_tilde, B, b_tilde) = model.sample(N, H, U)
    assert R.shape == (N, U) and R.dtype == np.dtype('bool')
    assert T.shape == (C, U) and T.dtype == np.dtype('bool')
    assert Fm.shape == (C, 3) and Fm.dtype == np.dtype('bool')
    assert f_tilde.shape == (C, U, 3) and f_tilde.dtype == np.dtype('bool')
    assert B.shape == (C, H) and B.dtype == np.dtype('float64')
    assert b_tilde.shape == (C, U) and b_tilde.dtype == np.dtype('float64')
    assert np.all(Fm.sum(axis=1) == 1) and np.all(f_tilde.sum(axis=2) == 1)


def test_sample_R_pi():
    model = fcdiff.UnsharedRegionModel()
    r = model.sample_R(3, 10000)
    nptest.assert_allclose(np.mean(r, axis=1), model.pi, atol=0.02)


def test_sample_T_cases():
    model = fcdiff.UnsharedRegionModel()
    r = np.tile(np.array([[1], [0], [0]], dtype='bool'), (1, 10000))
    t = model.sample_T(r)
    nptest.assert_equal(t[2, :], 0)
    nptest.assert_allclose(np.mean(t[0:2, :], axis=1), model.eta, atol=0.05)
    nptest.assert_array_equal(model.sample_T(np.ones((3, 1), dtype='bool')), np.ones((3, 1), dtype='bool'))
    nptest.assert_array_equal(model.sample_T(np.zeros((3, 1), dtype='bool')), np.zeros((3, 1), dtype='bool'))


def test_sample_F_gamma():
    model = fcdiff.UnsharedRegionModel()
    f = model.sample_F(100)
    nptest.assert_allclose(np.mean(f, axis=0), model.gamma, atol=0.05)


@pytest.mark.parametrize("k", [0, 1, 2])
@pytest.mark.parametrize("tval", [0, 1])
def test_sample_F_tilde_probabilities(k, tval):
    model = fcdiff.UnsharedRegionModel()
    U = 20000
    f = np.zeros((1, 3), dtype=bool)
    f[0, k] = True
    t = np.full((1, U), bool(tval))
    ft = model.sample_F_tilde(f, t)
    e = model.epsilon
    exp = np.full(3, (e / 2) if not tval else (1 - e) / 2)
    exp[k] = (1 - e) if not tval else e
    nptest.assert_allclose(ft[0].mean(axis=0), exp, atol=0.02)


@pytest.mark.parametrize("k", [0, 1, 2])
def test_sample_B_moments_and_ks(k):
    model = fcdiff.UnsharedRegionModel()
    f = np.zeros((1, 3), dtype=bool)
    f[0, k] = True
    b = model.sample_B(f, 50000)
    assert b.min() >= -1 and b.max() <= 1
    nptest.assert_allclose(b.mean(), model.mu[k], atol=0.002)
    nptest.assert_allclose(b.std(), model.sigma[k], atol=0.002)
    (_, p) = scipy.stats.kstest(b[0], scipy.stats.norm(model.mu[k], model.sigma[k]).cdf)
    assert p > 1e-3
    ft = np.zeros((1, 50000, 3), dtype=bool)
    ft[0, :, k] = True
    bt = model.sample_B_tilde(ft)
    (_, p) = scipy.stats.kstest(bt[0], scipy.stats.norm(model.mu[k], model.sigma[k]).cdf)
    assert p > 1e-3


def test_sample_B_clipped():
    model = fcdiff.UnsharedRegionModel()
    model.sigma = np.array([5.0, 5.0, 5.0])
    f = np.zeros((4, 3), dtype=bool)
    f[:, 1] = True
    b = model.sample_B(f, 1000)
    assert b.min() == -1.0 and b.max() == 1.0


def test_sampler_reseed_and_shard_invariance():
    """Counter-based: the same key gives the same draw whatever the launch
    geometry; an edge shard equals the slice of the full draw."""
    m1 = fcdiff.UnsharedRegionModel()
    m2 = fcdiff.UnsharedRegionModel()
    a = m1.sample(12, 6, 7)
    b = m2.sample(12, 6, 7)
    for (x, y) in zip(a, b):
        nptest.assert_array_equal(x, y)
    c = m1.sample(12, 6, 7)                 # the stream advances between calls
    assert not np.array_equal(a[5], c[5])
    m3 = fcdiff.UnsharedRegionModel()
    (c0, Cl) = (20, 30)
    part = m3.sample_device(12, 6, 7, c0=c0, C=Cl)
    nptest.assert_array_equal(_dev.download(part[0]) > 0, a[0])
    nptest.assert_array_equal(_dev.download(part[1]) > 0, a[1][c0:c0 + Cl])
    nptest.assert_array_equal(_dev.download(part[2]) > 0, a[2][c0:c0 + Cl])
    nptest.assert_array_equal(_dev.download(part[3]) > 0, a[3][c0:c0 + Cl])
    nptest.assert_array_equal(_dev.download(part[4]), a[4][c0:c0 + Cl])
    nptest.assert_array_equal(_dev.download(part[5]), a[5][c0:c0 + Cl])


def test_joint_sample_matches_oracle_sampler_in_distribution():
    model = fcdiff.UnsharedRegionModel()
    (N, H, U) = (40, 60, 80)
    (r, t, f, ft, b, bt) = model.sample(N, H, U)
    th = O.Theta()
    (ro, to, fo, fto, bo, bto) = O.sample(th, N, H, U, np.random.RandomState(123))
    nptest.assert_allclose(r.mean(), ro.mean(), atol=0.02)
    nptest.assert_allclose(t.mean(), to.mean(), atol=0.02)
    nptest.assert_allclose(f.mean(axis=0), fo.mean(axis=0), atol=0.05)
    nptest.assert_allclose(ft.mean(axis=(0, 1)), fto.mean(axis=(0, 1)), atol=0.02)
    assert scipy.stats.ks_2samp(b.ravel()[::7], bo.ravel()[::7]).pvalue > 1e-4
    assert scipy.stats.ks_2samp(bt.ravel()[::7], bto.ravel()[::7]).pvalue > 1e-4
    # T is consistent with R on the util edge order
    (n, m) = O.edge_pairs(N)
    both = r[n] & r[m]
    neither = ~r[n] & ~r[m]
    assert np.all(t[both]) and not np.any(t[neither])


# ------------------------------------------------------------------ K1
@pytest.mark.parametrize("S,N,T", [(1, 2, 2), (3, 6, 50), (5, 33, 97), (2, 90, 200), (4, 128, 256), (2, 130, 64),
                                   # tensor-core path: odd subject counts (a lone subject in the last pair), tail
                                   # blocks of 2 / 16 / 72 rows (transposed tiles, UMMA N = 16 / 16 / 80), no tail,
                                   # more work items than SMs (persistent CTAs, both TMEM buffers reused)
                                   (5, 130, 64), (3, 272, 96), (7, 200, 128), (1, 256, 64), (61, 300, 40),
                                   # the last SIMT size and the first tensor-core one (a single 64-row tile)
                                   (3, 63, 64), (3, 64, 64),
                                   # tail 112 (the widest transposed tile, UMMA N = 112), tail 113 (a full
                                   # 128-wide tile with masked rows), tail 127, no tail with three tiles
                                   (3, 240, 96), (3, 241, 96), (3, 255, 64), (3, 384, 64),
                                   # Schaefer-1000: eight tiles, tail 104
                                   (2, 1000, 96),
                                   # T around kKChunk = 32: one K chunk with 1 / 0 padded columns, two chunks
                                   (3, 130, 31), (3, 130, 32), (3, 130, 33), (3, 40, 33)])
@pytest.mark.parametrize("fisher", [True, False])
def test_corr_fisherz_vs_numpy(S, N, T, fisher):
    rng = np.random.RandomState(S * 1000 + N)
    mix = rng.standard_normal((N, N)) * 0.4 + np.eye(N)
    ts = np.einsum("nm,smt->snt", mix, rng.standard_normal((S, N, T))).astype(np.float32)
    ts += rng.uniform(-50, 50, (S, N, 1)).astype(np.float32)          # large row means
    got = corr.correlations(ts, fisher=fisher)
    exp = O.corr_fisherz(ts, fisher=fisher)
    assert got.shape == (N * (N - 1) // 2, S) and got.dtype == np.float64
    if T == 2:
        nptest.assert_allclose(np.abs(np.tanh(got)) if fisher else np.abs(got), 1.0, rtol=1e-5)
        return
    r_got = np.tanh(got) if fisher else got
    r_exp = np.tanh(exp) if fisher else exp
    # tolerance of the stage (parity unpinned by the reference): fp32 inputs,
    # split-TF32 products with fp32 accumulation -> |dr| <= 2e-6
    nptest.assert_allclose(r_got, r_exp, rtol=0, atol=2e-6)


def test_corr_config3_shape():
    """BASELINE.json configs[2]'s time series: Schaefer-400, 1200 TRs (8 subjects of the 1000).  The fp32
    accumulation over T / 8 = 150 MMAs per product bounds |dr| by 2.4e-6 (DESIGN.md 4); N = 400 has a
    16-row tail block."""
    (S, N, T) = (8, 400, 1200)
    rng = np.random.RandomState(7)
    mix = rng.standard_normal((N, N)) * 0.2 + np.eye(N)
    ts = np.einsum("nm,smt->snt", mix, rng.standard_normal((S, N, T))).astype(np.float32)
    got = corr.correlations(ts, fisher=False)
    exp = O.corr_fisherz(ts, fisher=False)
    nptest.assert_allclose(got, exp, rtol=0, atol=2.4e-6)
    z = corr.correlations(ts, fisher=True)
    nptest.assert_allclose(np.tanh(z), exp, rtol=0, atol=2.4e-6)


def test_corr_feeds_fit():
    rng = np.random.RandomState(0)
    ts = rng.standard_normal((8, 6, 120)).astype(np.float32)
    z = corr.correlations(ts, fisher=False)
    fit = fcdiff.fit.UnsharedRegionFit()
    fit.b, fit.bt = z[:, :4], z[:, 4:]
    fit.model = fcdiff.UnsharedRegionModel()
    fit.max_iters = 2
    fit.run()
    assert len(fit.energy) >= 2 and np.all(np.isfinite(fit.energy))
