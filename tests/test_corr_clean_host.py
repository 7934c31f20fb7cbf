"""CPU: the cleaned correlation stage's NumPy oracle (oracle/clean.py), the host packing / validation
(corr.pack_clean) and the file loaders (io.load_timeseries_list, io.load_confounds)."""
import numpy as np
import numpy.testing as nptest
import pytest

from oracle import clean as OC
from oracle import iar_oracle as O
from fcdiff_b200 import corr, io


def series(N, T, K, seed):
    rng = np.random.RandomState(seed)
    g = rng.standard_normal((T, K))
    x = rng.standard_normal((N, N)) @ rng.standard_normal((N, T)) + rng.standard_normal((N, K)) @ g.T
    return (x + rng.uniform(-5, 5, (N, 1))).astype(np.float32), g


@pytest.mark.parametrize("K", [0, 1, 3, 6])
def test_oracle_matches_precision_matrix_partial_correlation(K):
    (N, T) = (7, 90)
    (x, g) = series(N, T, K, 10 + K)
    keep = np.random.RandomState(K).rand(T) > 0.3
    (r, bad) = OC.subject_r(x, keep, g if K else None)
    assert not bad.any()
    exp = OC.partial_corr_precision(x.astype(np.float64), keep, g if K else None)
    nptest.assert_allclose(r, exp, atol=1e-12)


def test_oracle_without_confounds_is_pearson_over_kept_frames():
    (x, _) = series(6, 50, 0, 3)
    keep = np.ones(50, dtype=bool)
    keep[[4, 9, 33]] = False
    (r, _) = OC.subject_r(x, keep)
    nptest.assert_allclose(r, np.corrcoef(x[:, keep].astype(np.float64)), atol=1e-13)
    ts = x[None]
    nptest.assert_allclose(OC.corr_clean(ts, np.ones((1, 50), bool), fisher=True), O.corr_fisherz(ts), atol=1e-13)


def test_spike_regressor_is_censoring():
    (x, g) = series(6, 60, 3, 5)
    keep = np.ones(60, dtype=bool)
    spikes = [7, 31]
    gs = np.hstack([g] + [np.eye(60)[:, [t]] for t in spikes])
    (r_spike, _) = OC.subject_r(x, keep, gs)
    keep2 = keep.copy()
    keep2[spikes] = False
    (r_cens, _) = OC.subject_r(x, keep2, g)
    nptest.assert_allclose(r_spike, r_cens, atol=1e-12)


def test_oracle_unusable_rows_and_nan_convention():
    (x, g) = series(6, 40, 2, 8)
    keep = np.ones(40, dtype=bool)
    keep[[3, 4]] = False
    x[0, 3] = np.nan                     # censored: harmless
    x[1, 10] = np.inf                    # kept: unusable
    x[2] = np.float32(2.0)
    x[2, 4] = 7.0                        # constant over the kept frames
    x[3] = g[:, 1].astype(np.float32)    # explained by a confound
    ts = x[None]
    k = keep[None]
    G = g[None]
    out = OC.corr_clean(ts, k, G, fisher=False, mark_missing=True)
    out0 = OC.corr_clean(ts, k, G, fisher=False, mark_missing=False)
    (n, m) = O.edge_pairs(6)
    bad = np.isin(n, [1, 2, 3]) | np.isin(m, [1, 2, 3])
    assert np.isnan(out[bad, 0]).all() and np.isfinite(out[~bad, 0]).all()
    assert (out0[bad, 0] == 0).all()
    nptest.assert_array_equal(out[~bad, 0], out0[~bad, 0])


# ------------------------------------------------------------------ packing / validation
def test_pack_ragged_lists():
    rng = np.random.RandomState(0)
    ts = [rng.standard_normal((5, T)).astype(np.float32) for T in (30, 41, 35)]
    masks = [rng.rand(T) > 0.2 for T in (30, 41, 35)]
    conf = [rng.standard_normal((T, 3)) for T in (30, 41, 35)]
    conf[1][0] = np.nan
    masks[1][0] = False                  # a non-finite confound on a censored frame is fine
    (p, keep, c) = corr.pack_clean(ts, masks, conf)
    assert p.shape == (3, 5, 41) and p.dtype == np.float32
    assert keep.shape == (3, 41) and keep.dtype == np.uint8
    assert c.shape == (3, 41, 3) and c.dtype == np.float64
    for (s, T) in enumerate((30, 41, 35)):
        nptest.assert_array_equal(p[s, :, :T], ts[s])
        assert (p[s, :, T:] == 0).all()
        nptest.assert_array_equal(keep[s, :T], masks[s])
        assert (keep[s, T:] == 0).all()
        assert (c[s, T:] == 0).all()


def test_pack_array_without_mask_keeps_everything():
    ts = np.random.RandomState(1).standard_normal((2, 4, 20))
    (p, keep, c) = corr.pack_clean(ts)
    assert keep.all() and c is None and p.dtype == np.float32


def test_pack_rejections():
    rng = np.random.RandomState(2)
    ts = rng.standard_normal((2, 4, 20)).astype(np.float32)
    with pytest.raises(ValueError, match="regions"):
        corr.pack_clean([ts[0], ts[1][:3]])
    with pytest.raises(ValueError, match="sample_mask"):
        corr.pack_clean(ts, np.ones((2, 19), bool))
    with pytest.raises(ValueError, match="bool"):
        corr.pack_clean(ts, np.ones((2, 20), np.int32))
    with pytest.raises(ValueError, match="confounds"):
        corr.pack_clean(ts, None, rng.standard_normal((2, 21, 3)))
    with pytest.raises(ValueError, match="K = 65"):
        corr.pack_clean(ts, None, rng.standard_normal((2, 20, 65)))
    g = rng.standard_normal((2, 20, 3))
    g[1, 5, 2] = np.inf
    with pytest.raises(ValueError, match="non-finite"):
        corr.pack_clean(ts, None, g)
    m = np.ones((2, 20), bool)
    m[1, 5] = False
    corr.pack_clean(ts, m, g)                                         # censored: accepted
    m[0, :16] = False                                                 # 4 kept frames, K + 2 = 5
    with pytest.raises(ValueError, match="at least 5"):
        corr.pack_clean(ts, m, g)
    with pytest.raises(ValueError, match="subject 1"):
        corr.pack_clean([ts[0], ts[1]], [np.ones(20, bool), np.ones(19, bool)])
    with pytest.raises(ValueError, match="confounds"):
        corr.pack_clean([ts[0], ts[1][:, :15]], None, [g[0], g[1]])
    with pytest.raises(ValueError):
        corr.pack_clean(ts[0])


# ------------------------------------------------------------------ loaders
def test_load_timeseries_list(tmp_path):
    rng = np.random.RandomState(3)
    a = rng.standard_normal((4, 30)).astype(np.float32)
    b = rng.standard_normal((4, 25)).astype(np.float32)
    np.save(tmp_path / "a.npy", a.T)
    np.savetxt(tmp_path / "b.csv", b.T, delimiter=",", header=",".join("r%d" % i for i in range(4)), comments="")
    out = io.load_timeseries_list([str(tmp_path / "a.npy"), str(tmp_path / "b.csv")], time_major=True)
    assert [o.shape for o in out] == [(4, 30), (4, 25)]
    nptest.assert_array_equal(out[0], a)
    nptest.assert_allclose(out[1], b, rtol=1e-6)
    np.save(tmp_path / "a.npy", a)
    np.save(tmp_path / "c.npy", rng.standard_normal((5, 30)))
    with pytest.raises(ValueError, match="regions"):
        io.load_timeseries_list([str(tmp_path / "a.npy"), str(tmp_path / "c.npy")])
    with pytest.raises(ValueError, match="differ"):
        io.load_timeseries([str(tmp_path / "a.npy"), str(tmp_path / "b.csv")])


@pytest.mark.parametrize("ext", [".tsv", ".csv"])
def test_load_confounds_table(tmp_path, ext):
    d = "\t" if ext == ".tsv" else ","
    names = ["global_signal", "csf", "trans_x", "trans_x_derivative1"]
    rows = [["1.5", "2", "0.1", "n/a"], ["1.25", "2.5", "-0.2", "-0.3"], ["1", "3e-1", "0", "0.2"]]
    p = tmp_path / ("conf" + ext)
    p.write_text(d.join(names) + "\n" + "\n".join(d.join(r) for r in rows) + "\n")
    g = io.load_confounds(str(p))
    assert g.shape == (3, 4) and g.dtype == np.float64
    assert np.isnan(g[0, 3]) and g[1, 3] == -0.3
    g = io.load_confounds(str(p), columns=["trans_x", "global_signal"])
    nptest.assert_array_equal(g, [[0.1, 1.5], [-0.2, 1.25], [0.0, 1.0]])
    with pytest.raises(ValueError, match="no column"):
        io.load_confounds(str(p), columns=["white_matter"])


def test_load_confounds_npy(tmp_path):
    g = np.random.RandomState(4).standard_normal((12, 5))
    np.save(tmp_path / "g.npy", g)
    nptest.assert_array_equal(io.load_confounds(str(tmp_path / "g.npy")), g)
    nptest.assert_array_equal(io.load_confounds(str(tmp_path / "g.npy"), columns=[4, 0]), g[:, [4, 0]])
    np.save(tmp_path / "v.npy", g[:, 0])
    assert io.load_confounds(str(tmp_path / "v.npy")).shape == (12, 1)
