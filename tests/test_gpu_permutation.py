"""Permutation inference on the GPU: the max-T counting kernel (csrc/fcd_permutation.cu) against the NumPy
oracle (oracle/permutation.py), the statistics of ``sweep.permutation_inference`` against individual fits,
its p-values against the oracle, streams and rank splits, planted recovery, and the configs[4] shape."""
import copy

import numpy as np
import numpy.testing as nptest
import pytest
import scipy.stats
import torch

from oracle import iar_oracle as O
from oracle import permutation as OP

pytestmark = pytest.mark.gpu

import fcdiff_b200 as fcdiff          # noqa: E402
from fcdiff_b200 import sweep         # noqa: E402

CHUNK = 512                           # kMtChunk of csrc/fcd_permutation.cu


def _matrix(kind, R1, K, seed=0):
    rng = np.random.RandomState(seed + 7 * R1 + K)
    if kind == "continuous":
        return rng.randn(R1, K)
    if kind == "ties3":
        return rng.choice([0.1, 0.2, 0.3], (R1, K))
    if kind == "equal":
        return np.full((R1, K), 0.25)
    if kind == "obs_max":
        T = rng.rand(R1, K)
        T[0] = 2.0 + rng.rand(K)
        return T
    if kind == "obs_min":
        T = rng.rand(R1, K) + 1.0
        T[0] = rng.rand(K) * 0.5
        return T
    if kind == "zeros":
        return rng.choice([-0.0, 0.0], (R1, K))
    raise ValueError(kind)


def _check(T, families=None, device=True):
    (p, pf) = sweep.maxt_pvalues(torch.from_numpy(T).cuda() if device else T, families)
    (po, pfo) = OP.maxt_pvalues(T, families)
    nptest.assert_array_equal(p, po)
    nptest.assert_array_equal(pf, pfo)
    return p, pf


@pytest.mark.parametrize("R1", [1, 2, 31, 1001])
@pytest.mark.parametrize("K", [1, CHUNK - 1, CHUNK, CHUNK + 1, 2 * CHUNK + 1])
def test_kernel_equals_oracle_continuous(R1, K):
    _check(_matrix("continuous", R1, K))


@pytest.mark.parametrize("kind", ["ties3", "equal", "obs_max", "obs_min", "zeros"])
@pytest.mark.parametrize("R1,K", [(1, 7), (2, CHUNK + 1), (31, CHUNK), (31, 2 * CHUNK + 1), (1001, CHUNK - 1)])
def test_kernel_equals_oracle_ties_and_extremes(kind, R1, K):
    (p, pf) = _check(_matrix(kind, R1, K), device=(R1 != 2))     # one shape from a host array
    if kind == "obs_max":
        nptest.assert_array_equal(p, 1.0 / R1)
        nptest.assert_array_equal(pf, 1.0 / R1)
    if kind in ("obs_min", "equal", "zeros"):
        nptest.assert_array_equal(p, 1.0)
        nptest.assert_array_equal(pf, 1.0)


@pytest.mark.parametrize("kind", ["continuous", "ties3"])
def test_kernel_equals_oracle_atlas_width(kind):
    """K = 80,200: the 400 region and 79,800 connection columns of one Schaefer-400 row, one family and two."""
    T = _matrix(kind, 1001, 80200)
    _check(T)
    _check(T, [(0, 400), (400, 80200)])


def test_families_are_independent():
    T = _matrix("continuous", 31, 3 * CHUNK + 5)
    fams = [(0, 700), (700, 3 * CHUNK + 5)]
    (p1, pf1) = _check(T, fams)
    T2 = T.copy()
    T2[:, 700:] = _matrix("ties3", 31, T.shape[1] - 700, seed=3)
    (p2, pf2) = _check(T2, fams)
    nptest.assert_array_equal(p1[:700], p2[:700])
    nptest.assert_array_equal(pf1[:700], pf2[:700])
    # a column outside every family is NaN
    (p3, pf3) = _check(T, [(5, 700)])
    assert np.isnan(p3[:5]).all() and np.isnan(pf3[700:]).all()


def test_kernel_rejects_sizes_beyond_its_limits():
    from fcdiff_b200 import _dev, _lib
    lib = _lib.load()
    assert lib.fcd_maxt_ws_bytes(10001, 500500) == 8 * 10001 * (500500 + (500500 + CHUNK - 1) // CHUNK)
    assert lib.fcd_maxt_ws_bytes((1 << 20) + 1, 10) == 0
    assert lib.fcd_maxt_ws_bytes(10, (1 << 24) + 1) == 0
    buf = _dev.zeros((64,))
    idx = _dev.zeros((8,), torch.int64)
    n0 = lib.fcd_launch_count()
    for (R1, K, k0, k1) in (((1 << 20) + 1, 8, 0, 8), (4, (1 << 24) + 1, 0, 8), (4, 8, 3, 3), (4, 8, 0, 9), (0, 8, 0, 8)):
        rc = lib.fcd_maxt_counts(_dev.ptr(buf), R1, K, K, _dev.ptr(idx), k0, k1, _dev.ptr(idx), _dev.ptr(idx),
                                 _dev.ptr(buf), _dev.stream())
        assert rc != 0
    assert lib.fcd_launch_count() == n0


# ------------------------------------------------------------------ statistics of permutation_inference
def _problem(N=12, H=14, U=10, seed=3):
    (_, _, _, _, b, bt) = O.sample(O.Theta(), N, H, U, np.random.RandomState(seed))
    corr = np.concatenate([b, bt], axis=1)
    labels = np.r_[np.zeros(H, bool), np.ones(U, bool)]
    return corr, labels


def _individual(corr, labels, n_perm, seed, i, opts, model=None, shared_planes=True):
    """Region and connection statistics of replica i fitted on its own, the way the sweep builds it."""
    model = fcdiff.UnsharedRegionModel() if model is None else model
    lab = sweep.permuted_labels(labels, n_perm, seed)
    corr_dev = (corr if torch.is_tensor(corr) else torch.from_numpy(corr)).cuda().to(torch.float64)
    con = torch.from_numpy(np.flatnonzero(~lab[i])).cuda()
    pat = torch.from_numpy(np.flatnonzero(lab[i])).cuda()
    fit = fcdiff.fit.UnsharedRegionFit()
    fit.model = copy.deepcopy(model)
    sweep._configure(fit, opts)
    if shared_planes and not opts.get("update_mu_sigma"):
        fit.set_shared_inputs(sweep.SharedPlanes(corr_dev, model, missing=opts.get("missing", "reject")), con, pat)
    else:
        (fit.b, fit.bt) = (corr_dev.index_select(1, con), corr_dev.index_select(1, pat))
    fit.run()
    return np.exp(fit._lq_R[:, :, 1]).mean(1), fit.connection_posteriors(maps=False).anomalous_rate


def _nan_corr(corr, frac=0.03, seed=4):
    rng = np.random.RandomState(seed)
    out = corr.copy()
    out[rng.uniform(size=out.shape) < frac] = np.nan
    return out


@pytest.mark.parametrize("case", ["reference", "symmetric", "marginalize", "update_mu_sigma", "regions_only"])
def test_statistics_equal_individual_fits(case):
    (corr, labels) = _problem(N=14, H=12, U=11, seed=5)
    opts = dict(max_iters=4, rel_tol=-1.0)
    kw = dict(connections=True, shared_planes=True)
    if case == "symmetric":
        opts["edge_lookup"] = "symmetric"
    if case == "marginalize":
        opts["missing"] = "marginalize"
        corr = _nan_corr(corr)
    if case == "update_mu_sigma":
        opts["update_mu_sigma"] = True
        kw["shared_planes"] = False
    if case == "regions_only":
        kw["connections"] = False
    (N, C) = (14, 91)
    res = sweep.permutation_inference(corr, labels, 4, seed=2, fit_options=opts, streams=2, **kw)
    stats = res.statistics.cpu().numpy()
    assert stats.shape == (5, N + (C if kw["connections"] else 0))
    nptest.assert_array_equal(res.replica_index, np.arange(5))
    for i in (0, 3):
        (region, conn) = _individual(corr, labels, 4, 2, i, opts, shared_planes=kw["shared_planes"])
        nptest.assert_array_equal(stats[i, :N], region)
        if kw["connections"]:
            nptest.assert_array_equal(stats[i, N:], conn)
    nptest.assert_array_equal(res.region_rate, stats[0, :N])
    if kw["connections"]:
        nptest.assert_array_equal(res.connection_rate, stats[0, N:])
    else:
        assert res.connection_rate is None and res.connection_p is None and res.connection_q is None


def test_pvalues_equal_the_oracle_and_bh():
    (corr, labels) = _problem(N=16, H=12, U=12, seed=8)
    (N, C) = (16, 120)
    res = sweep.permutation_inference(corr, labels, 19, seed=1, fit_options=dict(max_iters=3, rel_tol=-1.0))
    stats = res.statistics.cpu().numpy()
    (p, pf) = OP.maxt_pvalues(stats, [(0, N), (N, N + C)])
    nptest.assert_array_equal(res.region_p, p[:N])
    nptest.assert_array_equal(res.region_p_fwer, pf[:N])
    nptest.assert_array_equal(res.connection_p, p[N:])
    nptest.assert_array_equal(res.connection_p_fwer, pf[N:])
    nptest.assert_array_equal(res.region_q, scipy.stats.false_discovery_control(p[:N], method="bh"))
    nptest.assert_array_equal(res.connection_q, scipy.stats.false_discovery_control(p[N:], method="bh"))
    # the summaries are those of permutation_sweep
    ref = sweep.permutation_sweep(corr, labels, 19, seed=1, fit_options=dict(max_iters=3, rel_tol=-1.0))
    assert sorted(ref) == sorted(res.replicas)
    for i in ref:
        assert ref[i]["energy"] == res.replicas[i]["energy"]
    # no permutation: every p-value is 1
    res0 = sweep.permutation_inference(corr, labels, 0, fit_options=dict(max_iters=2))
    for name in ("region_p", "region_p_fwer", "connection_p", "connection_p_fwer"):
        nptest.assert_array_equal(getattr(res0, name), 1.0)


def test_streams_and_rank_splits_are_bit_identical():
    (corr, labels) = _problem(N=12, H=14, U=10, seed=3)
    opts = dict(max_iters=4, rel_tol=-1.0)
    runs = [sweep.permutation_inference(corr, labels, 6, seed=5, fit_options=opts, streams=s) for s in (1, 2, 3)]
    ref = runs[0].statistics.cpu().numpy()
    for r in runs[1:]:
        nptest.assert_array_equal(r.statistics.cpu().numpy(), ref)
        for name in ("region_p", "region_p_fwer", "region_q", "connection_p", "connection_p_fwer", "connection_q"):
            nptest.assert_array_equal(getattr(r, name), getattr(runs[0], name))
    parts = [sweep.permutation_inference(corr, labels, 6, seed=5, fit_options=opts, rank=k, world=2, gather=False)
             for k in range(2)]
    assert parts[0].region_p is None and parts[1].region_rate is None
    nptest.assert_array_equal(parts[0].region_rate, runs[0].region_rate)
    idx = np.concatenate([q.replica_index for q in parts])
    rows = np.concatenate([q.statistics.cpu().numpy() for q in parts])
    stacked = rows[np.argsort(idx)]
    nptest.assert_array_equal(np.sort(idx), np.arange(7))
    nptest.assert_array_equal(stacked, ref)
    (p, pf) = sweep.maxt_pvalues(stacked, [(0, 12), (12, 12 + 66)])
    nptest.assert_array_equal(p[:12], runs[0].region_p)
    nptest.assert_array_equal(pf[12:], runs[0].connection_p_fwer)


def test_planted_regions_are_found():
    """Regions 3 and 17 anomalous in 60 % of the patients.  The fits read each region's edges by the unordered
    pair (``edge_lookup="symmetric"``): the reference's lookup reads, for some pairs, the edge of another pair
    and moves region 3's evidence to region 16.  eta = 0.8 makes most edges of an anomalous region anomalous."""
    th = O.Theta(eta=0.8)
    (N, H, U) = (30, 40, 40)
    pi = np.full(N, 0.01)
    pi[[3, 17]] = 0.6
    (_, _, _, _, b, bt) = OP.sample_planted(th, N, H, U, pi, np.random.RandomState(0))
    corr = np.concatenate([b, bt], axis=1)
    labels = np.r_[np.zeros(H, bool), np.ones(U, bool)]
    res = sweep.permutation_inference(corr, labels, 99, seed=0,
                                      fit_options=dict(max_iters=10, edge_lookup="symmetric"))
    print("planted region_p_fwer", res.region_p_fwer[[3, 17]], "smallest unplanted",
          np.delete(res.region_p_fwer, [3, 17]).min())
    assert res.region_p_fwer[3] <= 0.05 and res.region_p_fwer[17] <= 0.05


def test_config4_shape():
    """Schaefer-400 x (500 + 500) from the device sampler, 15 permutations: rows 0 and 7 against individual
    fits; the peak device memory is printed."""
    (N, H, U) = (400, 500, 500)
    model = fcdiff.UnsharedRegionModel()
    (_, _, _, _, b, bt) = model.sample_device(N, H, U)
    corr = torch.cat([b, bt], dim=1)
    del b, bt
    labels = np.r_[np.zeros(H, bool), np.ones(U, bool)]
    start = fcdiff.UnsharedRegionModel()
    start.eta += 0.1
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    res = sweep.permutation_inference(corr, labels, 15, model=start)
    torch.cuda.synchronize()
    print("configs[4] shape, 16 replicas: peak device memory %.2f GB" % (torch.cuda.max_memory_allocated() / 1e9))
    stats = res.statistics.cpu().numpy()
    assert stats.shape == (16, N + N * (N - 1) // 2)
    for i in (0, 7):
        (region, conn) = _individual(corr, labels, 15, 0, i, {}, model=start)
        nptest.assert_array_equal(stats[i, :N], region)
        nptest.assert_array_equal(stats[i, N:], conn)
    (p, pf) = OP.maxt_pvalues(stats, [(0, N), (N, stats.shape[1])])
    nptest.assert_array_equal(res.region_p_fwer, pf[:N])
    nptest.assert_array_equal(res.connection_p, p[N:])
