"""GPU: partial correlations (fcd_corr_partial, csrc/fcd_corr_partial.cu) through corr and the C-ABI.

Against the fp64 oracle (oracle/partial.py): N = 2 .. 1000, fewer and more kept frames than regions,
confounds, censoring and ragged lengths, Ledoit-Wolf and fixed shrinkage: the accuracy standard against the
longdouble reference (oracle/partial.py: accuracy) for Ledoit-Wolf, |dr| <= 1e-9 (|dz| the same over
1 - r^2) and delta within 1e-12 elsewhere.  Bit-identity: samples of censored frames are never read, a subject's column
does not depend on the batch, the padding or the internal batch size.  Unusable regions, singular subjects,
the output layout and the unchanged Pearson default.  An entry that is exactly zero may differ in the sign
of zero only."""
import numpy as np
import pytest
import torch

from oracle import iar_oracle as O
from oracle import partial as OP

pytestmark = pytest.mark.gpu

import fcdiff_b200 as fcdiff                  # noqa: E402
from fcdiff_b200 import _dev, _lib, corr      # noqa: E402

R_TOL = 1e-9
DELTA_TOL = 1e-12
SENTINEL = 0x7FF4DEADBEEF0001


def data(S, N, T, K, seed, censor=0.0, lengths=None, factors=8):
    """Planted-factor series (the K1 workload's structure) plus a confound component and an offset."""
    rng = np.random.RandomState(seed)
    a = np.where(rng.rand(N) < 0.5, 0.55, -0.27)
    z = rng.standard_normal((S, factors, T))
    ts = np.sqrt(1 - a * a)[None, :, None] * rng.standard_normal((S, N, T)) + \
        a[None, :, None] * z[:, np.arange(N) % factors, :]
    g = rng.standard_normal((S, T, K))
    ts += np.einsum("nk,stk->snt", 0.5 * rng.standard_normal((N, K)), g) + rng.uniform(-50, 50, (S, N, 1))
    keep = rng.rand(S, T) >= censor
    if lengths is not None:
        keep &= np.arange(T)[None, :] < np.asarray(lengths)[:, None]
    return ts.astype(np.float32), keep, (g if K else None)


def gpu(ts, keep=None, g=None, fisher=True, missing=False, shrinkage="ledoit-wolf", out=None, s0=0):
    S = ts.shape[0]
    delta = _dev.empty((S,))
    o = corr.correlations_device(_dev.upload(ts, np.float32), fisher=fisher, missing=missing, out=out, s0=s0,
                                 sample_mask=None if keep is None else _dev.upload(keep, np.bool_),
                                 confounds=None if g is None else _dev.upload(g, np.float64), kind="partial",
                                 shrinkage=shrinkage, shrinkage_out=delta)
    return _dev.download(o), _dev.download(delta)


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    eq = (a.view(np.int64) == b.view(np.int64)) | ((a == 0) & (b == 0))
    assert eq.all(), "%d entries differ, max |d| = %g" % ((~eq).sum(), np.nanmax(np.abs(a - b)))


def check(got_r, got_z, ref_r, ref_z, got_d=None, ref_d=None, what=""):
    dr = np.abs(got_r - ref_r)
    bound_z = R_TOL / np.maximum(1.0 - ref_r * ref_r, 2.0 ** -52)
    dz = np.abs(got_z - ref_z)
    print("partial %s: max |dr| = %.3g, max |dz|(1 - r^2) = %.3g, max |r| = %.3f%s" % (
        what, dr.max(), (dz * (1.0 - ref_r * ref_r)).max(), np.abs(ref_r).max(),
        "" if got_d is None else ", max |d delta| = %.3g" % np.abs(got_d - ref_d).max()))
    assert dr.max() <= R_TOL
    assert (dz <= bound_z).all()
    if got_d is not None:
        assert np.abs(got_d - ref_d).max() <= DELTA_TOL


CASES = [  # (S, N, T, K, censor, ragged)
    (3, 2, 40, 0, 0.0, False),
    (3, 3, 50, 1, 0.2, False),
    (4, 31, 25, 0, 0.0, False),                 # T < N: Ledoit-Wolf carries the rank deficiency
    (3, 64, 200, 2, 0.1, True),
    (3, 65, 50, 0, 0.1, False),                 # T < N
    (2, 200, 150, 3, 0.1, True),                # T < N
    (2, 400, 1200, 0, 0.0, False),
    (2, 400, 200, 6, 0.05, False),              # T < N with confounds
    (2, 400, 900, 4, 0.1, True),
    (1, 1000, 1200, 0, 0.0, False),
    (1, 1000, 600, 2, 0.1, False),              # T < N
]


@pytest.mark.parametrize("case", CASES, ids=["S%d-N%d-T%d-K%d" % c[:4] for c in CASES])
def test_against_oracle(case):
    (S, N, T, K, censor, ragged) = case
    lengths = np.linspace(T // 2, T, S).astype(int) if ragged else None
    (ts, keep, g) = data(S, N, T, K, 100 + N + K, censor, lengths)
    (ref_r, _) = OP.corr_partial(ts, keep, g, fisher=False)
    ref_z = np.arctanh(np.clip(ref_r, -1 + 2.0 ** -53, 1 - 2.0 ** -53))
    (got_r, got_d) = gpu(ts, keep, g, fisher=False)
    (got_z, got_d2) = gpu(ts, keep, g, fisher=True)
    same_bits(got_d, got_d2)
    # the accuracy standard against the longdouble reference (oracle/partial.py: accuracy); z follows r
    for s in range(S):
        a = OP.accuracy(got_r[:, s], got_d[s], OP.references(ts[s], keep[s], None if g is None else g[s]))
        print("partial N=%d T=%d K=%d s%d: kappa %.3g, err_gpu %.3g, err_np %.3g, ratio %.2f, delta ratio %.2f" % (
            N, T, K, s, a["kappa"], a["err_gpu"], a["err_np"], a["ratio"], a["dratio"]))
        assert a["ratio"] <= OP.F_R and a["dratio"] <= OP.F_DELTA
        tol = (OP.F_R + 1) * max(a["err_np"], OP.ERR_FLOOR)
        bound_z = tol / np.maximum(1.0 - ref_r[:, s] ** 2, 2.0 ** -52) + 2.0 ** -50 * np.abs(ref_z[:, s])
        assert (np.abs(got_z[:, s] - ref_z[:, s]) <= bound_z).all()


@pytest.mark.parametrize("N,T,K", [(40, 300, 0), (400, 1200, 3)])
def test_fixed_shrinkage(N, T, K):
    (ts, keep, g) = data(2, N, T, K, 7, censor=0.1)
    for d in (0.0, 0.3):
        (ref, _) = OP.corr_partial(ts, keep, g, fisher=False, shrinkage=d)
        (got, delta) = gpu(ts, keep, g, fisher=False, shrinkage=d)
        assert (delta == d).all()
        check(got, got, ref, ref, what="fixed %g N=%d" % (d, N))
    # delta = 0 is the inverse of the sample correlation matrix itself
    (z, _) = OP.unit_rows(ts[0], keep[0], None if g is None else g[0])
    P = np.linalg.inv(z @ z.T / keep[0].sum())
    (n, m) = O.edge_pairs(N)
    (got, _) = gpu(ts, keep, g, fisher=False, shrinkage=0.0)
    assert np.abs(got[:, 0] - (-P[n, m] / np.sqrt(P[n, n] * P[m, m]))).max() <= R_TOL
    (one, _) = gpu(ts, keep, g, shrinkage=1.0)
    assert (one == 0).all()


def test_censored_samples_are_never_read():
    (ts, keep, g) = data(3, 70, 120, 2, 3, censor=0.25)
    (base, d0) = gpu(ts, keep, g)
    bad = ts.copy()
    idx = np.argwhere(~keep)
    for (i, (s, t)) in enumerate(idx):
        bad[s, :, t] = (np.nan, np.inf, -np.inf, 1e30)[i % 4]
    (got, d1) = gpu(bad, keep, g)
    same_bits(got, base)
    same_bits(d1, d0)


def test_column_independent_of_batch_padding_and_internal_batch(monkeypatch):
    (S, N, T) = (5, 90, 140)
    (ts, keep, g) = data(S, N, T, 3, 11, censor=0.1, lengths=[140, 100, 120, 70, 140])
    (full, dfull) = gpu(ts, keep, g)
    for s in (0, 3):                                        # alone
        (one, d1) = gpu(ts[s:s + 1], keep[s:s + 1], g[s:s + 1])
        same_bits(one[:, 0], full[:, s])
        same_bits(d1[0], dfull[s])
    pad = 77                                                # padded to a longer T with censored frames
    ts_p = np.concatenate([ts, np.full((S, N, pad), np.nan, np.float32)], axis=2)
    keep_p = np.concatenate([keep, np.zeros((S, pad), bool)], axis=1)
    g_p = np.concatenate([g, np.zeros((S, pad, 3))], axis=1)
    (padded, dpad) = gpu(ts_p, keep_p, g_p)
    same_bits(padded, full)
    same_bits(dpad, dfull)
    for b in ("1", "2", "3"):                               # batch boundaries inside the call
        monkeypatch.setenv("FCD_CORR_PARTIAL_BATCH", b)
        (small, dsmall) = gpu(ts, keep, g)
        same_bits(small, full)
        same_bits(dsmall, dfull)


@pytest.mark.parametrize("missing", [False, True])
def test_unusable_regions(missing):
    (S, N, T, K) = (3, 50, 160, 2)
    (ts, keep, g) = data(S, N, T, K, 21, censor=0.1)
    t_kept = int(np.argmax(keep[0]))
    ts[0, 7, t_kept] = np.nan                               # non-finite kept sample
    ts[1, 20] = np.float32(3.25)                            # constant
    ts[2, 33] = (2.0 * g[2, :, 1] - 4.0).astype(np.float32)  # explained by a confound
    (got, delta) = gpu(ts, keep, g, fisher=False, missing=missing)
    (n, m) = O.edge_pairs(N)
    for (s, r) in ((0, 7), (1, 20), (2, 33)):
        on = (n == r) | (m == r)
        col = got[:, s]
        if missing:
            assert np.isnan(col[on]).all()
        else:
            assert (col[on] == 0).all()
        use = np.arange(N) != r
        (ref, dref) = OP.corr_partial(ts[s:s + 1, use], keep[s:s + 1], g[s:s + 1], fisher=False)
        assert np.abs(col[~on] - ref[:, 0]).max() <= R_TOL
        assert abs(delta[s] - dref[0]) <= DELTA_TOL


def test_singular_subject():
    (S, N, T) = (3, 30, 200)
    (ts, keep, _) = data(S, N, T, 0, 31)
    ts[1, 12] = ts[1, 4]                                   # duplicated region: R singular at shrinkage 0
    with pytest.raises(ValueError, match=r"subject\(s\) \[1\]"):
        corr.correlations(ts, kind="partial", shrinkage=0.0)
    # through the C-ABI: status set, column NaN, the other columns those of the subjects alone
    lib = _lib.load()
    ts_dev = _dev.upload(ts, np.float32)
    out = _dev.empty((N * (N - 1) // 2, S))
    status = torch.full((S,), -1, dtype=torch.int32, device="cuda")
    zws = torch.empty(lib.fcd_corr_partial_workspace_bytes(S, N, T, 0), dtype=torch.uint8, device="cuda")
    _lib.check(lib.fcd_corr_partial(_dev.ptr(ts_dev), S, N, T, None, None, 0, 0.0, _dev.ptr(out), S, 0, 1, 0, None,
                                    None, _dev.ptr(status), _dev.ptr(zws), _dev.stream()), "fcd_corr_partial")
    got = _dev.download(out)
    assert status.cpu().tolist() == [0, 1, 0]
    assert np.isnan(got[:, 1]).all()
    for s in (0, 2):
        (one, _) = gpu(ts[s:s + 1], shrinkage=0.0)
        same_bits(got[:, s], one[:, 0])
    # a shrunk matrix is not singular
    (shrunk, delta) = gpu(ts)
    assert np.isfinite(shrunk).all() and (delta > 0).all()


@pytest.mark.parametrize("s0,pitch", [(0, 4), (1, 4), (3, 7), (2, 9)])
def test_layout(s0, pitch):
    (S, N, T) = (3, 40, 90)
    (ts, keep, g) = data(S, N, T, 1, 41, censor=0.1)
    (ref, _) = gpu(ts, keep, g)
    C = N * (N - 1) // 2
    if s0 + S > pitch:
        pitch = s0 + S
    host = np.full((C, pitch), SENTINEL, dtype=np.int64).view(np.float64)
    out = _dev.upload(host, np.float64)
    (got, _) = gpu(ts, keep, g, out=out, s0=s0)
    same_bits(got[:, s0:s0 + S], ref)
    other = np.ones(pitch, bool)
    other[s0:s0 + S] = False
    assert (got[:, other].view(np.int64) == SENTINEL).all()


def test_cabi_matches_corr():
    (S, N, T, K) = (2, 45, 80, 2)
    (ts, keep, g) = data(S, N, T, K, 51, censor=0.1)
    (ref, dref) = gpu(ts, keep, g, missing=True)
    lib = _lib.load()
    out = _dev.empty((N * (N - 1) // 2, S))
    (ts_d, keep_d, g_d) = (_dev.upload(ts, np.float32), _dev.upload(keep.astype(np.uint8), np.uint8),
                           _dev.upload(g, np.float64))
    rank = torch.empty((S,), dtype=torch.int32, device="cuda")
    delta = _dev.empty((S,))
    status = torch.empty((S,), dtype=torch.int32, device="cuda")
    zws = torch.empty(lib.fcd_corr_partial_workspace_bytes(S, N, T, K), dtype=torch.uint8, device="cuda")
    _lib.check(lib.fcd_corr_partial(_dev.ptr(ts_d), S, N, T, _dev.ptr(keep_d), _dev.ptr(g_d), K, -1.0, _dev.ptr(out),
                                    S, 0, 1, 1, _dev.ptr(rank), _dev.ptr(delta), _dev.ptr(status), _dev.ptr(zws),
                                    _dev.stream()), "fcd_corr_partial")
    same_bits(_dev.download(out), ref)
    same_bits(_dev.download(delta), dref)
    assert rank.cpu().tolist() == [K, K] and status.cpu().tolist() == [0, 0]
    assert lib.fcd_corr_partial(_dev.ptr(ts_d), S, N, T, None, None, 0, 1.5, _dev.ptr(out), S, 0, 1, 0, None, None,
                                _dev.ptr(status), _dev.ptr(zws), _dev.stream()) != 0


def test_pearson_default_is_unchanged():
    (S, N, T, K) = (3, 70, 120, 2)
    (ts, keep, g) = data(S, N, T, K, 61, censor=0.1)
    same_bits(corr.correlations(ts, kind="pearson"), corr.correlations(ts))
    lib = _lib.load()
    ts_d = _dev.upload(ts, np.float32)
    out = _dev.empty((N * (N - 1) // 2, S))
    zws = torch.empty(lib.fcd_corr_workspace_bytes(S, N, T), dtype=torch.uint8, device="cuda")
    _lib.check(lib.fcd_corr_fisherz(_dev.ptr(ts_d), S, N, T, _dev.ptr(out), S, 0, 1, _dev.ptr(zws), _dev.stream()),
               "fcd_corr_fisherz")
    same_bits(corr.correlations(ts), _dev.download(out))
    (keep_d, g_d) = (_dev.upload(keep.astype(np.uint8), np.uint8), _dev.upload(g, np.float64))
    zws = torch.empty(lib.fcd_corr_clean_workspace_bytes(S, N, T, K), dtype=torch.uint8, device="cuda")
    _lib.check(lib.fcd_corr_fisherz_clean(_dev.ptr(ts_d), S, N, T, _dev.ptr(keep_d), _dev.ptr(g_d), K, _dev.ptr(out), S,
                                          0, 1, 0, None, _dev.ptr(zws), _dev.stream()), "fcd_corr_fisherz_clean")
    same_bits(corr.correlations(ts, sample_mask=keep, confounds=g, kind="pearson"), _dev.download(out))


def test_partial_correlations_feed_the_fit():
    (H, U, N, T) = (12, 10, 24, 300)
    (ts, _, _) = data(H + U, N, T, 0, 71)
    z = corr.correlations(ts, kind="partial")
    (b, bt) = (np.ascontiguousarray(z[:, :H]), np.ascontiguousarray(z[:, H:]))
    fit = fcdiff.fit.UnsharedRegionFit()
    (fit.b, fit.bt) = (b, bt)
    fit.model = fcdiff.UnsharedRegionModel()
    fit.update_mu_sigma = True
    fit.max_iters = 3
    fit.run()
    assert len(fit.energy) >= 2 and np.isfinite(fit.energy).all()
    ts[H + 2, 5, 40] = np.nan                              # a region without a usable series: marginalised
    zm = corr.correlations(ts, kind="partial", missing=True)
    assert np.isnan(zm).any()
    fit = fcdiff.fit.UnsharedRegionFit()
    (fit.b, fit.bt) = (np.ascontiguousarray(zm[:, :H]), np.ascontiguousarray(zm[:, H:]))
    fit.model = fcdiff.UnsharedRegionModel()
    fit.model.mu = np.array([-0.05, 0.0, 0.05])            # partial z are smaller than the default mu / sigma assume
    fit.model.sigma = np.array([0.03, 0.04, 0.05])
    fit.missing = "marginalize"
    fit.max_iters = 3
    fit.run()
    assert len(fit.energy) >= 2 and np.isfinite(fit.energy).all()
