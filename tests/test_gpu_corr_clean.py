"""GPU: correlations from cleaned time series (fcd_corr_fisherz_clean, csrc/fcd_corr_clean.cu).

Bit-identity contracts: an all-kept mask without confounds gives the bits of fcd_corr_fisherz (+ the
missing marks); samples of censored frames are never read; a subject's column does not depend on the
padding of the batch or on extra censored frames; dropped confound columns leave the bits of zero columns.
Against the fp64 oracle (oracle/clean.py): random masks, ragged lengths and K = 1 .. 64 confounds on the
tensor-core and SIMT paths; spike regressors against censoring; the missing marks; the output layout.
An entry that is exactly zero may differ in the sign of zero only."""
import numpy as np
import pytest
import torch

from oracle import clean as OC
from oracle import iar_oracle as O

pytestmark = pytest.mark.gpu

from fcdiff_b200 import _dev, corr       # noqa: E402

SENTINEL = 0x7FF4DEADBEEF0001
TC_DELTA = 2e-6                          # tensor cores, <= 256 kept frames (tests/test_gpu_corr_edges.py)
TC_LONG = 6e-6                           # tensor cores, ~1000 kept frames: the T = 2400 figure of DESIGN.md 4
SIMT_DELTA = 2.0 ** -23 + 1e-12          # fp32 rounding of both standardised rows
SIMT_CLEAN = SIMT_DELTA + 1e-10          # ... plus the residue of the fp64 projection


@pytest.fixture(params=["tc", "simt"])
def path(request, monkeypatch):
    monkeypatch.delenv("FCD_CORR_SIMT", raising=False)
    if request.param == "simt":
        monkeypatch.setenv("FCD_CORR_SIMT", "1")
    return request.param


def simt(monkeypatch):
    monkeypatch.setenv("FCD_CORR_SIMT", "1")


def data(S, N, T, K, seed, censor=0.2, lengths=None):
    """Mixed region series with a confound component, random masks and (optionally) ragged lengths."""
    rng = np.random.RandomState(seed)
    g = rng.standard_normal((S, T, K))
    mix = rng.standard_normal((N, N)) * 0.4 + np.eye(N)
    ts = np.einsum("nm,smt->snt", mix, rng.standard_normal((S, N, T)))
    ts += np.einsum("nk,stk->snt", rng.standard_normal((N, K)), g) + rng.uniform(-50, 50, (S, N, 1))
    keep = rng.rand(S, T) >= censor
    if lengths is not None:
        keep &= np.arange(T)[None, :] < np.asarray(lengths)[:, None]
    return ts.astype(np.float32), keep, g


def gpu(ts, keep=None, g=None, fisher=True, missing=False, out=None, s0=0, rank=None):
    o = corr.correlations_device(_dev.upload(ts, np.float32), fisher=fisher, missing=missing, out=out, s0=s0,
                                 sample_mask=None if keep is None else _dev.upload(keep, np.bool_),
                                 confounds=None if g is None else _dev.upload(g, np.float64), rank=rank)
    return _dev.download(o)


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    eq = (a.view(np.int64) == b.view(np.int64)) | ((a == 0) & (b == 0))
    assert eq.all(), "%d entries differ, max |d| = %g" % ((~eq).sum(), np.nanmax(np.abs(a - b)))


# ------------------------------------------------------------------ 1. all kept, no confounds
@pytest.mark.parametrize("fisher", [True, False])
@pytest.mark.parametrize("missing", [False, True])
def test_all_kept_is_plain_path(path, fisher, missing):
    (ts, _, _) = data(3, 70, 203, 0, 1)
    ts[1, 5] = np.float32(4.0)                        # zero variance: r = 0, or NaN with missing
    ts_dev = _dev.upload(ts, np.float32)
    plain = _dev.download(corr.correlations_device(ts_dev, fisher=fisher, missing=missing))
    got = gpu(ts, np.ones((3, 203), bool), None, fisher, missing)
    same_bits(got, plain)
    assert np.isnan(got).any() == missing


# ------------------------------------------------------------------ 2. censored samples are never read
@pytest.mark.parametrize("K", [0, 3])
def test_censored_samples_are_never_read(path, K):
    (ts, keep, g) = data(3, 66, 150, K, 2)
    keep[:, 7] = False
    ref = gpu(ts, keep, g if K else None, missing=True)
    assert not np.isnan(ref).any()
    bad = ts.copy()
    cens = ~keep
    junk = np.array([np.nan, np.inf, -np.inf, 1e30], dtype=np.float32)
    idx = np.argwhere(np.broadcast_to(cens[:, None, :], ts.shape))
    bad[tuple(idx.T)] = junk[np.arange(len(idx)) % 4]
    bad[:, :, 7] = np.nan                             # a frame NaN in every region
    gb = None
    if K:
        gb = g.copy()
        gb[cens] = np.nan
    for missing in (False, True):
        got = gpu(bad, keep, gb, missing=missing)
        same_bits(got, ref)
        assert not np.isnan(got).any()


# ------------------------------------------------------------------ 3. ragged lengths
@pytest.mark.parametrize("K", [0, 4])
def test_ragged_subject_bits(path, K):
    (ts, keep, g) = data(3, 64, 400, K, 3, lengths=[400, 233, 310])
    conf = g if K else None
    batch = gpu(ts, keep, conf)
    for s in range(3):
        Ts = int(np.nonzero(keep[s])[0].max()) + 1
        alone = gpu(ts[s:s + 1, :, :Ts], keep[s:s + 1, :Ts], None if conf is None else conf[s:s + 1, :Ts])
        same_bits(alone[:, 0], batch[:, s])
    # the same subject followed by 37 extra censored frames holding junk (a longer scan cut by the mask)
    s = 1
    T2 = ts.shape[2] + 37
    ts2 = np.full((1, ts.shape[1], T2), np.nan, np.float32)
    ts2[0, :, :ts.shape[2]] = ts[s]
    ts2[0, :, ts.shape[2]::2] = 1e30
    keep2 = np.zeros((1, T2), bool)
    keep2[0, :ts.shape[2]] = keep[s]
    g2 = None
    if K:
        g2 = np.full((1, T2, K), 3.0)
        g2[0, :ts.shape[2]] = g[s]
    same_bits(gpu(ts2, keep2, g2)[:, 0], batch[:, s])


def test_ragged_lists_through_correlations(path):
    rng = np.random.RandomState(5)
    subjects = [rng.standard_normal((64, T)).astype(np.float32) for T in (120, 97, 150)]
    masks = [rng.rand(T) > 0.15 for T in (120, 97, 150)]
    conf = [rng.standard_normal((T, 2)) for T in (120, 97, 150)]
    got = corr.correlations(subjects, fisher=False, sample_mask=masks, confounds=conf)
    (p, keep, c) = corr.pack_clean(subjects, masks, conf)
    exp = OC.corr_clean(p, keep.astype(bool), c, fisher=False)
    assert np.abs(got - exp).max() <= (TC_DELTA if path == "tc" else SIMT_CLEAN)


# ------------------------------------------------------------------ 4. against the fp64 oracle
@pytest.mark.parametrize("S,N,T,K,lengths", [
    (3, 63, 240, 6, [240, 200, 170]),
    (3, 64, 240, 1, [190, 240, 211]),
    (5, 64, 256, 24, None),
    (3, 64, 250, 64, [250, 230, 249]),
    (3, 400, 1200, 24, [1200, 1150, 1199]),
])
def test_vs_oracle(path, S, N, T, K, lengths):
    rng = np.random.RandomState(S * N + K)
    (ts, keep, g) = data(S, N, T, K, S + N + T + K, censor=0.0, lengths=lengths)
    for s in range(S):                                            # 10 - 50 % censored per subject
        keep[s] &= rng.rand(T) >= (0.1 if T > 1000 else rng.uniform(0.1, 0.5))
    rank = torch.zeros(S, dtype=torch.int32, device=_dev.device())
    got = gpu(ts, keep, g, fisher=False, rank=rank)
    assert rank.cpu().tolist() == [K] * S
    exp = OC.corr_clean(ts, keep, g, fisher=False)
    nkept = int(keep.sum(axis=1).max())
    tol = SIMT_CLEAN if path == "simt" else (TC_DELTA if nkept <= 256 else TC_LONG)
    d = float(np.abs(got - exp).max())
    print("clean K1 %s S=%d N=%d T=%d K=%d kept<=%d: max |dr| = %.3e (tolerance %.1e)" % (
        path, S, N, T, K, nkept, d, tol))
    assert d <= tol
    # Fisher z is the epilogue of the same Gram entries
    z = gpu(ts, keep, g, fisher=True)
    assert np.all(np.isfinite(z))
    assert np.abs(np.tanh(z) - got).max() <= 1e-6


# ------------------------------------------------------------------ 5. rank deficiency
def test_rank_deficient_confounds(path, monkeypatch):
    (S, N, T, K) = (3, 64, 200, 5)
    (ts, keep, g) = data(S, N, T, K, 6)
    keep[:, 11] = False
    extra = np.stack([g[:, :, 2], np.full((S, T), 0.37), np.eye(T)[11][None].repeat(S, 0)], axis=2)
    full = np.concatenate([g[:, :, :2], extra[:, :, :1], g[:, :, 2:], extra[:, :, 1:]], axis=2)   # K + 3
    zeroed = full.copy()
    zeroed[:, :, [2, K + 1, K + 2]] = 0.0
    rank = torch.zeros(S, dtype=torch.int32, device=_dev.device())
    a = gpu(ts, keep, full, rank=rank)
    assert rank.cpu().tolist() == [K] * S
    rank.zero_()
    b = gpu(ts, keep, zeroed, rank=rank)
    assert rank.cpu().tolist() == [K] * S
    same_bits(a, b)
    c = gpu(ts, keep, g, fisher=False)
    a_r = gpu(ts, keep, full, fisher=False)
    assert np.abs(a_r - c).max() <= (SIMT_DELTA if path == "simt" else TC_DELTA)


# ------------------------------------------------------------------ 6. spike regressor == censoring
def test_spike_regressor_is_censoring(monkeypatch):
    simt(monkeypatch)
    (S, N, T, K) = (2, 64, 180, 3)
    (ts, keep, g) = data(S, N, T, K, 7, censor=0.0)
    spikes = [0, 17, 95, 179]
    gs = np.concatenate([g, np.eye(T)[spikes].T[None].repeat(S, 0)], axis=2)
    a = gpu(ts, keep, gs, fisher=False)
    kc = keep.copy()
    kc[:, spikes] = False
    b = gpu(ts, kc, g, fisher=False)
    d = float(np.abs(a - b).max())
    print("spike vs censoring: max |dr| = %.3e" % d)
    assert d <= SIMT_DELTA


# ------------------------------------------------------------------ 7. missing marks with masks
@pytest.mark.parametrize("K", [0, 2])
def test_missing_marks(path, K):
    (S, N, T) = (2, 64, 160)
    (ts, keep, g) = data(S, N, T, max(K, 1), 8)
    keep[:, [5, 6]] = True
    keep[:, [20, 21]] = False
    keep[0, 30] = True
    ts[0, 3, 30] = np.nan                                     # non-finite on a kept frame
    ts[1, 9] = np.float32(1.5)
    ts[1, 9, [20, 21]] = [4.0, -3.0]                          # constant over the kept frames only
    flagged = {(0, 3), (1, 9)}
    conf = g[:, :, :K] if K else None
    if K:
        ts[1, 12] = g[1, :, 1].astype(np.float32)              # explained by a confound
        flagged.add((1, 12))
    a = gpu(ts, keep, conf, missing=True)
    b = gpu(ts, keep, conf, missing=False)
    (n, m) = O.edge_pairs(N)
    for s in range(S):
        rows = [r for (ss, r) in flagged if ss == s]
        bad = np.isin(n, rows) | np.isin(m, rows)
        assert np.isnan(a[bad, s]).all() and not np.isnan(a[~bad, s]).any()
        assert (b[bad, s] == 0).all()
        same_bits(a[~bad, s], b[~bad, s])


# ------------------------------------------------------------------ 8. layout
@pytest.mark.parametrize("s0,extra", [(0, 0), (1, 2), (2, 3), (3, 1)])
def test_layout_columns(path, s0, extra):
    (S, N, T, K) = (3, 64, 130, 2)
    (ts, keep, g) = data(S, N, T, K, 9)
    C = N * (N - 1) // 2
    pitch = s0 + S + extra
    out = torch.full((C, pitch), SENTINEL, dtype=torch.int64, device=_dev.device()).view(torch.float64)
    got = gpu(ts, keep, g, out=out, s0=s0)
    ref = gpu(ts, keep, g)
    same_bits(got[:, s0:s0 + S], ref)
    others = np.r_[0:s0, s0 + S:pitch]
    assert (np.ascontiguousarray(got[:, others]).view(np.int64) == SENTINEL).all()
