"""GPU: the correlation stage (K1, csrc/fcd_corr.cu, csrc/fcd_corr_tc.cu) at its edges.

* long series (concatenated runs, T = 2400 / 4800) against numpy.corrcoef in fp64;
* Fisher z checked in z-space, without tanh: z must lie in atanh([r - delta, r + delta] clipped to the
  path's saturation limit), widened by the rounding of the epilogue -- strongly correlated rows up to |r| ~ 1,
  exact and negated duplicates, square waves whose Gram entry is exactly -1 (z = the saturation value) and
  constant rows (exactly 0);
* the output layout: columns [s0, s0 + S) of a (C, pitch) matrix, odd / even s0 and pitch, an 8- but not
  16-byte aligned pointer; every other column keeps its bits;
* batch invariance: a subject's column has the same bits alone, first or second of a pair, at even or odd
  s0 (16-byte or scalar stores) and in a repeated call;
* isolation of non-finite samples, including the first rows of subject s + 1 that the tail tile of subject
  s reads as padding;
* agreement of the tensor-core path, the SIMT path (fp64 accumulation) and full tiles (FCD_CORR_NO_TAIL).
Both paths are selected per call through FCD_CORR_SIMT, which fcd_corr_fisherz reads on every call."""
import ctypes

import numpy as np
import numpy.testing as nptest
import pytest
import torch

from oracle import iar_oracle as O

pytestmark = pytest.mark.gpu

from fcdiff_b200 import _dev, _lib, corr       # noqa: E402

SENTINEL = 0x7FF4DEADBEEF0001                   # a signalling-NaN bit pattern no kernel writes
LIM32 = float(np.float32(1 - 2.0 ** -24))       # saturation of the tensor-core path (fp32 epilogue)
LIM64 = 1 - 2.0 ** -53                          # saturation of the SIMT path (fp64 epilogue)
TC_DELTA = 2e-6                                 # |dr| of the tensor-core path at T <= 256, |r| < 0.99
TC_DELTA_SAT = 4e-6                             # ... at T = 256 on common-factor rows (3.1e-6 measured on a B200)
SIMT_DELTA = 2.0 ** -23 + 1e-12                 # fp32 rounding of both standardised rows: 2 * 2^-24 sum|z w|
LONG_T_TOL = {2400: 6e-6, 4800: 1.2e-5}         # 1.5 x the |dr| measured on a B200 (DESIGN.md 4)


def use_path(mp, path):
    mp.delenv("FCD_CORR_SIMT", raising=False)
    mp.delenv("FCD_CORR_NO_TAIL", raising=False)
    if path == "simt":
        mp.setenv("FCD_CORR_SIMT", "1")
    elif path == "notail":
        mp.setenv("FCD_CORR_NO_TAIL", "1")


def mixed(S, N, T, seed, scale=0.4):
    rng = np.random.RandomState(seed)
    mix = rng.standard_normal((N, N)) * scale + np.eye(N)
    ts = np.einsum("nm,smt->snt", mix, rng.standard_normal((S, N, T))).astype(np.float32)
    ts += rng.uniform(-50, 50, (S, N, 1)).astype(np.float32)
    return ts


def sentinel_out(C, pitch):
    return torch.full((C, pitch), SENTINEL, dtype=torch.int64, device=_dev.device()).view(torch.float64)


def bits(a):
    return np.ascontiguousarray(a).view(np.int64)


def gpu_corr(ts, fisher=True, missing=False):
    return _dev.download(corr.correlations_device(_dev.upload(ts, np.float32), fisher=fisher, missing=missing))


# ------------------------------------------------------------------ long series
@pytest.mark.parametrize("T", [2400, 4800])
def test_long_series_vs_fp64(T):
    """Schaefer-400 with two / four concatenated 1200-TR runs: K = T / 8 fp32 accumulations per MMA chain."""
    (S, N) = (4, 400)
    ts = mixed(S, N, T, T, scale=0.2)
    got = gpu_corr(ts, fisher=False)
    exp = O.corr_fisherz(ts, fisher=False)
    d = float(np.abs(got - exp).max())
    print("K1 T=%d: max |dr| = %.3e (tolerance %.1e)" % (T, d, LONG_T_TOL[T]))
    assert d <= LONG_T_TOL[T]


# ------------------------------------------------------------------ Fisher z in z-space
def strong_series(S, N, T, seed):
    """Rows 0..N/2: a common factor plus noise of amplitude 1e-7 .. 3 (|r| from ~0.1 to 1 - 1e-14, both
    signs, large means); an exact duplicate, a negated duplicate, a negated duplicate of the duplicate, two
    constant rows; two square waves (+-c, T = 256: the standardised samples are +-1/16, exact in TF32, so
    the Gram entry of the pair is exactly +-1 on both paths); the rest mixed."""
    rng = np.random.RandomState(seed)
    ts = mixed(S, N, T, seed + 1).astype(np.float64)
    k = N // 2
    f = rng.standard_normal((S, 1, T))
    amp = np.logspace(-7, 0.5, k)[None, :, None]
    sign = np.where(np.arange(k) % 3 == 2, -1.0, 1.0)[None, :, None]
    ts[:, :k] = sign * f + amp * rng.standard_normal((S, k, T)) + rng.uniform(-20, 20, (S, k, 1))
    ts = ts.astype(np.float32)
    ts[:, k] = ts[:, 1]
    ts[:, k + 1] = -ts[:, 1]
    ts[:, k + 2] = -ts[:, k]
    ts[:, k + 3] = np.float32(3.7)
    ts[:, k + 4] = np.float32(0.0)
    wave = np.where(rng.permutation(T) % 2 == 0, 1.0, -1.0)
    ts[:, k + 5] = 2.5 * wave + 4.0
    ts[:, k + 6] = -0.75 * wave
    return ts, [k + 3, k + 4]


def z_contract(z, r_ref, path):
    """Checks z against atanh([r_ref - delta, r_ref + delta] n [-lim, lim]) widened by the epilogue's
    rounding; returns the largest excursion beyond the unwidened interval in units of 2^-23 |z| (tensor
    cores: fp32 log1pf, 1 ulp each, and one fp32 rounding -> 1.5 * 2^-23 relative) or 2^-52 |z| (SIMT:
    fp64 atanh, 2 ulp)."""
    (lim, delta, unit, allowed) = ((LIM32, TC_DELTA_SAT, 2.0 ** -23, 2.0) if path != "simt"
                                   else (LIM64, SIMT_DELTA, 2.0 ** -52, 2.0))
    r = r_ref.astype(np.longdouble)
    lo = np.arctanh(np.clip(r - delta, -lim, lim))
    hi = np.arctanh(np.clip(r + delta, -lim, lim))
    zl = z.astype(np.longdouble)
    out = np.maximum(np.maximum(lo - zl, zl - hi), 0) / (unit * np.maximum(np.abs(zl), 1e-300))
    worst = float(out.max()) if out.size else 0.0
    assert np.all(np.isfinite(z))
    assert worst <= allowed, "z outside its interval by %.2f x %g |z|" % (worst, unit)
    return worst


@pytest.mark.parametrize("path", ["tc", "simt"])
@pytest.mark.parametrize("N", [63, 96, 241])
def test_fisher_z_space_contract(monkeypatch, path, N):
    if path == "tc" and N < 64:
        pytest.skip("N < 64 always takes the SIMT path")
    use_path(monkeypatch, path)
    (S, T) = (3, 256)
    (ts, const) = strong_series(S, N, T, N)
    z = gpu_corr(ts, fisher=True)
    r = gpu_corr(ts, fisher=False)
    (n, m) = O.edge_pairs(N)
    is_const = np.isin(n, const) | np.isin(m, const)
    lim = LIM32 if path == "tc" else LIM64
    zsat = np.arctanh(np.longdouble(lim))
    k = N // 2
    (worst, dr) = (0.0, 0.0)
    for s in range(S):
        with np.errstate(invalid="ignore", divide="ignore"):
            rr = np.corrcoef(ts[s].astype(np.float64))[n, m]
        assert np.all(bits(z[is_const, s]) == 0) and np.all(bits(r[is_const, s]) == 0)    # +0.0 exactly
        worst = max(worst, z_contract(z[~is_const, s], rr[~is_const], path))
        dr = max(dr, float(np.abs(r[~is_const, s] - rr[~is_const]).max()))
        assert np.abs(z[:, s]).max() <= zsat * (1 + 2.0 ** -22)
        # duplicates and negated duplicates: r_ref = +-1, z within [atanh(1 - delta), atanh(lim)] of its sign
        for (a, b, sgn) in ((k, 1, 1), (k + 1, 1, -1), (k + 2, k, -1), (k + 2, 1, -1), (k + 2, k + 1, 1)):
            assert sgn * z[a * (a - 1) // 2 + b, s] > 6.0
        # the square waves: r = -1 exactly on both paths, so z is the saturation value itself
        c = (k + 6) * (k + 5) // 2 + k + 5
        assert r[c, s] == -1.0
        nptest.assert_allclose(z[c, s], -float(zsat), rtol=2.0 ** -22 if path == "tc" else 2.0 ** -51)
    print("K1 z-space %s N=%d: max |dr| %.3e, largest excursion %.3f units (allowed 2)" % (path, N, dr, worst))
    # the fp32 epilogue saturates at 1 - 2^-24 (|z| <= 8.67), the fp64 one at 1 - 2^-53 (|z| <= 18.7)
    assert np.abs(z).max() <= (8.67 if path == "tc" else 18.72)


# ------------------------------------------------------------------ output layout
def with_bad_rows(ts):
    ts = ts.copy()
    ts[1, 4] = np.float32(2.5)                  # constant row
    ts[2, 7, 3] = np.nan                        # non-finite sample
    ts[3, 0, 0] = np.inf
    return ts


@pytest.mark.parametrize("path", ["tc", "simt"])
@pytest.mark.parametrize("s0,pitch", [(1, 8), (2, 7), (3, 10), (2, 9), (1, 5)])
def test_output_layout_columns(monkeypatch, path, s0, pitch):
    """correlations_device(out=..., s0=...) + fcd_corr_mark_missing write exactly columns [s0, s0 + S), with
    the bits of the default (C, S) layout; all other columns keep the sentinel."""
    use_path(monkeypatch, path)
    (S, N, T) = (4, 200, 64)
    ts = with_bad_rows(mixed(S, N, T, 5))
    ts_dev = _dev.upload(ts, np.float32)
    C = N * (N - 1) // 2
    ref = _dev.download(corr.correlations_device(ts_dev, missing=True))
    out = sentinel_out(C, pitch)
    corr.correlations_device(ts_dev, out=out, s0=s0, missing=True)
    got = bits(_dev.download(out))
    assert np.all(got[:, :s0] == SENTINEL) and np.all(got[:, s0 + S:] == SENTINEL)
    nptest.assert_array_equal(got[:, s0:s0 + S], bits(ref))
    assert np.isnan(ref[:, 1]).sum() == N - 1 and np.isnan(ref[:, 2]).sum() == N - 1


@pytest.mark.parametrize("path", ["tc", "simt"])
def test_output_pointer_8_byte_aligned(monkeypatch, path):
    """An out pointer one double past a 16-byte boundary, even pitch and s0: the tensor-core epilogue must
    take the scalar stores.  (correlations_device takes the pitch from out.shape[1], so the C-ABI is called
    directly.)"""
    use_path(monkeypatch, path)
    lib = _lib.load()
    (S, N, T, s0, pitch) = (4, 241, 64, 2, 8)
    ts = with_bad_rows(mixed(S, N, T, 6))
    ts_dev = _dev.upload(ts, np.float32)
    C = N * (N - 1) // 2
    ref = _dev.download(corr.correlations_device(ts_dev, missing=True))
    buf = sentinel_out(C * pitch + 2, 1).view(-1)
    assert buf.data_ptr() % 16 == 0
    ptr = ctypes.c_void_p(buf.data_ptr() + 8)
    zws = torch.empty(lib.fcd_corr_workspace_bytes(S, N, T), dtype=torch.uint8, device=ts_dev.device)
    _lib.check(lib.fcd_corr_fisherz(_dev.ptr(ts_dev), S, N, T, ptr, pitch, s0, 1, _dev.ptr(zws), _dev.stream()),
               "fcd_corr_fisherz")
    _lib.check(lib.fcd_corr_mark_missing(_dev.ptr(ts_dev), S, N, T, ptr, pitch, s0, _dev.stream()),
               "fcd_corr_mark_missing")
    got = bits(_dev.download(buf))
    assert got[0] == SENTINEL and got[-1] == SENTINEL
    mat = got[1:1 + C * pitch].reshape(C, pitch)
    assert np.all(mat[:, :s0] == SENTINEL) and np.all(mat[:, s0 + S:] == SENTINEL)
    nptest.assert_array_equal(mat[:, s0:s0 + S], bits(ref))


# ------------------------------------------------------------------ batch invariance
@pytest.mark.parametrize("path", ["tc", "simt", "notail"])
@pytest.mark.parametrize("N", [64, 200, 241])
def test_subject_column_batch_invariant(monkeypatch, path, N):
    """Per subject, the column is a function of that subject's rows only: alone, first or second of a
    pair, a lone last subject, even s0 (16-byte stores of a pair) or odd (scalar stores), repeated."""
    use_path(monkeypatch, path)
    (S, T) = (5, 96)
    ts = mixed(S, N, T, N + 11)
    ts_dev = _dev.upload(ts, np.float32)
    C = N * (N - 1) // 2
    alone = np.stack([_dev.download(corr.correlations_device(_dev.upload(ts[s:s + 1], np.float32)))[:, 0]
                      for s in range(S)], axis=1)
    runs = {"batch": _dev.download(corr.correlations_device(ts_dev)),
            "repeat": _dev.download(corr.correlations_device(ts_dev))}
    for s0 in (1, 2):
        out = sentinel_out(C, s0 + S + 1)
        corr.correlations_device(ts_dev, out=out, s0=s0)
        runs["s0=%d" % s0] = _dev.download(out)[:, s0:s0 + S]
    rev = _dev.download(corr.correlations_device(_dev.upload(ts[::-1].copy(), np.float32)))
    runs["reversed"] = rev[:, ::-1]
    for (name, got) in runs.items():
        nptest.assert_array_equal(bits(got), bits(alone), err_msg=name)


# ------------------------------------------------------------------ isolation of non-finite samples
@pytest.mark.parametrize("missing", [False, True])
@pytest.mark.parametrize("path", ["tc", "simt", "notail"])
@pytest.mark.parametrize("N,bad", [(200, 1), (241, 2), (255, 3)])
def test_nonfinite_samples_stay_in_their_region(monkeypatch, missing, path, N, bad):
    """NaN / +-Inf samples in subject `bad`, in its first rows (rows that the tail tiles of subject bad - 1
    load as padding: 128 - tail rows of the full-width box, 1 at N = 255, 15 at 241; 8 of the transposed
    box at N = 200) and in its last: no bit of another subject changes; in
    subject `bad` only the edges of those regions change, to the negative clip (missing=False) or NaN."""
    use_path(monkeypatch, path)
    (S, T) = (4, 64)
    ts = mixed(S, N, T, N + bad)
    badrows = [0, 2, 5, 7, N - 1]
    dirty = ts.copy()
    dirty[bad, 0, 3] = np.nan
    dirty[bad, 2, :] = np.nan
    dirty[bad, 5, 10] = np.inf
    dirty[bad, 7, 0] = -np.inf
    dirty[bad, N - 1, T - 1] = np.nan
    clean = gpu_corr(ts, missing=missing)
    got = gpu_corr(dirty, missing=missing)
    others = [s for s in range(S) if s != bad]
    nptest.assert_array_equal(bits(got[:, others]), bits(clean[:, others]))
    (n, m) = O.edge_pairs(N)
    touched = np.isin(n, badrows) | np.isin(m, badrows)
    nptest.assert_array_equal(bits(got[~touched, bad]), bits(clean[~touched, bad]))
    v = got[touched, bad]
    if missing:
        assert np.all(np.isnan(v))
    else:
        assert np.all(bits(v) == bits(v[:1]))
        zlim = np.arctanh(LIM64 if path == "simt" else LIM32)
        nptest.assert_allclose(v[0], -zlim, rtol=2.0 ** -21)


# ------------------------------------------------------------------ path agreement
@pytest.mark.parametrize("N", [64, 200, 241, 400])
def test_tensor_core_simt_and_full_tiles_agree(monkeypatch, N):
    (S, T) = (3, 128)
    ts = mixed(S, N, T, N + 3)
    res = {}
    for path in ("tc", "simt", "notail"):
        use_path(monkeypatch, path)
        res[path] = gpu_corr(ts, fisher=False)
    exp = O.corr_fisherz(ts, fisher=False)
    nptest.assert_allclose(res["simt"], exp, rtol=0, atol=SIMT_DELTA)
    for path in ("tc", "notail"):
        nptest.assert_allclose(res[path], res["simt"], rtol=0, atol=TC_DELTA)
    same = bool(np.array_equal(bits(res["tc"]), bits(res["notail"])))
    ndiff = int((bits(res["tc"]) != bits(res["notail"])).sum())
    print("K1 N=%d: transposed tail tiles %s the full-tile form (%d values differ, max |d| %.2e)"
          % (N, "equal" if same else "differ from", ndiff, np.abs(res["tc"] - res["notail"]).max()))

