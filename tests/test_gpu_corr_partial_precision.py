"""GPU: partial correlations (fcd_corr_partial, csrc/fcd_corr_partial.cu) against the longdouble reference
(oracle/partial.py: subject_partial_ld), where the numerics are hard.

The standard (oracle/partial.py: accuracy), per subject: err_gpu = max |r_gpu - r_ld| and err_np =
max |r_np - r_ld| (r_np: the fp64 oracle, numpy.linalg.inv) over the edges of usable regions;
err_gpu <= F_R * max(err_np, 4 * 2^-53), and delta the same with F_DELTA.  Every case prints kappa_2(Sigma),
err_gpu, err_np and their ratio.

Cases: N across the 64-pivot sweep blocks and 64-wide tiles, T above and below N, Ledoit-Wolf and delta = 0;
a conditioning ladder to kappa ~ 1e10 (small delta, n_s just above N + K, nearly collinear regions); the
pivot test (a subject whose smallest reference pivot is >= 4 * 2^-40 comes back finite, one whose smallest
pivot is <= 2^-40 / 4 is flagged, in the first, a middle and the last block); unusable regions on block
boundaries and down to no usable region; K up to 64 confounds (every fp64 clean_kernel instantiation),
rank-deficient and nearly collinear confounds; long series (clean_kernel from 8 warps down to 1, and the T
where none fits) and short ones; the reversed region order; the batch split the workspace budget makes."""
import numpy as np
import pytest
import torch

from oracle import iar_oracle as O
from oracle import partial as OP

pytestmark = pytest.mark.gpu

from fcdiff_b200 import _dev, _lib, corr      # noqa: E402

PIVOT_TOL = 2.0 ** -40                        # kPivotTol
SENTINEL = 0x7FF4DEADBEEF0001


def series(S, N, T, K=0, seed=0, censor=0.0, offset=50.0, load=0.5):
    """Planted 8-factor series (the K1 workload's structure), confound components of loading ~``load`` and a
    per-region offset; keep (S, T) and g (S, T, K) or None."""
    rng = np.random.RandomState(seed)
    a = np.where(rng.rand(N) < 0.5, 0.55, -0.27)
    f = rng.standard_normal((S, 8, T))
    ts = np.sqrt(1 - a * a)[None, :, None] * rng.standard_normal((S, N, T)) + a[None, :, None] * f[:, np.arange(N) % 8]
    g = rng.standard_normal((S, T, K))
    ts += np.einsum("nk,stk->snt", load * rng.standard_normal((N, K)), g) + rng.uniform(-offset, offset, (S, N, 1))
    keep = rng.rand(S, T) >= censor
    return ts.astype(np.float32), keep, (g if K else None)


def collinear(ts, s, j, srcs, eps, seed):
    """Region j of subject s := a combination of regions srcs + eps * noise (in fp64, then rounded)."""
    rng = np.random.RandomState(seed)
    x = ts[s].astype(np.float64)
    x = x - x.mean(axis=1, keepdims=True)
    v = sum(c * x[i] / x[i].std() for (c, i) in zip((1.0, -0.5, 0.75), srcs))
    ts[s, j] = (v + eps * rng.standard_normal(ts.shape[2])).astype(np.float32)


def gpu(ts, keep=None, g=None, shrinkage="ledoit-wolf", missing=False, rank=None):
    S = ts.shape[0]
    delta = _dev.empty((S,))
    o = corr.correlations_device(_dev.upload(ts, np.float32), fisher=False, missing=missing, rank=rank,
                                 sample_mask=None if keep is None else _dev.upload(keep, np.bool_),
                                 confounds=None if g is None else _dev.upload(g, np.float64), kind="partial",
                                 shrinkage=shrinkage, shrinkage_out=delta)
    return _dev.download(o), _dev.download(delta)


def cabi(ts, keep, g, shrinkage):
    """Through the C-ABI with a workspace of exactly fcd_corr_partial_workspace_bytes: (out, delta, status)."""
    (S, N, T) = ts.shape
    K = 0 if g is None else g.shape[2]
    lib = _lib.load()
    out = _dev.empty((N * (N - 1) // 2, S))
    delta = _dev.empty((S,))
    status = torch.full((S,), -1, dtype=torch.int32, device="cuda")
    zws = torch.empty(lib.fcd_corr_partial_workspace_bytes(S, N, T, K), dtype=torch.uint8, device="cuda")
    (ts_d, keep_d) = (_dev.upload(ts, np.float32), None if keep is None else _dev.upload(keep, np.uint8))
    g_d = None if g is None else _dev.upload(g, np.float64)
    _lib.check(lib.fcd_corr_partial(_dev.ptr(ts_d), S, N, T, _dev.ptr(keep_d), _dev.ptr(g_d), K, shrinkage,
                                    _dev.ptr(out), S, 0, 0, 0, None, _dev.ptr(delta), _dev.ptr(status),
                                    _dev.ptr(zws), _dev.stream()), "fcd_corr_partial")
    return _dev.download(out), _dev.download(delta), status.cpu().numpy()


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    eq = (a.view(np.int64) == b.view(np.int64)) | ((a == 0) & (b == 0))
    assert eq.all(), "%d entries differ, max |d| = %g" % ((~eq).sum(), np.nanmax(np.abs(a - b)))


def oracle_shrinkage(shrinkage):
    return None if shrinkage == "ledoit-wolf" else shrinkage


def refs(ts, keep, g, shrinkage):
    sh = oracle_shrinkage(shrinkage)
    return [OP.references(ts[s], np.ones(ts.shape[2], bool) if keep is None else keep[s],
                          None if g is None else g[s], sh) for s in range(ts.shape[0])]


def meets_standard(col, delta, ref, what, fixed=False):
    """The standard for one subject that must come back (smallest reference pivot >= 4 * 2^-40); returns
    the accuracy record.  Edges of an unusable region must be exactly 0 (missing=False)."""
    assert ref["min_piv"] >= 4 * PIVOT_TOL, "%s: reference pivot %.3g is not a passing case" % (what, ref["min_piv"])
    assert (ref["bad"] == ref["bad64"]).all()
    N = ref["bad"].shape[0]
    (n, m) = O.edge_pairs(N)
    off = ref["bad"][n] | ref["bad"][m]
    assert (col[off] == 0).all()
    a = OP.accuracy(col, delta, ref)
    print("%-34s kappa %8.2e  err_gpu %8.2e  err_np %8.2e  ratio %6.2f  min pivot %8.2e  delta %.3g "
          "(err_gpu %.2g, err_np %.2g, ratio %.2f)" % (what, a["kappa"], a["err_gpu"], a["err_np"], a["ratio"],
                                                        ref["min_piv"], delta, a["derr_gpu"], a["derr_np"],
                                                        a["dratio"]))
    assert a["ratio"] <= OP.F_R, what
    if fixed:
        assert delta == ref["delta64"]
    else:
        assert a["dratio"] <= OP.F_DELTA, what
    return a


def run(ts, keep, g, shrinkage, what):
    """Every subject of a case against both references; all must be passing cases."""
    rs = refs(ts, keep, g, shrinkage)
    (got, delta) = gpu(ts, keep, g, shrinkage)
    return [meets_standard(got[:, s], delta[s], rs[s], "%s s%d" % (what, s), shrinkage != "ledoit-wolf")
            for s in range(ts.shape[0])]


# ------------------------------------------------------------------ sweep blocks and Gram tiles
EDGE_N = [63, 64, 65, 127, 128, 129, 191, 192, 193, 257]
EDGE_CASES = [(N, T, sh) for N in EDGE_N for (T, sh) in ((N + N // 2, "ledoit-wolf"), (N + 3, 0.0),
                                                          (2 * N // 3, "ledoit-wolf"))]
EDGE_CASES += [(1131, 1200, 0.0), (1131, 700, "ledoit-wolf")]


@pytest.mark.parametrize("N,T,shrinkage", EDGE_CASES,
                         ids=["N%d-T%d-%s" % (N, T, "lw" if sh == "ledoit-wolf" else "d0") for (N, T, sh) in EDGE_CASES])
def test_block_and_tile_edges(N, T, shrinkage):
    S = 1 if N > 1000 else 2
    (ts, keep, _) = series(S, N, T, seed=N + T, censor=0.0 if shrinkage == 0.0 else 0.1)
    run(ts, keep, None, shrinkage, "edges N=%d T=%d %s" % (N, T, shrinkage))


# ------------------------------------------------------------------ conditioning ladder
LADDER = [("lw-2N", "ledoit-wolf", 2, None), ("d1e-2", 1e-2, 1, None), ("d1e-5", 1e-5, 1, None),
          ("d1e-8", 1e-8, 1, None), ("d0-N+1", 0.0, 1, None), ("d0-5N/4", 0.0, 1.25, None), ("d0-2N", 0.0, 2, None),
          ("col1e-3", 0.0, 2, 1e-3), ("col3e-5", 0.0, 2, 3e-5), ("col3e-5-lw", "ledoit-wolf", 2, 3e-5)]


@pytest.mark.parametrize("N", [65, 200, 400])
def test_conditioning_ladder(N):
    kappas = []
    for (name, shrinkage, f, eps) in LADDER:
        T = N + 1 if f == 1 else int(f * N)                # n_s = N + K + 1 (K = 0) .. 2N
        (ts, keep, _) = series(1, N, T, seed=N + T, offset=1.0)
        if eps is not None:                                 # a region nearly a combination of three others
            collinear(ts, 0, N // 2 + 1, (3, N // 3, N // 2 - 5), eps, N)
        a = run(ts, None, None, shrinkage, "ladder N=%d %s" % (N, name))
        kappas.append(a[0]["kappa"])
    print("ladder N=%d: kappa %.2e .. %.2e" % (N, min(kappas), max(kappas)))
    assert min(kappas) < 1e2 and max(kappas) > 1e9


# ------------------------------------------------------------------ the pivot test
PIVOT_N = 193                                  # blocks [0, 64) [64, 128) [128, 192) [192]
PIVOT_AT = {10: (3, 7, 1), 100: (20, 70, 90), 192: (64, 150, 5)}


@pytest.mark.parametrize("j", sorted(PIVOT_AT), ids=["first-block", "middle-block", "last-pivot"])
def test_pivot_threshold(j):
    (S, N, T) = (3, PIVOT_N, 400)
    (ts, _, _) = series(S, N, T, seed=j, offset=1.0)
    for (s, eps) in ((0, 1e-5), (1, 3e-8), (2, 6e-6)):      # passing, failing, passing
        collinear(ts, s, j, PIVOT_AT[j], eps, 10 * j + s)
    rs = refs(ts, None, None, 0.0)
    for s in range(S):
        piv = rs[s]["piv"].astype(np.float64)
        print("pivot at %d: subject %d smallest pivot %.3g at %d" % (j, s, rs[s]["min_piv"], np.nanargmin(piv)))
        assert np.nanargmin(piv) == j
    assert rs[0]["min_piv"] >= 4 * PIVOT_TOL and rs[2]["min_piv"] >= 4 * PIVOT_TOL
    assert rs[1]["min_piv"] <= PIVOT_TOL / 4
    with pytest.raises(ValueError, match=r"subject\(s\) \[1\]"):
        corr.correlations(ts, kind="partial", shrinkage=0.0)
    (got, delta, status) = cabi(ts, None, None, 0.0)
    assert status.tolist() == [0, 1, 0]
    assert np.isnan(got[:, 1]).all()
    for s in (0, 2):
        meets_standard(got[:, s], delta[s], rs[s], "pivot at %d s%d" % (j, s), fixed=True)
        (one, d1) = gpu(ts[s:s + 1], shrinkage=0.0)
        same_bits(got[:, s], one[:, 0])
        same_bits(delta[s], d1[0])


# ------------------------------------------------------------------ unusable regions
def spoil(ts, g, s, regions, keep):
    """Make regions of subject s unusable, in turn: constant, a non-finite kept sample, explained by a
    confound (when there are confounds)."""
    t_kept = int(np.argmax(keep[s]))
    for (i, r) in enumerate(regions):
        how = i % (3 if g is not None else 2)
        if how == 0:
            ts[s, r] = np.float32(3.25)
        elif how == 1:
            ts[s, r, t_kept] = np.nan
        else:
            ts[s, r] = (2.0 * g[s, :, 0] - 4.0).astype(np.float32)


@pytest.mark.parametrize("what,N,T,K,shrinkage", [
    ("block-edges", 193, 300, 2, "ledoit-wolf"), ("block-edges", 193, 300, 2, 0.0),
    ("half", 130, 260, 1, "ledoit-wolf"), ("half", 130, 260, 1, 0.0)])
def test_unusable_regions(what, N, T, K, shrinkage):
    (ts, keep, g) = series(2, N, T, K, seed=N + K, censor=0.1)
    regions = [0, 63, 64, 127, 128, N - 1] if what == "block-edges" else list(range(1, N, 2))
    spoil(ts, g, 0, regions, keep)
    spoil(ts, g, 1, regions[::-1], keep)
    rs = refs(ts, keep, g, shrinkage)
    for r in rs:
        assert r["bad"].tolist() == [n in regions for n in range(N)]
    (got, delta) = gpu(ts, keep, g, shrinkage)
    (gotm, deltam) = gpu(ts, keep, g, shrinkage, missing=True)
    same_bits(delta, deltam)
    (n, m) = O.edge_pairs(N)
    for s in range(2):
        meets_standard(got[:, s], delta[s], rs[s], "unusable %s N=%d %s s%d" % (what, N, shrinkage, s),
                       shrinkage != "ledoit-wolf")
        off = rs[s]["bad"][n] | rs[s]["bad"][m]
        assert np.isnan(gotm[off, s]).all()
        same_bits(gotm[~off, s], got[~off, s])


def test_two_one_and_no_usable_regions():
    (N, T, K) = (6, 50, 1)
    (ts, keep, g) = series(3, N, T, K, seed=6, censor=0.1)
    ts[0, 1] += 2 * ts[0, 4]                               # a strong partial correlation between the two left
    spoil(ts, g, 0, [0, 2, 3, 5], keep)                    # 2 usable
    spoil(ts, g, 1, [0, 1, 2, 4, 5], keep)                 # 1 usable
    spoil(ts, g, 2, list(range(N)), keep)                  # none
    rs = refs(ts, keep, g, "ledoit-wolf")
    assert [int((~r["bad"]).sum()) for r in rs] == [2, 1, 0]
    (got, delta, status) = cabi(ts, keep, g, -1.0)
    assert status.tolist() == [0, 0, 0]
    (got2, delta2) = gpu(ts, keep, g)
    same_bits(got2, got)
    same_bits(delta2, delta)
    (gotm, _) = gpu(ts, keep, g, missing=True)
    (n, m) = O.edge_pairs(N)
    for s in range(3):
        meets_standard(got[:, s], delta[s], rs[s], "usable %d" % (2 - s))
        off = rs[s]["bad"][n] | rs[s]["bad"][m]
        assert np.isnan(gotm[off, s]).all() and (got[off, s] == 0).all()
    assert 0 < delta[0] < 1 and delta[1] == 0 and delta[2] == 0
    on = ~(rs[0]["bad"][n] | rs[0]["bad"][m])
    assert abs(got[on, 0][0]) > 0.5


# ------------------------------------------------------------------ confounds
@pytest.mark.parametrize("K", [7, 8, 9, 16, 17, 32, 33, 64])
def test_confounds(K):
    (ts, keep, g) = series(1, 65, 400, K, seed=K, censor=0.1)
    for shrinkage in ("ledoit-wolf", 0.0):
        run(ts, keep, g, shrinkage, "confounds K=%d %s" % (K, shrinkage))


def test_rank_deficient_confounds():
    (S, N, T, K) = (2, 65, 300, 9)
    (ts, keep, g) = series(S, N, T, K, seed=3, censor=0.1)
    g[:, :, 3] = g[:, :, 1]                                # duplicate
    g[:, :, 6] = 7.0                                       # constant: the intercept
    g[:, :, 8] = np.where(keep, 0.0, 5.0)                  # zero on every kept frame
    gz = g.copy()
    gz[:, :, [3, 6, 8]] = 0.0
    rank = torch.full((S,), -1, dtype=torch.int32, device="cuda")
    for shrinkage in ("ledoit-wolf", 0.0):
        rs = refs(ts, keep, g, shrinkage)
        (got, delta) = gpu(ts, keep, g, shrinkage, rank=rank)
        assert rank.cpu().tolist() == [K - 3] * S
        (gotz, deltaz) = gpu(ts, keep, gz, shrinkage)
        same_bits(got, gotz)
        same_bits(delta, deltaz)
        for s in range(S):
            meets_standard(got[:, s], delta[s], rs[s], "rank-deficient %s s%d" % (shrinkage, s),
                           shrinkage != "ledoit-wolf")


def test_unshrunk_frame_boundary():
    (N, K) = (65, 8)
    (ts, _, g) = series(1, N, 90, K, seed=5)
    keep = np.zeros((1, 90), bool)
    keep[0, :N + K] = True
    with pytest.raises(ValueError, match="subject 0 keeps %d frames" % (N + K)):
        corr.correlations(ts, kind="partial", shrinkage=0.0, sample_mask=keep, confounds=g)
    keep[0, N + K] = True                                  # n_s = N + K + 1: accepted
    rs = refs(ts, keep, g, 0.0)
    got = corr.correlations(ts, kind="partial", shrinkage=0.0, sample_mask=keep, confounds=g, fisher=False)
    a = meets_standard(got[:, 0], 0.0, rs[0], "n_s = N + K + 1", fixed=True)
    assert a["kappa"] > 1e3


@pytest.mark.parametrize("shrinkage", ["ledoit-wolf", 0.0])
def test_nearly_collinear_confounds(shrinkage):
    (S, N, T, K) = (2, 65, 400, 8)
    (ts, keep, g) = series(S, N, T, K, seed=8, censor=0.1, load=0.0)
    rng = np.random.RandomState(9)
    g[:, :, 1] = g[:, :, 0] + 1e-7 * rng.standard_normal((S, T))
    g[:, :, 5] = g[:, :, 2] - g[:, :, 3] + 1e-6 * rng.standard_normal((S, T))
    # The regions are ~1e4 times more confound than signal.  An error of the projection that stays in the
    # confounds' span moves r only at second order, so it needs this weight to show: a basis that lost
    # orthogonality (one Gram-Schmidt pass: ~eps * cond) leaves ~1e-8 in r, the fp64 oracle ~1e-11.
    ts = (0.1 * ts + np.einsum("nk,stk->snt", 1000.0 * rng.standard_normal((N, K)), g)).astype(np.float32)
    for s in range(S):
        gk = g[s][keep[s]]
        c = np.linalg.cond(np.hstack([np.ones((len(gk), 1)), gk - gk.mean(axis=0)]))
        print("confound condition number, subject %d: %.2e" % (s, c))
        assert 1e6 <= c <= 1e9
    run(ts, keep, g, shrinkage, "collinear confounds %s" % shrinkage)


# ------------------------------------------------------------------ series length
def clean_warps(T, K):
    """clean_kernel's warps per CTA (csrc/fcd_corr_clean.cu), 225 KiB of shared memory."""
    Tp = (T + 31) // 32 * 32
    return min(8, (225 * 1024 - K * 64 * 8) // (Tp * 8))


LONG = [(T, K) for T in (2400, 4800, 12000) for K in (0, 24, 64)] + [(24000, 64)]


@pytest.mark.parametrize("T,K", LONG, ids=["T%d-K%d" % c for c in LONG])
def test_long_series(T, K):
    print("T=%d K=%d: clean_kernel warps %d" % (T, K, clean_warps(T, K)))
    (ts, keep, g) = series(1, 65, T, K, seed=T + K, censor=0.05)
    run(ts, keep, g, "ledoit-wolf", "T=%d K=%d" % (T, K))


def test_long_series_warp_counts_are_covered():
    warps = {clean_warps(T, K) for (T, K) in LONG if K > 0}
    assert {1, 8} <= warps and len(warps) >= 4


def test_series_too_long_for_a_warp_launches_nothing():
    (N, T, K) = (8, 25000, 64)
    assert clean_warps(T, K) == 0
    (ts, keep, g) = series(1, N, T, K, seed=1)
    lib = _lib.load()
    host = np.full((N * (N - 1) // 2, 1), SENTINEL, dtype=np.int64).view(np.float64)
    out = _dev.upload(host, np.float64)
    torch.cuda.synchronize()
    before = lib.fcd_launch_count()
    with pytest.raises(_lib.FcdError, match="T=25000 too long for K=64 confounds"):
        corr.correlations_device(_dev.upload(ts, np.float32), confounds=_dev.upload(g, np.float64), kind="partial",
                                 out=out)
    assert lib.fcd_launch_count() == before
    assert (_dev.download(out).view(np.int64) == SENTINEL).all()


@pytest.mark.parametrize("T", [2, 3, 17])
def test_short_series(T):
    (S, N) = (2, 10)
    (ts, keep, _) = series(S, N, T, seed=T)
    rs = refs(ts, None, None, "ledoit-wolf")
    (got, delta, status) = cabi(ts, None, None, -1.0)
    for s in range(S):
        if T == 2:                       # R has rank 1 and Ledoit-Wolf's b^2 is 0: Sigma = R is singular
            assert rs[s]["min_piv"] <= PIVOT_TOL / 4
            assert status[s] == 1 and np.isnan(got[:, s]).all()
        else:
            assert status[s] == 0
            meets_standard(got[:, s], delta[s], rs[s], "short T=%d s%d" % (T, s))
    if T == 2:
        with pytest.raises(ValueError, match=r"subject\(s\) \[0, 1\]"):
            corr.correlations(ts, kind="partial")


# ------------------------------------------------------------------ permutation
@pytest.mark.parametrize("shrinkage", ["ledoit-wolf", 0.0])
def test_reversed_region_order(shrinkage):
    (N, T) = (193, 260)
    (ts, keep, g) = series(1, N, T, 2, seed=12, censor=0.05)
    (fwd, dfwd) = gpu(ts, keep, g, shrinkage)
    (rev, drev) = gpu(np.ascontiguousarray(ts[:, ::-1]), keep, g, shrinkage)
    (n, m) = O.edge_pairs(N)
    (F, R) = (np.eye(N), np.eye(N))
    F[n, m] = F[m, n] = fwd[:, 0]
    R[n, m] = R[m, n] = rev[:, 0]
    a = meets_standard(fwd[:, 0], dfwd[0], refs(ts, keep, g, shrinkage)[0], "forward order %s" % shrinkage,
                       shrinkage != "ledoit-wolf")
    d = np.abs(R[::-1, ::-1] - F).max()
    print("reversed order %s: max |r_rev - r_fwd| %.2e" % (shrinkage, d))
    assert d <= 2 * OP.F_R * max(a["err_np"], OP.ERR_FLOOR)
    assert abs(drev[0] - dfwd[0]) <= 2 * OP.F_DELTA * max(a["derr_np"], OP.ERR_FLOOR)


# ------------------------------------------------------------------ the natural batch split
def partial_ws_for(B, N, Tp, K):
    """csrc/fcd_corr_partial.cu: partial_ws_for."""
    def pal(b):
        return (b + 1023) & ~1023
    return 1024 + pal(B * N * Tp * 8) + pal(B * N * N * 8) + pal(B * N * 64 * 8) + pal(B * K * Tp * 8) + \
        pal(B * Tp * 8) + pal(B * 8) + pal(B * N)


def test_natural_batch_split():
    (S, N, T) = (81, 1131, 4800)
    B = (4 << 30) // partial_ws_for(1, N, T, 0)
    assert S - 3 < B < S                                  # the last three subjects straddle the split
    lib = _lib.load()
    assert lib.fcd_corr_partial_workspace_bytes(S, N, T, 0) == partial_ws_for(B, N, T, 0)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(81)
    ts = torch.randn((S, N, T), generator=gen, device="cuda", dtype=torch.float32)
    ts += 0.5 * torch.randn((S, 8, T), generator=gen, device="cuda", dtype=torch.float32)[:, torch.arange(N) % 8]
    out = _dev.empty((N * (N - 1) // 2, S))
    delta = _dev.empty((S,))
    status = torch.full((S,), -1, dtype=torch.int32, device="cuda")
    zws = torch.empty(lib.fcd_corr_partial_workspace_bytes(S, N, T, 0), dtype=torch.uint8, device="cuda")
    _lib.check(lib.fcd_corr_partial(_dev.ptr(ts), S, N, T, None, None, 0, -1.0, _dev.ptr(out), S, 0, 1, 0, None,
                                    _dev.ptr(delta), _dev.ptr(status), _dev.ptr(zws), _dev.stream()),
               "fcd_corr_partial")
    assert (status.cpu() == 0).all()
    for s in range(S - 3, S):
        d1 = _dev.empty((1,))
        one = corr.correlations_device(ts[s:s + 1].contiguous(), kind="partial", shrinkage_out=d1)
        same_bits(_dev.download(out[:, s].contiguous()), _dev.download(one[:, 0].contiguous()))
        same_bits(_dev.download(delta[s:s + 1]), _dev.download(d1))
    assert np.isfinite(_dev.download(out[:, :3].contiguous())).all()
