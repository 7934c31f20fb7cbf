"""GPU: the K3b code pass (dominant-state plane, code bytes, records), the evaluator over it, the
small-vector exchange and the patient gather staging -- each through the C-ABI against NumPy."""
import ctypes

import numpy as np
import numpy.testing as nptest
import pytest
import torch

from oracle import iar_oracle as O

pytestmark = pytest.mark.gpu

import fcdiff_b200 as fcdiff            # noqa: E402
from fcdiff_b200 import _dev, _lib      # noqa: E402
from fcdiff_b200 import util            # noqa: E402


def _pair_code(sn, sm):
    """code of an element from the two regions' peak states (csrc/fcd_streams.cu:pair_code):
    0..2 pair state of two decided regions, 4 + s one undecided normalised region (state 2) beside a
    region in state s, 3 anything else."""
    o = sn | sm
    if o < 2:
        return ((sn ^ sm) << 1) + (sn & sm)
    if sn == 2 and sm < 2:
        return 4 + sm
    if sm == 2 and sn < 2:
        return 4 + sn
    return 3


@pytest.mark.parametrize("N,U", [(9, 7), (23, 130), (40, 300)])
def test_code_plane_evaluator_and_estep_match_numpy(N, U):
    lib = _lib.load()
    rng = np.random.RandomState(N * 1000 + U)
    C = N * (N - 1) // 2
    pitchU = U + (U & 1)
    pitchS = (U + 255) // 256 * 256
    pitchQ = int(lib.fcd_code_pitch(U))
    assert pitchQ % 16 == 0 and pitchU <= pitchQ <= pitchS
    P = rng.dirichlet([1.0, 1.0, 1.0], size=(C, pitchU)).transpose(2, 0, 1).copy()      # [3][C][pitchU]
    L = rng.randn(C, pitchU)
    fstate = rng.choice([0, 1, 2, 3], size=C, p=[0.3, 0.3, 0.3, 0.1]).astype(np.uint8)
    rstate = np.full((N, pitchS), 4, np.uint8)
    rstate[:, :U] = rng.choice([0, 1, 2, 3], size=(N, U), p=[0.55, 0.25, 0.15, 0.05])
    # posteriors consistent with the states (peaked rows are exactly one-hot)
    qF = np.zeros((C, 3))
    for c in range(C):
        qF[c] = rng.dirichlet([2.0, 2.0, 2.0]) if fstate[c] == 3 else np.eye(3)[fstate[c]]
    qR = np.zeros((N, U, 2))
    for n in range(N):
        for u in range(U):
            s = rstate[n, u]
            if s == 2:
                qR[n, u] = rng.dirichlet([2.0, 2.0])                    # undecided, normalised
            elif s == 3:
                qR[n, u] = rng.dirichlet([2.0, 2.0]) * 1.25             # undecided, not normalised ("loose")
            else:
                qR[n, u] = np.eye(2)[s]
    nm = np.array([(util.c_to_nm(c)[0] | (util.c_to_nm(c)[1] << 16)) for c in range(C)], dtype=np.int32)

    d = {k: _dev.upload(v) for (k, v) in dict(P=P, L=L, qF=qF.reshape(-1), qR=qR.reshape(-1)).items()}
    fs = torch.from_numpy(fstate).cuda()
    rs = torch.from_numpy(rstate).cuda()
    nmd = torch.from_numpy(nm).cuda()
    PsE = _dev.zeros((C, pitchQ))
    kc = torch.full((C,), 255, dtype=torch.uint8, device="cuda")
    code = _dev.empty((C * pitchQ + 256,), torch.uint8)
    counts = _dev.empty((C, 2), torch.int32)
    offs = _dev.empty((4 * int(lib.fcd_bucket_blocks(C)),), torch.int64)
    tot = _dev.zeros((2,))
    # the peak states the library derives from these posteriors are the ones drawn above
    rs_lib = _dev.empty((N, pitchS), torch.uint8)
    _lib.check(lib.fcd_peak_states_R(_dev.ptr(d['qR']), N, U, pitchS, _dev.ptr(rs_lib), _dev.stream()), "fcd_peak_states_R")
    nptest.assert_array_equal(rs_lib.cpu().numpy(), rstate)
    st = _dev.stream()
    _lib.check(lib.fcd_code_plane(_dev.ptr(d['P']), C * pitchU, C, U, pitchU, _dev.ptr(fs), _dev.ptr(rs), pitchS,
                                  _dev.ptr(nmd), _dev.ptr(PsE), _dev.ptr(kc), _dev.ptr(code), pitchQ, _dev.ptr(counts),
                                  _dev.ptr(offs), _dev.ptr(tot), st), "fcd_code_plane")
    # ---- NumPy restatement of the code pass
    want_code = np.full((C, pitchQ), 3, np.uint8)
    want_cnt = np.zeros((C, 2), np.int64)
    for c in range(C):
        (n, m) = util.c_to_nm(c)
        if fstate[c] == 3:
            want_cnt[c, 0] = 3 * U
            continue
        for u in range(U):
            want_code[c, u] = _pair_code(int(rstate[n, u]), int(rstate[m, u]))
        want_cnt[c] = (int((want_code[c, :U] == 3).sum()), int((want_code[c, :U] >= 4).sum()))
    got_code = code[:C * pitchQ].cpu().numpy().reshape(C, pitchQ)
    nptest.assert_array_equal(got_code, want_code)
    nptest.assert_array_equal(counts.cpu().numpy(), want_cnt)
    (nd, nh) = (int(v) for v in tot.cpu().numpy())
    assert (nd, nh) == tuple(want_cnt.sum(axis=0)) and nh > 0
    got_PsE = PsE.cpu().numpy()
    for c in range(C):
        if fstate[c] < 3:
            nptest.assert_array_equal(got_PsE[c, :pitchU], P[fstate[c], c])
            assert not got_PsE[c, pitchU:].any()
    nptest.assert_array_equal(kc.cpu().numpy()[fstate < 3], fstate[fstate < 3])

    # ---- records + evaluation against the plain triple sum (fit.py:489-511, 600-697)
    Lsum = _dev.zeros((1,))
    ws = _dev.workspace()
    _lib.check(lib.fcd_plane_sum(_dev.ptr(d['L']), C, U, pitchU, _dev.ptr(Lsum), _dev.ptr(ws), st), "fcd_plane_sum")
    nptest.assert_allclose(Lsum.cpu().numpy()[0], L[:, :U].sum(), rtol=1e-12, atol=1e-9)
    D = _dev.empty((4 * max(nd, 1),))
    K = _dev.empty((max(nd, 1),), torch.int64)
    KH = _dev.empty((max(nh, 1),), torch.int64)
    Hh = _dev.empty((2 * max(nh, 1),))
    RO = _dev.empty((C, 2), torch.int64)
    out = _dev.zeros((4,))
    _lib.check(lib.fcd_code_records(_dev.ptr(d['P']), C * pitchU, _dev.ptr(PsE), _dev.ptr(code), pitchQ, _dev.ptr(d['L']),
                                    _dev.ptr(Lsum), C, U, pitchU, _dev.ptr(d['qF']), _dev.ptr(fs), _dev.ptr(d['qR']),
                                    _dev.ptr(rs), pitchS, N, _dev.ptr(nmd), _dev.ptr(counts), _dev.ptr(offs), _dev.ptr(K),
                                    _dev.ptr(KH), _dev.ptr(RO), _dev.ptr(D), nd, _dev.ptr(Hh), nh,
                                    _dev.ptr(out[3:]), _dev.ptr(ws), st), "fcd_code_records")
    # half records: {p of the dominant state, +-q_s of the undecided region}, in row order
    keysH = KH.cpu().numpy()[:nh].astype(np.uint64)
    half = Hh.cpu().numpy()[:2 * nh].reshape(nh, 2)
    for i in range(0, nh, max(1, nh // 50)):
        (u, c, sx) = (int(keysH[i] & np.uint64(0xffff)), int((keysH[i] >> np.uint64(16)) & np.uint64(0xffffffff)), int(keysH[i] >> np.uint64(48)))
        (n, m) = util.c_to_nm(c)
        who = n if rstate[n, u] == 2 else m
        assert want_code[c, u] == 4 + sx and half[i, 0] == P[fstate[c], c, u]
        assert abs(half[i, 1]) == qR[who, u, sx] and bool(np.signbit(half[i, 1])) == bool(sx)
    (eta, eps) = (0.37, 0.12)
    th = _lib.make_theta(0.1, eta, eps, [0.2, 0.5, 0.3], [-0.1, 0.0, 0.1], [0.1, 0.1, 0.1])
    _lib.check(lib.fcd_elm_coded(_dev.ptr(PsE), _dev.ptr(code), C * pitchQ, _dev.ptr(D), nd, _dev.ptr(Hh), nh, ctypes.byref(th), 1,
                                 _dev.ptr(out), _dev.ptr(ws), st), "fcd_elm_coded")
    got = out.cpu().numpy()
    epsl = np.array([1 - eps, eps, eta * eps + (1 - eta) * (1 - eps)])
    (al, bl) = ((1 - epsl) / 2, epsl - (1 - epsl) / 2)
    sl = np.array([-1.0, 1.0, 2 * eta - 1])
    (obj, const, ge, gh) = (0.0, 0.0, 0.0, 0.0)
    for c in range(C):
        (n, m) = util.c_to_nm(c)
        for u in range(U):
            (qn, qm) = (qR[n, u], qR[m, u])
            w = np.array([qn[0] * qm[0], qn[1] * qm[1], qn[0] * qm[1] + qn[1] * qm[0]])
            const += qF[c].sum() * w.sum() * L[c, u]
            for k in range(3):
                p = P[k, c, u]
                M = al + bl * p
                obj += qF[c, k] * (w * np.log(M)).sum()
                dd = qF[c, k] * w * (1.5 * p - 0.5) / M
                ge += (sl * dd).sum()
                gh += dd[2]
    scale = max(1.0, abs(obj))
    nptest.assert_allclose(got[0], obj, rtol=1e-11, atol=1e-11 * scale)
    nptest.assert_allclose(got[3], const, rtol=1e-11, atol=1e-10)
    nptest.assert_allclose(got[1], -(2 * eps - 1) * gh, rtol=0, atol=1e-10 * scale)
    nptest.assert_allclose(got[2], -ge, rtol=0, atol=1e-10 * scale)

    # ---- the E-step driven by the same code plane / key lists (fit.py:157-174)
    H = 6
    (S1, S2) = (rng.randn(C), np.abs(rng.randn(C)) + 1.0)
    (lqF_c, qF_c) = (_dev.zeros((C * 3,)), _dev.zeros((C * 3,)))
    (S1d, S2d) = (_dev.upload(S1), _dev.upload(S2))
    _lib.check(lib.fcd_estep_qF_coded(_dev.ptr(S1d), _dev.ptr(S2d), None, H, _dev.ptr(d['P']), C * pitchU, C, U,
                                      pitchU, _dev.ptr(d['qR']), N, _dev.ptr(nmd), _dev.ptr(code), pitchQ,
                                      _dev.ptr(counts), _dev.ptr(K), _dev.ptr(KH), _dev.ptr(RO), _dev.ptr(Hh),
                                      ctypes.byref(th), None, 0.0, 0.0, _dev.ptr(lqF_c), _dev.ptr(qF_c), st),
               "fcd_estep_qF_coded")
    (lqF_p, qF_p) = (_dev.zeros((C * 3,)), _dev.zeros((C * 3,)))
    _lib.check(lib.fcd_estep_qF(_dev.ptr(S1d), _dev.ptr(S2d), None, H, _dev.ptr(d['P']), C * pitchU, C, U, pitchU,
                                _dev.ptr(d['qR']), _dev.ptr(rs), pitchS, N, _dev.ptr(nmd), ctypes.byref(th),
                                _dev.ptr(lqF_p), _dev.ptr(qF_p), st), "fcd_estep_qF")
    # NumPy: lqF[c,k] = log gamma_k + healthy_k + sum_u sum_l w_l log(a_l + b_l p_k) - logsumexp_k  (L cancels)
    mu = np.array([-0.1, 0.0, 0.1]); sg = np.array([0.1, 0.1, 0.1]); gam = np.array([0.2, 0.5, 0.3])
    want = np.zeros((C, 3))
    for c in range(C):
        (n, m) = util.c_to_nm(c)
        l = np.log(gam) - (S2[c] - 2 * mu * S1[c] + H * mu ** 2) / (2 * sg ** 2) - H * (np.log(sg) + 0.5 * np.log(2 * np.pi))
        for u in range(U):
            (qn, qm) = (qR[n, u], qR[m, u])
            w = np.array([qn[0] * qm[0], qn[1] * qm[1], qn[0] * qm[1] + qn[1] * qm[0]])
            p3 = np.array([P[0, c, u], P[1, c, u], 1.0 - P[0, c, u] - P[1, c, u]])
            for k in range(3):
                l[k] += (w * np.log(al + bl * p3[k])).sum()
        want[c] = l - (l.max() + np.log(np.exp(l - l.max()).sum()))
    nptest.assert_allclose(lqF_c.cpu().numpy().reshape(C, 3), want, rtol=1e-10, atol=1e-9)
    nptest.assert_allclose(lqF_p.cpu().numpy().reshape(C, 3), want, rtol=1e-10, atol=1e-9)
    nptest.assert_allclose(qF_c.cpu().numpy(), np.exp(lqF_c.cpu().numpy()), rtol=1e-12, atol=1e-300)


def test_small_exchange_world1_publishes_to_the_host():
    from fcdiff_b200.dist import PeerWindow
    pw = PeerWindow()
    st = _dev.stream()
    for n in (1, 4, 8):
        x = np.random.RandomState(n).randn(n)
        v = _dev.upload(x)
        for _ in range(3):                      # consecutive exchanges reuse the window and the result slot
            nptest.assert_array_equal(pw.allreduce(v, n, st), x)
    pw.close()


@pytest.mark.parametrize("N,U,world", [(5, 7, 2), (12, 500, 8), (3, 3, 4)])
def test_patient_gather_staging_roundtrip(N, U, world):
    lib = _lib.load()
    rng = np.random.RandomState(U)
    (a, b) = (rng.randn(N, U, 2), rng.randn(N, U, 2))
    ch = (U + world - 1) // world
    st = _dev.stream()
    gathered = _dev.empty((world, 2 * N * ch * 2))
    (ad, bd) = (_dev.upload(a.reshape(-1)), _dev.upload(b.reshape(-1)))
    for r in range(world):
        u0 = min(r * ch, U)
        Ul = min(ch, U - u0)
        _lib.check(lib.fcd_pack_patients(_dev.ptr(ad), _dev.ptr(bd), N, U, u0, Ul, ch, _dev.ptr(gathered[r]), st),
                   "fcd_pack_patients")
    (oa, ob) = (_dev.zeros((N * U * 2,)), _dev.zeros((N * U * 2,)))
    _lib.check(lib.fcd_unpack_patients(_dev.ptr(gathered), world, N, U, ch, _dev.ptr(oa), _dev.ptr(ob), st),
               "fcd_unpack_patients")
    nptest.assert_array_equal(oa.cpu().numpy().reshape(N, U, 2), a)
    nptest.assert_array_equal(ob.cpu().numpy().reshape(N, U, 2), b)


@pytest.mark.parametrize("N,U,lookup,scale",
                         [(37, 5, 0, 0.05),                 # N < 64: one region per step
                          # blocked forward substitution (N >= 64): 256 threads below 700 regions, 512 from 700 on
                          (600, 3, 0, 0.05), (600, 2, 1, 0.05), (1100, 2, 0, 0.05), (1400, 2, 1, 0.05),
                          (2100, 1, 0, 0.05),
                          # more than 2 x SMs patients: 128 threads up to 512 regions, 256 above
                          (100, 300, 1, 0.05), (530, 300, 0, 0.05),
                          # whole / ragged last blocks, both lookups, shared memory beyond 48 KB
                          (64, 9, 0, 0.05), (65, 4, 1, 0.05), (96, 3, 0, 0.05), (100, 3, 1, 0.05), (400, 6, 0, 0.05),
                          (400, 5, 1, 0.05), (3300, 1, 1, 0.05),
                          # large weights: most regions come out decided (|l_0 - l_1| > 37.5, the short form of
                          # the in-block step), a few do not
                          (37, 5, 0, 2.0), (100, 3, 1, 2.0), (400, 6, 0, 2.0), (400, 5, 1, 2.0), (1100, 2, 0, 1.0),
                          (600, 2, 1, 0.5),
                          # from 700 regions on and with few patients two CTAs of a cluster share a patient
                          # (partial sums and solved blocks travel through distributed shared memory)
                          (800, 3, 1, 0.5), (715, 2, 0, 0.02)])
def test_sweep_launch_shapes_match_numpy(N, U, lookup, scale):
    """Gauss-Seidel sweep of fit.py:184-197 over the two weight differences, for every launch shape of
    fcd_estep_qR (the kernel and its threads per patient depend on N and on the number of patients), both edge
    lookups."""
    lib = _lib.load()
    rng = np.random.RandomState(N + U)
    C = N * (N - 1) // 2
    WT = scale * rng.randn(U, C + 1, 2)                      # {W_0 - W_2, W_2 - W_1}; one edge of slack (fit.py:186 quirk)
    q = rng.dirichlet([1.0, 1.0], size=(N, U))
    lp = np.log(np.array([0.7, 0.3]))
    WTd = _dev.upload(WT[:, :C].copy().reshape(-1))
    (qd, lqd) = (_dev.upload(q.reshape(-1)), _dev.zeros((N * U * 2,)))
    _lib.check(lib.fcd_estep_qR(_dev.ptr(WTd), C, N, U, 0, U, _lib.d3(lp), lookup, _dev.ptr(qd), _dev.ptr(lqd),
                                _dev.stream()), "fcd_estep_qR")
    want_q = q.copy()
    want_lq = np.zeros((N, U, 2))
    for u in range(U):
        for n in range(N):
            base = n * (n - 1) // 2
            m = np.arange(N)
            if lookup == 0:
                c = base + m                                  # nm_to_c(n, m) for every m != n (SURVEY 0.3)
            else:
                c = np.where(m < n, base + m, m * (m - 1) // 2 + n)
            keep = (m != n) & (c < C)
            D = (lp[0] - lp[1]) + (want_q[keep, u, 0] * WT[u, c[keep], 0] + want_q[keep, u, 1] * WT[u, c[keep], 1]).sum()
            l = np.array([0.0, -D])
            l -= l.max() + np.log(np.exp(l - l.max()).sum())
            want_lq[n, u] = l
            want_q[n, u] = np.exp(l)
    nptest.assert_allclose(lqd.cpu().numpy().reshape(N, U, 2), want_lq, rtol=1e-9, atol=1e-11)
    nptest.assert_allclose(qd.cpu().numpy().reshape(N, U, 2), want_q, rtol=1e-9, atol=1e-13)
