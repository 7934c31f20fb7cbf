"""GPU: every stage of the Philox sampler (K5, csrc/fcd_sample.cu) through the C-ABI against its NumPy
restatement (oracle/philox.py).  R, T, F and F~ are compared bit for bit; the normals of B and B~ against a
long-double evaluation under the error bound of the device's fp64 math (derived in `normal_bound`).  Every
output buffer has guard bytes on both sides that must keep their pattern."""
import ctypes

import numpy as np
import numpy.testing as nptest
import pytest
import torch

from oracle import philox as P

pytestmark = pytest.mark.gpu

import fcdiff_b200 as fcdiff            # noqa: E402
from fcdiff_b200 import _dev, _lib      # noqa: E402

GUARD = 64                              # bytes of guard pattern before and after every output
PATTERN = 0xA5
DEFAULT = dict(pi=0.05, eta=0.3, gamma=[0.1, 0.8, 0.1], epsilon=0.03, mu=[-0.15, 0.0, 0.3],
               sigma=[0.025, 0.035, 0.05])
SEED = 0xC0FFEE1234ABCDEF               # both key words non-zero
OFFSET = 0x00A5A5A5DEADBEEF             # offset bits 32..55 set (c3 = offset >> 32 << 8 | var)


class Out:
    """Device output of `shape` framed by guard bytes."""

    def __init__(self, shape, dtype):
        self.shape, self.dtype = shape, dtype
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self.buf = torch.full((self.nbytes + 2 * GUARD,), PATTERN, dtype=torch.uint8, device=_dev.device())

    def ptr(self):
        return ctypes.c_void_p(self.buf.data_ptr() + GUARD)

    def get(self):
        h = _dev.download(self.buf)
        assert np.all(h[:GUARD] == PATTERN) and np.all(h[GUARD + self.nbytes:] == PATTERN), "write outside the output"
        return h[GUARD:GUARD + self.nbytes].view(self.dtype).reshape(self.shape)


def u8(a):
    """Device copy of an input; the caller keeps it alive until the launch (a freed block is reused by the
    next upload)."""
    return _dev.upload(np.asarray(a), np.uint8)


def call(name, *args):
    _lib.check(getattr(_lib.load(), name)(*args, _dev.stream()), name)


def gpu_R(seed, offset, N, U, pi):
    o = Out((N, U), np.uint8)
    call("fcd_sample_R", seed, offset, N, U, float(pi), o.ptr())
    return o.get()


def gpu_T(seed, offset, r, eta, c0, C):
    (N, U) = r.shape
    (o, rd) = (Out((C, U), np.uint8), u8(r))
    call("fcd_sample_T", seed, offset, _dev.ptr(rd), N, U, float(eta), c0, C, o.ptr())
    return o.get()


def gpu_F(seed, offset, c0, C, gamma):
    o = Out((C, 3), np.uint8)
    call("fcd_sample_F", seed, offset, c0, C, _lib.d3(gamma), o.ptr())
    return o.get()


def gpu_F_tilde(seed, offset, f, t, c0, epsilon):
    (C, U) = t.shape
    (o, fd, td) = (Out((C, U, 3), np.uint8), u8(f), u8(t))
    call("fcd_sample_F_tilde", seed, offset, _dev.ptr(fd), _dev.ptr(td), c0, C, U, float(epsilon), o.ptr())
    return o.get()


def gpu_B(seed, offset, f, c0, H, mu, sigma):
    (o, fd) = (Out((len(f), H), np.float64), u8(f))
    call("fcd_sample_B", seed, offset, _dev.ptr(fd), c0, len(f), H, _lib.d3(mu), _lib.d3(sigma), o.ptr())
    return o.get()


def gpu_B_tilde(seed, offset, ft, c0, mu, sigma):
    (C, U) = ft.shape[:2]
    (o, ftd) = (Out((C, U), np.float64), u8(ft))
    call("fcd_sample_B_tilde", seed, offset, _dev.ptr(ftd), c0, C, U, _lib.d3(mu), _lib.d3(sigma), o.ptr())
    return o.get()


def normal_bound(b_ref, mu_abs, sz):
    """Bound on |b_gpu - b| for b = clip(mu + sigma z), z = sqrt(-2 log u1) cospi(2 u2), in float64 on the
    device.  CUDA documents log at 1 ulp (relative 2^-52) and cospi at 2 ulp (2^-51); sqrt, the product and
    fma round correctly (2^-53 each).  sqrt halves the log's relative error, so
        |z_gpu - z| <= (2^-53 + 2^-53 + 2^-51 + 2^-53) |z| = 3.5 * 2^-52 |z|,
    and the fma adds one rounding of |mu + sigma z_gpu| <= |mu| + |sigma z|.  Clipping is 1-Lipschitz.  The
    long-double reference contributes ~2^-63 |sigma z| (2^-60 covers it)."""
    del b_ref
    sz = np.abs(sz)
    return (3.5 * 2.0 ** -52 + 2.0 ** -60) * sz + 2.0 ** -53 * (1 + 2.0 ** -50) * (mu_abs + sz)


def mu_scale(mu, k):
    return np.abs(np.asarray(mu, dtype=np.float64))[k].astype(np.longdouble)


def check_normals(name, got, ref, sz, k, mu):
    """got: float64 device values; ref, sz: long-double clipped value and sigma z of the restatement."""
    assert got.dtype == np.float64 and got.shape == ref.shape
    assert np.all(np.abs(got) <= 1.0)
    err = np.abs(got.astype(np.longdouble) - ref)
    bound = normal_bound(ref, mu_scale(mu, k), sz)
    nz = err > 0                                        # (a zero bound, b = 0 exactly, needs a zero error)
    worst = float(np.max(err[nz] / bound[nz], initial=0.0))
    # in ulps of the fma's operand scale |mu| + |sigma z| (b itself may be a cancellation residue)
    scale = np.asarray(mu_scale(mu, k) + np.abs(sz), dtype=np.float64)
    in_ulp = float(np.max(err[nz] / np.spacing(scale[nz]), initial=0.0))
    print("%s: max |db| = %.2f ulp of |mu| + |sigma z|, %.3f of the bound (%d values)" % (name, in_ulp, worst, got.size))
    assert worst <= 1.0, "%s: %.3f of the fp64 error bound" % (name, worst)


def all_stages(seed, offset, N, H, U, th, c0=0, C=None):
    """Runs every stage on an edge shard and compares it with the restatement; returns the device draws."""
    if C is None:
        C = N * (N - 1) // 2 - c0
    r = gpu_R(seed, offset, N, U, th["pi"])
    nptest.assert_array_equal(r, P.sample_R(seed, offset, N, U, th["pi"]), err_msg="R")
    t = gpu_T(seed, offset, r, th["eta"], c0, C)
    nptest.assert_array_equal(t, P.sample_T(seed, offset, r, th["eta"], c0, C), err_msg="T")
    f = gpu_F(seed, offset, c0, C, th["gamma"])
    nptest.assert_array_equal(f, P.sample_F(seed, offset, c0, C, th["gamma"]), err_msg="F")
    ft = gpu_F_tilde(seed, offset, f, t, c0, th["epsilon"])
    nptest.assert_array_equal(ft, P.sample_F_tilde(seed, offset, f, t, c0, th["epsilon"]), err_msg="F~")
    b = gpu_B(seed, offset, f, c0, H, th["mu"], th["sigma"])
    (b_ref, sz) = P.sample_B(seed, offset, f, c0, H, th["mu"], th["sigma"], exact=True)
    check_normals("b", b, b_ref, sz, np.broadcast_to(P.onehot_state(f)[:, None], b.shape), th["mu"])
    bt = gpu_B_tilde(seed, offset, ft, c0, th["mu"], th["sigma"])
    (bt_ref, szt) = P.sample_B_tilde(seed, offset, ft, c0, th["mu"], th["sigma"], exact=True)
    check_normals("b~", bt, bt_ref, szt, P.onehot_state(ft), th["mu"])
    return (r, t, f, ft, b, bt)


def test_long_double_reference_available():
    assert np.finfo(np.longdouble).nmant >= 63, "the normals' reference needs an extended long double"


@pytest.mark.parametrize("N,H,U", [(2, 1, 1), (37, 9, 5), (400, 10, 3)])
def test_stages_exact_default_theta(N, H, U):
    """N = 2 / U = 1: one edge, one patient.  400 x 10: 798 000 normals of B, more than one pass of the
    grid-stride loop (16 blocks of 256 threads per SM)."""
    all_stages(SEED, OFFSET, N, H, U, DEFAULT)


@pytest.mark.parametrize("seed,offset", [(0, 0), (0xFFFFFFFFFFFFFFFF, 0x00FFFFFFFFFFFFFF), (1 << 32, 1 << 32),
                                         (0x00000001FFFFFFFF, 0x0000000100000000 | 0x12345)])
def test_stages_exact_keys(seed, offset):
    all_stages(seed, offset, 23, 4, 6, dict(DEFAULT, pi=0.4, eta=0.5, epsilon=0.3))


@pytest.mark.parametrize("pi,eta,epsilon,gamma", [(0.0, 0.0, 0.0, [1.0, 0.0, 0.0]),
                                                  (1.0, 1.0, 1.0, [0.0, 0.0, 1.0]),
                                                  (0.5, 0.0, 1.0, [0.0, 1.0, 0.0]),
                                                  (0.5, 1.0, 0.0, [0.5, 0.0, 0.5]),
                                                  (0.5, 0.5, 0.5, [0.0, 0.3, 0.7])])
def test_stages_exact_probability_edges(pi, eta, epsilon, gamma):
    th = dict(DEFAULT, pi=pi, eta=eta, epsilon=epsilon, gamma=gamma)
    (r, t, f, ft, _, _) = all_stages(SEED, OFFSET, 30, 3, 40, th)
    if pi in (0.0, 1.0):
        assert np.all(r == pi)
    if epsilon == 0.0:                                  # t = 0 keeps the template state, t = 1 never does
        keep = np.all(ft == f[:, None, :], axis=2)
        assert np.all(keep[t == 0]) and not np.any(keep[t == 1])
    for k in range(3):
        if gamma[k] == 0.0:
            assert not np.any(f[:, k])


@pytest.mark.parametrize("N,c0,C", [(50, 0, 1), (50, 3, 17), (50, 1000, 225), (50, 1224, 1), (200, 777, 5000)])
def test_ragged_edge_shards(N, c0, C):
    """Edge shards [c0, c0 + C) of any length, ending at C_total or not: the counter is the global edge."""
    all_stages(SEED ^ 0x5555, OFFSET, N, 5, 7, dict(DEFAULT, pi=0.3), c0=c0, C=C)


def test_element_indices_beyond_32_bits():
    """Counters with a non-zero high word (c1 = idx >> 32) through edge shards far from 0."""
    th = dict(DEFAULT, eta=0.45, epsilon=0.2, sigma=[0.5, 0.035, 0.3])
    rng = np.random.RandomState(8)
    # F: c0 >= 2^32 and a shard straddling 2^32
    for c0 in (2 ** 32 + 3, 2 ** 32 - 1000, 3 * 2 ** 32 + 12345):
        nptest.assert_array_equal(gpu_F(SEED, OFFSET, c0, 4096, th["gamma"]),
                                  P.sample_F(SEED, OFFSET, c0, 4096, th["gamma"]))
    # T, F~, B~ at the last edges of N = 65535, U = 3: element index c*U + u ~ 6.4e9
    (N, U, C) = (65535, 3, 3000)
    c0 = N * (N - 1) // 2 - C
    assert c0 * U >= 2 ** 32
    r = (rng.uniform(size=(N, U)) < 0.5).astype(np.uint8)
    t = gpu_T(SEED, OFFSET, r, th["eta"], c0, C)
    t_ref = P.sample_T(SEED, OFFSET, r, th["eta"], c0, C)
    nptest.assert_array_equal(t, t_ref)
    (n, m) = P.c_to_nm(c0 + np.arange(C))
    assert n.max() == N - 1 and np.any(r[n] != r[m])
    f = P.onehot(rng.randint(0, 3, C))
    ft = gpu_F_tilde(SEED, OFFSET, f, t, c0, th["epsilon"])
    nptest.assert_array_equal(ft, P.sample_F_tilde(SEED, OFFSET, f, t, c0, th["epsilon"]))
    bt = gpu_B_tilde(SEED, OFFSET, ft, c0, th["mu"], th["sigma"])
    (bt_ref, sz) = P.sample_B_tilde(SEED, OFFSET, ft, c0, th["mu"], th["sigma"], exact=True)
    check_normals("b~", bt, bt_ref, sz, P.onehot_state(ft), th["mu"])
    # B: (c0 + cl) * H + h beyond 2^33
    (c0, H) = (2 ** 31 + 17, 5)
    b = gpu_B(SEED, OFFSET, f, c0, H, th["mu"], th["sigma"])
    (b_ref, sz) = P.sample_B(SEED, OFFSET, f, c0, H, th["mu"], th["sigma"], exact=True)
    check_normals("b", b, b_ref, sz, np.broadcast_to(P.onehot_state(f)[:, None], b.shape), th["mu"])


def test_non_onehot_states_and_clipping():
    """States that are not one-hot are read as `onehot_state` does (f[1], else f[2], else 0; any non-zero
    byte counts); sigma large enough to clip at both ends, and sigma = 0 (b = mu exactly)."""
    rng = np.random.RandomState(4)
    (C, U, H) = (600, 9, 7)
    mu, sigma = [-0.4, 0.9, 0.25], [3.0, 0.0, 1.5]
    f = rng.choice(np.array([0, 1, 2, 255], dtype=np.uint8), size=(C, 3))
    ft = rng.choice(np.array([0, 1, 3], dtype=np.uint8), size=(C, U, 3))
    t = rng.choice(np.array([0, 1, 9], dtype=np.uint8), size=(C, U))
    for c0 in (0, 5000):
        ftd = gpu_F_tilde(SEED, OFFSET, f, t, c0, 0.35)
        nptest.assert_array_equal(ftd, P.sample_F_tilde(SEED, OFFSET, f, t, c0, 0.35))
        b = gpu_B(SEED, OFFSET, f, c0, H, mu, sigma)
        (b_ref, sz) = P.sample_B(SEED, OFFSET, f, c0, H, mu, sigma, exact=True)
        k = np.broadcast_to(P.onehot_state(f)[:, None], b.shape)
        check_normals("b", b, b_ref, sz, k, mu)
        bt = gpu_B_tilde(SEED, OFFSET, ft, c0, mu, sigma)
        (bt_ref, szt) = P.sample_B_tilde(SEED, OFFSET, ft, c0, mu, sigma, exact=True)
        check_normals("b~", bt, bt_ref, szt, P.onehot_state(ft), mu)
        for (x, kk) in ((b, k), (bt, P.onehot_state(ft))):
            assert np.all(x[kk == 1] == 0.9)
            assert np.any(x[kk == 0] == -1.0) and np.any(x[kk == 0] == 1.0)
            assert np.any(x[kk == 2] == -1.0) and np.any(x[kk == 2] == 1.0)


@pytest.mark.parametrize("seed", [0, 77])
def test_public_sample_equals_restatement(seed):
    """`UnsharedRegionModel.sample` with a seeded `rng`: the key is `_next_key`'s four randint draws, and
    successive calls take successive keys."""
    model = fcdiff.UnsharedRegionModel()
    model.rng = np.random.RandomState(seed)
    model.pi, model.eta, model.epsilon = 0.2, 0.4, 0.1
    rs = np.random.RandomState(seed)
    th = dict(pi=model.pi, eta=model.eta, gamma=model.gamma, epsilon=model.epsilon, mu=model.mu,
              sigma=model.sigma)
    (N, H, U) = (19, 6, 11)
    for _ in range(2):
        got = model.sample(N, H, U)
        (key, off) = P.next_key(rs)
        ref = P.sample(key, off, N, H, U, exact=True, **th)
        for (g, e, name) in zip(got[:4], ref[:4], ("r", "t", "f", "f~")):
            assert g.dtype == np.bool_
            nptest.assert_array_equal(g, e != 0, err_msg=name)
        k = np.broadcast_to(P.onehot_state(ref[2])[:, None], got[4].shape)
        check_normals("b", got[4], ref[4][0], ref[4][1], k, model.mu)
        check_normals("b~", got[5], ref[5][0], ref[5][1], P.onehot_state(ref[3]), model.mu)

