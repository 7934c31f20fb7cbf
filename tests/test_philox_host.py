"""Host: the NumPy restatement of the Philox sampler (oracle/philox.py) against the Random123 known-answer
vectors of Philox4x32-10, a scalar copy of the round function, and the kernels' key / counter packing and
uniform conversion (fcdiff_b200/csrc/fcd_sample.cu).  The GPU side is tests/test_gpu_sampler_exact.py."""
import numpy as np
import numpy.testing as nptest
import pytest

from oracle import philox as P


# Random123 kat_vectors, philox4x32 with 10 rounds: (counter, key, output)
KAT = [((0x00000000, 0x00000000, 0x00000000, 0x00000000), (0x00000000, 0x00000000),
        (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
       ((0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff), (0xffffffff, 0xffffffff),
        (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
       ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
        (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]


def philox_scalar(ctr, key):
    """One block with Python integers, the loop of philox4x32_10 in fcd_sample.cu written out."""
    (c0, c1, c2, c3) = ctr
    (k0, k1) = key
    for _ in range(10):
        (p0, p1) = (0xD2511F53 * c0, 0xCD9E8D57 * c2)
        (c0, c1, c2, c3) = ((p1 >> 32) ^ c1 ^ k0, p1 & 0xFFFFFFFF, (p0 >> 32) ^ c3 ^ k1, p0 & 0xFFFFFFFF)
        (k0, k1) = ((k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF)
    return (c0, c1, c2, c3)


@pytest.mark.parametrize("ctr,key,out", KAT)
def test_known_answers(ctr, key, out):
    assert philox_scalar(ctr, key) == out
    got = P.philox4x32_10(key[0], key[1], *ctr)
    assert tuple(int(v) for v in got) == out
    assert all(v.dtype == np.uint64 for v in got)


def test_vectorised_equals_scalar():
    rng = np.random.RandomState(11)
    words = rng.randint(0, 2 ** 32, size=(6, 200), dtype=np.uint64)
    words[:, :4] = [0, 0xFFFFFFFF, 1, 0x80000000]                   # extreme words in every lane
    got = np.stack(P.philox4x32_10(*words))
    for i in range(words.shape[1]):
        w = [int(v) for v in words[:, i]]
        assert tuple(int(v) for v in got[:, i]) == philox_scalar(w[2:], w[:2])


def test_key_and_counter_packing():
    seed = 0xFEDCBA9876543210
    offset = 0x00ABCDEF01234567                                      # bits 32..55 set: _next_key's range
    for var in range(1, 7):
        assert P.philox_make(seed, offset, var) == (0x76543210, 0xFEDCBA98, 0x01234567, 0xABCDEF00 | var)
    # bits 56..63 of the offset are shifted out of the 32-bit c3, as in the kernel
    assert P.philox_make(seed, offset | (0x5A << 56), 3) == P.philox_make(seed, offset, 3)
    # the element index is the low counter pair: (c0, c1) = (idx low, idx high)
    idx = np.array([0, 1, 2 ** 32 - 1, 2 ** 32, 3 * 2 ** 32 + 7, 2 ** 63 + 5], dtype=np.uint64)
    got = np.stack(P.blocks(seed, offset, 4, idx))
    (k0, k1, c2, c3) = P.philox_make(seed, offset, 4)
    for j, i in enumerate(idx.tolist()):
        assert tuple(int(v) for v in got[:, j]) == philox_scalar((i & 0xFFFFFFFF, i >> 32, c2, c3), (k0, k1))
    # every variable id and every offset word gives another stream
    streams = {tuple(np.stack(P.blocks(seed, o, v, idx[:2])).ravel().tolist())
               for v in range(1, 7) for o in (offset, offset + 1, offset + (1 << 32))}
    assert len(streams) == 18


def test_u01_range_and_resolution():
    m = 0xFFFFFFFF
    assert P.u01(0, 0) == 0.0
    assert P.u01(m, m) == 1.0 - 2.0 ** -53                          # the largest value, below 1
    assert P.u01(0, 1 << 6) == 2.0 ** -53                            # the smallest step
    assert P.u01(1 << 5, 0) == 2.0 ** -27
    assert P.u01(m, 0) == 1.0 - 2.0 ** -27
    # the low 5 bits of a and 6 bits of b are dropped
    assert P.u01(0x1F, 0x3F) == 0.0
    rng = np.random.RandomState(3)
    (a, b) = rng.randint(0, 2 ** 32, size=(2, 100000), dtype=np.uint64)
    u = P.u01(a, b)
    assert u.dtype == np.float64 and u.min() >= 0.0 and u.max() < 1.0
    v = np.array([((int(x) >> 5) << 26) | (int(y) >> 6) for (x, y) in zip(a[:1000], b[:1000])], dtype=np.float64)
    nptest.assert_array_equal(u[:1000] * 2.0 ** 53, v)                # exact


def test_box_muller_reference():
    # u01(x, y) = 0 -> 1 - u = 1 -> z = 0; the cosine's quadrants are exact
    assert P.std_normal_ld((np.uint64(0),) * 4) == 0
    x = np.array([0.0, 0.5, 1.0, 1.5, 0.25, 1.75, 1.0 / 3.0, 1.9])
    c = P.cospi_ld(x)
    nptest.assert_array_equal(c[:4], [1, 0, -1, 0])
    nptest.assert_allclose(c.astype(np.float64), np.cos(np.pi * x), rtol=0, atol=1e-15)
    assert abs(P.PI_LD - np.longdouble(np.pi)) < 2e-16              # pi beyond float64 where long double has it
    rng = np.random.RandomState(5)
    w = rng.randint(0, 2 ** 32, size=(4, 20000), dtype=np.uint64)
    z = P.std_normal_ld(w).astype(np.float64)
    u1 = 1.0 - P.u01(w[0], w[1])
    nptest.assert_allclose(z, np.sqrt(-2 * np.log(u1)) * np.cos(2 * np.pi * P.u01(w[2], w[3])), rtol=0, atol=1e-13)
    assert abs(z.mean()) < 0.03 and abs(z.std() - 1) < 0.02


def test_stage_shards_and_consistency():
    """The restatement's stages: an edge shard is the slice of the whole draw (counter-based), T agrees with R,
    the states are one-hot, and the correlations lie in [-1, 1]."""
    th = dict(pi=0.3, eta=0.4, gamma=[0.2, 0.5, 0.3], epsilon=0.25, mu=[-0.15, 0.0, 0.3], sigma=[0.6, 0.035, 0.05])
    (seed, offset, N, H, U) = (0x0123456789ABCDEF, 0x00FEDCBA00000011, 13, 4, 6)
    (r, t, f, ft, b, bt) = P.sample(seed, offset, N, H, U, **th)
    C = N * (N - 1) // 2
    assert r.shape == (N, U) and t.shape == (C, U) and f.shape == (C, 3) and ft.shape == (C, U, 3)
    assert b.shape == (C, H) and bt.shape == (C, U)
    assert np.all(f.sum(1) == 1) and np.all(ft.sum(2) == 1)
    (n, m) = P.c_to_nm(np.arange(C))
    nptest.assert_array_equal(n * (n - 1) // 2 + m, np.arange(C))
    rb = r != 0
    assert np.all(t[rb[n] & rb[m]] == 1) and np.all(t[~rb[n] & ~rb[m]] == 0)
    assert b.min() >= -1 and b.max() <= 1 and b.min() == -1               # sigma_0 = 0.6 clips
    (c0, Cl) = (17, 40)
    nptest.assert_array_equal(P.sample_T(seed, offset, r, th["eta"], c0, Cl), t[c0:c0 + Cl])
    nptest.assert_array_equal(P.sample_F(seed, offset, c0, Cl, th["gamma"]), f[c0:c0 + Cl])
    nptest.assert_array_equal(P.sample_F_tilde(seed, offset, f[c0:c0 + Cl], t[c0:c0 + Cl], c0, th["epsilon"]),
                              ft[c0:c0 + Cl])
    nptest.assert_array_equal(P.sample_B(seed, offset, f[c0:c0 + Cl], c0, H, th["mu"], th["sigma"]), b[c0:c0 + Cl])
    nptest.assert_array_equal(P.sample_B_tilde(seed, offset, ft[c0:c0 + Cl], c0, th["mu"], th["sigma"]),
                              bt[c0:c0 + Cl])


def test_onehot_state_rule():
    f = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1, 0], [1, 0, 1], [0, 1, 1], [1, 1, 1],
                  [0, 0, 7]], dtype=np.uint8)
    nptest.assert_array_equal(P.onehot_state(f), [0, 0, 1, 2, 1, 2, 1, 1, 2])


def test_next_key_matches_model():
    rs = np.random.RandomState(2024)
    w = np.random.RandomState(2024).randint(0, 2 ** 32, size=4, dtype=np.uint64)
    (seed, offset) = P.next_key(rs)
    assert seed == int(w[0]) + (int(w[1]) << 32)
    assert offset == int(w[2]) + ((int(w[3]) & 0xFFFFFF) << 32) and offset < 2 ** 56
