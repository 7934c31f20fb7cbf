"""
NumPy restatement of the Philox sampler (K5, ``fcdiff_b200/csrc/fcd_sample.cu``).

Every random variable of the IAR model is one Philox4x32-10 block (Salmon et al.,
SC'11) at the counter (element index, stream offset, variable id) under the 64-bit
key ``seed``; this module recomputes those blocks on the host with uint64 arrays
and applies the kernels' decisions to them.  The uniforms and every threshold are
exact doubles on both sides, so R, T, F and F~ are reproduced bit for bit.  The
normals of B and B~ are evaluated in ``np.longdouble`` (Box-Muller with pi taken
in long double and the cosine argument reduced exactly), as the reference the
device's ``log`` / ``cospi`` are measured against.

Stage  var  element index  draws used
R      1    n*U + u        u01(x, y) < pi
T      2    c*U + u        u01(x, y) < eta, only where r_n != r_m
F      3    c              u01(x, y) against g0, g0 + g1
F~     4    c*U + u        (x, y): keep the state; (z, w): which other state
B      5    c*H + h        Box-Muller of (x, y, z, w)
B~     6    c*U + u        Box-Muller of (x, y, z, w)

Edges are in util order (c = n(n-1)/2 + m, m < n); ``c0`` is the first edge of a
shard, as in the C-ABI.
"""
import numpy as np

MASK32 = 0xFFFFFFFF
PHILOX_M0, PHILOX_M1 = 0xD2511F53, 0xCD9E8D57
PHILOX_W0, PHILOX_W1 = 0x9E3779B9, 0xBB67AE85
VAR_R, VAR_T, VAR_F, VAR_FT, VAR_B, VAR_BT = 1, 2, 3, 4, 5, 6

PI_LD = np.longdouble("3.14159265358979323846264338327950288")
_U64 = np.uint64


def philox4x32_10(k0, k1, c0, c1, c2, c3):
    """Philox4x32-10 on arrays of 32-bit words held in uint64 (broadcast)."""
    m0, m1, mask = _U64(PHILOX_M0), _U64(PHILOX_M1), _U64(MASK32)
    w0, w1 = _U64(PHILOX_W0), _U64(PHILOX_W1)
    (k0, k1, c0, c1, c2, c3) = (np.asarray(v, dtype=np.uint64) for v in (k0, k1, c0, c1, c2, c3))
    for _ in range(10):
        p0 = m0 * c0                        # 32 x 32 -> 64 bits: hi = __umulhi, lo = the 32-bit product
        p1 = m1 * c2
        (c0, c1, c2, c3) = ((p1 >> _U64(32)) ^ c1 ^ k0, p1 & mask, (p0 >> _U64(32)) ^ c3 ^ k1, p0 & mask)
        k0 = (k0 + w0) & mask
        k1 = (k1 + w1) & mask
    return (c0, c1, c2, c3)


def philox_make(seed, offset, var):
    """Key and the two upper counter words of ``philox_make``: (k0, k1, c2, c3).  Offset bits 56..63
    fall out of c3 (the 32-bit shift of the kernel)."""
    seed, offset = int(seed), int(offset)
    return (seed & MASK32, (seed >> 32) & MASK32, offset & MASK32,
            ((((offset >> 32) & MASK32) << 8) & MASK32) | int(var))


def blocks(seed, offset, var, idx):
    """The Philox blocks of element indices ``idx`` (uint64 array) of variable ``var``."""
    (k0, k1, c2, c3) = philox_make(seed, offset, var)
    idx = np.asarray(idx, dtype=np.uint64)
    return philox4x32_10(k0, k1, idx & _U64(MASK32), idx >> _U64(32), c2, c3)


def u01(a, b):
    """53-bit uniform in [0, 1): ((a >> 5) << 26 | b >> 6) / 2^53, exact in float64."""
    v = ((np.asarray(a, dtype=np.uint64) >> _U64(5)) << _U64(26)) | (np.asarray(b, dtype=np.uint64) >> _U64(6))
    return v.astype(np.float64) * 2.0 ** -53


def cospi_ld(x):
    """cos(pi x) in long double for float64 x: x = q/2 + y with |y| <= 1/4 exactly, then the quadrant."""
    x = np.asarray(x, dtype=np.float64)
    q = np.rint(2.0 * x)
    a = (x - 0.5 * q).astype(np.longdouble) * PI_LD
    qm = q.astype(np.int64) % 4
    return np.select([qm == 0, qm == 1, qm == 2], [np.cos(a), -np.sin(a), -np.cos(a)], np.sin(a))


def std_normal_ld(w):
    """Box-Muller of one block, sqrt(-2 log(1 - u01(x, y))) * cos(2 pi u01(z, w)), in long double."""
    u1 = 1.0 - u01(w[0], w[1])                          # exact: a multiple of 2^-53 in (0, 1]
    u2 = u01(w[2], w[3])
    return np.sqrt(-2 * np.log(u1.astype(np.longdouble))) * cospi_ld(2.0 * u2)


def onehot_state(f):
    """State of a (..., 3) state array as the kernels read it: 1 if f[1], else 2 if f[2], else 0."""
    f = np.asarray(f) != 0
    return np.where(f[..., 1], 1, np.where(f[..., 2], 2, 0))


def onehot(k):
    return np.stack([k == 0, k == 1, k == 2], axis=-1).astype(np.uint8)


def c_to_nm(c):
    """util edge index -> (n, m), exact for any int64 c."""
    c = np.asarray(c, dtype=np.int64)
    n = ((np.sqrt(8.0 * c + 1.0) - 1.0) * 0.5).astype(np.int64) + 1
    for _ in range(2):
        n = np.where(n * (n - 1) // 2 > c, n - 1, n)
        n = np.where((n + 1) * n // 2 <= c, n + 1, n)
    return (n, c - n * (n - 1) // 2)


def _edge_index(c0, C, K):
    """Element indices (c0 + cl) * K + k of a (C, K) shard, uint64."""
    return ((np.uint64(c0) + np.arange(C, dtype=np.uint64))[:, None] * np.uint64(K)
            + np.arange(K, dtype=np.uint64)[None, :])


def sample_R(seed, offset, N, U, pi):
    """(N, U) uint8: r[n, u] = u01 < pi."""
    w = blocks(seed, offset, VAR_R, np.arange(N * U, dtype=np.uint64))
    return (u01(w[0], w[1]) < float(pi)).astype(np.uint8).reshape(N, U)


def sample_T(seed, offset, r, eta, c0, C):
    """(C, U) uint8 of edges [c0, c0 + C): r_n if r_n == r_m, else u01 < eta."""
    r = np.asarray(r) != 0
    U = r.shape[1]
    (n, m) = c_to_nm(c0 + np.arange(C, dtype=np.int64))
    (rn, rm) = (r[n], r[m])
    w = blocks(seed, offset, VAR_T, _edge_index(c0, C, U))
    return np.where(rn == rm, rn, u01(w[0], w[1]) < float(eta)).astype(np.uint8)


def sample_F(seed, offset, c0, C, gamma):
    """(C, 3) uint8 one-hot: state (x >= g0) + (x >= g0 + g1), the sum in double."""
    (g0, g1) = (float(gamma[0]), float(gamma[1]))
    w = blocks(seed, offset, VAR_F, np.uint64(c0) + np.arange(C, dtype=np.uint64))
    x = u01(w[0], w[1])
    return onehot((x >= g0).astype(np.int64) + (x >= g0 + g1))


def sample_F_tilde(seed, offset, f, t, c0, epsilon):
    """(C, U, 3) uint8 one-hot: keep the template state if u01(x, y) < (epsilon if t else 1 - epsilon),
    else move to state (k + 1 + [u01(z, w) < 0.5]) mod 3."""
    t = np.asarray(t) != 0
    (C, U) = t.shape
    fk = onehot_state(f)[:, None]
    p_keep = np.where(t, float(epsilon), 1.0 - float(epsilon))
    w = blocks(seed, offset, VAR_FT, _edge_index(c0, C, U))
    keep = u01(w[0], w[1]) < p_keep
    other = (fk + 1 + (u01(w[2], w[3]) < 0.5)) % 3
    return onehot(np.where(keep, fk, other))


def _normal_stage(seed, offset, var, k, c0, K, mu, sigma):
    """Unclipped long-double mu_k + sigma_k z and the z of each element; k broadcasts to (C, K)."""
    C = k.shape[0]
    z = std_normal_ld(blocks(seed, offset, var, _edge_index(c0, C, K)))
    mu = np.asarray(mu, dtype=np.float64)[k]
    sigma = np.asarray(sigma, dtype=np.float64)[k]
    return (mu.astype(np.longdouble) + sigma.astype(np.longdouble) * z, z)


def sample_B(seed, offset, f, c0, H, mu, sigma, exact=False):
    """(C, H): mu_k + sigma_k z clipped to [-1, 1], k the state of edge row c.  Long double;
    ``exact`` also returns sigma_k z (the scale of the error of a float64 evaluation)."""
    k = np.broadcast_to(onehot_state(f)[:, None], (len(f), H))
    (b, z) = _normal_stage(seed, offset, VAR_B, k, c0, H, mu, sigma)
    return _clipped(b, z, k, sigma, exact)


def sample_B_tilde(seed, offset, ft, c0, mu, sigma, exact=False):
    """(C, U) as :func:`sample_B`, with the state of each element of the (C, U, 3) ``ft``."""
    k = onehot_state(ft)
    (b, z) = _normal_stage(seed, offset, VAR_BT, k, c0, k.shape[1], mu, sigma)
    return _clipped(b, z, k, sigma, exact)


def _clipped(b, z, k, sigma, exact):
    b = np.clip(b, -1, 1)
    if exact:
        return (b, np.asarray(sigma, dtype=np.float64)[k].astype(np.longdouble) * z)
    return b.astype(np.float64)


def next_key(rs):
    """``UnsharedRegionModel._next_key``: the 64-bit seed and 56-bit offset from four 32-bit draws."""
    w = rs.randint(0, 2 ** 32, size=4, dtype=np.uint64)
    return (int(w[0]) | (int(w[1]) << 32), int(w[2]) | ((int(w[3]) & 0xFFFFFF) << 32))


def sample(seed, offset, N, H, U, pi, eta, gamma, epsilon, mu, sigma, exact=False):
    """``UnsharedRegionModel.sample_device`` (all edges) under one key: (r, t, f, ft, b, bt) as uint8
    arrays and the clipped correlations (long double pairs with ``exact``, see :func:`sample_B`)."""
    C = N * (N - 1) // 2
    r = sample_R(seed, offset, N, U, pi)
    t = sample_T(seed, offset, r, eta, 0, C)
    f = sample_F(seed, offset, 0, C, gamma)
    ft = sample_F_tilde(seed, offset, f, t, 0, epsilon)
    b = sample_B(seed, offset, f, 0, H, mu, sigma, exact)
    bt = sample_B_tilde(seed, offset, ft, 0, mu, sigma, exact)
    return (r, t, f, ft, b, bt)
