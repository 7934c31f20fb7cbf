"""The fp64 routines of csrc/fcd_math.cuh against extended-precision references.

Every logarithm, reciprocal and exponential of the hot kernels comes from fast_log / fast_rcp / fast_log_rcp /
log_pos / rcp_newton / exp_nonpos(_short) and the -log r8 table in shared memory; the kernel-level parity tests
cannot see an error below ~1e-11 per term.  Here each routine runs elementwise in a test-only harness
(tests/math_probe.cu) on the arguments where it can go wrong -- slot boundaries of the 9-bit reciprocal, binade
edges, the switch points of the exponential's argument reduction, the clamp -- and is compared with np.longdouble
(64-bit mantissa).  The table window (log_table_window) is checked as a property over theta, and the uniform-start
row sums and the (eta, epsilon) objective / gradient at Schaefer-400 scale (10^7 cancelling terms) against
high-precision sums."""
import ctypes
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "fcdiff_b200", "csrc")
LD = np.longdouble

TAB_SIZE = 21 << 9                    # kLogTabSize
TAB_MIN_EXP = -1                      # kLogTabMinExp: slot i holds -log(2^(i // 512 - 1) (1 + (i % 512) / 512))
TWO_M19 = 2.0 ** -19                  # log_table_covers: every weight bound must lie above 2^-19

# bounds stated in fcd_math.cuh
FAST_LOG_ABS = 3e-13                  # fast_log: u - u^2/2 + u^3/3, |u| <= 2^-10, truncation u^4/4 <= 2.3e-13
FAST_RCP_REL = 9.1e-13                # fast_rcp: 1 - u + u^2 - u^3, truncation u^4 <= 2^-40
LOG_RCP_REL = 2.0 ** -50              # fast_log_rcp: ... + u^4, truncation u^5 <= 2^-50 (+ 2 ulp of rounding)
EXP_REL = 1e-14                       # exp_nonpos / exp_nonpos_short
# Estrin against Horner: 3 ulp of the result.  The two forms round independently -- Horner last at fma(p, r, 1),
# Estrin along 1 + r, r^2 p23 + p01, r^4 q1 + q0, r^8 q2 + (.) -- so each carries up to ~1.5 ulp; the earlier
# "~1e-16" in fcd_math.cuh was one ulp, and 10^6 arguments on a B200 show 2 ulp (4.3e-16 relative).
EXP_FORMS_ULP = 3


def _nvcc():
    cand = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return cand if os.path.isfile(cand) else shutil.which("nvcc")


def _build_probe(outdir):
    """nvcc flags of csrc/Makefile (no fast-math); fcd_runtime.cu supplies the real table and window code."""
    so = os.path.join(str(outdir), "libmath_probe.so")
    cmd = [_nvcc(), "-O3", "-std=c++17", "--expt-relaxed-constexpr", "-gencode", "arch=compute_100a,code=sm_100a",
           "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared", "-I" + os.path.join(ROOT, "include"), "-I" + CSRC,
           os.path.join(ROOT, "tests", "math_probe.cu"), os.path.join(CSRC, "fcd_runtime.cu"), "-o", so, "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    return so


def test_math_probe_compiles(tmp_path):
    """The harness compiles for sm_100a against the current headers (no device needed)."""
    if _nvcc() is None:
        pytest.skip("nvcc not found")
    assert os.path.getsize(_build_probe(tmp_path)) > 0


# ---------------------------------------------------------------------------------------------- device side

@pytest.fixture(scope="session")
def probe(tmp_path_factory):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    if _nvcc() is None:
        pytest.skip("nvcc not found")
    if np.finfo(LD).nmant < 63:
        pytest.skip("np.longdouble has %d mantissa bits here; the reference needs 63" % np.finfo(LD).nmant)
    lib = ctypes.CDLL(_build_probe(tmp_path_factory.mktemp("math_probe")))
    P, I64, I32, D = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_double
    sig = {"probe_window": [P, P, I32, P, P], "probe_copy_table": [P, P], "probe_table_size": [],
           "probe_fast_log": [P, I64, P, P, I32, P, P, P], "probe_fast_log_rcp": [P, I64, P, P, I32, P, P, P],
           "probe_log_pos": [P, I64, P, P, P, P], "probe_mix_slots": [P, I64, D, D, P, P, I32, P, P, P, P],
           "probe_plain": [I32, P, I64, P, P]}
    for (name, args) in sig.items():
        getattr(lib, name).argtypes = args
        getattr(lib, name).restype = ctypes.c_int
    lib.probe_last_error.restype = ctypes.c_char_p
    assert lib.probe_table_size() == TAB_SIZE
    return Probe(lib, torch)


def _d3(v):
    return (ctypes.c_double * 3)(*[float(x) for x in v])


class Probe:
    """Elementwise evaluation of one routine on the device; numpy in, numpy out."""

    def __init__(self, lib, torch):
        (self.lib, self.torch) = (lib, torch)

    def _st(self):
        return ctypes.c_void_p(self.torch.cuda.current_stream().cuda_stream)

    def _check(self, rc, what):
        assert rc == 0, "%s: %s" % (what, self.lib.probe_last_error())
        self.torch.cuda.synchronize()

    def _in(self, x):
        return self.torch.from_numpy(np.ascontiguousarray(x, np.float64)).cuda()

    def _out(self, n, dtype=None):
        return self.torch.empty(n, dtype=dtype or self.torch.float64, device="cuda")

    @staticmethod
    def _p(t):
        return ctypes.c_void_p(t.data_ptr())

    def window(self, epsl, al, with_mantissa=True):
        w = (ctypes.c_int * 3)()
        self._check(self.lib.probe_window(_d3(epsl), _d3(al), int(with_mantissa), w, self._st()), "probe_window")
        return (w[0], w[1], bool(w[2]))

    def table(self):
        t = self._out(TAB_SIZE)
        self._check(self.lib.probe_copy_table(self._p(t), self._st()), "probe_copy_table")
        return t.cpu().numpy()

    def fast_log(self, y, epsl, al, with_mantissa=True):
        (x, out, slot) = (self._in(y), self._out(len(y)), self._out(len(y), self.torch.int32))
        self._check(self.lib.probe_fast_log(self._p(x), len(y), _d3(epsl), _d3(al), int(with_mantissa), self._p(out),
                                            self._p(slot), self._st()), "probe_fast_log")
        return (out.cpu().numpy(), slot.cpu().numpy())

    def fast_log_rcp(self, y, epsl, al):
        (x, lg, rcp) = (self._in(y), self._out(len(y)), self._out(len(y)))
        self._check(self.lib.probe_fast_log_rcp(self._p(x), len(y), _d3(epsl), _d3(al), 1, self._p(lg), self._p(rcp),
                                                self._st()), "probe_fast_log_rcp")
        return (lg.cpu().numpy(), rcp.cpu().numpy())

    def log_pos(self, v, epsl, al):
        (x, out) = (self._in(v), self._out(len(v)))
        self._check(self.lib.probe_log_pos(self._p(x), len(v), _d3(epsl), _d3(al), self._p(out), self._st()),
                    "probe_log_pos")
        return out.cpu().numpy()

    def mix_slots(self, p, eta, eps, w_epsl, w_al, with_mantissa):
        n = len(p)
        (x, y, slot, lg) = (self._in(p), self._out(3 * n), self._out(3 * n, self.torch.int32), self._out(3 * n))
        self._check(self.lib.probe_mix_slots(self._p(x), n, float(eta), float(eps), _d3(w_epsl), _d3(w_al),
                                             int(with_mantissa), self._p(y), self._p(slot), self._p(lg), self._st()),
                    "probe_mix_slots")
        return (y.cpu().numpy(), slot.cpu().numpy(), lg.cpu().numpy())

    def plain(self, which, v):
        (x, out) = (self._in(v), self._out(len(v)))
        self._check(self.lib.probe_plain(which, self._p(x), len(v), self._p(out), self._st()), "probe_plain")
        return out.cpu().numpy()

    def fast_rcp(self, v):
        return self.plain(0, v)

    def rcp_newton(self, v):
        return self.plain(1, v)

    def exp_nonpos(self, v):
        return self.plain(2, v)

    def exp_nonpos_short(self, v):
        return self.plain(3, v)


# ---------------------------------------------------------------------------------------------- arguments

# the widest FAST window: min weight just above 2^-19, with the mantissa binade -> slots [0, slot(2^-19) + 4]
WIDE_EPSL = [np.nextafter(TWO_M19, 1.0)] * 3
WIDE_AL = WIDE_EPSL


def _ulps(x, ks):
    """x moved by k ulp for every k in ks (x > 0 finite)."""
    b = np.asarray(x, np.float64).view(np.int64)
    return np.concatenate([(b + k).view(np.float64) for k in ks])


def _r8(i):
    """the 9-bit reciprocal of table slot i (exact)."""
    i = np.asarray(i)
    return np.ldexp(1.0 + (i % 512) / 512.0, i // 512 + TAB_MIN_EXP)


def log_arguments(rng, n_random=10 ** 6):
    """(edge arguments, random arguments) of fast_log / fast_rcp / fast_log_rcp in (2^-19, 2):
    the rounding midpoints 1/((r8_i + r8_{i+1}) / 2) between neighbouring 9-bit reciprocals (|u| largest) and
    +-1..4 ulp around them, for every slot of the widest window (slots below 512 are the mantissa binade [1, 2)
    of log_pos); exact binade edges +-1..4 ulp; y = 1 + k ulp; log-uniform values in (2^-19, 1]."""
    i = np.arange(0, 10240)
    mid = ((_r8(i) + _r8(i + 1)) / 2).astype(LD)
    mids = (LD(1) / mid).astype(np.float64)
    edges = np.ldexp(1.0, -np.arange(0, 20))
    y = np.concatenate([mids, _ulps(mids, [-4, -3, -2, -1, 1, 2, 3, 4]), edges, _ulps(edges, [-4, -3, -2, -1, 1, 2, 3, 4]),
                        _ulps([1.0], [1, 2, 3, 4])])
    y = y[(y > TWO_M19) & (y < 2.0)]
    r = np.exp2(-19.0 * (1.0 - rng.random_sample(n_random)))           # (2^-19, 1]
    return (y, r[r > TWO_M19])


@pytest.fixture(scope="module")
def log_args():
    return log_arguments(np.random.RandomState(11))


def _abs_err(got, ref):
    return np.abs(got.astype(LD) - ref)


def _report(name, value):
    print("%-34s %.3e" % (name, float(value)))


# ---------------------------------------------------------------------------------------------- routines

@pytest.mark.gpu
def test_log_table_entries_within_one_ulp(probe):
    tab = probe.table()
    ref = -np.log(_r8(np.arange(TAB_SIZE)).astype(LD))
    err = _abs_err(tab, ref)
    _report("table max |err| / ulp", (err / LD(2.0 ** -52) / np.maximum(np.abs(ref), LD(2.0 ** -1022))).max())
    assert tab[512] == 0.0                                             # r8 = 1
    ulp = np.spacing(np.abs(ref.astype(np.float64)))
    bad = np.nonzero(err > ulp)[0]
    assert bad.size == 0, "slots %s off by more than 1 ulp" % bad[:8]


@pytest.mark.gpu
def test_fast_log_against_longdouble(probe, log_args):
    lo, n, covers = probe.window(WIDE_EPSL, WIDE_AL)
    assert covers and lo == 0 and n >= 10242
    for (what, y) in zip(("edges", "random"), log_args):
        (got, slot) = probe.fast_log(y, WIDE_EPSL, WIDE_AL)
        assert ((slot >= lo) & (slot < lo + n)).all(), "slot outside the staged window: %s" % y[(slot < lo) | (slot >= lo + n)][:4]
        assert not np.isnan(got).any()
        # slot i of the reduction is the rounded reciprocal: |u| = |y r8 - 1| <= 2^-10 (+ MUFU error)
        u = (y.astype(LD) * _r8(slot).astype(LD) - 1)
        _report("fast_log max |u| (%s) * 2^10" % what, np.abs(u).max() * 1024)
        err = _abs_err(got, np.log(y.astype(LD)))
        _report("fast_log max abs err (%s)" % what, err.max())
        assert err.max() < FAST_LOG_ABS, y[np.argmax(err)]


@pytest.mark.gpu
def test_fast_rcp_against_longdouble(probe, log_args):
    for (what, y) in zip(("edges", "random"), log_args):
        got = probe.fast_rcp(y)
        rel = got.astype(LD) * y.astype(LD) - 1
        _report("fast_rcp max rel err (%s)" % what, np.abs(rel).max())
        assert np.abs(rel).max() <= FAST_RCP_REL, y[np.argmax(np.abs(rel))]


@pytest.mark.gpu
def test_fast_log_rcp_against_longdouble(probe, log_args):
    for (what, y) in zip(("edges", "random"), log_args):
        (lg, rcp) = probe.fast_log_rcp(y, WIDE_EPSL, WIDE_AL)
        assert not np.isnan(lg).any()
        err = _abs_err(lg, np.log(y.astype(LD)))
        assert err.max() < FAST_LOG_ABS
        ref = LD(1) / y.astype(LD)
        d = rcp.astype(LD) - ref
        bound = LD(LOG_RCP_REL) * ref + 2 * np.spacing(ref.astype(np.float64)).astype(LD)
        _report("fast_log_rcp max rel err (%s)" % what, (np.abs(d) / ref).max())
        assert (np.abs(d) <= bound).all(), y[np.argmax(np.abs(d) / bound)]
        if what == "random":
            # the gradient sums ~10^7 such reciprocals with cancellation: no one-sided truncation
            bias = (d / ref).mean()
            _report("fast_log_rcp mean signed rel err", bias)
            assert abs(bias) <= 2.0 ** -52


@pytest.mark.gpu
def test_log_pos_against_longdouble(probe):
    rng = np.random.RandomState(5)
    e = np.concatenate([np.arange(-1022, 1), [1, 2, 7, 100, 1023]])
    m = np.array([1.0, np.nextafter(1.0, 2.0), np.nextafter(2.0, 0.0), _ulps([2.0], [-4])[0]])
    x = np.ldexp(np.repeat(m[None, :], len(e), 0), e[:, None]).ravel()
    x = np.concatenate([x, np.ldexp(1.0 + rng.random_sample(10 ** 6), rng.randint(-1022, 1024, 10 ** 6)),
                        np.exp2(-19.0 * rng.random_sample(10 ** 5))])      # the running products of weights
    got = probe.log_pos(x, WIDE_EPSL, WIDE_AL)
    ref = np.log(x.astype(LD))
    err = _abs_err(got, ref)
    _report("log_pos max abs err", err.max())
    bound = LD(FAST_LOG_ABS) + LD(2.0 ** -52) * np.abs(ref)
    assert (err <= bound).all(), x[np.argmax(err / bound)]


@pytest.mark.gpu
def test_rcp_newton_within_one_ulp(probe):
    rng = np.random.RandomState(7)
    # positive normals whose reciprocal is normal too (MUFU.RCP64H flushes subnormal results)
    e = np.arange(-1021, 1022)
    edges = np.ldexp(1.0, e)
    x = np.concatenate([edges, _ulps(edges, [-2, -1, 1, 2]), 1.5 * edges, [np.ldexp(1.0, -1022)], _ulps([np.ldexp(1.0, 1022)], [-1])])
    rnd = np.ldexp(1.0 + rng.random_sample(10 ** 6), rng.randint(-1021, 1022, 10 ** 6))
    for (what, v) in (("edges", x), ("random", rnd)):
        got = probe.rcp_newton(v)
        ref = LD(1) / v.astype(LD)
        d = got.astype(LD) - ref
        ulp = np.spacing(ref.astype(np.float64)).astype(LD)
        _report("rcp_newton max err / ulp (%s)" % what, (np.abs(d) / ulp).max())
        assert (np.abs(d) <= ulp).all(), v[np.argmax(np.abs(d) / ulp)]
        if what == "random":
            bias = (d / ref).mean()
            _report("rcp_newton mean signed rel err", bias)
            assert abs(bias) <= 2.0 ** -53


def exp_arguments(rng):
    """edge arguments of exp_nonpos: 0, -0, the smallest subnormal, -k ln2 and -(k + 1/2) ln2 +-1..2 ulp (the
    points where n of the argument reduction switches and where |r| is largest) for every k up to 1010,
    -700 and its neighbours above."""
    k = np.arange(0, 1011).astype(LD)
    ln2 = np.log(LD(2))
    pts = np.concatenate([-(k * ln2), -((k + LD(0.5)) * ln2)]).astype(np.float64)
    pts = pts[pts < 0]
    near = -_ulps(-pts, [-2, -1, 0, 1, 2])
    edge = np.concatenate([[0.0, -0.0, -np.ldexp(1.0, -1074), -1e-300, -700.0], -_ulps([700.0], [-4, -3, -2, -1])])
    x = np.concatenate([edge, near])
    return (x[x >= -700.0], -700.0 * rng.random_sample(10 ** 6))


@pytest.mark.gpu
def test_exp_nonpos_against_longdouble(probe):
    (edges, rnd) = exp_arguments(np.random.RandomState(3))
    for (what, d) in (("edges", edges), ("random", rnd)):
        h = probe.exp_nonpos(d)
        s = probe.exp_nonpos_short(d)
        ref = np.exp(d.astype(LD))
        for (name, got) in (("exp_nonpos", h), ("exp_nonpos_short", s)):
            rel = np.abs(got.astype(LD) - ref) / ref
            _report("%s max rel err (%s)" % (name, what), rel.max())
            assert rel.max() < EXP_REL, (name, d[np.argmax(rel)])
        forms = np.abs(s.astype(LD) - h.astype(LD)) / np.spacing(h).astype(LD)
        _report("Estrin - Horner max ulp (%s)" % what, forms.max())
        assert forms.max() <= EXP_FORMS_ULP, d[np.argmax(forms)]


@pytest.mark.gpu
def test_exp_nonpos_clamp_and_nan(probe):
    """Arguments below -700 are clamped to -700 (bit for bit).  NaN comes out as e^-700 as well: fmax drops
    the NaN operand.  The callers pass differences of finite log-weights, so this is the recorded behaviour, not
    a guarantee to rely on."""
    low = np.array([-700.0, np.nextafter(-700.0, -np.inf), -700.5, -745.2, -1e4, -1e300, -np.inf, np.nan])
    for f in (probe.exp_nonpos, probe.exp_nonpos_short):
        got = f(low)
        assert (got.view(np.int64) == got[0].view(np.int64)).all(), got
        assert abs(float(got[0].astype(LD) / np.exp(LD(-700)) - 1)) < EXP_REL


# ---------------------------------------------------------------------------------------------- the window

def _theta_weights(eta, eps):
    """make_theta_dev: eps_l, a_l, b_l (same double operations)."""
    epsl = np.array([1.0 - eps, eps, eta * eps + (1.0 - eta) * (1.0 - eps)])
    al = (1.0 - epsl) * 0.5
    return (epsl, al, epsl - al)


EPS_FAST = 2.0 ** -18 + 2.0 ** -53    # smallest eps above 2^-18 whose a_0 = (1 - (1 - eps)) / 2 stays above 2^-19
BOX = (1e-5, 1 - 1e-5)                # the solver box of eta and epsilon


def _p_grid():
    """p in [0, 1] on a fine grid, the endpoints, and p_2 = (1 - p_0) - p_1 rounded just below 0 or 1."""
    p = np.linspace(0.0, 1.0, (1 << 16) + 1)
    p0 = np.random.RandomState(1).random_sample(4096)
    p2 = (1.0 - p0) - np.nextafter(1.0 - p0, 2.0)                     # -ulp(1 - p0), e.g. -2^-53
    tiny = np.array([-2.0 ** -53, -2.0 ** -52, -2.0 ** -54, 2.0 ** -53, np.nextafter(1.0, 2.0), np.nextafter(1.0, 0.0),
                     5e-324, -5e-324])
    return np.concatenate([p, p2[p2 < 0], tiny])


def _window_cases():
    grid = [BOX[0], 0.25, 0.5, 0.75, BOX[1]]
    cases = []
    for eta in grid:
        for eps in grid + [0.12, EPS_FAST, 1.0 - EPS_FAST, 2.0 ** -18]:
            (epsl, al, _) = _theta_weights(eta, eps)
            cases += [("theta", eta, eps, epsl, al, wm) for wm in (True, False)]
    # the solved E-step / fcd_elm_coded_solve: window of the box, weights of any theta inside it
    m = min(BOX[0], 1.0 - BOX[1])
    for eta in grid:
        for eps in grid:
            cases += [("box", eta, eps, [m] * 3, [0.5 * m] * 3, wm) for wm in (True, False)]
    return cases


@pytest.mark.gpu
def test_window_covers_every_slot_the_weights_use(probe):
    p = _p_grid()
    n_fast = 0
    for (form, eta, eps, w_epsl, w_al, wm) in _window_cases():
        (lo, n, covers) = probe.window(w_epsl, w_al, wm)
        assert lo % 2 == 0 and n % 2 == 0 and 0 <= lo and lo + n <= TAB_SIZE
        if not covers:
            assert (lo, n) == (0, TAB_SIZE)
            assert form == "theta" and min(min(_theta_weights(eta, eps)[0]), min(_theta_weights(eta, eps)[1])) <= TWO_M19
            continue
        n_fast += 1
        (y, slot, lg) = probe.mix_slots(p, eta, eps, w_epsl, w_al, wm)
        out = (slot < lo) | (slot >= lo + n)
        assert not out.any(), (form, eta, eps, wm, lo, n, np.unique(slot[out])[:8], y[out][:4])
        assert not np.isnan(lg).any()
        ok = y > 0
        assert np.abs(lg[ok].astype(LD) - np.log(y[ok].astype(LD))).max() < FAST_LOG_ABS
    assert n_fast > 100


@pytest.mark.gpu
def test_fast_safe_threshold(probe):
    """a_0 = eps / 2 must lie strictly above 2^-19 for the table kernels.  eps = 2^-18 (1 + 2^-40) is not enough:
    1 - eps rounds back to 1 - 2^-18, and a_0 = 2^-19 exactly."""
    for (eps, fast) in ((EPS_FAST, True), (2.0 ** -18, False), (2.0 ** -18 * (1 + 2.0 ** -40), False)):
        (epsl, al, _) = _theta_weights(0.5, eps)
        assert probe.window(epsl, al)[2] is fast, eps
        (epsl, al, _) = _theta_weights(0.5, 1.0 - eps)               # the mirrored edge: a_1 = (1 - eps_1) / 2
        assert probe.window(epsl, al)[2] is fast, 1.0 - eps


# ---------------------------------------------------------------------------------------------- kernels

def _theta(eta, eps):
    from fcdiff_b200 import _lib
    return _lib.make_theta(0.1, eta, eps, [0.2, 0.5, 0.3], [-0.1, 0.0, 0.1], [0.1, 0.1, 0.1])


def _slot_covering_p(eta, eps, per_slot=3):
    """p in [0, 1] whose weights a_l + b_l p step through every table slot between the weights' bounds, for each l."""
    (epsl, al, bl) = _theta_weights(eta, eps)
    ps = [np.array([0.0, 1.0])]
    for l in range(3):
        (ya, yb) = sorted((al[l], epsl[l]))
        nslots = int(np.ceil(np.log2(yb / ya) * 512)) + 2
        y = np.exp2(np.linspace(np.log2(ya), np.log2(yb), per_slot * nslots))
        ps.append(np.clip((y - al[l]) / bl[l], 0.0, 1.0))
    return np.concatenate(ps)


@pytest.mark.gpu
@pytest.mark.parametrize("eta,eps", [(0.37, 0.12), (0.5, EPS_FAST), (0.5, 2.0 ** -18), (0.5, 1.0 - EPS_FAST),
                                     (BOX[1], BOX[0]), (BOX[0], BOX[1]), (0.5, 0.5)])
@pytest.mark.parametrize("U", [1, 2, 3])
def test_row_logsums_against_longdouble(probe, eta, eps, U):
    """fcd_row_logsums (uniform start): S9[c][3k + l] = sum_u log(a_l + b_l p_k) through running products and
    log_pos, with p_0 stepping through every slot of the window, p_1 = t (1 - p_0) and p_2 rounded below 0."""
    from fcdiff_b200 import _dev, _lib
    lib = _lib.load()
    rng = np.random.RandomState(U)
    p0 = _slot_covering_p(eta, eps)
    p0 = np.concatenate([p0, rng.random_sample(64)])
    p1 = rng.random_sample(len(p0)) * (1.0 - p0)
    # elements whose p_2 = (1 - p_0) - p_1 rounds to just below 0
    q0 = rng.random_sample(256)
    p0 = np.concatenate([p0, q0])
    p1 = np.concatenate([p1, np.nextafter(1.0 - q0, 2.0)])
    C = -(-len(p0) // U)
    pitchU = U + (U & 1)
    pad = C * U - len(p0)
    perm = rng.permutation(len(p0))
    planes = np.full((2, C, pitchU), np.nan)                          # padding lanes must not enter the sums
    planes[0, :, :U] = np.concatenate([p0[perm], np.full(pad, 0.5)]).reshape(C, U)
    planes[1, :, :U] = np.concatenate([p1[perm], np.full(pad, 0.25)]).reshape(C, U)
    P = _dev.upload(planes.reshape(-1))
    S9 = _dev.zeros((C * 9,))
    th = _theta(eta, eps)
    _lib.check(lib.fcd_row_logsums(_dev.ptr(P), C * pitchU, C, U, pitchU, ctypes.byref(th), _dev.ptr(S9), _dev.stream()),
               "fcd_row_logsums")
    got = S9.cpu().numpy().reshape(C, 3, 3)
    (_, al, bl) = _theta_weights(eta, eps)
    pk = planes[:, :, :U].astype(LD)
    pk = np.stack([pk[0], pk[1], (1 - planes[0, :, :U]) - planes[1, :, :U]])   # p_2 as the kernel forms it
    want = np.log(al.astype(LD)[None, :, None, None] + bl.astype(LD)[None, :, None, None] * pk[:, None]).sum(-1)
    want = np.moveaxis(want, 2, 0)                                    # [C][k][l]
    err = np.abs(got.astype(LD) - want)
    assert err.max() <= 1e-12 * U, (np.unravel_index(np.argmax(err), err.shape), float(err.max()))


# --------------------------------------------------------- the (eta, epsilon) objective at Schaefer-400 scale

N_BIG, U_BIG = 400, 128               # C = 79 800 edges x 128 patients ~ 10^7 edge-patient elements


@pytest.fixture(scope="module")
def big_problem(probe):
    """Half the responsibilities near 1/3 (Dirichlet(50, 50, 50)), where the (3 p - 1) / 2 factors of the gradient
    cancel; the other half decided as in a fitted cohort (one p_k within 1e-7 of 1), where every weight of a
    state sits at the same a_l or eps_l, so that its reduction u -- and the truncation error of a reciprocal --
    is the same for all of them and adds up instead of averaging out.  q_F: 80 % peaked (one-hot), the rest
    Dirichlet(2, 2, 2); q_R: 65 % peaked, the rest undecided -- every tier (one plane and one log / three logs /
    nine logs per element) is read."""
    N, U = N_BIG, U_BIG
    C = N * (N - 1) // 2
    rng = np.random.default_rng(2024)
    g = rng.standard_gamma(50.0, size=(3, C, U))
    P = g / g.sum(axis=0)
    del g
    dec = rng.random((C, U)) < 0.5
    nd = int(dec.sum())
    (s, delta, t) = (rng.integers(0, 3, nd), 1e-7 * rng.random(nd), rng.random(nd))
    pd = np.empty((3, nd))
    pd[0] = delta * t
    pd[1] = delta - pd[0]
    pd[2] = 1.0 - delta
    rot = (np.arange(3)[:, None] - s[None, :] + 2) % 3                 # p_s = 1 - delta
    P[:, dec] = np.take_along_axis(pd, rot, axis=0)
    fstate = np.where(rng.random(C) < 0.8, rng.integers(0, 3, C), 3).astype(np.uint8)
    qF = np.eye(3)[np.minimum(fstate, 2)]
    qF[fstate == 3] = rng.dirichlet([2.0, 2.0, 2.0], size=int((fstate == 3).sum()))
    pitchS = 256
    rstate = np.full((N, pitchS), 4, np.uint8)
    rstate[:, :U] = np.where(rng.random((N, U)) < 0.65, rng.integers(0, 2, (N, U)), 2)
    qR = np.eye(2)[np.minimum(rstate[:, :U], 1)]
    und = rstate[:, :U] == 2
    qR[und] = rng.dirichlet([2.0, 2.0], size=int(und.sum()))
    nn = np.repeat(np.arange(N), np.arange(N))                      # c = n (n - 1) / 2 + m, m < n
    mm = np.concatenate([np.arange(n) for n in range(N)])
    return dict(N=N, U=U, C=C, P=P, qF=qF, fstate=fstate, qR=qR, rstate=rstate, pitchS=pitchS, nn=nn, mm=mm)


def _elm_reference(pb, eta, eps, chunk=2000):
    """out3 of fcd_elm_obj_grad in float64 with per-chunk np.sum and math.fsum across chunks, and the sums of
    |term| of the objective and of both gradient components."""
    (_, al, bl) = _theta_weights(eta, eps)
    sl = np.array([-1.0, 1.0, 2.0 * eta - 1.0])
    (P, qF, qR, nn, mm) = (pb['P'], pb['qF'], pb['qR'], pb['nn'], pb['mm'])
    parts = {k: [] for k in ("obj", "aobj", "ge", "age", "gh", "agh")}
    for c0 in range(0, pb['C'], chunk):
        c1 = min(c0 + chunk, pb['C'])
        (qn, qm) = (qR[nn[c0:c1]], qR[mm[c0:c1]])
        w = (qn[..., 0] * qm[..., 0], qn[..., 1] * qm[..., 1], qn[..., 0] * qm[..., 1] + qn[..., 1] * qm[..., 0])
        for k in range(3):
            p = P[k, c0:c1]
            num = 1.5 * p - 0.5
            qk = qF[c0:c1, k][:, None]
            for l in range(3):
                M = al[l] + bl[l] * p
                t = qk * w[l]
                o = t * np.log(M)
                d = t * num / M
                parts["obj"].append(o.sum())
                parts["aobj"].append(np.abs(o).sum())
                parts["ge"].append(sl[l] * d.sum())
                parts["age"].append(abs(sl[l]) * np.abs(d).sum())
                if l == 2:
                    parts["gh"].append(d.sum())
                    parts["agh"].append(np.abs(d).sum())
    s = {k: math.fsum(v) for (k, v) in parts.items()}
    want = np.array([s["obj"], -(2.0 * eps - 1.0) * s["gh"], -s["ge"]])
    scale = np.array([s["aobj"], abs(2.0 * eps - 1.0) * s["agh"], s["age"]])
    return (want, scale)


@pytest.fixture(scope="module")
def big_device(big_problem):
    import torch
    from fcdiff_b200 import _dev
    pb = big_problem
    d = dict(P=_dev.upload(pb['P'].reshape(-1)), qF=_dev.upload(pb['qF'].reshape(-1)), qR=_dev.upload(pb['qR'].reshape(-1)),
             fs=torch.from_numpy(pb['fstate']).cuda(), rs=torch.from_numpy(pb['rstate']).cuda(),
             nm=torch.from_numpy((pb['nn'] | (pb['mm'] << 16)).astype(np.int32)).cuda())
    return d


THETA_BIG = [(0.37, 0.12), (0.6, 1e-5)]


@pytest.mark.gpu
@pytest.mark.parametrize("eta,eps", THETA_BIG)
def test_elm_objective_and_gradient_at_scale(big_problem, big_device, eta, eps):
    """fcd_elm_obj_grad (tiered) and fcd_elm_coded (code pass as in test_gpu_code_pass.py) over ~10^7 elements:
    |error| <= 1e-12 sum |term| for the objective and both gradient components.  A one-sided error of 1e-9 per
    reciprocal would miss this by three orders of magnitude."""
    import torch
    from fcdiff_b200 import _dev, _lib
    lib = _lib.load()
    (pb, d) = (big_problem, big_device)
    (N, U, C, pitchS) = (pb['N'], pb['U'], pb['C'], pb['pitchS'])
    pitchU = U
    st = _dev.stream()
    ws = _dev.workspace()
    th = _theta(eta, eps)
    (want, scale) = _elm_reference(pb, eta, eps)

    out = _dev.zeros((3,))
    _lib.check(lib.fcd_elm_obj_grad(_dev.ptr(d['P']), C * pitchU, C, U, pitchU, _dev.ptr(d['qF']), _dev.ptr(d['fs']),
                                    _dev.ptr(d['qR']), _dev.ptr(d['rs']), pitchS, N, _dev.ptr(d['nm']), ctypes.byref(th), 1,
                                    _dev.ptr(out), _dev.ptr(ws), st), "fcd_elm_obj_grad")
    tiered = out.cpu().numpy()

    pitchQ = int(lib.fcd_code_pitch(U))
    PsE = _dev.zeros((C, pitchQ))
    kc = torch.full((C,), 255, dtype=torch.uint8, device="cuda")
    code = _dev.empty((C * pitchQ + 256,), torch.uint8)
    counts = _dev.empty((C, 2), torch.int32)
    offs = _dev.empty((4 * int(lib.fcd_bucket_blocks(C)),), torch.int64)
    tot = _dev.zeros((2,))
    _lib.check(lib.fcd_code_plane(_dev.ptr(d['P']), C * pitchU, C, U, pitchU, _dev.ptr(d['fs']), _dev.ptr(d['rs']), pitchS,
                                  _dev.ptr(d['nm']), _dev.ptr(PsE), _dev.ptr(kc), _dev.ptr(code), pitchQ, _dev.ptr(counts),
                                  _dev.ptr(offs), _dev.ptr(tot), st), "fcd_code_plane")
    (nd, nh) = (int(v) for v in tot.cpu().numpy())
    assert nd > 0 and nh > 0
    L = _dev.zeros((C * pitchU,))
    Lsum = _dev.zeros((1,))
    D = _dev.empty((4 * nd,))
    K = _dev.empty((nd,), torch.int64)
    KH = _dev.empty((nh,), torch.int64)
    Hh = _dev.empty((2 * nh,))
    RO = _dev.empty((C, 2), torch.int64)
    out4 = _dev.zeros((4,))
    _lib.check(lib.fcd_code_records(_dev.ptr(d['P']), C * pitchU, _dev.ptr(PsE), _dev.ptr(code), pitchQ, _dev.ptr(L),
                                    _dev.ptr(Lsum), C, U, pitchU, _dev.ptr(d['qF']), _dev.ptr(d['fs']), _dev.ptr(d['qR']),
                                    _dev.ptr(d['rs']), pitchS, N, _dev.ptr(d['nm']), _dev.ptr(counts), _dev.ptr(offs),
                                    _dev.ptr(K), _dev.ptr(KH), _dev.ptr(RO), _dev.ptr(D), nd, _dev.ptr(Hh), nh,
                                    _dev.ptr(out4[3:]), _dev.ptr(ws), st), "fcd_code_records")
    _lib.check(lib.fcd_elm_coded(_dev.ptr(PsE), _dev.ptr(code), C * pitchQ, _dev.ptr(D), nd, _dev.ptr(Hh), nh,
                                 ctypes.byref(th), 1, _dev.ptr(out4), _dev.ptr(ws), st), "fcd_elm_coded")
    coded = out4.cpu().numpy()[:3]
    for (name, got) in (("tiered", tiered), ("coded", coded)):
        rel = np.abs(got - want) / scale
        print("%s eta=%g eps=%g |err| / sum|term| = %s (net / sum|term| = %s)" % (name, eta, eps, rel, np.abs(want) / scale))
        assert (rel <= 1e-12).all(), (name, got, want, scale)
