"""The device math building blocks of the kernels, called directly, against independent high-precision references.

tests/devmath/devmath.cu wraps the product headers unchanged: the canonical arithmetic of octet.cuh (canon_sincos,
canon_log, canon_rsqrt / canon_pivot_ok, canon_acos), the SE(3) functions of fb_math.cuh, the task-space pose error of
task_space_cost.cuh (log3_canon, jlog3_canon, task_evaluate), the warp Cholesky of warp_llt.cuh and the fraction-to-
boundary rule of pdipm.cuh.  It builds two ways: with g++ against the SIMT emulator of tests/emu (every machine) and
with nvcc and the product's flags for the B200 (-m gpu).  The GPU build must give the emulator's results bit for bit
on every input (NaN matches any NaN), and both must meet the same bounds.

The references are mpmath at 50 digits and share no formula with the port: mp.sin / cos / log / acos / sqrt,
mp.expm of the 4x4 homogeneous matrix, Jexp6 by central differences of that exponential (Jlog6 is its inverse),
mp.cholesky / mp.inverse and exact rationals.  Bounds are multiples of eps times the operation's condition number;
where the port keeps a formula of upstream that is less accurate than that, the bound has the shape of that formula's
error and says so.  The inputs reach the branch points and domain edges that the solver scenarios never produce.
"""
import ctypes
import functools
import math
import os
import subprocess
import sys
from fractions import Fraction

import mpmath as mp
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "devmath", "devmath.cu")
CSRC = os.path.join(ROOT, "idocp_b200", "csrc")
EMU = os.path.join(ROOT, "tests", "emu")
BUILD = os.path.join(ROOT, "build", "devmath")
EPS = np.finfo(float).eps
TAYLOR = 1.220703125e-04   # the Taylor thresholds FB_TAYLOR / TASK_TAYLOR = eps^(1/4) = 2^-13
mp.mp.dps = 50

# function ids of k_dm_scalar (enum DmFn in devmath.cu)
(SINCOS, LOG, RSQRT, PIVOT_OK, ACOS, LOG3_CANON, JLOG3_CANON, FB_LOG3, FB_JLOG3, FB_LOG6, FB_JLOG6, FB_EXP6, FB_JEXP6,
 FB_JEXP3, FB_R_TO_QUAT, FB_QUAT_TO_R, FB_INV33, FB_INTEGRATE, FB_SUBTRACT, FB_DSUBTRACT_DPLUS, FB_DSUBTRACT_DMINUS,
 FB_DSUBTRACT_INVERSE, FB_DINTEGRATE_DQ, FB_DINTEGRATE_DV, FRACTION_ROW, NUM_FN) = range(26)
DM_IN = DM_OUT = 40
TASK_IN, TASK_OUT = 8 * 12 + 12, 6 + 8 * 6
LLT_SIZES = (3, 6, 12, 14, 18, 21)   # contact-space S (3 .. 12), UnParNMPC (14, 21), joint-space inertia (18)


# ---------------------------------------------------------------------------------------------------------------------
# the harness, built two ways
# ---------------------------------------------------------------------------------------------------------------------
def _emu_flags():
    """CXXFLAGS of tests/emu/Makefile, so that the harness is compiled like the emulator build of the kernels."""
    for line in open(os.path.join(EMU, "Makefile")):
        if line.startswith("CXXFLAGS"):
            return line.split(":=", 1)[1].split()
    raise RuntimeError("no CXXFLAGS in tests/emu/Makefile")


def _build(kind):
    os.makedirs(BUILD, exist_ok=True)
    if kind == "emu":
        out = os.path.join(BUILD, "libdevmath_emu.so")
        flags = [f for f in _emu_flags() if not f.startswith("-I")]
        cmd = ["g++"] + flags + ["-I" + EMU, "-I" + CSRC, "-shared", "-o", out, "-x", "c++", SRC,
                                 os.path.join(EMU, "cuda_emu.cpp")]
    else:
        sys.path.insert(0, ROOT)
        import __graft_entry__ as G
        out = os.path.join(BUILD, "libdevmath.so")
        cmd = [os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")] + G.NVCC_FLAGS + ["-I" + CSRC, "-o", out, SRC]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, " ".join(cmd) + "\n" + res.stdout + res.stderr
    return out


def _same(a, b):
    """bit-identical, except that any NaN matches any NaN (NaN payloads of constant-folded 0/0 differ by compiler)"""
    a, b = np.asarray(a, float), np.asarray(b, float)
    nan = np.isnan(a)
    return np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.int64), b[~nan].view(np.int64))


class Harness:
    """ctypes front of one build of devmath.cu.  With a `twin` (the emulator build), every call is repeated on the
    twin and the two results must agree bit for bit."""

    def __init__(self, path, twin=None):
        self.lib = ctypes.CDLL(path)
        self.twin = twin
        P = ctypes.POINTER(ctypes.c_double)
        for name, args in (("dm_scalar", [ctypes.c_int, P, P, ctypes.c_int]), ("dm_task", [P, P, ctypes.c_int]),
                           ("dm_llt", [ctypes.c_int, P, P, ctypes.c_int])):
            getattr(self.lib, name).argtypes = args
            getattr(self.lib, name).restype = ctypes.c_int
        assert self.lib.dm_num_fn() == NUM_FN

    @staticmethod
    def _p(a):
        return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))

    def _check_twin(self, method, out, *args):
        if self.twin is not None:
            ref = getattr(self.twin, method)(*args)
            assert _same(out, ref), "GPU and emulator builds differ in %s: %s" % (method, args[:1])

    def scalar(self, fn, rows, nout):
        rows = [np.atleast_1d(np.asarray(r, float)) for r in rows]
        inp = np.zeros((len(rows), DM_IN))
        for i, r in enumerate(rows):
            inp[i, :len(r)] = r
        out = np.zeros((len(rows), DM_OUT))
        assert self.lib.dm_scalar(fn, self._p(inp), self._p(out), len(rows)) == 0
        out = out[:, :nout].copy()
        self._check_twin("scalar", out, fn, rows, nout)
        return out

    def task(self, inp):
        inp = np.ascontiguousarray(inp, float).reshape(-1, TASK_IN)
        out = np.zeros((len(inp), TASK_OUT))
        assert self.lib.dm_task(self._p(inp), self._p(out), len(inp)) == 0
        self._check_twin("task", out, inp)
        return out

    def llt_raw(self, n, mats):
        mats = np.asarray(mats, float).reshape(-1, n, n)
        inp = np.ascontiguousarray(mats.transpose(0, 2, 1)).copy()   # column-major
        out = np.zeros((len(mats), 2 * n * n + n + 1))
        assert self.lib.dm_llt(n, self._p(inp), self._p(out), len(mats)) == 0
        self._check_twin("llt_raw", out, n, mats)
        return out

    def llt(self, n, mats):
        """column-major factor as left in A, pivot reciprocals, return value, inverse (column-major) of each matrix"""
        out = self.llt_raw(n, mats)
        fac = out[:, :n * n].reshape(-1, n, n).transpose(0, 2, 1)
        inv = out[:, n * n + n + 1:].reshape(-1, n, n).transpose(0, 2, 1)
        return fac, out[:, n * n:n * n + n], out[:, n * n + n].astype(int), inv


_BUILT = {}


@pytest.fixture(scope="module")
def emu():
    if "emu" not in _BUILT:
        _BUILT["emu"] = Harness(_build("emu"))
    return _BUILT["emu"]


@pytest.fixture(scope="module", params=["emu", pytest.param("gpu", marks=pytest.mark.gpu)])
def dev(request, emu):
    if request.param == "emu":
        return emu
    if "gpu" not in _BUILT:
        _BUILT["gpu"] = Harness(_build("gpu"), twin=emu)
    return _BUILT["gpu"]


# ---------------------------------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------------------------------
def ulp(y):
    return np.spacing(np.abs(np.asarray(y, float)))


def mpf_array(f, xs):
    return [f(mp.mpf(float(x))) for x in xs]


def hat6(nu):
    v, w = nu[:3], nu[3:]
    return mp.matrix([[0, -w[2], w[1], v[0]], [w[2], 0, -w[0], v[1]], [-w[1], w[0], 0, v[2]], [0, 0, 0, 0]])


def vee6(H):
    return [H[0, 3], H[1, 3], H[2, 3], H[2, 1], H[0, 2], H[1, 0]]


def exp6_mp(nu):
    return mp.expm(hat6([mp.mpf(x) for x in nu]))


@functools.lru_cache(maxsize=None)
def jexp6_mp(nu):
    """right Jacobian of exp6 at nu: column i = vee(T^-1 dT/dnu_i), dT/dnu_i by a central difference at h = 1e-20
    (truncation error h^2, 30 digits left after the cancellation at 50)"""
    nu = [mp.mpf(x) for x in nu]
    Ti = mp.inverse(mp.expm(hat6(nu)))
    h = mp.mpf("1e-20")
    J = mp.matrix(6, 6)
    for i in range(6):
        a, b = list(nu), list(nu)
        a[i] += h
        b[i] -= h
        col = vee6(Ti * (mp.expm(hat6(a)) - mp.expm(hat6(b))) / (2 * h))
        for r in range(6):
            J[r, i] = col[r]
    return J


def to_np(M):
    return np.array(M.tolist(), dtype=float)


def rot_R_p(T):
    return (np.array([[float(T[r, c]) for c in range(3)] for r in range(3)]),
            np.array([float(T[r, 3]) for r in range(3)]))


def unit(v):
    v = np.asarray(v, float)
    return v / np.linalg.norm(v)


# rotation angles at the branch points of log3 / Jlog3 / exp6 / Jexp3 (Taylor switch at eps^(1/4), pi switch at pi - 1e-2)
THETAS = [0.0, 1e-9, 1e-5, TAYLOR * (1 - 1e-3), TAYLOR * (1 + 1e-3), 2e-4, 1e-3, 1e-2, 0.5, 2.0,
          math.pi - 1e-2 - 1e-4, math.pi - 1e-2 + 1e-4, math.pi - 1e-4, math.pi - 1e-7, math.pi]


@functools.lru_cache(maxsize=None)
def se3_cases():
    """(nu, R, p): nu = [v; w] with |w| = theta on a random axis and a random translation, (R, p) = exp6(nu) at 50 digits
    rounded to doubles.  Two axes per angle, plus rotations by 2.5 and pi about each coordinate axis (trace <= 0)."""
    rng = np.random.default_rng(2024)
    nus = []
    for theta in THETAS:
        for _ in range(2):
            nus.append(np.concatenate([rng.uniform(-1, 1, 3), theta * unit(rng.normal(size=3))]))
    for ang in (2.5, math.pi):
        for ax in np.eye(3):
            nus.append(np.concatenate([rng.uniform(-1, 1, 3), ang * ax]))
    out = []
    for nu in nus:
        R, p = rot_R_p(exp6_mp(nu))
        out.append((nu, R, p))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# canonical arithmetic (octet.cuh)
# ---------------------------------------------------------------------------------------------------------------------
PIO2_HI, PIO2_LO = 1.57079632673412561417e+00, 6.07710050650619224932e-11   # canon_sincos's two-part pi/2


def _sincos_check(dev, xs):
    xs = np.asarray(xs, float)
    out = dev.scalar(SINCOS, xs, 2)
    rs, rc = np.array(mpf_array(mp.sin, xs), float), np.array(mpf_array(mp.cos, xs), float)
    # The reduced argument r = x - k pi/2 carries |k| |pi/2 - (hi + lo)| from the two-part constant and an ulp of r from
    # the two fmas; sin and cos have absolute condition 1 in r.  On top of that one ulp of the result.
    k = np.rint(xs * (2 / np.pi))
    dpi = abs(float(mp.pi / 2 - (mp.mpf(PIO2_HI) + mp.mpf(PIO2_LO))))
    r = np.array([float(mp.mpf(float(x)) - int(kk) * mp.pi / 2) for x, kk in zip(xs, k)])
    tol = ulp(np.maximum(np.abs(rs), np.abs(rc))) + ulp(r) + np.abs(k) * dpi
    es, ec = np.abs(out[:, 0] - rs), np.abs(out[:, 1] - rc)
    bad = np.flatnonzero((es > np.maximum(ulp(rs), tol)) | (ec > np.maximum(ulp(rc), tol)))
    assert bad.size == 0, [(xs[i], out[i], rs[i], rc[i]) for i in bad[:5]]
    return out, rs, rc


def test_canon_sincos_random_and_joint_ranges(dev):
    rng = np.random.default_rng(1)
    xs = np.concatenate([rng.uniform(-1e9, 1e9, 1500), rng.uniform(-1e3, 1e3, 500),
                         rng.uniform(-3.05, 3.05, 500), rng.uniform(-9.42, 9.42, 500)])   # iiwa14 / ANYmal joint ranges
    out, rs, rc = _sincos_check(dev, xs)
    small = np.abs(xs) <= 10   # within the joint ranges both results are within one ulp
    assert np.all(np.abs(out[small, 0] - rs[small]) <= ulp(rs[small]))
    assert np.all(np.abs(out[small, 1] - rc[small]) <= ulp(rc[small]))


def test_canon_sincos_multiples_of_half_pi(dev):
    k = np.arange(-200, 201)
    _sincos_check(dev, np.concatenate([k * (np.pi / 2), np.nextafter(k * (np.pi / 2), np.inf)]))


def test_canon_sincos_quadrant_beyond_int_range(dev):
    """k = rint(x 2/pi) passes 2^31 at |x| = 2^31 pi/2 ~ 3.37e9: the quadrant must still be k mod 4"""
    rng = np.random.default_rng(2)
    edge = 2.0 ** 31 * np.pi / 2
    xs = np.concatenate([[5e9, -5e9, edge, -edge, 2 * edge, 1e12, -1e12, 2.0 ** 40, 3e15],
                         rng.uniform(edge, 4e9, 200), -rng.uniform(edge, 1e12, 200)])
    out, rs, rc = _sincos_check(dev, xs)
    assert np.all(np.sign(out[:, 0]) == np.sign(rs)) and np.all(np.sign(out[:, 1]) == np.sign(rc))


def _log_ref(xs):
    return np.array([float(mp.log(mp.mpf(float(x)))) for x in xs])


def test_canon_log_normals(dev):
    rng = np.random.default_rng(3)
    k = np.arange(1, 53)
    # the sqrt(2) switch of the reduction: high mantissa word 0x6a09c / 0x6a09d (hx + 0x95f64 carries into bit 20)
    sw = [np.ldexp(1.0 + (0x6a09c + d) / 2.0 ** 20 + j * 2.0 ** -52, e)
          for d in (-1, 0, 1) for j in (0, 1, 2 ** 32 - 1) for e in (-1000, -1, 0, 1, 1000)]
    xs = np.concatenate([np.exp(rng.uniform(-708, 709, 3000)), 1 + np.ldexp(1.0, -k), 1 - np.ldexp(1.0, -k),
                         np.ldexp(1.0, np.arange(-1022, 1024, 7)), sw, [np.finfo(float).max, np.finfo(float).tiny, 2.0]])
    y = dev.scalar(LOG, xs, 1)[:, 0]
    ref = _log_ref(xs)
    assert np.all(np.abs(y - ref) <= ulp(ref)), np.max(np.abs(y - ref) / np.maximum(ulp(ref), 1e-300))


def test_canon_log_subnormals_and_specials(dev):
    sub = np.array([5e-324, 1e-323, 1e-320, 1e-310, 2.2250738585072009e-308, np.finfo(float).tiny / 3])
    y = dev.scalar(LOG, sub, 1)[:, 0]
    ref = _log_ref(sub)
    assert np.all(np.abs(y - ref) <= ulp(ref)), (y, ref)
    sp = np.array([0.0, -0.0, -1.0, -5e-324, -np.inf, np.nan, np.inf])
    y = dev.scalar(LOG, sp, 1)[:, 0]
    with np.errstate(divide="ignore", invalid="ignore"):
        assert _same(y, np.log(sp)), y


def test_canon_rsqrt_within_one_ulp(dev):
    rng = np.random.default_rng(4)
    lo, hi = np.nextafter(1e-36, np.inf), np.nextafter(1e36, 0.0)
    xs = np.concatenate([10.0 ** rng.uniform(-36, 36, 6000), rng.uniform(0.5, 4.0, 1000), [lo, hi, 1.0, 2.0, 4.0, 0.25]])
    y = dev.scalar(RSQRT, xs, 1)[:, 0]
    ref = np.array([float(1 / mp.sqrt(mp.mpf(float(x)))) for x in xs])
    assert np.all(np.abs(y - ref) <= ulp(ref))


def test_canon_pivot_ok_boundaries(dev):
    xs = np.array([1e-36, np.nextafter(1e-36, np.inf), 1e36, np.nextafter(1e36, 0.0), 1.0, 0.0, -1.0, 5e-324,
                   np.inf, -np.inf, np.nan, np.nextafter(1e-36, 0.0), np.nextafter(1e36, np.inf)])
    ok = dev.scalar(PIVOT_OK, xs, 1)[:, 0]
    assert list(ok) == [0, 1, 0, 1, 1, 0, 0, 0, 0, 0, 0, 0, 0]


def test_canon_acos(dev):
    k = np.arange(1, 53)
    xs = np.concatenate([np.linspace(-1, 1, 4001), 1 - np.ldexp(1.0, -k), -1 + np.ldexp(1.0, -k),
                         [0.5, -0.5, np.nextafter(0.5, 0), np.nextafter(-0.5, 0), 1.0, -1.0]])
    y = dev.scalar(ACOS, xs, 1)[:, 0]
    ref = np.array([float(mp.acos(mp.mpf(float(x)))) for x in xs])
    assert np.all(np.abs(y - ref) <= ulp(ref))
    # outside [-1, 1] the argument is clamped (log3 of a rotation matrix whose trace rounds past 3 or -1)
    y = dev.scalar(ACOS, [1.5, np.nextafter(1.0, 2.0), np.inf, -1.5, np.nextafter(-1.0, -2.0), -np.inf, np.nan], 1)[:, 0]
    assert list(y[:6]) == [0.0, 0.0, 0.0, 3.14159265358979311600, 3.14159265358979311600, 3.14159265358979311600]
    assert np.isnan(y[6])


# ---------------------------------------------------------------------------------------------------------------------
# SE(3) (fb_math.cuh, task_space_cost.cuh)
# ---------------------------------------------------------------------------------------------------------------------
def _delta(theta):
    return max(math.pi - theta, 1e-300)


def log6_tol(theta, p):
    """max-abs bound of log6 at a rotation angle theta, translation p, against the log of the unrounded placement"""
    s = 1.0 + float(np.abs(p).max())
    if theta < TAYLOR:
        # the Taylor branch of log3 takes theta / sin(theta) = 1: relative error theta^2 / 6 in w, ~ |p| theta^3 / 12 in v
        return theta ** 3 / 6 * s + 4 * EPS * s
    if theta < math.pi - 1e-2:
        # theta = acos of the trace, then theta / sin(theta): near pi the error of sin(theta) is cot(theta) eps / delta
        return 2 * EPS * s * (1 + _delta(theta) ** -2)
    # the rounded input itself moves the axis by eps / delta; at pi the axis components come from square roots of the
    # diagonal, so a component near zero is known to sqrt(eps)
    return 2 * EPS * s + 4 * s * min(EPS / _delta(theta), math.sqrt(EPS))


def jlog6_tol(theta, p):
    """relative (to max(1, max|J|)) bound of Jlog6"""
    s = 1.0 + float(np.abs(p).max())
    if theta < TAYLOR:
        return theta ** 3 / 6 * s + 4 * EPS * s
    if theta < math.pi - 1e-2:
        return 4 * EPS * s * (1 / theta + _delta(theta) ** -2)   # acos of the trace: relative error eps / theta in theta
    return 4 * EPS * s * (1 + 1 / _delta(theta))


def jexp6_tol(theta, v):
    s = 1.0 + float(np.abs(v).max())
    if theta < TAYLOR:
        # Jexp3's Taylor branch: b = -1/2 - n^2/24 where the series has -1/2 + n^2/24 (the port's formula), error n^3 / 12
        return theta ** 3 / 6 * s + 4 * EPS * s
    # B = -A C with C built from beta = 1/theta^2 - sin/(2 theta (1 - cos)) at theta = |w|: 1 - cos(theta) is rounded
    # independently of theta, relative error eps / theta^2, times 1 / theta^2 and |w| |p| ~ theta: eps / theta^3
    return 4 * EPS * s * (1 + theta ** -3)


def _log6_reference(nu, R, p, out):
    """reference log of the placement: nu itself, except at theta = pi where +-w are both logs and |nu_w| may have rounded
    past pi: there the kernel's own output is checked by exponentiating it back.  Returns None at theta = pi about an
    axis with more than one non-zero component: log3 takes the sign of each component from R - R^T, which is rounding
    noise at pi (upstream's formula), so only |w_i| is determined; the caller checks that."""
    theta = float(np.linalg.norm(nu[3:]))
    if theta < math.pi - 1e-9:
        return nu, theta
    if np.count_nonzero(nu[3:]) > 1:
        assert np.abs(np.abs(out[3:]) - np.abs(nu[3:])).max() <= log6_tol(theta, p)
        return None, theta
    T = exp6_mp(out)
    Rr, pr = rot_R_p(T)
    assert np.abs(Rr - R).max() <= log6_tol(theta, p) and np.abs(pr - p).max() <= log6_tol(theta, p)
    return out, theta


def test_fb_log6_exp6(dev):
    cases = se3_cases()
    log = dev.scalar(FB_LOG6, [np.concatenate([R.ravel(), p]) for _, R, p in cases], 6)
    exp = dev.scalar(FB_EXP6, [nu for nu, _, _ in cases], 12)
    for (nu, R, p), o, e in zip(cases, log, exp):
        ref, theta = _log6_reference(nu, R, p, o)
        assert ref is None or np.abs(o - ref).max() <= log6_tol(theta, p), (theta, o - ref)
        Rr, pr = rot_R_p(exp6_mp(nu))   # exp6 of the double input: a well-conditioned map
        s = 1 + np.abs(nu).max()
        assert np.abs(e[:9] - Rr.ravel()).max() <= 4 * EPS, theta
        # alpha_w = (1 - sin(t) / t) / t^2 cancels for t above the Taylor switch: eps / t^2, times (w . v) ~ t
        assert np.abs(e[9:] - pr).max() <= 4 * EPS * s * (1 + 1 / max(theta, TAYLOR)), theta


def test_fb_jlog6_jexp6(dev):
    cases = se3_cases()
    log = dev.scalar(FB_LOG6, [np.concatenate([R.ravel(), p]) for _, R, p in cases], 6)
    jl = dev.scalar(FB_JLOG6, [np.concatenate([R.ravel(), p]) for _, R, p in cases], 36).reshape(-1, 6, 6)
    je = dev.scalar(FB_JEXP6, [nu for nu, _, _ in cases], 36).reshape(-1, 6, 6)
    dv = dev.scalar(FB_DINTEGRATE_DV, [nu for nu, _, _ in cases], 36).reshape(-1, 6, 6)
    assert _same(dv, je)   # dIntegratedVelocity is Jexp6
    for (nu, R, p), o, Jl, Je in zip(cases, log, jl, je):
        ref, theta = _log6_reference(nu, R, p, o)
        Jeref = to_np(jexp6_mp(tuple(nu)))
        assert np.abs(Je - Jeref).max() / max(1, np.abs(Jeref).max()) <= jexp6_tol(theta, nu[:3]), theta
        if ref is not None:
            Jlref = to_np(mp.inverse(jexp6_mp(tuple(float(x) for x in ref))))
            assert np.abs(Jl - Jlref).max() / max(1, np.abs(Jlref).max()) <= jlog6_tol(theta, p), theta


def test_log3_of_the_task_cost_equals_fb_log3(dev):
    """task_space_cost.cuh restates log3 / Jlog3 with its own threshold TASK_TAYLOR; fb_math.cuh's are pinned above"""
    cases = se3_cases()
    a = dev.scalar(LOG3_CANON, [R.ravel() for _, R, _ in cases], 4)
    b = dev.scalar(FB_LOG3, [R.ravel() for _, R, _ in cases], 4)
    assert _same(a, b)
    thw = [np.concatenate([[t], unit(nu[3:]) * t if t > 0 else np.zeros(3)])
           for nu in (c[0] for c in cases) for t in [np.linalg.norm(nu[3:])]]
    assert _same(dev.scalar(JLOG3_CANON, thw, 9), dev.scalar(FB_JLOG3, thw, 9))


def _quat_mp(axis, ang):
    return [mp.sin(mp.mpf(ang) / 2) * a for a in axis] + [mp.cos(mp.mpf(ang) / 2)]


def test_fb_quaternion_conversions(dev):
    """R_to_quat's four branches: trace > 0, and trace <= 0 with the largest diagonal entry at x, y or z"""
    cases = [(unit(a), ang) for ang in (0.3, 2.0, 2.5, 3.0, math.pi)
             for a in ([1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 0.2, -0.1], [0.1, -1, 0.3], [-0.2, 0.1, 1], [1, 1, 1])]
    R = []
    for axis, ang in cases:
        T = mp.expm(hat6([0, 0, 0] + [mp.mpf(float(a)) * mp.mpf(ang) for a in axis]))
        R.append(rot_R_p(T)[0].ravel())
    q = dev.scalar(FB_R_TO_QUAT, R, 4)
    for (axis, ang), qq in zip(cases, q):
        ref = np.array([float(x) for x in _quat_mp([mp.mpf(float(a)) for a in axis], ang)])
        assert min(np.abs(qq - ref).max(), np.abs(qq + ref).max()) <= 4 * EPS, (axis, ang, qq, ref)
    qs = [np.array([float(x) for x in _quat_mp([mp.mpf(float(a)) for a in axis], ang)]) for axis, ang in cases]
    Rq = dev.scalar(FB_QUAT_TO_R, qs, 9)
    for qq, r in zip(qs, Rq):
        x, y, z, w = [mp.mpf(float(t)) for t in qq]
        ref = [1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w), 2 * (x * y + z * w), 1 - 2 * (x * x + z * z),
               2 * (y * z - x * w), 2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]
        assert np.abs(r - np.array(ref, float)).max() <= 4 * EPS


def test_fb_inv33_and_dsubtract_inverse(dev):
    rng = np.random.default_rng(5)
    As = [rng.normal(size=(3, 3)) + 3 * np.eye(3) for _ in range(20)] + [np.diag([1e-8, 1.0, 1e8])]
    Ai = dev.scalar(FB_INV33, [A.ravel() for A in As], 9)
    for A, X in zip(As, Ai):
        ref = to_np(mp.inverse(mp.matrix(A.tolist())))
        assert np.abs(X - ref.ravel()).max() <= 8 * EPS * np.linalg.cond(A) * np.abs(ref).max()
    cases = [c for c in se3_cases() if np.linalg.norm(c[0][3:]) < 3.0]
    J = dev.scalar(FB_JLOG6, [np.concatenate([R.ravel(), p]) for _, R, p in cases], 36)
    Ji = dev.scalar(FB_DSUBTRACT_INVERSE, J, 36)
    for j, ji in zip(J, Ji):
        ref = to_np(mp.inverse(mp.matrix(j.reshape(6, 6).tolist())))
        assert np.abs(ji.reshape(6, 6) - ref).max() <= 64 * EPS * np.linalg.cond(j.reshape(6, 6)) * np.abs(ref).max()


def _quat_of(nu_w):
    theta = float(np.linalg.norm(nu_w))
    axis = [mp.mpf(float(a)) / mp.mpf(theta) for a in nu_w] if theta > 0 else [mp.mpf(0)] * 3
    return np.array([float(x) for x in _quat_mp(axis, theta)])


def test_fb_integrate_subtract_round_trip(dev):
    """q (+) alpha v (-) q = alpha v on the base across the Taylor threshold; the subtract Jacobians against the
    reference Jlog6 and adjoint"""
    rng = np.random.default_rng(6)
    rows, nus = [], []
    for theta in [0.0, 1e-9, 1e-5, TAYLOR * (1 - 1e-3), TAYLOR * (1 + 1e-3), 2e-4, 1e-2, 0.5, 2.0, 3.0]:
        q = np.concatenate([rng.uniform(-1, 1, 3), _quat_of(rng.uniform(-2, 2, 3)), rng.uniform(-1, 1, 12)])
        v = np.concatenate([rng.uniform(-1, 1, 3), theta * unit(rng.normal(size=3)), rng.uniform(-1, 1, 12)])
        for alpha in (1.0, 0.5):
            rows.append(np.concatenate([q, v / alpha if alpha != 1.0 else v, [alpha]]))
            nus.append(v[:6])
    qo = dev.scalar(FB_INTEGRATE, rows, 19)
    diff = dev.scalar(FB_SUBTRACT, [np.concatenate([a, r[:19]]) for a, r in zip(qo, rows)], 18)
    for r, a, d, nu in zip(rows, qo, diff, nus):
        theta = float(np.linalg.norm(nu[3:]))
        assert abs(np.linalg.norm(a[3:7]) - 1) <= 4 * EPS
        # exp6 (its translation loses eps / theta above the Taylor switch, see test_fb_log6_exp6), two products by the
        # base rotation and a quaternion round trip on top of the log
        s = 1 + np.abs(r[:3]).max() + np.abs(nu[:3]).max()
        tol = log6_tol(theta, nu[:3]) + 16 * EPS * s * (1 + 1 / max(theta, TAYLOR))
        assert np.abs(d[:6] - nu).max() <= tol, (theta, d[:6] - nu)
        assert np.abs(d[6:] - r[19 + 6:19 + 18] * r[-1]).max() <= 4 * EPS
    # Jacobians at q_plus = q (+) nu, q_minus = q
    pairs = [np.concatenate([a, r[:19]]) for a, r in zip(qo, rows)]
    jp = dev.scalar(FB_DSUBTRACT_DPLUS, pairs, 36).reshape(-1, 6, 6)
    jm = dev.scalar(FB_DSUBTRACT_DMINUS, pairs, 36).reshape(-1, 6, 6)
    for nu, p_, m_ in zip(nus, jp, jm):
        theta = float(np.linalg.norm(nu[3:]))
        Jl = to_np(mp.inverse(jexp6_mp(tuple(nu))))
        tol = jlog6_tol(theta, nu[:3]) + 64 * EPS
        assert np.abs(p_ - Jl).max() / max(1, np.abs(Jl).max()) <= tol, theta
        Ti = mp.inverse(exp6_mp(nu))
        Ad = mp.zeros(6, 6)
        for i in range(3):
            for j in range(3):
                Ad[i, j] = Ad[3 + i, 3 + j] = Ti[i, j]
        P = mp.matrix([[0, -Ti[2, 3], Ti[1, 3]], [Ti[2, 3], 0, -Ti[0, 3]], [-Ti[1, 3], Ti[0, 3], 0]]) * Ti[0:3, 0:3]
        for i in range(3):
            for j in range(3):
                Ad[i, 3 + j] = P[i, j]
        ref = -to_np(mp.matrix(Jl.tolist()) * Ad)
        assert np.abs(m_ - ref).max() / max(1, np.abs(ref).max()) <= 4 * tol, theta
    dq = dev.scalar(FB_DINTEGRATE_DQ, nus, 36).reshape(-1, 6, 6)
    for nu, d in zip(nus, dq):
        Ti = mp.inverse(exp6_mp(nu))
        Ri, pi = rot_R_p(Ti)
        ref = np.zeros((6, 6))
        ref[:3, :3] = ref[3:, 3:] = Ri
        ref[:3, 3:] = np.array([[0, -pi[2], pi[1]], [pi[2], 0, -pi[0]], [-pi[1], pi[0], 0]]) @ Ri
        assert np.abs(d - ref).max() <= 16 * EPS * (1 + np.abs(nu).max()) * (1 + 1 / max(np.linalg.norm(nu[3:]), TAYLOR))


def test_task_evaluate(dev):
    """the pose error of the 6D task cost and its JJ columns, octet-parallel: lane 6 carries the end-effector pose"""
    rng = np.random.default_rng(7)
    perm = np.array([[0.0, -1.0, 0.0], [0.0, 0.0, 1.0], [-1.0, 0.0, 0.0]])   # exact rotation: the reference's R^T is exact
    rows, refs = [], []
    for nu, _, _ in se3_cases():
        if np.linalg.norm(nu[3:]) >= math.pi - 1e-9:
            continue
        pref = rng.uniform(-1, 1, 3)
        Tref = mp.matrix(4, 4)
        for i in range(3):
            for j in range(3):
                Tref[i, j] = perm[i, j]
            Tref[i, 3] = pref[i]
        Tref[3, 3] = 1
        R6, p6 = rot_R_p(Tref * exp6_mp(nu))
        lanes = []
        for l in range(8):
            if l == 6:
                lanes.append(np.concatenate([R6.ravel(), p6]))
            else:
                Rl, _ = rot_R_p(mp.expm(hat6([0, 0, 0] + list(rng.normal(size=3)))))
                lanes.append(np.concatenate([Rl.ravel(), rng.uniform(-1, 1, 3)]))
        rows.append(np.concatenate(lanes + [perm.ravel(), pref]))
        refs.append(nu)
    out = dev.task(np.array(rows))
    for row, nu, o in zip(rows, refs, out):
        theta = float(np.linalg.norm(nu[3:]))
        s = 1 + np.abs(nu[:3]).max()
        assert np.abs(o[:6] - nu).max() <= log6_tol(theta, nu[:3]) + 8 * EPS * s, theta
        Jl = mp.inverse(jexp6_mp(tuple(nu)))
        R6 = mp.matrix(row[72:81].reshape(3, 3).tolist())
        pf = mp.matrix(row[81:84].tolist())
        for l in range(8):
            z = mp.matrix(row[12 * l:12 * l + 9].reshape(3, 3)[:, 2].tolist())
            pl = mp.matrix(row[12 * l + 9:12 * l + 12].tolist())
            d = pf - pl
            lin = R6.T * mp.matrix([z[1] * d[2] - z[2] * d[1], z[2] * d[0] - z[0] * d[2], z[0] * d[1] - z[1] * d[0]])
            ang = R6.T * z
            col = to_np(Jl * mp.matrix([lin[0], lin[1], lin[2], ang[0], ang[1], ang[2]])).ravel()
            JJ = o[6 + 6 * l:12 + 6 * l]
            assert np.abs(JJ - col).max() / max(1, np.abs(col).max()) <= 4 * (jlog6_tol(theta, nu[:3]) + 8 * EPS * s), (theta, l)


# ---------------------------------------------------------------------------------------------------------------------
# warp Cholesky (warp_llt.cuh)
# ---------------------------------------------------------------------------------------------------------------------
def spd(n, kappa, rng):
    Q, _ = np.linalg.qr(rng.normal(size=(n, n)))
    lam = np.geomspace(1.0, 1.0 / kappa, n) if n > 1 else np.ones(1)
    A = (Q * lam) @ Q.T
    return (A + A.T) / 2


@pytest.mark.parametrize("n", LLT_SIZES)
def test_warp_llt_backward_and_inverse_error(dev, n):
    rng = np.random.default_rng(100 + n)
    kappas = (1.0, 1e4, 1e8, 1e12)
    mats = [spd(n, k, rng) for k in kappas]
    fac, rd, fail, inv = dev.llt(n, mats)
    assert np.all(fail == 0)
    for A, Lraw, r, X, kappa in zip(mats, fac, rd, inv, kappas):
        L = np.tril(Lraw)
        Am = mp.matrix(A.tolist())
        Lm = mp.matrix(L.tolist())
        nA = mp.mnorm(Am, 1)
        assert mp.mnorm(Lm * Lm.T - Am, 1) / nA <= 2 * n * EPS, kappa
        assert np.all(np.abs(r * np.diag(L) - 1) <= 4 * EPS)   # rd = 1 / L_kk within a few ulps
        Ainv = mp.inverse(Am)
        assert mp.mnorm(mp.matrix(X.tolist()) - Ainv, 1) / mp.mnorm(Ainv, 1) <= 4 * n * kappa * EPS, kappa


@pytest.mark.parametrize("n", LLT_SIZES)
def test_warp_llt_reads_only_the_lower_triangle(dev, n):
    rng = np.random.default_rng(200 + n)
    A = spd(n, 1e4, rng)
    B = A.copy()
    B[np.triu_indices(n, 1)] = np.nan
    fa, ra, ka, ia = dev.llt(n, [A])
    fb, rb, kb, ib = dev.llt(n, [B])
    low = np.tril_indices(n)
    assert _same(fa[0][low], fb[0][low]) and _same(ra, rb) and _same(ka, kb) and _same(ia, ib)


@pytest.mark.parametrize("n", LLT_SIZES)
def test_warp_llt_reports_the_first_bad_pivot(dev, n):
    rng = np.random.default_rng(300 + n)
    mats, expect = [], []
    for k in sorted({0, n // 2, n - 1}):
        A = spd(n, 10.0, rng)
        piv = float(A[k, k] - A[k, :k] @ np.linalg.solve(A[:k, :k], A[:k, k])) if k else float(A[0, 0])
        A[k, k] -= piv + 1.0   # pivot k becomes -1, the leading k x k block stays positive definite
        mats.append(A)
        expect.append(k + 1)
    # pivots outside (1e-36, 1e36) fail as well (the single-precision seed of canon_rsqrt would vanish or overflow)
    A = spd(n, 10.0, rng)
    mats += [A * 1e-37, A * 1e37]
    expect += [1, 1]
    D = np.eye(n)
    D[n - 1, n - 1] = 1e-37
    mats.append(D)
    expect.append(n)
    _, _, fail, _ = dev.llt(n, mats)
    assert list(fail) == expect


# ---------------------------------------------------------------------------------------------------------------------
# interior point (pdipm.cuh)
# ---------------------------------------------------------------------------------------------------------------------
def test_pdipm_fraction_row(dev):
    rows = [(0.995, 1.0, 0.0, 1.0), (0.995, 1.0, -0.0, 1.0), (0.995, 1.0, 2.0, 1.0), (0.995, 1.0, 1e-300, 0.7),
            (0.5, 2.0, -1.0, 1.0),            # lands exactly on the boundary: f = 1 does not count
            (0.995, 1.0, -4.0, 1.0), (0.995, 1.0, -4.0, 0.1), (0.995, 3.0, -7.0, 0.9), (0.995, 1e-300, -1e-10, 1.0),
            (0.995, 0.3, -0.1, 1.0)]         # f > 1
    y = dev.scalar(FRACTION_ROW, rows, 1)[:, 0]
    for (rate, x, dx, cur), got in zip(rows, y):
        if dx == 0.0:
            ref = cur
        else:
            f = -Fraction(rate) * (Fraction(x) / Fraction(dx))
            ref = float(f) if 0 < f < 1 and f < Fraction(cur) else cur
        assert abs(got - ref) <= ulp(ref), (rate, x, dx, cur, got, ref)
