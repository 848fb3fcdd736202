"""The hand-written device math routines, run on the GPU and compared with high-precision references.

Every parity claim of the tracer rests on a few device routines written for speed (csrc/lp_sincr.cuh,
lp_internal.cuh, lp_remap.cuh).  The end-to-end tests cannot stand in for direct tests of them: their
allowances (a sine moved one ulp for up to 1 % of a batch, one-float32-step flips near rounding boundaries,
whole-trajectory comparisons) would absorb a routine that is slightly wrong.  Here each routine runs
elementwise on the device (tests/device_math_probe.cu, compiled with the library's own NVCC_FLAGS, so with
-fmad=false like the library) over inputs chosen where such routines go wrong — table knots, branch
switches, exponent limits, multiples of pi, clamp edges — and is compared with mpmath at 200 bits rounded
once to double (or, for the integer results, with the reference's own integer arithmetic).

The bars are the routines' documented contracts, tightened to the worst case measured on a B200 rounded up
to the next 0.25 ulp (so that a regression fails; the constants below carry both numbers).  Each test
prints the worst case it measured.

One bar is stated on a different scale from the coordinate contract's plain "1e-12 relative": the pinhole
coordinate px = fx sx / sz + W/2 of source_coords_xy.  The direction (sx, sy, sz) is a sum of products of
O(1) factors (cos / sin of the viewing angle and of the screen angle), so any double evaluation of it —
the reference's numpy one included — carries an absolute error of a few 1e-16, which the division by sz
amplifies by 1/sz.  The bar is therefore 1e-12 max(1, |p|) plus that conditioning term,
4 eps f (1 + |sx / sz|) / sz with eps = 2^-53; for sz above ~1e-3 the extra term is below the plain bar.
"""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROBE_SRC = os.path.join(ROOT, "tests", "device_math_probe.cu")

PREC = 200
EPS = 2.0 ** -53
PI_HI = float.fromhex("0x1.921fb54442d18p+1")        # np.pi

# bars (see the module docstring)
SIN_CR_NEAR_MIDPOINT = 2.0 ** -14      # ulp: where correct rounding may be missed
SIN_CR_MAX_EXCEPTIONS = 2
# measured on an NVIDIA B200 (power limit 1000 W) over the inputs below, and rounded up to the next 0.25 ulp:
LIBM_SIN_ULP = 1.5                     # CUDA sin on pi < |x| <= 10 (its contract: 2 ulp); measured 1.269
LIBM_ACOS_ULP = 1.5                    # CUDA acos on |x| <= 0.5625 (contract: 2 ulp); measured 1.387
ACOS_ULP = 0.75                        # contract < 0.75 (tools/acos_study.c); measured 0.651
SINCOS_ABS = 1.5 * 2.0 ** -53          # contract 2^-52; measured 1.423 x 2^-53
SINCOS_REL_ULP = 1.5                   # where |result| >= 2^-10; measured 1.423
INV_TENTH_ULP = 1.0                    # contract "a few ulp" (3); measured 0.995
RCP_ULP = 0.75                         # contract 2 ulp; measured 0.500
RSQRT_ULP = 1.25                       # contract 2 ulp; measured 1.000
COORD_REL = 1e-12


# ---------------------------------------------------------------------------------------------------------
# the probe
# ---------------------------------------------------------------------------------------------------------
class _Probe:
    """ctypes launchers of tests/device_math_probe.cu, driven with torch CUDA tensors (numpy in, numpy out)."""

    _UNARY = {"sin_cr": "f8", "acos_unit": "f8", "inv_tenth_root": "f8", "fast_rcp": "f8", "fast_rsqrt": "f8",
              "mid_range": "i4", "half_orbits": "i8", "half_orbits_fast": "i8", "half_orbits_quadrant": "i8"}

    def __init__(self, so_path, native):
        import torch
        self.torch = torch
        self.lib = ctypes.CDLL(so_path)
        vp, i64 = ctypes.c_void_p, ctypes.c_longlong
        for name in self._UNARY:
            fn = getattr(self.lib, "probe_" + name)
            fn.restype, fn.argtypes = ctypes.c_int, [vp, vp, i64, vp]
        fn = self.lib.probe_sincos_moderate
        fn.restype, fn.argtypes = ctypes.c_int, [vp, vp, vp, vp, vp, i64, vp]
        fn = self.lib.probe_source_coords
        fn.restype = ctypes.c_int
        fn.argtypes = [ctypes.POINTER(native.lp_camera), ctypes.c_int] + [vp] * 9 + [i64, vp]

    def _dev(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a)).cuda()

    def _out(self, n, dtype):
        return self.torch.empty(n, dtype=getattr(self.torch, {"f8": "float64", "i4": "int32", "i8": "int64"}[dtype]),
                                device="cuda")

    def _call(self, fn, *args):
        stream = self.torch.cuda.current_stream().cuda_stream
        rc = fn(*[a.data_ptr() if hasattr(a, "data_ptr") else a for a in args], stream)
        assert rc == 0, "probe launch failed: %d" % rc
        self.torch.cuda.synchronize()

    def unary(self, name, x):
        x = np.asarray(x, dtype=np.float64)
        dx, dy = self._dev(x), self._out(x.size, self._UNARY[name])
        self._call(getattr(self.lib, "probe_" + name), dx, dy, x.size)
        return dy.cpu().numpy()

    def sincos_moderate(self, x):
        x = np.asarray(x, dtype=np.float64)
        dx = self._dev(x)
        s, c, r, q = self._out(x.size, "f8"), self._out(x.size, "f8"), self._out(x.size, "f8"), self._out(x.size, "i4")
        self._call(self.lib.probe_sincos_moderate, dx, s, c, q, r, x.size)
        return s.cpu().numpy(), c.cpu().numpy(), q.cpu().numpy(), r.cpu().numpy()

    def source_coords(self, cam, direct, xc, yc, fa32, fa64=None, cfa=None, sfa=None):
        n = len(xc)
        zeros = np.zeros(n)
        ins = [self._dev(np.asarray(a, dtype=t)) for a, t in
               ((xc, np.float64), (yc, np.float64), (fa32, np.float32), (zeros if fa64 is None else fa64, np.float64),
                (zeros if cfa is None else cfa, np.float64), (zeros if sfa is None else sfa, np.float64))]
        px, py, front = self._out(n, "f8"), self._out(n, "f8"), self._out(n, "i4")
        self._call(self.lib.probe_source_coords, ctypes.byref(cam), int(direct), *ins, px, py, front, n)
        return px.cpu().numpy(), py.cpu().numpy(), front.cpu().numpy().astype(bool)


@pytest.fixture(scope="module")
def probe(native, tmp_path_factory):
    from light_path_tracer_b200 import build as b
    so = str(tmp_path_factory.mktemp("device_math") / "device_math_probe.so")
    cmd = [b._nvcc()] + b.NVCC_FLAGS + ["-shared", "-Xcompiler", "-fPIC", "-I" + b.CSRC, PROBE_SRC, "-o", so,
                                        "-L" + b.OUT, "-llightpath", "-Xlinker", "-rpath," + b.OUT]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    return _Probe(so, native)


# ---------------------------------------------------------------------------------------------------------
# references and error measures
# ---------------------------------------------------------------------------------------------------------
def _mp():
    import mpmath
    return mpmath


def _ulp(e):
    """ulp of the double nearest to the (non-zero) exact value e."""
    mp = _mp()
    _, ex = mp.frexp(e)                         # |e| = m 2^ex, 1/2 <= m < 1
    return mp.ldexp(1, max(int(ex), -1021) - 53)


def _ulp_err(got, exact):
    """|got - exact| in ulps of exact (both lists; exact entries are mpf)."""
    mp = _mp()
    out = np.empty(len(got))
    with mp.workprec(PREC):
        for i, (g, e) in enumerate(zip(got, exact)):
            if e == 0:
                out[i] = 0.0 if g == 0 else np.inf
            elif not math.isfinite(g):
                out[i] = np.inf
            else:
                out[i] = float(abs(mp.mpf(float(g)) - e) / _ulp(e))
    return out


def _exact(fn, xs):
    mp = _mp()
    with mp.workprec(PREC):
        return [fn(mp.mpf(float(x))) for x in xs]


def _around(x, k):
    """the doubles within +-k ulp of each x (sorted, unique)"""
    x = np.atleast_1d(np.asarray(x, dtype=np.float64))
    out = [x]
    up, dn = x.copy(), x.copy()
    for _ in range(k):
        up, dn = np.nextafter(up, np.inf), np.nextafter(dn, -np.inf)
        out += [up, dn]
    return np.unique(np.concatenate(out))


def _report(name, text):
    print("\ndevice math | %-22s | %s" % (name, text))


# ---------------------------------------------------------------------------------------------------------
# lp_sin_cr
# ---------------------------------------------------------------------------------------------------------
def _sin_cr_inputs(rng):
    """non-negative normal arguments of the correctly rounded range [2^-26 - 20 ulp, pi_hi]"""
    k = np.arange(403)
    parts = [rng.uniform(0.0, np.pi, 12000),
             rng.uniform(0.0, np.pi, 12000).astype(np.float32).astype(np.float64),
             _around(np.concatenate([k / 256.0, (k + 0.5) / 256.0]), 3),
             _around([2.0 ** -26, 1.5707963267948966, PI_HI], 20)]
    x = np.unique(np.concatenate(parts))
    return x[(x > 0.0) & (x <= PI_HI)]


def test_sin_cr(probe):
    """lp_sin_cr: bit-identical to the correctly rounded sine on [-pi, pi] except within 2^-14 ulp of a
    half-way point (at most two such inputs); CUDA sin (contract 2 ulp) beyond; +-0 keep their sign."""
    mp = _mp()
    rng = np.random.default_rng(20261021)
    x = _sin_cr_inputs(rng)
    exact = _exact(mp.sin, x)
    ref = np.array([float(e) for e in exact])
    mid_dist = np.empty(x.size)
    with mp.workprec(PREC):
        for i, e in enumerate(exact):
            pos = abs(e) / _ulp(e)
            mid_dist[i] = float(abs(pos - mp.floor(pos) - mp.mpf(0.5)))
    got = probe.unary("sin_cr", np.concatenate([x, -x]))
    gp, gn = got[:x.size], got[x.size:]
    assert np.array_equal(gn, -gp), "lp_sin_cr is not odd"
    bad = gp != ref
    exceptions = int(np.count_nonzero(bad))
    assert not np.any(bad & (mid_dist >= SIN_CR_NEAR_MIDPOINT)), \
        "not correctly rounded at %s" % [(float.hex(v), float.hex(g), float.hex(r))
                                         for v, g, r in zip(x[bad][:8], gp[bad][:8], ref[bad][:8])]
    assert exceptions <= SIN_CR_MAX_EXCEPTIONS
    worst_range = float(np.max(_ulp_err(gp, exact)))

    # below 2^-26 sin x rounds to x: zeros (with their sign) and subnormals come back unchanged
    tiny = np.array([0.0, -0.0, 5e-324, -5e-324, 2.0 ** -1030, -(2.0 ** -1022), 2.0 ** -60, -(2.0 ** -27)])
    gt = probe.unary("sin_cr", tiny)
    assert np.array_equal(gt.view(np.int64), tiny.view(np.int64))

    # outside [-pi, pi]: CUDA sin; non-finite -> NaN
    far = np.concatenate([np.nextafter(PI_HI, 4.0) + np.array([0.0]), rng.uniform(np.pi, 10.0, 3000)])
    far = np.concatenate([far, -far])
    gf = probe.unary("sin_cr", far)
    worst_far = float(np.max(_ulp_err(gf, _exact(mp.sin, far))))
    assert worst_far <= LIBM_SIN_ULP
    assert np.isnan(probe.unary("sin_cr", [np.nan, np.inf, -np.inf])).all()
    _report("lp_sin_cr", "%d args in [-pi, pi]: %d not correctly rounded (all within 2^-14 ulp of a midpoint), "
            "worst %.4f ulp; (pi, 10]: worst %.4f ulp" % (2 * x.size, 2 * exceptions, worst_range, worst_far))


# ---------------------------------------------------------------------------------------------------------
# lp_acos_unit
# ---------------------------------------------------------------------------------------------------------
def test_acos_unit(probe):
    """lp_acos_unit: < 0.75 ulp for |x| > 0.5625 (the polynomial branch with the MUFU.RSQ64H seed),
    contract 2 ulp below (CUDA acos); np.clip semantics: |x| > 1 gives exactly 0.0 / np.pi, NaN stays NaN."""
    mp = _mp()
    rng = np.random.default_rng(7)
    one_minus = 1.0 - np.arange(4097) * 2.0 ** -53
    pos = np.unique(np.concatenate([rng.uniform(0.5625, 1.0, 12000), 1.0 - 10.0 ** (-16.0 * rng.uniform(0, 1, 5000)),
                                    one_minus, _around(0.5625, 8), [1.0]]))
    pos = pos[(pos > 0.5625) & (pos <= 1.0)]
    x = np.concatenate([pos, -pos])
    got = probe.unary("acos_unit", x)
    with mp.workprec(PREC):
        ep = [mp.acos(mp.mpf(float(v))) for v in pos]
        exact = ep + [mp.pi - e for e in ep]
    err = _ulp_err(got, exact)
    worst = float(np.max(err))
    assert worst < ACOS_ULP, "worst %.3f ulp at x = %s" % (worst, float.hex(float(x[np.argmax(err)])))

    small = np.unique(np.concatenate([rng.uniform(-0.5625, 0.5625, 4000), _around([0.5625, -0.5625], 8), [0.0, -0.0]]))
    small = small[np.abs(small) <= 0.5625]
    worst_small = float(np.max(_ulp_err(probe.unary("acos_unit", small), _exact(mp.acos, small))))
    assert worst_small <= LIBM_ACOS_ULP

    edges = np.array([1.0 + 2.0 ** -52, 2.0, 1e300, np.inf, 1.0, -1.0 - 2.0 ** -52, -2.0, -1e300, -np.inf, -1.0])
    ge = probe.unary("acos_unit", edges)
    assert np.array_equal(ge[:5], np.zeros(5)) and np.array_equal(ge[5:], np.full(5, np.pi))
    assert np.isnan(probe.unary("acos_unit", [np.nan, -np.nan])).all()
    _report("lp_acos_unit", "|x| > 0.5625: worst %.4f ulp (%d args); |x| <= 0.5625: worst %.4f ulp"
            % (worst, x.size, worst_small))


# ---------------------------------------------------------------------------------------------------------
# sincos_moderate
# ---------------------------------------------------------------------------------------------------------
def _sincos_inputs(rng):
    k = np.arange(-40, 41)
    ks = rng.integers(41, int(1e4 * 2 / np.pi), 200)
    with _mp().workprec(PREC):
        pi2 = _mp().pi / 2
        near = [float(int(j) * pi2) for j in k]
        near_s = [float(int(j) * pi2) for j in ks]
    x = np.concatenate([rng.uniform(0, np.pi / 2, 8000), rng.uniform(-4 * np.pi, 4 * np.pi, 8000),
                        rng.uniform(0, 60, 8000), rng.uniform(0, 1e4, 8000), _around(near, 64), _around(near_s, 16)])
    return np.unique(x[np.abs(x) <= 1e4])


def test_sincos_moderate(probe):
    """sincos_moderate on |x| <= 1e4 (the largest argument its callers pass): sine and cosine within 2^-52
    absolute everywhere and within the measured relative bound where |result| >= 2^-10; the reduction
    x = q pi/2 + r exact but for the rounding of r, with |r| <= pi/4 (1 + 2^-50)."""
    mp = _mp()
    rng = np.random.default_rng(11)
    x = _sincos_inputs(rng)
    s, c, q, r = probe.sincos_moderate(x)
    worst_abs, worst_rel, worst_red = 0.0, 0.0, 0.0
    with mp.workprec(PREC):
        pi2 = mp.pi / 2
        es, ec = [], []
        for v, qi, ri in zip(x, q, r):
            xv = mp.mpf(float(v))
            es.append(mp.sin(xv))
            ec.append(mp.cos(xv))
            # the reduction: exact but for the rounding of r (half an ulp) and the 2^-107 tail of pi/2
            dev = abs(xv - (int(qi) * pi2 + mp.mpf(float(ri))))
            bound = mp.mpf(float(np.spacing(abs(ri)))) / 2 + abs(int(qi)) * mp.ldexp(1, -104)
            worst_red = max(worst_red, float(dev / bound))
        for got, exact in ((s, es), (c, ec)):
            err = [abs(mp.mpf(float(g)) - e) for g, e in zip(got, exact)]
            worst_abs = max(worst_abs, float(max(err)) / 2.0 ** -53)
            big = [i for i, e in enumerate(exact) if abs(e) >= 2.0 ** -10]
            worst_rel = max(worst_rel, float(np.max(_ulp_err(got[big], [exact[i] for i in big]))))
    assert worst_abs * 2.0 ** -53 <= SINCOS_ABS, "absolute error %.3f x 2^-53" % worst_abs
    assert worst_rel <= SINCOS_REL_ULP, "relative error %.3f ulp" % worst_rel
    assert worst_red <= 1.0, "x = q pi/2 + r off by %.3g of the rounding bound" % worst_red
    assert np.all(np.abs(r) <= np.pi / 4 * (1 + 2.0 ** -50))
    _report("sincos_moderate", "%d args: worst |err| %.4f x 2^-53, worst %.4f ulp where |result| >= 2^-10, "
            "reduction within %.3f of its rounding bound" % (x.size, worst_abs, worst_rel, worst_red))


# ---------------------------------------------------------------------------------------------------------
# inv_tenth_root
# ---------------------------------------------------------------------------------------------------------
def test_inv_tenth_root(probe):
    """inv_tenth_root: x^-0.1 within a few ulp (contract 3) on [1e-14, 1e10]; below (0, negatives, subnormals, -inf) exactly
    the value at 1e-14, at and above 1e10 (+inf, NaN) exactly the value at 1e10."""
    mp = _mp()
    rng = np.random.default_rng(13)
    edges = _around([1e-14, 1e10], 8)
    x = np.unique(np.concatenate([10.0 ** rng.uniform(-14, 10, 20000), edges, [1.0, 0.5, 2.0]]))
    x = x[(x >= 1e-14) & (x <= 1e10)]
    got = probe.unary("inv_tenth_root", x)
    err = _ulp_err(got, _exact(lambda v: mp.power(v, -mp.mpf(1) / 10), x))
    worst = float(np.max(err))
    assert worst <= INV_TENTH_ULP, "worst %.3f ulp at x = %r" % (worst, float(x[np.argmax(err)]))

    lo_v, hi_v = probe.unary("inv_tenth_root", [1e-14, 1e10])
    below = np.array([0.0, -0.0, -1.0, -1e300, -np.inf, 5e-324, 2.0 ** -1030, np.nextafter(1e-14, 0), 1e-300])
    above = np.array([np.nextafter(1e10, np.inf), 1e20, 1e300, np.inf, np.nan])
    assert np.array_equal(probe.unary("inv_tenth_root", below), np.full(below.size, lo_v))
    assert np.array_equal(probe.unary("inv_tenth_root", above), np.full(above.size, hi_v))
    _report("inv_tenth_root", "[1e-14, 1e10]: worst %.4f ulp (%d args)" % (worst, x.size))


# ---------------------------------------------------------------------------------------------------------
# fast_rcp, fast_rsqrt, mid_range
# ---------------------------------------------------------------------------------------------------------
def _mid_range_operands(rng, n, signed):
    mant = rng.integers(0, 1 << 52, n, dtype=np.int64)
    pattern = np.arange(n) % 5
    mant = np.where(pattern == 1, (1 << 52) - 1, mant)                            # all ones
    mant = np.where(pattern == 2, mant | ((1 << 52) - (1 << 12)), mant)           # near all ones
    mant = np.where(pattern == 3, 0, mant)                                        # power of two
    mant = np.where(pattern == 4, mant & 0xFFF, mant)                             # just above a power of two
    ex = rng.integers(-900, 900, n)
    x = ((ex + 1023).astype(np.int64) << 52 | mant).view(np.float64)
    if signed:
        x = np.where(rng.integers(0, 2, n) == 1, -x, x)
    return x


def test_fast_rcp_rsqrt(probe):
    """fast_rcp and fast_rsqrt (MUFU seed + two Newton steps): contract 2 ulp on mid_range's domain
    2^-900 <= |x| < 2^900, over random, all-ones and power-of-two mantissas."""
    mp = _mp()
    rng = np.random.default_rng(17)
    x = np.concatenate([_mid_range_operands(rng, 10000, True), [2.0 ** -900, -(2.0 ** -900)],
                        np.nextafter([2.0 ** 900, -(2.0 ** 900)], 0)])
    err_rcp = _ulp_err(probe.unary("fast_rcp", x), _exact(lambda v: 1 / v, x))
    xs = np.abs(_mid_range_operands(rng, 10000, False))
    err_rsqrt = _ulp_err(probe.unary("fast_rsqrt", xs), _exact(lambda v: 1 / mp.sqrt(v), xs))
    w_rcp, w_rsqrt = float(np.max(err_rcp)), float(np.max(err_rsqrt))
    assert w_rcp <= RCP_ULP, "fast_rcp %.3f ulp at %r" % (w_rcp, float(x[np.argmax(err_rcp)]))
    assert w_rsqrt <= RSQRT_ULP, "fast_rsqrt %.3f ulp at %r" % (w_rsqrt, float(xs[np.argmax(err_rsqrt)]))
    _report("fast_rcp / fast_rsqrt", "worst %.4f / %.4f ulp (%d / %d args)" % (w_rcp, w_rsqrt, x.size, xs.size))


def test_mid_range_boundaries(probe):
    """mid_range: true exactly for finite 2^-900 <= |x| < 2^900 (three integer instructions on the high word)."""
    b = np.array([2.0 ** -900, 2.0 ** 900])
    x = np.concatenate([_around(b, 2), -_around(b, 2), [0.0, -0.0, 5e-324, -5e-324, 2.0 ** -1022, np.inf, -np.inf,
                                                         np.nan, 1.0, -1.0, 1e308]])
    want = np.isfinite(x) & (np.abs(x) >= 2.0 ** -900) & (np.abs(x) < 2.0 ** 900)
    got = probe.unary("mid_range", x).astype(bool)
    assert np.array_equal(got, want), [float.hex(float(v)) for v in x[got != want]]
    _report("mid_range", "%d boundary decisions exact" % x.size)


# ---------------------------------------------------------------------------------------------------------
# half-orbit counts
# ---------------------------------------------------------------------------------------------------------
def _half_orbit_inputs(rng):
    mp = _mp()
    with mp.workprec(PREC):
        kpi = [float(k * mp.pi) for k in range(41)]
        # both edges of half_orbits_fast's window: |phi| / pi within 1e-9 of an integer
        n = list(range(0, 41)) + [int(v) for v in rng.integers(41, 3183, 40)]
        win = [float((j + s) * mp.pi) for j in n for s in (mp.mpf("1e-9"), 1 - mp.mpf("1e-9"))]
        big = float(mp.mpf("4e9") * mp.pi)
    parts = [_around(kpi, 64), _around(win, 8), rng.uniform(0, 60, 10000), rng.uniform(0, 1e4, 10000),
             _around(big, 8), rng.uniform(4e9 * np.pi, 1e15, 2000)]
    return np.unique(np.concatenate(parts))


def test_half_orbit_counts(probe):
    """half_orbits, half_orbits_fast and binet_finish's quadrant rule (half_orbits_quadrant, for
    0 <= phi < 1e4): bit-exact abs(phi) // pi with CPython's float floor division, which numba's
    compilation of the reference's np.abs(phi_f) // np.pi follows."""
    rng = np.random.default_rng(19)
    x = _half_orbit_inputs(rng)
    x = np.concatenate([x, -x[x > 0]])
    want = np.array([int(abs(v) // math.pi) for v in x], dtype=np.int64)
    for name in ("half_orbits", "half_orbits_fast"):
        got = probe.unary(name, x)
        bad = got != want
        assert not bad.any(), "%s: %s" % (name, [(float.hex(float(v)), int(g), int(w)) for v, g, w in
                                                 zip(x[bad][:8], got[bad][:8], want[bad][:8])])
    m = (x >= 0) & (x < 1e4)
    got = probe.unary("half_orbits_quadrant", x[m])
    bad = got != want[m]
    assert not bad.any(), [(float.hex(float(v)), int(g), int(w)) for v, g, w in
                           zip(x[m][bad][:8], got[bad][:8], want[m][bad][:8])]
    _report("half-orbit counts", "%d args (%d in the quadrant rule's range): all exact" % (x.size, int(m.sum())))


# ---------------------------------------------------------------------------------------------------------
# source_coords_xy
# ---------------------------------------------------------------------------------------------------------
def _cameras(native, golden):
    meta = golden("golden_meta.json")["frames"]
    geoms = [(g["H"], g["W"], g["hfov"], g["vfov"], tuple(g["psi"])) for k, g in sorted(meta.items())
             if not k.startswith("_")]
    geoms.append((90, 160, 1.2, 0.75, (1.3, -2.6)))      # large psi: the black hole behind the camera
    lib = native.capi()
    cams = []
    for H, W, hf, vf, psi in geoms:
        cam = native.lp_camera()
        assert lib.lp_camera_init(H, W, hf, vf, psi[0], psi[1], ctypes.byref(cam)) == 0
        cams.append((psi, cam))
    return cams


def _coords_exact(cam, xc, yc, fa32):
    """the reference's source direction and pinhole coordinates (image_lens.py:310-375) in mpmath:
    (sz, px, py) per pixel, px / py None behind the camera"""
    mp = _mp()
    d = [mp.mpf(v) for v in cam.d]
    ex = [mp.mpf(v) for v in cam.e_x]
    ey = [mp.mpf(v) for v in cam.e_y]
    fx, fy, hw, hh = mp.mpf(cam.fx), mp.mpf(cam.fy), mp.mpf(cam.width) / 2, mp.mpf(cam.height) / 2
    out = []
    with mp.workprec(PREC):
        for x, y, a in zip(xc, yc, fa32):
            x, y, a = mp.mpf(float(x)), mp.mpf(float(y)), mp.mpf(float(a))
            A = x * ex[0] + y * ex[1] + ex[2]
            B = x * ey[0] + y * ey[1] + ey[2]
            n = mp.sqrt(A * A + B * B)
            st, ct = (A / n, B / n) if n != 0 else (mp.mpf(0), mp.mpf(1))     # arctan2(0, 0) = 0
            sf, cf = mp.sin(a), mp.cos(a)
            s = [cf * d[i] + sf * (st * ex[i] + ct * ey[i]) for i in range(3)]
            if s[2] > mp.mpf(1e-12):                                   # the double 1e-12, as numpy compares
                out.append((s[2], s[0] / s[2] * fx + hw, s[1] / s[2] * fy + hh, s[0] / s[2], s[1] / s[2]))
            else:
                out.append((s[2], None, None, None, None))
    return out


def _coord_pixels(rng, cam, n_random):
    """(xc, yc, fa32): random pixels and viewing angles, the centre pixel, and float32 angles that step sz
    across 1e-12"""
    H, W = cam.height, cam.width
    rows = rng.integers(0, H, n_random)
    cols = rng.integers(0, W, n_random)
    xc = list((cols - W / 2) / cam.fx)
    yc = list((rows - H / 2) / cam.fy)
    fa = list(rng.uniform(0, np.pi / 2, n_random).astype(np.float32))
    for a in (0.0, 0.3, 1.0, 1.5707962):               # the centre pixel: on the axis when psi = 0
        xc.append((W // 2 - W / 2) / cam.fx)
        yc.append((H // 2 - H / 2) / cam.fy)
        fa.append(np.float32(a))
    d, ex, ey = np.array(cam.d), np.array(cam.e_x), np.array(cam.e_y)
    for i in range(60):
        x0, y0 = (int(rng.integers(0, W)) - W / 2) / cam.fx, (int(rng.integers(0, H)) - H / 2) / cam.fy
        A, B = x0 * ex[0] + y0 * ex[1] + ex[2], x0 * ey[0] + y0 * ey[1] + ey[2]
        nrm = math.hypot(A, B)
        if nrm == 0:
            continue
        tz = (A * ex[2] + B * ey[2]) / nrm
        # sz(fa) = d2 cos fa + tz sin fa = R cos(fa - phi): the angle where it falls through 1e-12
        R, phi = math.hypot(d[2], tz), math.atan2(tz, d[2])
        if R < 1e-6:
            continue
        for root in (phi + math.acos(1e-12 / R), phi - math.acos(1e-12 / R)):
            if 0.0 <= root <= np.pi / 2:
                a = np.float32(root)
                for _ in range(8):
                    a = np.nextafter(a, np.float32(0))
                for _ in range(17):
                    xc.append(x0)
                    yc.append(y0)
                    fa.append(a)
                    a = np.nextafter(a, np.float32(4))
    return np.array(xc), np.array(yc), np.array(fa, dtype=np.float32)


def _check_coords(tag, exact, px, py, front, fx, fy):
    mp = _mp()
    worst_plain, worst = 0.0, 0.0
    n_front = 0
    with mp.workprec(PREC):
        for i, (sz, ex_px, ex_py, qx, qy) in enumerate(exact):
            if abs(sz - mp.mpf(1e-12)) > mp.mpf("1e-20"):
                assert bool(front[i]) == (sz > mp.mpf(1e-12)), "%s: front differs at pixel %d (sz = %s)" % (
                    tag, i, mp.nstr(sz, 5))
            if ex_px is None or sz < mp.mpf("1e-6"):
                continue
            n_front += 1
            for got, ref, q, f in ((px[i], ex_px, qx, fx), (py[i], ex_py, qy, fy)):
                plain = COORD_REL * max(1.0, abs(float(ref)))
                cond = 4 * EPS * f * (1 + abs(float(q))) / float(sz)
                dev = float(abs(mp.mpf(float(got)) - ref))
                worst_plain = max(worst_plain, dev / plain)
                worst = max(worst, dev / (plain + cond))
    return worst_plain, worst, n_front


def test_source_coords(probe, native, golden):
    """source_coords_xy, plain (sincos of fa32) and DIR (cos / sin of the fp64 final_alpha from the tracer,
    corrected to fa32): `front` equals the exact sz > 1e-12 wherever |sz - 1e-12| > 1e-20, and where
    sz >= 1e-6 the pinhole coordinates are within 1e-12 max(1, |p|) plus the conditioning term of the
    module docstring — the margin the integer source index rint(p) has against the reference."""
    mp = _mp()
    rng = np.random.default_rng(23)
    lines = []
    for psi, cam in _cameras(native, golden):
        xc, yc, fa32 = _coord_pixels(rng, cam, 2500)
        exact = _coords_exact(cam, xc, yc, fa32)
        px, py, front = probe.source_coords(cam, False, xc, yc, fa32)
        plain_p, worst_p, n_front = _check_coords("plain %r" % (psi,), exact, px, py, front, cam.fx, cam.fy)
        # DIR: fa64 within half a float32 step of fa32; cfa, sfa its correctly rounded cosine / sine moved by
        # up to 2 ulp (the accuracy of the tracer's heading)
        half = (np.nextafter(fa32, np.float32(4)) - fa32).astype(np.float64) / 2
        fa64 = fa32.astype(np.float64) + rng.uniform(-1, 1, fa32.size) * half
        with mp.workprec(PREC):
            cfa = np.array([float(mp.cos(mp.mpf(float(v)))) for v in fa64])
            sfa = np.array([float(mp.sin(mp.mpf(float(v)))) for v in fa64])
        cfa = cfa + rng.integers(-2, 3, cfa.size) * np.spacing(np.abs(cfa))
        sfa = sfa + rng.integers(-2, 3, sfa.size) * np.spacing(np.abs(sfa))
        px, py, front = probe.source_coords(cam, True, xc, yc, fa32, fa64, cfa, sfa)
        plain_d, worst_d, _ = _check_coords("DIR %r" % (psi,), exact, px, py, front, cam.fx, cam.fy)
        assert worst_p <= 1.0 and worst_d <= 1.0, (psi, worst_p, worst_d)
        lines.append("psi %r: %d pixels (%d in front, sz >= 1e-6): worst |dp| / (1e-12 max(1, |p|)) "
                     "plain %.3g, DIR %.3g; against the bar with conditioning %.3g, %.3g"
                     % (psi, xc.size, n_front, plain_p, plain_d, worst_p, worst_d))
    _report("source_coords_xy", "\n    ".join([""] + lines))
