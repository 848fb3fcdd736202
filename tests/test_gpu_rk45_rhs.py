"""The generic RK45 integrator's right-hand sides, run on the GPU and compared with an exact evaluation of
the reference's formulas.

rk_rhs (Schwarzschild) and rk_rhs_kerr (csrc/lp_rk45_rhs.cuh) do not evaluate the reference's expressions
(metrics.py: Schwarzschild.geodesic_equations, Kerr.geodesic_equations): they replace its divisions with
products of a few fast_rcp reciprocals and contract sums into fma, and claim every term stays within a few
ulp of the reference's.  The whole-integration tests cannot check that claim, and before this file no Kerr
state they integrated had p_phi != 0, so half of the Kerr formula was multiplied by zero.  Here each right-
hand side runs over arrays of states (tests/rk45_rhs_probe.cu, compiled with the library's NVCC_FLAGS, so
with -fmad=false like the library) and is compared with the reference's expressions evaluated in mpmath at
200 bits on the same double inputs.

Scale of the bar.  A component is a sum of terms, some of them with cancellation inside (f = 1 - R_S / r
and Delta = r^2 - 2 M r + a^2 near the horizon, cos(theta) near the equator).  Each component is held to
|device - exact| <= K 2^-53 S, where S is the first-order running error bound of the reference's own
expression: every sum contributes the sum of the absolute values of its terms, carried through the products
and quotients that use it, and every operation its own result (sin and cos two units).  A correctly rounded
evaluation of the reference's expression order stays within 1 x 2^-53 S; K is the B200's measured worst
case for the rewritten form, rounded up to the next 0.25 (the constants carry both numbers).

Besides accuracy: the theta cache must not change a result (a hit and a miss give the same bits); the
equatorial kernel's rk_rhs_eq<SPEC> must equal rk_rhs bit for bit at theta = pi/2, p_theta = 0 on
(t, r, phi, p_r); at r == r_floor every component is 0; where the reference gives a non-finite value
(sin theta = 0 exactly) the device must too.
"""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROBE_SRC = os.path.join(ROOT, "tests", "rk45_rhs_probe.cu")

PREC = 200
EPS = 2.0 ** -53
SEQ = 4                                # states per thread (one ThetaCache)
# bars in units of 2^-53 S (module docstring); measured on an NVIDIA B200 (power limit 1000 W) over the
# inputs below and rounded up to the next 0.25:
K_SCHW = 1.5                           # rk_rhs; measured 1.404
K_KERR = 0.75                          # rk_rhs_kerr; measured 0.690

KIND_SCHW, KIND_KERR, KIND_EQ_SPEC, KIND_EQ = 0, 1, 2, 3


class _Probe:
    def __init__(self, so_path):
        import torch
        self.torch = torch
        self.lib = ctypes.CDLL(so_path)
        vp = ctypes.c_void_p
        fn = self.lib.probe_rk45_rhs
        fn.restype = ctypes.c_int
        fn.argtypes = [ctypes.c_int, vp, vp, vp, vp, ctypes.c_longlong, ctypes.c_int, vp]

    def rhs(self, kind, par, y, seq=SEQ):
        t = self.torch
        par = t.from_numpy(np.ascontiguousarray(par, dtype=np.float64)).cuda()
        y = t.from_numpy(np.ascontiguousarray(y, dtype=np.float64)).cuda()
        n = y.shape[0]
        d = t.empty((n, 6), dtype=t.float64, device="cuda")
        hit = t.empty(n, dtype=t.int32, device="cuda")
        rc = self.lib.probe_rk45_rhs(kind, par.data_ptr(), y.data_ptr(), d.data_ptr(), hit.data_ptr(), n, seq,
                                     t.cuda.current_stream().cuda_stream)
        assert rc == 0, "probe launch failed: %d" % rc
        t.cuda.synchronize()
        return d.cpu().numpy(), hit.cpu().numpy().astype(bool)


@pytest.fixture(scope="module")
def probe(native, tmp_path_factory):
    from light_path_tracer_b200 import build as b
    so = str(tmp_path_factory.mktemp("rk45_rhs") / "rk45_rhs_probe.so")
    cmd = [b._nvcc()] + b.NVCC_FLAGS + ["-shared", "-Xcompiler", "-fPIC", "-I" + b.CSRC, PROBE_SRC, "-o", so,
                                        "-L" + b.OUT, "-llightpath", "-Xlinker", "-rpath," + b.OUT]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    return _Probe(so)


# ---------------------------------------------------------------------------------------------------------
# the reference: metrics.py's expressions on a value (mpf, 200 bits) carrying its running error scale
# ---------------------------------------------------------------------------------------------------------
class _V:
    """An exact value and the first-order error scale of computing it in doubles, in units of 2^-53."""
    __slots__ = ("v", "s")

    def __init__(self, v, s=0.0):
        self.v, self.s = v, s

    @staticmethod
    def _w(x):
        return x if isinstance(x, _V) else _V(_mp().mpf(x))

    def _out(self, v, s):
        return _V(v, s + abs(float(v)))

    def __add__(self, o):
        o = self._w(o)
        return self._out(self.v + o.v, self.s + o.s)
    __radd__ = __add__

    def __sub__(self, o):
        o = self._w(o)
        return self._out(self.v - o.v, self.s + o.s)

    def __rsub__(self, o):
        return self._w(o) - self

    def __neg__(self):
        return _V(-self.v, self.s)

    def __mul__(self, o):
        o = self._w(o)
        return self._out(self.v * o.v, self.s * abs(float(o.v)) + abs(float(self.v)) * o.s)
    __rmul__ = __mul__

    def __truediv__(self, o):
        o = self._w(o)
        q = self.v / o.v
        return self._out(q, (self.s + abs(float(q)) * o.s) / abs(float(o.v)))

    def __rtruediv__(self, o):
        return self._w(o) / self

    def __pow__(self, k):                     # numpy's x**k for a small integer k: one rounding
        assert k in (2, 3)
        return self._out(self.v ** k, k * abs(float(self.v)) ** (k - 1) * self.s)


def _mp():
    import mpmath
    return mpmath


def _trig(th):
    mp = _mp()
    s, c = mp.sin(th), mp.cos(th)
    return _V(s, 2 * abs(float(s))), _V(c, 2 * abs(float(c)))


def _ref_schw(R_S, st):
    """Schwarzschild.geodesic_equations (metrics.py) for (t, r, theta, phi, p_r, p_theta), floor included"""
    t, r, th, phi, p_t, p_r, p_th, p_phi = st
    mp = _mp()
    R_S, r, p_t, p_r, p_th, p_phi = (_V(mp.mpf(x)) for x in (R_S, r, p_t, p_r, p_th, p_phi))
    f = 1 - R_S / r
    sin_th, cos_th = _trig(mp.mpf(th))
    s2 = sin_th ** 2
    if s2.v < mp.mpf(1e-15):
        s2 = _V(mp.mpf(1e-15))
    half = R_S / (2 * r ** 2)
    return [-p_t / f, f * p_r, p_th / r ** 2, p_phi / (r ** 2 * s2),
            (-half * (p_t ** 2 / f ** 2) - half * p_r ** 2 + (p_th ** 2 + p_phi ** 2 / s2) / r ** 3),
            cos_th * p_phi ** 2 / (r ** 2 * s2 * sin_th)]


def _ref_kerr(M, a, st):
    """Kerr.geodesic_equations (metrics.py) for the six moving components"""
    t, r, th, phi, p_t, p_r, p_th, p_phi = st
    mp = _mp()
    M, a, r, p_t, p_r, p_th, p_phi = (_V(mp.mpf(x)) for x in (M, a, r, p_t, p_r, p_th, p_phi))
    s, c = _trig(mp.mpf(th))
    Sigma = r ** 2 + a ** 2 * c ** 2
    Delta = r ** 2 - 2 * M * r + a ** 2
    A = (r ** 2 + a ** 2) ** 2 - a ** 2 * Delta * s ** 2
    g = dict(tt=-A / (Sigma * Delta), tphi=-2 * M * a * r / (Sigma * Delta), rr=Delta / Sigma,
             thth=1.0 / Sigma, phiphi=(Delta - a ** 2 * s ** 2) / (Sigma * Delta * s ** 2))
    SD = Sigma * Delta
    dS_r, dD_r = 2 * r, 2 * r - 2 * M
    dA_r = 4 * r * (r ** 2 + a ** 2) - a ** 2 * dD_r * s ** 2
    dSD_r = dS_r * Delta + Sigma * dD_r
    d_r = dict(tt=-(dA_r * SD - A * dSD_r) / SD ** 2,
               tphi=-(2 * M * a * (SD - r * dSD_r)) / SD ** 2,
               rr=(dD_r * Sigma - Delta * dS_r) / Sigma ** 2,
               thth=-dS_r / Sigma ** 2,
               phiphi=(dD_r * SD * s ** 2 - (Delta - a ** 2 * s ** 2) * dSD_r * s ** 2) / (SD * s ** 2) ** 2)
    dS_th = -2 * a ** 2 * s * c
    dA_th = -a ** 2 * Delta * 2 * s * c
    num, den = Delta - a ** 2 * s ** 2, SD * s ** 2
    dnum, dden = -a ** 2 * 2 * s * c, dS_th * Delta * s ** 2 + SD * 2 * s * c
    d_th = dict(tt=-(dA_th * SD - A * dS_th * Delta) / SD ** 2,
                tphi=2 * M * a * r * dS_th / (Sigma ** 2 * Delta),
                rr=-Delta * dS_th / Sigma ** 2,
                thth=-dS_th / Sigma ** 2,
                phiphi=(dnum * den - num * dden) / den ** 2)

    def contract(d):
        return -0.5 * (d["tt"] * p_t ** 2 + 2 * d["tphi"] * p_t * p_phi + d["rr"] * p_r ** 2
                       + d["thth"] * p_th ** 2 + d["phiphi"] * p_phi ** 2)
    return [g["tt"] * p_t + g["tphi"] * p_phi, g["rr"] * p_r, g["thth"] * p_th,
            g["tphi"] * p_t + g["phiphi"] * p_phi, contract(d_r), contract(d_th)]


def _reference(kind, par, y):
    """exact values [n][6] (mpf) and scales [n][6] (float, units of 2^-53) above the floor"""
    mp = _mp()
    ex, sc = [], []
    with mp.workprec(PREC):
        for p, yi in zip(par, y):
            st = (yi[0], yi[1], yi[2], yi[3], p[3], yi[4], yi[5], p[4])
            out = _ref_schw(p[0], st) if kind == KIND_SCHW else _ref_kerr(p[0], p[1], st)
            ex.append([o.v for o in out])
            sc.append([o.s for o in out])
    return ex, np.array(sc)


def _err_units(got, ex, sc):
    """|got - exact| / (2^-53 S), elementwise; 0 where both are exactly 0"""
    mp = _mp()
    out = np.zeros(got.shape)
    with mp.workprec(PREC):
        for i in range(got.shape[0]):
            for j in range(got.shape[1]):
                e = abs(mp.mpf(float(got[i, j])) - ex[i][j]) if math.isfinite(got[i, j]) else mp.inf
                if e == 0:
                    continue
                out[i, j] = float(e / (EPS * sc[i, j])) if sc[i, j] > 0 else np.inf
    return out


def _report(name, text):
    print("\nrk45 rhs | %-12s | %s" % (name, text))


# ---------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------
PI_2 = np.pi / 2
THETAS = np.array([PI_2, np.nextafter(PI_2, 4.0), np.nextafter(PI_2, 0.0), 1e-3, 1e-8, np.pi - 1e-8, -1e-8,
                   -0.7, -PI_2, 4.0, 2 * np.pi - 0.3, 1.1, 0.3, 2.9, 3e-8, 3.3e-8])
A_OVER_M = np.array([0.0, 1e-6, -1e-6, 0.5, -0.5, 0.9, -0.9, 0.998, -0.998, 1.0, -1.0])


def _theta_walk(rng, n, pool):
    """theta for n states in chunks of SEQ (one thread each): the first of a chunk drawn, the next equal to
    the previous one (a cache hit), one ulp away (a miss that a stale cache would not notice) or drawn"""
    th = np.empty(n)
    for i in range(n):
        u = rng.random()
        if i % SEQ == 0 or u < 0.3:
            th[i] = pool(rng) if i % SEQ == 0 or u < 0.15 else rng.uniform(0.05, np.pi - 0.05)
        elif u < 0.7:
            th[i] = th[i - 1]
        else:
            th[i] = np.nextafter(th[i - 1], np.inf if rng.random() < 0.5 else -np.inf)
    return th


def _states(rng, n, r_floor, M, p_phi_zero_share=0.2):
    """n states above the floor: r from the floor to 1e6 M (the near-horizon shell dense), theta from THETAS
    or uniform (walked in cache chunks), momenta of both signs, p_phi in {0, O(1), O(10)}"""
    u = rng.random(n)
    shell = r_floor * (1 + 10.0 ** rng.uniform(-9, -1, n))
    far = M * 10.0 ** rng.uniform(np.log10(3.0), 6.0, n)
    mid = rng.uniform(r_floor, 12 * M, n)
    r = np.where(u < 0.3, shell, np.where(u < 0.65, mid, far))
    r = np.maximum(r, np.nextafter(r_floor, np.inf))
    th = _theta_walk(rng, n, lambda g: THETAS[g.integers(THETAS.size)] if g.random() < 0.7
                     else g.uniform(-0.5, np.pi + 0.5))
    p_phi = np.where(rng.random(n) < 0.5, rng.uniform(-3, 3, n), rng.uniform(-30, 30, n))
    p_phi[rng.random(n) < p_phi_zero_share] = 0.0
    p_t = np.where(rng.random(n) < 0.7, -1.0, -rng.uniform(0.3, 3.0, n))
    y = np.stack([rng.uniform(0, 500, n), r, th, rng.uniform(-20, 20, n),
                  rng.normal(0, 2, n), rng.normal(0, 5, n)], axis=1)
    return y, p_t, p_phi


def _schw_batch(seed, n_per):
    rng = np.random.default_rng(seed)
    pars, ys = [], []
    for M in (1.0, 2.5):
        R_S = 2 * M
        r_floor = R_S * 1.001
        y, p_t, p_phi = _states(rng, n_per, r_floor, M)
        pars.append(np.stack([np.full(n_per, R_S), np.zeros(n_per), np.full(n_per, r_floor), p_t, p_phi], axis=1))
        ys.append(y)
    return np.concatenate(pars), np.concatenate(ys)


def _kerr_batch(seed, n_per):
    from light_path_tracer_b200.metrics import Kerr
    rng = np.random.default_rng(seed)
    pars, ys = [], []
    for M in (1.0, 2.5):
        for q in A_OVER_M:
            a = q * M
            r_floor = float(Kerr(M, a).r_plus) * 1.001
            y, p_t, p_phi = _states(rng, n_per, r_floor, M)
            pars.append(np.stack([np.full(n_per, M), np.full(n_per, a), np.full(n_per, r_floor), p_t, p_phi], axis=1))
            ys.append(y)
    return np.concatenate(pars), np.concatenate(ys)


@pytest.fixture(scope="module")
def schw_inputs():
    return _schw_batch(11, 1200)


@pytest.fixture(scope="module")
def kerr_inputs():
    return _kerr_batch(12, 160)


# ---------------------------------------------------------------------------------------------------------
# tests
# ---------------------------------------------------------------------------------------------------------
def _accuracy(probe, kind, par, y, K, name):
    d, hit = probe.rhs(kind, par, y)
    assert hit.mean() > 0.2 and (~hit).mean() > 0.2, hit.mean()
    ex, sc = _reference(kind, par, y)
    err = _err_units(d, ex, sc)
    i, j = np.unravel_index(int(np.argmax(err)), err.shape)
    per = ", ".join("%.3f" % v for v in err.max(axis=0))
    _report(name, "%d states: worst %.3f x 2^-53 S (component %d at r=%r theta=%r p_phi=%r); per component %s"
            % (y.shape[0], err.max(), j, y[i, 1], y[i, 2], par[i, 4], per))
    bad = np.argwhere(err > K)
    assert bad.size == 0, "%d components above %.2f x 2^-53 S, first: state %s component %d (%.3f)" % (
        bad.shape[0], K, (par[bad[0, 0]].tolist(), y[bad[0, 0]].tolist()), bad[0, 1], err[tuple(bad[0])])
    return d, hit


def test_schwarzschild_rhs_accuracy(probe, schw_inputs):
    """rk_rhs against metrics.py's expressions at 200 bits: within K_SCHW x 2^-53 S on every component,
    the sin^2 floor engaged (theta within ~3e-8 of a pole) and not"""
    par, y = schw_inputs
    s2 = np.sin(y[:, 2]) ** 2
    assert (s2 < 1e-15).sum() >= 50 and ((s2 >= 1e-15) & (s2 < 1e-6)).sum() >= 50
    _accuracy(probe, KIND_SCHW, par, y, K_SCHW, "rk_rhs")


def test_kerr_rhs_accuracy(probe, kerr_inputs):
    """rk_rhs_kerr against metrics.py's expressions at 200 bits, p_phi != 0 and off the equator included:
    within K_KERR x 2^-53 S on every component"""
    par, y = kerr_inputs
    assert (par[:, 4] != 0).mean() > 0.7 and (np.abs(np.cos(y[:, 2])) > 0.1).mean() > 0.2
    _accuracy(probe, KIND_KERR, par, y, K_KERR, "rk_rhs_kerr")


@pytest.mark.parametrize("kind", [KIND_SCHW, KIND_KERR], ids=["schwarzschild", "kerr"])
def test_theta_cache_invariance(probe, schw_inputs, kerr_inputs, kind):
    """a result is the same bits whether its theta hit the cache (a thread walking SEQ states) or not (one
    state per thread); the walks include thetas one ulp from their predecessor, which a cache keyed on
    fewer bits than theta's would serve stale sin / cos"""
    par, y = schw_inputs if kind == KIND_SCHW else kerr_inputs
    d_walk, hit = probe.rhs(kind, par, y, seq=SEQ)
    d_cold, hit_cold = probe.rhs(kind, par, y, seq=1)
    assert not hit_cold.any() and hit.sum() > 0.2 * hit.size
    one_ulp = np.zeros(y.shape[0], dtype=bool)
    one_ulp[1:] = (np.arange(1, y.shape[0]) % SEQ != 0) & (y[1:, 2] != y[:-1, 2]) & \
        (np.abs(y[1:, 2] - y[:-1, 2]) <= np.spacing(np.abs(y[:-1, 2])))
    assert one_ulp.sum() >= 100
    same = (d_walk == d_cold) | (np.isnan(d_walk) & np.isnan(d_cold))
    assert same.all(), "%d states differ with and without the cache" % int((~same.all(axis=1)).sum())


def test_equatorial_rhs_equals_six_component(probe):
    """rk_rhs_eq<true> and rk_rhs_eq<false> (the batch path's equatorial system) against rk_rhs at
    theta = pi/2, p_theta = 0: bit-identical on (t, r, phi, p_r) for r above the floor"""
    rng = np.random.default_rng(13)
    pars, ys = [], []
    for M in (1.0, 2.5):
        r_floor = 2 * M * 1.001
        y, p_t, p_phi = _states(rng, 3000, r_floor, M, p_phi_zero_share=0.1)
        y[:, 2], y[:, 5] = PI_2, 0.0
        y[:8, 1] = np.nextafter(r_floor, np.inf)
        pars.append(np.stack([np.full(y.shape[0], 2 * M), np.zeros(y.shape[0]), np.full(y.shape[0], r_floor),
                              p_t, p_phi], axis=1))
        ys.append(y)
    par, y = np.concatenate(pars), np.concatenate(ys)
    d6, _ = probe.rhs(KIND_SCHW, par, y)
    for kind in (KIND_EQ_SPEC, KIND_EQ):
        d4, _ = probe.rhs(kind, par, y)
        live = [0, 1, 3, 4]
        assert np.array_equal(d4[:, live], d6[:, live]), (kind, int((d4[:, live] != d6[:, live]).any(axis=1).sum()))
    # the tested form at and below the floor
    y[:, 1] = np.where(np.arange(y.shape[0]) % 2 == 0, par[:, 2], par[:, 2] * 0.5)
    d4, _ = probe.rhs(KIND_EQ, par, y)
    assert (d4 == 0.0).all() and not np.signbit(d4).any()


@pytest.mark.parametrize("kind", [KIND_SCHW, KIND_KERR], ids=["schwarzschild", "kerr"])
def test_floor(probe, schw_inputs, kerr_inputs, kind):
    """r == r_floor: every component exactly +0 (metrics.py's early return); r one ulp above: non-zero
    and within the accuracy bar"""
    par, y = schw_inputs if kind == KIND_SCHW else kerr_inputs
    par, y = par[::7].copy(), y[::7].copy()
    y[:, 1] = par[:, 2]
    d, _ = probe.rhs(kind, par, y)
    assert (d == 0.0).all() and not np.signbit(d).any()
    y[:, 1] = np.nextafter(par[:, 2], np.inf)
    y[:, 2] = np.where(np.abs(np.sin(y[:, 2])) < 1e-6, 1.2, y[:, 2])
    d, _ = probe.rhs(kind, par, y)
    assert (d[:, [0, 1]] != 0.0).all()               # dt/dlambda and dr/dlambda (p_r != 0)
    ex, sc = _reference(kind, par, y)
    err = _err_units(d, ex, sc)
    K = K_SCHW if kind == KIND_SCHW else K_KERR
    _report("floor " + ("schw" if kind == KIND_SCHW else "kerr"), "one ulp above r_floor: worst %.3f x 2^-53 S"
            % err.max())
    assert err.max() <= K


@pytest.mark.parametrize("kind", [KIND_SCHW, KIND_KERR], ids=["schwarzschild", "kerr"])
def test_non_finite_at_the_pole(probe, kind):
    """sin(theta) = 0 exactly (theta = +-0): where metrics.py's formula (float64, the product's own host
    right-hand side) gives a non-finite value the device does too, and only there"""
    from light_path_tracer_b200.metrics import Schwarzschild, Kerr
    rows, metrics = [], []
    for M in (1.0, 2.5):
        for q in ((0.0,) if kind == KIND_SCHW else (0.0, 0.5, -0.9, 1.0)):
            m = Schwarzschild(M) if kind == KIND_SCHW else Kerr(M, q * M)
            r_floor = (m.R_S if kind == KIND_SCHW else float(m.r_plus)) * 1.001
            for th in (0.0, -0.0):
                for p_phi in (0.0, 1.5, -12.0):
                    for r in (3.0 * M, 40.0 * M):
                        rows.append(([m.R_S if kind == KIND_SCHW else M, q * M, r_floor, -1.0, p_phi],
                                     [1.0, r, th, 0.5, -0.8, 0.3]))
                        metrics.append(m)
    par = np.array([p for p, _ in rows])
    y = np.array([s for _, s in rows])
    d, _ = probe.rhs(kind, par, y)
    with np.errstate(all="ignore"):
        ref = np.array([np.array(m.geodesic_equations(0.0, [yi[0], yi[1], yi[2], yi[3], p[3], yi[4], yi[5], p[4]]),
                                 dtype=np.float64)[[0, 1, 2, 3, 5, 6]] for m, p, yi in zip(metrics, par, y)])
    assert (~np.isfinite(ref)).any()
    assert np.array_equal(np.isfinite(d), np.isfinite(ref)), np.argwhere(np.isfinite(d) != np.isfinite(ref))
