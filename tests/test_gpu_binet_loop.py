"""The Binet RK4 loop's fast paths, bit for bit against the literal loop, at every exit position, step budget
and bound touch.

binet_trace_fast (lp_internal.cuh) runs the loop two trips of TRIP = 2 or 4 RK4 steps per iteration with an
integer test on the high word of u per trip, and leaves it through a handful of rare branches: an exit at
step i of the first or the second trip, a trip whose u only touched a bound (then the remaining full steps
one at a time), the step budget (then the remainder one at a time), the shortened last step.  It must equal
binet_trace_generic, the literal transcription of the reference's loop, bit for bit, and the strict literal
loop must equal the reference itself.  tests/binet_loop_probe.cu runs each variant (strict or FMA arithmetic x
literal loop / fast trip 2 / fast trip 4), the plain per-ray composition LP_TRACE_HYBRID stands for, and the
literal loop's u after every full step, over:

* configurations: the production one, budgets of 0 ... 19 full steps (every n_full mod 8, and the loop skipped
  below two trips), budgets with and without a shortened step, phi_shift 3 and 9 (the strided phi table's
  re-addition loop and, FMA, beyond its single fma), M = 2.5, observers at 2.3 ... 1000 M, a capture radius of
  4M (outside the photon sphere, so a periapsis can touch it without crossing) and observers outside the band;
* rays: random, a cluster at the critical angle, odd values (0, pi, tiny, negative, beyond pi, non-finite) and
  rays bisected, per arithmetic, onto every step-count and outcome boundary of a grid, i.e. rays whose u at
  step k sits within a few ulp of the bound they cross at step k + 1 (touched, then out).

A numpy replay of the fast path's control flow on the literal loop's history sorts every ray into the branch it
takes and requires each branch to have run, so the bit-for-bit comparisons are known to cover them.

More than one shortened step is unreachable: the host replays `phi += h` (lp_make_binet_consts), and once fewer
than h_max remain, phi_max - phi is exact (Sterbenz: phi >= phi_max / 2 there) and so is phi + (phi_max - phi).
"""
import ctypes
import hashlib
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.join(ROOT, "tests")
PROBE_SRC = os.path.join(TESTS, "binet_loop_probe.cu")

LP_ERR_UNSUPPORTED = -3
TRIPS = (2, 4)
HALF_PI_F32 = np.float32(np.pi / 2)

# final_alpha of the strict loop against the reference restated with the device's sine: the two differ only
# through the finish's own routines (sincos_moderate, lp_acos_unit, the straight-line t; lp_internal.cuh).  Bar:
# 2 arccos quanta (2^-52 / sin fa) plus FA_ULP ulp of fa.  Measured on an NVIDIA B200 (power limit 1000 W) over
# the rays below (2.0e5 rays): no ray beyond the 2 quanta (worst excess 0.000 ulp); FA_ULP is that rounded up to
# the next 0.25 ulp.
FA_QUANTA = 2.0
FA_ULP = 0.25
SIN_CR_NEAR_MIDPOINT = 2.0 ** -14      # ulp: lp_sin_cr may round either way this close to a half-way point
ORACLE_STEP_BUDGET = 2e8               # oracle RK4 steps per run (CPU)
MIN_PATH_COUNT = 10

# ---------------------------------------------------------------------------------------------------------
# configurations (M, R_S, r_obs, phi_max, h_max)
# ---------------------------------------------------------------------------------------------------------
DEFAULT = (1.0, 2.0, 100.0, 50.0, 0.05)                      # the reference's budget: 1000 full steps + 1 shortened
CONFIGS = (
    [DEFAULT]
    + [(1.0, 2.0, r, 50.0, 0.05) for r in (2.3, 3.49, 15.0, 1000.0)]
    + [(1.0, 2.0, 3.49, 0.05 * n + 0.025, 0.05) for n in range(20)]     # n_full = n, one shortened step
    + [(1.0, 2.0, 2.3, 0.0625 * n, 0.0625) for n in (0, 7, 9, 16)]      # n_full = n, no shortened step
    + [(1.0, 2.0, 15.0, 0.05 * n + 0.025, 0.05) for n in (203, 405)]
    + [(1.0, 2.0, 100.0, 60.0, 0.05),                                  # phi_shift 3
       (1.0, 2.0, 100.0, 50.0, 0.0005),                                # phi_shift 9 (99 999 full steps)
       (2.5, 5.0, 40.0, 50.0, 0.05),
       (1.0, 4.0, 15.0, 50.0, 0.05), (1.0, 4.0, 100.0, 50.0, 0.05), (1.0, 4.0, 5.0, 20.0, 0.05),
       (1.0, 2.0, 2.01, 50.0, 0.05),                                   # observer beyond the capture bound
       (1.0, 2.0, 1.5, 50.0, 0.05)])                                   # inside R_S: every ray invalid
BIG = (1.0, 2.0, 100.0, 50.0, 0.0005)
HISTORY_MAX_STEPS = 1500               # the path classifier replays configurations up to this many full steps


def _cfg_id(cfg):
    return "M%g Rs%g r%g phi%g h%g" % cfg


# ---------------------------------------------------------------------------------------------------------
# the probe
# ---------------------------------------------------------------------------------------------------------
class ProbeError(RuntimeError):
    pass


class _Probe:
    """ctypes launchers of tests/binet_loop_probe.cu (numpy or CUDA tensors in, numpy out)."""

    def __init__(self, so_path):
        import torch
        self.torch = torch
        self.lib = ctypes.CDLL(so_path)
        d, vp, i64, ci = ctypes.c_double, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int
        self.lib.probe_binet_consts.argtypes = [d] * 5 + [vp, vp]
        self.lib.probe_binet_trace.argtypes = [ci] + [d] * 5 + [vp, i64, vp, vp, vp, vp, vp]
        self.lib.probe_binet_hybrid.argtypes = [d] * 5 + [vp, i64, vp, vp, vp, vp, vp]
        self.lib.probe_binet_history.argtypes = [ci] + [d] * 5 + [vp, i64, ci, vp, vp, vp, vp]
        for f in (self.lib.probe_binet_consts, self.lib.probe_binet_trace, self.lib.probe_binet_hybrid,
                  self.lib.probe_binet_history):
            f.restype = ci

    def consts(self, cfg):
        ints, hi = np.zeros(7, np.int32), np.zeros(4, np.uint32)
        rc = self.lib.probe_binet_consts(*cfg, ints.ctypes.data, hi.ctypes.data)
        if rc:
            raise ProbeError(rc)
        keys = ("n_full", "n_tail", "phi_shift", "fast_ok", "fast_ok_fused", "scaled_ok", "valid")
        out = {k: int(v) for k, v in zip(keys, ints)}
        out["hi"] = {"uc": int(hi[0]), "ue": int(hi[1]), "vc": int(hi[2]), "ve": int(hi[3])}
        return out

    def _dev(self, a):
        t = self.torch
        if isinstance(a, t.Tensor):
            return a.reshape(-1).to(device="cuda", dtype=t.float64).contiguous()
        return t.from_numpy(np.ascontiguousarray(a, dtype=np.float64).reshape(-1)).cuda()

    def _outs(self, n):
        t = self.torch
        return (t.empty(n, dtype=t.float64, device="cuda"), t.empty(n, dtype=t.int64, device="cuda"),
                t.empty(n, dtype=t.int8, device="cuda"), t.empty(n, dtype=t.int32, device="cuda"))

    def _run(self, fn, *args):
        stream = self.torch.cuda.current_stream().cuda_stream
        rc = fn(*[a.data_ptr() if hasattr(a, "data_ptr") else a for a in args], stream)
        if rc:
            raise ProbeError(rc)
        self.torch.cuda.synchronize()

    def trace(self, variant, cfg, alphas):
        """binet_trace per ray -> (fa, nh, status, steps); variant = 3 * fused + {0 literal, 1 trip 2, 2 trip 4}"""
        a = self._dev(alphas)
        outs = self._outs(a.numel())
        self._run(self.lib.probe_binet_trace, variant, *cfg, a, a.numel(), *outs)
        return tuple(o.cpu().numpy() for o in outs)

    def hybrid(self, cfg, alphas):
        a = self._dev(alphas)
        outs = self._outs(a.numel())
        self._run(self.lib.probe_binet_hybrid, *cfg, a, a.numel(), *outs)
        return tuple(o.cpu().numpy() for o in outs)

    def history(self, fused, cfg, alphas, max_steps):
        """the literal loop's variable after each full step -> (hist[n, max_steps], orbit status, steps)"""
        t = self.torch
        a = self._dev(alphas)
        n = a.numel()
        hist = t.empty((n, max_steps), dtype=t.float64, device="cuda")
        ost, steps = t.empty(n, dtype=t.int8, device="cuda"), t.empty(n, dtype=t.int32, device="cuda")
        self._run(self.lib.probe_binet_history, int(fused), *cfg, a, n, int(max_steps), hist, ost, steps)
        return hist.cpu().numpy(), ost.cpu().numpy(), steps.cpu().numpy()


def _compile_probe(so):
    from light_path_tracer_b200 import build as b
    cmd = [b._nvcc()] + b.NVCC_FLAGS + ["-shared", "-Xcompiler", "-fPIC", "-I" + b.CSRC, PROBE_SRC, "-o", so,
                                        "-L" + b.OUT, "-llightpath", "-Xlinker", "-rpath," + b.OUT]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]


@pytest.fixture(scope="module")
def probe_so(native, tmp_path_factory):
    so = str(tmp_path_factory.mktemp("binet_loop") / "binet_loop_probe.so")
    _compile_probe(so)
    return so


@pytest.fixture(scope="module")
def probe(probe_so):
    return _Probe(probe_so)


# ---------------------------------------------------------------------------------------------------------
# rays
# ---------------------------------------------------------------------------------------------------------
ODD_ALPHAS = np.array([0.0, np.pi, np.nextafter(np.pi, 0.0), np.nextafter(np.pi, 4.0), np.pi / 2, 1e-12, 5e-324,
                       -1e-12, -0.3, -np.pi / 2, -np.pi, 3.5, 4.0, 2 * np.pi, 7.0, 100.0, 1e300,
                       np.nan, -np.nan, np.inf, -np.inf])


def _critical_angles(cfg):
    M, R_S, r_obs = cfg[:3]
    f0 = 1.0 - R_S / r_obs
    if not f0 > 0:
        return []
    s = 3.0 * math.sqrt(3.0) * M * math.sqrt(f0) / r_obs
    return [math.asin(s), math.pi - math.asin(s)] if s < 1.0 else []


def _common_rays(cfg, rng):
    n_random = 1000 if cfg == BIG else 4000
    parts = [rng.uniform(0.0, np.pi, n_random), ODD_ALPHAS]
    for ac in _critical_angles(cfg):
        e = 10.0 ** -rng.uniform(3, 15, 150 if cfg == BIG else 300)
        parts.append(ac * (1.0 + np.concatenate([e, -e])))
    return np.concatenate(parts)


def _key(status, steps):
    return status.astype(np.int64) * (1 << 32) + steps.astype(np.int64)


def _edge_rays(probe, cfg, fused, rng, n_grid=2048, max_pairs=400):
    """Adjacent doubles either side of each (status, steps) boundary of a grid over (0, pi), found by
    bisection with the literal loop of one arithmetic: all outcome changes, up to max_pairs step-count changes."""
    grid = np.linspace(0.0, np.pi, n_grid + 1)[1:-1]
    _, _, st, steps = probe.trace(3 * int(fused), cfg, grid)
    key = _key(st, steps)
    idx = np.nonzero(key[1:] != key[:-1])[0]
    outcome = st[idx] != st[idx + 1]
    steps_only = idx[~outcome]
    if steps_only.size > max_pairs:
        steps_only = rng.choice(steps_only, max_pairs, replace=False)
    idx = np.concatenate([idx[outcome], steps_only])
    lo, hi = grid[idx].view(np.int64).copy(), grid[idx + 1].view(np.int64).copy()
    klo = key[idx]
    for _ in range(64):
        act = np.nonzero(hi - lo > 1)[0]
        if act.size == 0:
            break
        mid = lo[act] + (hi[act] - lo[act]) // 2
        _, _, st, steps = probe.trace(3 * int(fused), cfg, mid.view(np.float64))
        same = _key(st, steps) == klo[act]
        lo[act] = np.where(same, mid, lo[act])
        hi[act] = np.where(same, hi[act], mid)
    return np.concatenate([lo, hi]).view(np.float64)


@pytest.fixture(scope="module")
def cases(probe):
    """per configuration: its constants and its rays (random, critical, odd, and both arithmetics' edge rays)"""
    t0 = time.time()
    rng = np.random.default_rng(20261022)
    out = []
    for cfg in CONFIGS:
        k = probe.consts(cfg)
        rays = [_common_rays(cfg, rng)]
        if k["valid"]:
            for fused in (False, True):
                rays.append(_edge_rays(probe, cfg, fused, rng, n_grid=512 if cfg == BIG else 2048,
                                       max_pairs=100 if cfg == BIG else 400))
        out.append(dict(cfg=cfg, k=k, alphas=np.concatenate(rays)))
    print("\nbinet loop | %d configurations, %d rays, prepared in %.1f s"
          % (len(out), sum(c["alphas"].size for c in out), time.time() - t0))
    return out


def _diff(a, b, alphas):
    """indices of the rays where two (fa, nh, status, steps) results differ (fa compared as int64 bits), and a
    description of the first few"""
    ka, kb = (a[0].view(np.int64),) + tuple(a[1:]), (b[0].view(np.int64),) + tuple(b[1:])
    idx = np.nonzero(np.any([x != y for x, y in zip(ka, kb)], axis=0))[0]
    desc = ["alpha %s: (fa %s, nh %d, status %d, steps %d) vs (fa %s, nh %d, status %d, steps %d)" % (
        float.hex(float(alphas[i])), float.hex(float(a[0][i])), a[1][i], a[2][i], a[3][i],
        float.hex(float(b[0][i])), b[1][i], b[2][i], b[3][i]) for i in idx[:5]]
    return idx, desc


# ---------------------------------------------------------------------------------------------------------
# 1. fast == literal
# ---------------------------------------------------------------------------------------------------------
def test_configurations(probe):
    """the list covers what it claims: every n_full 0 ... 19, n_full < 4 and < 8, every n_full mod 8, n_tail 0 and 1
    (and never more), phi_shift 2, 3 and > 8, configurations with and without the fast path's precondition"""
    ks = [probe.consts(c) for c in CONFIGS]
    n_full = {k["n_full"] for k in ks}
    assert set(range(20)) <= n_full
    assert {n % 8 for n in n_full} == set(range(8))
    assert {k["n_tail"] for k in ks} == {0, 1}
    assert {2, 3} <= {k["phi_shift"] for k in ks} and max(k["phi_shift"] for k in ks) > 8
    assert {k["fast_ok"] for k in ks} == {0, 1} and {k["fast_ok_fused"] for k in ks} == {0, 1}
    assert probe.consts(DEFAULT)["n_full"] == 1000 and probe.consts(DEFAULT)["n_tail"] == 1


def test_fast_equals_generic(probe, cases):
    """binet_trace_fast<FUSED, 2> and <FUSED, 4> equal binet_trace_generic<FUSED> bit for bit (final_alpha as int64
    bits, n_half_orbits, status, steps) on every ray of every configuration where the precondition holds; where it
    does not, the probe refuses the fast variant."""
    bad, lines = [], {}
    for c in cases:
        cfg, k, a = c["cfg"], c["k"], c["alphas"]
        for fused in (False, True):
            ok = k["fast_ok_fused"] if fused else k["fast_ok"]
            if not ok:
                for v in (1, 2):
                    with pytest.raises(ProbeError) as e:
                        probe.trace(3 * fused + v, cfg, a[:4])
                    assert e.value.args[0] == LP_ERR_UNSUPPORTED
                continue
            ref = probe.trace(3 * fused, cfg, a)
            for v, trip in ((1, 2), (2, 4)):
                idx, desc = _diff(probe.trace(3 * fused + v, cfg, a), ref, a)
                if idx.size:
                    bad.append("%s %s trip %d: %d rays differ: %s" % (_cfg_id(cfg), "FMA" if fused else "strict",
                                                                      trip, idx.size, desc))
            lines[fused] = lines.get(fused, 0) + a.size
    print("\nbinet loop | fast == literal: %d strict rays, %d FMA rays, each against trip 2 and trip 4"
          % (lines.get(False, 0), lines.get(True, 0)))
    assert not bad, "\n".join(bad)


# ---------------------------------------------------------------------------------------------------------
# 2. which branch each ray took
# ---------------------------------------------------------------------------------------------------------
def _path_names(trip):
    return (["exit trip %d step %d" % (t, i) for t in (0, 1) for i in range(1, trip + 1)]
            + ["touched trip, then remainder", "exit in remainder", "loop skipped", "exit in shortened step",
               "ran out", "NaN"])


def _classify(hist, ost, steps, alphas, n_full, lo_hi, span, trip):
    """binet_trace_fast's branch for each ray, replayed on the literal loop's history: the trip test is
    (hi(u) - lo_hi) >= span as uint32 over the trip's steps; the exit step (the first u out of the band, under
    the precondition) is the literal loop's.  None for invalid rays."""
    n = alphas.size
    labels = np.array([None] * n, dtype=object)
    exit_full = np.isin(ost, (-1, 1)) & (steps <= n_full)
    exit_idx = np.where(exit_full, steps - 1, n_full)
    n_iter = n_full // (2 * trip)
    span_l = 2 * trip * n_iter
    first = np.full(n, -1)
    if span_l:
        hiw = (hist[:, :span_l].view(np.uint64) >> np.uint64(32)).astype(np.uint32)
        touch = (hiw - np.uint32(lo_hi)) >= np.uint32(span)
        touch &= np.arange(span_l)[None, :] <= exit_idx[:, None]          # (NaN padding after the exit)
        tt = touch.reshape(n, 2 * n_iter, trip).any(axis=2)
        first = np.where(tt.any(axis=1), tt.argmax(axis=1), -1)
    for i in range(n):
        if ost[i] == 0:
            continue
        if not np.isfinite(alphas[i]):
            labels[i] = "NaN"
        elif n_full < 2 * trip:
            labels[i] = "loop skipped"
        elif first[i] >= 0:
            m = int(first[i])
            pos = int(exit_idx[i]) - m * trip
            assert pos >= 0, "exit before the first touched trip"
            labels[i] = ("exit trip %d step %d" % (m % 2, pos + 1)) if pos < trip else "touched trip, then remainder"
        elif exit_full[i]:
            assert exit_idx[i] >= span_l, "an exit in an untouched trip"
            labels[i] = "exit in remainder"
        elif ost[i] == 2:
            labels[i] = "ran out"
        else:
            labels[i] = "exit in shortened step"
    return labels


def test_loop_paths_covered(probe, cases):
    """Every branch of binet_trace_fast ran, for both arithmetics and both trips, at least MIN_PATH_COUNT times
    over the rays the bit-for-bit tests use: exits at each step of either trip, a touched trip followed by the
    remainder loop, exits in the remainder after the whole iterations, the loop skipped, exits in the shortened
    step, rays that run out, NaN rays."""
    counts = {(f, t): dict.fromkeys(_path_names(t), 0) for f in (False, True) for t in TRIPS}
    for c in cases:
        cfg, k, a = c["cfg"], c["k"], c["alphas"]
        if not k["fast_ok"] or k["n_full"] > HISTORY_MAX_STEPS:
            continue
        for fused in (False, True):
            hist, ost, steps = probe.history(fused, cfg, a, k["n_full"])
            ref = probe.trace(3 * fused, cfg, a)
            assert np.array_equal(steps, ref[3]), "history and literal loop disagree on the step count"
            hi_c, hi_e = (k["hi"]["vc"], k["hi"]["ve"]) if fused else (k["hi"]["uc"], k["hi"]["ue"])
            lo_hi, span = (hi_e + 1) & 0xffffffff, (hi_c - hi_e - 1) & 0xffffffff
            for trip in TRIPS:
                for lab in _classify(hist, ost, steps, a, k["n_full"], lo_hi, span, trip):
                    if lab is not None:
                        counts[(fused, trip)][lab] += 1
    lines, short = [], []
    for (fused, trip), cnt in counts.items():
        tag = "%s trip %d" % ("FMA" if fused else "strict", trip)
        lines.append("%-13s " % tag + ", ".join("%s: %d" % kv for kv in cnt.items()))
        short += ["%s: %s (%d)" % (tag, p, v) for p, v in cnt.items() if v < MIN_PATH_COUNT]
    print("\nbinet loop | paths\n    " + "\n    ".join(lines))
    assert not short, "paths run fewer than %d times: %s" % (MIN_PATH_COUNT, short)


# ---------------------------------------------------------------------------------------------------------
# 3. the strict loop against the reference with the device's sine
# ---------------------------------------------------------------------------------------------------------
def _sines(x):
    """sin(x) correctly rounded (mpmath at 200 bits, rounded once) and, where the exact sine lies within
    SIN_CR_NEAR_MIDPOINT ulp of a half-way point, the other neighbouring double (NaN elsewhere)"""
    import mpmath as mp
    rn, other = np.empty(x.size), np.full(x.size, np.nan)
    with mp.workprec(200):
        for i, v in enumerate(x):
            e = mp.sin(mp.mpf(float(v)))
            rn[i] = float(e)
            if e == 0:
                continue
            _, ex = mp.frexp(e)
            pos = abs(e) / mp.ldexp(1, max(int(ex), -1021) - 53)
            if abs(pos - mp.floor(pos) - mp.mpf(0.5)) < SIN_CR_NEAR_MIDPOINT:
                other[i] = np.nextafter(rn[i], np.inf if e > rn[i] else -np.inf)
    return rn, other


def test_strict_equals_oracle_with_device_sine(probe, cases, oracle):
    """The strict literal loop (and with it both strict fast trips, test_fast_equals_generic) against the
    reference's loop restated on the CPU, fed the correctly rounded sine on [0, pi]: status, steps and
    n_half_orbits identical on every ray; final_alpha within FA_QUANTA arccos quanta plus FA_ULP ulp.

    lp_sin_cr is correctly rounded except within SIN_CR_NEAR_MIDPOINT ulp of a half-way point
    (test_gpu_device_math).  The bisected edge rays find such arguments wherever an outcome hinges on the
    sine's last bit: with R_S = 2M, w0^2 = 0 exactly at sin alpha = 1, and next to pi/2 the sine is flat, so
    adjacent alphas straddle the half-way point between 1 - 2^-53 and 1 within 2^-22 ulp.  A ray whose exact
    sine lies that close to a half-way point must equal the reference fed the other rounding instead,
    exactly; those rays are counted."""
    budget = ORACLE_STEP_BUDGET / len(cases)
    worst, worst_at, n_rays, n_steps, n_mid, bad = 0.0, None, 0, 0, 0, []
    for c in cases:
        cfg, a = c["cfg"], c["alphas"]
        a = np.unique(a[(a >= 0.0) & (a <= np.pi)])
        fa, nh, st, steps = probe.trace(0, cfg, a)
        # within the CPU budget: a random subset when the configuration's rays need more steps than its share
        sel = np.random.default_rng(5).permutation(a.size)
        sel = np.sort(sel[np.cumsum(steps[sel].astype(np.int64) + 1) <= budget])
        a, fa, nh, st, steps = a[sel], fa[sel], nh[sel], st[sel], steps[sel]
        sin_rn, sin_other = _sines(a)
        o_fa, o_nh, o_st, o_steps = oracle.trace_rays_batch_sin(*cfg[:3], a, sin_rn, phi_max=cfg[3], h_max=cfg[4])
        n_rays += a.size
        n_steps += int(o_steps.astype(np.int64).sum())
        diff = (st != o_st) | (steps != o_steps) | (nh != o_nh)
        mid = np.nonzero(diff & ~np.isnan(sin_other))[0]
        if mid.size:
            m_fa, m_nh, m_st, m_steps = oracle.trace_rays_batch_sin(*cfg[:3], a[mid], sin_other[mid], phi_max=cfg[3],
                                                                    h_max=cfg[4])
            same = (st[mid] == m_st) & (steps[mid] == m_steps) & (nh[mid] == m_nh)
            mid, m = mid[same], same
            o_fa[mid], o_nh[mid], o_st[mid], o_steps[mid] = m_fa[m], m_nh[m], m_st[m], m_steps[m]
            n_mid += mid.size
            diff[mid] = False
        for i in np.nonzero(diff)[0][:5]:
            bad.append("%s alpha %s: gpu (status %d, steps %d, nh %d) vs reference (%d, %d, %d)" % (
                _cfg_id(cfg), float.hex(float(a[i])), st[i], steps[i], nh[i], o_st[i], o_steps[i], o_nh[i]))
        esc = (o_st == 1) & (st == 1)
        d = np.abs(fa[esc] - o_fa[esc])
        with np.errstate(divide="ignore"):
            quanta = FA_QUANTA * 2.0 ** -52 / np.sin(o_fa[esc])
        ulps = np.maximum(d - quanta, 0.0) / np.spacing(np.abs(o_fa[esc]))
        if ulps.size and ulps.max() > worst:
            j = int(np.argmax(ulps))
            worst, worst_at = float(ulps[j]), (_cfg_id(cfg), float.hex(float(a[esc][j])), float(d[j]))
    print("\nbinet loop | strict literal loop vs reference with the correctly rounded sine: %d rays, %d reference "
          "steps; status / steps / n_half_orbits identical on all but %d (%d more equal the reference with the other "
          "rounding of a sine within 2^-14 ulp of a half-way point); final_alpha beyond %g arccos quanta: "
          "worst %.4f ulp (bar %g) at %r" % (n_rays, n_steps, len(bad), n_mid, FA_QUANTA, worst, FA_ULP, worst_at))
    assert n_steps <= ORACLE_STEP_BUDGET * 1.01
    assert not bad, "\n".join(bad)
    assert worst <= FA_ULP


# ---------------------------------------------------------------------------------------------------------
# 4. the production tracers
# ---------------------------------------------------------------------------------------------------------
def _f32_bits(x):
    """float32 bits with every NaN as 0x7fc00000 (the device's double -> float conversion and numpy's give NaN
    different payloads; the kernels store no meaning in them)"""
    x = np.asarray(x, dtype=np.float32)
    return np.where(np.isnan(x), np.int32(0x7fc00000), x.view(np.int32))


def _stats_of(fa, nh, status, steps, warp_steps=False):
    """lp_frame_stats of per-ray results (fa: the float64 final_alpha, NaN unless escaped)"""
    esc = status == 1
    fin = fa[esc & ~np.isnan(fa)]
    with np.errstate(invalid="ignore"):
        wind = esc & (fa.astype(np.float32) > HALF_PI_F32)
    s = dict(n_rays=int(fa.size), n_escaped=int(esc.sum()), n_captured=int((status == -1).sum()),
             n_invalid=int((status == 0).sum()), n_winding=int(wind.sum()),
             sum_steps=int(steps.astype(np.int64).sum()), max_steps=int(steps.max()) if steps.size else 0,
             max_winding=int(np.clip(nh, 0, 65535).max()) if nh.size else 0,
             min_final_alpha=float(fin.min()) if fin.size else math.inf,
             max_final_alpha=float(fin.max()) if fin.size else 0.0)
    if warp_steps:     # the one-ray-per-thread tracer: warps of 32 consecutive rays
        pad = np.zeros(-steps.size % 32, np.int64)
        s["sum_warp_steps"] = int(32 * np.concatenate([steps.astype(np.int64), pad]).reshape(-1, 32).max(1).sum())
    return s


def _stats_diff(got, want):
    return {k: (got[k], v) for k, v in want.items() if got[k] != v}


def test_production_tracers_equal_probe(probe, cases):
    """ext.trace_batch_f64 and ext.trace_alpha32 (the fast loop wherever its precondition holds) equal the probe's
    literal loops bit for bit in every output, steps included — flags 0: strict, 1: FMA, 4: the hybrid
    composition — and their statistics equal the sums and maxima of the probe's outputs."""
    import torch
    from light_path_tracer_b200 import _lib, _device as dev
    e = _lib.ext()
    bad = []
    for c in cases:
        cfg, a = c["cfg"], c["alphas"]
        for flags in (0, 1, 4):
            ref = probe.hybrid(cfg, a) if flags == 4 else probe.trace(3 if flags == 1 else 0, cfg, a)
            n = a.size
            da = torch.from_numpy(a).cuda()
            fa, w = torch.empty(n, dtype=torch.float64, device="cuda"), torch.empty(n, dtype=torch.int64, device="cuda")
            st, steps = torch.empty(n, dtype=torch.int8, device="cuda"), torch.empty(n, dtype=torch.int32, device="cuda")
            stats = dev.new_stats()
            e.trace_batch_f64(da, *cfg, fa, w, st, steps, stats, flags)
            got = (fa.cpu().numpy(), w.cpu().numpy(), st.cpu().numpy(), steps.cpu().numpy())
            idx, desc = _diff(got, ref, a)
            if idx.size:
                bad.append("trace_batch_f64 %s flags %d: %d rays: %s" % (_cfg_id(cfg), flags, idx.size, desc))
            sd = _stats_diff(dev.read_stats(stats), _stats_of(*ref, warp_steps=True))
            if sd:
                bad.append("trace_batch_f64 %s flags %d stats: %s" % (_cfg_id(cfg), flags, sd))

            with np.errstate(over="ignore"):                # (1e300 becomes inf: one more odd value)
                a32 = a.astype(np.float32)
            ref = probe.hybrid(cfg, a32) if flags == 4 else probe.trace(3 if flags == 1 else 0, cfg, a32)
            fa32, w16 = torch.empty(n, dtype=torch.float32, device="cuda"), torch.empty(n, dtype=torch.uint16, device="cuda")
            stats = dev.new_stats()
            e.trace_alpha32(torch.from_numpy(a32).cuda(), *cfg, fa32, w16, st, steps, stats, flags)
            got = (_f32_bits(fa32.cpu().numpy()), w16.cpu().numpy().astype(np.int64), st.cpu().numpy(),
                   steps.cpu().numpy())
            want = (_f32_bits(ref[0].astype(np.float32)), np.clip(ref[1], 0, 65535), ref[2], ref[3])
            diff = np.nonzero((got[0] != want[0]) | (got[1] != want[1]) | (got[2] != want[2]) | (got[3] != want[3]))[0]
            if diff.size:
                i = diff[0]
                bad.append("trace_alpha32 %s flags %d: %d rays, first alpha %r: %r vs %r" % (
                    _cfg_id(cfg), flags, diff.size, float(a32[i]), [g[i] for g in got], [x[i] for x in want]))
            sd = _stats_diff(dev.read_stats(stats), _stats_of(*ref, warp_steps=True))
            if sd:
                bad.append("trace_alpha32 %s flags %d stats: %s" % (_cfg_id(cfg), flags, sd))
    assert not bad, "\n".join(bad[:20])


# ---------------------------------------------------------------------------------------------------------
# 5. the frame kernels at odd budgets
# ---------------------------------------------------------------------------------------------------------
# n_full mod 8 = 1, 3, 5, 7 (201, 403, 605, 807), n_full < 4 (3), phi_shift 3 (60 / 0.05)
FRAME_BUDGETS = [(0.05 * n + 0.025, 0.05) for n in (3, 201, 403, 605, 807)] + [(60.0, 0.05)]


def _frame_geometries():
    """(H, W, r_obs, fov, psi): psi = 0 takes the mirror-image kernel, psi != 0 the one-ray-per-pixel kernel"""
    def fov_of(H, W, vfov):
        return (2 * np.arctan(np.tan(vfov / 2) * W / H), vfov)
    a_c = math.asin(3.0 * math.sqrt(3.0) * math.sqrt(1.0 - 2.0 / 100.0) / 100.0)
    return [(101, 250, 15.0, fov_of(101, 250, np.radians(40.0)), (0.0, 0.0)),
            (101, 250, 15.0, fov_of(101, 250, np.radians(40.0)), (0.04, -0.03)),
            (270, 480, 100.0, fov_of(270, 480, np.radians(12.0)), (0.0, 0.0)),
            (270, 480, 100.0, fov_of(270, 480, np.radians(12.0)), (0.02, 0.03)),
            (101, 250, 100.0, fov_of(101, 250, 0.004), (0.0, a_c))]          # narrow, across the critical ring


def _frame_child(so_path):
    """Render every (budget, geometry, strict / hybrid, schedule, source type) and compare with the probe; prints
    one RESULT line (failures, frame digests).  Runs in a subprocess: LP_RENDER_TRIP is read once per process."""
    import torch
    from light_path_tracer_b200 import _lib, _device as dev, image_lens as il
    probe = _Probe(so_path)
    e = _lib.ext()
    g = torch.Generator(device="cuda").manual_seed(11)
    bad, digests, n_frames = [], {}, 0
    for phi_max, h_max in FRAME_BUDGETS:
        for H, W, r_obs, fov, psi in _frame_geometries():
            cfg = (1.0, 2.0, r_obs, phi_max, h_max)
            cam = dev.camera_vector((H, W), fov, psi, il._psi_frame)
            a32 = il.build_alpha_lookup((H, W), fov, psi=psi, device=True)
            src = torch.rand(H, W, 3, device="cuda", generator=g)
            srcs = {"f32": (src, False), "u8": ((src * 255).to(torch.uint8), True)}
            for flags in (0, 4):
                ref = probe.hybrid(cfg, a32) if flags else probe.trace(0, cfg, a32)
                want_fa = torch.from_numpy(_f32_bits(ref[0].astype(np.float32)).reshape(H, W)).cuda()
                want_w = torch.from_numpy(np.clip(ref[1], 0, 65535).astype(np.uint16).reshape(H, W)).cuda()
                want_stats = _stats_of(*ref)
                frames = {}
                for sched in (0, dev.TRACE_REPACK):
                    for name, (s, unit) in srcs.items():
                        tag = "budget %g/%g %dx%d r%g psi %r flags %d %s" % (phi_max, h_max, W, H, r_obs, psi,
                                                                             flags | sched, name)
                        out = torch.empty_like(s)
                        fa = torch.empty((H, W), dtype=torch.float32, device="cuda")
                        w = torch.empty((H, W), dtype=torch.uint16, device="cuda")
                        stats = dev.new_stats()
                        e.render_frame(s, 3, cam, 0, H, *cfg, False, il.SAMPLE_NEAREST, out, fa, w, stats,
                                       flags | sched, unit, 0, 0)
                        n_frames += 1
                        got_fa = torch.where(torch.isnan(fa), torch.full_like(fa.view(torch.int32), 0x7fc00000),
                                             fa.view(torch.int32))
                        if not torch.equal(got_fa, want_fa):
                            bad.append("%s: final_alpha lookup differs at %d pixels" % (
                                tag, int((got_fa != want_fa).sum())))
                        if not torch.equal(w, want_w):
                            bad.append("%s: winding lookup differs at %d pixels" % (tag, int((w != want_w).sum())))
                        sd = _stats_diff(dev.read_stats(stats), want_stats)
                        if sd:
                            bad.append("%s: stats %s" % (tag, sd))
                        frames[(sched, name)] = out
                for name in srcs:
                    if not torch.equal(frames[(0, name)], frames[(dev.TRACE_REPACK, name)]):
                        bad.append("budget %g/%g %dx%d r%g psi %r flags %d %s: frame differs from the re-packing "
                                   "kernel's" % (phi_max, h_max, W, H, r_obs, psi, flags, name))
                    digests["%g %dx%d r%g %r %d %s" % (phi_max, W, H, r_obs, psi, flags, name)] = hashlib.sha256(
                        frames[(0, name)].cpu().numpy().tobytes()).hexdigest()
    print("RESULT " + json.dumps({"bad": bad, "digests": digests, "frames": n_frames}))


def _run_frame_child(so, trip):
    env = dict(os.environ)
    env.pop("LP_RENDER_TRIP", None)
    if trip:
        env["LP_RENDER_TRIP"] = str(trip)
    code = "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import test_gpu_binet_loop as T; " \
           "T._frame_child(%r)" % (ROOT, TESTS, so)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    return json.loads(line[len("RESULT "):])


def test_frame_kernels_odd_budgets(probe_so):
    """ext.render_frame at budgets of n_full mod 8 = 1, 3, 5, 7, n_full < 4 and phi_shift 3, through the mirror-image
    kernel (psi = 0), the one-ray-per-pixel kernel (psi != 0) and the re-packing kernel (LP_TRACE_REPACK), strict and
    hybrid, 8-bit unit and float32 sources, with LP_RENDER_TRIP unset, 2 and 4 (one subprocess each): the
    final_alpha / winding lookups and the statistics equal the probe's literal loops (hybrid: its composition) on
    build_alpha_lookup's float32 table; the frames equal the re-packing kernel's and do not depend on the trip."""
    results = {trip: _run_frame_child(probe_so, trip) for trip in (None, 2, 4)}
    bad = ["LP_RENDER_TRIP=%s: %s" % (t, b) for t, r in results.items() for b in r["bad"]]
    base = results[None]["digests"]
    for t in (2, 4):
        diff = [k for k, v in results[t]["digests"].items() if base.get(k) != v]
        if diff:
            bad.append("LP_RENDER_TRIP=%d: frames differ from the default's: %s" % (t, diff[:5]))
    print("\nbinet loop | frames: %d renders per trip setting, %d budgets" % (results[None]["frames"],
                                                                           len(FRAME_BUDGETS)))
    assert not bad, "\n".join(bad[:30])
