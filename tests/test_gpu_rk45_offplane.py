"""Whole integrations of the generic RK45 integrator off the equator and with angular momentum, against
the oracle's restatement of scipy's RK45 (oracle/lp_oracle_rk45.c), ray by ray.

Kerr rays come from Kerr.initial_conditions at every screen angle, so p_phi != 0 and theta leaves the
equator: the frame-dragging, p_phi^2 and 1/sin^2(theta) terms of the Kerr right-hand side all steer the
ray.  They run through both Kerr kernels: the batch path (geodesic_tracer._paths(Kerr, state0=...),
lp_kerr_rk45_integrate_paths) and the dense single-ray path (integrate_geodesic).  Off-plane Schwarzschild
states (tilted orbital planes, polar planes, rays that pass the pole closer than the right-hand side's
sin^2(theta) floor of 1e-15) run through the six-component kernel.

The bar is test_gpu_rk45.py's test_batch_vs_oracle:
- status and outcome exact, except for a ray whose own oracle outcome changes when its initial state moves
  by one ulp; a Schwarzschild ray whose oracle trajectory reaches the floor (sin^2(theta) < 1e-15) is held
  to its outcome only: there the 1 / sin^3(theta) term of p_theta' makes any rounding decide whether the
  step size collapses at the pole (status -1), and on which side of the pole the ray leaves it;
- accepted points and nfev exact for at least 99.8 % of the Kerr and of the Schwarzschild rays, not counting
  rays whose own oracle step sequence changes when the initial state moves by one ulp or that reach the floor
  (the near-polar Schwarzschild rays: there one ulp of sin(theta) decides the steps); the rest agree to 1e-5
  (plus the movement below);
- final 8-state and lambda within 1e-9 relative (FLOOR), plus 3 x the oracle's own movement when state0's
  r, theta, p_r and p_theta move one ulp each way (it stands in for CUDA's sincos against glibc and for the
  conditioning near photon orbits; computed only for the rays the plain bar does not already pass);
- dense path: trajectories within 1e-7 as in the golden test, plus 3 x the oracle's own trajectory movement
  under the same one-ulp moves (the step-size controller's jitter moves intermediate points by up to ~1e-6);
  final state, nfev and status bit-identical to the batch kernel's;
- p_t and p_phi bit-identical to state0 in every output row;
- for rays with the same step sequence, the drift of the Carter constant (Kerr) or of the total angular
  momentum p_theta^2 + p_phi^2 / sin^2(theta) (Schwarzschild, on orbits that stay above the floor) at most
  2 x the oracle's drift + 1e-9 max(1, |Q0|).  This check depends on no restatement.
Both batches run once with the library's defaults and once with LP_RK45_POW=1 (the step controller's
inv_tenth_root form), each in a subprocess because the library reads the knob once per process.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import record_parity

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REL_TOL = 1e-9
FLOOR = np.array([1.0, 1.0, 1.0, 1e-3, 1.0, 1e-3, 1e-6, 1.0])
SPREAD_FACTOR = 3.0
FLIP_SHARE = 2e-3
FLIP_TOL = 1e-5
PERTURBED = (1, 2, 5, 6)                  # r, theta, p_r, p_theta of state0

# (M, a / M, r_obs / M, theta_obs)
KERR_CONFIGS = [(1.0, 0.9, 30.0, 1.1), (1.0, -0.998, 12.0, 0.3), (2.5, 0.3, 100.0, np.pi / 2),
                (1.0, 1e-6, 6.0, 1.1), (1.0, 0.3, 1000.0, 0.05), (2.5, 0.998, 12.0, np.pi - 0.2),
                (1.0, 1.0, 30.0, 0.3), (1.0, -0.9, 100.0, 1.1), (2.5, 0.9, 6.0, np.pi / 2),
                (1.0, 0.998, 100.0, 0.05)]
KERR_RAYS = 2000
DENSE_RAYS = 20                           # per configuration, through integrate_geodesic


def _kerr_states(M, q, r_obs_M, th_obs, seed):
    from light_path_tracer_b200.metrics import Kerr
    m = Kerr(M, q * M)
    r_obs = r_obs_M * M
    rng = np.random.default_rng(seed)
    ac = float(m.alpha_crit(r_obs, th_obs))
    n_band = KERR_RAYS * 3 // 10
    alpha = np.concatenate([rng.uniform(0, 2 * ac, KERR_RAYS - n_band), ac * rng.uniform(0.6, 1.05, n_band)])
    screen = -np.pi + (np.pi - rng.uniform(0, 2 * np.pi, KERR_RAYS))          # (-pi, pi]
    screen[DENSE_RAYS:DENSE_RAYS + 40] = np.tile([0.0, np.pi / 2, -np.pi / 2, np.pi], 10)
    return np.array([m.initial_conditions(r_obs, float(al), float(sc), th_obs) for al, sc in zip(alpha, screen)])


def _schw_states(M, r0, seed):
    """photons at r0 heading inwards: tilted orbital planes, polar planes (p_phi = 0) and near-polar planes
    (|p_phi| / L = 1e-6, 1e-8, 1e-10: the orbit's closest approach to the pole has sin(theta) = |p_phi| / L,
    so the last two cross the sin^2 floor)"""
    rng = np.random.default_rng(seed)
    n = SCHW_RAYS
    R_S = 2 * M
    f = 1 - R_S / r0
    b_crit = 3 * np.sqrt(3) * M
    L = np.concatenate([rng.uniform(0.05, 2.5, n // 2), rng.uniform(0.9, 1.1, n - n // 2)]) * b_crit
    th0 = rng.uniform(0.2, np.pi - 0.2, n)
    kind = np.arange(n) % 5
    psi = rng.uniform(-np.pi, np.pi, n)
    ratio = np.choose(kind, [np.cos(psi), np.zeros(n), np.full(n, 1e-6), np.full(n, 1e-8), np.full(n, 1e-10)])
    sgn = np.where(rng.random(n) < 0.5, -1.0, 1.0)
    p_phi = ratio * L * np.where(kind == 0, np.sin(th0), sgn)
    p_th = np.where(rng.random(n) < 0.5, -1.0, 1.0) * np.sqrt(np.maximum(L ** 2 - p_phi ** 2 / np.sin(th0) ** 2, 0))
    p_r_sq = (1 / f - L ** 2 / r0 ** 2) / f
    keep = p_r_sq > 0
    s0 = np.stack([np.zeros(n), np.full(n, r0), th0, rng.uniform(-1, 1, n), np.full(n, -1.0),
                   -np.sqrt(np.where(keep, p_r_sq, 0)), p_th, p_phi], axis=1)
    return s0[keep]


SCHW_CONFIGS = [(1.0, 10.0), (1.0, 30.0), (2.5, 100.0), (1.0, 300.0)]
SCHW_RAYS = 600


@pytest.fixture(scope="module")
def batches():
    """{tag: (metric (M, a) or (M,), state0 [n, 8])}"""
    out = {}
    for k, (M, q, r_obs_M, th_obs) in enumerate(KERR_CONFIGS):
        out["kerr%d" % k] = ((M, q * M), _kerr_states(M, q, r_obs_M, th_obs, 100 + k))
    for k, (M, r0) in enumerate(SCHW_CONFIGS):
        out["schw%d" % k] = ((M,), _schw_states(M, r0, 200 + k))
    return out


def _oracle_run(oracle, metric, s0, max_points=4):
    if len(metric) == 2:
        return oracle.rk45_integrate_kerr(metric[0], metric[1], s0, max_points=max_points)
    return oracle.rk45_trace_ray(metric[0], None, None, state0=s0, max_points=max_points)


class _Oracle:
    """the oracle's result per ray, and (on demand) its results from the eight one-ulp moves of state0"""

    def __init__(self, oracle, batches):
        self.oracle, self.batches, self.res, self.moved = oracle, batches, {}, {}
        for tag, (metric, s0) in batches.items():
            rs = [_oracle_run(oracle, metric, s) for s in s0]
            self.res[tag] = dict(state=np.array([r["y_final"] for r in rs]), lam=np.array([r["t_final"] for r in rs]),
                                 oc=np.array([r["outcome"] for r in rs]), st=np.array([r["status"] for r in rs]),
                                 ns=np.array([(r["n_points"], r["nfev"]) for r in rs]))

    def spread(self, tag, i):
        """(largest relative movement of the final state, of lambda; did the outcome or status change; did the
        accepted points or nfev change)"""
        key = (tag, i)
        if key not in self.moved:
            metric, s0 = self.batches[tag]
            ref = self.res[tag]
            sp, sp_l, flips, steps = 0.0, 0.0, False, False
            for c in PERTURBED:
                for to in (np.inf, -np.inf):
                    s = s0[i].copy()
                    s[c] = np.nextafter(s[c], to)
                    o = _oracle_run(self.oracle, metric, s)
                    flips |= (o["outcome"] != ref["oc"][i]) or (o["status"] != ref["st"][i])
                    steps |= (o["n_points"], o["nfev"]) != tuple(ref["ns"][i])
                    with np.errstate(invalid="ignore"):
                        sp = max(sp, float(np.nanmax(np.abs(o["y_final"] - ref["state"][i]) /
                                                     np.maximum(np.abs(ref["state"][i]), FLOOR))))
                        sp_l = max(sp_l, abs(o["t_final"] - ref["lam"][i]) / max(abs(ref["lam"][i]), 1.0))
            self.moved[key] = (sp, sp_l, flips, steps)
        return self.moved[key]

    def at_floor(self, tag, i):
        """does the oracle's Schwarzschild trajectory reach sin^2(theta) < 1e-15, where the floor decides the
        motion and the 1 / sin^3(theta) term of p_theta' makes every rounding decisive"""
        metric, s0 = self.batches[tag]
        if len(metric) == 2:
            return False
        o = _oracle_run(self.oracle, metric, s0[i], max_points=1 << 20)
        return bool((np.sin(o["y"][2]) ** 2 < 1e-15).any())

    def traj_spread(self, tag, i):
        """largest movement of the oracle's trajectory (_traj_err) under the one-ulp moves of state0 that keep
        its step sequence: the step-size controller's jitter moves intermediate points far more than the end"""
        metric, s0 = self.batches[tag]
        ref = _oracle_run(self.oracle, metric, s0[i], max_points=8192)
        worst = 0.0
        for c in PERTURBED:
            for to in (np.inf, -np.inf):
                s = s0[i].copy()
                s[c] = np.nextafter(s[c], to)
                o = _oracle_run(self.oracle, metric, s, max_points=8192)
                if o["n_points"] == ref["n_points"]:
                    worst = max(worst, _traj_err(o["t"], o["y"], ref))
        return worst


def _traj_err(t, y, o):
    """t and r as the golden test, the other components relative above 1 (p_theta and phi cross 0)"""
    tf = max(1.0, float(o["t"][-1]))
    return max(np.abs(t - o["t"]).max() / tf, (np.abs(y[1] - o["y"][1]) / o["y"][1]).max(),
               (np.abs(y - o["y"]) / np.maximum(np.abs(o["y"]), 1.0)).max())


@pytest.fixture(scope="module")
def oracle_res(oracle, batches):
    return _Oracle(oracle, batches)


CHILD = r'''
import sys
import numpy as np
sys.path.insert(0, %(root)r)
from light_path_tracer_b200 import geodesic_tracer as gt
from light_path_tracer_b200.metrics import Schwarzschild, Kerr
src = np.load(sys.argv[1])
out = {}
for tag in sorted({k.split("__")[0] for k in src.files}):
    metric, s0 = src[tag + "__metric"], src[tag + "__state0"]
    m = Kerr(*metric) if metric.size == 2 else Schwarzschild(*metric)
    # the first 2048 points of every trajectory (a ray the floor traps near a pole takes 1e5 steps)
    traj, npts, state, lam, oc, ns, st, _, _ = gt._paths(m, state0=s0, max_points=2048)
    live = np.arange(traj.shape[1])[None, :] < npts[:, None]
    bits = lambda x: np.ascontiguousarray(x).view(np.int64)
    const = (bits(traj[:, :, 5]) == bits(s0[:, 4])[:, None]) & (bits(traj[:, :, 8]) == bits(s0[:, 7])[:, None])
    const = (const | ~live).all(axis=1) & (npts >= 1) & (bits(state[:, 4]) == bits(s0[:, 4])) & \
        (bits(state[:, 7]) == bits(s0[:, 7]))
    for k, v in (("state", state), ("lam", lam), ("oc", oc), ("ns", ns), ("st", st), ("const", const)):
        out[tag + "__" + k] = v
np.savez(sys.argv[2], **out)
'''


def _device(batches, tmp_path, pow_knob):
    src = str(tmp_path / ("in_%s.npz" % pow_knob))
    dst = str(tmp_path / ("out_%s.npz" % pow_knob))
    np.savez(src, **{k: v for tag, (metric, s0) in batches.items()
                     for k, v in ((tag + "__metric", np.array(metric)), (tag + "__state0", s0))})
    env = dict(os.environ)
    env.pop("LP_RK45_POW", None)
    if pow_knob != "default":
        env["LP_RK45_POW"] = pow_knob
    r = subprocess.run([sys.executable, "-c", CHILD % {"root": ROOT}, src, dst], env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    res = np.load(dst)
    return {tag: {k: res[tag + "__" + k] for k in ("state", "lam", "oc", "ns", "st", "const")} for tag in batches}


def _conserved(metric, y):
    """Carter constant (Kerr) or total angular momentum (Schwarzschild) of states y [n, 8]"""
    th, p_t, p_th, p_phi = y[:, 2], y[:, 4], y[:, 6], y[:, 7]
    s2, c2 = np.sin(th) ** 2, np.cos(th) ** 2
    if len(metric) == 2:
        return p_th ** 2 + c2 * (p_phi ** 2 / s2 - metric[1] ** 2 * p_t ** 2)
    return p_th ** 2 + p_phi ** 2 / s2


def _check(tag, metric, s0, dev, orc, setting):
    ref = orc.res[tag]
    n = s0.shape[0]
    assert dev["const"].all(), "%s: p_t / p_phi moved in %d rays" % (tag, int((~dev["const"]).sum()))
    same = (dev["ns"] == ref["ns"]).all(axis=1)
    err = (np.abs(dev["state"] - ref["state"]) / np.maximum(np.abs(ref["state"]), FLOOR)).max(axis=1)
    err_l = np.abs(dev["lam"] - ref["lam"]) / np.maximum(np.abs(ref["lam"]), 1.0)
    match = (dev["oc"] == ref["oc"]) & (dev["st"] == ref["st"])
    base = np.where(same, REL_TOL, FLIP_TOL)
    worst_spread, n_spread, n_floor = 0.0, 0, 0
    for i in np.nonzero(~same | ~match | ~(err <= base) | ~(err_l <= base))[0]:
        # a ray that reaches the floor: only the outcome is held (the rounding decides the status and on which
        # side of the pole the ray leaves it)
        if dev["oc"][i] == ref["oc"][i] and orc.at_floor(tag, int(i)):
            n_floor += 1
            continue
        sp, sp_l, moved, _ = orc.spread(tag, int(i))
        worst_spread, n_spread = max(worst_spread, sp), n_spread + 1
        if not match[i]:
            assert moved, "%s ray %d: outcome / status %s vs oracle %s, stable under 1-ulp moves" % (
                tag, i, (dev["oc"][i], dev["st"][i]), (ref["oc"][i], ref["st"][i]))
            continue
        assert err[i] <= base[i] + SPREAD_FACTOR * sp and err_l[i] <= base[i] + SPREAD_FACTOR * sp_l, (
            tag, int(i), s0[i].tolist(), err[i], err_l[i], sp, sp_l)
    flips = int((~same).sum())
    unstable = np.array([not same[i] and (orc.spread(tag, int(i))[3] or orc.at_floor(tag, int(i)))
                         for i in range(n)])
    stable = np.nonzero(~same & ~unstable)[0]
    stable_flips = int(stable.size)
    for i in stable:
        print("\n%s %s ray %d: steps %s vs oracle %s, |p_phi| / sqrt(Q0) = %.1e, final rel err %.2e"
              % (setting, tag, i, dev["ns"][i].tolist(), ref["ns"][i].tolist(),
                 abs(s0[i, 7]) / max(np.sqrt(abs(_conserved(metric, s0[i:i + 1])[0])), 1e-300), err[i]))
    # drift of the conserved quantity, on the rays with the oracle's step sequence
    q0 = _conserved(metric, s0)
    fin = same & match & np.isfinite(ref["state"]).all(axis=1)
    if len(metric) == 1:        # away from the floor: the orbit's sin^2(theta) >= p_phi^2 / L^2 stays above it
        fin &= s0[:, 7] ** 2 >= 1e-14 * q0
    drift = np.abs(_conserved(metric, dev["state"][fin]) - q0[fin])
    drift_o = np.abs(_conserved(metric, ref["state"][fin]) - q0[fin])
    allowed = 2 * drift_o + 1e-9 * np.maximum(1.0, np.abs(q0[fin]))
    assert (drift <= allowed).all(), (tag, int((drift > allowed).sum()), float((drift - allowed).max()))
    rel = lambda x: float((x / np.maximum(1.0, np.abs(q0[fin]))).max()) if fin.any() else 0.0
    ok = same & match
    print("\n%s %-6s %s: %d rays, %d flips (%d of them where the oracle's own steps are stable), worst rel err "
          "%.2e (state) %.2e (lambda) on the same steps; %d needed the 1-ulp spread (largest %.2e); "
          "conserved-quantity drift %.2e (oracle %.2e); %d differing rays that reach the floor"
          % (setting, tag, metric, n, flips, stable_flips, err[ok].max(), err_l[ok].max(), n_spread, worst_spread,
             rel(drift), rel(drift_o), n_floor))
    return flips, stable_flips, n, worst_spread


@pytest.mark.parametrize("pow_knob", ["default", "1"], ids=["pow_default", "pow_1"])
def test_offplane_batches_vs_oracle(batches, oracle_res, tmp_path, native, pow_knob):
    """Kerr rays with angular momentum (lp_kerr_rk45_integrate_paths) and off-plane Schwarzschild states
    (the six-component kernel) against the oracle, ray by ray (module docstring)"""
    dev = _device(batches, tmp_path, pow_knob)
    totals = {"kerr": [0, 0, 0, 0.0], "schw": [0, 0, 0, 0.0]}
    for tag, (metric, s0) in batches.items():
        flips, stable_flips, n, sp = _check(tag, metric, s0, dev[tag], oracle_res, "LP_RK45_POW=" + pow_knob)
        t = totals[tag[:4]]
        t[0], t[1], t[2], t[3] = t[0] + flips, t[1] + stable_flips, t[2] + n, max(t[3], sp)
    for fam, (flips, stable_flips, n, sp) in totals.items():
        record_parity("rk45_offplane_%s_pow_%s" % (fam, pow_knob), rays=n, step_sequence_flips=flips,
                      flips_where_oracle_steps_stable=stable_flips, worst_one_ulp_spread=sp)
        print("\nLP_RK45_POW=%s %s: %d rays, %d flips, %d where the oracle's own steps are stable; largest 1-ulp "
              "spread %.2e" % (pow_knob, fam, n, flips, stable_flips, sp))
    for fam, (flips, stable_flips, n, sp) in totals.items():
        assert stable_flips <= FLIP_SHARE * n, "%s: %d of %d rays with a different step sequence where the " \
            "oracle's own sequence is stable under one-ulp moves" % (fam, stable_flips, n)


def test_dense_single_ray_path(batches, oracle_res, native):
    """integrate_geodesic (the dense Kerr and six-component kernels) on the first rays of every batch:
    trajectory within 1e-7 of the oracle's, as in the golden test; final state, lambda, nfev, status and
    outcome bit-identical to the batch kernel's; p_t and p_phi constant in every row"""
    from light_path_tracer_b200 import geodesic_tracer as gt
    from light_path_tracer_b200.metrics import Schwarzschild, Kerr
    worst, n_spread = 0.0, 0
    for tag, (metric, s0) in batches.items():
        m = Kerr(*metric) if len(metric) == 2 else Schwarzschild(*metric)
        ref = oracle_res.res[tag]
        sub = s0[:DENSE_RAYS]
        _, npts_b, state_b, lam_b, oc_b, ns_b, st_b, _, _ = gt._paths(m, state0=sub)
        for i, s in enumerate(sub):
            sol, outcome = gt.integrate_geodesic(m, s)
            assert np.array_equal(sol.y[:, -1], state_b[i]) and sol.t[-1] == lam_b[i], (tag, i)
            assert (sol.t.size, sol.nfev, sol.status) == (npts_b[i], ns_b[i, 1], st_b[i]), (tag, i)
            assert outcome == {1: "escaped", -1: "captured"}[int(oc_b[i])]
            assert (sol.y[4] == s[4]).all() and (sol.y[7] == s[7]).all()
            if (sol.t.size, sol.nfev) != tuple(ref["ns"][i]):
                continue
            o = _oracle_run(oracle_res.oracle, metric, s, max_points=8192)
            e = _traj_err(sol.t, sol.y, o)
            if e > 1e-7:        # the oracle's own movement under one-ulp moves, as for the final state
                sp = oracle_res.traj_spread(tag, i)
                assert e <= 1e-7 + SPREAD_FACTOR * sp, (tag, i, e, sp)
                n_spread += 1
            worst = max(worst, e)
    print("\ndense single-ray path: %d rays, worst trajectory difference %.2e (%d above 1e-7 needed the oracle's "
          "own 1-ulp movement)" % (DENSE_RAYS * len(batches), worst, n_spread))
