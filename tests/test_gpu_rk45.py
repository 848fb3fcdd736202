"""GPU parity of kernel (1b), the batched 8-D Hamiltonian tracer with scipy-RK45 semantics,
through the reference-facing API (light_path_tracer_b200.geodesic_tracer -> torch extension
-> C ABI lp_schw_rk45_*).

Checkers: tests/golden/rk45_rays.npz (the UNMODIFIED reference: geodesic_tracer.trace_ray on
scipy 1.18.1) and the oracle's restatement of scipy's RK45 (oracle/lp_oracle_rk45.c, pinned to
the same fixture in test_oracle_golden.py).

Bar: outcome exact (except within 1e-9 of the critical impact parameter); number of accepted
points and nfev exact (they are integers: the whole accept/reject sequence is reproduced);
final 8-state and affine parameter within 1e-9 relative.  scipy forms its stage sums with
BLAS, so bit equality is not defined (SURVEY.md 7.3 H7).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

REL_TOL = 1e-9
# absolute floors per state component (t, r, theta, phi, p_t, p_r, p_theta, p_phi): theta and
# p_theta hover at pi/2 and ~1e-17 (cos(pi/2) = 6e-17 drives them), phi can be exactly 0
FLOOR = np.array([1.0, 1.0, 1.0, 1e-3, 1.0, 1e-3, 1e-6, 1.0])


def _gt():
    from light_path_tracer_b200 import geodesic_tracer
    return geodesic_tracer


def _metric(M):
    from light_path_tracer_b200.metrics import Schwarzschild
    return Schwarzschild(M)


def test_golden_rays_single_ray_api(native, golden):
    """Every ray of the reference fixture through trace_ray: OdeResult-shaped solution,
    whole accepted-step trajectory, event point, nfev, outcome."""
    gt = _gt()
    g = golden("rk45_rays.npz")
    off = g["traj_offsets"]
    names = {1: "escaped", -1: "captured"}
    worst_final, worst_traj = 0.0, 0.0
    for i in range(g["alpha"].size):
        metric = _metric(float(g["M"][i]))
        sol, outcome = gt.trace_ray(metric, float(g["r_obs"][i]), float(g["alpha"][i]))
        assert outcome == names[int(g["outcome"][i])], i
        assert sol.y.shape == (8, int(g["n_points"][i])) and sol.t.shape == (int(g["n_points"][i]),), i
        assert sol.nfev == int(g["nfev"][i]) and sol.status == int(g["status"][i]), i
        assert sol.success and sol.t[0] == 0.0
        np.testing.assert_array_equal(sol.y[:, 0], g["state0"][i])
        e_final = np.abs(sol.y[:, -1] - g["y_final"][i]) / np.maximum(np.abs(g["y_final"][i]), FLOOR)
        assert e_final.max() <= REL_TOL, (i, e_final)
        assert abs(sol.t[-1] - g["t_final"][i]) <= REL_TOL * max(1.0, g["t_final"][i])
        tr_t, tr_r, tr_p = (g[k][off[i]:off[i + 1]] for k in ("traj_t", "traj_r", "traj_phi"))
        # intermediate points carry the controller's step-size jitter (pow / dot rounding): 1e-7
        e_traj = max(np.abs(sol.t - tr_t).max() / max(1.0, tr_t.max()), (np.abs(sol.y[1] - tr_r) / tr_r).max(),
                     np.abs(sol.y[3] - tr_p).max())
        assert e_traj <= 1e-7, (i, e_traj)
        # the terminal event is recorded like scipy does
        k = 0 if outcome == "captured" else 1
        assert sol.t_events[k].shape == (1,) and sol.t_events[1 - k].shape == (0,)
        assert sol.t_events[k][0] == sol.t[-1] and np.array_equal(sol.y_events[k][0], sol.y[:, -1])
        worst_final, worst_traj = max(worst_final, e_final.max()), max(worst_traj, e_traj)
    print("30 reference rays: worst final-state rel err %.2e, worst trajectory err %.2e" % (worst_final, worst_traj))


def test_invalid_and_reference_table(native):
    """geodesic_tracer.py:153-172: the printed alpha -> outcome table at r_obs = 50 M
    (0..5.5 deg captured, 5.97..15 deg escaped); trace_ray returns (None, 'invalid') when
    initial_conditions returns None."""
    gt = _gt()
    metric = _metric(1.0)
    rows = gt.outcome_table(metric, 50.0, [0, 2, 4, 5, 5.5, 5.97, 6.5, 8, 10, 15])
    assert [r[2] for r in rows] == ["CAPTURED"] * 5 + ["ESCAPED"] * 5

    class NoRay(type(metric)):
        def initial_conditions(self, r_obs, alpha, theta=0.0, theta_obs=np.pi / 2):
            return None
    assert gt.trace_ray(NoRay(1.0), 50.0, 0.1) == (None, 'invalid')


@pytest.mark.parametrize("M,r_obs", [(1.0, 100.0), (1.0, 50.0), (2.0, 30.0), (1.0, 8.0)])
def test_batch_vs_oracle(native, oracle, M, r_obs):
    """Seeded batch (uniform + a cluster at the critical angle + odd inputs) against the
    oracle's scipy restatement, ray by ray."""
    gt = _gt()
    metric = _metric(M)
    rng = np.random.default_rng(int(r_obs))
    ac = float(oracle.alpha_crit(M, r_obs))
    alpha = np.concatenate([rng.uniform(0, np.pi, 6000), ac * (1 + rng.normal(0, 1e-2, 3000)),
                            ac * (1 + rng.normal(0, 1e-5, 1000)), rng.uniform(0, 2 * ac, 2000),
                            [0.0, np.pi / 2, np.pi, 1e-9, -0.2, 3.5, np.nan]])
    state, lam, outcome, nsteps, status = gt.trace_rays(metric, r_obs, alpha, return_status=True)
    s_o, l_o, oc_o, ns_o, st_o = oracle.rk45_trace_batch(M, r_obs, alpha)
    b = r_obs * np.sin(alpha) / np.sqrt(1 - 2 * M / r_obs)
    in_band = np.abs(b - 3 * np.sqrt(3) * M) <= 1e-9
    assert np.array_equal(outcome[~in_band], oc_o[~in_band])
    assert np.array_equal(status, st_o)
    valid = oc_o != 0
    assert np.isnan(state[~valid]).all() and np.isnan(lam[~valid]).all() and (~valid).sum() >= 1
    same_steps = (nsteps == ns_o).all(axis=1)
    # The batch path integrates the four live components of an equatorial ray and reports
    # theta = pi/2, p_theta = 0 (csrc/lp_rk45.cu, lp_rk45_eq_kernel).  What the reference holds in
    # those two slots is the rounding noise of cos(pi/2) = 6.1e-17 integrated along the ray: checked
    # to BE noise here (|p_theta| <= 1e-12, theta within 1e-14 of pi/2) and compared on that scale;
    # the six-component kernel behind the single-ray API reproduces it (tests above / below).
    assert np.abs(s_o[valid, 6]).max() <= 1e-12 and np.abs(s_o[valid, 2] - np.pi / 2).max() <= 1e-14
    assert np.abs(state[valid, 6]).max() <= 1e-12 and np.abs(state[valid, 2] - np.pi / 2).max() <= 1e-14
    live = [0, 1, 3, 4, 5, 7]
    err = (np.abs(state - s_o) / np.maximum(np.abs(s_o), FLOOR))[:, live].max(axis=1)
    err_l = np.abs(lam - l_o) / np.maximum(np.abs(l_o), 1.0)
    ok = valid & same_steps
    # Conditioning clause: a ray that grazes the photon sphere amplifies ANY rounding
    # difference (the kernel's reciprocals and fma sums, scipy's BLAS sums) like 1/|b - b_crit|.
    # Measure that amplification with the oracle itself — how far does the reference's own
    # result move when the viewing angle moves by ONE ulp — and allow twice that on top of 1e-9.
    # It is below 1e-12 for all but a handful of rays per batch.
    spread = np.zeros(alpha.size)
    spread_l = np.zeros(alpha.size)
    for shifted in (np.nextafter(alpha, np.inf), np.nextafter(alpha, -np.inf)):
        s_p, l_p, _, _, _ = oracle.rk45_trace_batch(M, r_obs, shifted)
        with np.errstate(invalid="ignore"):
            spread = np.fmax(spread, (np.abs(s_p - s_o) / np.maximum(np.abs(s_o), FLOOR))[:, live].max(axis=1))
            spread_l = np.fmax(spread_l, np.abs(l_p - l_o) / np.maximum(np.abs(l_o), 1.0))
    tol, tol_l = REL_TOL + 2 * spread, REL_TOL + 2 * spread_l
    print("M=%g r_obs=%g: %d rays, %d with a different accept/reject sequence; worst rel err %.2e (state) "
          "%.2e (lambda); %d rays with 1-ulp sensitivity above 1e-10 (max %.2e)"
          % (M, r_obs, alpha.size, int((valid & ~same_steps).sum()), err[ok].max(), err_l[ok].max(),
             int((spread > 1e-10).sum()), spread.max()))
    assert (err[ok] <= tol[ok]).all() and (err_l[ok] <= tol_l[ok]).all()
    assert (spread > 1e-10).sum() <= 0.005 * alpha.size
    # a borderline error norm may flip one accept/reject decision (SURVEY.md 7.3 H7): rare, and
    # the result then still agrees to the integrator's own tolerance
    flipped = valid & ~same_steps
    assert flipped.mean() <= 2e-3
    if flipped.any():
        assert err[flipped].max() <= 1e-5


def test_explicit_state_non_equatorial(native, oracle):
    """integrate_geodesic with a caller-made state0 (off the equator, p_theta != 0) and
    non-default stop radii / lambda_max (status 0 = ran to lambda_max)."""
    gt = _gt()
    metric = _metric(1.0)
    s0 = [0.0, 30.0, 1.1, 0.3, -1.0, -0.93, 2.5, 6.0]
    for kw in (dict(), dict(lambda_max=20.0), dict(r_stop_inner=3.5, r_stop_outer=45.0)):
        sol, outcome = gt.integrate_geodesic(metric, s0, **kw)
        ref = oracle.rk45_trace_ray(1.0, None, None, state0=s0, **kw)
        assert sol.status == ref["status"] and sol.nfev == ref["nfev"] and sol.t.size == ref["n_points"], kw
        assert outcome == {1: "escaped", -1: "captured"}[ref["outcome"]]
        e = np.abs(sol.y[:, -1] - ref["y_final"]) / np.maximum(np.abs(ref["y_final"]), FLOOR)
        assert e.max() <= REL_TOL, (kw, e)
        assert np.abs(sol.y - ref["y"]).max() <= 1e-6
    sol, _ = gt.integrate_geodesic(metric, s0, lambda_max=20.0)
    assert sol.status == 0 and sol.t[-1] == 20.0 and sol.t_events[0].size == 0 and sol.t_events[1].size == 0


def test_device_tensor_batch_and_main(native, oracle, capsys):
    import torch
    gt = _gt()
    metric = _metric(1.0)
    alpha = torch.linspace(0.01, 1.5, 4097, dtype=torch.float64, device="cuda").reshape(17, 241)
    state, lam, outcome, nsteps = gt.trace_rays(metric, 100.0, alpha)
    assert state.is_cuda and state.shape == (17, 241, 8) and outcome.dtype == torch.int8
    s_o, l_o, oc_o, ns_o, _ = oracle.rk45_trace_batch(1.0, 100.0, alpha.cpu().numpy().ravel())
    assert np.array_equal(outcome.cpu().numpy().ravel(), oc_o)
    assert (nsteps.cpu().numpy().reshape(-1, 2) == ns_o).all(axis=1).mean() >= 0.998
    # empty batch
    st, _, oc, _ = gt.trace_rays(metric, 100.0, np.empty(0))
    assert st.shape == (0, 8) and oc.shape == (0,)
    # main.main() (main.py:12-33): prints the summary of the 8 deg ray at r_obs = 50 M
    from light_path_tracer_b200 import main as main_mod
    main_mod.main()
    out = capsys.readouterr().out
    assert "ESCAPED" in out and "b = 7.1" in out


def test_kerr_generic_path_golden(native, golden, oracle):
    """geodesic_tracer.trace_ray with a Kerr metric (scipy RK45 on Kerr.geodesic_equations,
    metrics.py:946-1029) against the reference fixture: outcome, accepted points and nfev exact,
    final state within 1e-9, trajectory within 1e-7."""
    from light_path_tracer_b200.metrics import Kerr
    gt = _gt()
    g = golden("kerr_rk45_rays.npz")
    off = g["traj_offsets"]
    worst = 0.0
    for i, row in enumerate(g["rows"]):
        M, a, r_obs, al, oc, npts, nfev, status, tf = row
        sol, outcome = gt.trace_ray(Kerr(float(M), float(a)), float(r_obs), float(al))
        assert outcome == {1: "escaped", -1: "captured"}[int(oc)], i
        assert sol.t.size == int(npts) and sol.nfev == int(nfev) and sol.status == int(status), i
        np.testing.assert_array_equal(sol.y[:, 0], g["state0"][i])
        e = np.abs(sol.y[:, -1] - g["y_final"][i]) / np.maximum(np.abs(g["y_final"][i]), FLOOR)
        assert e.max() <= REL_TOL, (i, e)
        assert abs(sol.t[-1] - tf) <= REL_TOL * max(1.0, tf)
        sl = slice(off[i], off[i + 1])
        assert np.abs(sol.t - g["traj_t"][sl]).max() <= 1e-7 * max(1.0, tf)
        assert (np.abs(sol.y[1] - g["traj_r"][sl]) / g["traj_r"][sl]).max() <= 1e-7
        worst = max(worst, e.max())
    print("20 Kerr reference rays through the generic integrator: worst final-state rel err %.2e" % worst)
    # several rays in one launch (plot_trajectories) and main.main(metric=Kerr)
    res = gt.trace_paths(Kerr(1.0, 0.9), 50.0, np.radians([3.0, 10.0]))
    assert [o for _, o in res] == ["captured", "escaped"]


def test_config3_4k_generic_vs_binet(native):
    """BASELINE config 3 at its full size (the generic 8-D RK45 integrator on every pixel of the
    3840x2160 alpha table), checked against the INDEPENDENT Binet RK4 tracer on the same rays —
    two different integrators of the same geodesics: escaped / captured must agree for every
    pixel outside a 1e-6 band around the critical angle, and the number of half orbits
    floor(|phi_f| / pi) wherever phi_f is not within 1e-4 of a multiple of pi (RK4 with
    h = 0.05 carries ~1e-6 of phase error)."""
    import torch
    from light_path_tracer_b200 import image_lens as il
    gt = _gt()
    metric = _metric(1.0)
    H, W = 2160, 3840
    vfov = np.radians(40.0)
    fov = (2 * np.arctan(np.tan(vfov / 2) * W / H), vfov)
    a32 = il.build_alpha_lookup((H, W), fov, device=True)
    status = torch.empty((H, W), dtype=torch.int8, device="cuda")
    fa, w = metric.trace_alpha_table(a32, 100.0, status=status)
    state, lam, outcome, nsteps = gt.trace_rays(metric, 100.0, a32.double())
    ac = float(metric.alpha_crit(100.0))
    clear = (a32.double() - ac).abs() > 1e-6 * ac
    # the centre pixel (alpha = 0, a radial ray): the generic path captures it
    # (geodesic_tracer.py:153-172 table, "0 deg captured"), the Binet fast path reports it
    # invalid (b = 0, metrics.py:57-58)
    valid = status != 0
    assert int((~valid).sum().item()) == 1 and int((outcome == 0).sum().item()) == 0
    assert int(outcome[~valid].item()) == -1
    assert torch.equal(outcome[clear & valid], status[clear & valid])
    assert int((~clear).sum().item()) < 64
    phi = state[..., 3].abs()
    frac = torch.remainder(phi / np.pi, 1.0)
    safe = clear & valid & (frac > 1e-4) & (frac < 1 - 1e-4)
    nh = torch.floor(phi / np.pi).to(torch.int64)
    assert torch.equal(nh[safe], w.view(torch.int16).to(torch.int64)[safe])
    assert int(safe.sum().item()) > 0.999 * H * W
    esc = outcome == 1
    r_f = state[..., 1][esc]
    assert float((r_f - 200.0).abs().max().item()) < 1e-6            # terminal event at 2 r_obs
    assert int(nsteps[..., 0].min().item()) >= 1 and int(nsteps[..., 1].max().item()) < 20000


def test_dense_output_sol_vs_scipy(native):
    """OdeResult.sol (the reference calls solve_ivp(dense_output=True), geodesic_tracer.py:57-67):
    the continuous solution rebuilt from the kernel's per-step (h, Q = K^T P) against scipy's own
    OdeSolution on the same right-hand side, at the breakpoints, mid-step points and the event —
    <= 1e-10 relative on the path (theta / p_theta hover at pi/2 and 1e-17: absolute floors)."""
    scipy_integrate = pytest.importorskip("scipy.integrate")
    gt = _gt()
    from light_path_tracer_b200.metrics import Schwarzschild, Kerr
    # (metric, r_obs, alpha, screen angle, theta_obs); the last two Kerr rays have angular momentum and
    # leave the equator
    cases = [(Schwarzschild(1.0), 50.0, np.radians(8.0), 0.0, np.pi / 2),
             (Schwarzschild(1.0), 50.0, np.radians(3.0), 0.0, np.pi / 2),
             (Schwarzschild(2.0), 120.0, np.radians(7.0), 0.0, np.pi / 2),
             (Schwarzschild(1.0), 30.0, np.radians(120.0), 0.0, np.pi / 2),
             (Kerr(1.0, 0.6), 40.0, np.radians(10.0), 0.0, np.pi / 2),
             (Kerr(1.0, 0.9), 40.0, np.radians(10.0), 1.0, 1.2),
             (Kerr(1.0, -0.998), 40.0, np.radians(8.0), 2.0, 0.3)]
    states = [(metric, metric.initial_conditions(r_obs, alpha, screen, theta_obs))
              for metric, r_obs, alpha, screen, theta_obs in cases]
    # an off-plane Schwarzschild state (Schwarzschild.initial_conditions only makes equatorial ones)
    states.append((Schwarzschild(1.0), [0.0, 30.0, 1.1, 0.3, -1.0, -0.93, 2.5, 6.0]))
    worst = 0.0
    for metric, state0 in states:
        sol, outcome = gt.integrate_geodesic(metric, state0)
        assert callable(sol.sol) and sol.sol.n_segments == sol.t.size - 1
        r_in, r_out = metric.capture_radius(), 2.0 * state0[1]

        def ev_in(t, y):
            return y[1] - r_in
        ev_in.terminal, ev_in.direction = True, -1

        def ev_out(t, y):
            return y[1] - r_out
        ev_out.terminal, ev_out.direction = True, 1
        ref = scipy_integrate.solve_ivp(metric.geodesic_equations, [0, 1000.0], state0, method='RK45', max_step=1.0,
                                        rtol=1e-8, atol=1e-10, events=[ev_in, ev_out], dense_output=True)
        assert ref.t.size == sol.t.size and ref.nfev == sol.nfev
        mids = 0.5 * (ref.t[:-1] + ref.t[1:])
        thirds = ref.t[:-1] + 0.31 * np.diff(ref.t)
        tt = np.concatenate([ref.t, mids, thirds])
        got, want = sol.sol(tt), ref.sol(tt)
        assert got.shape == want.shape == (8, tt.size)
        err = np.abs(got - want) / np.maximum(np.abs(want), FLOOR[:, None])
        assert err.max() <= 1e-10, (type(metric).__name__, state0, err.max(axis=1))
        worst = max(worst, float(err.max()))
        one = sol.sol(float(mids[3]))
        assert one.shape == (8,) and np.allclose(one, got[:, ref.t.size + 3], rtol=1e-14, atol=0.0)
        # the event point is sol(t_event), as solve_ivp builds it (ivp.py:676-697)
        e_evt = np.abs(sol.sol(sol.t[-1]) - sol.y[:, -1]) / np.maximum(np.abs(sol.y[:, -1]), FLOOR)
        assert e_evt.max() <= 1e-12
    print("sol(t) vs scipy OdeSolution: worst relative difference %.2e" % worst)


_EQ_SCRIPT = r"""
import sys, numpy as np, torch
sys.path.insert(0, %r)
from light_path_tracer_b200 import geodesic_tracer as gt
from light_path_tracer_b200.metrics import Schwarzschild
rng = np.random.default_rng(5)
out = {}
for tag, M, r_obs in (("a", 1.0, 100.0), ("b", 1.0, 15.0), ("c", 2.5, 40.0), ("d", 1.0, 2.9)):
    m = Schwarzschild(M)
    ac = float(m.alpha_crit(r_obs)) if r_obs > 3 * M else 1.0
    al = np.concatenate([rng.uniform(0, np.pi, 6000), ac * (1 + rng.normal(0, 1e-3, 3000)), [0.0, np.pi, 1e-12]])
    st, lam, oc, ns = gt.trace_rays(m, r_obs, al)
    out[tag + "_state"], out[tag + "_lam"], out[tag + "_oc"], out[tag + "_ns"] = st, lam, oc, ns
np.savez(sys.argv[1], **out)
"""


def test_equatorial_kernel_equals_six_component_kernel(native, tmp_path):
    """The batch path's equatorial kernel (four live components; theta = pi/2, p_theta = 0 carried
    as the constants they are to within rounding noise) against the six-component kernel that
    integrates the reference's full state: same outcome, same accepted points and nfev for every
    ray, (t, r, phi, p_r) and lambda within 1e-11, theta / p_theta within the noise they integrate
    to in the reference (<= 1e-14 / 1e-12 absolute)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = {}
    for eq in ("0", "1"):
        path = str(tmp_path / ("eq%s.npz" % eq))
        r = subprocess.run([sys.executable, "-c", _EQ_SCRIPT % root, path], env=dict(os.environ, LP_RK45_EQ=eq),
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        res[eq] = dict(np.load(path))
    worst = 0.0
    for tag in "abcd":
        s0, s1 = res["0"][tag + "_state"], res["1"][tag + "_state"]
        assert np.array_equal(res["0"][tag + "_oc"], res["1"][tag + "_oc"])
        assert np.array_equal(res["0"][tag + "_ns"], res["1"][tag + "_ns"]), "accept / reject sequences differ"
        ok = res["0"][tag + "_oc"] != 0
        assert np.array_equal(np.isnan(s0), np.isnan(s1))
        for c, floor in ((0, 1.0), (1, 1.0), (3, 1e-3), (5, 1e-3)):
            e = np.abs(s1[ok, c] - s0[ok, c]) / np.maximum(np.abs(s0[ok, c]), floor)
            worst = max(worst, float(e.max()))
            assert e.max() <= 1e-11, (tag, c, e.max())
        assert np.array_equal(s0[ok, 4], s1[ok, 4]) and np.array_equal(s0[ok, 7], s1[ok, 7])      # constants of the motion
        assert np.abs(s1[ok, 2] - s0[ok, 2]).max() <= 1e-14 and np.abs(s1[ok, 6] - s0[ok, 6]).max() <= 1e-12
        e = np.abs(res["1"][tag + "_lam"][ok] - res["0"][tag + "_lam"][ok]) / np.maximum(res["0"][tag + "_lam"][ok], 1.0)
        assert e.max() <= 1e-11
    print("equatorial vs six-component kernel: worst relative difference %.2e" % worst)
