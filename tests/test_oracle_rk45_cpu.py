"""CPU anchors of the generic RK45 integrator's off-plane checks (no GPU).

test_gpu_rk45_rhs.py holds the device right-hand sides to metrics.py's expressions, and
test_gpu_rk45_offplane.py holds whole Kerr and off-plane integrations to the oracle's RK45
(oracle/lp_oracle_rk45.c).  Two links of that chain are checked here:
- metrics.py's right-hand sides are Hamilton's equations: x' = dH/dp and p' = -dH/dx for
  H = 1/2 g^{mu nu} p_mu p_nu, differentiated with mpmath at 200 bits, on states with p_phi != 0 and off
  the equator (where the frame-dragging, p_phi^2 and 1/sin^2(theta) terms all count);
- the oracle's Kerr RK45 is scipy's: solve_ivp(method='RK45') on Kerr.geodesic_equations with the
  reference's events, tolerances and max_step takes the same accepted points and right-hand-side
  evaluations on rays with angular momentum, and ends at the same state.
"""
import numpy as np
import pytest

PREC = 200


def _hamiltonian(M, a, y, kerr):
    """H = 1/2 g^{mu nu} p_mu p_nu (mpmath), y = (r, theta, p_t, p_r, p_theta, p_phi)"""
    import mpmath as mp
    r, th, p_t, p_r, p_th, p_phi = y
    s, c = mp.sin(th), mp.cos(th)
    if not kerr:
        f = 1 - 2 * M / r
        return (-p_t ** 2 / f + f * p_r ** 2 + p_th ** 2 / r ** 2 + p_phi ** 2 / (r ** 2 * s ** 2)) / 2
    Sigma = r ** 2 + a ** 2 * c ** 2
    Delta = r ** 2 - 2 * M * r + a ** 2
    A = (r ** 2 + a ** 2) ** 2 - a ** 2 * Delta * s ** 2
    g_tt, g_tphi = -A / (Sigma * Delta), -2 * M * a * r / (Sigma * Delta)
    g_rr, g_thth = Delta / Sigma, 1 / Sigma
    g_phiphi = (Delta - a ** 2 * s ** 2) / (Sigma * Delta * s ** 2)
    return (g_tt * p_t ** 2 + 2 * g_tphi * p_t * p_phi + g_rr * p_r ** 2 + g_thth * p_th ** 2
            + g_phiphi * p_phi ** 2) / 2


def _hamilton_rhs(M, a, state, kerr):
    """(dt, dr, dtheta, dphi, dp_r, dp_theta) = (dH/dp_t, dH/dp_r, dH/dp_theta, dH/dp_phi, -dH/dr, -dH/dtheta)"""
    import mpmath as mp
    with mp.workprec(PREC):
        y = [mp.mpf(float(state[k])) for k in (1, 2, 4, 5, 6, 7)]
        M, a = mp.mpf(M), mp.mpf(a)

        def d(k):
            def h(x):
                z = list(y)
                z[k] = x
                return _hamiltonian(M, a, z, kerr)
            return mp.diff(h, y[k])
        return [d(2), d(3), d(4), d(5), -d(0), -d(1)]


def _random_states(rng, n, M, r_lo):
    return [[0.0, float(rng.uniform(r_lo, 60 * M)), float(rng.uniform(0.15, np.pi - 0.15)), 0.0,
             float(-rng.uniform(0.5, 2.0)), float(rng.normal()), float(rng.normal() * 3),
             float(rng.choice([-1, 1]) * rng.uniform(0.5, 12.0))] for _ in range(n)]


@pytest.mark.parametrize("kerr", [False, True], ids=["schwarzschild", "kerr"])
def test_metrics_rhs_is_hamiltons_equations(kerr):
    """metrics.py's geodesic_equations = Hamilton's equations of H = 1/2 g^{mu nu} p p to 1e-12 (measured
    2e-14), relative to max(|exact|, 1e-3), on 60 random states with p_phi != 0 off the equator"""
    from light_path_tracer_b200.metrics import Schwarzschild, Kerr
    rng = np.random.default_rng(31 if kerr else 32)
    worst = 0.0
    for k in range(60):
        M = float(rng.choice([1.0, 2.5]))
        a = float(rng.uniform(-1, 1) * M) if kerr else 0.0
        m = Kerr(M, a) if kerr else Schwarzschild(M)
        r_lo = (float(m.r_plus) if kerr else 2 * M) * 1.05
        for st in _random_states(rng, 1, M, r_lo):
            got = np.array(m.geodesic_equations(0.0, st), dtype=np.float64)[[0, 1, 2, 3, 5, 6]]
            exact = np.array([float(v) for v in _hamilton_rhs(M, a, st, kerr)])
            assert got[5] != 0.0 or not kerr
            err = np.abs(got - exact) / np.maximum(np.abs(exact), 1e-3)
            assert err.max() <= 1e-12, (M, a, st, err)
            worst = max(worst, float(err.max()))
    print("\n%s geodesic_equations vs Hamilton's equations: worst %.2e" % ("Kerr" if kerr else "Schwarzschild", worst))


# (M, a / M, r_obs / M, theta_obs, alpha / alpha_c, screen angle)
KERR_RAYS = [(1.0, 0.9, 30.0, 1.1), (1.0, -0.998, 12.0, 0.3), (2.5, 0.3, 100.0, np.pi / 2), (1.0, 1.0, 30.0, 0.3),
             (1.0, -0.9, 50.0, np.pi - 0.2), (2.5, 0.998, 20.0, 0.05)]


def _kerr_ray_states(n_per, seed):
    from light_path_tracer_b200.metrics import Kerr
    rng = np.random.default_rng(seed)
    out = []
    for M, q, r_obs_M, th_obs in KERR_RAYS:
        m = Kerr(M, q * M)
        ac = float(m.alpha_crit(r_obs_M * M, th_obs))
        for al, sc in zip(ac * rng.uniform(0.1, 1.9, n_per), rng.uniform(-np.pi, np.pi, n_per)):
            out.append((M, q * M, m.initial_conditions(r_obs_M * M, float(al), float(sc), th_obs)))
    return out


def _scipy_kerr(M, a, s0):
    scipy_integrate = pytest.importorskip("scipy.integrate")
    from light_path_tracer_b200.metrics import Kerr
    m = Kerr(M, a)
    r_in, r_out = m.capture_radius(), 2.0 * s0[1]

    def ev_in(t, y):
        return y[1] - r_in
    ev_in.terminal, ev_in.direction = True, -1

    def ev_out(t, y):
        return y[1] - r_out
    ev_out.terminal, ev_out.direction = True, 1
    return scipy_integrate.solve_ivp(m.geodesic_equations, [0, 1000.0], s0, method='RK45', max_step=1.0, rtol=1e-8,
                                     atol=1e-10, events=[ev_in, ev_out])


def test_oracle_kerr_rk45_vs_scipy(oracle):
    """oracle.rk45_integrate_kerr against scipy's solve_ivp on Kerr.geodesic_equations, 24 rays with
    angular momentum from six configurations: accepted points, nfev and status exact, final state within
    1e-11 relative (absolute below 1)"""
    worst = 0.0
    rays = _kerr_ray_states(4, 41)
    for M, a, s0 in rays:
        assert s0[7] != 0.0
        ref = _scipy_kerr(M, a, s0)
        o = oracle.rk45_integrate_kerr(M, a, s0)
        assert (o["n_points"], o["nfev"], o["status"]) == (ref.t.size, ref.nfev, ref.status), (M, a, s0)
        e = np.abs(o["y_final"] - ref.y[:, -1]) / np.maximum(np.abs(ref.y[:, -1]), 1.0)
        assert e.max() <= 1e-11, (M, a, s0, e)
        assert abs(o["t_final"] - ref.t[-1]) <= 1e-11 * max(1.0, ref.t[-1])
        worst = max(worst, float(e.max()))
    print("\noracle Kerr RK45 vs scipy, %d rays with L != 0: worst final-state difference %.2e" % (len(rays), worst))
