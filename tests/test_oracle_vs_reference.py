"""Live pin of the oracle against the UNMODIFIED reference, where the reference tree exists
(/root/reference in the build container; skipped on the GPU box).  The committed fixtures in
tests/golden/ are a frozen subset of exactly this comparison."""
import numpy as np
import pytest

import ref_harness
from conftest import bits_equal

pytestmark = pytest.mark.skipif(not ref_harness.available(), reason="reference tree not present")


@pytest.fixture(scope="module")
def ref():
    return ref_harness.load()


def test_binet_batch_live(oracle, ref):
    """Schwarzschild.trace_rays_batch (numba) vs the C restatement, 4 x 250k rays, bit for bit."""
    rng = np.random.default_rng(77)
    for M, r_obs in [(1.0, 100.0), (1.0, 15.0), (2.5, 40.0), (1.0, 1000.0)]:
        m = ref.metrics.Schwarzschild(M)
        ac = float(m.alpha_crit(r_obs))
        alpha = np.concatenate([rng.uniform(0, np.pi, 150000), ac * (1 + rng.normal(0, 1e-3, 60000)),
                                ac * (1 + rng.normal(0, 1e-7, 40000))])
        fa = np.empty(alpha.size)
        w = np.empty(alpha.size, dtype=np.int64)
        m.trace_rays_batch(r_obs, alpha, fa, w)
        fa_o, w_o, _, _ = oracle.trace_rays_batch(M, r_obs, alpha)
        assert bits_equal(fa, fa_o) and np.array_equal(w, w_o), (M, r_obs)


def test_frame_pipeline_live(oracle, ref):
    """build_alpha_lookup -> precompute_final_alpha_lookup -> render_lensed_image at 135x240."""
    IL = ref.image_lens
    H, W = 135, 240
    vfov = np.radians(40.0)
    fov = (2 * np.arctan(np.tan(vfov / 2) * W / H), vfov)
    for psi in ((0.0, 0.0), (0.07, -0.11)):
        m = ref.metrics.Schwarzschild(1.0)
        a = IL.build_alpha_lookup((H, W), fov, psi=psi)
        assert np.array_equal(a, oracle.build_alpha_lookup((H, W), fov, psi=psi))
        fa, w, n, _ = IL.precompute_final_alpha_lookup(a, m.alpha_crit(100.0), 100.0, m)
        fa_o, w_o, _, _ = oracle.precompute_final_alpha_lookup(a, 1.0, 100.0)
        assert bits_equal(fa, fa_o) and np.array_equal(w, w_o)
        src = oracle.checkerboard(H, W)
        assert np.array_equal(IL.render_lensed_image(src, a, fa, w, 0.0, fov, False, psi=psi),
                              oracle.render_lensed_image(src, fa, w, fov, False, psi))


def test_kerr_batch_live(oracle, ref):
    rng = np.random.default_rng(5)
    M, a, r_obs, th_obs = 1.0, 0.7, 60.0, 1.3
    m = ref.metrics.Kerr(M, a)
    ac = float(m.alpha_crit(r_obs, th_obs))
    alpha = np.concatenate([rng.uniform(0, 3 * ac, 3000), rng.uniform(0, np.pi, 500)])
    theta = rng.uniform(-np.pi, np.pi, alpha.size)
    refine = rng.random(alpha.size) < 0.3
    fa = np.empty(alpha.size)
    w = np.empty(alpha.size, dtype=np.int64)
    m.trace_rays_batch(r_obs, alpha, theta, th_obs, refine, fa, w)
    fa_o, w_o, _, _ = oracle.kerr_trace_rays_batch(M, a, r_obs, alpha, theta, th_obs, refine)
    assert bits_equal(fa, fa_o) and np.array_equal(w, w_o)


def test_rk45_live(oracle, ref):
    """geodesic_tracer.trace_ray (scipy) vs the restated stepper: same accepted points / nfev."""
    m = ref.metrics.Schwarzschild(1.0)
    for deg in (1.0, 5.7, 5.9, 9.0, 33.0, 140.0):
        sol, outcome = ref.geodesic_tracer.trace_ray(m, 50.0, float(np.radians(deg)))
        r = oracle.rk45_trace_ray(1.0, 50.0, float(np.radians(deg)))
        assert (sol.t.size, sol.nfev, sol.status) == (r["n_points"], r["nfev"], r["status"]), deg
        assert outcome == {1: "escaped", -1: "captured"}[r["outcome"]]
        assert np.abs(sol.y[:, -1] - r["y_final"]).max() <= 1e-10 * max(1.0, np.abs(sol.y[:, -1]).max())


def test_rk45_kerr_live(oracle, ref):
    """geodesic_tracer.integrate_geodesic(Kerr) (scipy) vs the restated Kerr stepper on rays with angular
    momentum, off the equator and at both spins: same accepted points / nfev / status, final state to 1e-11."""
    rng = np.random.default_rng(43)
    for M, a, r_obs, th_obs in ((1.0, 0.9, 30.0, 1.1), (1.0, -0.998, 12.0, 0.3), (2.5, 2.0, 100.0, np.pi / 2),
                                (1.0, 1.0, 50.0, np.pi - 0.2)):
        m = ref.metrics.Kerr(M, a)
        ac = float(m.alpha_crit(r_obs, th_obs))
        for al, sc in zip(ac * rng.uniform(0.1, 1.9, 4), rng.uniform(-np.pi, np.pi, 4)):
            s0 = m.initial_conditions(r_obs, float(al), float(sc), th_obs)
            assert s0[7] != 0.0
            sol, outcome = ref.geodesic_tracer.integrate_geodesic(m, s0)
            r = oracle.rk45_integrate_kerr(M, a, s0)
            assert (sol.t.size, sol.nfev, sol.status) == (r["n_points"], r["nfev"], r["status"]), (a, s0)
            assert outcome == {1: "escaped", -1: "captured"}[r["outcome"]]
            e = np.abs(sol.y[:, -1] - r["y_final"]) / np.maximum(np.abs(sol.y[:, -1]), 1.0)
            assert e.max() <= 1e-11, (a, s0, e)
