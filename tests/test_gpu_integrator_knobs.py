"""GPU parity of the integrator builds selected by environment knobs (the library reads a knob once per
process, so every setting runs in its own subprocess): resident CTAs per SM of the six-component and
equatorial RK45 kernels (LP_RK45_MINB, LP_RK45_EQ_MINB), the RK45 refill threshold (LP_RK45_REFILL) and the
Kerr schedule knobs (LP_KERR_MINB, LP_KERR_REFILL, LP_KERR_QUEUE=0 = the parked schedule).  They change
register limits or which lane runs a ray, never the operations of a ray, so no output byte may change.
LP_RK45_POW and LP_RK45_EQ=0 do change results within the parity bar and are not covered here; the
LP_RK45_EQ pair is held together by test_gpu_rk45.py."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KNOBS = ("LP_RK45_MINB", "LP_RK45_EQ_MINB", "LP_RK45_REFILL", "LP_RK45_POW", "LP_RK45_EQ",
         "LP_KERR_MINB", "LP_KERR_REFILL", "LP_KERR_QUEUE")

CHILD = r'''
import hashlib, json, sys
import numpy as np, torch
sys.path.insert(0, %(root)r)
from light_path_tracer_b200 import geodesic_tracer as gt, image_lens as il, _device as dev
from light_path_tracer_b200.metrics import Schwarzschild, Kerr
out = {}
def digest(*arrays):
    h = hashlib.sha256()
    for x in arrays:
        x = x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
        h.update(np.ascontiguousarray(x).tobytes())
    return h.hexdigest()
m = Schwarzschild(1.0)
for r_obs in (100.0, 15.0):
    # uniform, a cluster at the critical angle and the odd inputs of test_batch_vs_oracle
    rng = np.random.default_rng(int(r_obs))
    ac = float(np.arcsin(3 * np.sqrt(3) / r_obs * np.sqrt(1 - 2 / r_obs)))
    alpha = np.concatenate([rng.uniform(0, np.pi, 2000), ac * (1 + rng.normal(0, 1e-3, 1000)),
                            [0.0, np.pi / 2, np.pi, 1e-9, -0.2, 3.5, np.nan]])
    out["trace_rays r%%g" %% r_obs] = digest(*gt.trace_rays(m, r_obs, alpha, return_status=True))
    # the six-component kernel: the batch entry runs the equatorial one
    paths = gt.trace_paths(m, r_obs, alpha[::10])
    out["trace_paths r%%g" %% r_obs] = [outcome if sol is None else digest(sol.t, sol.y, [sol.nfev, sol.status]) + outcome
                                        for sol, outcome in paths]
sol, outcome = gt.integrate_geodesic(m, [0.0, 30.0, 1.1, 0.3, -1.0, -0.93, 2.5, 6.0])
out["integrate_geodesic"] = digest(sol.t, sol.y, [sol.nfev, sol.status]) + outcome
H, W = 135, 243
vfov = np.radians(40.0)
fov = (2 * np.arctan(np.tan(vfov / 2) * W / H), vfov)
a32 = il.build_alpha_lookup((H, W), fov, device=True)
cam = dev.camera_vector((H, W), fov, (0.0, 0.0), il._psi_frame)
steps = torch.empty((H, W, 2), dtype=torch.int32, device="cuda")
fa, w = Kerr(1.0, 0.9).trace_alpha_table_2d(a32, cam, 100.0, 1.1, steps=steps)
out["kerr_2d"] = digest(fa, w, steps)
print("RESULT " + json.dumps(out, sort_keys=True))
'''


def _run(env_extra):
    env = dict(os.environ)
    for k in KNOBS:
        env.pop(k, None)
    env.update(env_extra)
    r = subprocess.run([sys.executable, "-c", CHILD % {"root": ROOT}], env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    return json.loads(line[len("RESULT "):])


@pytest.fixture(scope="module")
def default_outputs(native):
    return _run({})


@pytest.mark.parametrize("knobs", [
    {"LP_RK45_MINB": "2"},
    {"LP_RK45_MINB": "4"},
    {"LP_RK45_EQ_MINB": "3"},
    {"LP_RK45_EQ_MINB": "5"},
    {"LP_RK45_EQ_MINB": "6"},
    {"LP_RK45_REFILL": "1"},
    {"LP_RK45_REFILL": "32"},
    {"LP_KERR_MINB": "3"},
    {"LP_KERR_MINB": "5"},
    {"LP_KERR_QUEUE": "0", "LP_KERR_MINB": "2"},
    {"LP_KERR_QUEUE": "0", "LP_KERR_MINB": "6"},
    {"LP_KERR_QUEUE": "0", "LP_KERR_REFILL": "1"},
], ids=lambda k: ",".join("%s=%s" % kv for kv in sorted(k.items())))
def test_integrator_knob_variants_are_bit_identical(native, default_outputs, knobs):
    got = _run(knobs)
    assert set(got) == set(default_outputs)
    differing = [k for k in got if got[k] != default_outputs[k]]
    assert not differing, "outputs differ under %s: %s" % (knobs, differing)
