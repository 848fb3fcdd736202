"""GPU parity of the opt-in KERNEL VARIANTS that are selected by environment knobs (the library reads a
knob once per process, so every variant renders in its own subprocess): 2-step loop trips of the frame
kernel (LP_RENDER_TRIP, lp_trace.cu), warp-tile shapes (LP_RENDER_TILE_H), CTA sizes (LP_TRACE_BLOCK)
and the TMA-staged remap (LP_REMAP_TMA, lp_remap_tma.cu).  None of them may change a single output
byte: they only move work between warps or stage the same source texels differently (reference:
metrics.py:49-145, image_lens.py:133-178, :296-397)."""
import hashlib
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r'''
import hashlib, json, sys
import numpy as np, torch
sys.path.insert(0, %(root)r)
from light_path_tracer_b200 import image_lens as il, _device as dev
from light_path_tracer_b200.metrics import Schwarzschild
m = Schwarzschild(1.0)
out = {}
def digest(*ts):
    h = hashlib.sha256()
    for t in ts:
        h.update(t.detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()
g = torch.Generator(device="cuda").manual_seed(7)
# frames larger than one wave of CTAs, a ragged one, a close observer (divergent warps), a rotated
# camera, uint8 and float32, strict and hybrid
for (H, W, r_obs, vf, psi) in [(1080, 1920, 100.0, 40.0, (0.0, 0.0)), (1000, 1500, 15.0, 40.0, (0.04, -0.03)),
                               (1031, 1217, 30.0, 25.0, (0.0, 0.1)), (96, 128, 100.0, 12.0, (0.0, 0.0))]:
    vfov = np.radians(vf); fov = (2 * np.arctan(np.tan(vfov / 2) * W / H), vfov)
    src = torch.rand(H, W, 3, device="cuda", generator=g)
    src8 = (src * 255).to(torch.uint8)
    for flags in (0, 4, 4 | 8):
        f32, fa, w = il.render_frame(src, fov, r_obs, m, psi=psi, flags=flags, return_lookups=True)
        u8 = il.render_frame(src8, fov, r_obs, m, psi=psi, flags=flags, unit_u8=True)
        out["frame %%dx%%d r%%g f%%d" %% (W, H, r_obs, flags)] = digest(f32, fa.view(torch.int32), w.view(torch.int16), u8)
    stats = dev.new_stats()
    il.render_frame(src8, fov, r_obs, m, psi=psi, flags=4 | 8, unit_u8=True, stats=stats)
    s = dev.read_stats(stats)
    out["stats %%dx%%d r%%g" %% (W, H, r_obs)] = [int(s[k]) for k in ("n_rays", "n_escaped", "n_captured", "n_invalid",
                                                                   "n_winding", "sum_steps", "max_steps", "max_winding")]
    a = il.build_alpha_lookup((H, W), fov, psi=psi, device=True)
    fa, w = m.trace_alpha_table(a, r_obs)
    for loop_around in (False, True):
        for sampling in (il.SAMPLE_NEAREST, il.SAMPLE_BILINEAR):
            r32 = il.render_lensed_image(src, a, fa, w, 0.0, fov, render_loop_around=loop_around, psi=psi, sampling=sampling)
            r8 = il.render_lensed_image(src8, a, fa, w, 0.0, fov, render_loop_around=loop_around, psi=psi, sampling=sampling)
            out["remap %%dx%%d r%%g loop%%d s%%s" %% (W, H, r_obs, loop_around, sampling)] = digest(r32, r8)
print("RESULT " + json.dumps(out, sort_keys=True))
'''


def _run(env_extra):
    env = dict(os.environ)
    for k in ("LP_RENDER_TRIP", "LP_RENDER_TILE_H", "LP_TRACE_BLOCK", "LP_REMAP_TMA"):
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
    {"LP_RENDER_TRIP": "2"},
    {"LP_RENDER_TILE_H": "1"},
    {"LP_RENDER_TILE_H": "2", "LP_TRACE_BLOCK": "128"},
    {"LP_TRACE_BLOCK": "32"},
    {"LP_REMAP_TMA": "1"},
], ids=lambda k: ",".join("%s=%s" % kv for kv in sorted(k.items())))
def test_knob_variants_are_bit_identical(native, default_outputs, knobs):
    got = _run(knobs)
    assert set(got) == set(default_outputs)
    differing = [k for k in got if got[k] != default_outputs[k]]
    assert not differing, "outputs differ under %s: %s" % (knobs, differing)
