"""Which kernel a request runs (lp_trace.cu, lp_repack.cu).  Every schedule and build of the Binet kernels
produces the same bytes, so the parity tests cannot see a routing change; the speed of a frame depends on it
(the mirror-image kernel takes a third of the time of the one-ray-per-pixel kernel on the 4K bench frame).
These tests record each request's launch with torch.profiler and check the kernel's template arguments and
CTA size.  Knobs are read once per process, so each knob setting runs in its own subprocess."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))

SIZES = {"1080p": (1080, 1920), "4K": (2160, 3840), "8K": (4320, 7680)}
PSI_OFF = (0.03, -0.02)          # no mirror symmetry
HYB, STRICT = 4, 0               # LP_TRACE_HYBRID, strict arithmetic
STAGED, REPACK, ROW_RUNS = 8, 2, 32


def run_case(case, trace_path):
    """Runs one request under the profiler: [(kernel with template arguments, threads per CTA)] of every
    lp_* kernel it launched."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from light_path_tracer_b200 import _device as dev, _lib, image_lens as il
    from light_path_tracer_b200.metrics import Schwarzschild
    m = Schwarzschild(1.0)
    kind, size, psi, flags, dtype, extra = case
    H, W = SIZES[size]
    vfov = np.radians(40.0)
    fov = (2 * np.arctan(np.tan(vfov / 2) * W / H), vfov)
    r_obs = extra.get("r_obs", 100.0)
    if kind == "frame":
        src = torch.zeros((H, W, 3), dtype=getattr(torch, dtype), device="cuda")
        call = lambda: il.render_frame(src, fov, r_obs, m, psi=psi, flags=flags, unit_u8=dtype == "uint8",
                                       rows=extra.get("rows"), bands=extra.get("bands"))
    elif kind == "trace_rays_batch":
        a = torch.linspace(0.0, 0.5, H * W, dtype=torch.float64, device="cuda")
        fa, w = torch.empty_like(a), torch.empty(H * W, dtype=torch.int64, device="cuda")
        call = lambda: m.trace_rays_batch(r_obs, a, fa, w, flags=flags)
    elif kind == "trace_alpha_table":
        a = il.build_alpha_lookup((H, W), fov, psi=psi, device=True)
        call = lambda: m.trace_alpha_table(a, r_obs, flags=flags)
    else:                        # trace_frame: the stand-alone tracer's own camera source
        fa = torch.empty((H, W), dtype=torch.float32, device="cuda")
        w = torch.empty((H, W), dtype=torch.uint16, device="cuda")
        cam = dev.camera_vector((H, W), fov, psi, il._psi_frame)
        call = lambda: _lib.ext().trace_frame(cam, 0, H, float(m.M), float(m.R_S), r_obs, dev.PHI_MAX, dev.H_MAX,
                                              None, fa, w, None, None, None, flags)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    prof.export_chrome_trace(trace_path)
    with open(trace_path) as f:
        events = json.load(f)["traceEvents"]
    out = []
    for e in events:
        k = re.search(r"\b(lp_\w+_kernel<[^>]*>)", e.get("name", ""))
        if e.get("cat") == "kernel" and k:
            out.append((k.group(1), int(e["args"]["block"][0])))
    return out


# (request, expected kernel, expected threads per CTA)
CASES = [
    # the bench frame: 2.08M traced rays (a quarter of the frame plus its mirror axes), under the 4M threshold
    (("frame", "4K", (0.0, 0.0), HYB | STAGED, "uint8", {}),
     "lp_render_mirror_kernel<true, true, unsigned char, 4, 2>", 256),
    (("frame", "8K", (0.0, 0.0), HYB | STAGED, "uint8", {}),
     "lp_render_mirror_kernel<true, true, unsigned char, 4, 4>", 256),
    (("frame", "4K", (0.0, 0.0), STRICT, "uint8", {}),
     "lp_render_mirror_kernel<false, true, unsigned char, 4, 2>", 256),
    (("frame", "4K", (0.0, 0.0), HYB, "float32", {}),
     "lp_render_mirror_kernel<true, true, float, 4, 2>", 256),
    (("frame", "4K", PSI_OFF, HYB | STAGED, "uint8", {}),
     "lp_render_kernel<true, true, unsigned char, 4, 4>", 256),
    (("frame", "1080p", PSI_OFF, HYB, "uint8", {}),
     "lp_render_kernel<true, true, unsigned char, 4, 2>", 256),
    (("frame", "1080p", PSI_OFF, STRICT, "uint8", {}),
     "lp_render_kernel<false, true, unsigned char, 4, 2>", 256),
    (("frame", "1080p", PSI_OFF, HYB, "float32", {}),
     "lp_render_kernel<true, true, float, 4, 2>", 256),
    (("frame", "1080p", PSI_OFF, HYB, "float64", {}),
     "lp_render_kernel<true, true, double, 4, 2>", 256),
    (("frame", "1080p", (0.0, 0.0), HYB | REPACK, "uint8", {}),
     "lp_render_repack_kernel<true, unsigned char, 16>", 64),
    (("frame", "1080p", (0.0, 0.0), STRICT | REPACK, "float32", {}),
     "lp_render_repack_kernel<false, float, 16>", 64),
    # mirror symmetry, but a tile the mirror kernel does not take
    (("frame", "1080p", (0.0, 0.0), HYB, "uint8", {"rows": (0, 540), "bands": (8, 16)}),
     "lp_render_kernel<true, true, unsigned char, 4, 2>", 256),
    (("frame", "1080p", (0.0, 0.0), HYB | ROW_RUNS, "uint8", {}),
     "lp_render_kernel<true, true, unsigned char, 4, 2>", 256),
    # r_obs = 2.01 M lies inside the capture radius 1.01 R_S: the fast path's precondition fails
    (("frame", "1080p", PSI_OFF, HYB, "uint8", {"r_obs": 2.01}),
     "lp_render_kernel<true, false, unsigned char, 4, 2>", 256),
    # the stand-alone tracer: SRC 0 / 1 / 2 = float64 angles, float32 angles, the camera
    (("trace_rays_batch", "1080p", (0.0, 0.0), STRICT, None, {}), "lp_trace_kernel<false, true, 0, true>", 256),
    (("trace_alpha_table", "1080p", (0.0, 0.0), HYB, None, {}), "lp_trace_kernel<true, true, 1, false>", 256),
    (("trace_frame", "1080p", (0.0, 0.0), HYB, None, {}), "lp_trace_kernel<true, true, 2, false>", 256),
]


def _case_id(c):
    kind, size, psi, flags, dtype, extra = c[0]
    return "-".join([kind, size, "psi%g,%g" % psi, "f%d" % flags] + ([dtype] if dtype else []) +
                    ["%s=%s" % kv for kv in sorted(extra.items())]).replace(" ", "")


@pytest.mark.parametrize("case,kernel,block", CASES, ids=[_case_id(c) for c in CASES])
def test_frame_request_runs_kernel(native, tmp_path, case, kernel, block):
    assert run_case(case, str(tmp_path / "trace.json")) == [(kernel, block)]


CHILD = r'''
import json, sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(here)r)
import test_gpu_dispatch as t
print("RESULT " + json.dumps(t.run_case(t.CASES[%(index)d][0], %(trace)r)))
'''


@pytest.mark.parametrize("knobs,index,kernel,block", [
    ({"LP_RENDER_TRIP": "2"}, 1, "lp_render_mirror_kernel<true, true, unsigned char, 4, 2>", 256),
    ({"LP_RENDER_TRIP": "3"}, 1, "lp_render_mirror_kernel<true, true, unsigned char, 4, 4>", 256),
    ({"LP_TRACE_BLOCK": "128"}, 0, "lp_render_mirror_kernel<true, true, unsigned char, 4, 2>", 128),
    ({"LP_TRACE_BLOCK": "128"}, 5, "lp_render_kernel<true, true, unsigned char, 4, 2>", 128),
], ids=["trip2-8K", "trip3-ignored-8K", "block128-mirror", "block128-render"])
def test_knob_routing(native, tmp_path, knobs, index, kernel, block):
    env = dict(os.environ)
    for k in ("LP_RENDER_TRIP", "LP_RENDER_TILE_H", "LP_TRACE_BLOCK"):
        env.pop(k, None)
    env.update(knobs)
    root = os.path.dirname(HERE)
    code = CHILD % {"root": root, "here": HERE, "index": index, "trace": str(tmp_path / "trace.json")}
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    assert [tuple(x) for x in json.loads(line[len("RESULT "):])] == [(kernel, block)]
