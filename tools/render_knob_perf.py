"""Frame-kernel timing under one tuning knob (the library reads knobs once per process, so every value
runs in its own subprocess).

    python tools/render_knob_perf.py LP_RENDER_TRIP 2 4
"""
import os
import subprocess
import sys

CHILD = r'''
import sys, os
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(sys.argv[0]))) if False else os.getcwd())
from light_path_tracer_b200 import image_lens as il
from light_path_tracer_b200.metrics import Schwarzschild
flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
def timeit(fn, n=20, warm=3):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return min(ts), float(np.median(ts))
m = Schwarzschild(1.0)
out = []
for (H, W, r_obs, vf) in [(2160, 3840, 100.0, 40.0), (1080, 1920, 100.0, 40.0), (2160, 3840, 15.0, 40.0), (1024, 1024, 100.0, 12.0), (4320, 7680, 100.0, 40.0)]:
    vfov = np.radians(vf); fov = (2*np.arctan(np.tan(vfov/2)*W/H), vfov)
    src = torch.rand(H, W, 3, device='cuda')
    src8 = (src * 255).to(torch.uint8)
    t8 = timeit(lambda: il.render_frame(src8, fov, r_obs, m, flags=4 | 8, unit_u8=True))
    t32 = timeit(lambda: il.render_frame(src, fov, r_obs, m, flags=4 | 8))
    ts = timeit(lambda: il.render_frame(src, fov, r_obs, m, flags=0 | 8))
    out.append("%dx%d r%g v%g: u8 %.4f/%.4f  f32 %.4f/%.4f  strict %.4f/%.4f" % (W, H, r_obs, vf, *t8, *t32, *ts))
print(" | ".join(out))
'''

if __name__ == "__main__":
    knob, values = sys.argv[1], sys.argv[2:]
    for v in values:
        env = dict(os.environ)
        if v != "default":
            env[knob] = v
        r = subprocess.run([sys.executable, "-c", CHILD], env=env, capture_output=True, text=True)
        print("%s=%s  %s" % (knob, v, (r.stdout.strip().splitlines() or [r.stderr[-400:]])[-1]), flush=True)
