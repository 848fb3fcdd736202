"""Stand-alone remap (render_lensed_image) timings at 4K (r_obs 100 and 15) and 1080p, float32 and
uint8 RGB, nearest and bilinear.  CUDA events, L2 flushed between launches."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from light_path_tracer_b200 import image_lens as il  # noqa: E402
from light_path_tracer_b200.metrics import Schwarzschild  # noqa: E402
from light_path_tracer_b200.synthetic import checkerboard  # noqa: E402

metric = Schwarzschild(1.0)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
for H, W, r_obs in ((2160, 3840, 100.0), (2160, 3840, 15.0), (1080, 1920, 100.0)):
    vfov = np.radians(40.0)
    fov = (2 * np.arctan(np.tan(vfov / 2) * W / H), vfov)
    a32 = il.build_alpha_lookup((H, W), fov, device=True)
    fa32, w16 = metric.trace_alpha_table(a32, r_obs)
    for dt in (np.float32, np.uint8):
        src = torch.from_numpy(checkerboard(H, W, dt)).cuda()
        for sampling in (0, 1):
            fn = lambda: il.render_lensed_image(src, a32, fa32, w16, 0.0, fov, sampling=sampling)  # noqa: E731
            fn(); fn()
            ts = []
            for _ in range(10):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); out = fn(); b.record(); torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
            bpp = (4 + 2 + 2 * 3 * src.element_size())
            print("%dx%d r_obs=%g %-7s %-8s  best %.4f ms  median %.4f ms  %.0f GB/s (algorithmic %d B/px)  checksum %d"
                  % (W, H, r_obs, np.dtype(dt).name, "bilinear" if sampling else "nearest", min(ts), float(np.median(ts)),
                     H * W * bpp / min(ts) / 1e6, bpp, int(out.view(torch.uint8).to(torch.int64).sum().item())), flush=True)
