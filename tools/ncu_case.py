"""One small, fixed workload per case for ncu captures (gpurun: plain run first, then under ncu).

    python tools/ncu_case.py render_hybrid | render_u8 | render_strict | trace_hybrid | remap | rk45 | rk45_full | kerr | shadow
(rk45_full sets LP_RK45_EQ=0 for its process)
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from light_path_tracer_b200 import image_lens as il, geodesic_tracer as gt, black_hole_shadow as bs  # noqa: E402
from light_path_tracer_b200.metrics import Schwarzschild  # noqa: E402

case = sys.argv[1]
if case == "rk45_full":
    os.environ["LP_RK45_EQ"] = "0"
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
H, W = 2160, 3840
vfov = np.radians(40.0)
fov = (2 * np.arctan(np.tan(vfov / 2) * W / H), vfov)
m = Schwarzschild(1.0)
src = torch.rand(H, W, 3, device="cuda")
for _ in range(reps):
    if case == "render_hybrid":
        il.render_frame(src, fov, 100.0, m, flags=4)
    elif case == "render_u8":
        il.render_frame((src * 255).to(torch.uint8), fov, 100.0, m, flags=4 | 8, unit_u8=True)
    elif case == "render_strict":
        il.render_frame(src, fov, 100.0, m, flags=0)
    elif case == "trace_hybrid":
        a = il.build_alpha_lookup((H, W), fov, device=True)
        m.trace_alpha_table(a, 100.0, flags=4)
    elif case == "remap":
        a = il.build_alpha_lookup((H, W), fov, device=True)
        fa, w = m.trace_alpha_table(a, 100.0)
        il.render_lensed_image(src, a, fa, w, 0.0, fov)
    elif case in ("rk45", "rk45_full"):
        h, w_ = 540, 960
        f2 = (2 * np.arctan(np.tan(vfov / 2) * w_ / h), vfov)
        a = il.build_alpha_lookup((h, w_), f2, device=True).double()
        gt.trace_rays(m, 100.0, a)
    elif case == "kerr":
        from light_path_tracer_b200.metrics import Kerr
        from light_path_tracer_b200 import _device as dev
        h, w_ = 540, 960
        f2 = (2 * np.arctan(np.tan(vfov / 2) * w_ / h), vfov)
        a = il.build_alpha_lookup((h, w_), f2, device=True)
        cam = dev.camera_vector((h, w_), f2, (0.0, 0.0), il._psi_frame)
        Kerr(1.0, 0.9).trace_alpha_table_2d(a, cam, 100.0, np.pi / 2)
    elif case == "shadow":
        bs.shadow_image(m, 4096, 4096, np.radians(40), 50.0, device=True)
torch.cuda.synchronize()
print("ok", case)
