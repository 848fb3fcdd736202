"""GPU parity of the mirror-image frame kernel for cameras whose basis does not carry a mirror over to the
remap's source direction.  The kernel forms a ray's source direction once and negates qx / qy for its mirror
images only when the basis has the exact zeros that make this exact (lp_render_mirror_kernel, lp_trace.cu);
any other basis around a view direction with d0 == d1 == 0 keeps both mirrors (the viewing angle depends on
d alone) but forms each image's direction from its own camera coordinates.  The frames must be the ones of
the lane re-packing schedule (LP_TRACE_REPACK), which traces and remaps one pixel per lane, BIT FOR BIT."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROLL = 0.3


def _rolled(psi):
    """Basis rolled about d = (0, 0, 1): both mirrors, no shared direction."""
    c, s = np.cos(ROLL), np.sin(ROLL)
    return (np.array([0.0, 0.0, 1.0]), np.array([c, s, 0.0]), np.array([-s, c, 0.0]), True)


def _tilted_ey(psi):
    """e_x = (1, 0, 0), e_y tilted towards d: both mirrors, the direction shared in x only."""
    c, s = np.cos(ROLL), np.sin(ROLL)
    return (np.array([0.0, 0.0, 1.0]), np.array([1.0, 0.0, 0.0]), np.array([0.0, c, s]), True)


@pytest.mark.parametrize("frame", [_rolled, _tilted_ey], ids=["rolled", "tilted_ey"])
def test_mirror_unshared_direction_bit_identical(native, monkeypatch, frame):
    import torch
    from light_path_tracer_b200 import image_lens as il, _device as dev
    from light_path_tracer_b200.metrics import Schwarzschild
    monkeypatch.setattr(il, "_psi_frame", frame)
    metric = Schwarzschild(1.0)
    for H, W in ((270, 480), (101, 250), (99, 97)):
        vfov = np.radians(40.0)
        fov = (2 * np.arctan(np.tan(vfov / 2) * W / H), vfov)
        base = torch.rand(H, W, 3, device="cuda", generator=torch.Generator(device="cuda").manual_seed(H + W))
        for src, unit in (((base * 255).to(torch.uint8), True), (base, False)):
            for sampling in (il.SAMPLE_NEAREST, il.SAMPLE_BILINEAR):
                ref = il.render_frame(src, fov, 100.0, metric, sampling=sampling, unit_u8=unit,
                                      flags=dev.TRACE_HYBRID | dev.TRACE_REPACK)
                for extra in (0, dev.RENDER_STAGED_STORES):
                    out = il.render_frame(src, fov, 100.0, metric, sampling=sampling, unit_u8=unit,
                                          flags=dev.TRACE_HYBRID | extra)
                    assert torch.equal(out, ref), (frame.__name__, H, W, src.dtype, sampling, extra)
