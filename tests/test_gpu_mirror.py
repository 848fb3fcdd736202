"""GPU parity of the mirror-image frame kernel (lp_render_mirror_kernel, lp_trace.cu).  When the view
direction has d0 == 0 (psi_x = 0) the columns col and W - col see the same float32 viewing angle, and
with d1 == 0 (psi_y = 0) the rows row and H - row: the default frame kernel then traces one ray per set
of mirror images and remaps every image with its own camera coordinates.  Frames, lookups and statistics
must be the ones of a schedule that still traces one ray per pixel, BIT FOR BIT: the lane re-packing
kernel (LP_TRACE_REPACK) for frames, build_alpha_lookup + trace_alpha_table for lookups and statistics
(reference: image_lens.py:133-178, :296-397, metrics.py:49-145)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

STAT_KEYS = ("n_rays", "n_escaped", "n_captured", "n_invalid", "n_winding", "sum_steps", "max_steps",
             "max_winding", "min_final_alpha", "max_final_alpha")


def _setup(H, W, vfov_deg=40.0):
    from light_path_tracer_b200 import image_lens as il, _device as dev
    from light_path_tracer_b200.metrics import Schwarzschild
    vfov = np.radians(vfov_deg)
    fov = (2 * np.arctan(np.tan(vfov / 2) * W / H), vfov)
    return il, dev, Schwarzschild(1.0), fov


def _sources(H, W, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    base = torch.rand(H, W, 4, device="cuda", dtype=torch.float64, generator=g)
    rgb = base[..., :3].float().contiguous()
    return [("f32x3", rgb, False), ("f32x1", base[..., 0].float().contiguous(), False),
            ("f32x4", base.float().contiguous(), False),
            ("u8x3", (base[..., :3] * 255).to(torch.uint8).contiguous(), False),
            ("u8x3unit", (base[..., :3] * 255).to(torch.uint8).contiguous(), True),
            ("u8x4unit", (base * 255).to(torch.uint8).contiguous(), True)]


def _check_lookups_and_stats(il, dev, metric, fov, src, r_obs, psi, flags, unit, rows=None):
    """return_lookups and statistics of the frame kernel against the per-pixel tracer of the same tile."""
    import torch
    H, W = src.shape[0], src.shape[1]
    row0, n = (0, H) if rows is None else rows
    s0, s1 = dev.new_stats(), dev.new_stats()
    _, fa0, w0 = il.render_frame(src, fov, r_obs, metric, psi=psi, rows=rows, return_lookups=True, stats=s0,
                                 flags=flags, unit_u8=unit)
    a = il.build_alpha_lookup((H, W), fov, psi=psi, device=True)[row0:row0 + n].contiguous()
    fa1, w1 = metric.trace_alpha_table(a, r_obs, stats=s1, flags=flags)
    assert torch.equal(fa0.view(torch.int32), fa1.view(torch.int32))
    assert torch.equal(w0.view(torch.int16), w1.view(torch.int16))
    a0, a1 = dev.read_stats(s0), dev.read_stats(s1)
    for k in STAT_KEYS:
        assert a0[k] == a1[k], (k, a0[k], a1[k])
    assert a0["sum_steps"] <= a0["sum_warp_steps"]


@pytest.mark.parametrize("mode", ["hybrid", "strict"])
@pytest.mark.parametrize("psi", [(0.0, 0.0), (0.1, 0.0), (0.0, 0.1), (0.03, -0.02)],
                         ids=["psi0_0", "psi01_0", "psi0_01", "psi003_m002"])
def test_mirror_frames_bit_identical(native, mode, psi):
    """Frames of every image layout, nearest and bilinear, with and without staged stores, full frames
    and contiguous row tiles, even, odd and mixed sizes: identical to the re-packing schedule."""
    import torch
    flags0 = 4 if mode == "hybrid" else 0
    for H, W in ((270, 480), (101, 250), (99, 97), (64, 1)):
        il, dev, metric, fov = _setup(H, W)
        for name, src, unit in _sources(H, W, H * 1000 + W):
            for sampling in (il.SAMPLE_NEAREST, il.SAMPLE_BILINEAR):
                ref = il.render_frame(src, fov, 100.0, metric, psi=psi, sampling=sampling, unit_u8=unit,
                                      flags=flags0 | dev.TRACE_REPACK)
                for extra in (0, dev.RENDER_STAGED_STORES):
                    out = il.render_frame(src, fov, 100.0, metric, psi=psi, sampling=sampling, unit_u8=unit,
                                          flags=flags0 | extra)
                    assert torch.equal(out, ref), (H, W, name, sampling, extra)
                    for rows in ((0, 1), (3, H - 5), (H - 1, 1), (7, H // 2)):
                        if rows[1] <= 0:
                            continue
                        out = il.render_frame(src, fov, 100.0, metric, psi=psi, sampling=sampling, unit_u8=unit,
                                              rows=rows, flags=flags0 | extra)
                        assert torch.equal(out, ref[rows[0]:rows[0] + rows[1]]), (H, W, name, sampling, extra, rows)
        src = _sources(H, W, 5)[0][1]
        _check_lookups_and_stats(il, dev, metric, fov, src, 100.0, psi, flags0, False)
        if H > 8:
            _check_lookups_and_stats(il, dev, metric, fov, src, 100.0, psi, flags0, False, rows=(3, H - 8))


def test_mirror_staged_stores_misaligned_views(native):
    """Staged 8-bit and float32 RGB stores into views that start off the vector grid: every pixel of the
    view is written and nothing around it."""
    import torch
    for H, W in ((270, 480), (101, 250), (99, 97)):
        il, dev, metric, fov = _setup(H, W)
        for name, src, unit in _sources(H, W, 3):
            if src.dim() != 3 or src.shape[2] != 3:
                continue
            ref = il.render_frame(src, fov, 100.0, metric, unit_u8=unit, flags=dev.TRACE_HYBRID | dev.TRACE_REPACK)
            esz = src.element_size()
            for shift, rows in ((0, (0, H)), (1, (0, H)), (3, (7, H - 20)), (16 // esz, (3, 50))):
                n = rows[1] * W * 3
                big = torch.full((H * W * 3 + 32,), 77, device="cuda", dtype=src.dtype)
                view = big[shift:shift + n].view(rows[1], W, 3)
                il.render_frame(src, fov, 100.0, metric, rows=rows, out=view, unit_u8=unit,
                                flags=dev.TRACE_HYBRID | dev.RENDER_STAGED_STORES)
                assert torch.equal(view, ref[rows[0]:rows[0] + rows[1]]), (H, W, name, shift, rows)
                assert (big[:shift] == 77).all() and (big[shift + n:] == 77).all()


def test_mirror_4k(native):
    """The 3840 x 2160 frame at psi = 0, 8-bit in and out with staged stores (the benchmark's frame), and
    float32: frame, lookups and statistics of the per-pixel schedules."""
    import torch
    H, W = 2160, 3840
    il, dev, metric, fov = _setup(H, W)
    base = torch.rand(H, W, 3, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    src8 = (base * 255).to(torch.uint8)
    for src, unit in ((src8, True), (base, False)):
        ref = il.render_frame(src, fov, 100.0, metric, unit_u8=unit, flags=dev.TRACE_HYBRID | dev.TRACE_REPACK)
        out = il.render_frame(src, fov, 100.0, metric, unit_u8=unit,
                              flags=dev.TRACE_HYBRID | dev.RENDER_STAGED_STORES)
        assert torch.equal(out, ref)
    _check_lookups_and_stats(il, dev, metric, fov, base, 100.0, (0.0, 0.0), dev.TRACE_HYBRID, False)
    _check_lookups_and_stats(il, dev, metric, fov, base, 100.0, (0.0, 0.0), dev.TRACE_HYBRID, False,
                             rows=(540, 1080))
