"""GPU parity of the mirror-image frame kernel's CTA strips (lp_render_mirror_kernel, lp_trace.cu).  A CTA
owns eight warp tiles side by side (a 64 x 4 strip of the traced domain), stages every image's rows for the
whole strip and stores them in one pass across the CTA; the tiles of column 0 and row 0 run in CTAs of their
own.  Frames, lookups and statistics must be the ones of the lane re-packing schedule (LP_TRACE_REPACK) and
the per-pixel tracer, BIT FOR BIT, at every strip remainder and output alignment."""
import pytest

from test_gpu_mirror import _check_lookups_and_stats, _setup, _sources

pytestmark = pytest.mark.gpu

# traced half W // 2 = 64 k + r for r in (0, 1, 7, 8, 63): full strips, and last strips of one pixel, of part
# of a warp tile, of one warp tile and of all but one pixel; even and odd widths
WIDTHS = [2 * (64 + r) + odd for r in (0, 1, 7, 8, 63) for odd in (0, 1)]
PSI = [(0.0, 0.0), (0.1, 0.0), (0.0, 0.1)]     # both mirrors, the x mirror alone, the y mirror alone
PSI_IDS = ["both", "x_only", "y_only"]


@pytest.mark.parametrize("psi", PSI, ids=PSI_IDS)
def test_mirror_strips_frames(native, psi):
    """Every strip remainder, odd and even heights, contiguous row tiles: 8-bit and float32 RGB through
    the staged strips, 1- and 4-channel images through the one-image-at-a-time path, nearest and bilinear."""
    import torch
    for W in WIDTHS:
        for H in (37, 24):
            il, dev, metric, fov = _setup(H, W)
            for name, src, unit in _sources(H, W, H * 1000 + W):
                if name == "u8x3":          # (u8x3unit covers the 8-bit RGB layout)
                    continue
                for sampling in (il.SAMPLE_NEAREST, il.SAMPLE_BILINEAR):
                    ref = il.render_frame(src, fov, 100.0, metric, psi=psi, sampling=sampling, unit_u8=unit,
                                          flags=dev.TRACE_HYBRID | dev.TRACE_REPACK)
                    out = il.render_frame(src, fov, 100.0, metric, psi=psi, sampling=sampling, unit_u8=unit,
                                          flags=dev.TRACE_HYBRID | dev.RENDER_STAGED_STORES)
                    assert torch.equal(out, ref), (psi, H, W, name, sampling)
                    for rows in ((5, H - 9), (0, 7)):
                        out = il.render_frame(src, fov, 100.0, metric, psi=psi, sampling=sampling, unit_u8=unit,
                                              rows=rows, flags=dev.TRACE_HYBRID | dev.RENDER_STAGED_STORES)
                        assert torch.equal(out, ref[rows[0]:rows[0] + rows[1]]), (psi, H, W, name, sampling, rows)


@pytest.mark.parametrize("psi", PSI, ids=PSI_IDS)
def test_mirror_strips_lookups_and_stats(native, psi):
    """Lookups and statistics of the strip schedule against the per-pixel tracer, whole frames and tiles."""
    for W in WIDTHS:
        for H in (37, 24):
            il, dev, metric, fov = _setup(H, W)
            src = _sources(H, W, 5)[0][1]
            for flags in (dev.TRACE_HYBRID, 0):
                _check_lookups_and_stats(il, dev, metric, fov, src, 100.0, psi, flags, False)
                _check_lookups_and_stats(il, dev, metric, fov, src, 100.0, psi, flags, False, rows=(3, H - 8))


def test_mirror_strips_offset_views(native):
    """Staged 8-bit and float32 RGB strips into views that start 1 .. 15 bytes off the 16-byte grid (float32:
    4, 8, 12): every pixel of the view is written and nothing around it."""
    import torch
    for H, W in ((37, 2 * (64 + 7) + 1), (24, 2 * (64 + 63)), (31, 2 * 128)):
        il, dev, metric, fov = _setup(H, W)
        for name, src, unit in _sources(H, W, 11):
            if name not in ("f32x3", "u8x3unit"):
                continue
            ref = il.render_frame(src, fov, 100.0, metric, unit_u8=unit, flags=dev.TRACE_HYBRID | dev.TRACE_REPACK)
            esz = src.element_size()
            for shift in range(1, 16 // esz):
                for rows in ((0, H), (3, H - 10)):
                    n = rows[1] * W * 3
                    big = torch.full((H * W * 3 + 32,), 77, device="cuda", dtype=src.dtype)
                    view = big[shift:shift + n].view(rows[1], W, 3)
                    il.render_frame(src, fov, 100.0, metric, rows=rows, out=view, unit_u8=unit,
                                    flags=dev.TRACE_HYBRID | dev.RENDER_STAGED_STORES)
                    assert torch.equal(view, ref[rows[0]:rows[0] + rows[1]]), (H, W, name, shift, rows)
                    assert (big[:shift] == 77).all() and (big[shift + n:] == 77).all()
