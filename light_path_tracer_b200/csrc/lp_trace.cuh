// lp_trace.cuh — launch arguments shared by the Binet tracer kernels (lp_trace.cu) and the
// lane re-packing frame kernel (lp_repack.cu).
#pragma once
#include "lp_internal.cuh"
#include "lp_remap.cuh"

#define LP_TRACE_BLOCK 256          /* launch bound (max threads per CTA) */

enum { SRC_F64 = 0, SRC_F32 = 1, SRC_CAM = 2 };

struct TraceArgs {
    const void *alphas;     // SRC_F64: const double*, SRC_F32: const float*, SRC_CAM: unused
    long long n;            // rays in this launch
    void *out_fa;           // WIDE: double*, else float*
    void *out_w;            // WIDE: int64_t*, else uint16_t*
    float *out_alpha32;     // SRC_CAM only, optional
    int8_t *out_status;     // optional
    int32_t *out_steps;     // optional
    lp_frame_stats *stats;  // optional
    int32_t row0;           // SRC_CAM: first frame row of the tile
    int32_t retrace_steps_small;   // ... and the step count below which no ray is (see hybrid_needs_retrace)
    float retrace_h, retrace_off;  // step size and exponent offset as floats, for that test
    int32_t retrace_steps;  // FUSED kernels: a ray that ran more RK4 steps than this is traced
                            // again with strict arithmetic (LP_TRACE_HYBRID); INT_MAX = never
    // interleaved row bands (lp_render_frame_bands): tile-local row r is frame row
    // row0 + (r / band_rows) * band_stride + (r % band_rows); band_rows == 0: contiguous
    int32_t band_rows, band_stride;
    int32_t out_frame_rows; // the pixel tile is frame-addressed (LP_RENDER_OUT_FRAME_ROWS)
    // warp tile of the one-ray-per-thread frame kernel: a warp owns tile_h rows x (32 / tile_h)
    // columns of pixels instead of 32 consecutive pixels of one row (tile_h = 1).  The RK4 step count
    // of a ray is a smooth function of its viewing angle, i.e. of the pixel's distance from the black
    // hole's image, so a compact 8x4 tile has a smaller spread of step counts than a 32x1 strip
    // (fewer idle lanes around the shadow edge).  tiles_x = width / (32 / tile_h).
    int32_t tile_h, tiles_x;
    // tile_shift = log2(tile_h); tiles_x_magic = ceil(2^32 / tiles_x) when the host has verified that
    // __umulhi(w, magic) == w / tiles_x for every warp tile index w of this launch, else 0 (plain division)
    uint32_t tile_shift, tiles_x_magic;
    uint32_t m_edge;        // mirror-image frame kernel: warp tiles of column 0 / row 0 (placed here so that
                            // the 4-byte fields below share 8-byte words in pairs as the kernels load them)
    // staged stores of the frame kernel (host-side arithmetic of the warp's write-out, so that the kernel
    // has no integer division): bytes of one run of the warp tile, vector width (16 / 8), vectors per run,
    // lanes that store (tile_h * per_run), and ceil(2^16 / per_run) for lane / per_run by multiply-shift
    int32_t st_run_bytes, st_vb, st_per_run, st_lanes;
    uint32_t st_magic;
    // mirror-image frame kernel (lp_render_mirror_kernel): the traced columns are mx_base .. mx_base + mx_main - 1
    // in mtx_main warp-tile columns of 8, then (x mirror) one more tile column whose first lane traces column 0;
    // the same for tile-local rows in tiles of 4 (my_*).  Image k = 0..3 of a ray is mirrored in x when k & 1 and
    // in y when k & 2; the images with k & mir_skip do not exist in this launch.  Bit 1 (x) / 2 (y) of mir_share:
    // the camera basis carries that mirror over to the remap's source direction exactly (lp_render_mirror_kernel).
    int16_t mir_skip, mir_share;
    int32_t mx_main, mx_base, mtx_main, my_main, my_base, mty_main;
    // CTA b < m_ctas owns strip b % m_strips of tile row b / m_strips: its warps' tiles side by side (m_strips
    // strips per tile row); the CTAs after them hold the m_edge tiles of column 0 and row 0, one per warp
    uint32_t m_strips, m_ctas;
};

// frame row of tile-local row r (interleaved bands, see above)
__device__ __forceinline__ int tile_row(const TraceArgs &a, int r)
{
    if (a.band_rows > 0) r += (r / a.band_rows) * (a.band_stride - a.band_rows);
    return a.row0 + r;
}

// thread index -> tile-local (row r, column) under the warp-tile mapping
__device__ __forceinline__ void warp_tile_rc(const TraceArgs &a, int width, long long i, int &r, int &col)
{
    if (a.tile_h <= 1 && !a.tiles_x_magic) { pixel_row_col(i, a.n, width, 0, r, col); return; }   // (32 x 1 tiles of a width that is a multiple of 32 take the multiply-high path)
    const unsigned wi = (unsigned)(i >> 5), l = (unsigned)i & 31u;
    const unsigned tw_shift = 5u - a.tile_shift;
    const unsigned ty = a.tiles_x_magic ? __umulhi(wi, a.tiles_x_magic) : wi / (unsigned)a.tiles_x;
    const unsigned tx = wi - ty * (unsigned)a.tiles_x;
    r = (int)((ty << a.tile_shift) + (l >> tw_shift));
    col = (int)((tx << tw_shift) + (l & ((1u << tw_shift) - 1u)));
}

// tile-local pixel index -> (frame row, column, element index of the pixel in the output tile)
__device__ __forceinline__ void tile_pixel(const TraceArgs &a, int width, long long i,
                                           int &row, int &col, long long &oi)
{
    int r;
    pixel_row_col(i, a.n, width, 0, r, col);
    if (a.band_rows > 0) {
        const int q = r / a.band_rows;
        r += q * (a.band_stride - a.band_rows);
    }
    row = a.row0 + r;
    oi = a.out_frame_rows ? (long long)r * width + col : i;
}

// LP_TRACE_HYBRID (lp_trace.cu): fills retrace_steps, retrace_steps_small, retrace_h, retrace_off of `a`
void lp_hybrid_rule(uint32_t flags, double M, double r_obs, double h_max, TraceArgs *a);

// Does the FMA loop's result have to be replaced by a strict re-trace?  With phi = steps * h:
//   steps > retrace_steps                                     (phi - phi_out > 11.5), or
//   steps > retrace_steps_small (phi - phi_out > 4.6) and max(final_alpha, 1e-3) < exp(phi - retrace_off)
// where retrace_off = 11.5 + phi_out and phi_out is the part of the swept angle that cannot amplify (lp_trace.cu).
__device__ __forceinline__ bool hybrid_needs_retrace(const RayResult &r, int retrace_steps, int retrace_steps_small,
                                                     float h, float off)
{
    if (r.steps <= retrace_steps_small) return false;                 // 99.9 % of a frame's rays stop here
    if (r.steps > retrace_steps) return true;
    if (r.status != 1) return false;
    return fmaxf((float)r.fa, 1.0e-3f) < __expf((float)r.steps * h - off);
}

// The build of the Binet loop a request runs: the FMA loop (FUSED) for LP_TRACE_FUSED / LP_TRACE_HYBRID, and the
// fast path (FAST, "icmp") where its precondition holds for the loops that kernel runs.
struct BinetVariant { bool fused, icmp; };
static inline BinetVariant lp_binet_variant(uint32_t flags, const BinetConsts &c)
{
    // the FMA loop integrates 3M u: without a usable scale (c.scaled_ok) the request runs strictly
    const bool fused = (flags & (LP_TRACE_FUSED | LP_TRACE_HYBRID)) != 0 && c.scaled_ok;
    return {fused, (fused ? lp_binet_fast_ok_fused(&c) : lp_binet_fast_ok(&c)) != 0};
}

// The Binet kernels' tuning knobs (DESIGN.md §4), read once per process (lp_trace.cu).
struct TraceKnobs {
    int block;          // LP_TRACE_BLOCK = 32 | 64 | 128 | 256: threads per CTA of the tracer and frame kernels
    int trip;           // LP_RENDER_TRIP = 2 | 4: RK4 steps per loop trip of the frame kernels; 0: by frame size
    int tile_h;         // LP_RENDER_TILE_H = 1 | 2 | 4: rows of lp_render_kernel's warp tile; 0: not set
    int repack_refill;  // LP_REPACK_REFILL = 1..32: idle lanes that trigger a refill of the re-packing kernel
};
const TraceKnobs &lp_trace_knobs();

// element type of a frame's source and output image: the index of the frame kernel tables
enum { ELEM_U8 = 0, ELEM_F32 = 1, ELEM_F64 = 2 };

int lp_launch_render_repack(TraceArgs a, RemapArgs ra, const BinetConsts &c, const CamConsts &cam, int elem,
                            bool fused, cudaStream_t stream);
