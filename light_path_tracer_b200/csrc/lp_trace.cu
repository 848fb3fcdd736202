// lp_trace.cu — kernel (1a): one-thread-per-ray Schwarzschild Binet-equation RK4 tracer
// (replaces metrics.py:49-145, :661-668 and the drivers at image_lens.py:133-178).
//
// Layout: one thread per ray, non-persistent CTAs (256 rays) back-filled by the hardware work
// distributor; a warp owns 32 consecutive rays (= 32 consecutive pixels of a row), so
// the alpha loads and the fa / winding stores are fully coalesced.  The ray state
// (u, w, step index) lives in registers in fp64; the per-configuration constants and the
// strided phi table arrive through the kernel parameter (constant) bank.
#include "lp_trace.cuh"

#include <stdlib.h>

#define LP_RENDER_DEFAULT_TRIP 4
#define LP_RENDER_DEFAULT_TILE_H 4
#define LP_TRACE_DEFAULT_BLOCK 256  /* rays per CTA; LP_TRACE_BLOCK=32|64|128|256 overrides (tuning).  Measured on the
                                       14-instruction kernel (profiles/r2af_knob_sweep*.log): 256 is 4 % faster than 64 at 4K
                                       and 8K, 8-9 % on 1080p / divergent frames (with the 18-instruction step of the first
                                       half of the round 64 and 128 were equal; 512-thread CTAs are no faster than 256:
                                       profiles/r2ak_block512.log) */
/* frames of fewer rays than this run two RK4 steps per trip instead of four (less speculation past the exit and a
   smaller loop: 7 % faster at 1024 x 1024, 1 % at 4K r_obs = 15; four steps are 2.5-3.5 % faster at 4K / 8K r_obs = 100;
   measured on the one-ray-per-pixel kernel).  The mirror-image kernel applies it to the rays it traces: 2 steps for a
   mirrored 4K frame (2.08M traces; within 2 % either way) and 1080p (12 % faster), 4 for 8K (3 % faster):
   profiles/r3a_trip_sweep.log */
#define LP_RENDER_TRIP4_MIN_RAYS 4000000LL

// LP_TRACE_HYBRID rule.  The FMA loop (scaled second-order form, lp_internal.cuh) differs from the strict one
// by ~1e-16 per operation.  A perturbation d of the orbit obeys d'' = (-1 + 6 M u) d: it can only grow where
// r < 6M, at a rate <= 1 per radian for r >= 3M (= 1 at the photon sphere; an escaping ray never goes below 3M),
// so the difference is amplified by at most e^(phi - phi_out), phi_out = the angle the ray sweeps outside 6M.
// phi_out is smallest for the critical impact parameter, where it has a closed integrand
//     phi_out >= I(1/r_obs) + I(1/(2 r_obs)),  I(u0) = int_{u0}^{1/6M} du / sqrt(1/(27 M^2) - u^2 + 2 M u^3)
// (way in from the observer, way out to the escape radius; 1.87 rad at r_obs = 100 M, 0.16 at 3.49 M).
// The parity bar is |d final_alpha| <= 1e-9 max(final_alpha, 1e-3), so with ~1e-15 accumulated per ray and a
// factor ten of margin a ray may keep its FMA result while
//     e^(phi - phi_out) <= 1e5 max(final_alpha, 1e-3),   i.e.   phi - phi_out <= 11.5 + ln max(final_alpha, 1e-3):
// nobody is re-traced below phi - phi_out = 4.6, everybody above 11.5, and in between the rays whose
// final_alpha is small — the thin Einstein rings.  Re-traced rays are traced again strictly by the same thread
// (its warp waits: a re-traced ray costs about three warps' worth of time, which is why the rule is not simply
// "everything above 4.6 rad").  Measured: tools/nystrom_study.c (rays of <= 249 steps agree to a few 1e-11 over
// r_obs = 3.5 .. 1000 — relative to final_alpha >= 1e-3, which is what the final_alpha term is for:
// tools/parity_fuzz.py seed 31 found a 1.08e-12 difference at final_alpha = 9e-4, r_obs = 3.49 M, under the
// single 12-rad threshold this replaces).
#define LP_HYBRID_RETRACE_PHI 11.5
#define LP_HYBRID_RETRACE_PHI_SMALL 4.6

static double hybrid_phi_outside(double M, double r_obs)
{
    if (!(M > 0.0) || !(r_obs > 0.0) || !isfinite(M) || !isfinite(r_obs)) return 0.0;
    const double u6 = 1.0 / (6.0 * M), c0 = 1.0 / (27.0 * M * M);
    double total = 0.0;
    for (int leg = 0; leg < 2; ++leg) {
        const double u0 = 1.0 / (leg == 0 ? r_obs : 2.0 * r_obs);
        if (!(u0 < u6)) continue;
        const int n = 2000;                              // Simpson; the integrand is smooth below the double root at 1/3M
        const double hq = (u6 - u0) / n;
        double acc = 0.0;
        for (int i = 0; i <= n; ++i) {
            const double u = u0 + hq * i;
            const double f = 1.0 / sqrt(c0 - u * u + 2.0 * M * u * u * u);
            acc += f * ((i == 0 || i == n) ? 1.0 : (i & 1) ? 4.0 : 2.0);
        }
        total += acc * hq / 3.0;
    }
    return (total > 0.0 && isfinite(total)) ? total : 0.0;
}

static int steps_for_phi(double phi, double h_max)
{
    if (!(h_max > 0.0)) return 0;                       // degenerate step: everything strict
    const double k = floor(phi / h_max + 1e-9);
    return k < 1.0 ? 0 : (k > 1.0e9 ? 0x7fffffff : (int)k);
}

void lp_hybrid_rule(uint32_t flags, double M, double r_obs, double h_max, TraceArgs *a)
{
    a->retrace_steps = a->retrace_steps_small = 0x7fffffff;
    a->retrace_h = (float)h_max; a->retrace_off = 0.0f;
    if (!(flags & LP_TRACE_HYBRID)) return;
    // (the quadrature is ~20 us of host time: remembered per thread for the last configuration)
    static thread_local double last_M = 0.0, last_r = 0.0, last_phi = 0.0;
    if (!(M == last_M && r_obs == last_r)) { last_phi = hybrid_phi_outside(M, r_obs); last_M = M; last_r = r_obs; }
    const double phi_out = 0.95 * last_phi;              // (5 % off the bound for the quadrature and the float test)
    a->retrace_steps = steps_for_phi(LP_HYBRID_RETRACE_PHI + phi_out, h_max);
    a->retrace_steps_small = steps_for_phi(LP_HYBRID_RETRACE_PHI_SMALL + phi_out, h_max);
    a->retrace_off = (float)(LP_HYBRID_RETRACE_PHI + phi_out);
}

extern "C" int lp_hybrid_retrace_rule(double M, double r_obs, double h_max,
                                      int32_t *steps_all, int32_t *steps_none, double *exp_offset, double *phi_outside)
{
    TraceArgs a = {};
    lp_hybrid_rule(LP_TRACE_HYBRID, M, r_obs, h_max, &a);
    if (steps_all) *steps_all = a.retrace_steps;
    if (steps_none) *steps_none = a.retrace_steps_small;
    if (exp_offset) *exp_offset = (double)a.retrace_off;
    if (phi_outside) *phi_outside = hybrid_phi_outside(M, r_obs);
    return LP_OK;
}

// One ray per thread, one CTA per `blockDim.x` consecutive rays.  The grid is NOT
// persistent on purpose: the SMSP arbiter is unfair between always-eligible warps, so a
// resident-forever grid finishes its warps at very different times and the tail runs
// under-occupied (ncu, round 1: 5.6 of 8 warps active on average); one-shot CTAs let the
// hardware work distributor back-fill SMs as warps retire.
template <bool FUSED, bool FAST, int SRC, bool WIDE>
__global__ void __launch_bounds__(LP_TRACE_BLOCK)
lp_trace_kernel(const TraceArgs a, const BinetConsts c, const CamConsts cam)
{
    const LoopRegs L = load_loop_regs<FUSED>(c);
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < a.n;
    RayResult r;
    r.status = 0; r.steps = 0; r.nh = 0; r.fa = 0.0;
    if (live) {
        double alpha;
        if (SRC == SRC_F64) {
            alpha = __ldg((const double *)a.alphas + i);
        } else if (SRC == SRC_F32) {
            alpha = (double)__ldg((const float *)a.alphas + i);   // image_lens.py:157
        } else {
            int row, col;
            pixel_row_col(i, a.n, cam.width, a.row0, row, col);
            const double xc = cam_x(cam, col);
            const double yc = cam_y(cam, row);
            const float a32 = (float)pixel_alpha64(cam, xc, yc);     // image_lens.py:152
            if (a.out_alpha32) a.out_alpha32[i] = a32;
            alpha = (double)a32;
        }
        binet_trace<FUSED, FAST, (FUSED && FAST) ? LP_RENDER_DEFAULT_TRIP : 2>(c, L, alpha, r);
        if (__builtin_expect(FUSED && hybrid_needs_retrace(r, a.retrace_steps, a.retrace_steps_small, a.retrace_h, a.retrace_off), 0))
            binet_trace<false, FAST>(c, load_loop_regs<false>(c), alpha, r);   // cold: its own constants
        const double fa = (r.status == 1) ? r.fa : __longlong_as_double(0x7ff8000000000000LL);
        if (WIDE) {
            ((double *)a.out_fa)[i] = fa;                          // metrics.py:667
            ((long long *)a.out_w)[i] = r.nh;                      // metrics.py:668
        } else {
            ((float *)a.out_fa)[i] = (float)fa;                    // image_lens.py:176
            const long long nh = r.nh < 0 ? 0 : (r.nh > 65535 ? 65535 : r.nh);
            ((unsigned short *)a.out_w)[i] = (unsigned short)nh;   // image_lens.py:177
        }
        if (a.out_status) a.out_status[i] = (int8_t)r.status;
        if (a.out_steps) a.out_steps[i] = r.steps;
    }
    if (a.stats) {
        StatAcc acc;
        acc.init();
        acc.add(r, live);
        lp_stats_flush(acc, live ? 1ull : 0ull, a.stats);
    }
}

static int trace_block_size()
{
    static int cached = 0;
    if (!cached) {
        int v = LP_TRACE_DEFAULT_BLOCK;
        const char *e = getenv("LP_TRACE_BLOCK");
        if (e) { const int t = atoi(e); if (t == 32 || t == 64 || t == 128 || t == 256) v = t; }
        cached = v;
    }
    return cached;
}

template <int SRC, bool WIDE>
static int launch_trace(const TraceArgs &a, const BinetConsts &c, const CamConsts &cam,
                        uint32_t flags, cudaStream_t stream)
{
    if (a.n == 0) return LP_OK;
    // the FMA loop integrates 3M u: without a usable scale (c.scaled_ok) the request runs strictly
    const bool fused = (flags & (LP_TRACE_FUSED | LP_TRACE_HYBRID)) != 0 && c.scaled_ok;
    const bool icmp = (fused ? lp_binet_fast_ok_fused(&c) : lp_binet_fast_ok(&c)) != 0;
    const int block = trace_block_size();
    const long long chunks = (a.n + block - 1) / block;
    if (chunks > 0x7fffffffLL) return LP_ERR_UNSUPPORTED;
    const unsigned grid = (unsigned)chunks;
    if (fused) {
        if (icmp) lp_trace_kernel<true, true, SRC, WIDE><<<grid, block, 0, stream>>>(a, c, cam);
        else      lp_trace_kernel<true, false, SRC, WIDE><<<grid, block, 0, stream>>>(a, c, cam);
    } else {
        if (icmp) lp_trace_kernel<false, true, SRC, WIDE><<<grid, block, 0, stream>>>(a, c, cam);
        else      lp_trace_kernel<false, false, SRC, WIDE><<<grid, block, 0, stream>>>(a, c, cam);
    }
    return lp_check_launch();
}

extern "C" int lp_schw_trace_batch_f64(const double *alphas, int64_t n,
                                       double M, double R_S, double r_obs,
                                       double phi_max, double h_max,
                                       double *out_fa, int64_t *out_w,
                                       int8_t *out_status, int32_t *out_steps,
                                       lp_frame_stats *stats, uint32_t flags, void *stream)
{
    if (n < 0) return LP_ERR_INVALID_ARG;
    if (n > 0 && (!alphas || !out_fa || !out_w)) return LP_ERR_INVALID_ARG;
    BinetConsts c;
    int rc = lp_make_binet_consts(M, R_S, r_obs, phi_max, h_max, &c);
    if (rc != LP_OK) return rc;
    CamConsts cam = {};
    TraceArgs a = {};
    lp_hybrid_rule(flags, M, r_obs, h_max, &a);
    a.alphas = alphas; a.n = n; a.out_fa = out_fa; a.out_w = out_w;
    a.out_status = out_status; a.out_steps = out_steps; a.stats = stats;
    return launch_trace<SRC_F64, true>(a, c, cam, flags, (cudaStream_t)stream);
}

extern "C" int lp_schw_trace_alpha32(const float *alpha32, int64_t n,
                                     double M, double R_S, double r_obs,
                                     double phi_max, double h_max,
                                     float *out_fa32, uint16_t *out_w16,
                                     int8_t *out_status, int32_t *out_steps,
                                     lp_frame_stats *stats, uint32_t flags, void *stream)
{
    if (n < 0) return LP_ERR_INVALID_ARG;
    if (n > 0 && (!alpha32 || !out_fa32 || !out_w16)) return LP_ERR_INVALID_ARG;
    BinetConsts c;
    int rc = lp_make_binet_consts(M, R_S, r_obs, phi_max, h_max, &c);
    if (rc != LP_OK) return rc;
    CamConsts cam = {};
    TraceArgs a = {};
    lp_hybrid_rule(flags, M, r_obs, h_max, &a);
    a.alphas = alpha32; a.n = n; a.out_fa = out_fa32; a.out_w = out_w16;
    a.out_status = out_status; a.out_steps = out_steps; a.stats = stats;
    return launch_trace<SRC_F32, false>(a, c, cam, flags, (cudaStream_t)stream);
}

extern "C" int lp_schw_trace_frame(const lp_camera *h_cam, int32_t row0, int32_t rows,
                                   double M, double R_S, double r_obs,
                                   double phi_max, double h_max,
                                   float *out_alpha32, float *out_fa32, uint16_t *out_w16,
                                   int8_t *out_status, int32_t *out_steps,
                                   lp_frame_stats *stats, uint32_t flags, void *stream)
{
    CamConsts cam;
    int rc = lp_make_cam_consts(h_cam, &cam);
    if (rc != LP_OK) return rc;
    if (row0 < 0 || rows < 0 || (long long)row0 + rows > cam.height) return LP_ERR_INVALID_ARG;
    const long long n = (long long)rows * cam.width;
    if (n > 0 && (!out_fa32 || !out_w16)) return LP_ERR_INVALID_ARG;
    BinetConsts c;
    rc = lp_make_binet_consts(M, R_S, r_obs, phi_max, h_max, &c);
    if (rc != LP_OK) return rc;
    TraceArgs a = {};
    lp_hybrid_rule(flags, M, r_obs, h_max, &a);
    a.n = n; a.out_fa = out_fa32; a.out_w = out_w16; a.out_alpha32 = out_alpha32;
    a.out_status = out_status; a.out_steps = out_steps; a.stats = stats; a.row0 = row0;
    return launch_trace<SRC_CAM, false>(a, c, cam, flags, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------
// Fully fused frame: pixel -> alpha(f32) -> trace -> fa(f32), w(u16) -> remap -> pixel.
// Same per-ray code as the kernels above followed by remap_pixel() on the float32-rounded
// result, so the output is bit-identical to trace_frame + remap run back to back.
// ---------------------------------------------------------------------------
// One warp tile (32 pixels) per warp, one CTA per blockDim.x pixels, CTAs back-filled by the hardware
// work distributor.
template <bool FUSED, bool FAST, typename T, int MINB, int TRIP>
__global__ void __launch_bounds__(LP_TRACE_BLOCK, MINB)
lp_render_kernel(const TraceArgs a, const RemapArgs ra, const BinetConsts c, const CamConsts cam)
{
    const LoopRegs L = load_loop_regs<FUSED>(c);
    // RGB (float32 or 8-bit) into an aligned tile: the warp's 32 pixels — tile_h runs of 32 / tile_h
    // consecutive pixels — are staged in shared memory and leave as 16-byte (8-byte for 24-byte runs)
    // vector stores instead of 96 4-byte / 1-byte ones: full sectors, which is what peer (NVLink)
    // destinations need (dist.PeerFrame).
    __shared__ __align__(16) float stage[LP_TRACE_BLOCK / 32][96];
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const long long wt = (long long)blockIdx.x * (blockDim.x >> 5) + wrp;
    const long long i = wt * 32 + lane;
    const bool live = i < a.n;
    const bool vec = (sizeof(T) == 4 || sizeof(T) == 1) && ra.vec_ok && (wt * 32 + 31 < a.n);      // warp-uniform
    RayResult r;
    r.status = 0; r.steps = 0; r.nh = 0; r.fa = 0.0;
    int tr = 0, col = 0;
    if (live) {
        warp_tile_rc(a, cam.width, i, tr, col);
        const int row = tile_row(a, tr);
        const long long pi = (long long)tr * cam.width + col;                    // compact tile index
        const double xc = cam_x(cam, col), yc = cam_y(cam, row);     // also the remap's (kept across the loop)
        const float a32 = (float)pixel_alpha64(cam, xc, yc);
        binet_trace<FUSED, FAST, TRIP>(c, L, (double)a32, r);
        if (FUSED && hybrid_needs_retrace(r, a.retrace_steps, a.retrace_steps_small, a.retrace_h, a.retrace_off))
            binet_trace<false, FAST>(c, load_loop_regs<false>(c), (double)a32, r);   // cold
        const float fa32 = (float)((r.status == 1) ? r.fa : __longlong_as_double(0x7ff8000000000000LL));
        const long long nh = r.nh < 0 ? 0 : (r.nh > 65535 ? 65535 : r.nh);
        if (a.out_fa) ((float *)a.out_fa)[pi] = fa32;
        if (a.out_w) ((unsigned short *)a.out_w)[pi] = (unsigned short)nh;
        const long long oi = a.out_frame_rows ? (long long)(row - a.row0) * cam.width + col : pi;
        // two call sites so that each store has a known address space (shared / global) instead of
        // a generic pointer
        if (vec) remap_pixel_xy<T, true>(ra, cam, (T *)&stage[wrp][0] + lane * 3, xc, yc, fa32, (unsigned)nh, r.fa, r.cf, r.sf);
        else remap_pixel_xy<T, true>(ra, cam, (T *)ra.out + oi * ra.channels, xc, yc, fa32, (unsigned)nh, r.fa, r.cf, r.sf);
    }
    if (vec) {
        // vec_ok (host): every run of the warp tile is contiguous in the output and starts on a
        // vector boundary.  Vector v of the staged 96 floats / bytes belongs to run v / per_run.
        __syncwarp();
        const int r0 = __shfl_sync(0xffffffffu, tr, 0), c0 = __shfl_sync(0xffffffffu, col, 0);
        if (lane < a.st_lanes) {
            const int run = (int)(((unsigned)lane * a.st_magic) >> 16), part = lane - run * a.st_per_run;
            const int rr = r0 + run;
            const long long o0 = a.out_frame_rows ? (long long)(tile_row(a, rr) - a.row0) * cam.width + c0
                                                  : (long long)rr * cam.width + c0;
            unsigned char *g = (unsigned char *)((T *)ra.out + o0 * 3) + part * a.st_vb;
            const unsigned char *sm = (const unsigned char *)stage[wrp] + run * a.st_run_bytes + part * a.st_vb;
            if (a.st_vb == 16) *reinterpret_cast<uint4 *>(g) = *reinterpret_cast<const uint4 *>(sm);
            else *reinterpret_cast<uint2 *>(g) = *reinterpret_cast<const uint2 *>(sm);
        }
        __syncwarp();      // reconverge the warp after the lane-divergent stores
    }
    if (a.stats) {
        StatAcc acc;
        acc.init();
        acc.add(r, live);
        lp_stats_flush(acc, live ? 1ull : 0ull, a.stats);         // CTA-uniform: one pass per CTA
    }
}

// ---------------------------------------------------------------------------
// Mirror-image frame kernel: one ray per SET of mirror-image pixels.
// final_alpha, the winding and the step count of a pixel depend on its float32 viewing angle a32 alone, and
// a32 is mirror-symmetric bit for bit when the view direction d has d0 == 0 (x) or d1 == 0 (y) and d2 != 0:
// cam_x(W - col) == -cam_x(col) exactly (an exact integer / half-integer subtraction, then RN(x / f) or the
// Markstein sequence, both odd under round-to-nearest), pixel_alpha64 sees xc only as xc * xc and as
// xc * d0 = +-0, and a signed zero added to the nonzero d2 (or to yc * d1) disappears.  Pairs are col <-> W - col
// and row <-> H - row; column 0 / row 0 have no partner and W / 2, H / 2 (even sizes) are their own.
// So a lane traces a pixel of the traced quarter (or half) once and then remaps and stores each of its
// images with that image's own camera coordinates: the frame, the lookups and the statistics are the ones
// of the one-ray-per-pixel kernel.  8x4 warp tiles over the traced domain (see TraceArgs::mx_main).
// Staged stores (RGB, float32 / 8-bit): each run of an image (a tile row: up to 8 pixels, contiguous in the
// output, in reverse order for an x mirror) is staged at the same address modulo 16 as its destination; the
// run's lanes then store the 16-byte (float32) / 8-byte (8-bit) windows that lie inside it as vectors and the
// run's ends element by element.  A mirror image starts one pixel off the vector grid (column 0 is unpaired).
// ---------------------------------------------------------------------------
#define LP_MIRROR_RUN_SLOT 112      /* bytes of one staged run: 96 + up to 15 of alignment offset, rounded */

template <bool FUSED, bool FAST, typename T, int MINB, int TRIP>
__global__ void __launch_bounds__(LP_TRACE_BLOCK, MINB)
lp_render_mirror_kernel(const TraceArgs a, const RemapArgs ra, const BinetConsts c, const CamConsts cam)
{
    const LoopRegs L = load_loop_regs<FUSED>(c);
    __shared__ __align__(16) unsigned char stage[LP_TRACE_BLOCK / 32][4][LP_MIRROR_RUN_SLOT];
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5, j = lane & 7, q = lane >> 3;
    const unsigned wt = blockIdx.x * (blockDim.x >> 5) + wrp;
    const unsigned ty = wt / a.mtiles_x, tx = wt - ty * a.mtiles_x;
    int col, r;                  // frame column, tile-local row of the traced pixel
    bool live;
    if ((int)tx < a.mtx_main) { col = (int)(tx * 8u) + j; live = col < a.mx_main; col += a.mx_base; }
    else { col = 0; live = j == 0; }
    if ((int)ty < a.mty_main) { r = (int)(ty * 4u) + q; live = live && r < a.my_main; r += a.my_base; }
    else { r = 0; live = live && q == 0; }
    live = live && wt < a.m_warps;
    RayResult res;
    res.status = 0; res.steps = 0; res.nh = 0; res.fa = 0.0;
    if (live) {
        const float a32 = (float)pixel_alpha64(cam, cam_x(cam, col), cam_y(cam, a.row0 + r));
        binet_trace<FUSED, FAST, TRIP>(c, L, (double)a32, res);
        if (FUSED && hybrid_needs_retrace(res, a.retrace_steps, a.retrace_steps_small, a.retrace_h, a.retrace_off))
            binet_trace<false, FAST>(c, load_loop_regs<false>(c), (double)a32, res);   // cold
    }
    // (formed again rather than kept across the loop: fewer registers live in it)
    const double xc = cam_x(cam, col), yc = cam_y(cam, a.row0 + r);
    const float fa32 = (float)((res.status == 1) ? res.fa : __longlong_as_double(0x7ff8000000000000LL));
    const unsigned nh = (unsigned)(res.nh < 0 ? 0 : (res.nh > 65535 ? 65535 : res.nh));
    const int W = cam.width, H = cam.height;
    const bool xm = live && !(a.mir_skip & 1) && col != 0 && 2 * col != W;     // has an x mirror image
    const bool ym = live && !(a.mir_skip & 2) && r != 0 && 2 * r != H;         // (y mirror: row0 == 0, rows == H)
    const bool vec = (sizeof(T) == 4 || sizeof(T) == 1) && ra.vec_ok;
    const int px = 3 * (int)sizeof(T);               // bytes of a staged (RGB) pixel
#pragma unroll 1
    for (int k = 0; k < 4; ++k) {
        if (k & a.mir_skip) continue;                                   // warp-uniform
        const bool fx = (k & 1) != 0, fy = (k & 2) != 0;
        const bool has = live && (!fx || xm) && (!fy || ym);
        const int ic = fx ? W - col : col, ir = fy ? H - r : r;
        const long long pi = (long long)ir * W + ic;                    // compact tile index of this image
        if (has) {
            if (a.out_fa) ((float *)a.out_fa)[pi] = fa32;
            if (a.out_w) ((unsigned short *)a.out_w)[pi] = (unsigned short)nh;
        }
        // cam_x(W - col) == -cam_x(col), cam_y(H - r) == -cam_y(r) bit for bit (see above)
        const double xi = fx ? -xc : xc, yi = fy ? -yc : yc;
        if (vec) {
            // the run of tile row q in this image: columns [cmin, cmax] of tile-local row rr
            int cmin = has ? ic : 0x7fffffff, cmax = has ? ic : -1, rr = has ? ir : -1;
#pragma unroll
            for (int off = 1; off < 8; off <<= 1) {
                cmin = min(cmin, __shfl_xor_sync(0xffffffffu, cmin, off));
                cmax = max(cmax, __shfl_xor_sync(0xffffffffu, cmax, off));
                rr = max(rr, __shfl_xor_sync(0xffffffffu, rr, off));
            }
            uintptr_t lo = 0, hi = 0;
            unsigned char *sb = stage[wrp][q];
            if (cmax >= 0) {
                lo = (uintptr_t)ra.out + (uintptr_t)(((long long)rr * W + cmin) * px);
                hi = lo + (uintptr_t)((cmax - cmin + 1) * px);
                sb += lo & 15u;                                         // same address modulo 16 as the run
            }
            if (has) remap_pixel_xy<T, true>(ra, cam, (T *)(sb + (ic - cmin) * px), xi, yi, fa32, nh, res.fa, res.cf, res.sf);
            __syncwarp();
            if (cmax >= 0) {
                const unsigned vb = (sizeof(T) == 4) ? 16u : 8u;
                const uintptr_t g = (lo & ~(uintptr_t)(vb - 1u)) + j * vb;      // lane j: the run's window j
                const unsigned char *s = sb - (lo & (vb - 1u)) + j * vb;
                if (g < hi) {
                    if (g >= lo && g + vb <= hi) {
                        if (vb == 16u) *reinterpret_cast<uint4 *>(g) = *reinterpret_cast<const uint4 *>(s);
                        else *reinterpret_cast<uint2 *>(g) = *reinterpret_cast<const uint2 *>(s);
                    } else {
#pragma unroll
                        for (unsigned e = 0; e < vb; e += (unsigned)sizeof(T))
                            if (g + e >= lo && g + e < hi) *reinterpret_cast<T *>(g + e) = *reinterpret_cast<const T *>(s + e);
                    }
                }
            }
            __syncwarp();      // the staging slots are reused by the next image
        } else if (has) {
            remap_pixel_xy<T, true>(ra, cam, (T *)ra.out + pi * ra.channels, xi, yi, fa32, nh, res.fa, res.cf, res.sf);
        }
    }
    if (a.stats) {
        const unsigned m = (xm ? 2u : 1u) * (ym ? 2u : 1u);
        StatAcc acc;
        acc.init();
        acc.add_mult(res, live, m);
        lp_stats_flush(acc, live ? m : 0ull, a.stats);
    }
}

// RK4 steps per loop trip of the fast path: LP_RENDER_TRIP=2|4 (tuning knob).
static int render_trip(long long n_rays)
{
    static int cached = -1;
    if (cached < 0) {
        const char *e = getenv("LP_RENDER_TRIP");
        cached = (e && atoi(e) == 2) ? 2 : (e && atoi(e) == 4) ? 4 : 0;      // 0: by frame size
    }
    if (cached) return cached;
    return n_rays >= LP_RENDER_TRIP4_MIN_RAYS ? 4 : 2;
}

// MINB = 4 CTAs of LP_TRACE_BLOCK threads per SM -> ptxas keeps the kernel at 64 registers
// (32 warps/SM); a 48-register build (40 warps/SM, spills outside the loop) measured 1 % slower.
template <typename T>
static int launch_render(const TraceArgs &a, const RemapArgs &ra, const BinetConsts &c,
                         const CamConsts &cam, uint32_t flags, cudaStream_t stream)
{
    const bool fused = (flags & (LP_TRACE_FUSED | LP_TRACE_HYBRID)) != 0 && c.scaled_ok;
    const bool icmp = (fused ? lp_binet_fast_ok_fused(&c) : lp_binet_fast_ok(&c)) != 0;
    const int block = trace_block_size();
    const long long chunks = (a.n + block - 1) / block;
    if (chunks > 0x7fffffffLL) return LP_ERR_UNSUPPORTED;
    const unsigned grid = (unsigned)chunks;
    if (fused) {
        if (icmp && render_trip(a.n) == 4) lp_render_kernel<true, true, T, 4, 4><<<grid, block, 0, stream>>>(a, ra, c, cam);
        else if (icmp) lp_render_kernel<true, true, T, 4, 2><<<grid, block, 0, stream>>>(a, ra, c, cam);
        else      lp_render_kernel<true, false, T, 4, 2><<<grid, block, 0, stream>>>(a, ra, c, cam);
    } else {
        if (icmp && render_trip(a.n) == 4) lp_render_kernel<false, true, T, 4, 4><<<grid, block, 0, stream>>>(a, ra, c, cam);
        else if (icmp) lp_render_kernel<false, true, T, 4, 2><<<grid, block, 0, stream>>>(a, ra, c, cam);
        else      lp_render_kernel<false, false, T, 4, 2><<<grid, block, 0, stream>>>(a, ra, c, cam);
    }
    return lp_check_launch();
}

// The mirror-image kernel for a contiguous row tile: x mirror when mir_x, y mirror when mir_y (whole frame).
template <typename T>
static int launch_render_mirror(const TraceArgs &a_in, const RemapArgs &ra, const BinetConsts &c,
                                const CamConsts &cam, int32_t rows, bool mir_x, bool mir_y, uint32_t flags,
                                cudaStream_t stream)
{
    const bool fused = (flags & (LP_TRACE_FUSED | LP_TRACE_HYBRID)) != 0 && c.scaled_ok;
    const bool icmp = (fused ? lp_binet_fast_ok_fused(&c) : lp_binet_fast_ok(&c)) != 0;
    TraceArgs a = a_in;
    const int W = cam.width;
    a.mir_skip = (mir_x ? 0 : 1) | (mir_y ? 0 : 2);
    a.mx_main = mir_x ? W / 2 : W;           a.mx_base = mir_x ? W - W / 2 : 0;
    a.my_main = mir_y ? rows / 2 : rows;     a.my_base = mir_y ? rows - rows / 2 : 0;
    a.mtx_main = (a.mx_main + 7) / 8;        a.mty_main = (a.my_main + 3) / 4;
    const long long tiles_x = a.mtx_main + (mir_x ? 1 : 0), tiles_y = a.mty_main + (mir_y ? 1 : 0);
    const long long warps = tiles_x * tiles_y;
    const int block = trace_block_size();
    if (warps * 32 > 0x7fffffffLL) return LP_ERR_UNSUPPORTED;
    a.mtiles_x = (uint32_t)tiles_x; a.m_warps = (uint32_t)warps;
    const unsigned grid = (unsigned)((warps * 32 + block - 1) / block);
    const long long traced = (long long)(a.mx_main + (mir_x ? 1 : 0)) * (a.my_main + (mir_y ? 1 : 0));
    const int trip = render_trip(traced);
    if (fused) {
        if (icmp && trip == 4) lp_render_mirror_kernel<true, true, T, 4, 4><<<grid, block, 0, stream>>>(a, ra, c, cam);
        else if (icmp) lp_render_mirror_kernel<true, true, T, 4, 2><<<grid, block, 0, stream>>>(a, ra, c, cam);
        else      lp_render_mirror_kernel<true, false, T, 4, 2><<<grid, block, 0, stream>>>(a, ra, c, cam);
    } else {
        if (icmp && trip == 4) lp_render_mirror_kernel<false, true, T, 4, 4><<<grid, block, 0, stream>>>(a, ra, c, cam);
        else if (icmp) lp_render_mirror_kernel<false, true, T, 4, 2><<<grid, block, 0, stream>>>(a, ra, c, cam);
        else      lp_render_mirror_kernel<false, false, T, 4, 2><<<grid, block, 0, stream>>>(a, ra, c, cam);
    }
    return lp_check_launch();
}

// Frame rows of a (possibly interleaved) tile: last frame row + 1, or -1 for a bad request.
static long long tile_row_end(int32_t row0, int32_t rows, int32_t band_rows, int32_t band_stride)
{
    if (row0 < 0 || rows < 0 || band_rows < 0) return -1;
    if (band_rows == 0 || rows == 0) return (long long)row0 + rows;
    if (band_stride < band_rows) return -1;
    const long long r = rows - 1;
    return (long long)row0 + (r / band_rows) * band_stride + (r % band_rows) + 1;
}

extern "C" int lp_render_frame_bands(const void *src, int32_t src_dtype, int32_t channels,
                                     const lp_camera *h_cam, int32_t row0, int32_t rows,
                                     int32_t band_rows, int32_t band_stride,
                                     double M, double R_S, double r_obs, double phi_max, double h_max,
                                     int32_t render_loop_around, int32_t sampling,
                                     void *out, float *out_fa32, uint16_t *out_w16,
                                     lp_frame_stats *stats, uint32_t flags, void *stream)
{
    CamConsts cam;
    int rc = lp_make_cam_consts(h_cam, &cam);
    if (rc != LP_OK) return rc;
    const long long row_end = tile_row_end(row0, rows, band_rows, band_stride);
    if (row_end < 0 || row_end > cam.height) return LP_ERR_INVALID_ARG;
    if (channels < 1 || channels > 4) return LP_ERR_INVALID_ARG;
    if (sampling != LP_SAMPLE_NEAREST && sampling != LP_SAMPLE_BILINEAR) return LP_ERR_INVALID_ARG;
    const long long n = (long long)rows * cam.width;
    if (n == 0) return LP_OK;
    if (!src || !out) return LP_ERR_INVALID_ARG;
    BinetConsts c;
    rc = lp_make_binet_consts(M, R_S, r_obs, phi_max, h_max, &c);
    if (rc != LP_OK) return rc;
    const bool frame_rows = (flags & LP_RENDER_OUT_FRAME_ROWS) != 0;
    TraceArgs a = {};
    lp_hybrid_rule(flags, M, r_obs, h_max, &a);
    a.n = n; a.out_fa = out_fa32; a.out_w = out_w16; a.stats = stats; a.row0 = row0;
    a.band_rows = band_rows; a.band_stride = band_stride;
    a.out_frame_rows = (frame_rows && band_rows > 0) ? 1 : 0;     // contiguous rows: frame-addressed == compact
    RemapArgs ra;
    ra.src = src; ra.out = out; ra.fa32 = nullptr; ra.w16 = nullptr; ra.n = n;
    ra.row0 = row0; ra.channels = channels; ra.loop_around = render_loop_around; ra.sampling = sampling;
    // warp tile: LP_RENDER_TILE_H = 1 | 2 | 4 rows per warp (tuning knob; default 4 = 8x4 pixels)
    static int tile_h_pref = 0, tile_h_env = 0;
    if (!tile_h_pref) {
        const char *e = getenv("LP_RENDER_TILE_H");
        const int v = e ? atoi(e) : 0;
        tile_h_env = (v == 1 || v == 2 || v == 4);
        tile_h_pref = tile_h_env ? v : LP_RENDER_DEFAULT_TILE_H;
    }
    int th = tile_h_pref;
    // LP_RENDER_ROW_RUNS: 8-bit row bands of a frame that MANY peers store into one GPU's memory over NVLink
    // (dist.PeerFrame at more than four ranks).  An 8 x 4 tile's runs are 24 bytes — 8-byte stores into partial
    // 32-byte sectors, ~200 GB/s into the root at 8 GPUs (measured: config 4 at 0.447 ms against 0.31 of compute)
    // — where a 32 x 1 tile's run is 96 bytes = three whole sectors in 16-byte stores, like the float32 tiles'.
    if (!tile_h_env && (flags & LP_RENDER_ROW_RUNS) && (src_dtype == LP_DTYPE_U8 || src_dtype == LP_DTYPE_U8_UNIT)) th = 1;
    while (th > 1 && (cam.width % (32 / th) != 0 || rows % th != 0)) th >>= 1;
    a.tile_h = th; a.tiles_x = cam.width / (32 / th);
    a.tile_shift = (th == 4) ? 2u : (th == 2) ? 1u : 0u;
    a.tiles_x_magic = 0u;
    if ((th > 1 || cam.width % 32 == 0) && a.tiles_x > 1) {
        // w / tiles_x == (w * ceil(2^32 / tiles_x)) >> 32 for all w <= w_max iff w_max * e < 2^32,
        // e = tiles_x * ceil(2^32 / tiles_x) - 2^32
        const unsigned long long d = (unsigned long long)a.tiles_x, two32 = 1ull << 32;
        const unsigned long long m = (two32 + d - 1) / d, e = m * d - two32;
        const unsigned long long w_max = (unsigned long long)((n + 31) / 32) + 64;
        if (m < two32 && w_max * e < two32) a.tiles_x_magic = (uint32_t)m;
    }
    const bool contiguous32 = !a.out_frame_rows || cam.width % 32 == 0;
    const bool runs_ok = th > 1 || contiguous32;        // every run of a warp tile contiguous and vector-aligned
    ra.vec_ok = ((flags & LP_RENDER_STAGED_STORES) && channels == 3 && runs_ok &&
                 (src_dtype == LP_DTYPE_F32 || src_dtype == LP_DTYPE_U8 || src_dtype == LP_DTYPE_U8_UNIT) &&
                 ((uintptr_t)out % 16) == 0) ? 1 : 0;
    {   // write-out geometry of a warp tile (see TraceArgs)
        const int esz = (src_dtype == LP_DTYPE_F32) ? 4 : (src_dtype == LP_DTYPE_F64) ? 8 : 1;
        a.st_run_bytes = (32 / th) * 3 * esz;
        a.st_vb = (a.st_run_bytes % 16 == 0) ? 16 : 8;
        a.st_per_run = a.st_run_bytes / a.st_vb;
        a.st_lanes = th * a.st_per_run;
        a.st_magic = (65536u + (uint32_t)a.st_per_run - 1u) / (uint32_t)a.st_per_run;
        if (a.st_run_bytes % 8 != 0 || a.st_lanes > 32) ra.vec_ok = 0;
    }
    ra.u8_scale = (src_dtype == LP_DTYPE_U8_UNIT) ? 255.0f : 1.0f;
    ra.fast3 = (channels == 3 && sampling == LP_SAMPLE_NEAREST &&
                (long long)cam.height * cam.width * 3 < 0x7fffffffLL) ? 1 : 0;
    if (src_dtype == LP_DTYPE_U8_UNIT) src_dtype = LP_DTYPE_U8;
    cudaStream_t st = (cudaStream_t)stream;
    // opt-in lane re-packing schedule; it needs the fast-path precondition (observer strictly inside
    // the integration band), otherwise the request falls through to the default kernel
    const bool rp_fused = (flags & (LP_TRACE_FUSED | LP_TRACE_HYBRID)) != 0 && c.scaled_ok;
    if ((flags & LP_TRACE_REPACK) && (rp_fused ? lp_binet_fast_ok_fused(&c) : lp_binet_fast_ok(&c)) && c.valid && n <= 0x7fffffffLL) {
        ra.vec_ok = (contiguous32 && ((uintptr_t)out % 16) == 0) ? 1 : 0;   // chunks are staged by construction
        return lp_launch_render_repack(a, ra, c, cam, src_dtype, flags, st);
    }
    // mirror images (lp_render_mirror_kernel): contiguous rows stored compactly, default schedule; x needs
    // d0 == 0 (either sign), y needs d1 == 0 and the whole frame, both need d2 != 0
    const bool mir_ok = band_rows == 0 && !(flags & (LP_RENDER_OUT_FRAME_ROWS | LP_RENDER_ROW_RUNS)) && cam.d2 != 0.0;
    const bool mir_x = mir_ok && cam.d0 == 0.0;
    const bool mir_y = mir_ok && cam.d1 == 0.0 && row0 == 0 && rows == cam.height;
    if (mir_x || mir_y) {
        const int esz = (src_dtype == LP_DTYPE_F32) ? 4 : 1;
        ra.vec_ok = ((flags & LP_RENDER_STAGED_STORES) && channels == 3 &&
                     (src_dtype == LP_DTYPE_F32 || src_dtype == LP_DTYPE_U8) && ((uintptr_t)out % esz) == 0) ? 1 : 0;
        switch (src_dtype) {
        case LP_DTYPE_U8: return launch_render_mirror<unsigned char>(a, ra, c, cam, rows, mir_x, mir_y, flags, st);
        case LP_DTYPE_F32: return launch_render_mirror<float>(a, ra, c, cam, rows, mir_x, mir_y, flags, st);
        case LP_DTYPE_F64: return launch_render_mirror<double>(a, ra, c, cam, rows, mir_x, mir_y, flags, st);
        default: return LP_ERR_INVALID_ARG;
        }
    }
    switch (src_dtype) {
    case LP_DTYPE_U8: return launch_render<unsigned char>(a, ra, c, cam, flags, st);
    case LP_DTYPE_F32: return launch_render<float>(a, ra, c, cam, flags, st);
    case LP_DTYPE_F64: return launch_render<double>(a, ra, c, cam, flags, st);
    default: return LP_ERR_INVALID_ARG;
    }
}

extern "C" int lp_render_frame(const void *src, int32_t src_dtype, int32_t channels,
                               const lp_camera *h_cam, int32_t row0, int32_t rows,
                               double M, double R_S, double r_obs, double phi_max, double h_max,
                               int32_t render_loop_around, int32_t sampling,
                               void *out, float *out_fa32, uint16_t *out_w16,
                               lp_frame_stats *stats, uint32_t flags, void *stream)
{
    return lp_render_frame_bands(src, src_dtype, channels, h_cam, row0, rows, 0, 0, M, R_S, r_obs, phi_max, h_max,
                                 render_loop_around, sampling, out, out_fa32, out_w16, stats, flags, stream);
}

// ---------------------------------------------------------------------------
// build_alpha_lookup alone (image_lens.py:133-152)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
lp_alpha_lookup_kernel(const CamConsts cam, int row0, long long n, int decimals, double scale,
                       float *__restrict__ out)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        int row, col;
        pixel_row_col(i, n, cam.width, row0, row, col);
        double al = pixel_alpha64(cam, cam_x(cam, col), cam_y(cam, row));
        if (decimals >= 0) al = __ddiv_rn(rint(mul_(al, scale)), scale);   // np.round(alpha, decimals)
        out[i] = (float)al;
    }
}

extern "C" int lp_build_alpha_lookup(const lp_camera *h_cam, int32_t row0, int32_t rows,
                                     int32_t decimals, float *out_alpha32, void *stream)
{
    CamConsts cam;
    int rc = lp_make_cam_consts(h_cam, &cam);
    if (rc != LP_OK) return rc;
    if (row0 < 0 || rows < 0 || (long long)row0 + rows > cam.height) return LP_ERR_INVALID_ARG;
    if (decimals > 300) return LP_ERR_INVALID_ARG;
    const long long n = (long long)rows * cam.width;
    if (n == 0) return LP_OK;
    if (!out_alpha32) return LP_ERR_INVALID_ARG;
    int grid = 0;
    rc = lp_grid_for((const void *)lp_alpha_lookup_kernel, 256, n, &grid);
    if (rc != LP_OK) return rc;
    double scale = 1.0;
    for (int i = 0; i < decimals; ++i) scale *= 10.0;
    lp_alpha_lookup_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(cam, row0, n, decimals, scale, out_alpha32);
    return lp_check_launch();
}

// ---------------------------------------------------------------------------
// FP64 pipe micro-benchmark (roofline denominator; see lightpath.h)
// ---------------------------------------------------------------------------
__global__ void lp_dfma_kernel(int iters, double *sink)
{
    double a0 = 1.0 + threadIdx.x * 1e-9, a1 = a0 + 1e-3, a2 = a0 + 2e-3, a3 = a0 + 3e-3;
    double a4 = a0 + 4e-3, a5 = a0 + 5e-3, a6 = a0 + 6e-3, a7 = a0 + 7e-3;
    const double m = 0.999999, b = 1e-7;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, m, b); a1 = fma(a1, m, b); a2 = fma(a2, m, b); a3 = fma(a3, m, b);
        a4 = fma(a4, m, b); a5 = fma(a5, m, b); a6 = fma(a6, m, b); a7 = fma(a7, m, b);
    }
    sink[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

extern "C" int lp_bench_dfma(int32_t blocks, int32_t threads, int32_t iters, double *sink, void *stream)
{
    if (blocks <= 0 || threads <= 0 || threads > 1024 || iters < 0 || !sink) return LP_ERR_INVALID_ARG;
    lp_dfma_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(iters, sink);
    return lp_check_launch();
}
