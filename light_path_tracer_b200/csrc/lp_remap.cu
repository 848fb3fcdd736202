// lp_remap.cu — kernel (2): deflection -> background remap
// (replaces image_lens.render_lensed_image, image_lens.py:296-397).
//
// One thread per output pixel; a warp covers 32 consecutive pixels of a row, so the
// fa / winding loads and the pixel stores are coalesced; the source gather follows the
// lensing map, which is smooth away from the photon ring, so neighbouring lanes hit
// neighbouring source texels (L1/L2 resident).  All direction math is fp64 like the
// reference's; what must match is the INTEGER source index.
#include "lp_remap.cuh"
#include <stdlib.h>

template <typename T>
__global__ void __launch_bounds__(256)
lp_remap_kernel(const RemapArgs a, const CamConsts cam)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += stride) {
        const float fa32 = __ldg(a.fa32 + i);
        const unsigned wnd = a.w16 ? (unsigned)__ldg(a.w16 + i) : 0u;
        int row, col;
        pixel_row_col(i, a.n, cam.width, a.row0, row, col);
        remap_pixel<T>(a, cam, (T *)a.out + i * a.channels, row, col, fa32, wnd);
    }
}

// Fast path for the common layout — float32 RGB, nearest sampling, width % 4 == 0, 16-byte
// aligned tile pointers: one thread owns FOUR consecutive pixels of a row.  The lookups arrive
// as one 16-byte (fa) and one 8-byte (winding) vector load per thread, the four source
// directions are four independent fp64 chains (the latency-bound math overlaps), the twelve
// gather loads are issued back to back before any of them is consumed, and the 48 output
// bytes leave as three 16-byte stores, so every warp keeps ~4x more memory in flight than
// the one-pixel-per-thread kernel (the remap is latency-, not bandwidth-limited otherwise).
// Same per-pixel decisions as remap_pixel(), same integer source index.
#define LP_REMAP4_BLOCK 128
#define LP_REMAP4_DEFAULT_QUADS 1
#define LP_REMAP_DEFAULT_TMA 0

int lp_remap_try_tma(const RemapArgs &a, const CamConsts &cam, int src_dtype, int rows, cudaStream_t stream);

// sin and cos on [0, pi/2] (final_alpha of a sampled pixel is a float32 in that range): one
// conditional reflection about pi/4 instead of a general quadrant reduction, the fdlibm kernel
// polynomials with their coefficients from the constant bank (c_sin_poly / c_cos_poly, lp_internal.cuh:
// an FP64 instruction of sm_100 takes a constant through a uniform register, and a literal double costs two
// UMOVs where a table entry costs half an LDCU.128).
static __constant__ double c_quadrant[3] = {0.78539816339744828, 1.5707963267948966, 6.123233995736766e-17};   // pi/4, pi/2 hi, lo
__device__ __forceinline__ void sincos_first_quadrant(double x, double &s, double &c)
{
    const bool hi = x > c_quadrant[0];
    // pi/2 - x with the low word of pi/2: exact enough for a float32-valued x
    const double r = hi ? (c_quadrant[1] - x) + c_quadrant[2] : x;
    const double z = r * r;
    double ps = c_sin_poly[5];
    double pc = c_cos_poly[5];
#pragma unroll
    for (int k = 4; k >= 0; --k) { ps = fma(ps, z, c_sin_poly[k]); pc = fma(pc, z, c_cos_poly[k]); }
    const double sr = fma(r * z, ps, r);
    const double cr = fma(z * z, pc, fma(-0.5, z, 1.0));
    s = hi ? cr : sr;
    c = hi ? sr : cr;
}

// The per-quad pieces of the fast path: decisions + source offsets (pure math), gather, store.
__device__ __forceinline__ void quad_offsets(const RemapArgs &a, const CamConsts &cam, int col, double Ay, double By,
                                             const float4 fa4, const ushort4 w4, float (&o)[12], int (&off)[4])
{
    const float fa[4] = {fa4.x, fa4.y, fa4.z, fa4.w};
    const unsigned wn[4] = {w4.x, w4.y, w4.z, w4.w};
    const int H = cam.height, W = cam.width;                 // the host checks H * W * 3 < 2^31 for this kernel
    double px[4], py[4];
    bool front[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        // straight-line (interleavable across the four pixels); pixels that do not sample the
        // source (captured, winding) run the math on a harmless angle
        const bool samp = fa[p] <= LP_HALF_PI_F32;               // false for NaN
        const double xc = cam_x(cam, col + p);
        const double A = fma(xc, cam.ex0, Ay), B = fma(xc, cam.ey0, By);
        const double n2r = fma(A, A, B * B);
        const double n2 = (n2r > 1e-300) ? n2r : 1e-300;         // the on-axis pixel itself is never sampled (compare + select: fmax is ~7 instructions)
        const double inv = fast_rsqrt(n2);
        const double st = A * inv, ct = B * inv;
        double sf, cf;
        sincos_first_quadrant(samp ? (double)fa[p] : 0.5, sf, cf);
        const double sx = fma(cf, cam.d0, sf * fma(st, cam.ex0, ct * cam.ey0));
        const double sy = fma(cf, cam.d1, sf * fma(st, cam.ex1, ct * cam.ey1));
        const double sz = fma(cf, cam.d2, sf * fma(st, cam.ex2, ct * cam.ey2));
        front[p] = sz > 1e-12;
        const double isz = fast_rcp(front[p] ? sz : 1.0);
        px[p] = fma(sx * isz, cam.fx, cam.half_w);
        py[p] = fma(sy * isz, cam.fy, cam.half_h);
    }
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        off[p] = -1;
        const float f = fa[p];
        if (!isfinite(f)) {
            o[3 * p] = 0.0f; o[3 * p + 1] = 0.0f; o[3 * p + 2] = 0.0f;
        } else if (f > LP_HALF_PI_F32) {
            const unsigned k = wn[p] > 4u ? 4u : wn[p];
            o[3 * p] = c_wind_rgb[k][0]; o[3 * p + 1] = c_wind_rgb[k][1]; o[3 * p + 2] = c_wind_rgb[k][2];
        } else {
            // np.rint -> index; cvt.rni.s32.f64 rounds half to even and saturates, so a far
            // out-of-frame coordinate stays out of frame
            int ix = __double2int_rn(front[p] ? px[p] : cam.half_w);       // image_lens.py:356-361
            int iy = __double2int_rn(front[p] ? py[p] : cam.half_h);
            bool ok;
            if (a.loop_around) {
                ix %= W; ix += (ix < 0) ? W : 0;
                iy %= H; iy += (iy < 0) ? H : 0;
                ok = true;
            } else {
                ok = front[p] && (unsigned)ix < (unsigned)W && (unsigned)iy < (unsigned)H;
            }
            if (ok) off[p] = (iy * W + ix) * 3;
            else { o[3 * p] = 1.0f; o[3 * p + 1] = 0.0f; o[3 * p + 2] = 1.0f; }
        }
    }
}

__device__ __forceinline__ void quad_gather(const float *__restrict__ src, const int (&off)[4], float (&o)[12])
{
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        if (off[p] >= 0) {
            // (an 8-byte + 4-byte pair per texel instead of three 4-byte loads measured no faster: the kernel is
            // bound neither by L1 wavefronts nor — after the constant-table trims — by the issue port)
            o[3 * p] = __ldg(src + off[p]);
            o[3 * p + 1] = __ldg(src + off[p] + 1);
            o[3 * p + 2] = __ldg(src + off[p] + 2);
        }
    }
}

__device__ __forceinline__ void quad_store(float *out, long long i, const float (&o)[12])
{
    float4 *dst = reinterpret_cast<float4 *>(out + i * 3);
    dst[0] = make_float4(o[0], o[1], o[2], o[3]);
    dst[1] = make_float4(o[4], o[5], o[6], o[7]);
    dst[2] = make_float4(o[8], o[9], o[10], o[11]);
}

// QUADS consecutive quads per thread, software-pipelined: all lookups are loaded up front, the
// gathers of quad q are issued before the math of quad q+1 starts (so they are in flight under
// it), all stores come last.
template <int MINB, int QUADS>
__global__ void __launch_bounds__(LP_REMAP4_BLOCK, MINB)
lp_remap_f32rgb_x4_kernel(const RemapArgs a, const CamConsts cam)
{
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * (4 * QUADS);
    if (i >= a.n) return;
    int row, col;
    pixel_row_col(i, a.n, cam.width, a.row0, row, col);
    float4 fa4[QUADS];
    ushort4 w4[QUADS];
#pragma unroll
    for (int q = 0; q < QUADS; ++q) {
        fa4[q] = __ldg(reinterpret_cast<const float4 *>(a.fa32 + i) + q);
        w4[q] = a.w16 ? __ldg(reinterpret_cast<const ushort4 *>(a.w16 + i) + q) : make_ushort4(0, 0, 0, 0);
    }
    const float *__restrict__ src = (const float *)a.src;
    // row-constant parts of the two dot products A = v.e_x, B = v.e_y (v = (x_cam, y_cam, 1))
    const double yc = cam_y(cam, row);
    const double Ay = fma(yc, cam.ex1, cam.ex2), By = fma(yc, cam.ey1, cam.ey2);
    float o[QUADS][12];
    int off[QUADS][4];
#pragma unroll
    for (int q = 0; q < QUADS; ++q) {
        quad_offsets(a, cam, col + 4 * q, Ay, By, fa4[q], w4[q], o[q], off[q]);
        quad_gather(src, off[q], o[q]);
    }
#pragma unroll
    for (int q = 0; q < QUADS; ++q) quad_store((float *)a.out, i + 4 * q, o[q]);
}

extern "C" int lp_remap(const void *src, int32_t src_dtype, int32_t channels,
                        const lp_camera *h_cam, const float *fa32, const uint16_t *w16,
                        int32_t render_loop_around, int32_t sampling,
                        int32_t row0, int32_t rows, void *out, void *stream)
{
    CamConsts cam;
    int rc = lp_make_cam_consts(h_cam, &cam);
    if (rc != LP_OK) return rc;
    if (row0 < 0 || rows < 0 || (long long)row0 + rows > cam.height) return LP_ERR_INVALID_ARG;
    if (channels < 1 || channels > 4) return LP_ERR_INVALID_ARG;
    if (sampling != LP_SAMPLE_NEAREST && sampling != LP_SAMPLE_BILINEAR) return LP_ERR_INVALID_ARG;
    RemapArgs a;
    a.src = src; a.out = out; a.fa32 = fa32; a.w16 = w16;
    a.n = (long long)rows * cam.width;
    a.row0 = row0; a.channels = channels; a.loop_around = render_loop_around; a.sampling = sampling;
    a.vec_ok = 0;
    a.fast3 = (channels == 3 && sampling == LP_SAMPLE_NEAREST &&
               (long long)cam.height * cam.width * 3 < 0x7fffffffLL) ? 1 : 0;
    a.u8_scale = (src_dtype == LP_DTYPE_U8_UNIT) ? 255.0f : 1.0f;
    if (src_dtype == LP_DTYPE_U8_UNIT) src_dtype = LP_DTYPE_U8;
    if (a.n == 0) return LP_OK;
    if (!src || !out || !fa32) return LP_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    // LP_REMAP_TMA = 1: the TMA-staged kernel (lp_remap_tma.cu) for float32 / uint8 RGB images
    static int use_tma = -1;
    if (use_tma < 0) {
        const char *e = getenv("LP_REMAP_TMA");
        use_tma = e ? atoi(e) : LP_REMAP_DEFAULT_TMA;
    }
    if (use_tma > 0) {
        const int t = lp_remap_try_tma(a, cam, src_dtype, rows, st);
        if (t != 0) return t > 0 ? LP_OK : t;
    }
    if (src_dtype == LP_DTYPE_F32 && channels == 3 && sampling == LP_SAMPLE_NEAREST && cam.width % 4 == 0 &&
        (long long)cam.height * cam.width * 3 < 0x7fffffffLL &&
        ((uintptr_t)out % 16) == 0 && ((uintptr_t)fa32 % 16) == 0 && (!w16 || ((uintptr_t)w16 % 8) == 0)) {
        const long long quads = a.n / 4;                 // width % 4 == 0 -> n % 4 == 0
        const long long blocks = (quads + LP_REMAP4_BLOCK - 1) / LP_REMAP4_BLOCK;
        if (blocks > 0x7fffffffLL) return LP_ERR_UNSUPPORTED;
        // LP_REMAP_QUADS = 1 | 2 quads per thread (tuning knob); 2 needs width % 8 == 0
        static int quads_per_thread = 0;
        if (!quads_per_thread) {
            const char *e = getenv("LP_REMAP_QUADS");
            const int v = e ? atoi(e) : 0;
            quads_per_thread = (v == 1 || v == 2) ? v : LP_REMAP4_DEFAULT_QUADS;
        }
        const int qpt = (quads_per_thread == 2 && cam.width % 8 == 0) ? 2 : 1;
        const long long threads = (quads + qpt - 1) / qpt;
        const long long nblocks = (threads + LP_REMAP4_BLOCK - 1) / LP_REMAP4_BLOCK;
        if (qpt == 2) lp_remap_f32rgb_x4_kernel<8, 2><<<(unsigned)nblocks, LP_REMAP4_BLOCK, 0, st>>>(a, cam);
        else lp_remap_f32rgb_x4_kernel<12, 1><<<(unsigned)nblocks, LP_REMAP4_BLOCK, 0, st>>>(a, cam);
        return lp_check_launch();
    }
    const void *fn;
    switch (src_dtype) {
    case LP_DTYPE_U8: fn = (const void *)lp_remap_kernel<unsigned char>; break;
    case LP_DTYPE_F32: fn = (const void *)lp_remap_kernel<float>; break;
    case LP_DTYPE_F64: fn = (const void *)lp_remap_kernel<double>; break;
    default: return LP_ERR_INVALID_ARG;
    }
    int grid = 0;
    rc = lp_grid_for(fn, 256, a.n, &grid);
    if (rc != LP_OK) return rc;
    switch (src_dtype) {
    case LP_DTYPE_U8: lp_remap_kernel<unsigned char><<<grid, 256, 0, st>>>(a, cam); break;
    case LP_DTYPE_F32: lp_remap_kernel<float><<<grid, 256, 0, st>>>(a, cam); break;
    default: lp_remap_kernel<double><<<grid, 256, 0, st>>>(a, cam); break;
    }
    return lp_check_launch();
}
