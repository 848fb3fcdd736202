// lp_remap.cuh — per-pixel device code of the remap (shared by the stand-alone remap
// kernel and the fully fused frame kernel).
#pragma once
#include "lp_internal.cuh"

// WINDING_COLORS (image_lens.py:287-293) as float32, and WINDING_COLORS @ luma
// (image_lens.py:330-331) evaluated in float32 by numpy.
static __constant__ float c_wind_rgb[5][3] = {
    {0.0f, 0.2f, 1.0f}, {0.0f, 0.7f, 1.0f}, {0.0f, 1.0f, 0.4f}, {1.0f, 1.0f, 0.0f}, {1.0f, 0.4f, 0.0f}};
static __constant__ float c_wind_luma[5] = {
    0x1.d9e84p-3f, 0x1.0cbfb2p-1f, 0x1.43e426p-1f, 0x1.c5a1ccp-1f, 0x1.114e3cp-1f};

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ unsigned char from_f32<unsigned char>(float v) { return (unsigned char)v; }  // C cast, like numpy's assignment
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ double from_f32<double>(float v) { return (double)v; }

// A colour constant (winding colours, magenta) in the image's value range.  scale is 1 except
// for LP_DTYPE_U8_UNIT images, whose bytes stand for float32 value/255 (image_lens.py:448-450):
// there the constant c is stored as the byte trunc(c * 255), matplotlib's float -> 8-bit rule.
template <typename T> __device__ __forceinline__ T colour(float v, float scale) { return from_f32<T>(v); }
template <> __device__ __forceinline__ unsigned char colour<unsigned char>(float v, float scale)
{
    return (unsigned char)__fmul_rn(v, scale);
}

struct RemapArgs {
    const void *src;
    void *out;
    const float *fa32;
    const unsigned short *w16;   // optional
    long long n;                 // pixels in the tile
    int32_t row0;
    int32_t channels;
    int32_t loop_around;
    int32_t sampling;
    // vector (staged) stores of the frame kernels; each kernel's launcher decides it:
    //   lp_render_kernel: LP_RENDER_STAGED_STORES, RGB float32 / 8-bit, every run of a warp tile contiguous in the
    //     output and the output 16-byte aligned;
    //   lp_render_mirror_kernel: LP_RENDER_STAGED_STORES, RGB float32 / 8-bit, the output aligned to its elements;
    //   lp_render_repack_kernel: a chunk's 32-pixel batches contiguous in the output, the output 16-byte aligned.
    // The stand-alone remap kernel does not read it (0).
    int32_t vec_ok;
    float u8_scale;              // 255 for LP_DTYPE_U8_UNIT images, else 1
    int32_t fast3;               // RGB, nearest sampling, H*W*3 < 2^31: 32-bit index arithmetic
};

// python `a % n` for n > 0
__device__ __forceinline__ long long pymod(long long a, long long n)
{
    long long m = a % n;
    return m < 0 ? m + n : m;
}

// ---------------------------------------------------------------------------
// Branch-free fp64 helpers for the remap.  What has to match the reference there is the
// INTEGER source index rint(px), rint(py) (image_lens.py:367-375): the continuous coordinate
// only needs ~1e-12 relative accuracy (a tie would have to be that close to a half-integer to
// flip), so these trade the library routines' last-ulp guarantees and special-case branches
// (which keep ptxas from interleaving neighbouring pixels' dependency chains) for straight-line
// code accurate to a few ulp.
// ---------------------------------------------------------------------------
// Source direction of an escaped pixel -> pinhole plane coordinates (image_lens.py:310-352), in two parts:
// source_dir_xy forms the direction (front = src_vz > 1e-12, and (sx, sy) / sz), source_px the continuous
// source pixel coordinates.  The mirror-image frame kernel forms the direction once for all images of a ray.
//
// The reference normalises the pixel ray v, takes theta = arctan2(v.e_x, v.e_y) and then
// sin(theta), cos(theta).  theta is invariant under scaling of v, and sin/cos of an arctan2
// are the normalised components themselves, so here (st, ct) = (A, B)/hypot(A, B) with
// A, B the dot products of the UN-normalised ray (x_cam, y_cam, 1): no arctan2, no second
// sincos, no normalisation of v.  Straight-line code (see the helpers above).
//
// DIR (the fused frame kernel): the tracer has just formed c = cos(fa), s = sin(fa) of the fp64 final_alpha
// fa (RayResult::cf, sf, fa).  The lookup holds fa32 = float32(fa), so the angle the reference takes the
// sine and cosine of is fa + d with d = fa32 - fa, |d| <= 3e-8 fa: cos(fa32) = c - s d, sin(fa32) = s + c d
// up to d^2 / 2 < 5e-16 — far inside the 1e-12 the source index needs — instead of a second sincos.
struct SrcDir {
    double qx, qy;               // pinhole-plane direction of the source: (sx, sy) / sz
    bool front;                  // sz > 1e-12
};

template <bool DIR = false>
__device__ __forceinline__ SrcDir source_dir_xy(const CamConsts &cam, double xc, double yc, float fa32,
                                                double fa64 = 0.0, double cfa = 0.0, double sfa = 0.0)
{
    const double A = fma(xc, cam.ex0, fma(yc, cam.ex1, cam.ex2));
    const double B = fma(xc, cam.ey0, fma(yc, cam.ey1, cam.ey2));
    const double n2 = fma(A, A, B * B);
    const bool on_axis = !(n2 > 1e-300);                    // arctan2(0, 0) = 0
    const double inv = fast_rsqrt(on_axis ? 1.0 : n2);
    const double st = on_axis ? 0.0 : A * inv, ct = on_axis ? 1.0 : B * inv;
    double sf, cf;
    if (DIR) {
        const double d = (double)fa32 - fa64;
        cf = fma(-sfa, d, cfa);
        sf = fma(cfa, d, sfa);
    } else {
        sincos_moderate((double)fa32, sf, cf);              // image_lens.py:340-346
    }
    const double tx = fma(st, cam.ex0, ct * cam.ey0);
    const double ty = fma(st, cam.ex1, ct * cam.ey1);
    const double tz = fma(st, cam.ex2, ct * cam.ey2);
    const double sx = fma(cf, cam.d0, sf * tx);
    const double sy = fma(cf, cam.d1, sf * ty);
    const double sz = fma(cf, cam.d2, sf * tz);
    SrcDir s;
    s.front = sz > 1e-12;
    const double isz = fast_rcp(s.front ? sz : 1.0);
    s.qx = sx * isz;
    s.qy = sy * isz;
    return s;
}

// the per-pixel part: continuous source pixel coordinates of a direction
__device__ __forceinline__ void source_px(const CamConsts &cam, const SrcDir &s, double &px, double &py)
{
    // behind the camera: zeros * f + n/2 (image_lens.py:356-361)
    px = s.front ? fma(s.qx, cam.fx, cam.half_w) : cam.half_w;    // image_lens.py:374
    py = s.front ? fma(s.qy, cam.fy, cam.half_h) : cam.half_h;
}

template <bool DIR = false>
__device__ __forceinline__ bool source_coords_xy(const CamConsts &cam, double xc, double yc, float fa32,
                                                 double &px, double &py,
                                                 double fa64 = 0.0, double cfa = 0.0, double sfa = 0.0)
{
    const SrcDir s = source_dir_xy<DIR>(cam, xc, yc, fa32, fa64, cfa, sfa);
    source_px(cam, s, px, py);
    return s.front;
}

// fast3 layout (see remap_pixel_dir): the element offset o of the source pixel, or false when the pixel
// is out of frame (magenta).  cvt.rni.s32.f64 rounds half to even like np.rint and saturates, so a far
// out-of-frame coordinate stays out of frame (same as lp_remap_f32rgb_x4_kernel, pixel-identical).
__device__ __forceinline__ bool fast3_source(const RemapArgs &a, const CamConsts &cam, const SrcDir &s, int &o)
{
    double px, py;
    source_px(cam, s, px, py);
    const int H = cam.height, W = cam.width;
    int ix = __double2int_rn(px), iy = __double2int_rn(py);
    bool ok;
    if (a.loop_around) {
        ix %= W; ix += (ix < 0) ? W : 0;
        iy %= H; iy += (iy < 0) ? H : 0;
        ok = true;
    } else {
        ok = s.front && (unsigned)ix < (unsigned)W && (unsigned)iy < (unsigned)H;
    }
    o = (iy * W + ix) * 3;
    return ok;
}

__device__ __forceinline__ bool source_coords(const CamConsts &cam, int row, int col, float fa32,
                                              double &px, double &py)
{
    return source_coords_xy(cam, cam_x(cam, col), cam_y(cam, row), fa32, px, py);
}

// dir(): the pixel's SrcDir, formed only for escaped pixels that are not winding-coloured
template <typename T, typename Dir>
__device__ __forceinline__ void remap_pixel_dir(const RemapArgs &a, const CamConsts &cam, T *__restrict__ dst,
                                                float fa32, unsigned wnd, Dir dir)
{   // dst: where this pixel's `channels` values go (global memory, or a staging slot)
    const int C = a.channels;
    const T *__restrict__ src = (const T *)a.src;
    if (a.fast3) {
        // the common layout — three channels, nearest sampling, an image whose element count fits
        // 31 bits — with the decisions of the general code below on 32-bit integers (fast3_source)
        if (!isfinite(fa32)) { dst[0] = (T)0; dst[1] = (T)0; dst[2] = (T)0; return; }
        if (fa32 > LP_HALF_PI_F32) {
            const unsigned k = wnd > 4u ? 4u : wnd;
            dst[0] = colour<T>(c_wind_rgb[k][0], a.u8_scale); dst[1] = colour<T>(c_wind_rgb[k][1], a.u8_scale);
            dst[2] = colour<T>(c_wind_rgb[k][2], a.u8_scale);
            return;
        }
        int o;
        if (!fast3_source(a, cam, dir(), o)) {
            const T one = colour<T>(1.0f, a.u8_scale);
            dst[0] = one; dst[1] = (T)0; dst[2] = one;
            return;
        }
        const T *s = src + o;
        dst[0] = __ldg(s); dst[1] = __ldg(s + 1); dst[2] = __ldg(s + 2);
        return;
    }
    if (!isfinite(fa32)) {                                   // captured / invalid: zeros_like
        for (int ch = 0; ch < C; ++ch) dst[ch] = (T)0;
        return;
    }
    if (fa32 > LP_HALF_PI_F32) {                             // winding false colour, image_lens.py:322-333
        const unsigned k = wnd > 4u ? 4u : wnd;
        if (C == 1) {
            dst[0] = colour<T>(c_wind_luma[k], a.u8_scale);
        } else {
            for (int ch = 0; ch < C; ++ch) dst[ch] = (ch < 3) ? colour<T>(c_wind_rgb[k][ch], a.u8_scale) : (T)0;
        }
        return;
    }
    const SrcDir sd = dir();
    const bool front = sd.front;
    double px, py;
    source_px(cam, sd, px, py);
    const long long H = cam.height, W = cam.width;
    long long ix = (long long)rint(px), iy = (long long)rint(py);   // np.rint -> intp
    bool ok;
    if (a.loop_around) {                                     // image_lens.py:354-365
        ix = pymod(ix, W);
        iy = pymod(iy, H);
        ok = true;
    } else {                                                 // image_lens.py:367-379
        ok = front && iy >= 0 && iy < H && ix >= 0 && ix < W;
    }
    if (!ok) {                                               // magenta, image_lens.py:381-393
        const T one = colour<T>(1.0f, a.u8_scale);
        if (C == 1) dst[0] = one;
        else for (int ch = 0; ch < C; ++ch) dst[ch] = (ch == 0 || ch == 2) ? one : (T)0;
        return;
    }
    if (a.sampling == LP_SAMPLE_NEAREST) {
        const T *s = src + (iy * W + ix) * C;
        for (int ch = 0; ch < C; ++ch) dst[ch] = __ldg(s + ch);
        return;
    }
    // bilinear extension: same in/out-of-frame decision as nearest, 4-tap blend around the
    // continuous coordinate, taps clamped (or wrapped when loop_around) at the border.
    const double fxp = floor(px), fyp = floor(py);
    const double tx = px - fxp, ty = py - fyp;
    long long x0 = (long long)fxp, y0 = (long long)fyp, x1 = x0 + 1, y1 = y0 + 1;
    if (a.loop_around) {
        x0 = pymod(x0, W); x1 = pymod(x1, W); y0 = pymod(y0, H); y1 = pymod(y1, H);
    } else {
        x0 = min(max(x0, 0ll), W - 1); x1 = min(max(x1, 0ll), W - 1);
        y0 = min(max(y0, 0ll), H - 1); y1 = min(max(y1, 0ll), H - 1);
    }
    const double w00 = (1.0 - tx) * (1.0 - ty), w01 = tx * (1.0 - ty), w10 = (1.0 - tx) * ty, w11 = tx * ty;
    for (int ch = 0; ch < C; ++ch) {
        const double v = w00 * (double)__ldg(src + (y0 * W + x0) * C + ch)
                       + w01 * (double)__ldg(src + (y0 * W + x1) * C + ch)
                       + w10 * (double)__ldg(src + (y1 * W + x0) * C + ch)
                       + w11 * (double)__ldg(src + (y1 * W + x1) * C + ch);
        if (sizeof(T) == 1) dst[ch] = (T)(int)rint(v);
        else dst[ch] = (T)v;
    }
}

// xc, yc: the pixel's camera-plane coordinates cam_x(col), cam_y(row); DIR: see source_coords_xy
template <typename T, bool DIR = false>
__device__ __forceinline__ void remap_pixel_xy(const RemapArgs &a, const CamConsts &cam, T *__restrict__ dst,
                                               double xc, double yc, float fa32, unsigned wnd,
                                               double fa64 = 0.0, double cfa = 0.0, double sfa = 0.0)
{
    remap_pixel_dir<T>(a, cam, dst, fa32, wnd,
                       [&] { return source_dir_xy<DIR>(cam, xc, yc, fa32, fa64, cfa, sfa); });
}

template <typename T>
__device__ __forceinline__ void remap_pixel(const RemapArgs &a, const CamConsts &cam, T *__restrict__ dst,
                                            int row, int col, float fa32, unsigned wnd)
{
    remap_pixel_xy<T>(a, cam, dst, cam_x(cam, col), cam_y(cam, row), fa32, wnd);
}
