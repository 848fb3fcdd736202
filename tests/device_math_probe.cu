// tests/device_math_probe.cu — elementwise launchers of the hand-written device math routines
// (csrc/lp_sincr.cuh, lp_internal.cuh, lp_remap.cuh), for tests/test_gpu_device_math.py.
//
// Test infrastructure: not part of liblightpath.so and not part of the C ABI.  The test compiles it with
// light_path_tracer_b200.build.NVCC_FLAGS (the library's -fmad=false arithmetic) into a shared object that
// links against liblightpath.so for lp_make_cam_consts.  Every launcher takes device pointers, an element
// count and a stream, and returns 0 or a cudaError_t (a negative LP_ERR_* for an invalid camera).
#include <cstdint>
#include "lp_internal.cuh"
#include "lp_remap.cuh"

namespace {

constexpr int kBlock = 256;

template <typename Op, typename T>
__global__ void unary_kernel(const double *__restrict__ x, T *__restrict__ y, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = Op::eval(x[i]);
}

template <typename Op, typename T>
int launch_unary(const double *x, T *y, long long n, void *stream)
{
    if (n <= 0) return (int)cudaSuccess;
    unary_kernel<Op, T><<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, (cudaStream_t)stream>>>(x, y, n);
    return (int)cudaGetLastError();
}

struct SinCr { __device__ static double eval(double v) { return lp_sin_cr(v); } };
struct AcosUnit { __device__ static double eval(double v) { return lp_acos_unit(v); } };
struct InvTenthRoot { __device__ static double eval(double v) { return inv_tenth_root(v); } };
struct FastRcp { __device__ static double eval(double v) { return fast_rcp(v); } };
struct FastRsqrt { __device__ static double eval(double v) { return fast_rsqrt(v); } };
struct MidRange { __device__ static int32_t eval(double v) { return mid_range(v) ? 1 : 0; } };
struct HalfOrbits { __device__ static long long eval(double v) { return half_orbits(v); } };
struct HalfOrbitsFast { __device__ static long long eval(double v) { return half_orbits_fast(v); } };
// n_half_orbits as binet_finish forms it for 0 <= phi_f < 1e4: from the quadrant of the sincos reduction
struct HalfOrbitsQuadrant {
    __device__ static long long eval(double v)
    {
        double s, c, rr;
        int q;
        sincos_moderate(v, s, c, &q, &rr);
        return half_orbits_quadrant(v, q, rr);
    }
};

__global__ void sincos_kernel(const double *__restrict__ x, double *s, double *c, int32_t *q, double *r, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double si, ci, ri;
    int qi;
    sincos_moderate(x[i], si, ci, &qi, &ri);
    s[i] = si; c[i] = ci; q[i] = qi; r[i] = ri;
}

template <bool DIR>
__global__ void source_coords_kernel(const CamConsts cam, const double *__restrict__ xc, const double *__restrict__ yc,
                                     const float *__restrict__ fa32, const double *__restrict__ fa64,
                                     const double *__restrict__ cfa, const double *__restrict__ sfa,
                                     double *px, double *py, int32_t *front, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double x, y;
    const bool f = DIR ? source_coords_xy<true>(cam, xc[i], yc[i], fa32[i], x, y, fa64[i], cfa[i], sfa[i])
                       : source_coords_xy<false>(cam, xc[i], yc[i], fa32[i], x, y);
    px[i] = x; py[i] = y; front[i] = f ? 1 : 0;
}

}  // namespace

extern "C" int probe_sin_cr(const double *x, double *y, long long n, void *s) { return launch_unary<SinCr>(x, y, n, s); }
extern "C" int probe_acos_unit(const double *x, double *y, long long n, void *s) { return launch_unary<AcosUnit>(x, y, n, s); }
extern "C" int probe_inv_tenth_root(const double *x, double *y, long long n, void *s) { return launch_unary<InvTenthRoot>(x, y, n, s); }
extern "C" int probe_fast_rcp(const double *x, double *y, long long n, void *s) { return launch_unary<FastRcp>(x, y, n, s); }
extern "C" int probe_fast_rsqrt(const double *x, double *y, long long n, void *s) { return launch_unary<FastRsqrt>(x, y, n, s); }
extern "C" int probe_mid_range(const double *x, int32_t *y, long long n, void *s) { return launch_unary<MidRange>(x, y, n, s); }
extern "C" int probe_half_orbits(const double *x, long long *y, long long n, void *s) { return launch_unary<HalfOrbits>(x, y, n, s); }
extern "C" int probe_half_orbits_fast(const double *x, long long *y, long long n, void *s) { return launch_unary<HalfOrbitsFast>(x, y, n, s); }
extern "C" int probe_half_orbits_quadrant(const double *x, long long *y, long long n, void *s) { return launch_unary<HalfOrbitsQuadrant>(x, y, n, s); }

// s, c and the reduction x = q pi/2 + r
extern "C" int probe_sincos_moderate(const double *x, double *s, double *c, int32_t *q, double *r, long long n,
                                     void *stream)
{
    if (n <= 0) return (int)cudaSuccess;
    sincos_kernel<<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, (cudaStream_t)stream>>>(x, s, c, q, r, n);
    return (int)cudaGetLastError();
}

// source_coords_xy<DIR> on the CamConsts the library builds from *cam (a host pointer), as its frame and remap
// launchers do; fa64, cfa, sfa are read only when dir != 0.  front[i] is the routine's return value.
extern "C" int probe_source_coords(const lp_camera *cam, int dir, const double *xc, const double *yc, const float *fa32,
                                   const double *fa64, const double *cfa, const double *sfa, double *px, double *py,
                                   int32_t *front, long long n, void *stream)
{
    CamConsts cc;
    const int rc = lp_make_cam_consts(cam, &cc);
    if (rc != LP_OK) return rc;
    if (n <= 0) return (int)cudaSuccess;
    const unsigned grid = (unsigned)((n + kBlock - 1) / kBlock);
    if (dir)
        source_coords_kernel<true><<<grid, kBlock, 0, (cudaStream_t)stream>>>(cc, xc, yc, fa32, fa64, cfa, sfa, px, py,
                                                                             front, n);
    else
        source_coords_kernel<false><<<grid, kBlock, 0, (cudaStream_t)stream>>>(cc, xc, yc, fa32, fa64, cfa, sfa, px,
                                                                              py, front, n);
    return (int)cudaGetLastError();
}
