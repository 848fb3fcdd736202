// tests/rk45_rhs_probe.cu — launchers of the generic RK45 integrator's right-hand sides
// (csrc/lp_rk45_rhs.cuh: rk_rhs, rk_rhs_kerr, rk_rhs_eq<SPEC>) over arrays of states, for
// tests/test_gpu_rk45_rhs.py.
//
// Test infrastructure: not part of liblightpath.so and not part of the C ABI.  The test compiles it with
// light_path_tracer_b200.build.NVCC_FLAGS (the library's -fmad=false arithmetic), linked against
// liblightpath.so.  Every launcher takes device pointers, a state count and a stream, and returns 0 or a
// cudaError_t.
//
// Inputs: par[n][5] = (R_S for Schwarzschild or M for Kerr, a, r_floor, p_t, p_phi) and y[n][6] = (t, r,
// theta, phi, p_r, p_theta); outputs d[n][6] and hit[n] (1 where theta hit the cache).  Each thread walks
// `seq` consecutive states with one ThetaCache, initialised as RkSixSystem initialises it (th = NaN), so
// the cache hits and misses as it does in the integrator; seq = 1 makes every evaluation a miss.  The
// equatorial kinds take (t, r, phi, p_r) of y and leave d[2] = d[5] = 0.
#include <climits>
#include <cstdint>
#include "lp_rk45_rhs.cuh"

namespace {

constexpr int kBlock = 128;

// 0: rk_rhs, 1: rk_rhs_kerr, 2: rk_rhs_eq<true>, 3: rk_rhs_eq<false>
template <int KIND>
__global__ void rhs_kernel(const double *__restrict__ par, const double *__restrict__ y, double *d, int32_t *hit,
                           long long n, int seq)
{
    const long long first = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * seq;
    ThetaCache tc;
    tc.th = __longlong_as_double(0x7ff8000000000000LL); tc.s = 1.0; tc.c = 0.0;
    for (int k = 0; k < seq; ++k) {
        const long long i = first + k;
        if (i >= n) return;
        const double *p = par + i * 5;
        double yi[RK_NC], di[RK_NC];
        for (int j = 0; j < RK_NC; ++j) yi[j] = y[i * RK_NC + j];
        hit[i] = (yi[2] == tc.th) ? 1 : 0;
        if (KIND == 0) {
            rk_rhs(p[0], p[2], p[3], p[4], yi, tc, di);
        } else if (KIND == 1) {
            rk_rhs_kerr(p[0], p[1], p[2], p[3], p[4], yi, tc, di);
        } else {
            const double y4[RK_EQ] = {yi[0], yi[1], yi[3], yi[4]};
            double d4[RK_EQ];
            int r_hi_min = INT_MAX;
            rk_rhs_eq<KIND == 2>(p[0], p[2], p[3], p[4], p[4] * p[4], y4, d4, r_hi_min);
            di[0] = d4[0]; di[1] = d4[1]; di[2] = 0.0; di[3] = d4[2]; di[4] = d4[3]; di[5] = 0.0;
        }
        for (int j = 0; j < RK_NC; ++j) d[i * RK_NC + j] = di[j];
    }
}

}  // namespace

extern "C" int probe_rk45_rhs(int kind, const double *par, const double *y, double *d, int32_t *hit, long long n,
                              int seq, void *stream)
{
    if (n <= 0) return (int)cudaSuccess;
    if (seq < 1) return (int)cudaErrorInvalidValue;
    const long long threads = (n + seq - 1) / seq;
    const unsigned grid = (unsigned)((threads + kBlock - 1) / kBlock);
    cudaStream_t s = (cudaStream_t)stream;
    switch (kind) {
    case 0: rhs_kernel<0><<<grid, kBlock, 0, s>>>(par, y, d, hit, n, seq); break;
    case 1: rhs_kernel<1><<<grid, kBlock, 0, s>>>(par, y, d, hit, n, seq); break;
    case 2: rhs_kernel<2><<<grid, kBlock, 0, s>>>(par, y, d, hit, n, seq); break;
    case 3: rhs_kernel<3><<<grid, kBlock, 0, s>>>(par, y, d, hit, n, seq); break;
    default: return (int)cudaErrorInvalidValue;
    }
    return (int)cudaGetLastError();
}
