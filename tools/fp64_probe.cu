// fp64_probe.cu — stand-alone probe of the B200 FP64 pipe for the Binet RK4 loop (no torch):
//   (1) dependent-DFMA issue latency (one warp, one chain, clock64),
//   (2) FP64-pipe utilisation of the FMA-contracted RK4 loop of lp_internal.cuh as a function of
//       resident warps per SM sub-partition and of independent rays per thread (ILP), with the
//       4-steps-per-trip band test of binet_trace_fast<FUSED, 4>.
// Utilisation = FP64 warp instructions x 2 cycles / (elapsed cycles x 592 sub-partitions), SM clock
// taken as 1.965 GHz (the bench's NVML samples sit there under this load).
//   nvcc -gencode arch=compute_100a,code=sm_100a -I include -I light_path_tracer_b200/csrc \
//        -o tools/fp64_probe tools/fp64_probe.cu ; tools/fp64_probe
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include "lp_internal.cuh"

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e_), __LINE__); exit(1); } } while (0)

__global__ void lat_kernel(double *out, long long *cyc, int n)
{
    double a = 1.0 + threadIdx.x * 1e-9;
    const double m = 0.9999999, b = 1e-8;
    const long long t0 = clock64();
#pragma unroll 16
    for (int i = 0; i < n; ++i) a = fma(a, m, b);
    const long long t1 = clock64();
    out[threadIdx.x] = a;
    if (threadIdx.x == 0) *cyc = t1 - t0;
}

// ILP independent rays per thread, `trips` trips of 4 RK4 steps each, band test on the high words
template <int ILP>
__global__ void __launch_bounds__(128) rk4_kernel(double *out, int trips, double M3, double h, unsigned lo_hi, unsigned span)
{
    extern __shared__ unsigned char pad[];
    const double hh = 0.5 * h, h6 = h / 6.0;
    double u[ILP], w[ILP];
#pragma unroll
    for (int j = 0; j < ILP; ++j) { u[j] = 0.01 + 1e-6 * threadIdx.x + 1e-4 * j; w[j] = 1e-4; }
    int done = 0;
#pragma unroll 1
    for (int t = 0; t < trips; ++t) {
        unsigned worst = 0;
#pragma unroll
        for (int j = 0; j < ILP; ++j) {
            double u1, w1, u2, w2, u3, w3, u4, w4;
            rk4_step<true>(u[j], w[j], M3, h, hh, h6, u1, w1);
            rk4_step<true>(u1, w1, M3, h, hh, h6, u2, w2);
            rk4_step<true>(u2, w2, M3, h, hh, h6, u3, w3);
            rk4_step<true>(u3, w3, M3, h, hh, h6, u4, w4);
            const unsigned t1 = (unsigned)__double2hiint(u1) - lo_hi, t2 = (unsigned)__double2hiint(u2) - lo_hi;
            const unsigned t3 = (unsigned)__double2hiint(u3) - lo_hi, t4 = (unsigned)__double2hiint(u4) - lo_hi;
            worst = max(worst, max(max(t1, t2), max(t3, t4)));
            u[j] = u4; w[j] = w4;
        }
        if (worst >= span) { done = t + 1; break; }
    }
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < ILP; ++j) s += u[j] + w[j];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s + done + (pad[0] & 0);
}

template <int ILP>
static void run(int wps, int trips, double *d_out)
{
    // one 128-thread CTA = one warp per sub-partition; `wps` resident CTAs per SM through dynamic smem
    int smem = (220 * 1024) / wps - 1024;
    if (smem > 200 * 1024) smem = 200 * 1024;
    CK(cudaFuncSetAttribute(rk4_kernel<ILP>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, rk4_kernel<ILP>, 128, smem));
    const int waves = 6;
    const int grid = 148 * occ * waves;
    // u stays ~0.01 (far inside the band) for any trip count: a weak-field circular-ish orbit
    const double M3 = 3.0, h = 1e-5;
    const unsigned lo_hi = 0x3f000000u, span = 0x00f00000u;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        CK(cudaEventRecord(e0));
        rk4_kernel<ILP><<<grid, 128, smem>>>(d_out, trips, M3, h, lo_hi, span);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
        if (rep && ms < best) best = ms;
    }
    const double fp64_inst = (double)grid * 4.0 * trips * 4.0 * 18.0 * ILP;   // warp instructions
    const double cycles = best * 1e-3 * 1.965e9;
    printf("ILP %d  warps/SMSP %2d (occ %2d)  trips %d  %.3f ms  FP64 pipe utilisation %.3f\n", ILP, wps, occ, trips, best,
           fp64_inst * 2.0 / (cycles * 592.0));
    fflush(stdout);
}

int main()
{
    double *d_out; long long *d_cyc;
    CK(cudaMalloc(&d_out, (size_t)148 * 64 * 8 * 128 * sizeof(double)));
    CK(cudaMalloc(&d_cyc, 8));
    for (int rep = 0; rep < 2; ++rep) {
        lat_kernel<<<1, 32>>>(d_out, d_cyc, 4096);
        CK(cudaDeviceSynchronize());
    }
    long long cyc; CK(cudaMemcpy(&cyc, d_cyc, 8, cudaMemcpyDeviceToHost));
    printf("dependent DFMA chain: %.2f cycles per instruction\n", (double)cyc / 4096.0);
    const int trips = 400;
    for (int wps : {1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 16}) run<1>(wps, trips, d_out);
    for (int wps : {1, 2, 3, 4, 5, 6, 8}) run<2>(wps, trips, d_out);
    for (int wps : {1, 2, 3, 4}) run<3>(wps, trips, d_out);
    return 0;
}
