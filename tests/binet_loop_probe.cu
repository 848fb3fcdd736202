// tests/binet_loop_probe.cu — launchers of the Binet RK4 loop's variants (binet_trace, lp_internal.cuh) for
// tests/test_gpu_binet_loop.py: the literal loop (binet_trace_generic), the fast loop with two or four RK4 steps
// per trip (binet_trace_fast), each in strict and FMA arithmetic, the plain per-ray composition that
// LP_TRACE_HYBRID must equal, and the loop variable after every full step of the literal loop.
//
// Test infrastructure: not part of liblightpath.so and not part of the C ABI.  The test compiles it with
// light_path_tracer_b200.build.NVCC_FLAGS (the library's -fmad=false arithmetic) into a shared object that
// links against liblightpath.so for lp_make_binet_consts, the fast-path preconditions and the hybrid rule.
// Every launcher takes the configuration (M, R_S, r_obs, phi_max, h_max), builds BinetConsts with
// lp_make_binet_consts exactly as the production launchers do, takes device pointers and a stream, and
// returns 0, a negative LP_ERR_* or a cudaError_t.
#include <cstdint>
#include <cstring>
#include "lp_trace.cuh"

namespace {

constexpr int kBlock = 128;
constexpr long long kNaNBits = 0x7ff8000000000000LL;

struct RayOut {
    double *fa;         // final_alpha, NaN unless status == 1 (as the tracer kernels store it)
    long long *nh;      // n_half_orbits
    int8_t *status;
    int32_t *steps;
};

__device__ __forceinline__ void store(const RayOut &o, long long i, const RayResult &r)
{
    o.fa[i] = (r.status == 1) ? r.fa : __longlong_as_double(kNaNBits);
    o.nh[i] = r.nh;
    o.status[i] = (int8_t)r.status;
    o.steps[i] = r.steps;
}

template <bool FUSED, bool FAST, int TRIP>
__global__ void trace_kernel(const BinetConsts c, const double *__restrict__ alphas, long long n, RayOut o)
{
    const LoopRegs L = load_loop_regs<FUSED>(c);
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    RayResult r;
    binet_trace<FUSED, FAST, TRIP>(c, L, alphas[i], r);
    store(o, i, r);
}

// LP_TRACE_HYBRID per ray, written plainly: the FMA literal loop, then the strict literal loop where the rule says so
__global__ void hybrid_kernel(const BinetConsts c, const double *__restrict__ alphas, long long n, int retrace_steps,
                              int retrace_steps_small, float retrace_h, float retrace_off, RayOut o)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    RayResult r;
    binet_trace<true, false>(c, load_loop_regs<true>(c), alphas[i], r);
    if (hybrid_needs_retrace(r, retrace_steps, retrace_steps_small, retrace_h, retrace_off))
        binet_trace<false, false>(c, load_loop_regs<false>(c), alphas[i], r);
    store(o, i, r);
}

// binet_trace_generic's loop, recording the loop variable (u, or v = 3M u for FUSED) after each of the first
// max_steps full steps (NaN after the exit); orbit_status: 0 invalid, -1 / 1 a crossing (in a full or a
// shortened step), 2 phi_max reached.  steps: as binet_trace reports it.
template <bool FUSED>
__global__ void history_kernel(const BinetConsts c, const double *__restrict__ alphas, long long n, int max_steps,
                               double *hist, int8_t *orbit_status, int32_t *steps_out)
{
    const LoopRegs L = load_loop_regs<FUSED>(c);
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double *h = hist + i * (long long)max_steps;
    double u, w;
    int status = 0, k = 0, steps = 0;
    if (binet_init<FUSED>(c, alphas[i], u, w)) {
        binet_scale_in<FUSED>(c, u, w);
        const double uc = band_hi<FUSED>(c), ue = band_lo<FUSED>(c);
        bool ge_c = (u >= uc), le_e = (u <= ue);
        status = 2;
        for (; k < c.n_full; ++k) {
            const double up = u, wp = w;
            rk4_full_step<FUSED>(L, up, wp, u, w);
            if (k < max_steps) h[k] = u;
            const bool ge2 = (u >= uc), le2 = (u <= ue);
            if (!ge_c && ge2) { status = -1; break; }
            if (!le_e && le2) { status = 1; break; }
            ge_c = ge2; le_e = le2;
        }
        steps = (status == 2) ? c.n_full : k + 1;
        if (status != 2) ++k;
        for (int j = 0; status == 2 && j < c.n_tail; ++j) {
            const double hj = c.tail_h[j];
            const double up = u, wp = w;
            rk4_step<FUSED>(up, wp, L.M3, hj, mul_(0.5, hj), __ddiv_rn(hj, 6.0), u, w);
            steps++;
            const bool ge2 = (u >= uc), le2 = (u <= ue);
            if (!ge_c && ge2) status = -1;
            else if (!le_e && le2) status = 1;
            ge_c = ge2; le_e = le2;
        }
    }
    for (; k < max_steps; ++k) h[k] = __longlong_as_double(kNaNBits);
    orbit_status[i] = (int8_t)status;
    steps_out[i] = steps;
}

unsigned grid_for(long long n) { return (unsigned)((n + kBlock - 1) / kBlock); }

int finish() { return (int)cudaGetLastError(); }

}  // namespace

// The configuration's constants: ints = {n_full, n_tail, phi_shift, lp_binet_fast_ok, lp_binet_fast_ok_fused,
// scaled_ok, valid}, hi = the high words of {uc, ue, vc, ve}.  Host only.
extern "C" int probe_binet_consts(double M, double R_S, double r_obs, double phi_max, double h_max, int32_t *ints,
                                  uint32_t *hi)
{
    BinetConsts c;
    const int rc = lp_make_binet_consts(M, R_S, r_obs, phi_max, h_max, &c);
    if (rc != LP_OK) return rc;
    const int32_t v[7] = {c.n_full, c.n_tail, c.phi_shift, lp_binet_fast_ok(&c), lp_binet_fast_ok_fused(&c), c.scaled_ok,
                          c.valid};
    for (int j = 0; j < 7; ++j) ints[j] = v[j];
    const double b[4] = {c.uc, c.ue, c.vc, c.ve};
    for (int j = 0; j < 4; ++j) {
        uint64_t bits;
        memcpy(&bits, &b[j], 8);
        hi[j] = (uint32_t)(bits >> 32);
    }
    return LP_OK;
}

// binet_trace<FUSED, FAST, TRIP> per ray.  variant = 3 * fused + {0: literal loop, 1: fast, 2 steps per trip,
// 2: fast, 4 steps per trip}.  A fast variant whose precondition fails (lp_binet_fast_ok, or
// lp_binet_fast_ok_fused for the FMA loop), and the FMA loop without a usable scale, return
// LP_ERR_UNSUPPORTED without a launch.
extern "C" int probe_binet_trace(int variant, double M, double R_S, double r_obs, double phi_max, double h_max,
                                 const double *alphas, long long n, double *fa, long long *nh, int8_t *status,
                                 int32_t *steps, void *stream)
{
    BinetConsts c;
    const int rc = lp_make_binet_consts(M, R_S, r_obs, phi_max, h_max, &c);
    if (rc != LP_OK) return rc;
    if (variant < 0 || variant > 5) return LP_ERR_INVALID_ARG;
    const bool fused = variant >= 3;
    const int kind = variant % 3;
    if (fused && !c.scaled_ok) return LP_ERR_UNSUPPORTED;
    if (kind && !(fused ? lp_binet_fast_ok_fused(&c) : lp_binet_fast_ok(&c))) return LP_ERR_UNSUPPORTED;
    if (n <= 0) return (int)cudaSuccess;
    const RayOut o = {fa, nh, status, steps};
    cudaStream_t s = (cudaStream_t)stream;
    switch (variant) {
    case 0: trace_kernel<false, false, 2><<<grid_for(n), kBlock, 0, s>>>(c, alphas, n, o); break;
    case 1: trace_kernel<false, true, 2><<<grid_for(n), kBlock, 0, s>>>(c, alphas, n, o); break;
    case 2: trace_kernel<false, true, 4><<<grid_for(n), kBlock, 0, s>>>(c, alphas, n, o); break;
    case 3: trace_kernel<true, false, 2><<<grid_for(n), kBlock, 0, s>>>(c, alphas, n, o); break;
    case 4: trace_kernel<true, true, 2><<<grid_for(n), kBlock, 0, s>>>(c, alphas, n, o); break;
    default: trace_kernel<true, true, 4><<<grid_for(n), kBlock, 0, s>>>(c, alphas, n, o); break;
    }
    return finish();
}

// LP_TRACE_HYBRID as a plain composition of the literal loops, with the re-trace rule lp_hybrid_retrace_rule returns,
// narrowed to float as lp_hybrid_rule narrows it.  LP_ERR_UNSUPPORTED without a usable scale.
extern "C" int probe_binet_hybrid(double M, double R_S, double r_obs, double phi_max, double h_max, const double *alphas,
                                  long long n, double *fa, long long *nh, int8_t *status, int32_t *steps, void *stream)
{
    BinetConsts c;
    int rc = lp_make_binet_consts(M, R_S, r_obs, phi_max, h_max, &c);
    if (rc != LP_OK) return rc;
    if (!c.scaled_ok) return LP_ERR_UNSUPPORTED;
    int32_t steps_all = 0, steps_none = 0;
    double offset = 0.0;
    rc = lp_hybrid_retrace_rule(M, r_obs, h_max, &steps_all, &steps_none, &offset, nullptr);
    if (rc != LP_OK) return rc;
    if (n <= 0) return (int)cudaSuccess;
    const RayOut o = {fa, nh, status, steps};
    hybrid_kernel<<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(c, alphas, n, steps_all, steps_none, (float)h_max,
                                                                    (float)offset, o);
    return finish();
}

// The literal loop's variable after each of the first max_steps full steps: hist[i * max_steps + k] after step k + 1
// (u strict, v = 3M u FMA), NaN after the exit; the orbit's status and binet_trace's step count.
extern "C" int probe_binet_history(int fused, double M, double R_S, double r_obs, double phi_max, double h_max,
                                   const double *alphas, long long n, int max_steps, double *hist, int8_t *orbit_status,
                                   int32_t *steps, void *stream)
{
    BinetConsts c;
    const int rc = lp_make_binet_consts(M, R_S, r_obs, phi_max, h_max, &c);
    if (rc != LP_OK) return rc;
    if (fused && !c.scaled_ok) return LP_ERR_UNSUPPORTED;
    if (max_steps < 0) return LP_ERR_INVALID_ARG;
    if (n <= 0) return (int)cudaSuccess;
    cudaStream_t s = (cudaStream_t)stream;
    if (fused) history_kernel<true><<<grid_for(n), kBlock, 0, s>>>(c, alphas, n, max_steps, hist, orbit_status, steps);
    else history_kernel<false><<<grid_for(n), kBlock, 0, s>>>(c, alphas, n, max_steps, hist, orbit_status, steps);
    return finish();
}
