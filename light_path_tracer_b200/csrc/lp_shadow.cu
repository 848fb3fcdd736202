// lp_shadow.cu — kernel (3): analytic shadow classification (black_hole_shadow.py:7-37)
// and the frame reductions over finished lookups (image_lens.py:319-337, :178),
// both built on warp-level primitives.
#include "lp_internal.cuh"

// One CTA handles a tile of x-columns; the per-axis viewing-angle cosines only depend on
// one pixel coordinate each, so they are evaluated once per row/column into shared
// memory (width + height transcendental pairs instead of width*height).
// image[i*height + j], i = x, j = y  (the reference fills image[i, j], shape (width, height)).
#define SH_TILE 32
__global__ void __launch_bounds__(256)
lp_shadow_kernel(int width, int height, double tan_half, double alpha_crit,
                 double *__restrict__ image, unsigned long long *n_shadow)
{
    __shared__ double cx[SH_TILE];
    extern __shared__ double cy[];               // height entries
    const int i0 = blockIdx.x * SH_TILE;
    const double hw = width / 2.0, hh = height / 2.0;
    for (int t = threadIdx.x; t < SH_TILE; t += blockDim.x) {
        const int i = i0 + t;
        // pixel_to_viewing_angle: arctan(((i - n/2)/(n/2)) * tan(fov/2))
        const double iu = __ddiv_rn(sub_((double)i, hw), hw);
        cx[t] = cos(atan(mul_(iu, tan_half)));
    }
    for (int j = threadIdx.x; j < height; j += blockDim.x) {
        const double ju = __ddiv_rn(sub_((double)j, hh), hh);
        cy[j] = cos(atan(mul_(ju, tan_half)));
    }
    __syncthreads();
    unsigned int mine = 0;
    const int ni = min(SH_TILE, width - i0);
    const long long total = (long long)ni * height;
    for (long long e = threadIdx.x; e < total; e += blockDim.x) {
        const int t = (int)(e / height), j = (int)(e % height);
        const double alpha = acos(mul_(cx[t], cy[j]));          // black_hole_shadow.py:36
        const bool dark = alpha < alpha_crit;                   // black_hole_shadow.py:12-15
        image[(long long)(i0 + t) * height + j] = dark ? 0.0 : 1.0;
        mine += dark ? 1u : 0u;
    }
    if (n_shadow) {
        for (int off = 16; off > 0; off >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, off);
        __shared__ unsigned int blk;
        if (threadIdx.x == 0) blk = 0;
        __syncthreads();
        if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&blk, mine);
        __syncthreads();
        if (threadIdx.x == 0 && blk) atomicAdd(n_shadow, (unsigned long long)blk);
    }
}

extern "C" int lp_shadow_classify(int32_t width, int32_t height, double fov, double alpha_crit,
                                  double *image, uint64_t *n_shadow, void *stream)
{
    if (width < 0 || height < 0) return LP_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (n_shadow && cudaMemsetAsync(n_shadow, 0, sizeof(uint64_t), st) != cudaSuccess) { cudaGetLastError(); return LP_ERR_CUDA; }
    if (width == 0 || height == 0) return LP_OK;
    if (!image) return LP_ERR_INVALID_ARG;
    const size_t smem = (size_t)height * sizeof(double);
    if (smem > 200 * 1024) return LP_ERR_UNSUPPORTED;
    if (smem > 48 * 1024 &&
        cudaFuncSetAttribute((const void *)lp_shadow_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        cudaGetLastError();
        return LP_ERR_CUDA;
    }
    const int grid = (width + SH_TILE - 1) / SH_TILE;
    lp_shadow_kernel<<<grid, 256, smem, st>>>(width, height, tan(fov / 2), alpha_crit, image,
                                              (unsigned long long *)n_shadow);
    return lp_check_launch();
}

// ---------------------------------------------------------------------------
// frame statistics
// ---------------------------------------------------------------------------
__global__ void lp_stats_reset_kernel(lp_frame_stats *s)
{
    s->n_rays = s->n_escaped = s->n_captured = s->n_invalid = s->n_winding = 0;
    s->sum_steps = s->sum_warp_steps = 0;
    s->max_steps = s->max_winding = 0;
    s->min_final_alpha = __longlong_as_double(0x7ff0000000000000LL);   // +inf
    s->max_final_alpha = 0.0;
}

extern "C" int lp_frame_stats_reset(lp_frame_stats *stats, void *stream)
{
    if (!stats) return LP_ERR_INVALID_ARG;
    lp_stats_reset_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(stats);
    return lp_check_launch();
}

__global__ void __launch_bounds__(256)
lp_stats_reduce_kernel(const float *__restrict__ fa32, const unsigned short *__restrict__ w16,
                       const int8_t *__restrict__ status, const int32_t *__restrict__ steps,
                       long long n, lp_frame_stats *g)
{
    StatAcc acc;
    acc.init();
    unsigned long long n_mine = 0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long base = (long long)blockIdx.x * blockDim.x; base < n; base += stride) {
        const long long i = base + threadIdx.x;
        const bool live = i < n;
        RayResult r;
        r.status = 0; r.steps = 0; r.nh = 0; r.fa = 0.0;
        if (live) {
            const float f = __ldg(fa32 + i);
            r.fa = (double)f;
            r.nh = w16 ? (long long)__ldg(w16 + i) : 0;
            r.steps = steps ? __ldg(steps + i) : 0;
            // without a status array a finite final_alpha means escaped (image_lens.py:319)
            // and everything else counts as captured
            r.status = status ? (int)__ldg(status + i) : (isfinite(f) ? 1 : -1);
            n_mine++;
        }
        acc.add(r, live);
    }
    lp_stats_flush(acc, n_mine, g);
}

extern "C" int lp_frame_stats_reduce(const float *fa32, const uint16_t *w16,
                                     const int8_t *status, const int32_t *steps, int64_t n,
                                     lp_frame_stats *stats, void *stream)
{
    if (n < 0 || !stats) return LP_ERR_INVALID_ARG;
    if (n == 0) return LP_OK;
    if (!fa32) return LP_ERR_INVALID_ARG;
    int grid = 0;
    int rc = lp_grid_for((const void *)lp_stats_reduce_kernel, 256, n, &grid);
    if (rc != LP_OK) return rc;
    lp_stats_reduce_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(fa32, w16, status, steps, n, stats);
    return lp_check_launch();
}
