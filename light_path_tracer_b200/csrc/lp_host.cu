// lp_host.cu — host-side pieces of liblightpath: per-configuration constants,
// camera frame, error strings, launch helpers.  No device code here.
#include "lp_internal.cuh"
#include <stdlib.h>
#include <string.h>

extern "C" int lp_abi_version(void) { return LP_ABI_VERSION; }

extern "C" const char *lp_error_string(int code)
{
    switch (code) {
    case LP_OK: return "ok";
    case LP_ERR_INVALID_ARG: return "invalid argument";
    case LP_ERR_CUDA: return "CUDA error (no usable device, or a launch failed)";
    case LP_ERR_UNSUPPORTED: return "unsupported configuration";
    default: return "unknown error";
    }
}

extern "C" int lp_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" int lp_device_props(int32_t *sm_count, int32_t *clock_khz)
{
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return LP_ERR_CUDA; }
    if (sm_count) {
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return LP_ERR_CUDA;
        *sm_count = v;
    }
    if (clock_khz) {
        if (cudaDeviceGetAttribute(&v, cudaDevAttrClockRate, dev) != cudaSuccess) return LP_ERR_CUDA;
        *clock_khz = v;
    }
    return LP_OK;
}

int lp_check_launch(void)
{
    return cudaGetLastError() == cudaSuccess ? LP_OK : LP_ERR_CUDA;
}

// Persistent grid: (resident CTAs per SM) x (SM count) for this kernel / block size, but no more CTAs
// than the n items fill (ceil(n / block)).
int lp_grid_for(const void *kernel, int block, long long n, int *grid_out)
{
    int dev = 0, sms = 0, per_sm = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return LP_ERR_CUDA; }
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) { cudaGetLastError(); return LP_ERR_CUDA; }
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, 0) != cudaSuccess) { cudaGetLastError(); return LP_ERR_CUDA; }
    if (per_sm < 1) per_sm = 1;
    *grid_out = sms * per_sm;
    const long long chunks = (n + block - 1) / block;
    if (chunks < *grid_out) *grid_out = (int)chunks;
    return LP_OK;
}

int lp_launch_ctas(const void *kernel, long long n, long long per_cta, int block, size_t smem, void **args,
                   cudaStream_t stream)
{
    const long long ctas = (n + per_cta - 1) / per_cta;
    if (ctas > 0x7fffffffLL) return LP_ERR_UNSUPPORTED;
    cudaLaunchKernel(kernel, dim3((unsigned)ctas), dim3((unsigned)block), args, smem, stream);
    return lp_check_launch();
}

int lp_env_int(const char *name, int lo, int hi, int dflt)
{
    const char *e = getenv(name);
    const int v = e ? atoi(e) : 0;
    return (v >= lo && v <= hi) ? v : dflt;
}

// metrics.py:51-78 evaluated once per configuration instead of once per ray.  Every
// expression keeps the reference's operation order; this translation unit is compiled
// with host FMA contraction disabled.
// x / d == div_by(x, d, RN(1/d)) (lp_internal.cuh) for every x whose quotient is normal: d normal and far
// from the exponent limits, significand not all ones (the one case Markstein's theorem excludes).
static int div_const_exact(double d)
{
    if (!(d > 1e-100) || !(d < 1e100)) return 0;
    unsigned long long bits;
    memcpy(&bits, &d, 8);
    return (bits & 0xfffffffffffffull) != 0xfffffffffffffull;
}

int lp_make_binet_consts(double M, double R_S, double r_obs, double phi_max, double h_max,
                         BinetConsts *c)
{
    memset(c, 0, sizeof(*c));
    c->r_obs = r_obs;
    c->R_S = R_S;
    const double f0 = 1.0 - R_S / r_obs;
    c->valid = (f0 <= 0.0) ? 0 : 1;            // NaN f0 stays "valid", as in the reference
    c->sqrt_f0 = sqrt(f0);
    const double u = 1.0 / r_obs;
    c->u0 = u;
    c->u0sq = u * u;
    c->c3 = 2.0 * M * u * u * u;
    c->M3 = 3.0 * M;
    c->h = h_max;
    c->hh = 0.5 * h_max;
    c->h6 = h_max / 6.0;
    c->uc = 1.0 / (R_S * 1.01);
    c->ue = 1.0 / (2.0 * r_obs);
    c->cap_r = R_S * 1.1;
    c->r_esc = 1.0 / c->ue;
    c->ue_sq = c->ue * c->ue;
    c->inv_sqrt_f0 = 1.0 / c->sqrt_f0;
    c->inv_ue_sq = 1.0 / c->ue_sq;
    c->div_const_ok = div_const_exact(c->sqrt_f0) && div_const_exact(c->ue_sq);
    // the FMA loop's scaled variable v = 3M u (lp_internal.cuh, rk4_step)
    c->v0 = c->M3 * c->u0;
    c->vc = c->M3 * c->uc;
    c->ve = c->M3 * c->ue;
    c->inv_M3 = 1.0 / c->M3;
    c->hh2 = c->hh * c->hh;
    c->h2_2 = c->h * c->hh;
    c->h2_6 = c->h * c->h6;
    c->scaled_ok = (c->M3 > 1e-100 && c->M3 < 1e100 && isfinite(c->inv_M3)) ? 1 : 0;

    // replay the phi bookkeeping of the while-loop (metrics.py:72-78, :93, :115)
    int shift = 0;
    if (h_max > 0.0 && phi_max > 0.0) {
        const double est = phi_max / h_max + 4.0;
        if (!(est < (double)LP_MAX_STEPS)) return LP_ERR_UNSUPPORTED;
        while ((((long long)est) >> shift) >= LP_PHI_TAB) ++shift;
    }
    c->phi_shift = shift;
    const int mask = (1 << shift) - 1;
    double phi = 0.0;
    int k = 0;
    while (phi < phi_max) {
        double h = h_max;
        const double remaining = phi_max - phi;
        if (remaining < h) h = remaining;
        if (h <= 0.0) break;
        if (h == h_max && c->n_tail == 0) {
            if ((k & mask) == 0) {
                if ((k >> shift) >= LP_PHI_TAB) return LP_ERR_UNSUPPORTED;
                c->phi_tab[k >> shift] = phi;
            }
            c->n_full++;
        } else {
            if (c->n_tail >= LP_MAX_TAIL) return LP_ERR_UNSUPPORTED;
            c->tail_h[c->n_tail] = h;
            c->tail_phi[c->n_tail] = phi;
            c->n_tail++;
        }
        phi = phi + h;
        if (++k > LP_MAX_STEPS) return LP_ERR_UNSUPPORTED;
    }
    c->phi_end = phi;
    return LP_OK;
}

// Fast-path precondition: positive finite band, observer strictly inside it, and at least
// one representable high word strictly between the bounds' high words.
int lp_binet_fast_ok(const BinetConsts *c)
{
    if (!(c->uc > 0.0) || !(c->ue > 0.0) || !isfinite(c->uc) || !isfinite(c->ue)) return 0;
    if (!(c->ue < c->u0 && c->u0 < c->uc)) return 0;
    unsigned long long bc, be;
    memcpy(&bc, &c->uc, 8);
    memcpy(&be, &c->ue, 8);
    const unsigned hc = (unsigned)(bc >> 32), he = (unsigned)(be >> 32);
    return hc > he + 1u;
}

// The same for a kernel that runs the FMA loop (scaled band) and the strict re-trace (plain band).
int lp_binet_fast_ok_fused(const BinetConsts *c)
{
    if (!c->scaled_ok || !lp_binet_fast_ok(c)) return 0;
    if (!(c->vc > 0.0) || !(c->ve > 0.0) || !isfinite(c->vc) || !isfinite(c->ve)) return 0;
    if (!(c->ve < c->v0 && c->v0 < c->vc)) return 0;
    unsigned long long bc, be;
    memcpy(&bc, &c->vc, 8);
    memcpy(&be, &c->ve, 8);
    const unsigned hc = (unsigned)(bc >> 32), he = (unsigned)(be >> 32);
    return hc > he + 1u;
}

// 1 when the multiply + two-fma form of (i - half) / f used by cam_coord() equals the IEEE
// division bit for bit for every i in [0, n) (it always should, by Markstein's theorem, as long
// as inv_f = RN(1/f); this makes it a checked fact per frame rather than a proof obligation).
static int coord_div_is_exact(int n, double half, double f, double inv_f)
{
    if (!(f > 0.0) || !isfinite(f) || !isfinite(inv_f)) return 0;
    for (int i = 0; i < n; ++i) {
        const double x = (double)i - half;
        const double q = x * inv_f;
        const double q2 = fma(fma(-q, f, x), inv_f, q);
        if (q2 != x / f) return 0;
    }
    return 1;
}

int lp_make_cam_consts(const lp_camera *cam, CamConsts *o)
{
    if (!cam || cam->height < 0 || cam->width < 0) return LP_ERR_INVALID_ARG;
    o->height = cam->height;
    o->width = cam->width;
    o->fx = cam->fx;
    o->fy = cam->fy;
    o->half_w = cam->width / 2.0;
    o->half_h = cam->height / 2.0;
    o->d0 = cam->d[0]; o->d1 = cam->d[1]; o->d2 = cam->d[2];
    o->ex0 = cam->e_x[0]; o->ex1 = cam->e_x[1]; o->ex2 = cam->e_x[2];
    o->ey0 = cam->e_y[0]; o->ey1 = cam->e_y[1]; o->ey2 = cam->e_y[2];
    o->inv_fx = 1.0 / o->fx;
    o->inv_fy = 1.0 / o->fy;
    o->fast_x = coord_div_is_exact(o->width, o->half_w, o->fx, o->inv_fx);
    o->fast_y = coord_div_is_exact(o->height, o->half_h, o->fy, o->inv_fy);
    return LP_OK;
}

static double dot3(const double *a, const double *b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
static double norm3(const double *a) { return sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]); }

// image_lens.py:21-61 (_psi_to_bh_direction, _psi_frame) and :138-139 (fx, fy).
extern "C" int lp_camera_init(int32_t height, int32_t width, double hfov, double vfov,
                              double psi_y, double psi_x, lp_camera *cam)
{
    if (!cam || height < 0 || width < 0) return LP_ERR_INVALID_ARG;
    cam->height = height;
    cam->width = width;
    cam->fx = (width / 2.0) / tan(hfov / 2);
    cam->fy = (height / 2.0) / tan(vfov / 2);
    double *d = cam->d, *ex = cam->e_x, *ey = cam->e_y;
    d[0] = sin(psi_x) * cos(psi_y);
    d[1] = -sin(psi_y);
    d[2] = cos(psi_x) * cos(psi_y);
    const double cx[3] = {1.0, 0.0, 0.0}, cy[3] = {0.0, 1.0, 0.0};
    double t = dot3(cx, d);
    for (int i = 0; i < 3; ++i) ex[i] = cx[i] - t * d[i];
    double n = norm3(ex);
    if (n < 1e-12) {
        t = dot3(cy, d);
        for (int i = 0; i < 3; ++i) ex[i] = cy[i] - t * d[i];
        n = norm3(ex);
    }
    n = n > 1e-12 ? n : 1e-12;
    for (int i = 0; i < 3; ++i) ex[i] /= n;
    const double t1 = dot3(cy, d), t2 = dot3(cy, ex);
    for (int i = 0; i < 3; ++i) ey[i] = cy[i] - t1 * d[i] - t2 * ex[i];
    n = norm3(ey);
    if (n < 1e-12) {
        ey[0] = d[1] * ex[2] - d[2] * ex[1];
        ey[1] = d[2] * ex[0] - d[0] * ex[2];
        ey[2] = d[0] * ex[1] - d[1] * ex[0];
        n = norm3(ey);
    }
    n = n > 1e-12 ? n : 1e-12;
    for (int i = 0; i < 3; ++i) ey[i] /= n;
    return LP_OK;
}

extern "C" int lp_camera_fast_coords(const lp_camera *cam, int32_t *fast_x, int32_t *fast_y)
{
    CamConsts c;
    const int rc = lp_make_cam_consts(cam, &c);
    if (rc != LP_OK) return rc;
    if (fast_x) *fast_x = c.fast_x;
    if (fast_y) *fast_y = c.fast_y;
    return LP_OK;
}
