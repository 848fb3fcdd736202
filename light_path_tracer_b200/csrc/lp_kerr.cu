// lp_kerr.cu — Kerr null-geodesic tracer (SURVEY.md §8(f) rank 1): the reference's
// _kerr_trace_ray_numba (metrics.py:419-567) — Dormand-Prince 4(5) with FSAL and the
// reference's own step controller on the reduced 5-D Hamiltonian state [r, theta, phi, p_r,
// p_theta] (metrics.py:227-306), initial conditions metrics.py:148-224, final direction
// metrics.py:362-416 — batched as _trace_rays_batch_kerr (metrics.py:671-679) and as the
// per-pixel driver precompute_final_alpha_lookup_2d (image_lens.py:185-280).
//
// GPU layout: persistent warps, one ray per LANE, every trip of the main loop is one step
// ATTEMPT (accepted or rejected) for all 32 lanes; a lane whose ray has ended takes another ray
// of its warp's queue, so captured / escaped rays stop occupying lanes (adaptive step counts
// differ 3x between neighbouring rays near the shadow edge).  The divergent per-ray work
// (initial conditions + first right-hand side: ~1500 instructions; final direction: ~600) is
// never run for a single lane: lp_kerr_queued_kernel (the default, see there) prepares and
// retires rays 32 at a time through per-warp queues in shared memory; lp_kerr_kernel
// (LP_KERR_QUEUE=0) parks finished lanes and serves them in one flush phase once
// KERR_REFILL_MIN lanes wait.  State, the seven stage vectors and the controller live in
// registers, fp64; the right-hand side is one __noinline__ function (arguments and results in
// registers) so the hot loop stays inside the instruction cache.  No atomics, no hidden state.
//
// Arithmetic: every expression is written in the reference's order and the library is built
// with -fmad=false, so all +,-,*,/ and sqrt round exactly like the numba build; what differs
// from the host is the transcendental library (sin/cos of theta in the right-hand side, pow in
// the controller, arccos at the end), each within 1-2 ulp.  The right-hand side's 14 IEEE
// divisions share 7 denominators: each quotient is formed as the compiler's own division
// sequence with the reciprocal part hoisted (div_rcp / div_by, lp_internal.cuh) — bit-identical
// quotients, 204 instead of 235 FP64-pipe slots and 325 instead of 604 instructions per
// evaluation.  Three shared approximate reciprocals (a few ulp per term) would be cheaper, but with
// the axis_refine tolerances (rtol 1e-8) they move step sizes by ~1e-8, and the reference's linear
// interpolation at the exit radius turns that into up to 6e-9 in final_alpha, outside the 1e-9 bar.
#include "lp_internal.cuh"
#include <stdlib.h>

#define KERR_BLOCK 128
#define KERR_REFILL_MIN 8
#define KERR_DEFAULT_MINB 4

struct KerrArgs {
    // ray source A: explicit arrays
    const double *alphas, *thetas;
    const uint8_t *refine;           // optional per-ray axis_refine
    // ray source B: frame tile (alpha from a float32 table, theta from the pixel)
    const float *alpha32;            // [rows * width]
    const uint8_t *refine_cols;      // optional [width]
    int32_t frame_mode, row0;
    long long n;
    double M, a, r_plus, r_obs, theta_obs, lambda_max;
    double sin_th_obs, cos_th_obs;   // host libm (the reference's own), one value per launch
    // outputs (WIDE: f64 / i64, else f32 / u16)
    void *out_fa, *out_w;
    int32_t wide, refill_min;
    int8_t *out_status;              // optional
    int32_t *out_steps;              // optional [n][2]: accepted steps, attempts
};

static __constant__ double kA21 = 1.0 / 5.0, kA31 = 3.0 / 40.0, kA32 = 9.0 / 40.0, kA41 = 44.0 / 45.0,
    kA42 = -56.0 / 15.0, kA43 = 32.0 / 9.0, kA51 = 19372.0 / 6561.0, kA52 = -25360.0 / 2187.0,
    kA53 = 64448.0 / 6561.0, kA54 = -212.0 / 729.0, kA61 = 9017.0 / 3168.0, kA62 = -355.0 / 33.0,
    kA63 = 46732.0 / 5247.0, kA64 = 49.0 / 176.0, kA65 = -5103.0 / 18656.0, kB1 = 35.0 / 384.0,
    kB3 = 500.0 / 1113.0, kB4 = 125.0 / 192.0, kB5 = -2187.0 / 6784.0, kB6 = 11.0 / 84.0,
    kE1 = 71.0 / 57600.0, kE3 = -71.0 / 16695.0, kE4 = 71.0 / 1920.0, kE5 = -17253.0 / 339200.0,
    kE6 = 22.0 / 525.0, kE7 = -1.0 / 40.0;

// metrics.py:227-306
struct K5 { double v0, v1, v2, v3, v4; };

// All arguments and the five derivatives travel in registers (scalars by value, a plain struct
// back): array references to a __noinline__ function would go through local memory.
__device__ __noinline__ K5 kerr_rhs_regs(double r, double th, double p_r, double p_th, double p_t, double p_phi,
                                         double M, double a, double r_floor)
{
    K5 out;
    if (r <= r_floor) {
        out.v0 = out.v1 = out.v2 = out.v3 = out.v4 = 0.0;
        return out;
    }
    // theta is a polar angle (a few pi at most): the straight-line sincos of lp_internal.cuh (fdlibm kernel
    // polynomials, constants from the constant bank) instead of the library call with its immediates and
    // slow-path branch — either differs from the host's libm in the last place, which the Kerr bar allows for
    double sin_th, cos_th;
    if (fabs(th) < 1.0e4) sincos_moderate(th, sin_th, cos_th);
    else sincos(th, &sin_th, &cos_th);
    double sin_th_sq = sin_th * sin_th;
    if (sin_th_sq < 1e-15) sin_th_sq = 1e-15;
    // The reference's expression tree, one IEEE quotient per `/` (bit for bit: div_by), over the
    // 7 distinct denominators its 14 divisions share.
    const double Sigma = r * r + a * a * cos_th * cos_th;
    const double Delta = r * r - 2.0 * M * r + a * a;
    const double A = (r * r + a * a) * (r * r + a * a) - a * a * Delta * sin_th_sq;
    const double sigma_delta = Sigma * Delta;
    const double sigma_sq = Sigma * Sigma;
    const double sigma_sq_delta = sigma_sq * Delta;
    const double sigma_delta_sq = sigma_delta * sigma_delta;
    const double den = sigma_delta * sin_th_sq;
    const double den_sq = den * den;
    const double y_S = div_rcp(Sigma), y_SD = div_rcp(sigma_delta), y_S2 = div_rcp(sigma_sq);
    const double y_S2D = div_rcp(sigma_sq_delta), y_SD2 = div_rcp(sigma_delta_sq);
    const double y_den = div_rcp(den), y_den2 = div_rcp(den_sq);
    const double g_tphi_inv = div_by(-2.0 * M * a * r, sigma_delta, y_SD);
    const double g_rr_inv = div_by(Delta, Sigma, y_S);
    const double g_thth_inv = div_by(1.0, Sigma, y_S);
    const double g_phiphi_inv = div_by(Delta - a * a * sin_th_sq, den, y_den);
    const double dr = g_rr_inv * p_r;
    const double dth = g_thth_inv * p_th;
    const double dphi = g_tphi_inv * p_t + g_phiphi_inv * p_phi;
    const double dSigma_dr = 2.0 * r;
    const double dDelta_dr = 2.0 * r - 2.0 * M;
    const double dA_dr = 4.0 * r * (r * r + a * a) - a * a * dDelta_dr * sin_th_sq;
    const double dg_tt_inv_dr = div_by(-(dA_dr * sigma_delta - A * (dSigma_dr * Delta + Sigma * dDelta_dr)),
                                       sigma_delta_sq, y_SD2);
    const double dg_tphi_inv_dr = div_by(-(2.0 * M * a * (sigma_delta - r * (dSigma_dr * Delta + Sigma * dDelta_dr))),
                                         sigma_delta_sq, y_SD2);
    const double dg_rr_inv_dr = div_by(dDelta_dr * Sigma - Delta * dSigma_dr, sigma_sq, y_S2);
    const double dg_thth_inv_dr = div_by(-dSigma_dr, sigma_sq, y_S2);
    const double dg_phiphi_inv_dr = div_by(dDelta_dr * den
                                           - (Delta - a * a * sin_th_sq)
                                           * (dSigma_dr * Delta + Sigma * dDelta_dr) * sin_th_sq,
                                           den_sq, y_den2);
    const double dp_r = -0.5 * (dg_tt_inv_dr * p_t * p_t
                                + 2.0 * dg_tphi_inv_dr * p_t * p_phi
                                + dg_rr_inv_dr * p_r * p_r
                                + dg_thth_inv_dr * p_th * p_th
                                + dg_phiphi_inv_dr * p_phi * p_phi);
    const double dSigma_dth = -2.0 * a * a * sin_th * cos_th;
    const double dA_dth = -a * a * Delta * 2.0 * sin_th * cos_th;
    const double dg_tt_inv_dth = div_by(-(dA_dth * Sigma * Delta - A * dSigma_dth * Delta), sigma_delta_sq, y_SD2);
    const double dg_tphi_inv_dth = div_by(2.0 * M * a * r * dSigma_dth, sigma_sq_delta, y_S2D);
    const double dg_rr_inv_dth = div_by(-Delta * dSigma_dth, sigma_sq, y_S2);
    const double dg_thth_inv_dth = div_by(-dSigma_dth, sigma_sq, y_S2);
    const double num = Delta - a * a * sin_th_sq;
    const double dnum_dth = -a * a * 2.0 * sin_th * cos_th;
    const double dden_dth = dSigma_dth * Delta * sin_th_sq + Sigma * Delta * 2.0 * sin_th * cos_th;
    const double dg_phiphi_inv_dth = div_by(dnum_dth * den - num * dden_dth, den_sq, y_den2);
    const double dp_th = -0.5 * (dg_tt_inv_dth * p_t * p_t
                                 + 2.0 * dg_tphi_inv_dth * p_t * p_phi
                                 + dg_rr_inv_dth * p_r * p_r
                                 + dg_thth_inv_dth * p_th * p_th
                                 + dg_phiphi_inv_dth * p_phi * p_phi);
    out.v0 = dr; out.v1 = dth; out.v2 = dphi; out.v3 = dp_r; out.v4 = dp_th;
    return out;
}

__device__ __forceinline__ void kerr_rhs(const double (&s)[5], double p_t, double p_phi, double M, double a,
                                         double r_floor, double (&out)[5])
{
    const K5 k = kerr_rhs_regs(s[0], s[1], s[3], s[4], p_t, p_phi, M, a, r_floor);
    out[0] = k.v0; out[1] = k.v1; out[2] = k.v2; out[3] = k.v3; out[4] = k.v4;
}

// One Dormand-Prince attempt from (state, k1 = f(state)) with step h: stages 2-7 and the 5th-order
// solution (metrics.py:461-496).
__device__ __forceinline__ void kerr_dp_stages(const double (&state)[5], const double (&k1)[5], double h,
                                               double p_t, double p_phi, double M, double sp, double r_floor,
                                               double (&k3)[5], double (&k4)[5], double (&k5)[5], double (&k6)[5],
                                               double (&k7)[5], double (&nxt)[5])
{
    double k2[5], tmp[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) tmp[i] = state[i] + h * kA21 * k1[i];
    kerr_rhs(tmp, p_t, p_phi, M, sp, r_floor, k2);
#pragma unroll
    for (int i = 0; i < 5; ++i) tmp[i] = state[i] + h * (kA31 * k1[i] + kA32 * k2[i]);
    kerr_rhs(tmp, p_t, p_phi, M, sp, r_floor, k3);
#pragma unroll
    for (int i = 0; i < 5; ++i) tmp[i] = state[i] + h * (kA41 * k1[i] + kA42 * k2[i] + kA43 * k3[i]);
    kerr_rhs(tmp, p_t, p_phi, M, sp, r_floor, k4);
#pragma unroll
    for (int i = 0; i < 5; ++i)
        tmp[i] = state[i] + h * (kA51 * k1[i] + kA52 * k2[i] + kA53 * k3[i] + kA54 * k4[i]);
    kerr_rhs(tmp, p_t, p_phi, M, sp, r_floor, k5);
#pragma unroll
    for (int i = 0; i < 5; ++i)
        tmp[i] = state[i] + h * (kA61 * k1[i] + kA62 * k2[i] + kA63 * k3[i] + kA64 * k4[i] + kA65 * k5[i]);
    kerr_rhs(tmp, p_t, p_phi, M, sp, r_floor, k6);
#pragma unroll
    for (int i = 0; i < 5; ++i)
        nxt[i] = state[i] + h * (kB1 * k1[i] + kB3 * k3[i] + kB4 * k4[i] + kB5 * k5[i] + kB6 * k6[i]);
    kerr_rhs(nxt, p_t, p_phi, M, sp, r_floor, k7);
}

// Sum of squared scaled errors (metrics.py:505-513).  The five quotients e_i / scale_i go over a
// straight-line reciprocal (a few ulp; scale >= atol > 0): the norm only feeds the step controller,
// whose power is a few-ulp routine itself (inv_tenth_root), and an accept / reject decision could
// only change for an error norm within ~1e-16 of 1.  Anything non-finite takes the literal IEEE form.
__device__ __forceinline__ double kerr_err_sq(const double (&state)[5], const double (&nxt)[5],
                                              const double (&k1)[5], const double (&k3)[5], const double (&k4)[5],
                                              const double (&k5)[5], const double (&k6)[5], const double (&k7)[5],
                                              double h, double atol, double rtol)
{
    double e[5], sc[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        e[i] = h * (kE1 * k1[i] + kE3 * k3[i] + kE4 * k4[i] + kE5 * k5[i] + kE6 * k6[i] + kE7 * k7[i]);
        const double as = fabs(state[i]), an = fabs(nxt[i]);
        sc[i] = atol + rtol * ((as > an) ? as : an);       // compare + select: fmax is ~7 instructions on sm_100
    }
    double err_sq = 0.0;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        const double q = e[i] * fast_rcp(sc[i]);           // sc >= atol > 0; only the step controller sees the norm
        err_sq += q * q;
    }
    if (!isfinite(err_sq)) {
        err_sq = 0.0;
#pragma unroll
        for (int i = 0; i < 5; ++i) {
            const double q = e[i] / sc[i];
            err_sq += q * q;
        }
    }
    return err_sq;
}

// metrics.py:148-224.  false = (ok == False) -> status 0.
__device__ __forceinline__ bool kerr_init(double M, double a, double r_obs, double alpha, double theta,
                                          double theta_obs, double sin_th, double cos_th,
                                          double (&state)[5], double &p_t, double &p_phi)
{
    const double r = r_obs, th = theta_obs;
    double sin_th_sq = sin_th * sin_th;
    if (sin_th_sq < 1e-15) sin_th_sq = 1e-15;
    const double Sigma = r * r + a * a * cos_th * cos_th;
    const double Delta = r * r - 2.0 * M * r + a * a;
    if (Delta <= 0.0 || Sigma <= 0.0) return false;
    const double sin_alpha = lp_sin_cr(alpha);
    double sin_screen, cos_screen;
    sincos(theta, &sin_screen, &cos_screen);
    const double E = 1.0;
    const double sqrt_Delta = __dsqrt_rn(Delta), sqrt_Sigma = __dsqrt_rn(Sigma);
    const double rho = r * sin_alpha * sqrt_Sigma / sqrt_Delta;
    const double alpha_screen = -rho * sin_screen;
    const double beta_screen = -rho * cos_screen;
    const double xi = -alpha_screen * sin_th;
    const double eta = beta_screen * beta_screen + cos_th * cos_th * (alpha_screen * alpha_screen - a * a);
    const double L = xi * E;
    const double Q = eta * E * E;
    p_t = -E;
    p_phi = L;
    double Theta = Q - cos_th * cos_th * (L * L / sin_th_sq - a * a * E * E);
    if (Theta < 0.0) Theta = 0.0;
    const double p_th_sign = (cos_screen > 0.0) ? -1.0 : 1.0;
    const double p_theta = p_th_sign * __dsqrt_rn(Theta);
    const double A_val = (r * r + a * a) * (r * r + a * a) - a * a * Delta * sin_th_sq;
    const double g_tt_inv = -A_val / (Sigma * Delta);
    const double g_tphi_inv = -2.0 * M * a * r / (Sigma * Delta);
    const double g_rr_inv = Delta / Sigma;
    const double g_thth_inv = 1.0 / Sigma;
    const double g_phiphi_inv = (Delta - a * a * sin_th_sq) / (Sigma * Delta * sin_th_sq);
    const double other = (g_tt_inv * p_t * p_t
                          + 2.0 * g_tphi_inv * p_t * p_phi
                          + g_thth_inv * p_theta * p_theta
                          + g_phiphi_inv * p_phi * p_phi);
    double p_r_sq = -other / g_rr_inv;
    if (p_r_sq < 0.0) p_r_sq = 0.0;
    state[0] = r; state[1] = th; state[2] = 0.0; state[3] = -__dsqrt_rn(p_r_sq); state[4] = p_theta;
    return true;
}

// metrics.py:362-416
__device__ __noinline__ int kerr_extract_angle(const double (&state)[5], double p_t, double p_phi, double M, double a,
                                               double r_capture, int event_status, double &fa, long long &nh)
{
    const double r_f = state[0], th_f = state[1], phi_f = state[2], p_r_f = state[3], p_th_f = state[4];
    const long long n_half = half_orbits(phi_f);
    fa = __longlong_as_double(0x7ff8000000000000LL);
    if (r_f <= r_capture * 1.1 || event_status == -1) { nh = n_half; return -1; }
    if (!isfinite(r_f) || !isfinite(th_f) || !isfinite(phi_f)) { nh = 0; return 0; }
    double sin_th, cos_th;
    sincos(th_f, &sin_th, &cos_th);
    double sin_th_sq = sin_th * sin_th;
    if (sin_th_sq < 1e-15) sin_th_sq = 1e-15;
    const double Sigma_f = r_f * r_f + a * a * cos_th * cos_th;
    const double Delta_f = r_f * r_f - 2.0 * M * r_f + a * a;
    nh = n_half;
    if (Sigma_f <= 1e-15 || fabs(Delta_f) <= 1e-15) return 0;
    const double dr_dl = Delta_f / Sigma_f * p_r_f;
    const double dth_dl = p_th_f / Sigma_f;
    const double dphi_dl = (-2.0 * M * a * r_f / (Sigma_f * Delta_f) * p_t
                            + (Delta_f - a * a * sin_th_sq) / (Sigma_f * Delta_f * sin_th_sq) * p_phi);
    double sin_phi, cos_phi;
    sincos(phi_f, &sin_phi, &cos_phi);
    const double vx = (sin_th * cos_phi * dr_dl + r_f * cos_th * cos_phi * dth_dl - r_f * sin_th * sin_phi * dphi_dl);
    const double vy = (sin_th * sin_phi * dr_dl + r_f * cos_th * sin_phi * dth_dl + r_f * sin_th * cos_phi * dphi_dl);
    const double vz = cos_th * dr_dl - r_f * sin_th * dth_dl;
    if (!isfinite(vx) || !isfinite(vy) || !isfinite(vz)) return 0;
    const double v_mag = __dsqrt_rn(vx * vx + vy * vy + vz * vz);
    if (v_mag < 1e-30) return 1;
    fa = acos(clip_scalar(-vx / v_mag, -1.0, 1.0));
    return 1;
}

__device__ __forceinline__ bool finite5(const double (&x)[5])
{
    return isfinite(x[0]) && isfinite(x[1]) && isfinite(x[2]) && isfinite(x[3]) && isfinite(x[4]);
}

// image_lens.py:194-208: screen angle of a pixel (theta_pixel)
__device__ __forceinline__ double pixel_theta(const CamConsts &cam, int row, int col)
{
    const double xc = cam_x(cam, col), yc = cam_y(cam, row);
    const double denom = __dsqrt_rn(1.0 + xc * xc + yc * yc);
    const double vx = xc / denom, vy = yc / denom, vz = 1.0 / denom;
    return atan2(vx * cam.ex0 + vy * cam.ex1 + vz * cam.ex2, vx * cam.ey0 + vy * cam.ey1 + vz * cam.ey2);
}

// Viewing angle, screen angle and axis_refine flag of ray `ray`: from the caller's arrays, or from
// the float32 alpha table and the pixel position (image_lens.py:194-208, :247).
__device__ __forceinline__ void kerr_load_ray(const KerrArgs &a, const CamConsts &cam, long long ray,
                                              double &alpha, double &theta, bool &refine)
{
    if (a.frame_mode) {
        int row, col;
        pixel_row_col(ray, a.n, cam.width, a.row0, row, col);
        alpha = (double)__ldg(a.alpha32 + ray);
        theta = pixel_theta(cam, row, col);
        refine = a.refine_cols ? (__ldg(a.refine_cols + col) != 0) : false;
    } else {
        alpha = __ldg(a.alphas + ray);
        theta = __ldg(a.thetas + ray);
        refine = a.refine ? (__ldg(a.refine + ray) != 0) : false;
    }
}

__device__ __forceinline__ void kerr_store_result(const KerrArgs &a, long long idx, int status, double fa,
                                                  long long nh, int accepted, int attempts)
{
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    const double fa_out = (status == 1) ? fa : qnan;                         // metrics.py:678
    if (a.wide) {
        ((double *)a.out_fa)[idx] = fa_out;
        ((long long *)a.out_w)[idx] = nh;
    } else {
        ((float *)a.out_fa)[idx] = (float)fa_out;                            // image_lens.py:261
        const long long c = nh < 0 ? 0 : (nh > 65535 ? 65535 : nh);          // image_lens.py:262
        ((unsigned short *)a.out_w)[idx] = (unsigned short)c;
    }
    if (a.out_status) a.out_status[idx] = (int8_t)status;
    if (a.out_steps) { a.out_steps[2 * idx] = accepted; a.out_steps[2 * idx + 1] = attempts; }
}

// One trip of the reference's `for _step in range(max_steps)` (metrics.py:451-566) for one lane: the
// loop guards, one Dormand-Prince attempt, the controller, the exit events.  done: 0 running,
// 1 finished -> extract the final direction, 2 invalid (status 0).
__device__ __forceinline__ void kerr_trip(double (&state)[5], double (&k1)[5], double p_t, double p_phi,
                                          double M, double sp, double r_floor, double r_capture, double r_escape,
                                          double lambda_max, double h_min, double atol, double rtol,
                                          double &lam, double &h, int &accepted, int &attempts, int &iters,
                                          int &done, int &event_status)
{
    done = 0;
    event_status = 2;
    if (iters >= 200000 || lam >= lambda_max) {
        done = 1;
    } else {
        iters++;
        const double remaining = lambda_max - lam;
        if (h > remaining) h = remaining;
        if (h <= 0.0) {
            done = 1;
        } else {
            attempts++;
            double k3[5], k4[5], k5[5], k6[5], k7[5], nxt[5];
            kerr_dp_stages(state, k1, h, p_t, p_phi, M, sp, r_floor, k3, k4, k5, k6, k7, nxt);

            if (!finite5(nxt) || nxt[0] <= 0.0) {                        // metrics.py:498-503
                h *= 0.25;
                if (h < h_min) done = 2;
            } else {
                const double err_sq = kerr_err_sq(state, nxt, k1, k3, k4, k5, k6, k7, h, atol, rtol);
                // err_norm = sqrt(err_sq / 5) (metrics.py:514) only enters comparisons with constants and
                // 0.9 * err_norm ** -0.2, which feeds both the reject (metrics.py:517) and the accept
                // (metrics.py:562) controller: the controller works on the square, e2 = err_norm^2, and
                // 0.9 * e2^-0.1 comes from inv_tenth_root (lp_internal.cuh) instead of a square root, a
                // division and pow() — a few ulp, like the difference between CUDA's pow and the host's
                const double e2 = err_sq * 0.2;
                double pow_term = 0.9 * inv_tenth_root(e2);
                if (!(err_sq == err_sq)) pow_term = err_sq;              // NaN stays NaN (fmin / fmax below drop it)
                if (err_sq > 5.0) {                                      // err_norm > 1: reject, metrics.py:516-522
                    const double factor = (pow_term > 0.2) ? pow_term : 0.2;        // max(0.2, .): NaN -> 0.2 like fmax
                    h *= factor;
                    if (h < h_min) done = 2;
                } else {
                    accepted++;
                    const double r_prev = state[0], r_next = nxt[0];
                    const bool cap = (r_prev > r_capture && r_next <= r_capture);
                    const bool esc = !cap && (r_prev < r_escape && r_next >= r_escape);
                    if (cap || esc) {                                    // metrics.py:528-550
                        const double target = cap ? r_capture : r_escape;
                        const double denom = r_next - r_prev;
                        double frac = (denom == 0.0) ? 1.0 : (target - r_prev) / denom;
                        frac = clip_scalar(frac, 0.0, 1.0);
#pragma unroll
                        for (int i = 0; i < 5; ++i) state[i] = state[i] + frac * (nxt[i] - state[i]);
                        lam += frac * h;
                        event_status = cap ? -1 : 1;
                        done = 1;
                    } else {
#pragma unroll
                        for (int i = 0; i < 5; ++i) { state[i] = nxt[i]; k1[i] = k7[i]; }
                        lam += h;
                        if (!finite5(state)) {
                            done = 2;
                        } else if (e2 < 1e-20) {                        // err_norm < 1e-10
                            h *= 5.0;
                        } else {
                            h *= (pow_term < 5.0) ? pow_term : 5.0;                 // min(5.0, .): NaN -> 5.0 like fmin
                        }
                    }
                }
            }
        }
    }
}

template <int MINB>
__global__ void __launch_bounds__(KERR_BLOCK, MINB)
lp_kerr_kernel(const KerrArgs a, const CamConsts cam)
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const double M = a.M, sp = a.a, r_floor = a.r_plus * 1.001;
    const double r_capture = a.r_plus * 1.01, r_escape = a.r_obs * 2.0, lambda_max = a.lambda_max;
    const double h_min = 1e-12;
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);

    bool active = false;
    int pending = 0, pend_event = 2;   // a finished ray waiting for its flush: `done` code, event status
    long long idx = -1;
    double state[5], k1[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) { state[i] = 0.0; k1[i] = 0.0; }
    double p_t = -1.0, p_phi = 0.0, lam = 0.0, h = 1.0, atol = 1e-8, rtol = 1e-6;
    int accepted = 0, attempts = 0, iters = 0;

    LpWarpQueue queue(a.n);

    while (true) {
        // ---------------- lane refill ----------------
        const unsigned idle = __ballot_sync(full, !active);
        const bool flush = idle && (__popc(idle) >= a.refill_min || idle == full);
        // ---------------- finished rays: final direction + stores, for all waiting lanes at once ----------------
        if (flush && pending) {
            double fa = qnan;
            long long nh = 0;
            int status = 0;
            if (pending == 1) status = kerr_extract_angle(state, p_t, p_phi, M, sp, r_capture, pend_event, fa, nh);
            kerr_store_result(a, idx, status, fa, nh, accepted, attempts);
            pending = 0;
        }
        if (flush && !queue.empty) {
            const long long ray = queue.take(idle, lane);
            if (!active && ray < a.n) {
                idx = ray;
                double alpha, theta;
                bool refine;
                kerr_load_ray(a, cam, ray, alpha, theta, refine);
                atol = refine ? 1e-10 : 1e-8;                               // metrics.py:432-433
                rtol = refine ? 1e-8 : 1e-6;
                if (kerr_init(M, sp, a.r_obs, alpha, theta, a.theta_obs, a.sin_th_obs, a.cos_th_obs, state, p_t, p_phi)) {
                    kerr_rhs(state, p_t, p_phi, M, sp, r_floor, k1);   // FSAL seed, metrics.py:447
                    lam = 0.0;
                    h = fmax(1.0, 0.01 * a.r_obs);
                    accepted = 0; attempts = 0; iters = 0;
                    active = true;
                } else {
                    kerr_store_result(a, idx, 0, qnan, 0, 0, 0);      // initial conditions invalid: status 0
                }
            }
        }
        if (!__any_sync(full, active)) {
            if (queue.empty) break;
            continue;
        }
        if (!active) continue;

        // ---------------- one trip of the reference's `for _step in range(max_steps)` ----------------
        int done, event_status;
        kerr_trip(state, k1, p_t, p_phi, M, sp, r_floor, r_capture, r_escape, lambda_max, h_min, atol, rtol,
                  lam, h, accepted, attempts, iters, done, event_status);
        if (done) {          // park the lane: its result is produced in the next flush phase
            pending = done;
            pend_event = event_status;
            active = false;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Queued variant (the default): the two divergent per-ray phases run CONVERGED on whole batches.
//   * in-queue: when a warp runs out of prepared rays, all 32 lanes together compute the initial
//     conditions and the first right-hand side of the next 32 rays of its queue into shared
//     memory (coalesced alpha reads); empty lanes pop prepared rays one by one, in every trip,
//     so a finished lane is stepping again in the next trip (no refill threshold, no waiting);
//   * out-queue: a finished lane pushes its final state to shared memory and is free at once;
//     when 32 results have gathered, all 32 lanes extract the final directions together.
// Same rays, same operations per ray, bit-identical outputs; only the lane a ray runs in differs.
// Shared memory: 5.1 KB per warp.
#define KQ_IN 10      /* r, theta, p_r, p_theta, p_phi, k1[0..4] */
#define KQ_OUT 6      /* r, theta, phi, p_r, p_theta, p_phi */

struct KerrWarpQueues {
    double in[KQ_IN][32];
    double out[KQ_OUT][32];
    long long out_idx[32];
    int out_accepted[32], out_attempts[32], out_code[32];   // code = done | (event_status + 1) << 2
    int in_flag[32];                                        // bit 0 valid, bit 1 axis_refine
};

template <int MINB>
__global__ void __launch_bounds__(KERR_BLOCK, MINB)
lp_kerr_queued_kernel(const KerrArgs a, const CamConsts cam)
{
    __shared__ KerrWarpQueues queues[KERR_BLOCK / 32];
    KerrWarpQueues &Q = queues[threadIdx.x >> 5];
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned lt_mask = (1u << lane) - 1u;
    const double M = a.M, sp = a.a, r_floor = a.r_plus * 1.001;
    const double r_capture = a.r_plus * 1.01, r_escape = a.r_obs * 2.0, lambda_max = a.lambda_max;
    const double h_min = 1e-12;
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    const double p_t = -1.0;                    // -E with E = 1 (metrics.py:196, :203)

    bool active = false;
    int pending = 0, pend_event = 2;
    long long idx = -1;
    double state[5], k1[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) { state[i] = 0.0; k1[i] = 0.0; }
    double p_phi = 0.0, lam = 0.0, h = 1.0, atol = 1e-8, rtol = 1e-6;
    int accepted = 0, attempts = 0, iters = 0;

    // warp-uniform queue state: the warp's chunks of 32 rays (LpWarpQueue::chunk_ray), one chunk at a time
    LpWarpQueue queue(a.n);
    long long chunk = 0, in_ray0 = 0;
    int in_base = 0, in_avail = 0, out_count = 0;

    while (true) {
        // ---------------- finished lanes -> out-queue ----------------
        const unsigned fin = __ballot_sync(full, pending != 0);
        const bool last_round = !fin && queue.empty && in_avail == 0 && !__any_sync(full, active);
        if (out_count && (out_count + __popc(fin) > 32 || last_round)) {
            // all lanes together: final direction + stores for the gathered results
            __syncwarp();
            if (lane < out_count) {
                double st[5];
#pragma unroll
                for (int i = 0; i < 5; ++i) st[i] = Q.out[i][lane];
                const double o_p_phi = Q.out[5][lane];
                const int code = Q.out_code[lane];
                double fa = qnan;
                long long nh = 0;
                int status = 0;
                if ((code & 3) == 1)
                    status = kerr_extract_angle(st, p_t, o_p_phi, M, sp, r_capture, (code >> 2) - 1, fa, nh);
                kerr_store_result(a, Q.out_idx[lane], status, fa, nh, Q.out_accepted[lane], Q.out_attempts[lane]);
            }
            __syncwarp();
            out_count = 0;
        }
        if (fin) {
            if (pending) {
                const int slot = out_count + __popc(fin & lt_mask);
#pragma unroll
                for (int i = 0; i < 5; ++i) Q.out[i][slot] = state[i];
                Q.out[5][slot] = p_phi;
                Q.out_idx[slot] = idx;
                Q.out_accepted[slot] = accepted;
                Q.out_attempts[slot] = attempts;
                Q.out_code[slot] = pending | ((pend_event + 1) << 2);
                pending = 0;
            }
            out_count += __popc(fin);
        }
        if (last_round) {
            if (out_count) continue;            // (cannot happen: !fin on the last round)
            break;
        }

        // ---------------- empty lanes <- in-queue ----------------
#pragma unroll 1
        for (int pass = 0; pass < 2; ++pass) {
            const unsigned empty = __ballot_sync(full, !active);
            if (!empty) break;
            if (in_avail == 0) {
                if (queue.empty) break;
                // all lanes together: initial conditions + FSAL seed of the next 32 rays
                in_ray0 = queue.chunk_ray(chunk);
                const long long ray = in_ray0 + lane;
                int flag = 0;
                __syncwarp();
                if (ray < a.n) {
                    double alpha, theta;
                    bool refine;
                    kerr_load_ray(a, cam, ray, alpha, theta, refine);
                    double s0[5], kk[5], i_p_t, i_p_phi;
                    const bool ok = kerr_init(M, sp, a.r_obs, alpha, theta, a.theta_obs, a.sin_th_obs, a.cos_th_obs,
                                              s0, i_p_t, i_p_phi);
                    if (ok) {
                        kerr_rhs(s0, p_t, i_p_phi, M, sp, r_floor, kk);   // FSAL seed, metrics.py:447
                        Q.in[0][lane] = s0[0]; Q.in[1][lane] = s0[1]; Q.in[2][lane] = s0[3]; Q.in[3][lane] = s0[4];
                        Q.in[4][lane] = i_p_phi;
#pragma unroll
                        for (int i = 0; i < 5; ++i) Q.in[5 + i][lane] = kk[i];
                    }
                    flag = (ok ? 1 : 0) | (refine ? 2 : 0);
                }
                Q.in_flag[lane] = flag;
                __syncwarp();
                const long long left = a.n - in_ray0;
                in_avail = left < 32 ? (int)left : 32;
                in_base = 0;
                chunk++;
                queue.empty = (queue.chunk_ray(chunk) >= a.n);
            }
            const int rank = __popc(empty & lt_mask);
            if (!active && rank < in_avail) {
                const int e = in_base + rank;
                const int flag = Q.in_flag[e];
                idx = in_ray0 + e;
                if (flag & 1) {
                    state[0] = Q.in[0][e]; state[1] = Q.in[1][e]; state[2] = 0.0;
                    state[3] = Q.in[2][e]; state[4] = Q.in[3][e];
                    p_phi = Q.in[4][e];
#pragma unroll
                    for (int i = 0; i < 5; ++i) k1[i] = Q.in[5 + i][e];
                    atol = (flag & 2) ? 1e-10 : 1e-8;                       // metrics.py:432-433
                    rtol = (flag & 2) ? 1e-8 : 1e-6;
                    lam = 0.0;
                    h = fmax(1.0, 0.01 * a.r_obs);
                    accepted = 0; attempts = 0; iters = 0;
                    active = true;
                } else {
                    kerr_store_result(a, idx, 0, qnan, 0, 0, 0);            // initial conditions invalid: status 0
                }
            }
            const int taken = min(__popc(empty), in_avail);
            in_base += taken;
            in_avail -= taken;
        }
        if (!active) continue;

        // ---------------- one trip of the reference's `for _step in range(max_steps)` ----------------
        int done, event_status;
        kerr_trip(state, k1, p_t, p_phi, M, sp, r_floor, r_capture, r_escape, lambda_max, h_min, atol, rtol,
                  lam, h, accepted, attempts, iters, done, event_status);
        if (done) {
            pending = done;
            pend_event = event_status;
            active = false;
        }
    }
}

static int kerr_launch(KerrArgs &a, const CamConsts &cam, cudaStream_t stream)
{
    if (a.n == 0) return LP_OK;
    a.sin_th_obs = sin(a.theta_obs);
    a.cos_th_obs = cos(a.theta_obs);
    static int refill = 0;
    if (!refill) {
        const char *e = getenv("LP_KERR_REFILL");
        const int v = e ? atoi(e) : 0;
        refill = (v >= 1 && v <= 32) ? v : KERR_REFILL_MIN;
    }
    a.refill_min = refill;
    // resident CTAs per SM ptxas must fit (register cap): the kernel is latency-bound, so more
    // resident warps win until the spills cost more (LP_KERR_MINB = 2..6, tuning knob; the queued
    // kernel is built for 3..5 and runs 4 for the others)
    static int minb = 0;
    if (!minb) {
        const char *e = getenv("LP_KERR_MINB");
        const int v = e ? atoi(e) : 0;
        minb = (v >= 2 && v <= 6) ? v : KERR_DEFAULT_MINB;
    }
    const char *qe = getenv("LP_KERR_QUEUE");
    const bool queued = !(qe && atoi(qe) == 0);
    const void *fn;
    if (queued) {
        fn = minb == 3 ? (const void *)lp_kerr_queued_kernel<3>
           : minb == 5 ? (const void *)lp_kerr_queued_kernel<5> : (const void *)lp_kerr_queued_kernel<4>;
    } else {
        const void *parked[] = {(const void *)lp_kerr_kernel<2>, (const void *)lp_kerr_kernel<3>,
                                (const void *)lp_kerr_kernel<4>, (const void *)lp_kerr_kernel<5>,
                                (const void *)lp_kerr_kernel<6>};
        fn = parked[minb - 2];
    }
    int grid = 0;
    const int rc = lp_grid_for(fn, KERR_BLOCK, a.n, &grid);
    if (rc != LP_OK) return rc;
    void *args[] = {&a, (void *)&cam};
    cudaLaunchKernel(fn, grid, KERR_BLOCK, args, 0, stream);
    return lp_check_launch();
}

extern "C" int lp_kerr_trace_batch_f64(const double *alphas, const double *thetas, const uint8_t *axis_refines,
                                       int64_t n, double M, double a, double r_plus, double r_obs,
                                       double theta_obs, double lambda_max,
                                       double *out_fa, int64_t *out_w, int8_t *out_status, int32_t *out_steps,
                                       void *stream)
{
    if (n < 0) return LP_ERR_INVALID_ARG;
    if (n > 0 && (!alphas || !thetas || !out_fa || !out_w)) return LP_ERR_INVALID_ARG;
    KerrArgs k = {};
    k.alphas = alphas; k.thetas = thetas; k.refine = axis_refines; k.n = n;
    k.M = M; k.a = a; k.r_plus = r_plus; k.r_obs = r_obs; k.theta_obs = theta_obs; k.lambda_max = lambda_max;
    k.out_fa = out_fa; k.out_w = out_w; k.wide = 1; k.out_status = out_status; k.out_steps = out_steps;
    CamConsts cam = {};
    return kerr_launch(k, cam, (cudaStream_t)stream);
}

extern "C" int lp_kerr_trace_alpha32(const float *alpha32, const lp_camera *h_cam, int32_t row0, int32_t rows,
                                     const uint8_t *axis_refine_cols,
                                     double M, double a, double r_plus, double r_obs, double theta_obs,
                                     double lambda_max, float *out_fa32, uint16_t *out_w16,
                                     int8_t *out_status, int32_t *out_steps, void *stream)
{
    CamConsts cam;
    int rc = lp_make_cam_consts(h_cam, &cam);
    if (rc != LP_OK) return rc;
    if (row0 < 0 || rows < 0 || (long long)row0 + rows > cam.height) return LP_ERR_INVALID_ARG;
    const long long n = (long long)rows * cam.width;
    if (n > 0 && (!alpha32 || !out_fa32 || !out_w16)) return LP_ERR_INVALID_ARG;
    KerrArgs k = {};
    k.alpha32 = alpha32; k.refine_cols = axis_refine_cols; k.frame_mode = 1; k.row0 = row0; k.n = n;
    k.M = M; k.a = a; k.r_plus = r_plus; k.r_obs = r_obs; k.theta_obs = theta_obs; k.lambda_max = lambda_max;
    k.out_fa = out_fa32; k.out_w = out_w16; k.wide = 0; k.out_status = out_status; k.out_steps = out_steps;
    return kerr_launch(k, cam, (cudaStream_t)stream);
}
