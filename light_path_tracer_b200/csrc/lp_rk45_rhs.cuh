// lp_rk45_rhs.cuh — the right-hand sides of the generic RK45 integrator (lp_rk45.cu): the moving
// components of Schwarzschild.geodesic_equations (metrics.py:763-790) and Kerr.geodesic_equations
// (metrics.py:946-1029), and the four-component equatorial form of the batch path.
//
// In a header of their own so that tests/rk45_rhs_probe.cu evaluates the production functions
// (tests/test_gpu_rk45_rhs.py holds them to an exact reference); the kernels are the only other user.
#pragma once
#include "lp_internal.cuh"

#define RK_NC 6            /* moving components: t, r, theta, phi, p_r, p_theta */

struct ThetaCache { double th, s, c; };

// Schwarzschild.geodesic_equations (metrics.py:763-790) for the moving components.
// y = (t, r, theta, phi, p_r, p_theta); p_t and p_phi are constants of the motion.
__device__ __forceinline__ void rk_rhs(double R_S, double r_floor, double p_t, double p_phi,
                                       const double (&y)[RK_NC], ThetaCache &tc, double (&d)[RK_NC])
{
    const double r = y[1], th = y[2], p_r = y[4], p_th = y[5];
    if (r <= r_floor) {                                   // metrics.py:766-767
#pragma unroll
        for (int i = 0; i < RK_NC; ++i) d[i] = 0.0;
        return;
    }
    if (th != tc.th) { sincos(th, &tc.s, &tc.c); tc.th = th; }
    double s2 = tc.s * tc.s;
    if (s2 < 1e-15) s2 = 1e-15;
    const double pp2 = p_phi * p_phi;
    // The reference's expressions with its nine divisions replaced by products of three reciprocals
    // (1/r, 1/f and, off the equator only, 1/sin theta): every term within a few ulp of the
    // reference's.  That is the level at which scipy's own BLAS stage sums already differ from
    // any restatement, and it removes most of the FP64-pipe work of an evaluation (an IEEE
    // division is ~12 dependent pipe slots); tests/test_gpu_rk45.py holds the result to the same
    // bar (identical accept/reject sequences, final state <= 1e-9).
    // (sums contracted into fma: 18 FP64 instructions on the equator instead of 24 — the rounding differs from the
    // separately rounded form at the level the reciprocals already do)
    const double ir = fast_rcp(r);
    const double ir2 = ir * ir, ir3 = ir2 * ir;
    const double f = fma(-R_S, ir, 1.0);
    const double inv_f = fast_rcp(f);
    double is2 = 1.0, is1 = tc.s;                          // equatorial plane: sin(theta) = +-1 exactly
    if (s2 != 1.0) { is2 = fast_rcp(s2); is1 = fast_rcp(tc.s); }
    const double a = (0.5 * R_S) * ir2;
    const double ptf = p_t * inv_f;
    d[0] = -ptf;
    d[1] = f * p_r;
    d[2] = p_th * ir2;
    d[3] = p_phi * ir2 * is2;
    d[4] = fma(-a, fma(ptf, ptf, p_r * p_r), fma(pp2, is2, p_th * p_th) * ir3);
    d[5] = tc.c * pp2 * ir2 * is2 * is1;
}

// Kerr.geodesic_equations (metrics.py:946-1029) for the moving components (same six: p_t and
// p_phi are cyclic), over three shared reciprocals like the Schwarzschild form above.  The
// generic path has no sin^2(theta) floor (metrics.py:953-959), unlike the numba tracer.
__device__ __forceinline__ void rk_rhs_kerr(double M, double a, double r_floor, double p_t, double p_phi,
                                            const double (&y)[RK_NC], ThetaCache &tc, double (&d)[RK_NC])
{
    const double r = y[1], th = y[2], p_r = y[4], p_th = y[5];
    if (r <= r_floor) {                                   // metrics.py:950-951
#pragma unroll
        for (int i = 0; i < RK_NC; ++i) d[i] = 0.0;
        return;
    }
    if (th != tc.th) { sincos(th, &tc.s, &tc.c); tc.th = th; }
    const double sn = tc.s, cs = tc.c, s2 = sn * sn, a2 = a * a, r2 = r * r;
    const double Sigma = r2 + a2 * (cs * cs);
    const double Delta = r2 - 2.0 * M * r + a2;
    const double A = (r2 + a2) * (r2 + a2) - a2 * Delta * s2;
    const double iS = fast_rcp(Sigma), iD = fast_rcp(Delta), is2 = fast_rcp(s2);
    const double iSD = iS * iD, iS2 = iS * iS, iSD2 = iSD * iSD, iden2 = iSD2 * (is2 * is2);
    const double twoMa = 2.0 * M * a, SD = Sigma * Delta;
    const double num = Delta - a2 * s2, den = SD * s2;
    const double g_tt = -A * iSD, g_tphi = -twoMa * r * iSD, g_phiphi = num * iSD * is2;
    d[0] = g_tt * p_t + g_tphi * p_phi;
    d[1] = Delta * iS * p_r;
    d[2] = iS * p_th;
    d[3] = g_tphi * p_t + g_phiphi * p_phi;
    const double dS_r = 2.0 * r, dD_r = 2.0 * r - 2.0 * M;
    const double dA_r = 4.0 * r * (r2 + a2) - a2 * dD_r * s2;
    const double X = dS_r * Delta + Sigma * dD_r;
    const double pt2 = p_t * p_t, ptpp = p_t * p_phi, pr2 = p_r * p_r, pth2 = p_th * p_th, pp2 = p_phi * p_phi;
    d[4] = -0.5 * (-(dA_r * SD - A * X) * iSD2 * pt2 + 2.0 * (-(twoMa * (SD - r * X)) * iSD2) * ptpp
                   + (dD_r * Sigma - Delta * dS_r) * iS2 * pr2 + (-dS_r * iS2) * pth2
                   + (dD_r * den - num * X * s2) * iden2 * pp2);
    const double sc2 = 2.0 * sn * cs;
    const double dS_th = -a2 * sc2, dA_th = -a2 * Delta * sc2;
    const double dden_th = dS_th * Delta * s2 + SD * sc2;
    d[5] = -0.5 * (-(dA_th * SD - A * dS_th * Delta) * iSD2 * pt2 + 2.0 * (twoMa * r * dS_th * iS2 * iD) * ptpp
                   + (-Delta * dS_th * iS2) * pr2 + (-dS_th * iS2) * pth2
                   + (-a2 * sc2 * den - num * dden_th) * iden2 * pp2);
}

// The equatorial system's right-hand side (RkEquatorialSystem in lp_rk45.cu): the four live components.
#define RK_EQ 4

// SPEC: no test inside — the caller collects the smallest high word of r over the evaluations of a step
// attempt (one integer min each; a negative r is a negative word, a NaN a large one, as in the fp64 test)
// and repeats the attempt with the tested form in the rare case that a stage may have landed at or below
// the floor (the test, its branch and the zero defaults cost ~10 issue slots per evaluation).
template <bool SPEC>
__device__ __forceinline__ void rk_rhs_eq(double R_S, double r_floor, double p_t, double p_phi, double pp2,
                                          const double (&y)[RK_EQ], double (&d)[RK_EQ], int &r_hi_min)
{
    const double r = y[1], p_r = y[3];
    if (SPEC) {
        r_hi_min = min(r_hi_min, __double2hiint(r));
    } else if (r <= r_floor) {                            // metrics.py:766-767
#pragma unroll
        for (int i = 0; i < RK_EQ; ++i) d[i] = 0.0;
        return;
    }
    // rk_rhs with sin(theta) = 1, p_theta = 0: the same operations on the same operands
    const double ir = fast_rcp(r);
    const double ir2 = ir * ir, ir3 = ir2 * ir;
    const double f = fma(-R_S, ir, 1.0);
    const double inv_f = fast_rcp(f);
    const double a = (0.5 * R_S) * ir2;
    const double ptf = p_t * inv_f;
    d[0] = -ptf;
    d[1] = f * p_r;
    d[2] = p_phi * ir2;
    d[3] = fma(-a, fma(ptf, ptf, p_r * p_r), pp2 * ir3);
}
