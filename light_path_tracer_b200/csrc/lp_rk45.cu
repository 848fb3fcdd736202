// lp_rk45.cu — kernel (1b): batched 8-D Hamiltonian null-geodesic tracer with the semantics of
// the reference's GENERIC path, geodesic_tracer.trace_ray / integrate_geodesic
// (geodesic_tracer.py:22-82): scipy solve_ivp(method='RK45', rtol, atol, max_step,
// dense_output, two terminal events) on Schwarzschild.geodesic_equations (metrics.py:763-790)
// from Schwarzschild.initial_conditions (metrics.py:794-809).
//
// The stepper is scipy's (third-party, unpinned by the reference; restated from scipy 1.18.1,
// scipy/integrate/_ivp/rk.py:14-176, :538-566, :715-737, common.py:63-134, ivp.py:52-157,
// :676-697, optimize/Zeros/brentq.c): Dormand-Prince 5(4) with FSAL, scipy's step controller
// and first-step selection, events located with brentq on the quartic dense output.
//
// GPU layout — persistent warps, lane-level re-packing.  One ray per LANE; every trip of the
// main loop is one step ATTEMPT (accepted or rejected) for all 32 lanes, so lanes never wait
// for each other's rejections.  A lane whose ray has hit an event takes the next ray of its
// warp's queue (queue = the chunks of 32 consecutive rays w, w + NW, w + 2 NW, ... of the
// batch, NW = warps in the grid), so finished rays stop occupying lanes: the refill runs when
// at least RK_REFILL_MIN lanes are idle (ballot), which bounds both the idle-lane time and the
// number of partially filled refill passes.  No global atomics, no shared memory, no hidden
// state: re-entrant.
//
// Per-lane state in registers, fp64: of the 8 state components only 6 move — p_t and p_phi
// have identically zero derivatives (metrics.py:782, :789), so their K rows are exact zeros,
// y_new = y exactly and their error terms vanish; they are carried as constants and enter
// only where scipy's formulas see them (the y0/scale term of the first-step norm, the RHS).
// theta stays at (a few 1e-17 around) pi/2; sin/cos(theta) are re-evaluated only when theta's
// bits change.
//
// Arithmetic: the right-hand side keeps the reference's operation order with separately
// rounded operations (the library is built with -fmad=false); the stage / error / dense-output
// sums use fma chains — scipy forms them with BLAS dot products whose order and contraction
// are build specific, so bit equality with scipy is not attainable by any order (SURVEY.md
// 7.3 H7); measured agreement with the reference: see tests/test_gpu_rk45.py.
#include "lp_internal.cuh"
#include <stdlib.h>

#define RK_BLOCK 128
#define RK_REFILL_MIN 8
#define RK_DEFAULT_MINB 3
#define RK_DEFAULT_EQ 1
#define RK_DEFAULT_EQ_MINB 4
#define RK_NC 6            /* moving components: t, r, theta, phi, p_r, p_theta */

static __constant__ double c_A[6][5] = {
    {0, 0, 0, 0, 0},
    {1.0 / 5, 0, 0, 0, 0},
    {3.0 / 40, 9.0 / 40, 0, 0, 0},
    {44.0 / 45, -56.0 / 15, 32.0 / 9, 0, 0},
    {19372.0 / 6561, -25360.0 / 2187, 64448.0 / 6561, -212.0 / 729, 0},
    {9017.0 / 3168, -355.0 / 33, 46732.0 / 5247, 49.0 / 176, -5103.0 / 18656}};
static __constant__ double c_B[6] = {35.0 / 384, 0, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84};
static __constant__ double c_E[7] = {-71.0 / 57600, 0, 71.0 / 16695, -71.0 / 1920, 17253.0 / 339200,
                                     -22.0 / 525, 1.0 / 40};
static __constant__ double c_P[7][4] = {
    {1, -8048581381.0 / 2820520608, 8663915743.0 / 2820520608, -12715105075.0 / 11282082432},
    {0, 0, 0, 0},
    {0, 131558114200.0 / 32700410799, -68118460800.0 / 10900136933, 87487479700.0 / 32700410799},
    {0, -1754552775.0 / 470086768, 14199869525.0 / 1410260304, -10690763975.0 / 1880347072},
    {0, 127303824393.0 / 49829197408, -318862633887.0 / 49829197408, 701980252875.0 / 199316789632},
    {0, -282668133.0 / 205662961, 2019193451.0 / 616988883, -1453857185.0 / 822651844},
    {0, 40617522.0 / 29380423, -110615467.0 / 29380423, 69997945.0 / 29380423}};

struct Rk45Args {
    const double *alphas;       // viewing angles [n] (initial_conditions, metrics.py:794-809) ...
    const double *state0;       // ... or explicit initial states [n][8] (integrate_geodesic's state0)
    long long n;
    double R_S, r_obs, lambda_max, rtol, atol, max_step;
    double kerr_M, kerr_a, r_floor;   // METRIC 1; r_floor = 1.001 R_S (metrics.py:766) or 1.001 r_plus (:950)
    double r_in, r_out;         // r_out <= 0: 2 * state0[1] (geodesic_tracer.py:44-45)
    double sqrt_f0, f0;         // metrics.py:797 / :757-759, hoisted
    double *out_state;          // [n][8]
    double *out_lambda;         // [n]
    int8_t *out_outcome;        // [n]
    int32_t *out_nsteps;        // [n][2] optional: points (1 + accepted steps), nfev
    int8_t *out_status;         // [n] optional: scipy status 1 / 0 / -1, -2 for invalid
    double *traj;               // optional [n][max_points][9]
    int32_t max_points;
    int32_t *n_points;          // optional [n]
    double *dense;              // optional [n][max_points][25]: row k >= 1 = (h, Q[6][4]) of the accepted step
                                // that ended in point k — scipy's RkDenseOutput (rk.py:178-180, :715-737)
    int32_t refill_min;         // lanes that must be waiting before a flush (RK_REFILL_MIN)
    int32_t fast_pow;           // step controller: 0.9 err^-0.2 by inv_tenth_root on the squared norm instead of pow()
};

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

// METRIC 0: Schwarzschild (R_S), 1: Kerr (M, a)
template <int METRIC>
__device__ __forceinline__ void rk_f(const Rk45Args &a, double r_floor, double p_t, double p_phi,
                                     const double (&y)[RK_NC], ThetaCache &tc, double (&d)[RK_NC])
{
    if (METRIC == 0) rk_rhs(a.R_S, r_floor, p_t, p_phi, y, tc, d);
    else rk_rhs_kerr(a.kerr_M, a.kerr_a, r_floor, p_t, p_phi, y, tc, d);
}

// Quartic dense output of one component (rk.py:723-737), sequential like the oracle.
__device__ __forceinline__ double dense_comp(const double (&q)[4], double h, double y_old, double x)
{
    const double p1 = x, p2 = p1 * x, p3 = p2 * x, p4 = p3 * x;
    double s = q[0] * p1;
    s = s + q[1] * p2;
    s = s + q[2] * p3;
    s = s + q[3] * p4;
    return h * s + y_old;
}

// Row i of the dense-output coefficients Q = K^T P (rk.py:178-180).
template <int NC>
__device__ __forceinline__ void dense_q(const double (&K)[7][NC], int i, double (&q)[4])
{
#pragma unroll
    for (int m = 0; m < 4; ++m) {
        double acc = K[0][i] * c_P[0][m];
#pragma unroll
        for (int j = 2; j < 7; ++j) acc = fma(K[j][i], c_P[j][m], acc);
        q[m] = acc;
    }
}

// scipy/optimize/Zeros/brentq.c on event(t) = r(t) - r_stop, xtol = rtol = 4 EPS, 100 iterations.
__device__ __noinline__ double rk_brentq(const double (&q)[4], double h, double y_old, double t_old,
                                         double r_stop, double xa, double xb)
{
    const double tol = 4 * 2.220446049250313e-16;
#define EV(tt) (dense_comp(q, h, y_old, ((tt) - t_old) / h) - r_stop)
    double xpre = xa, xcur = xb, xblk = 0., fpre = EV(xpre), fcur = EV(xcur), fblk = 0., spre = 0., scur = 0.;
    if (fpre == 0) return xpre;
    if (fcur == 0) return xcur;
    if (signbit(fpre) == signbit(fcur)) return __longlong_as_double(0x7ff8000000000000LL);
    for (int i = 0; i < 100; ++i) {
        if (fpre != 0 && fcur != 0 && (signbit(fpre) != signbit(fcur))) {
            xblk = xpre; fblk = fpre; spre = scur = xcur - xpre;
        }
        if (fabs(fblk) < fabs(fcur)) {
            xpre = xcur; xcur = xblk; xblk = xpre;
            fpre = fcur; fcur = fblk; fblk = fpre;
        }
        const double delta = (tol + tol * fabs(xcur)) / 2;
        const double sbis = (xblk - xcur) / 2;
        if (fcur == 0 || fabs(sbis) < delta) return xcur;
        if (fabs(spre) > delta && fabs(fcur) < fabs(fpre)) {
            double stry;
            if (xpre == xblk) {
                stry = -fcur * (xcur - xpre) / (fcur - fpre);
            } else {
                const double dpre = (fpre - fcur) / (xpre - xcur);
                const double dblk = (fblk - fcur) / (xblk - xcur);
                stry = -fcur * (fblk * dblk - fpre * dpre) / (dblk * dpre * (fblk - fpre));
            }
            if (2 * fabs(stry) < fmin(fabs(spre), 3 * fabs(sbis) - delta)) { spre = scur; scur = stry; }
            else { spre = sbis; scur = sbis; }
        } else {
            spre = sbis; scur = sbis;
        }
        xpre = xcur; fpre = fcur;
        if (fabs(scur) > delta) xcur += scur;
        else xcur += (sbis > 0 ? delta : -delta);
        fcur = EV(xcur);
    }
#undef EV
    return xcur;
}

// max / min as one compare and a select (fmax / fmin expand to ~7 instructions on sm_100: no DMNMX).  A NaN in
// the SECOND operand is returned, a NaN in the first is dropped; the call sites below only ever see a NaN
// where the result is discarded or where that is the reference's behaviour (max(MIN_FACTOR, nan)).
__device__ __forceinline__ double max_sel(double a, double b) { return (a > b) ? a : b; }
__device__ __forceinline__ double min_sel(double a, double b) { return (a < b) ? a : b; }

__device__ __forceinline__ double rms8(double sumsq)     // common.py:63-65 with x.size == 8
{
    return __dsqrt_rn(sumsq) / 2.8284271247461903;       // 8 ** 0.5
}

__device__ __forceinline__ void write_point(const Rk45Args &a, long long idx, int k, double t,
                                            const double (&y)[RK_NC], double p_t, double p_phi)
{
    if (!a.traj || k >= a.max_points) return;
    double *row = a.traj + ((size_t)idx * a.max_points + k) * 9;
    row[0] = t; row[1] = y[0]; row[2] = y[1]; row[3] = y[2]; row[4] = y[3];
    row[5] = p_t; row[6] = y[4]; row[7] = y[5]; row[8] = p_phi;
}

// ---------------------------------------------------------------------------------------------
// The pieces of scipy's RK45 that every component system runs.  Scalars (rtol, atol, max_step, ...)
// come by value from the kernel's locals: re-reading them from Rk45Args changes the generated code.
// ---------------------------------------------------------------------------------------------

// Schwarzschild.initial_conditions, metrics.py:794-809: the six moving components and p_phi (p_t = -1).
// false where the reference returns None (`p_r_sq < 0`; a NaN would hang solve_ivp).
__device__ __forceinline__ bool rk_initial_conditions(const Rk45Args &a, long long ray, double (&y)[RK_NC],
                                                      double &p_phi)
{
    const double alpha = __ldg(a.alphas + ray);
    const double b = a.r_obs * lp_sin_cr(alpha) / a.sqrt_f0;
    const double L = b;
    const double p_r_sq = (1.0 / a.f0 - (L * L) / (a.r_obs * a.r_obs)) / a.f0;
    if (!(p_r_sq >= 0.0)) return false;
    y[0] = 0.0; y[1] = a.r_obs; y[2] = LP_PI_D / 2; y[3] = 0.0;
    y[4] = -__dsqrt_rn(p_r_sq); y[5] = 0.0;
    p_phi = L;
    return true;
}

// f = rhs(y) (rk.py:95) and select_initial_step (common.py:68-134, direction = +1) on the six-component state.
template <int METRIC>
__device__ __forceinline__ double rk_select_initial_step(const Rk45Args &a, double r_floor, double p_t, double p_phi,
                                                         const double (&y)[RK_NC], ThetaCache &tc, double (&f)[RK_NC],
                                                         double interval, double rtol, double atol, double max_step)
{
    rk_f<METRIC>(a, r_floor, p_t, p_phi, y, tc, f);
    double sc[RK_NC], d0s = 0.0, d1s = 0.0;
#pragma unroll
    for (int i = 0; i < RK_NC; ++i) {
        sc[i] = atol + fabs(y[i]) * rtol;
        const double v0 = y[i] / sc[i], v1 = f[i] / sc[i];
        d0s = fma(v0, v0, d0s); d1s = fma(v1, v1, d1s);
    }
    {   // the two constant components contribute to d0 only
        const double v4 = p_t / (atol + fabs(p_t) * rtol), v7 = p_phi / (atol + fabs(p_phi) * rtol);
        d0s = fma(v4, v4, d0s); d0s = fma(v7, v7, d0s);
    }
    const double d0 = rms8(d0s), d1 = rms8(d1s);
    double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
    h0 = fmin(h0, interval);
    double y1[RK_NC], f1[RK_NC], d2s = 0.0;
#pragma unroll
    for (int i = 0; i < RK_NC; ++i) y1[i] = y[i] + h0 * f[i];
    rk_f<METRIC>(a, r_floor, p_t, p_phi, y1, tc, f1);
#pragma unroll
    for (int i = 0; i < RK_NC; ++i) { const double v2 = (f1[i] - f[i]) / sc[i]; d2s = fma(v2, v2, d2s); }
    const double d2 = rms8(d2s) / h0;
    double h1;
    if (d1 <= 1e-15 && d2 <= 1e-15) h1 = fmax(1e-6, h0 * 1e-3);
    else h1 = pow(0.01 / fmax(d1, d2), 0.2);
    return fmin(fmin(100 * h0, h1), fmin(interval, max_step));
}

// The stages of one step attempt (rk_step, rk.py:14-73): K[0] = f on entry; K[1..6] and y_new on exit.
template <int NC, class Rhs>
__device__ __forceinline__ void rk_stages(double h, const double (&y)[NC], double (&K)[7][NC], double (&y_new)[NC],
                                          Rhs rhs)
{
#pragma unroll
    for (int s = 1; s < 6; ++s) {
        double ys[NC];
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            double dy = K[0][i] * c_A[s][0];
#pragma unroll
            for (int j = 1; j < s; ++j) dy = fma(K[j][i], c_A[s][j], dy);
            ys[i] = fma(dy, h, y[i]);
        }
        rhs(ys, K[s]);
    }
#pragma unroll
    for (int i = 0; i < NC; ++i) {
        double acc = K[0][i] * c_B[0];
        acc = fma(K[2][i], c_B[2], acc);
        acc = fma(K[3][i], c_B[3], acc);
        acc = fma(K[4][i], c_B[4], acc);
        acc = fma(K[5][i], c_B[5], acc);
        y_new[i] = fma(h, acc, y[i]);
    }
    rhs(y_new, K[6]);
}

// Sum of the squared scaled errors, 8 error_norm^2 (rk.py:105-109, :148-149).  The NC quotients use the
// branch-free division halves (bit-identical to `/` for finite operands, scale >= atol > 0) so their
// dependent chains interleave; anything non-finite takes the literal IEEE form.
template <int NC>
__device__ __forceinline__ double rk_error_sq(const double (&K)[7][NC], const double (&y)[NC], const double (&y_new)[NC],
                                              double h, double rtol, double atol)
{
    double esum = 0.0, en[NC], es[NC];
#pragma unroll
    for (int i = 0; i < NC; ++i) {
        es[i] = atol + max_sel(fabs(y[i]), fabs(y_new[i])) * rtol;
        double acc = K[0][i] * c_E[0];
        acc = fma(K[2][i], c_E[2], acc);
        acc = fma(K[3][i], c_E[3], acc);
        acc = fma(K[4][i], c_E[4], acc);
        acc = fma(K[5][i], c_E[5], acc);
        acc = fma(K[6][i], c_E[6], acc);
        en[i] = acc * h;
    }
#pragma unroll
    for (int i = 0; i < NC; ++i) {
        const double e = en[i] * fast_rcp(es[i]);        // es >= atol > 0; only the controller sees it
        esum = fma(e, e, esum);
    }
    if (!isfinite(esum)) {
        esum = 0.0;
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const double e = en[i] / es[i];
            esum = fma(e, e, esum);
        }
    }
    return esum;
}

// Terminal events on an accepted step (ivp.py:676-699): r falls to r_in (act0) or rises to r_out (act1).  The
// earlier root of the two by brentq on r's dense output, every component interpolated there into yf.
template <int NC>
__device__ __forceinline__ double rk_event_root(const double (&K)[7][NC], const double (&y)[NC], double t, double h,
                                                double t_new, double r_in, double r_out, bool act0, bool act1,
                                                double (&yf)[NC])
{
    double q[4];
    dense_q(K, 1, q);
    double root = 0.0;
    if (act0) root = rk_brentq(q, h, y[1], t, r_in, t, t_new);
    if (act1) {
        const double r1 = rk_brentq(q, h, y[1], t, r_out, t, t_new);
        root = (act0 && root <= r1) ? root : r1;
    }
    const double x = (root - t) / h;
#pragma unroll
    for (int i = 0; i < NC; ++i) {
        double qi[4];
        dense_q(K, i, qi);
        yf[i] = dense_comp(qi, h, y[i], x);
    }
    return root;
}

// (None, 'invalid'), geodesic_tracer.py:79-81
template <bool PATHS>
__device__ __forceinline__ void rk_write_invalid(const Rk45Args &a, long long idx)
{
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    for (int k = 0; k < 8; ++k) a.out_state[idx * 8 + k] = qnan;
    a.out_lambda[idx] = qnan;
    a.out_outcome[idx] = 0;
    if (a.out_nsteps) { a.out_nsteps[2 * idx] = 0; a.out_nsteps[2 * idx + 1] = 0; }
    if (a.out_status) a.out_status[idx] = -2;
    if (PATHS && a.n_points) a.n_points[idx] = 0;
}

// A finished ray: outcome (geodesic_tracer.py:69-70) and outputs.  y[1] is r in every system.
template <class Sys>
__device__ __forceinline__ void rk_write_result(const Rk45Args &a, const Sys &sys, long long idx,
                                                const double (&y)[Sys::NC], double t, int npts, int nfev, int status)
{
    sys.pack(y, a.out_state + idx * 8);
    a.out_lambda[idx] = t;
    a.out_outcome[idx] = (y[1] <= a.r_in * 1.1) ? -1 : 1;
    if (a.out_nsteps) { a.out_nsteps[2 * idx] = npts; a.out_nsteps[2 * idx + 1] = nfev; }
    if (a.out_status) a.out_status[idx] = (int8_t)status;
    if (Sys::PATHS && a.n_points) a.n_points[idx] = npts;
}

// ---------------------------------------------------------------------------------------------
// Component systems.  A system carries NC moving components in registers and supplies
//   start():  the initial conditions of a ray, then rk_select_initial_step; false for an invalid ray;
//   stages(): K[1..6] and y_new of one step attempt;
//   pack():   the 8-slot output state;
// and the compile-time flags PATHS (trajectory points, n_points) and DENSE (per-step interpolant rows).
// ---------------------------------------------------------------------------------------------

// The six moving components (t, r, theta, phi, p_r, p_theta) from alphas or state0, Schwarzschild or Kerr.
template <int METRIC, bool DENSE_ROWS>
struct RkSixSystem {
    static constexpr int NC = RK_NC;
    static constexpr bool PATHS = true, DENSE = DENSE_ROWS;
    double p_t, p_phi;
    ThetaCache tc;                                        // kept across the rays of the lane

    __device__ __forceinline__ RkSixSystem() : p_t(-1.0), p_phi(0.0)
    {
        tc.th = __longlong_as_double(0x7ff8000000000000LL); tc.s = 1.0; tc.c = 0.0;
    }
    __device__ __forceinline__ bool start(const Rk45Args &a, long long ray, double r_floor, double interval,
                                          double rtol, double atol, double max_step,
                                          double (&y)[NC], double (&f)[NC], double &h_abs)
    {
        if (a.state0) {                                   // integrate_geodesic(metric, state0, ...)
            const double *s0 = a.state0 + ray * 8;
            y[0] = __ldg(s0 + 0); y[1] = __ldg(s0 + 1); y[2] = __ldg(s0 + 2); y[3] = __ldg(s0 + 3);
            p_t = __ldg(s0 + 4); y[4] = __ldg(s0 + 5); y[5] = __ldg(s0 + 6); p_phi = __ldg(s0 + 7);
        } else {
            p_t = -1.0;
            if (!rk_initial_conditions(a, ray, y, p_phi)) return false;
        }
        h_abs = rk_select_initial_step<METRIC>(a, r_floor, p_t, p_phi, y, tc, f, interval, rtol, atol, max_step);
        return true;
    }
    __device__ __forceinline__ void stages(const Rk45Args &a, double r_floor, double h, const double (&y)[NC],
                                           double (&K)[7][NC], double (&y_new)[NC])
    {
        rk_stages(h, y, K, y_new, [&](const double (&ys)[NC], double (&d)[NC]) {
            rk_f<METRIC>(a, r_floor, p_t, p_phi, ys, tc, d);
        });
    }
    __device__ __forceinline__ void pack(const double (&y)[NC], double *o) const
    {
        o[0] = y[0]; o[1] = y[1]; o[2] = y[2]; o[3] = y[3];
        o[4] = p_t; o[5] = y[4]; o[6] = y[5]; o[7] = p_phi;
    }
};

// ---------------------------------------------------------------------------------------------
// Equatorial system of the batch path (the `alphas` entry: every ray starts from
// Schwarzschild.initial_conditions, metrics.py:794-809, i.e. theta = pi/2 and p_theta = 0 EXACTLY).
//
// In the reference's own integration those two components only carry rounding noise: d theta/d lambda
// = p_theta / r^2 and d p_theta/d lambda = cos(theta) p_phi^2 / (r^2 sin^3 theta) with cos(pi/2) =
// 6.1e-17, so |p_theta| stays below ~1e-15 and theta within one ulp of pi/2.  They do not feed back:
// sin^2(theta) rounds to exactly 1.0 and p_theta^2 + p_phi^2 to p_phi^2, so the right-hand side of the
// other four components (t, r, phi, p_r) is BIT-IDENTICAL with or without them; their terms of the
// error norm are ~1e-24 against a sum that is >= 1e-10 whenever the step-size factor is not clamped.
// This system therefore integrates the four live components only (28 stage values instead of 42 in
// registers, ~2/3 of the FP64 work per step attempt) and reports theta = pi/2, p_theta = 0 — within
// 3e-16 absolute of what the reference's noise integrates to.  The first-step selection is the full
// six-component arithmetic (it sees theta / scale = 1e8).  tests/test_gpu_rk45.py holds it to the
// six-component system: same accept/reject sequences, (t, r, phi, p_r) within 1e-12.
// ---------------------------------------------------------------------------------------------
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

struct RkEquatorialSystem {
    static constexpr int NC = RK_EQ;                      // (t, r, phi, p_r)
    static constexpr bool PATHS = false, DENSE = false;
    double p_t, p_phi, pp2;

    __device__ __forceinline__ RkEquatorialSystem() : p_t(-1.0), p_phi(0.0), pp2(0.0) {}
    __device__ __forceinline__ bool start(const Rk45Args &a, long long ray, double r_floor, double interval,
                                          double rtol, double atol, double max_step,
                                          double (&y)[NC], double (&f)[NC], double &h_abs)
    {
        double y6[RK_NC], f6[RK_NC];                      // the six-component state of the reference
        if (!rk_initial_conditions(a, ray, y6, p_phi)) return false;
        pp2 = p_phi * p_phi;
        ThetaCache tc;
        tc.th = __longlong_as_double(0x7ff8000000000000LL); tc.s = 1.0; tc.c = 0.0;
        h_abs = rk_select_initial_step<0>(a, r_floor, p_t, p_phi, y6, tc, f6, interval, rtol, atol, max_step);
        y[0] = y6[0]; y[1] = y6[1]; y[2] = y6[3]; y[3] = y6[4];
        f[0] = f6[0]; f[1] = f6[1]; f[2] = f6[3]; f[3] = f6[4];
        return true;
    }
    __device__ __forceinline__ void stages(const Rk45Args &a, double r_floor, double h, const double (&y)[NC],
                                           double (&K)[7][NC], double (&y_new)[NC])
    {
        int r_hi_min = 0x7fffffff;
        rk_stages(h, y, K, y_new, [&](const double (&ys)[NC], double (&d)[NC]) {
            rk_rhs_eq<true>(a.R_S, r_floor, p_t, p_phi, pp2, ys, d, r_hi_min);
        });
        // a stage at or (by less than one high word) above the floor: the tested form decides — cold
        if (r_hi_min <= __double2hiint(r_floor))
            rk_stages(h, y, K, y_new, [&](const double (&ys)[NC], double (&d)[NC]) {
                rk_rhs_eq<false>(a.R_S, r_floor, p_t, p_phi, pp2, ys, d, r_hi_min);
            });
    }
    __device__ __forceinline__ void pack(const double (&y)[NC], double *o) const
    {
        o[0] = y[0]; o[1] = y[1]; o[2] = LP_PI_D / 2; o[3] = y[2];
        o[4] = p_t; o[5] = y[3]; o[6] = 0.0; o[7] = p_phi;
    }
};

// ---------------------------------------------------------------------------------------------
// The step body: warp-queue refill, one step attempt per trip, accept / reject, finish.
// ---------------------------------------------------------------------------------------------
template <class Sys>
__device__ __forceinline__ void rk45_solve(const Rk45Args &a)
{
    constexpr int NC = Sys::NC;
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const double r_floor = a.r_floor, rtol = a.rtol, atol = a.atol;
    const double t_bound = a.lambda_max, max_step = a.max_step;

    // per-lane ray state
    Sys sys;
    bool active = false, fresh = true, rejected = false;
    long long idx = -1;
    double t = 0.0, h_abs = 0.0, g0 = 0.0, g1 = 0.0, r_out = 0.0;
    double y[NC], f[NC];
#pragma unroll
    for (int i = 0; i < NC; ++i) { y[i] = 0.0; f[i] = 0.0; }
    int npts = 0, attempts = 0;
    LpWarpQueue queue(a.n);

    while (true) {
        // ---------------- lane refill (ballot + rank) ----------------
        const unsigned idle = __ballot_sync(full, !active);
        if (idle && !queue.empty && (__popc(idle) >= a.refill_min || idle == full)) {
            const long long ray = queue.take(idle, lane);
            if (!active && ray < a.n) {
                idx = ray;
                const double interval = fabs(t_bound - 0.0);              // t starts at 0
                if (!sys.start(a, ray, r_floor, interval, rtol, atol, max_step, y, f, h_abs)) {
                    rk_write_invalid<Sys::PATHS>(a, idx);
                } else {
                    t = 0.0;
                    r_out = a.r_out > 0.0 ? a.r_out : y[1] * 2.0;
                    g0 = y[1] - a.r_in; g1 = y[1] - r_out;                        // ivp.py:650
                    npts = 1; attempts = 0; fresh = true; rejected = false;
                    if constexpr (Sys::PATHS) write_point(a, idx, 0, t, y, sys.p_t, sys.p_phi);
                    active = (interval != 0.0);
                    // zero-length interval: solve_ivp returns the initial point, status 0
                    if (!active) rk_write_result(a, sys, idx, y, t, 1, 2, 0);
                }
            }
        }
        if (!__any_sync(full, active)) {
            if (queue.empty) break;
            continue;
        }
        if (!active) continue;

        // ---------------- one step attempt (RungeKutta._step_impl, rk.py:111-176) ----------------
        const double min_step = 10 * fabs((__longlong_as_double(__double_as_longlong(t) + 1LL)) - t);
        double ha = h_abs;
        if (fresh) {
            if (ha > max_step) ha = max_step; else if (ha < min_step) ha = min_step;
            fresh = false; rejected = false;
        }
        int status = 2;                 // 2 = still running
        double t_fin = t;
        double yf[NC];
#pragma unroll
        for (int i = 0; i < NC; ++i) yf[i] = y[i];

        if (ha < min_step) {
            status = -1;                // TOO_SMALL_STEP -> solve_ivp status -1, last accepted point stays
        } else {
            double t_new = t + ha;
            if (t_new - t_bound > 0) t_new = t_bound;
            const double h = t_new - t;
            ha = fabs(h);
            attempts++;
            double K[7][NC], y_new[NC];
#pragma unroll
            for (int i = 0; i < NC; ++i) K[0][i] = f[i];
            sys.stages(a, r_floor, h, y, K, y_new);
            const double esum = rk_error_sq(K, y, y_new, h, rtol, atol);
            // one power for the accept and the reject controller (rk.py:155-170): divergent branches
            // would each run their own copy for the whole warp
            // (fast_pow: the controller on the SQUARED norm, 0.9 err^-0.2 = 0.9 (esum / 8)^-0.1 by
            // inv_tenth_root — a few ulp, the level at which scipy's own BLAS stage sums already differ
            // from any restatement; error_norm is then only compared with 0 and 1, which the square
            // preserves; tests hold the accept/reject sequences identical)
            double error_norm, pow_term;
            if (a.fast_pow) { error_norm = esum * 0.125; pow_term = 0.9 * inv_tenth_root(error_norm); }
            else { error_norm = rms8(esum); pow_term = 0.9 * pow(error_norm, -0.2); }
            if (error_norm < 1) {
                double factor = (error_norm == 0) ? 10.0 : min_sel(pow_term, 10.0);
                if (rejected) factor = min_sel(factor, 1.0);
                ha *= factor;
                // ---- accepted: events on the new point (ivp.py:676-699) ----
                const double gn0 = y_new[1] - a.r_in, gn1 = y_new[1] - r_out;
                const bool act0 = (g0 >= 0) && (gn0 <= 0);       // direction -1
                const bool act1 = (g1 <= 0) && (gn1 >= 0);       // direction +1
                t_fin = t_new;
#pragma unroll
                for (int i = 0; i < NC; ++i) yf[i] = y_new[i];
                if (t_new - t_bound >= 0) status = 0;            // OdeSolver.step: finished
                if (act0 || act1) {
                    t_fin = rk_event_root(K, y, t, h, t_new, a.r_in, r_out, act0, act1, yf);
                    status = 1;
                }
                g0 = gn0; g1 = gn1;
                if constexpr (Sys::DENSE) {
                    if (a.dense && npts < a.max_points) {
                        // the step's interpolant for OdeResult.sol: h and Q = K^T P (rk.py:178-180)
                        double *row = a.dense + ((size_t)idx * a.max_points + npts) * 25;
                        row[0] = h;
#pragma unroll
                        for (int i = 0; i < NC; ++i) {
                            double q[4];
                            dense_q(K, i, q);
#pragma unroll
                            for (int m = 0; m < 4; ++m) row[1 + 4 * i + m] = q[m];
                        }
                    }
                }
                if constexpr (Sys::PATHS) write_point(a, idx, npts, t_fin, yf, sys.p_t, sys.p_phi);
                npts++;
                t = t_new;
#pragma unroll
                for (int i = 0; i < NC; ++i) { y[i] = y_new[i]; f[i] = K[6][i]; }
                fresh = true;
            } else {
                ha *= max_sel(pow_term, 0.2);
                rejected = true;
            }
        }
        h_abs = ha;

        if (status != 2) {
            rk_write_result(a, sys, idx, yf, t_fin, npts, 2 + 6 * attempts, status);
            active = false;
        }
    }
}

template <int MINB, int METRIC, bool DENSE = false>
__global__ void __launch_bounds__(RK_BLOCK, MINB)
lp_rk45_kernel(const Rk45Args a)
{
    rk45_solve<RkSixSystem<METRIC, DENSE>>(a);
}

template <int MINB>
__global__ void __launch_bounds__(RK_BLOCK, MINB)
lp_rk45_eq_kernel(const Rk45Args a)
{
    rk45_solve<RkEquatorialSystem>(a);
}

// The RK45 tuning knobs (DESIGN.md §4), read once per process.
struct Rk45Knobs {
    int minb;       // LP_RK45_MINB = 2..4: resident CTAs per SM of the six-component kernel
    int eq_minb;    // LP_RK45_EQ_MINB = 3..6: the same for the equatorial kernel
    int refill;     // LP_RK45_REFILL = 1..32: idle lanes before a refill
    int fast_pow;   // LP_RK45_POW = 0 | 1: pow() or inv_tenth_root() in the step controller; -1 unset
    int eq;         // LP_RK45_EQ = 0 | 1: the equatorial kernel for the `alphas` batch entry
};

static int env_int(const char *name, int lo, int hi, int dflt)
{
    const char *e = getenv(name);
    const int v = e ? atoi(e) : 0;
    return (v >= lo && v <= hi) ? v : dflt;
}

static const Rk45Knobs &rk45_knobs()
{
    static const Rk45Knobs k = [] {
        Rk45Knobs r;
        // resident CTAs per SM ptxas must fit: the kernels are bound by the latency of the right-hand side's
        // dependent chains, so resident warps win until the spills start.  Six-component kernel: 2 -> 240
        // registers, no spills; 3 -> 168; 4 -> 128 (spills).  Round 1 measured 3 best on the 4K frame, which
        // that kernel then integrated; the frame now runs the equatorial kernel (4 -> 128 registers).
        r.minb = env_int("LP_RK45_MINB", 2, 4, RK_DEFAULT_MINB);
        r.eq_minb = env_int("LP_RK45_EQ_MINB", 3, 6, RK_DEFAULT_EQ_MINB);
        r.refill = env_int("LP_RK45_REFILL", 1, 32, RK_REFILL_MIN);
        const char *p = getenv("LP_RK45_POW");
        r.fast_pow = p ? (atoi(p) != 0) : -1;
        const char *e = getenv("LP_RK45_EQ");
        r.eq = e ? (atoi(e) != 0) : RK_DEFAULT_EQ;
        return r;
    }();
    return k;
}

static int rk45_launch(bool metric_is_kerr, double kerr_a, const double *alphas, const double *state0, int64_t n,
                       double M, double R_S, double r_obs,
                       double lambda_max, double rtol, double atol, double max_step,
                       double r_stop_inner, double r_stop_outer,
                       double *out_state, double *out_lambda, int8_t *out_outcome,
                       int32_t *out_nsteps, int8_t *out_status,
                       double *traj, int32_t max_points, int32_t *n_points, cudaStream_t stream,
                       double *dense = nullptr)
{
    if (n < 0 || max_points < 0) return LP_ERR_INVALID_ARG;
    if (n == 0) return LP_OK;
    if ((!alphas && !state0) || !out_state || !out_lambda || !out_outcome) return LP_ERR_INVALID_ARG;
    if (!(rtol > 0.0) || !(atol >= 0.0) || !(max_step > 0.0) || !(lambda_max >= 0.0)) return LP_ERR_INVALID_ARG;
    Rk45Args a;
    a.alphas = alphas; a.state0 = state0; a.n = n;
    a.R_S = R_S; a.r_obs = r_obs; a.lambda_max = lambda_max;
    a.kerr_M = M; a.kerr_a = kerr_a;
    // R_S carries r_plus for Kerr: capture_radius() = 1.01 r_plus (metrics.py:861-862)
    a.r_floor = R_S * 1.001;
    a.rtol = rtol < 100 * 2.220446049250313e-16 ? 100 * 2.220446049250313e-16 : rtol;   // common.py validate_tol
    a.atol = atol; a.max_step = max_step;
    a.r_in = r_stop_inner > 0.0 ? r_stop_inner : R_S * 1.01;                           // metrics.py:750-751
    a.r_out = r_stop_outer;
    a.f0 = 1 - R_S / r_obs;                                                            // metrics.py:746-748
    a.sqrt_f0 = sqrt(a.f0);
    a.out_state = out_state; a.out_lambda = out_lambda; a.out_outcome = out_outcome;
    a.out_nsteps = out_nsteps; a.out_status = out_status;
    a.traj = traj; a.max_points = max_points; a.n_points = n_points; a.dense = dense;
    const Rk45Knobs &k = rk45_knobs();
    a.refill_min = k.refill;
    const bool kerr = metric_is_kerr;
    // the equatorial four-component kernel serves the `alphas` batch entry (no trajectory, no dense output)
    const bool eq = k.eq && !kerr && !dense && alphas && !traj && !n_points;
    // fast_pow default: on in the equatorial batch kernel (4K frame 94 -> 86 ms), off in the six-component
    // kernel of the single-ray API, whose fixtures were pinned with pow()
    a.fast_pow = k.fast_pow < 0 ? eq : k.fast_pow;
    const void *fn;
    if (eq) {
        const void *eq_kernels[] = {(const void *)lp_rk45_eq_kernel<3>, (const void *)lp_rk45_eq_kernel<4>,
                                    (const void *)lp_rk45_eq_kernel<5>, (const void *)lp_rk45_eq_kernel<6>};
        fn = eq_kernels[k.eq_minb - 3];
    } else if (dense) {     // single-ray API (OdeResult.sol): the variant that also stores every step's interpolant
        fn = kerr ? (const void *)lp_rk45_kernel<2, 1, true> : (const void *)lp_rk45_kernel<2, 0, true>;
    } else if (kerr) {
        fn = (const void *)lp_rk45_kernel<2, 1>;
    } else {
        const void *six_kernels[] = {(const void *)lp_rk45_kernel<2, 0>, (const void *)lp_rk45_kernel<3, 0>,
                                     (const void *)lp_rk45_kernel<4, 0>};
        fn = six_kernels[k.minb - 2];
    }
    int grid = 0;
    const int rc = lp_grid_for(fn, RK_BLOCK, n, &grid);
    if (rc != LP_OK) return rc;
    void *args[] = {&a};
    cudaLaunchKernel(fn, grid, RK_BLOCK, args, 0, stream);
    return lp_check_launch();
}

extern "C" int lp_schw_rk45_trace_batch(const double *alphas, int64_t n,
                                        double M, double R_S, double r_obs,
                                        double lambda_max, double rtol, double atol, double max_step,
                                        double r_stop_inner, double r_stop_outer,
                                        double *out_state, double *out_lambda,
                                        int8_t *out_outcome, int32_t *out_nsteps, int8_t *out_status,
                                        void *stream)
{
    return rk45_launch(false, 0.0, alphas, nullptr, n, M, R_S, r_obs, lambda_max, rtol, atol, max_step, r_stop_inner,
                       r_stop_outer, out_state, out_lambda, out_outcome, out_nsteps, out_status,
                       nullptr, 0, nullptr, (cudaStream_t)stream);
}

extern "C" int lp_schw_rk45_trace_paths(const double *alphas, int64_t n,
                                        double M, double R_S, double r_obs,
                                        double lambda_max, double rtol, double atol, double max_step,
                                        double r_stop_inner, double r_stop_outer,
                                        double *traj, int32_t max_points, int32_t *n_points,
                                        double *out_state, double *out_lambda,
                                        int8_t *out_outcome, int32_t *out_nsteps, int8_t *out_status,
                                        void *stream)
{
    if (n > 0 && (!traj || !n_points || max_points < 1)) return LP_ERR_INVALID_ARG;
    return rk45_launch(false, 0.0, alphas, nullptr, n, M, R_S, r_obs, lambda_max, rtol, atol, max_step, r_stop_inner,
                       r_stop_outer, out_state, out_lambda, out_outcome, out_nsteps, out_status,
                       traj, max_points, n_points, (cudaStream_t)stream);
}

extern "C" int lp_schw_rk45_integrate_paths(const double *state0, int64_t n,
                                            double M, double R_S,
                                            double lambda_max, double rtol, double atol, double max_step,
                                            double r_stop_inner, double r_stop_outer,
                                            double *traj, int32_t max_points, int32_t *n_points,
                                            double *out_state, double *out_lambda,
                                            int8_t *out_outcome, int32_t *out_nsteps, int8_t *out_status,
                                            void *stream)
{
    if (n > 0 && traj && (!n_points || max_points < 1)) return LP_ERR_INVALID_ARG;
    // r_obs only feeds initial_conditions, which explicit states bypass
    return rk45_launch(false, 0.0, nullptr, state0, n, M, R_S, 4.0 * R_S, lambda_max, rtol, atol, max_step, r_stop_inner,
                       r_stop_outer, out_state, out_lambda, out_outcome, out_nsteps, out_status,
                       traj, max_points, n_points, (cudaStream_t)stream);
}

// The same for a Kerr metric (Kerr.geodesic_equations, metrics.py:946-1029): explicit initial
// states only (Kerr.initial_conditions is host arithmetic).  r_plus = M + sqrt(M^2 - a^2).
extern "C" int lp_kerr_rk45_integrate_paths(const double *state0, int64_t n,
                                            double M, double a, double r_plus,
                                            double lambda_max, double rtol, double atol, double max_step,
                                            double r_stop_inner, double r_stop_outer,
                                            double *traj, int32_t max_points, int32_t *n_points,
                                            double *out_state, double *out_lambda,
                                            int8_t *out_outcome, int32_t *out_nsteps, int8_t *out_status,
                                            void *stream)
{
    if (n > 0 && traj && (!n_points || max_points < 1)) return LP_ERR_INVALID_ARG;
    return rk45_launch(true, a, nullptr, state0, n, M, r_plus, 4.0 * r_plus, lambda_max, rtol, atol, max_step,
                       r_stop_inner, r_stop_outer, out_state, out_lambda, out_outcome, out_nsteps, out_status,
                       traj, max_points, n_points, (cudaStream_t)stream);
}

// Trajectories WITH their dense output (what solve_ivp(dense_output=True) keeps for OdeResult.sol,
// geodesic_tracer.py:57-67): as the *_paths entry points above, plus dense[n][max_points][25] —
// row k >= 1 holds (h, Q[6][4]) of the accepted step that ended in point k, Q = K^T P restricted
// to the six moving components (t, r, theta, phi, p_r, p_theta; p_t and p_phi are constants of
// the motion: their rows of Q are exactly zero).  sol(t) = y_old + h * Q @ (x, x^2, x^3, x^4),
// x = (t - t_old) / h (rk.py:723-737).  Exactly one of alphas / state0 is given; metric 0 =
// Schwarzschild (a ignored, R_S_or_r_plus = R_S), 1 = Kerr (R_S_or_r_plus = r_plus, state0 only).
extern "C" int lp_rk45_paths_dense(int32_t metric, const double *alphas, const double *state0, int64_t n,
                                   double M, double a, double R_S_or_r_plus, double r_obs,
                                   double lambda_max, double rtol, double atol, double max_step,
                                   double r_stop_inner, double r_stop_outer,
                                   double *traj, int32_t max_points, int32_t *n_points, double *dense,
                                   double *out_state, double *out_lambda,
                                   int8_t *out_outcome, int32_t *out_nsteps, int8_t *out_status,
                                   void *stream)
{
    if (metric != 0 && metric != 1) return LP_ERR_INVALID_ARG;
    if ((alphas != nullptr) == (state0 != nullptr)) return LP_ERR_INVALID_ARG;
    if (metric == 1 && alphas) return LP_ERR_UNSUPPORTED;
    if (n > 0 && (!traj || !n_points || !dense || max_points < 1)) return LP_ERR_INVALID_ARG;
    const double r_obs_used = alphas ? r_obs : 4.0 * R_S_or_r_plus;      // only feeds initial_conditions
    return rk45_launch(metric == 1, a, alphas, state0, n, M, R_S_or_r_plus, r_obs_used, lambda_max, rtol, atol,
                       max_step, r_stop_inner, r_stop_outer, out_state, out_lambda, out_outcome, out_nsteps,
                       out_status, traj, max_points, n_points, (cudaStream_t)stream, dense);
}
