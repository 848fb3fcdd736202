"""CPU oracle for the Schwarzschild lensing hot path — TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
``--impl reference`` legs may import this module; the product package
(``light_path_tracer_b200``) never does and has no CPU fallback.

Two halves:

* the integrator (the reference's numba kernels, metrics.py:35-145, 661-668) is
  restated in C (``lp_oracle.c``, built by ``oracle/Makefile`` into
  ``oracle/_build/liblp_oracle.so``) and called here through ctypes;
* the numpy stages either side of it (image_lens.py:21-178, 287-397) are
  restated below with numpy, keeping the reference's operation order wherever a
  rounding could change a result.

Pinning ("parity unpinned" upstream — the reference has no tests): every
function here is checked against outputs of the UNMODIFIED reference, either
the committed fixtures in tests/golden/ (made by tests/golden/make_golden.py in
the build container) or live when /root/reference is present
(tests/test_oracle_vs_reference.py).
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "liblp_oracle.so")
_lib = None

PHI_MAX = 50.0      # metrics.py:833 (hard-coded in trace_rays_batch)
H_MAX = 0.05        # metrics.py:833
WINDING_MAX = 65535  # image_lens.py:12-13 (uint16)


def build(force=False):
    """Compile the C restatement (gcc only; a few hundred ms)."""
    srcs = [os.path.join(_HERE, f) for f in ("lp_oracle.c", "lp_oracle_rk45.c", "lp_oracle_kerr.c", "Makefile")]
    if (not force and os.path.exists(_SO)
            and all(os.path.getmtime(_SO) >= os.path.getmtime(s) for s in srcs)):
        return _SO
    subprocess.run(["make", "-C", _HERE, "-s"] + (["-B"] if force else []), check=True)
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(_SO)
        d, i64, i32, vp = ctypes.c_double, ctypes.c_int64, ctypes.c_int32, ctypes.c_void_p
        L.lp_oracle_binet_orbit.restype = ctypes.c_int
        L.lp_oracle_binet_orbit.argtypes = [d, d, d, d, d, d] + [vp] * 4
        L.lp_oracle_binet_ray.restype = ctypes.c_int
        L.lp_oracle_binet_ray.argtypes = [d, d, d, d, d, d] + [vp] * 3
        L.lp_oracle_trace_rays_batch.restype = None
        L.lp_oracle_trace_rays_batch.argtypes = [d, d, d, vp, i64, d, d, vp, vp, vp, vp]
        L.lp_oracle_trace_rays_batch_shift.restype = None
        L.lp_oracle_trace_rays_batch_shift.argtypes = [d, d, d, vp, i64, ctypes.c_int, d, d, vp, vp, vp]
        L.lp_oracle_trace_rays_batch_sin.restype = None
        L.lp_oracle_trace_rays_batch_sin.argtypes = [d, d, d, vp, vp, i64, d, d, vp, vp, vp, vp]
        L.lp_oracle_trace_frame_f32.restype = None
        L.lp_oracle_trace_frame_f32.argtypes = [d, d, d, vp, i64, d, d, vp, vp, vp, vp]
        L.lp_oracle_shadow.restype = None
        L.lp_oracle_shadow.argtypes = [ctypes.c_int, ctypes.c_int, d, d, vp]
        L.lp_oracle_num_threads.restype = ctypes.c_int
        L.lp_oracle_rk45_initial_conditions.restype = ctypes.c_int
        L.lp_oracle_rk45_initial_conditions.argtypes = [d, d, d, vp]
        L.lp_oracle_rk45_integrate.restype = ctypes.c_int
        L.lp_oracle_rk45_integrate.argtypes = [d, d, vp, d, d, d, d, d, d, vp, i32, vp, vp, vp, vp, vp]
        L.lp_oracle_rk45_trace_batch.restype = None
        L.lp_oracle_rk45_trace_batch.argtypes = [d, d, vp, i64, d, d, d, d, d, d, vp, vp, vp, vp, vp]
        L.lp_oracle_rk45_integrate_kerr.restype = ctypes.c_int
        L.lp_oracle_rk45_integrate_kerr.argtypes = [d, d, d, vp, d, d, d, d, d, d, vp, i32, vp, vp, vp, vp, vp]
        L.lp_oracle_kerr_trace_ray.restype = ctypes.c_int
        L.lp_oracle_kerr_trace_ray.argtypes = [d, d, d, d, d, d, d, d, ctypes.c_int, vp, vp, vp]
        L.lp_oracle_kerr_trace_batch.restype = None
        L.lp_oracle_kerr_trace_batch.argtypes = [d, d, d, d, vp, vp, d, d, vp, i64, vp, vp, vp, vp]
        L.lp_oracle_kerr_trace_batch_trigshift.restype = None
        L.lp_oracle_kerr_trace_batch_trigshift.argtypes = [d, d, d, d, vp, vp, d, d, vp, i64, ctypes.c_int, vp, vp, vp, vp]
        _lib = L
    return _lib


def num_threads():
    return int(lib().lp_oracle_num_threads())


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


# --------------------------------------------------------------------------
# integrator (C)
# --------------------------------------------------------------------------

def binet_orbit(M, R_S, r_obs, alpha, phi_max=PHI_MAX, h_max=H_MAX):
    """metrics.py:49-117 -> (status, phi_f, u_f, w_f, steps)."""
    phi, u, w = ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
    steps = ctypes.c_int32()
    s = lib().lp_oracle_binet_orbit(M, R_S, r_obs, alpha, phi_max, h_max,
                                    ctypes.addressof(phi), ctypes.addressof(u),
                                    ctypes.addressof(w), ctypes.addressof(steps))
    return int(s), phi.value, u.value, w.value, int(steps.value)


def binet_ray(M, R_S, r_obs, alpha, phi_max=PHI_MAX, h_max=H_MAX):
    """metrics.py:120-145 -> (status, final_alpha, n_half_orbits, steps)."""
    fa = ctypes.c_double()
    nh = ctypes.c_int64()
    steps = ctypes.c_int32()
    s = lib().lp_oracle_binet_ray(M, R_S, r_obs, alpha, phi_max, h_max,
                                  ctypes.addressof(fa), ctypes.addressof(nh),
                                  ctypes.addressof(steps))
    return int(s), fa.value, int(nh.value), int(steps.value)


def trace_rays_batch(M, r_obs, alphas, phi_max=PHI_MAX, h_max=H_MAX, R_S=None,
                     want_status=True):
    """metrics.py:661-668 / 831-833 -> (out_fa f64[n], out_w i64[n], status i8[n], steps i32[n])."""
    alphas = np.ascontiguousarray(alphas, dtype=np.float64)
    n = alphas.size
    R_S = 2 * M if R_S is None else R_S
    fa = np.empty(n, np.float64)
    w = np.empty(n, np.int64)
    st = np.empty(n, np.int8) if want_status else None
    steps = np.empty(n, np.int32) if want_status else None
    lib().lp_oracle_trace_rays_batch(M, R_S, r_obs, _p(alphas), n, phi_max, h_max,
                                     _p(fa), _p(w), _p(st), _p(steps))
    return fa, w, st, steps


def trace_rays_batch_sin_shift(M, r_obs, alphas, sin_shift, phi_max=PHI_MAX, h_max=H_MAX):
    """Sensitivity probe, not a reference path: trace_rays_batch with np.sin(alpha)
    (metrics.py:55 — the one libm-dependent input of the integration) moved by
    ``sin_shift`` ulps.  -> (out_fa, out_w, status)."""
    alphas = np.ascontiguousarray(alphas, dtype=np.float64)
    n = alphas.size
    fa = np.empty(n, np.float64)
    w = np.empty(n, np.int64)
    st = np.empty(n, np.int8)
    lib().lp_oracle_trace_rays_batch_shift(M, 2 * M, r_obs, _p(alphas), n, int(sin_shift),
                                           phi_max, h_max, _p(fa), _p(w), _p(st))
    return fa, w, st


def trace_rays_batch_sin(M, R_S, r_obs, alphas, sins, phi_max=PHI_MAX, h_max=H_MAX):
    """Sensitivity entry, not a reference path: trace_rays_batch with the caller's sin(alpha)
    (``sins``, e.g. the correctly rounded sine the GPU kernels use) in place of the host libm's
    np.sin(alpha) at metrics.py:55.  -> (out_fa f64[n], out_w i64[n], status i8[n], steps i32[n])."""
    alphas = np.ascontiguousarray(alphas, dtype=np.float64)
    sins = np.ascontiguousarray(sins, dtype=np.float64)
    assert sins.shape == alphas.shape
    n = alphas.size
    fa = np.empty(n, np.float64)
    w = np.empty(n, np.int64)
    st = np.empty(n, np.int8)
    steps = np.empty(n, np.int32)
    lib().lp_oracle_trace_rays_batch_sin(M, R_S, r_obs, _p(alphas), _p(sins), n, phi_max, h_max,
                                         _p(fa), _p(w), _p(st), _p(steps))
    return fa, w, st, steps


# --------------------------------------------------------------------------
# generic path: geodesic_tracer.trace_ray (scipy RK45 on the 8-D Hamiltonian), C
# --------------------------------------------------------------------------
RK45_DEFAULTS = dict(lambda_max=1000.0, rtol=1e-8, atol=1e-10, max_step=1.0)   # geodesic_tracer.py:22, :57-67


def rk45_initial_conditions(M, r_obs, alpha):
    """metrics.py:794-809 -> float64[8] or None."""
    s0 = np.empty(8, np.float64)
    ok = lib().lp_oracle_rk45_initial_conditions(M, r_obs, alpha, _p(s0))
    return s0 if ok else None


def rk45_trace_ray(M, r_obs, alpha, lambda_max=1000.0, r_stop_inner=None, r_stop_outer=None,
                   rtol=1e-8, atol=1e-10, max_step=1.0, max_points=4096, state0=None):
    """geodesic_tracer.trace_ray (geodesic_tracer.py:74-82) -> dict(t, y[8, n], nfev, status,
    outcome) or None for 'invalid'.  With ``state0`` (8 values): integrate_geodesic
    (geodesic_tracer.py:22-71) from that explicit state instead."""
    if state0 is not None:
        s0 = np.ascontiguousarray(state0, dtype=np.float64).copy()
    else:
        s0 = rk45_initial_conditions(M, r_obs, alpha)
    if s0 is None:
        return None
    r_in = 2 * M * 1.01 if r_stop_inner is None else r_stop_inner
    r_out = s0[1] * 2.0 if r_stop_outer is None else r_stop_outer
    traj = np.empty((max_points, 9), np.float64)
    npts, nfev, status = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
    tf = ctypes.c_double()
    yf = np.empty(8, np.float64)
    oc = lib().lp_oracle_rk45_integrate(M, 2 * M, _p(s0), lambda_max, rtol, atol, max_step, r_in, r_out,
                                        _p(traj), max_points, ctypes.addressof(npts), ctypes.addressof(nfev),
                                        ctypes.addressof(status), ctypes.addressof(tf), _p(yf))
    n = min(int(npts.value), max_points)
    return dict(t=traj[:n, 0].copy(), y=traj[:n, 1:].T.copy(), nfev=int(nfev.value),
                status=int(status.value), outcome=int(oc), n_points=int(npts.value),
                t_final=tf.value, y_final=yf, state0=s0)


def rk45_integrate_kerr(M, a, state0, lambda_max=1000.0, r_stop_inner=None, r_stop_outer=None,
                        rtol=1e-8, atol=1e-10, max_step=1.0, max_points=8192):
    """integrate_geodesic(Kerr(M, a), state0, ...) (geodesic_tracer.py:22-71 on metrics.py:946-1029)."""
    s0 = np.ascontiguousarray(state0, dtype=np.float64).copy()
    r_plus = float(kerr_r_plus(M, a))
    r_in = r_plus * 1.01 if r_stop_inner is None else r_stop_inner
    r_out = s0[1] * 2.0 if r_stop_outer is None else r_stop_outer
    traj = np.empty((max_points, 9), np.float64)
    npts, nfev, status = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
    tf = ctypes.c_double()
    yf = np.empty(8, np.float64)
    oc = lib().lp_oracle_rk45_integrate_kerr(M, a, r_plus, _p(s0), lambda_max, rtol, atol, max_step, r_in, r_out,
                                             _p(traj), max_points, ctypes.addressof(npts), ctypes.addressof(nfev),
                                             ctypes.addressof(status), ctypes.addressof(tf), _p(yf))
    n = min(int(npts.value), max_points)
    return dict(t=traj[:n, 0].copy(), y=traj[:n, 1:].T.copy(), nfev=int(nfev.value), status=int(status.value),
                outcome=int(oc), n_points=int(npts.value), t_final=tf.value, y_final=yf, state0=s0)


def rk45_trace_batch(M, r_obs, alphas, lambda_max=1000.0, rtol=1e-8, atol=1e-10, max_step=1.0,
                     r_stop_inner=0.0, r_stop_outer=0.0):
    """Batched geodesic_tracer.trace_ray -> (state f64[n,8], lambda f64[n], outcome i8[n]
    (1/-1/0 invalid), nsteps i32[n,2] = (points, nfev), status i8[n])."""
    alphas = np.ascontiguousarray(alphas, dtype=np.float64)
    n = alphas.size
    state = np.empty((n, 8), np.float64)
    lam = np.empty(n, np.float64)
    oc = np.empty(n, np.int8)
    ns = np.empty((n, 2), np.int32)
    st = np.empty(n, np.int8)
    lib().lp_oracle_rk45_trace_batch(M, r_obs, _p(alphas), n, lambda_max, rtol, atol, max_step,
                                     r_stop_inner, r_stop_outer, _p(state), _p(lam), _p(oc), _p(ns), _p(st))
    return state, lam, oc, ns, st


# --------------------------------------------------------------------------
# Kerr (metrics.py:148-567, :671-679, :840-1132), C
# --------------------------------------------------------------------------
def kerr_r_plus(M, a):
    return M + np.sqrt(M**2 - a**2)                       # metrics.py:852


def kerr_lambda_max(r_obs):
    return max(5000.0, 6.0 * r_obs)                       # metrics.py:1120, :1131


def kerr_trace_rays_batch(M, a, r_obs, alphas, thetas, theta_obs, axis_refines=None, lambda_max=None,
                          trig_shift=0):
    """Kerr.trace_rays_batch (metrics.py:1128-1132) -> (out_fa f64[n], out_w i64[n], status i8[n],
    steps i32[n, 2] = (accepted, attempts)).  ``trig_shift`` != 0 is a sensitivity probe, not a
    reference path: sin/cos(theta) in the right-hand side moved by that many ulps."""
    alphas = np.ascontiguousarray(alphas, dtype=np.float64)
    thetas = np.ascontiguousarray(thetas, dtype=np.float64)
    n = alphas.size
    ar = None if axis_refines is None else np.ascontiguousarray(axis_refines, dtype=np.uint8)
    fa = np.empty(n, np.float64)
    w = np.empty(n, np.int64)
    st = np.empty(n, np.int8)
    steps = np.empty((n, 2), np.int32)
    lam = kerr_lambda_max(r_obs) if lambda_max is None else lambda_max
    if trig_shift:
        lib().lp_oracle_kerr_trace_batch_trigshift(M, a, float(kerr_r_plus(M, a)), r_obs, _p(alphas), _p(thetas),
                                                   theta_obs, lam, _p(ar), n, int(trig_shift), _p(fa), _p(w),
                                                   _p(st), _p(steps))
    else:
        lib().lp_oracle_kerr_trace_batch(M, a, float(kerr_r_plus(M, a)), r_obs, _p(alphas), _p(thetas), theta_obs,
                                         lam, _p(ar), n, _p(fa), _p(w), _p(st), _p(steps))
    return fa, w, st, steps


def precompute_final_alpha_lookup(alpha_lookup, M, r_obs, want_status=False):
    """image_lens.py:155-178 with a Schwarzschild(M) metric:
    float32[H,W] -> (fa float32[H,W], winding uint16[H,W], n, n[, status, steps])."""
    a32 = np.ascontiguousarray(alpha_lookup, dtype=np.float32)
    n = a32.size
    fa = np.empty(a32.shape, np.float32)
    w = np.empty(a32.shape, np.uint16)
    st = np.empty(a32.shape, np.int8) if want_status else None
    steps = np.empty(a32.shape, np.int32) if want_status else None
    if n:
        lib().lp_oracle_trace_frame_f32(M, 2 * M, r_obs, _p(a32), n, PHI_MAX, H_MAX,
                                        _p(fa), _p(w), _p(st), _p(steps))
    if want_status:
        return fa, w, n, (n if n else 0), st, steps
    return fa, w, n, (n if n else 0)


def shadow_image(width, height, fov, alpha_crit):
    """black_hole_shadow.py:30-37 -> float64[width, height] of {0., 1.}."""
    img = np.empty((width, height), np.float64)
    lib().lp_oracle_shadow(width, height, fov, alpha_crit, _p(img))
    return img


# --------------------------------------------------------------------------
# Schwarzschild scalars (metrics.py:740-759)
# --------------------------------------------------------------------------

def alpha_crit(M, r_obs):
    b_crit = 3 * np.sqrt(3) * M
    arg = b_crit * np.sqrt(1 - (2 * M) / r_obs) / r_obs
    return np.arcsin(np.clip(arg, -1.0, 1.0))


# --------------------------------------------------------------------------
# camera geometry and numpy stages (image_lens.py)
# --------------------------------------------------------------------------

def psi_frame(psi):
    """image_lens.py:21-61 -> (d, e_x, e_y, in_front); psi = (pitch_up, yaw_right)."""
    pitch, yaw = psi
    d = np.array([np.sin(yaw) * np.cos(pitch), -np.sin(pitch), np.cos(yaw) * np.cos(pitch)],
                 dtype=np.float64)
    ax = np.array([1.0, 0.0, 0.0])
    ay = np.array([0.0, 1.0, 0.0])
    e_x = ax - np.dot(ax, d) * d
    nx = np.linalg.norm(e_x)
    if nx < 1e-12:
        e_x = ay - np.dot(ay, d) * d
        nx = np.linalg.norm(e_x)
    e_x /= max(nx, 1e-12)
    e_y = ay - np.dot(ay, d) * d - np.dot(ay, e_x) * e_x
    ny = np.linalg.norm(e_y)
    if ny < 1e-12:
        e_y = np.cross(d, e_x)
        ny = np.linalg.norm(e_y)
    e_y /= max(ny, 1e-12)
    return d, e_x, e_y, bool(d[2] > 1e-12)


def focal(image_dimension, fov):
    """fx, fy as image_lens.py:138-139 / 304-305."""
    h, w = image_dimension
    hf, vf = fov
    return (w / 2) / np.tan(hf / 2), (h / 2) / np.tan(vf / 2)


def build_alpha_lookup(image_dimension, fov, decimals=None, psi=(0.0, 0.0), rows=None):
    """image_lens.py:133-152 -> float32[H,W].  ``rows`` (an index array) restricts the
    output to those frame rows (bounded CPU-baseline samples; not a reference feature)."""
    h, w = image_dimension
    fx, fy = focal(image_dimension, fov)
    xc = (np.arange(w) - w / 2) / fx
    yc = ((np.arange(h) if rows is None else np.asarray(rows)) - h / 2) / fy
    d = psi_frame(psi)[0]
    norm = np.sqrt(1.0 + xc[None, :] ** 2 + yc[:, None] ** 2)
    c = ((xc[None, :] * d[0]) + (yc[:, None] * d[1]) + d[2]) / norm
    a = np.arccos(np.clip(c, -1.0, 1.0))
    if decimals is not None:
        a = np.round(a, decimals)
    return a.astype(np.float32)


WINDING_COLORS = np.array([[0.0, 0.2, 1.0], [0.0, 0.7, 1.0], [0.0, 1.0, 0.4],
                           [1.0, 1.0, 0.0], [1.0, 0.4, 0.0]], dtype=np.float32)


def render_lensed_image(source, fa_lookup, winding_lookup, fov,
                        render_loop_around=False, psi=(0.0, 0.0), return_index=False, rows=None):
    """image_lens.py:296-397 (the arguments the reference never reads —
    alpha_lookup, alpha_crit — are dropped).  With return_index=True also
    returns the int64 source index map (src_y, src_x; -1 where not sampled)."""
    H, W = source.shape[:2]
    fx, fy = focal((H, W), fov)
    if rows is None:
        out = np.zeros_like(source)
        yc = (np.arange(H) - H / 2) / fy
    else:   # row subset (bounded CPU-baseline samples): lookups / output cover those rows only
        rows = np.asarray(rows)
        out = np.zeros((rows.size,) + source.shape[1:], dtype=source.dtype)
        yc = (rows - H / 2) / fy
    xc = (np.arange(W) - W / 2) / fx
    d, e_x, e_y, _ = psi_frame(psi)
    norm = np.sqrt(1.0 + xc[None, :] ** 2 + yc[:, None] ** 2)
    vx, vy, vz = xc[None, :] / norm, yc[:, None] / norm, 1.0 / norm
    theta = np.arctan2(vx * e_x[0] + vy * e_x[1] + vz * e_x[2],
                       vx * e_y[0] + vy * e_y[1] + vz * e_y[2])
    finite = np.isfinite(fa_lookup)
    # float32 lookup vs python float: comparison happens in float32 (NEP 50)
    wind = finite & (fa_lookup > np.pi / 2)
    if wind.any():
        if winding_lookup is not None:
            k = np.clip(winding_lookup[wind], 0, len(WINDING_COLORS) - 1)
        else:
            k = np.zeros(np.count_nonzero(wind), dtype=np.intp)
        if source.ndim == 2:
            out[wind] = (WINDING_COLORS @ np.array([0.299, 0.587, 0.114], np.float32))[k]
        else:
            out[wind] = WINDING_COLORS[k]
    esc = finite & (fa_lookup <= np.pi / 2)
    sy_map = np.full(fa_lookup.shape, -1, np.int64)
    sx_map = np.full(fa_lookup.shape, -1, np.int64)
    if np.count_nonzero(esc):
        fa = fa_lookup[esc].astype(np.float64)
        th = theta[esc]
        sf, cf, st, ct = np.sin(fa), np.cos(fa), np.sin(th), np.cos(th)
        sx_ = cf * d[0] + sf * (st * e_x[0] + ct * e_y[0])
        sy_ = cf * d[1] + sf * (st * e_x[1] + ct * e_y[1])
        sz_ = cf * d[2] + sf * (st * e_x[2] + ct * e_y[2])
        front = sz_ > 1e-12
        if render_loop_around:
            qx = np.zeros_like(sx_)
            qy = np.zeros_like(sy_)
            qx[front] = sx_[front] / sz_[front]
            qy[front] = sy_[front] / sz_[front]
            ix = np.rint(qx * fx + W / 2).astype(np.intp) % W
            iy = np.rint(qy * fy + H / 2).astype(np.intp) % H
            out[esc] = source[iy, ix]
            sy_map[esc], sx_map[esc] = iy, ix
        else:
            ix = np.full(sx_.shape, -1, dtype=np.intp)
            iy = np.full(sy_.shape, -1, dtype=np.intp)
            ix[front] = np.rint(sx_[front] / sz_[front] * fx + W / 2).astype(np.intp)
            iy[front] = np.rint(sy_[front] / sz_[front] * fy + H / 2).astype(np.intp)
            ok = front & (iy >= 0) & (iy < H) & (ix >= 0) & (ix < W)
            if source.ndim == 3:
                fill = np.zeros(source.shape[2], dtype=source.dtype)
                fill[0] = 1.0
                if source.shape[2] > 2:
                    fill[2] = 1.0
            else:
                fill = source.dtype.type(1.0)
            px = np.empty((fa.shape[0],) + source.shape[2:], dtype=source.dtype)
            px[:] = fill
            px[ok] = source[iy[ok], ix[ok]]
            out[esc] = px
            ty = np.where(ok, iy, -1)
            tx = np.where(ok, ix, -1)
            sy_map[esc], sx_map[esc] = ty, tx
    if return_index:
        return out, sy_map, sx_map
    return out


def checkerboard(H, W, dtype=np.float32):
    """Synthetic source of SURVEY.md §8(d) config 2: R=((y//32+x//32)&1), G=1-R, B=x/W."""
    y = np.arange(H)[:, None]
    x = np.arange(W)[None, :]
    r = (((y // 32) + (x // 32)) & 1).astype(np.float32)
    img = np.empty((H, W, 3), np.float32)
    img[..., 0] = r
    img[..., 1] = 1.0 - r
    img[..., 2] = (x / W).astype(np.float32) * np.ones((H, 1), np.float32)
    if dtype == np.uint8:
        return np.floor(255 * img).astype(np.uint8)
    return img.astype(dtype)


def frame_stats(fa32, w16, status=None, steps=None):
    """Frame reductions (SURVEY.md §8 a16) as plain numpy."""
    finite = np.isfinite(fa32)
    out = {
        "escaped": int(np.count_nonzero(finite)),
        "winding": int(np.count_nonzero(finite & (fa32 > np.float32(np.pi / 2)))),
        "max_winding": int(w16.max()) if w16.size else 0,
    }
    if status is not None:
        out["captured"] = int(np.count_nonzero(status == -1))
        out["invalid"] = int(np.count_nonzero(status == 0))
    if steps is not None:
        out["sum_steps"] = int(steps.astype(np.int64).sum())
        out["max_steps"] = int(steps.max()) if steps.size else 0
    return out
