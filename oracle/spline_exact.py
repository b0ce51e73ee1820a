"""CPU ORACLE (test infrastructure, NOT product code) -- closed cubic splines solved in extended precision.

The dense 4N x 4N route of tph_dense.calc_splines is exact to float64 rounding but costs O(N^3) time and O(N^2)
memory, so it cannot check tracks of several thousand points.  Here the same spline is computed from its periodic
tridiagonal moment system

    h_{i-1} m_{i-1} + 2 (h_{i-1} + h_i) m_i + h_i m_{i+1} = 6 ((p_{i+1} - p_i) / h_i - (p_i - p_{i-1}) / h_{i-1})

(x and y separately, indices modulo n), solved in O(N) by the Thomas algorithm with a Sherman-Morrison correction for
the two corner entries, in extended precision throughout:

* ``np.longdouble`` where it carries at least 63 mantissa bits (x87 80-bit on x86-64, IEEE quad on aarch64 Linux);
* ``mpmath`` at 30 significant digits everywhere else (``BACKEND`` records which one is in use).

Every output is built from the extended-precision moments and rounded to float64 once, at the end, so a float64
kernel can be held to a few ulp of the true spline through its float64 inputs.

Input convention: ``xy`` holds the n distinct points of the closed track (no repeated first point; segment i runs
from p_i to p_{(i+1) mod n}), like the batched device API; ``el_lengths`` has one entry per segment.

Only tests/ may import this module.
"""
from __future__ import annotations

from fractions import Fraction

import numpy as np

from . import tph_dense as T

MPMATH_DPS = 30

if np.finfo(np.longdouble).nmant >= 63:
    BACKEND = "longdouble"
    _num = np.longdouble
    _ctx = None
else:
    import mpmath

    BACKEND = "mpmath"
    _ctx = mpmath.MPContext()
    _ctx.dps = MPMATH_DPS
    _num = _ctx.mpf


def _to_ext(a) -> np.ndarray:
    """float64 values -> array of extended-precision scalars (exact)."""
    a = np.asarray(a, dtype=np.float64)
    if _ctx is None:
        return a.astype(np.longdouble)
    return np.array([_num(float(v)) for v in a.ravel()], dtype=object).reshape(a.shape)


def _sqrt(a: np.ndarray) -> np.ndarray:
    return np.sqrt(a) if _ctx is None else np.array([_ctx.sqrt(v) for v in a], dtype=object)


def _to_f64(a: np.ndarray) -> np.ndarray:
    """extended precision -> float64, rounded to nearest."""
    return a.astype(np.float64) if _ctx is None else np.array([float(v) for v in a.ravel()]).reshape(a.shape)


def solve_periodic_moments(h: np.ndarray, rx: np.ndarray, ry: np.ndarray):
    """Solve the periodic symmetric tridiagonal system diag_i = 2 (h_{i-1} + h_i), off(i, i+1) = h_i for two right-hand
    sides.  h, rx, ry: n >= 3 extended-precision values (see _to_ext).  Returns (mx, my) in the same precision."""
    n = len(h)
    if n < 3:
        raise ValueError("a closed spline needs at least 3 points")
    h = list(h)
    b = [2 * (h[i - 1] + h[i]) for i in range(n)]
    # T = T' + u v^T with gamma = -b_0: T' is tridiagonal (no corners), u = (gamma, 0, .., 0, h_{n-1}),
    # v = (1, 0, .., 0, h_{n-1} / gamma)
    gamma = -b[0]
    b[0] = b[0] - gamma
    b[n - 1] = b[n - 1] - h[n - 1] * h[n - 1] / gamma
    zero = 0 * h[0]
    du = [zero] * n
    du[0] = gamma
    du[n - 1] = h[n - 1]
    dx, dy = list(rx), list(ry)
    # forward elimination (sub-diagonal of row i and super-diagonal of row i-1: h_{i-1})
    bp = [zero] * n
    bp[0] = b[0]
    for i in range(1, n):
        hm = h[i - 1]
        w = hm / bp[i - 1]
        bp[i] = b[i] - w * hm
        dx[i] = dx[i] - w * dx[i - 1]
        dy[i] = dy[i] - w * dy[i - 1]
        du[i] = du[i] - w * du[i - 1]
    # back substitution
    xn, yn, un = dx[n - 1] / bp[n - 1], dy[n - 1] / bp[n - 1], du[n - 1] / bp[n - 1]
    dx[n - 1], dy[n - 1], du[n - 1] = xn, yn, un
    for i in range(n - 2, -1, -1):
        hi, d = h[i], bp[i]
        xn = (dx[i] - hi * xn) / d
        yn = (dy[i] - hi * yn) / d
        un = (du[i] - hi * un) / d
        dx[i], dy[i], du[i] = xn, yn, un
    # Sherman-Morrison: m = y - z (v.y) / (1 + v.z)
    vn = h[n - 1] / gamma
    den = 1 + du[0] + vn * du[n - 1]
    fx = (dx[0] + vn * dx[n - 1]) / den
    fy = (dy[0] + vn * dy[n - 1]) / den
    dt = np.longdouble if _ctx is None else object
    du = np.array(du, dtype=dt)
    return np.array(dx, dtype=dt) - fx * du, np.array(dy, dtype=dt) - fy * du


def calc_splines_exact(xy, el_lengths=None, use_dist_scaling: bool = True) -> dict:
    """Closed spline through the n points xy [n, 2] (the closing segment is implicit).

    Parameter scales h as in tph.calc_splines: 1 without distance scaling, else el_lengths if given, else the chord
    lengths |p_{i+1} - p_i| (computed in extended precision from the float64 points).
    Returns float64 arrays coeffs_x, coeffs_y [n, 4], normvec [n, 2], h [n], plus the extended-precision moments
    mx, my and the backend name."""
    xy = np.asarray(xy, dtype=np.float64)
    if xy.ndim != 2 or xy.shape[1] < 2 or xy.shape[0] < 3:
        raise ValueError("xy must be [n >= 3, 2]")
    n = xy.shape[0]
    px, py = _to_ext(xy[:, 0]), _to_ext(xy[:, 1])
    dpx, dpy = np.roll(px, -1) - px, np.roll(py, -1) - py
    if not use_dist_scaling:
        h = _to_ext(np.ones(n))
    elif el_lengths is not None:
        h = _to_ext(el_lengths)
        if h.shape != (n,):
            raise ValueError("el_lengths must have one entry per segment (n)")
    else:
        h = _sqrt(dpx * dpx + dpy * dpy)
    hm = np.roll(h, 1)
    rx = 6 * (dpx / h - np.roll(dpx, 1) / hm)
    ry = 6 * (dpy / h - np.roll(dpy, 1) / hm)
    mx, my = solve_periodic_moments(h, rx, ry)
    mx1, my1 = np.roll(mx, -1), np.roll(my, -1)
    h2 = h * h
    ax1 = dpx - h2 * (2 * mx + mx1) / 6
    ay1 = dpy - h2 * (2 * my + my1) / 6
    norm = _sqrt(ax1 * ax1 + ay1 * ay1)
    cx = np.column_stack((xy[:, 0], _to_f64(ax1), _to_f64(h2 * mx / 2), _to_f64(h2 * (mx1 - mx) / 6)))
    cy = np.column_stack((xy[:, 1], _to_f64(ay1), _to_f64(h2 * my / 2), _to_f64(h2 * (my1 - my) / 6)))
    nv = np.column_stack((_to_f64(ay1 / norm), _to_f64(-ax1 / norm)))
    return dict(coeffs_x=cx, coeffs_y=cy, normvec=nv, h=_to_f64(h), mx=mx, my=my, backend=BACKEND)


def create_raceline_exact(refline, normvectors, alpha, stepsize_interp: float) -> dict:
    """tph.create_raceline with the closed spline (no distance scaling) from calc_splines_exact in place of the dense
    4N x 4N solve; spline lengths, resampling and heading / curvature are tph_dense's restatements.

    Returns a dict keyed like batch.create_raceline_batch's result (n_out = number of resampled points), plus
    `total` = the summed spline lengths.

    The raceline points are refline + alpha * normvectors rounded once (as a fused multiply-add does), not twice
    like numpy's separate product and sum: on a track 1 km across the second rounding moves a point by up to 1e-13 m,
    which already shows in the smallest coefficient column at the 1e-12 level."""
    refline = np.asarray(refline, dtype=np.float64)[:, :2]
    alpha = np.asarray(alpha, dtype=np.float64)
    normvectors = np.asarray(normvectors, dtype=np.float64)
    raceline = np.array([[float(Fraction(p) + Fraction(a) * Fraction(v)) for p, v in zip(row, nrow)]
                         for row, a, nrow in zip(refline.tolist(), alpha.tolist(), normvectors.tolist())])
    spl = calc_splines_exact(raceline, use_dist_scaling=False)
    cx, cy = spl["coeffs_x"], spl["coeffs_y"]
    sl = T.calc_spline_lengths(cx, cy)
    ri, inds, tv, s = T.interp_splines(cx, cy, spline_lengths=sl, incl_last_point=False, stepsize_approx=stepsize_interp)
    total = float(np.sum(sl))
    el = np.append(np.diff(s), total - s[-1])
    psi, kappa = T.calc_head_curv_an(cx, cy, inds, tv)
    return dict(coeffs_x=cx, coeffs_y=cy, spline_lengths=sl, n_out=int(ri.shape[0]), raceline_interp=ri,
                spline_inds=inds, t_values=tv, s_interp=s, el_lengths_interp=el, psi=psi, kappa=kappa, total=total)


# ----------------------------------------------------------------------------------------------
# The acceptance norm for a float64 spline kernel against calc_splines_exact, shared by the CPU tests (which also
# prove that it rejects a parallel cyclic reduction one step short) and the GPU tests.
# ----------------------------------------------------------------------------------------------
COEF_REL_TOL = 1e-12      # every coefficient column: max |got - ref| / max |ref column|
NORMVEC_ABS_TOL = 1e-13   # unit normal vectors, absolute, weighted by |a1_i| / max |a1| (see spline_errors)
H_ULP_TOL = 4             # parameter scales, in float64 ulp of the reference


def spline_errors(ref: dict, coeffs_x, coeffs_y, normvec=None, h=None) -> dict:
    """Errors of a spline (float64 arrays of n rows) against calc_splines_exact's result `ref`:

    coef     worst column of max |diff| / max |ref column| over a0..a3 of x and y;
    a0_bits  number of a0 entries that are not bit-identical to the reference (= the input points);
    normvec  max over i of |diff of normal i| * |a1_i| / max |a1|.  The normal is a1 / |a1|, so any float64
             evaluation moves it by (error of a1) / |a1_i|, and the error of a1 is only bounded relative to its
             column maximum.  Where |a1_i| is of the order of the largest (every equidistant track) this is the
             plain absolute error; on the very short segments of a 1:1000 track without distance scaling it
             discounts the conditioning of the normalisation, not the solve;
    h_ulp    max difference of the parameter scales in ulp of the reference."""
    err = {}
    worst = 0.0
    for got, want in ((coeffs_x, ref["coeffs_x"]), (coeffs_y, ref["coeffs_y"])):
        got = np.asarray(got, dtype=np.float64)
        for c in range(4):
            scale = max(np.abs(want[:, c]).max(), 1e-300)
            worst = max(worst, float(np.abs(got[:, c] - want[:, c]).max() / scale))
    err["coef"] = worst
    err["a0_bits"] = int(np.count_nonzero(np.asarray(coeffs_x)[:, 0] != ref["coeffs_x"][:, 0])
                         + np.count_nonzero(np.asarray(coeffs_y)[:, 0] != ref["coeffs_y"][:, 0]))
    if normvec is not None:
        a1 = np.hypot(ref["coeffs_x"][:, 1], ref["coeffs_y"][:, 1])
        dn = np.abs(np.asarray(normvec, dtype=np.float64) - ref["normvec"]).max(axis=1)
        err["normvec"] = float((dn * (a1 / a1.max())).max())
    if h is not None:
        err["h_ulp"] = float((np.abs(np.asarray(h) - ref["h"]) / np.spacing(ref["h"])).max())
    return err


def check_splines(ref: dict, coeffs_x, coeffs_y, normvec=None, h=None, a0_exact: bool = True, what: str = "") -> dict:
    """Assert spline_errors() within COEF_REL_TOL / NORMVEC_ABS_TOL / H_ULP_TOL (a0 bit-identical if a0_exact);
    returns the errors."""
    err = spline_errors(ref, coeffs_x, coeffs_y, normvec, h)
    bad = []
    if not err["coef"] <= COEF_REL_TOL:
        bad.append(f"coefficients {err['coef']:.3e} > {COEF_REL_TOL:.0e}")
    if a0_exact and err["a0_bits"]:
        bad.append(f"{err['a0_bits']} a0 entries differ from the input points")
    if "normvec" in err and not err["normvec"] <= NORMVEC_ABS_TOL:
        bad.append(f"normal vectors {err['normvec']:.3e} > {NORMVEC_ABS_TOL:.0e}")
    if "h_ulp" in err and not err["h_ulp"] <= H_ULP_TOL:
        bad.append(f"h {err['h_ulp']:.1f} ulp > {H_ULP_TOL}")
    assert not bad, f"{what}: " + "; ".join(bad)
    return err


def spaced_track(n: int, seed: int = 0, fine: float = 2e-4, coarse: float = 5.0) -> np.ndarray:
    """Closed test track [n, 2] with strongly non-uniform spacing: stretches of `coarse` metres alternate with
    stretches of fine * coarse metres (1:5000 by default), entered by an abrupt drop and left by a five-step
    geometric ramp; the first two segments are coarse, so even n = 3 has a 1:1000+ spacing ratio.  The centre line is
    a star-shaped curve with features of ~70 m like synth.make_track's, evaluated analytically at the arc-length
    stations (no point lies on a straight interpolation segment)."""
    rng = np.random.default_rng(1000 + n + seed)
    d = [1.0, 1.0]
    while len(d) < n:
        d += [fine] * int(rng.integers(1, 24))
        d += list(np.geomspace(fine, 1.0, 6)[1:])
        d += [1.0] * int(rng.integers(1, 8))
    d = np.array(d[:n])
    length = coarse * d.sum()
    k = np.arange(2, max(4, int(round(length / 70.0))) + 1)
    a = 0.6 * rng.uniform(0.3, 1.0, k.size) / k ** 1.5
    ph = rng.uniform(0.0, 2.0 * np.pi, k.size)

    def radius(t):
        return 1.0 + (a[:, None] * np.cos(k[:, None] * t[None, :] + ph[:, None])).sum(axis=0)

    th = np.linspace(0.0, 2.0 * np.pi, 16 * n + 4096)
    r = radius(th)
    s_dense = np.concatenate(([0.0], np.cumsum(np.hypot(np.diff(r * np.cos(th)), np.diff(r * np.sin(th))))))
    t = np.interp(np.concatenate(([0.0], np.cumsum(d)[:-1])) / d.sum() * s_dense[-1], s_dense, th)
    r = length / s_dense[-1] * radius(t)
    return np.column_stack((r * np.cos(t), r * np.sin(t)))
