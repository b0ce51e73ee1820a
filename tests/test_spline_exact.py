"""CPU tests of oracle/spline_exact.py, the extended-precision closed-spline reference the GPU spline tests
(tests/test_gpu_splines.py) compare against, and of the acceptance norm they share with it (check_splines).

* the reference agrees with the dense 4N x 4N restatement (tph_dense.calc_splines) and, on tiny tracks, with an
  independent 40-digit mpmath solve -- so it is the spline tph defines, in more than float64 precision;
* a float64 numpy mirror of the kernel's parallel cyclic reduction (spline_moments_pcr in csrc/splines.cu) passes
  check_splines with the kernel's step counts on every geometry the GPU tests use, including the 5e5 m offset, and
  fails it when it stops one step early -- so the norm is attainable in float64 and tight enough to catch that."""
import math

import numpy as np
import pytest

from global_racetrajectory_optimization_b200 import synth
from oracle import spline_exact as E
from oracle import tph_dense as T

UTM = 5e5


def _closed(xy):
    return np.vstack((xy, xy[:1]))


def _col_rel(got, want):
    return max(float(np.abs(got[:, c] - want[:, c]).max() / max(np.abs(want[:, c]).max(), 1e-300)) for c in range(4))


def _geometry(kind, n):
    if kind == "synth":
        return synth.make_track(11, n)[:, :2]
    xy = E.spaced_track(n)
    return xy + UTM if kind == "utm" else xy


def _mode(xy, mode):
    """(el_lengths, use_dist_scaling) of the three ways a caller scales the parameter."""
    if mode == "el":
        d = np.roll(xy, -1, axis=0) - xy
        return np.sqrt(d[:, 0] ** 2 + d[:, 1] ** 2) * 1.0001, True
    return None, mode == "dist"


# ------------------------------------------------------------------------------------------------
def test_backend_is_extended():
    assert E.BACKEND in ("longdouble", "mpmath")
    if E.BACKEND == "longdouble":
        assert np.finfo(np.longdouble).nmant >= 63
    print(f"\nspline_exact backend: {E.BACKEND}")


def _dense_refined(xy, use_dist_scaling):
    """tph_dense.calc_splines' 4N x 4N system, solved by LU and then refined once with a residual formed in extended
    precision.  With distance scaling the float64 LU solve alone loses up to ~1e-11 of the smallest coefficient
    columns on 1:1000 tracks (the scaling factors enter its rows unbalanced); the refined solve is the same
    formulation without that loss."""
    cx, cy, M, nv = T.calc_splines(_closed(xy), use_dist_scaling=use_dist_scaling)
    n = xy.shape[0]
    out = []
    for c, co in ((0, cx), (1, cy)):
        b = np.zeros(4 * n)
        b[0::4], b[1::4] = xy[:, c], np.roll(xy[:, c], -1)
        x0 = co.ravel()
        r = (b.astype(np.longdouble) - M.astype(np.longdouble) @ x0.astype(np.longdouble)).astype(float)
        out.append((x0.astype(np.longdouble) + np.linalg.solve(M, r)).astype(float).reshape(n, 4))
    return cx, cy, out[0], out[1], nv


@pytest.mark.parametrize("n", [5, 40, 200, 333])
@pytest.mark.parametrize("kind", ["synth", "spaced"])
@pytest.mark.parametrize("use_dist_scaling", [True, False])
def test_matches_dense_oracle(n, kind, use_dist_scaling):
    xy = synth.make_track(3, n)[:, :2] if kind == "synth" else E.spaced_track(n)
    if kind == "spaced":
        d = np.hypot(*(np.roll(xy, -1, axis=0) - xy).T)
        assert d.max() / d.min() >= 1000.0
    ref = E.calc_splines_exact(xy, use_dist_scaling=use_dist_scaling)
    cx, cy, rcx, rcy, nv = _dense_refined(xy, use_dist_scaling)
    assert _col_rel(rcx, ref["coeffs_x"]) <= 1e-12 and _col_rel(rcy, ref["coeffs_y"]) <= 1e-12
    if not use_dist_scaling or (kind == "synth" and n <= 200):     # where the plain float64 LU solve is that accurate
        assert _col_rel(cx, ref["coeffs_x"]) <= 1e-12 and _col_rel(cy, ref["coeffs_y"]) <= 1e-12
    assert E.spline_errors(ref, cx, cy, nv)["normvec"] <= 1e-11
    assert np.array_equal(ref["coeffs_x"][:, 0], xy[:, 0]) and np.array_equal(ref["coeffs_y"][:, 0], xy[:, 1])


def test_el_lengths_are_the_parameter_scales():
    """Supplied el_lengths replace the chord lengths (and are ignored without distance scaling), as in tph."""
    xy = synth.make_track(4, 60)[:, :2]
    el = np.linspace(2.0, 4.0, 60)
    ref = E.calc_splines_exact(xy, el_lengths=el)
    assert np.array_equal(ref["h"], el)
    # tph_dense takes n + 1 points and n lengths; its closed branch appends el[0] itself
    cx, cy, _, nv = T.calc_splines(_closed(xy), el_lengths=el)
    assert _col_rel(cx, ref["coeffs_x"]) <= 1e-12 and _col_rel(cy, ref["coeffs_y"]) <= 1e-12
    ref1 = E.calc_splines_exact(xy, el_lengths=el, use_dist_scaling=False)
    assert np.all(ref1["h"] == 1.0)
    assert np.array_equal(ref1["coeffs_x"], E.calc_splines_exact(xy, use_dist_scaling=False)["coeffs_x"])


def _mp_moments(xy, h=None):
    """Moments by a dense 40-digit LU solve of the n x n periodic system (independent of the Thomas/Sherman-Morrison
    route); h=None: chord lengths."""
    import mpmath
    ctx = mpmath.MPContext()
    ctx.dps = 40
    n = xy.shape[0]
    if h is None:
        q = [(ctx.mpf(float(a)), ctx.mpf(float(b))) for a, b in xy]
        hh = [ctx.sqrt((q[(i + 1) % n][0] - q[i][0]) ** 2 + (q[(i + 1) % n][1] - q[i][1]) ** 2) for i in range(n)]
    else:
        hh = [ctx.mpf(float(v)) for v in h]
    A = ctx.matrix(n, n)
    for i in range(n):
        A[i, i] += 2 * (hh[i - 1] + hh[i])
        A[i, (i + 1) % n] += hh[i]
        A[i, (i - 1) % n] += hh[i - 1]
    out = []
    for c in range(2):
        p = [ctx.mpf(float(v)) for v in xy[:, c]]
        r = ctx.matrix([6 * ((p[(i + 1) % n] - p[i]) / hh[i] - (p[i] - p[i - 1]) / hh[i - 1]) for i in range(n)])
        out.append(ctx.lu_solve(A, r))
    return out, ctx


def _mpf(ctx, v):
    num, den = v.as_integer_ratio() if hasattr(v, "as_integer_ratio") else (v, 1)     # exact, whatever the backend
    return ctx.mpf(num) / den


@pytest.mark.parametrize("n", [3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("kind,mode", [("synth", "dist"), ("synth", "el"), ("spaced", "uniform")])
def test_matches_mpmath(n, kind, mode):
    """The moments agree with a 40-digit solve to 1e-17 of their largest value, three orders of magnitude below
    float64 rounding.  (Distance-scaled 1:1000 tracks are left out here: their system's condition number ~1e3
    amplifies the extended-precision rounding of the right-hand side to that level in the moments of the shortest
    segments, which are multiplied by h^2 before they reach a coefficient; test_matches_dense_oracle covers them.)"""
    xy = _geometry(kind, n)
    el, ds = _mode(xy, mode)
    ref = E.calc_splines_exact(xy, el, ds)
    (mx, my), ctx = _mp_moments(xy, None if (ds and el is None) else ref["h"])
    for got, want in ((ref["mx"], mx), (ref["my"], my)):
        scale = max(abs(want[i]) for i in range(n))
        err = max(abs(_mpf(ctx, got[i]) - want[i]) for i in range(n)) / scale
        assert err <= 1e-17, (n, float(err))


# ------------------------------------------------------------------------------------------------
# float64 mirror of csrc/splines.cu (normalised equations, wrapped stride, one reciprocal per step)
def pcr_moments(h, p, s_end):
    n = h.size
    idx = np.arange(n)
    hm = np.roll(h, 1)
    w = 6.0 * (1.0 / (2.0 * (hm + h)))
    A, C = hm * w * (1.0 / 6.0), h * w * (1.0 / 6.0)
    R = w[:, None] * ((np.roll(p, -1, axis=0) - p) * (1.0 / h)[:, None] - (p - np.roll(p, 1, axis=0)) * (1.0 / hm)[:, None])
    s = 1
    while s < s_end:
        st = s % n
        im, ip = (idx - st) % n, (idx + st) % n
        w = 1.0 / (1.0 - C[im] * A - A[ip] * C)
        A, C, R = (-A[im] * A * w, -C[ip] * C * w,
                   (R - R[im] * A[:, None] - R[ip] * C[:, None]) * w[:, None])
        s <<= 1
    return R


KERNEL_S_END = {True: 64, False: 32}      # closed_spline(): six PCR steps with distance scaling, five without


def pcr_splines(xy, el_lengths, use_dist_scaling, s_end):
    d = np.roll(xy, -1, axis=0) - xy
    if not use_dist_scaling:
        h = np.ones(xy.shape[0])
    elif el_lengths is not None:
        h = np.asarray(el_lengths, dtype=float)
    else:
        h = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1])
    m = pcr_moments(h, xy, s_end)
    m1, h2 = np.roll(m, -1, axis=0), (h * h)[:, None]
    a1 = d - h2 * (2.0 * m + m1) * (1.0 / 6.0)
    a2, a3 = 0.5 * h2 * m, h2 * (m1 - m) * (1.0 / 6.0)
    cx = np.column_stack((xy[:, 0], a1[:, 0], a2[:, 0], a3[:, 0]))
    cy = np.column_stack((xy[:, 1], a1[:, 1], a2[:, 1], a3[:, 1]))
    nv = np.column_stack((a1[:, 1], -a1[:, 0])) / np.sqrt((a1 * a1).sum(axis=1))[:, None]
    return cx, cy, nv, h


@pytest.mark.parametrize("n", [3, 4, 5, 7, 8, 31, 33, 64, 500, 1024])
@pytest.mark.parametrize("kind", ["synth", "spaced", "utm"])
@pytest.mark.parametrize("mode", ["dist", "uniform", "el"])
def test_float64_pcr_mirror_passes_the_norm(n, kind, mode):
    """The kernel's algorithm in float64 meets check_splines on the geometries of the GPU sweep: the tolerances are
    attainable from float64 inputs, also 5e5 m from the origin (the point differences the spline is built from
    are exact there, so the offset costs nothing in a float64 kernel that forms them first)."""
    xy = _geometry(kind, n)
    el, ds = _mode(xy, mode)
    ref = E.calc_splines_exact(xy, el, ds)
    cx, cy, nv, h = pcr_splines(xy, el, ds, KERNEL_S_END[ds])
    E.check_splines(ref, cx, cy, nv, h, what=f"mirror {kind} n={n} {mode}")


@pytest.mark.parametrize("n", [3, 5, 33, 500, 2000])
@pytest.mark.parametrize("kind", ["synth", "spaced", "utm"])
def test_pcr_one_step_short_fails_the_norm(n, kind):
    """Halving s_end (one PCR step fewer) leaves couplings of ~3e-5 (uniform scales) in the equations: the norm
    must reject it, by a wide margin."""
    xy = _geometry(kind, n)
    ref = E.calc_splines_exact(xy, use_dist_scaling=False)
    cx, cy, nv, h = pcr_splines(xy, None, False, KERNEL_S_END[False] // 2)
    err = E.spline_errors(ref, cx, cy, nv, h)
    assert err["coef"] > 100 * E.COEF_REL_TOL, err
    with pytest.raises(AssertionError):
        E.check_splines(ref, cx, cy, nv, h)


def test_norm_catches_a_sub_ulp_h_and_moved_a0():
    xy = synth.make_track(2, 50)[:, :2]
    ref = E.calc_splines_exact(xy)
    cx, cy, nv, h = ref["coeffs_x"].copy(), ref["coeffs_y"].copy(), ref["normvec"], ref["h"]
    E.check_splines(ref, cx, cy, nv, h)
    with pytest.raises(AssertionError):
        E.check_splines(ref, cx, cy, nv, h * (1.0 + 8 * np.finfo(float).eps))
    cx[7, 0] = np.nextafter(cx[7, 0], math.inf)
    with pytest.raises(AssertionError):
        E.check_splines(ref, cx, cy, nv, h)


def test_create_raceline_exact_matches_dense_route():
    rt = synth.make_track(9, 150)
    ref = E.calc_splines_exact(rt[:, :2])
    alpha = 1.2 * np.sin(np.linspace(0.0, 6.0 * np.pi, 150, endpoint=False))
    ex = E.create_raceline_exact(rt[:, :2], ref["normvec"], alpha, 2.0)
    de = T.create_raceline(rt[:, :2], ref["normvec"], alpha, 2.0)
    assert ex["n_out"] == de[0].shape[0]
    assert _col_rel(de[2], ex["coeffs_x"]) <= 1e-12 and _col_rel(de[3], ex["coeffs_y"]) <= 1e-12
    assert np.abs(de[0] - ex["raceline_interp"]).max() <= 1e-9
    assert np.array_equal(de[4], ex["spline_inds"])
    assert np.abs(de[8] - ex["el_lengths_interp"]).max() <= 1e-9
