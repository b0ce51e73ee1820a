"""GPU tests of the closed-spline kernels (csrc/splines.cu) on every solver tier against the extended-precision
reference oracle/spline_exact.py, with the acceptance norm it defines (check_splines: coefficients 1e-12 of each
column's maximum, a0 bit-identical to the input, normal vectors 1e-13, h 4 ulp).

closed_spline() picks its path from the track size n (256 threads per block) and the capacity n_max:
  pcr4     n <= 1024           parallel cyclic reduction, 4 points per thread
  pcr8     1025 <= n <= 2048   parallel cyclic reduction, 8 points per thread
  chunked  n >= 2049           periodic LDL^T recurrences after a warm-up of TRI_WARM points
and its eight scratch vectors live in shared memory up to n_max = 3488, in the HBM workspace above.  Tracks of
fewer than 64 points run the PCR with a wrapped stride.  Run with -s to see the largest error per tier."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from global_racetrajectory_optimization_b200 import batch as B_, synth  # noqa: E402
from oracle import spline_exact as E  # noqa: E402
from oracle import tph_dense as T  # noqa: E402

UTM = 5e5
SIZES = [3, 4, 5, 7, 8, 31, 33, 64, 1024, 1025, 2048, 2049, 2366, 3488, 3489, 4100]
KINDS = ["synth", "spaced", "utm"]
MODES = ["dist", "uniform", "el"]
SMEM_N_MAX = 3488             # largest n_max whose eight scratch vectors fit the 220 KiB of shared memory


def _tier(n, n_max):
    t = "pcr4" if n <= 1024 else "pcr8" if n <= 2048 else "chunked"
    if n < 64:
        t += "-wrap"
    return t + ("/hbm" if n_max > SMEM_N_MAX else "/smem")


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


@pytest.fixture(scope="module")
def worst():
    """largest error per tier and quantity over the module; printed at the end (-s)."""
    acc = {}
    yield acc
    print("\nlargest error per tier (coef: per-column relative, normvec: absolute, h: ulp):")
    for k in sorted(acc):
        print(f"  {k:24s} " + "  ".join(f"{q} {v:.2e}" for q, v in sorted(acc[k].items())))


def _note(worst, tier, err):
    d = worst.setdefault(tier, {})
    for q in ("coef", "normvec", "h_ulp"):
        if q in err:
            d[q] = max(d.get(q, 0.0), err[q])


def _geometry(kind, n, seed=0):
    if kind == "synth":
        return synth.make_track(11 + seed, n)[:, :2]
    xy = E.spaced_track(n, seed=seed)
    return xy + UTM if kind == "utm" else xy


def _mode(xy, mode):
    if mode == "el":
        d = np.roll(xy, -1, axis=0) - xy
        return np.sqrt(d[:, 0] ** 2 + d[:, 1] ** 2) * 1.0001, True
    return None, mode == "dist"


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _host(t):
    return t.cpu().numpy()


# ------------------------------------------------------------------------------------------------
# (a) every tier boundary, three geometries, three ways of scaling the parameter
@pytest.mark.parametrize("n", SIZES)
def test_calc_splines_tier_sweep(n, worst):
    for kind in KINDS:
        xy = _geometry(kind, n)
        for mode in MODES:
            el, ds = _mode(xy, mode)
            ref = E.calc_splines_exact(xy, el, ds)
            cx, cy, nv, h = B_.calc_splines_batch(_dev(xy[None]), el_lengths=None if el is None else _dev(el[None]),
                                                  use_dist_scaling=ds)
            torch.cuda.synchronize()
            err = E.check_splines(ref, _host(cx)[0], _host(cy)[0], _host(nv)[0], _host(h)[0],
                                  what=f"n={n} {kind} {mode}")
            _note(worst, _tier(n, n), err)
            print(f"n={n:5d} {kind:6s} {mode:7s} coef {err['coef']:.2e} normvec {err['normvec']:.2e} "
                  f"h {err['h_ulp']:.0f} ulp")


# ------------------------------------------------------------------------------------------------
# (b) ragged batches on both memory paths
@pytest.mark.parametrize("n_max,counts", [(2400, [3, 700, 1024, 1025, 2048, 2049, 2400]),
                                          (3600, [3, 700, 1024, 1025, 2048, 2049, 2400, 3600])])
@pytest.mark.parametrize("use_dist_scaling", [True, False])
def test_calc_splines_ragged(n_max, counts, use_dist_scaling, worst):
    counts = counts[:3] + [2] + counts[3:]           # a degenerate row between live neighbours
    Bn = len(counts)
    rng = np.random.default_rng(n_max)
    xy = rng.uniform(-1e3, 1e3, (Bn, n_max, 2))      # garbage past n_pts[b]: must not be read
    refs = {}
    for b, n in enumerate(counts):
        if n >= 3:
            xy[b, :n] = _geometry("spaced" if b % 2 else "synth", n, seed=b)
            refs[b] = E.calc_splines_exact(xy[b, :n], use_dist_scaling=use_dist_scaling)
    n_pts = torch.tensor(counts, dtype=torch.int32)
    dxy = _dev(xy)
    cx, cy, nv, h = (_host(t) for t in B_.calc_splines_batch(dxy, n_pts=n_pts, use_dist_scaling=use_dist_scaling))
    for b, n in enumerate(counts):
        if n < 3:
            assert not cx[b].any() and not cy[b].any() and not nv[b].any() and np.all(h[b] == 1.0)
            continue
        err = E.check_splines(refs[b], cx[b, :n], cy[b, :n], nv[b, :n], h[b, :n],
                              what=f"n_max={n_max} row {b} n={n}")
        _note(worst, _tier(n, n_max), err)
        assert not cx[b, n:].any() and not cy[b, n:].any() and not nv[b, n:].any() and np.all(h[b, n:] == 1.0)
        one = B_.calc_splines_batch(dxy[b:b + 1], n_pts=n_pts[b:b + 1], use_dist_scaling=use_dist_scaling)
        for got, single in zip((cx, cy, nv, h), one):
            assert np.array_equal(got[b], _host(single)[0]), f"row {b} differs from its single-track call"


# ------------------------------------------------------------------------------------------------
# (c) create_raceline against the exact spline
def _raceline_case(n, stepsize):
    rt = synth.make_track(5, n)
    xy = rt[:, :2]
    nv = E.calc_splines_exact(xy)["normvec"]
    u = np.arange(n) / n
    amp = min(1.5, 0.05 * n * synth.STEP_M / (2.0 * np.pi))
    alpha = amp * (np.sin(2.0 * np.pi * 3.0 * u + 0.4) + 0.5 * np.cos(2.0 * np.pi * 7.0 * u))
    ref = E.create_raceline_exact(xy, nv, alpha, stepsize)
    q = ref["total"] / stepsize
    assert abs(q - round(q)) > 1e-9, "the point count would hinge on the last bits of the track length"
    return xy, nv, alpha, ref


def _wrap(d):
    d = np.mod(d, 2.0 * np.pi)
    return np.minimum(d, 2.0 * np.pi - d)


@pytest.mark.parametrize("n", [5, 1024, 1025, 2049, 2366, 3489])
def test_create_raceline_matches_exact(n, worst):
    stepsize = 2.9
    xy, nv, alpha, ref = _raceline_case(n, stepsize)
    out = B_.create_raceline_batch(_dev(xy[None]), _dev(nv[None]), _dev(alpha[None]), stepsize)
    o = {k: (_host(v)[0] if v is not None else None) for k, v in out.items()}
    m = int(o["n_out"])
    assert m == ref["n_out"]
    # (the kernel forms the raceline points with a fused multiply-add, which is what the reference rounds to)
    err = E.check_splines(ref, o["coeffs_x"], o["coeffs_y"], what=f"create_raceline n={n}")
    _note(worst, "raceline " + _tier(n, n), err)
    sl_err = np.abs(o["spline_lengths"] - ref["spline_lengths"]).max() / ref["spline_lengths"].max()
    assert sl_err <= 1e-12
    for k in ("raceline_interp", "s_interp", "el_lengths_interp"):
        assert np.abs(o[k][:m] - ref[k]).max() <= 1e-9, k
    kappa_err = np.abs(o["kappa"][:m] - ref["kappa"]).max() / np.abs(ref["kappa"]).max()
    assert kappa_err <= 1e-9
    # heading of the exact spline at the kernel's own stations: the stations themselves differ from numpy's cumsum
    # by the summation order (~3e-11 m at N = 3489), which alone would turn the heading by kappa * ds ~ 2e-12 rad
    inds, tv = o["spline_inds"][:m], o["t_values"][:m]
    psi_at = T.calc_head_curv_an(ref["coeffs_x"], ref["coeffs_y"], inds.astype(int), tv)[0]
    psi_err = _wrap(o["psi"][:m] - psi_at).max()
    assert psi_err <= 1e-12
    assert _wrap(o["psi"][:m] - ref["psi"]).max() <= 1e-10
    # spline index: equal, except at a station within 1e-9 m of a knot, where (j - 1, t ~ 1) stands for (j, t ~ 0)
    knots = np.cumsum(ref["spline_lengths"])
    for i in np.nonzero(inds != ref["spline_inds"])[0]:
        j, jr = int(inds[i]), int(ref["spline_inds"][i])
        assert abs(j - jr) == 1, (i, j, jr)
        assert np.abs(knots - ref["s_interp"][i]).min() <= 1e-9, (i, j, jr)
        t_lo, t_hi = (tv[i], ref["t_values"][i]) if j < jr else (ref["t_values"][i], tv[i])
        assert abs(t_lo - 1.0) <= 1e-9 and abs(t_hi) <= 1e-9, (i, t_lo, t_hi)
    print(f"create_raceline n={n:5d} n_out {m}: coef {err['coef']:.2e} lengths {sl_err:.2e} "
          f"kappa {kappa_err:.2e} psi {psi_err:.2e}")


# ------------------------------------------------------------------------------------------------
# (d) output capacity
def test_create_raceline_capacity_protocol():
    stepsize = 2.9
    xy, nv, alpha, ref = _raceline_case(1025, stepsize)
    args = (_dev(xy[None]), _dev(nv[None]), _dev(alpha[None]), stepsize)
    small = B_.create_raceline_batch(*args, n_out_max=ref["n_out"] - 1)
    assert int(small["n_out"][0]) == -ref["n_out"]
    derived = B_.create_raceline_batch(*args)
    cap = ref["n_out"] + 7
    fixed = B_.create_raceline_batch(*args, n_out_max=cap)
    m = int(fixed["n_out"][0])
    assert m == ref["n_out"] and int(derived["n_out"][0]) == m
    for k, v in fixed.items():
        a, d = _host(v)[0], _host(derived[k])[0]
        if k in ("coeffs_x", "coeffs_y", "spline_lengths", "n_out"):
            assert np.array_equal(a, d), k
        else:
            assert np.array_equal(a[:m], d[:m]), k
            assert not a[m:].any() and not d[m:].any(), k


# ------------------------------------------------------------------------------------------------
# (e) the launches that put the track index on gridDim.y split B into chunks of 65535
def test_head_curv_and_scale_alpha_beyond_grid_y_limit():
    Bn, n_max, ne = 65537, 4, 3
    rng = np.random.default_rng(7)
    cx = rng.normal(size=(Bn, n_max, 4))
    cy = rng.normal(size=(Bn, n_max, 4))
    cx[:, :, 1] += 3.0                                   # keep |x'| away from zero
    ind = rng.integers(0, n_max, (Bn, ne)).astype(np.int32)
    t = rng.uniform(0.0, 1.0, (Bn, ne))
    n_eval = (1 + np.arange(Bn) % ne).astype(np.int32)
    psi, kappa, dkappa = (_host(a) for a in B_.calc_head_curv_batch(_dev(cx), _dev(cy), _dev(ind), _dev(t),
                                                                     n_eval=torch.from_numpy(n_eval), calc_dcurv=True))
    flat = (np.arange(Bn)[:, None] * n_max + ind).ravel()
    rpsi, rkap, rdk = (a.reshape(Bn, ne) for a in T.calc_head_curv_an(cx.reshape(-1, 4), cy.reshape(-1, 4), flat,
                                                                       t.ravel(), calc_dcurv=True))
    live = np.arange(ne)[None, :] < n_eval[:, None]
    for rows in (slice(None), slice(65534, 65537)):
        lv = live[rows]
        assert _wrap(psi[rows] - rpsi[rows])[lv].max() <= 1e-13
        assert (np.abs(kappa[rows] - rkap[rows]) / np.abs(rkap[rows]).max())[lv].max() <= 1e-13
        assert (np.abs(dkappa[rows] - rdk[rows]) / np.abs(rdk[rows]).max())[lv].max() <= 1e-12
        assert not psi[rows][~lv].any() and not kappa[rows][~lv].any() and not dkappa[rows][~lv].any()

    alpha = rng.normal(size=(Bn, 5))
    scale = 1.0 + 1e-6 * np.arange(Bn)
    da = _dev(alpha)
    B_.scale_alpha_batch(da, _dev(scale))
    assert np.array_equal(_host(da), alpha * scale[:, None])


# ------------------------------------------------------------------------------------------------
# (f) the IQP re-linearisation: create_raceline on the chunked tier, new normal vectors on the HBM tier
def test_iqp_relinearise_big_tiers(worst):
    n, stepsize, n_max_new = 2366, 3.0, 3600
    rt = synth.make_track(21, n)
    drt = _dev(rt[None])
    _, _, nv, _ = B_.calc_splines_batch(drt)
    u = np.arange(n) / n
    alpha = 1.2 * np.sin(2.0 * np.pi * 5.0 * u + 0.3) + 0.6 * np.cos(2.0 * np.pi * 11.0 * u)
    rnew, nvnew, nnew = B_.iqp_relinearise_batch(drt, nv, _dev(alpha[None]), stepsize, n_max_new=n_max_new)
    m = int(nnew[0])
    assert 2048 < m <= n_max_new and n_max_new > SMEM_N_MAX
    rnew, nvnew = _host(rnew)[0], _host(nvnew)[0]
    rl = E.create_raceline_exact(rt[:, :2], _host(nv)[0], alpha, stepsize)
    assert m == rl["n_out"] and np.abs(rnew[:m, :2] - rl["raceline_interp"]).max() <= 1e-9
    ref = E.calc_splines_exact(rnew[:m, :2], use_dist_scaling=False)
    err = E.spline_errors(ref, ref["coeffs_x"], ref["coeffs_y"], nvnew[:m])
    assert err["normvec"] <= E.NORMVEC_ABS_TOL, err
    assert np.abs(nvnew[:m] - ref["normvec"]).max() <= E.NORMVEC_ABS_TOL
    assert not nvnew[m:].any()
    _note(worst, "iqp normvec " + _tier(m, n_max_new), {"normvec": err["normvec"]})
    print(f"iqp_relinearise: n {n} -> {m} (n_max_new {n_max_new}): normvec {err['normvec']:.2e}")
