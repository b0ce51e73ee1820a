"""CPU tests (-m "not gpu") of the host side: the C-ABI library loads and exports every symbol declared in
include/*.h, argument validation happens before any CUDA work, the SplineSystem stand-in reproduces the
dense matrix of tph.calc_splines, and the package mirrors the tph call surface."""
import ctypes
import inspect
import os
import re

import numpy as np
import pytest

from conftest import ROOT
import global_racetrajectory_optimization_b200 as tph
from global_racetrajectory_optimization_b200 import _lib, spline_system, synth
from oracle import tph_dense as T


def _declared_symbols():
    names = set()
    inc = os.path.join(ROOT, "include")
    for fn in os.listdir(inc):
        if fn.endswith(".h"):
            txt = open(os.path.join(inc, fn)).read()
            txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
            names |= set(re.findall(r"\b(mc_[a-z0-9_]+)\s*\(", txt))
    return names


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    declared = _declared_symbols()
    assert declared, "no declarations parsed from include/*.h"
    assert declared == set(_lib.EXPORTED_SYMBOLS)
    for sym in declared:
        assert getattr(lib, sym) is not None
    assert lib.mc_version() >= 100


def test_workspace_queries_and_argument_validation_without_gpu():
    lib = _lib.load()
    assert lib.mc_mincurv_workspace_bytes(4, 1000) > 4 * 1000 * 34 * 8
    assert lib.mc_mincurv_workspace_bytes(4, 10) == 0            # below the supported minimum
    assert lib.mc_calc_splines_workspace_bytes(2, 500) % 256 == 0
    assert lib.mc_mincurv_workspace_bytes(8, 1000) - 256 == 2 * (lib.mc_mincurv_workspace_bytes(4, 1000) - 256)
    # NULL / bad arguments are rejected before any CUDA call
    assert lib.mc_calc_splines_batch(1, 100, None, None, 2, None, 1, None, None, None, None, None, 0, None) == -1
    assert b"bad argument" in lib.mc_last_error()
    assert lib.mc_mincurv_solve_batch(1, 100, None, None, None, None, 0.12, 2.0, None, None, None, None, None, None,
                                      None, 0, None) == -1
    dummy = ctypes.c_void_p(4096)
    assert lib.mc_mincurv_solve_batch(1, 10, None, dummy, dummy, dummy, 0.12, 2.0, None, dummy, dummy, None, dummy, None,
                                      None, 0, None) == -1        # n_max too small
    assert lib.mc_mincurv_solve_batch(1, 100, None, dummy, dummy, dummy, 0.12, 2.0, None, dummy, dummy, None, dummy, None,
                                      None, 0, None) == -3        # workspace too small
    assert lib.mc_create_raceline_batch(1, 100, None, dummy, 3, dummy, dummy, 2.0, 10, dummy, dummy, dummy, dummy, dummy,
                                        dummy, dummy, dummy, dummy, None, None, dummy, 1 << 30, None) == -1   # stride 3
    # velocity-profile stage: workspace = 5 interleaved vectors per profile; validation before any CUDA call
    assert lib.mc_vel_profile_workspace_bytes(3, 7, 1200) >= 3 * 7 * 5 * 1200 * 8
    assert lib.mc_vel_profile_workspace_bytes(3, 7, 1200) % 256 == 0 and lib.mc_vel_profile_workspace_bytes(0, 7, 1200) == 0
    vp = lambda **kw: lib.mc_vel_profile_batch(*[kw.get(k, d) for k, d in (
        ("B", 1), ("n_max", 100), ("n_pts", None), ("kappa", dummy), ("el", dummy), ("mu", None), ("V", 1), ("scale", None),
        ("vmb", None), ("v_max", 70.0), ("n_ggv", 4), ("ggv", dummy), ("n_mach", 4), ("mach", dummy), ("exp", 1.0),
        ("drag", 0.75), ("m", 1200.0), ("filt", 0), ("vx", None), ("ax", None), ("t", None), ("lap", dummy), ("st", None),
        ("ws", None), ("wsb", 0), ("stream", None))])
    assert vp() == -3                                              # workspace too small
    assert vp(kappa=None) == -1 and vp(lap=None) == -1 and vp(V=0) == -1 and vp(m=0.0) == -1 and vp(v_max=0.0) == -1
    assert vp(filt=4) == -1 and b"must be odd" in lib.mc_last_error()
    assert lib.mc_calc_ax_t_profile_batch(1, 100, None, dummy, 100, dummy, None, 0.0, dummy, None, None) == -1   # vx needs n + 1


def test_spline_system_materialises_the_tph_matrix():
    rt = synth.make_track(4, 90)
    path = np.vstack((rt[:, :2], rt[0, :2]))
    _, _, A, _ = T.calc_splines(path)
    el = np.sqrt(np.sum(np.diff(path, axis=0) ** 2, axis=1))
    S = spline_system.SplineSystem(el)
    assert S.shape == A.shape
    assert np.abs(np.asarray(S) - A).max() < 1e-12
    h = spline_system.h_from_system(A, 90)          # dense matrix -> scales (only ratios matter)
    assert np.allclose(h / h[0], el / el[0], rtol=1e-12)
    assert spline_system.h_from_system(S, 90) is S.h
    with pytest.raises(RuntimeError, match="wrong dimensions"):
        spline_system.h_from_system(A, 91)
    _, _, A1, _ = T.calc_splines(path, use_dist_scaling=False)
    assert np.abs(np.asarray(spline_system.SplineSystem(np.ones(90))) - A1).max() == 0.0


def test_call_surface_matches_the_reference_call_sites():
    """Keyword names used by /root/reference/main_globaltraj.py:264-290,371-387 and prep_track.py:50."""
    sig = lambda f: list(inspect.signature(f).parameters)
    assert sig(tph.calc_splines.calc_splines) == ["path", "el_lengths", "psi_s", "psi_e", "use_dist_scaling"]
    assert sig(tph.opt_min_curv.opt_min_curv)[:7] == ["reftrack", "normvectors", "A", "kappa_bound", "w_veh",
                                                       "print_debug", "plot_debug"]
    assert sig(tph.iqp_handler.iqp_handler) == ["reftrack", "normvectors", "A", "kappa_bound", "w_veh", "print_debug",
                                                "plot_debug", "stepsize_interp", "iters_min", "curv_error_allowed"]
    assert sig(tph.opt_shortest_path.opt_shortest_path) == ["reftrack", "normvectors", "w_veh", "print_debug"]
    assert sig(tph.create_raceline.create_raceline) == ["refline", "normvectors", "alpha", "stepsize_interp"]
    assert sig(tph.calc_head_curv_an.calc_head_curv_an) == ["coeffs_x", "coeffs_y", "ind_spls", "t_spls", "calc_curv",
                                                            "calc_dcurv"]
    # velocity-profile stage, /root/reference/main_globaltraj.py:211-213, :400-421 (all keyword calls)
    assert {"ggv", "ax_max_machines", "v_max", "kappa", "el_lengths", "closed", "filt_window", "dyn_model_exp", "drag_coeff",
            "m_veh"} <= set(sig(tph.calc_vel_profile.calc_vel_profile))
    assert sig(tph.calc_ax_profile.calc_ax_profile) == ["vx_profile", "el_lengths", "eq_length_output"]
    assert sig(tph.calc_t_profile.calc_t_profile) == ["vx_profile", "el_lengths", "t_start", "ax_profile"]
    assert sig(tph.import_veh_dyn_info.import_veh_dyn_info) == ["ggv_import_path", "ax_max_machines_import_path"]
    assert sig(tph.check_normals_crossing.check_normals_crossing) == ["track", "normvec_normalized", "horizon"]
    # the reference's in-tree back end, main_globaltraj.py:193-195, :520-553
    hf = tph.helper_funcs_glob.src
    assert sig(hf.import_track.import_track) == ["file_path", "imp_opts", "width_veh"]
    assert sig(hf.interp_track.interp_track) == ["reftrack", "stepsize_approx"]
    assert sig(hf.calc_min_bound_dists.calc_min_bound_dists) == ["trajectory", "bound1", "bound2", "length_veh", "width_veh"]
    assert sig(hf.check_traj.check_traj) == ["reftrack", "reftrack_normvec_normalized", "trajectory", "ggv", "ax_max_machines",
                                             "v_max", "length_veh", "width_veh", "debug", "dragcoeff", "mass_veh", "curvlim"]
    assert sig(hf.export_traj_race.export_traj_race) == ["file_paths", "traj_race"]
    assert sig(hf.export_traj_ltpl.export_traj_ltpl) == ["file_paths", "spline_lengths_opt", "trajectory_opt", "reftrack",
                                                         "normvec_normalized", "alpha_opt"]


def test_no_cpu_fallback_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    rt = synth.make_track(1, 100)
    path = np.vstack((rt[:, :2], rt[0, :2]))
    with pytest.raises(_lib.MinCurvLibError, match="no CPU fallback"):
        tph.calc_splines.calc_splines(path=path)
    with pytest.raises(RuntimeError, match="Headings must be provided"):
        tph.calc_splines.calc_splines(path=path[:-1])
    with pytest.raises(_lib.MinCurvLibError, match="no CPU fallback"):
        tph.calc_vel_profile.calc_vel_profile(ggv=np.array([[0.0, 12.0, 12.0], [80.0, 12.0, 12.0]]),
                                              ax_max_machines=np.array([[0.0, 5.0], [80.0, 5.0]]), v_max=70.0,
                                              kappa=np.full(100, 0.01), el_lengths=np.full(100, 2.0), closed=True,
                                              drag_coeff=0.75, m_veh=1200.0)
    with pytest.raises(_lib.MinCurvLibError, match="no CPU fallback"):
        tph.calc_ax_profile.calc_ax_profile(np.ones(11), np.ones(10))


def test_import_veh_dyn_info_reads_and_checks_the_tables(tmp_path):
    g = tmp_path / "ggv.csv"
    m = tmp_path / "axm.csv"
    g.write_text("# v_mps,ax_max_mps2,ay_max_mps2\n0.0,12.0,11.0\n40.0,10.0,9.5\n")
    m.write_text("# v_mps,ax_max_machines_mps2\n0.0,5.3\n")
    ggv, mach = tph.import_veh_dyn_info.import_veh_dyn_info(ggv_import_path=str(g), ax_max_machines_import_path=str(m))
    assert ggv.shape == (2, 3) and mach.shape == (1, 2) and ggv[1, 2] == 9.5 and mach[0, 1] == 5.3
    g.write_text("0.0,60.0,11.0\n")
    with pytest.raises(RuntimeError, match="ggv seems unreasonable"):
        tph.import_veh_dyn_info.import_veh_dyn_info(ggv_import_path=str(g))
    g.write_text("0.0,12.0\n")
    with pytest.raises(RuntimeError, match="three columns"):
        tph.import_veh_dyn_info.import_veh_dyn_info(ggv_import_path=str(g))


def test_synthetic_tracks_are_deterministic_and_well_posed():
    a, b = synth.make_track(7, 300), synth.make_track(7, 300)
    assert np.array_equal(a, b) and not np.array_equal(a, synth.make_track(8, 300))
    k = synth.discrete_curvature(a[:, :2])
    assert 0.02 < np.abs(k).max() < 0.25
    assert (np.maximum(a[:, 2], a[:, 3]) * np.abs(k)).max() <= 0.7 + 1e-9
    d = np.linalg.norm(np.diff(np.vstack((a[:, :2], a[0, :2])), axis=0), axis=1)
    assert d.std() / d.mean() < 0.02                  # equidistant points
    j = synth.jitter_widths(a, 3)
    assert np.array_equal(j[:, :2], a[:, :2]) and np.abs(j[:, 2:] / a[:, 2:] - 1).max() <= 0.1 + 1e-12


def test_default_pars_are_the_stock_racecar_ini_values():
    """globaltraj.default_pars() against the reference's params/racecar.ini, parsed the way main_globaltraj.py:160-183 does
    (configparser + json) and stored as tests/golden/racecar_pars.json by tools/make_golden_ref.py."""
    import json
    from global_racetrajectory_optimization_b200 import globaltraj
    with open(os.path.join(ROOT, "tests", "golden", "racecar_pars.json")) as f:
        ini = json.load(f)
    ref = {k: ini["GENERAL_OPTIONS"][k] for k in ("stepsize_opts", "veh_params", "vel_calc_opts")}
    ref["optim_opts"] = ini["OPTIMIZATION_OPTIONS"]["optim_opts_mincurv"]
    assert ini["OPTIMIZATION_OPTIONS"]["optim_opts_shortest_path"]["width_opt"] == ref["optim_opts"]["width_opt"]
    mine = globaltraj.default_pars()
    for section, values in mine.items():
        for key, val in values.items():
            assert ref[section][key] == val, (section, key)
