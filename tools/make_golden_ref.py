"""Generates tests/golden/refback_*.npz by executing the UNMODIFIED in-tree reference helpers

    /root/reference/helper_funcs_glob/src/interp_track.py          interp_track
    /root/reference/helper_funcs_glob/src/calc_min_bound_dists.py  calc_min_bound_dists
    /root/reference/helper_funcs_glob/src/check_traj.py            check_traj   (stdout captured)
    /root/reference/helper_funcs_glob/src/export_traj_race.py      export_traj_race
    /root/reference/helper_funcs_glob/src/export_traj_ltpl.py      export_traj_ltpl
    /root/reference/helper_funcs_glob/src/import_track.py          import_track

and tests/golden/racecar_pars.json from the reference's params/racecar.ini (write_default_pars), all
imported from /root/reference in the build container -- so, unlike the tph-based rows, the fixtures of this row are
PINNED to the reference's own code.  The package's __init__ also imports prep_track / result_plots, which need
trajectory_planning_helpers and matplotlib (absent offline); both are stubbed with empty modules -- none of the functions
executed here touches them.

Inputs: the raceline of the committed fixtures (tests/golden/<name>.npz, made by tools/make_golden.py) with the velocity
profile of oracle/tph_velprofile.py, assembled into the trajectory array exactly like
/root/reference/main_globaltraj.py:501-512.

    python tools/make_golden_ref.py
"""
from __future__ import annotations

import contextlib
import io
import os
import sys
import tempfile
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)


def load_reference_helpers():
    for name in ("trajectory_planning_helpers", "matplotlib", "matplotlib.pyplot", "mpl_toolkits", "mpl_toolkits.mplot3d"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__path__ = []
            sys.modules[name] = m
    sys.modules["mpl_toolkits.mplot3d"].Axes3D = object
    sys.path.insert(0, REF)
    import helper_funcs_glob  # noqa: E402  (the reference's own package)
    return helper_funcs_glob


def write_default_pars():
    """tests/golden/racecar_pars.json: the options of params/racecar.ini that globaltraj.default_pars() restates, parsed the
    way main_globaltraj.py:160-183 parses them (configparser, then json.loads of each value)."""
    import configparser
    import json
    parser = configparser.ConfigParser()
    assert parser.read(os.path.join(REF, "params", "racecar.ini"))
    keys = {"GENERAL_OPTIONS": ("stepsize_opts", "veh_params", "vel_calc_opts"),
            "OPTIMIZATION_OPTIONS": ("optim_opts_shortest_path", "optim_opts_mincurv")}
    pars = {sec: {k: json.loads(parser.get(sec, k)) for k in ks} for sec, ks in keys.items()}
    with open(os.path.join(GOLD, "racecar_pars.json"), "w") as f:
        json.dump(pars, f, indent=1)
        f.write("\n")


def main():
    write_default_pars()
    hf = load_reference_helpers()
    from oracle import tph_velprofile as VP
    ggv_file = os.path.join(REF, "inputs", "veh_dyn_info", "ggv.csv")
    ggv, axm = VP.import_veh_dyn_info(ggv_file, os.path.join(REF, "inputs", "veh_dyn_info", "ax_max_machines.csv"))
    veh = dict(v_max=70.0, length=4.7, width=2.0, mass=1200.0, dragcoeff=0.75, curvlim=0.12)   # params/racecar.ini:44-50
    for name in ("berlin", "handling", "synth333"):
        g = np.load(os.path.join(GOLD, name + ".npz"))
        rt, nv, alpha = g["reftrack"], g["normvec"], g["alpha_mincurv"]
        kappa, el = g["rl_kappa"], g["rl_el_lengths"]
        vx = VP.calc_vel_profile(ggv=ggv, ax_max_machines=axm, v_max=veh["v_max"], kappa=kappa, el_lengths=el, closed=True,
                                 drag_coeff=veh["dragcoeff"], m_veh=veh["mass"])
        ax = VP.calc_ax_profile(np.append(vx, vx[0]), el)
        # main_globaltraj.py:501-512
        trajectory_opt = np.column_stack((g["rl_s"], g["rl_raceline_interp"], g["rl_psi"], kappa, vx, ax))
        spline_data_opt = np.column_stack((g["rl_spline_lengths"], g["rl_coeffs_x"], g["rl_coeffs_y"]))
        traj_race_cl = np.vstack((trajectory_opt, trajectory_opt[0, :]))
        traj_race_cl[-1, 0] = np.sum(spline_data_opt[:, 0])
        out = dict(trajectory_opt=trajectory_opt, traj_race_cl=traj_race_cl, length_veh=veh["length"], width_veh=veh["width"],
                   v_max=veh["v_max"], dragcoeff=veh["dragcoeff"], mass=veh["mass"], curvlim=veh["curvlim"],
                   ggv=ggv, ax_max_machines=axm)
        # interp_track on the reftrack itself (prep_track.py:32-34 uses it on the imported track) and on the bounds
        for step in (1.0, 2.5):
            out[f"interp_track_{step}"] = hf.src.interp_track.interp_track(reftrack=rt, stepsize_approx=step)
        bound_r = rt[:, :2] + nv * np.expand_dims(rt[:, 2], 1)
        bound_l = rt[:, :2] - nv * np.expand_dims(rt[:, 3], 1)
        br = hf.src.interp_track.interp_track(np.column_stack((bound_r, np.zeros((rt.shape[0], 2)))), 1.0)
        bl = hf.src.interp_track.interp_track(np.column_stack((bound_l, np.zeros((rt.shape[0], 2)))), 1.0)
        out.update(bound_r_interp=br, bound_l_interp=bl)
        # calc_min_bound_dists against the full interpolated boundaries (what check_traj intends) ...
        out["min_dists_full"] = hf.src.calc_min_bound_dists.calc_min_bound_dists(
            trajectory=trajectory_opt, bound1=br, bound2=bl, length_veh=veh["length"], width_veh=veh["width"])
        # ... and what check_traj.py:58-69 actually passes: interp_track(...)[0], i.e. the FIRST point of each boundary
        out["min_dists_as_called"] = hf.src.calc_min_bound_dists.calc_min_bound_dists(
            trajectory=trajectory_opt, bound1=br[0], bound2=bl[0], length_veh=veh["length"], width_veh=veh["width"])
        # check_traj: messages + returned boundaries, for the stock car and for limits that trigger every warning
        for tag, kw in (("stock", {}), ("tight", dict(v_max=30.0, curvlim=0.05, ggv=ggv * np.array([1.0, 0.5, 0.5]),
                                                      ax_max_machines=axm * np.array([1.0, 0.5])))):
            args = dict(reftrack=rt, reftrack_normvec_normalized=nv, length_veh=veh["length"], width_veh=veh["width"],
                        debug=True, trajectory=trajectory_opt, ggv=ggv, ax_max_machines=axm, v_max=veh["v_max"],
                        curvlim=veh["curvlim"], mass_veh=veh["mass"], dragcoeff=veh["dragcoeff"])
            args.update(kw)
            buf = io.StringIO()
            with contextlib.redirect_stdout(buf):
                b1, b2 = hf.src.check_traj.check_traj(**args)
            out[f"check_traj_{tag}_stdout"] = np.array(buf.getvalue())
            out[f"check_traj_{tag}_bound_r"], out[f"check_traj_{tag}_bound_l"] = b1, b2
            if kw:
                out["tight_ggv"], out["tight_ax_max_machines"], out["tight_v_max"], out["tight_curvlim"] = \
                    kw["ggv"], kw["ax_max_machines"], kw["v_max"], kw["curvlim"]
        # exports (first line = random UUID, dropped; second line = SHA1 of the ggv file)
        with tempfile.TemporaryDirectory() as d:
            fp = dict(ggv_file=ggv_file, traj_race_export=os.path.join(d, "race.csv"), traj_ltpl_export=os.path.join(d, "ltpl.csv"))
            hf.src.export_traj_race.export_traj_race(file_paths=fp, traj_race=traj_race_cl)
            hf.src.export_traj_ltpl.export_traj_ltpl(file_paths=fp, spline_lengths_opt=g["rl_spline_lengths"],
                                                     trajectory_opt=trajectory_opt, reftrack=rt, normvec_normalized=nv,
                                                     alpha_opt=alpha)
            for key in ("traj_race_export", "traj_ltpl_export"):
                txt = open(fp[key]).read().split("\n", 1)[1]
                out[key] = np.array(txt if name != "berlin" else txt[:20000])       # keep the fixture small
            fp2 = dict(traj_race_export=os.path.join(d, "race2.csv"))                # no ggv file: hash of an empty array
            hf.src.export_traj_race.export_traj_race(file_paths=fp2, traj_race=traj_race_cl[:3])
            out["traj_race_export_noggv"] = np.array(open(fp2["traj_race_export"]).read().split("\n", 1)[1])
        out["ggv_file_bytes"] = np.frombuffer(open(ggv_file, "rb").read(), dtype=np.uint8)
        np.savez_compressed(os.path.join(GOLD, f"refback_{name}.npz"), **out)
        print(f"  refback_{name}: traj {trajectory_opt.shape}, bounds {br.shape[0]}+{bl.shape[0]} points, "
              f"min dist full {out['min_dists_full'].min():.3f} m / as called {out['min_dists_as_called'].min():.3f} m")
        print("   ", str(out["check_traj_stock_stdout"]).strip().replace("\n", "\n    "))
        print("   ", str(out["check_traj_tight_stdout"]).strip().replace("\n", "\n    "))
    # import_track on the reference's own CSVs (3-, 4-column forms; flip / new start / laps options)
    imp = {}
    for csv, opts in (("berlin_2018", dict(flip_imp_track=False, set_new_start=False, new_start=np.array([0.0, -47.0]), num_laps=1)),
                      ("handling_track", dict(flip_imp_track=True, set_new_start=True, new_start=np.array([0.0, -47.0]), num_laps=2)),
                      ("rounded_rectangle", dict(flip_imp_track=False, set_new_start=True, new_start=np.array([10.0, 5.0]), num_laps=1)),
                      ("modena_2019", dict(flip_imp_track=False, set_new_start=False, new_start=np.array([0.0, 0.0]), num_laps=1))):
        path = os.path.join(REF, "inputs", "tracks", csv + ".csv")
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            imp[csv] = hf.src.import_track.import_track(file_path=path, imp_opts=opts, width_veh=2.0)
        imp[csv + "_csv"] = np.frombuffer(open(path, "rb").read(), dtype=np.uint8)
        imp[csv + "_stdout"] = np.array(buf.getvalue())
        imp[csv + "_opts"] = np.array([float(opts["flip_imp_track"]), float(opts["set_new_start"]), opts["new_start"][0],
                                       opts["new_start"][1], float(opts["num_laps"])])
        print(f"  import_track {csv}: {imp[csv].shape}")
    np.savez_compressed(os.path.join(GOLD, "refback_import_track.npz"), **imp)


if __name__ == "__main__":
    main()
