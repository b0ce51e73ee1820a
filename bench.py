#!/usr/bin/env python
"""Benchmark of the batched minimum-curvature QP path (BASELINE.json metric: min-curv QPs/s, N=1000 closed tracks).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU)
    python bench.py --impl reference --steps K --warmup W    # the reference-style CPU path (oracle) on the host cores
    python bench.py --config c2|c3|c4|c5 ...                 # the other BASELINE.json configs (same JSON shape)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results as DIR/<name>.npy

One "step" = one pass of the hot path over one batch of synthetic closed tracks resident in HBM:
calc_splines -> assemble banded QP -> interior-point solve -> curvature check -> create_raceline + heading/curvature
(everything main_globaltraj.py does on its mincurv branch between prep_track and the velocity profile).
Prints ONE JSON line (rank 0).  See the task contract for the keys.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "min-curv QPs/sec (N=1000 closed track, batched)"
UNIT = "QP/s"
N_POINTS = 1000
BATCH_PER_GPU = 2368          # 4 instances per resident CTA (148 SMs x 4 CTAs)
N_BASE_LINES = 32          # distinct centre lines per rank; the rest of the batch are width-jitter variants
KAPPA_BOUND = 0.12
W_VEH = 2.0
STEP_INTERP = 2.0
ALG_BYTES_PER_POINT_K2 = 40.0      # SURVEY.md 8d: 32 B reftrack row in + 8 B alpha out
ALG_BYTES_PER_POINT_SP = 56.0      # shortest path: 32 B reftrack row + 16 B normal in, 8 B alpha out
IPM_SOURCE = os.path.join(ROOT, "global_racetrajectory_optimization_b200", "csrc", "mincurv_ipm.cu")
DUMP_LIMIT_BYTES = 64 * 10**6      # --dump-outputs: all files together

# BASELINE.json configs (configs[0] is the reference's own CPU run; c1 is the headline workload of the metric)
CONFIGS = {
    "c1": dict(n=N_POINTS, batch=BATCH_PER_GPU, what="synthetic closed tracks, mincurv (non-iterative) QP + raceline/kappa evaluation"),
    "c2": dict(n=500, batch=4096, what="Berlin FE track re-sampled to N=500, width-jitter variants generated on the device x "
                                       "vehicle-width grid 1.6..3.4 m, mincurv (non-iterative) QP, single PDIP launch"),
    "c3": dict(n=1000, batch=1024, what="iterative mincurv (iqp_handler, 5 outer iterations: 5 QPs per track) on synthetic closed tracks"),
    "c4": dict(n=2000, batch=32768, what="N=2000 sweep: vehicle-width x width-jitter grid generated on the device from 64 centre "
                                         "lines, mincurv (non-iterative) QP, chunked by free HBM"),
    "c5": dict(n=500, batch=32768, what="opt_shortest_path QP (32768 per GPU) interleaved with mincurv (4096 per GPU) on two streams"),
}


def make_inputs(batch: int, n: int, seed0: int) -> np.ndarray:
    from global_racetrajectory_optimization_b200 import synth
    base = synth.make_batch(seed0, min(N_BASE_LINES, batch), n)
    out = np.empty((batch, n, 4))
    for i in range(batch):
        out[i] = base[i] if i < len(base) else synth.jitter_widths(base[i % len(base)], seed0 + 7919 * i)
    return out


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU during the timed region (pynvml).  NVML is initialised in the
    constructor, i.e. BEFORE the timed region: nvmlInit inside the sampling thread took driver locks while the first timed
    steps were being launched (a step of 28 ms measured as 42 ms on some boxes)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt = threading.Event()
        self._nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)

            def const(new, old):
                return getattr(pynvml, new, None) or getattr(pynvml, old)
            names = {const("nvmlClocksEventReasonHwSlowdown", "nvmlClocksThrottleReasonHwSlowdown"): "hw_slowdown",
                     const("nvmlClocksEventReasonHwThermalSlowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"): "hw_thermal_slowdown",
                     const("nvmlClocksEventReasonSwThermalSlowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"): "sw_thermal_slowdown",
                     const("nvmlClocksEventReasonSwPowerCap", "nvmlClocksThrottleReasonSwPowerCap"): "sw_power_cap"}
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(pynvml, "nvmlDeviceGetCurrentClocksThrottleReasons")
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)          # first query outside the timed region too
            get_reasons(h)
            self._nv = (pynvml, h, names, get_reasons)
        except Exception as e:  # clocks are evidence, not a dependency of the measurement
            self.reasons.add(f"sampler_error:{type(e).__name__}")

    def run(self):
        if self._nv is None:
            return
        pynvml, h, names, get_reasons = self._nv
        try:
            # a few samples per timed region, not a tight poll: NVML queries take driver locks that the launching thread
            # needs too (sporadic ~100 ms gaps between launches were seen with a 20 ms poll)
            time.sleep(0.01)
            while not self._halt.is_set():
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                r = get_reasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                self._halt.wait(0.05)
        except Exception as e:
            self.reasons.add(f"sampler_error:{type(e).__name__}")

    def stop(self) -> dict:
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------
def source_sha256(path: str) -> str:
    import hashlib
    return hashlib.sha256(open(path, "rb").read()).hexdigest()


def measured_traffic():
    """DRAM bytes per QP of mincurv_pdip_kernel from the committed ncu capture -- valid only for the kernel source it was
    captured from: profiles/pdip_traffic.json carries the SHA-256 of csrc/mincurv_ipm.cu; a mismatch means the number is
    stale and `traffic` is reported as null."""
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "pdip_traffic.json")))
        if prof.get("source_sha256") != source_sha256(IPM_SOURCE):
            return None, "profiles/pdip_traffic.json was captured from a different mincurv_ipm.cu (hash mismatch): stale"
        return float(prof["dram_bytes_per_qp"]), prof.get("source", "")
    except Exception as e:
        return None, f"no traffic capture ({type(e).__name__})"


def dump_outputs(res: dict, out_dir: str, limit: int = DUMP_LIMIT_BYTES, seed: int = 0) -> None:
    """Writes the results of one step (what a caller of the path receives) as out_dir/<name>.npy in float64; integer
    results such as status and point counts convert exactly.  If the arrays together exceed `limit` bytes, each keeps the
    same fraction of its rows (instances), rows = np.sort(np.random.default_rng(seed).choice(len(a), k, replace=False)):
    the sample depends on the shapes only, and arrays of the same batch size keep the same instances, so the files of two
    builds run with the same arguments can be compared one to one."""
    arrs = {k: np.asarray(v.cpu() if hasattr(v, "cpu") else v, dtype=np.float64) for k, v in res.items()}
    budget = limit - 4096 * len(arrs)                    # (room for the .npy headers)
    total = sum(a.nbytes for a in arrs.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrs.items():
        if total > budget and a.ndim > 0:
            k = a.shape[0] * budget // total
            a = a[np.sort(np.random.default_rng(seed).choice(a.shape[0], k, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


class _Timer:
    """CUDA-event pairs on the launching stream, one pair per timed step and name."""

    def __init__(self, torch):
        self.torch, self.ev, self.on = torch, {}, False

    def span(self, name):
        t = self

        class _S:
            def __enter__(self_):
                if t.on:
                    self_.a, self_.b = t.torch.cuda.Event(enable_timing=True), t.torch.cuda.Event(enable_timing=True)
                    self_.a.record()

            def __exit__(self_, *exc):
                if t.on:
                    self_.b.record()
                    t.ev.setdefault(name, []).append((self_.a, self_.b))
        return _S()

    def mean_ms(self, name):
        p = self.ev.get(name, [])
        return float(np.mean([a.elapsed_time(b) for a, b in p])) if p else None


def build_workload(cfg_name, args, dev, rank, torch, B_, lib, _lib):
    """Returns dict(step=callable(inputs, timer) -> results, inputs (device), host_in (pinned or None), qps_per_step,
    d2h=list of result keys copied back in the e2e loop, launches_per_step, extra config facts)."""
    cfg = CONFIGS[cfg_name]
    n, bl = args.npoints or cfg["n"], args.batch or cfg["batch"]
    p, s_ = B_._ptr, B_._stream
    n_out_max = int(np.ceil(1.25 * n * 3.0 / STEP_INTERP)) + 64
    W = dict(cfg=cfg_name, n=n, batch=bl, n_out_max=n_out_max, facts={})

    if cfg_name in ("c1", "c3"):
        host = make_inputs(bl, n, seed0=10_000 + 1_000_003 * rank)
        W["host_in"] = torch.from_numpy(host).pin_memory()
        W["inputs"] = W["host_in"].to(dev)
        W["w_veh"] = W_VEH
    else:
        # sweep configs: a few centre lines on the host, the variants generated on the device from one seed each
        if cfg_name == "c2":
            base_np = np.load(os.path.join(ROOT, "tests", "golden", "berlin500_jitter_a.npz"))["reftrack"][None]
        else:
            from global_racetrajectory_optimization_b200 import synth
            base_np = synth.make_batch(20_000 + 97 * rank, 64 if cfg_name == "c4" else 32, n)
        base = torch.tensor(base_np, device=dev)
        W["base"] = base
        nsp = bl
        seeds = torch.arange(nsp, dtype=torch.int64, device=dev) + 1_000_003 * (rank + 1)
        W["seeds"] = seeds
        grid = torch.linspace(1.6, 3.4, 7, dtype=torch.float64, device=dev)
        W["w_veh"] = grid[torch.arange(nsp, device=dev) % 7].contiguous()          # vehicle-width grid of the sweep
        W["host_in"] = None
        W["inputs"] = None
        W["facts"]["inputs"] = f"{base_np.shape[0]} centre line(s) from the host, {nsp} variants generated on the device (mc_jitter_widths_batch)"
        if cfg_name == "c5":
            seeds_mc = torch.arange(4096, dtype=torch.int64, device=dev) + 77_000_003 * (rank + 1)
            W["seeds_mc"] = seeds_mc
            W["side"] = torch.cuda.Stream(device=dev)

    if cfg_name == "c1":
        ws = B_._workspace("mincurv", lib.mc_mincurv_workspace_bytes(bl, n), dev)
        # variant i is a width jitter of centre line i % N_BASE_LINES (make_inputs): H, f and k_ref depend on the centre line
        # only and are assembled once per centre line (centre_id of mc_mincurv_setup_batch_shared)
        W["centre_id"] = (torch.arange(bl, device=dev) % min(N_BASE_LINES, bl)).to(torch.int32)
        W["facts"]["shared_centre_lines"] = f"{min(N_BASE_LINES, bl)} centre lines for {bl} instances: QP matrices assembled once per centre line"

        def step(rt_dev, tm):
            with tm.span("splines"):
                cx, cy, nv, h = B_.calc_splines_batch(rt_dev, want_coeffs=False)
            Bq = rt_dev.shape[0]
            alpha = torch.empty((Bq, n), dtype=torch.float64, device=dev)
            cerr = torch.empty((Bq,), dtype=torch.float64, device=dev)
            kmax = torch.empty((Bq,), dtype=torch.float64, device=dev)
            st = torch.empty((Bq,), dtype=torch.int32, device=dev)
            iters = torch.empty((Bq,), dtype=torch.int32, device=dev)
            s = s_()
            with tm.span("setup"):
                _lib.check(lib.mc_mincurv_setup_batch_shared(Bq, n, None, p(rt_dev), p(nv), p(h), W_VEH, None, B_.F_SCALE,
                                                             p(W["centre_id"]), p(st), p(ws), ws.numel(), s), "setup")
            with tm.span("pdip"):
                _lib.check(lib.mc_mincurv_pdip_batch(Bq, n, None, p(alpha), p(st), p(iters), p(ws), ws.numel(), s), "pdip")
            _lib.check(lib.mc_mincurv_finalize_batch(Bq, n, None, p(alpha), KAPPA_BOUND, p(cerr), p(kmax), p(st), p(ws), ws.numel(), s), "finalize")
            # curvature-row phase for the instances the box-only phase flagged (none on this workload: the kernel scans
            # the status words and returns) + re-evaluation -- together the six launches of mc_mincurv_solve_batch_shared
            _lib.check(lib.mc_mincurv_kappa_batch(Bq, n, None, KAPPA_BOUND, p(alpha), p(st), p(iters), p(ws), ws.numel(), s), "kappa")
            _lib.check(lib.mc_mincurv_finalize_batch(Bq, n, None, p(alpha), KAPPA_BOUND, p(cerr), p(kmax), p(st), p(ws), ws.numel(), s), "finalize")
            with tm.span("raceline"):
                rl = B_.create_raceline_batch(rt_dev, nv, alpha, STEP_INTERP, n_out_max=n_out_max, with_head_curv=True)
            return dict(alpha=alpha, status=st, iters=iters, kappa=rl["kappa"], raceline=rl["raceline_interp"],
                        n_out=rl["n_out"], el=rl["el_lengths_interp"])
        W.update(step=step, qps_per_step=bl, launches=8)       # splines, setup, share, pdip, finalize, kappa, finalize, raceline

    elif cfg_name == "c3":
        def step(rt_dev, tm):
            with tm.span("splines"):
                cx, cy, nv, h = B_.calc_splines_batch(rt_dev, want_coeffs=False)
            with tm.span("iqp"):
                res = B_.iqp_batch(rt_dev, nv, h, KAPPA_BOUND, W_VEH, 3.0, fixed_iters=5)
            return dict(alpha=res["alpha"], status=res["status"], n_pts=res["n_pts"], qp_solves=res["qp_solves"])
        W.update(step=step, qps_per_step=5 * bl, launches=1 + 5 * 5 + 4 * 3)

    elif cfg_name in ("c2", "c4"):
        chunk = None

        def step(_unused, tm):
            # variants are generated chunk by chunk so that the N = 2000 sweep never holds more than one chunk of reftracks
            nonlocal chunk
            if chunk is None:
                per_item = lib.mc_mincurv_workspace_bytes(1, n) + 8 * n * 16
                chunk = max(1, min(bl, B_._chunk(bl, per_item, dev)))
                W["facts"]["chunk"] = chunk
            alpha = torch.empty((bl, n), dtype=torch.float64, device=dev)
            status = torch.empty((bl,), dtype=torch.int32, device=dev)
            iters = torch.empty((bl,), dtype=torch.int32, device=dev)
            for lo in range(0, bl, chunk):
                hi = min(bl, lo + chunk)
                with tm.span("jitter"):
                    rt_dev, _ = B_.jitter_widths_batch(W["base"], W["seeds"][lo:hi])
                with tm.span("splines"):
                    cx, cy, nv, h = B_.calc_splines_batch(rt_dev, want_coeffs=False)
                with tm.span("solve"):
                    cid = B_.shared_centre_ids(torch.arange(hi - lo, device=dev) % W["base"].shape[0])
                    res = B_.opt_min_curv_batch(rt_dev, nv, h, KAPPA_BOUND, W["w_veh"][lo:hi], max_chunk=hi - lo, centre_id=cid)
                alpha[lo:hi], status[lo:hi], iters[lo:hi] = res["alpha"], res["status"], res["iters"]
            return dict(alpha=alpha, status=status, iters=iters)
        W.update(step=step, qps_per_step=bl, launches=None)

    else:  # c5
        def step(_unused, tm):
            cur = torch.cuda.current_stream(dev)
            W["side"].wait_stream(cur)
            with torch.cuda.stream(W["side"]):                       # mincurv on the second stream
                rt_mc, _ = B_.jitter_widths_batch(W["base"], W["seeds_mc"])
                cx, cy, nv_mc, h_mc = B_.calc_splines_batch(rt_mc, want_coeffs=False)
                mc = B_.opt_min_curv_batch(rt_mc, nv_mc, h_mc, KAPPA_BOUND, W_VEH,
                                           centre_id=B_.shared_centre_ids(torch.arange(4096, device=dev) % W["base"].shape[0]))
            with tm.span("jitter"):
                rt_sp, _ = B_.jitter_widths_batch(W["base"], W["seeds"])
            with tm.span("splines"):
                cx, cy, nv, h = B_.calc_splines_batch(rt_sp, want_coeffs=False)
            with tm.span("shortest"):
                sp = B_.opt_shortest_path_batch(rt_sp, nv, W["w_veh"])
            cur.wait_stream(W["side"])
            return dict(alpha=sp["alpha"], status=sp["status"], iters=sp["iters"], alpha_mc=mc["alpha"], status_mc=mc["status"])
        W.update(step=step, qps_per_step=bl + 4096, launches=None)
    return W


def run_b200(args) -> dict:
    import torch
    import torch.distributed as dist
    from global_racetrajectory_optimization_b200 import _lib, batch as B_, sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs CUDA devices (no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # rank 0 must print exactly one line: some images export NCCL_DEBUG=VERSION, which makes NCCL write its banner to stdout
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    W = build_workload(args.config, args, dev, rank, torch, B_, lib, _lib)
    n, bl = W["n"], W["batch"]
    total = bl * world                                   # weak scaling: fixed work per GPU
    step, rt = W["step"], W["inputs"]
    tm = _Timer(torch)
    gather = sharding.BatchGatherer(total, n, dev) if world > 1 else None   # the single collective of the path (alpha + status)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def collect(res):
        if gather is not None:
            if gather._pending:
                gather.finish()
            gather.start(res["alpha"][:, :n].contiguous() if res["alpha"].shape[1] != n else res["alpha"], res["status"])

    # ---- device-resident measurement ("value") ----
    res = None
    for _ in range(args.warmup):
        res = step(rt, tm)                               # (the previous step's results stay alive while the next one runs,
        collect(res)                                     #  exactly as in the timed loop: the allocator's cache then holds both
                                                         #  sets of output buffers -- a cold second set cost one cudaMalloc burst
                                                         #  of ~100 ms inside the timed region in some runs)
    if gather is not None and gather._pending:
        gather.finish()
    sync_all()
    sampler = ClockSampler(local_rank)
    import gc
    gc.collect()
    gc.disable()                                         # no collector pauses between launches inside the timed region
    sampler.start()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tm.on = True
    t0.record()
    res = None
    marks, host_marks = [t0], [time.perf_counter()]
    for _ in range(args.steps):
        res = step(rt, tm)
        collect(res)                                     # gather of step k overlaps the kernels of step k + 1
        marks.append(torch.cuda.Event(enable_timing=True))
        marks[-1].record()
        host_marks.append(time.perf_counter())           # (launch-side time of the step: a gap here is a host stall)
    if gather is not None and gather._pending:
        gathered = gather.finish()                       # (the last gather ends inside the timed region)
    t1.record()
    tm.on = False
    sync_all()
    gc.enable()
    clocks = sampler.stop()
    ms_local = t0.elapsed_time(t1)
    step_ms = [round(marks[i].elapsed_time(marks[i + 1]), 3) for i in range(len(marks) - 1)]
    host_step_ms = [round(1e3 * (host_marks[i + 1] - host_marks[i]), 3) for i in range(len(host_marks) - 1)]
    tmax = torch.tensor([ms_local], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_total = float(tmax.item())
    st = res["status"].cpu().numpy()
    ok_frac = float(np.mean((st == 0) | (st == 4)))
    if "status_mc" in res:
        ok_frac = min(ok_frac, float((res["status_mc"] == 0).double().mean().item()))

    # ---- end-to-end measurement ("e2e"): through the public batched API with HOST buffers; inputs copied in and every
    #      result of the path (alpha, kappa profile, raceline x/y, point counts, status) copied out each step, on copy
    #      streams, double-buffered: the H2D of step k + 1 and the D2H of step k - 1 overlap the kernels of step k ----
    e2e = run_e2e(args, W, torch, B_, dev, world, sync_all, dist)

    qps = W["qps_per_step"] * world * args.steps / (ms_total * 1e-3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json (of measured)" if peaks else "fallback 6650 GB/s (of fallback)"

    def _k(name, bytes_per_qp, ms, count):
        if ms is None:
            return None
        gbs = bytes_per_qp * count / (ms * 1e-3) / 1e9
        return {"kernel": name, "ms": ms, "algorithmic_bytes_per_qp": bytes_per_qp, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / hbm_peak}

    cfg = args.config
    per_kernel, roof = [], None
    if cfg == "c1":
        pdip_ms, setup_ms = tm.mean_ms("pdip"), tm.mean_ms("setup")
        n_stations = float(res["n_out"].double().mean().item())
        # the two streaming kernels run ~0.1 ms per launch: inside the step their event pairs also span the wrapper's output
        # allocations and launch gaps, so they are timed here as back-to-back launches with pre-allocated outputs
        spl_ms, rl_ms = streaming_kernel_times(torch, B_, lib, _lib, rt, res["alpha"], n, W["n_out_max"], dev)
        per_kernel = [_k("calc_splines_kernel (x, y in; normals + h out: 40 B/point; back-to-back launches)", 40.0 * n, spl_ms, bl),
                      _k("mincurv_setup_kernel + mincurv_pdip_kernel", ALG_BYTES_PER_POINT_K2 * n, setup_ms + pdip_ms, bl),
                      _k("create_raceline_kernel (+ psi/kappa; 40 B in + 72 B coefficients/lengths per point, 60 B per station; back-to-back launches)", 112.0 * n + 60.0 * n_stations, rl_ms, bl)]
        alg_bytes = ALG_BYTES_PER_POINT_K2 * n * bl
        achieved = alg_bytes / (pdip_ms * 1e-3) / 1e9
        per_qp, tsrc = measured_traffic()
        traffic = per_qp * bl if per_qp else None
        roof = {"bound": "hbm", "kernel": "mincurv_pdip_kernel", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved / hbm_peak, "traffic": traffic, "traffic_source": tsrc, "peak_source": peak_src,
                "kernel_ms": pdip_ms, "setup_kernel_ms": setup_ms, "per_kernel": per_kernel,
                "algorithmic_bytes_per_launch": alg_bytes,
                "traffic_gbs": (traffic / (pdip_ms * 1e-3) / 1e9) if traffic else None,
                "traffic_frac_of_peak": (traffic / (pdip_ms * 1e-3) / 1e9 / hbm_peak) if traffic else None,
                "note": "algorithmic bytes = 40 B/point (SURVEY 8d). The kernel streams its bordered LDL^T factor (written "
                        "once, read three times per interior-point iteration): traffic >> algorithmic bytes by construction; "
                        "see DESIGN.md section 5 for what bounds it"}
    else:
        names = {"c2": [("jitter_widths_kernel", 32.0 * n, "jitter"), ("calc_splines_kernel", 96.0 * n, "splines"),
                        ("mincurv_setup + pdip + finalize kernels (mc_mincurv_solve_batch)", ALG_BYTES_PER_POINT_K2 * n, "solve")],
                 "c4": [("jitter_widths_kernel", 32.0 * n, "jitter"), ("calc_splines_kernel", 96.0 * n, "splines"),
                        ("mincurv_setup + pdip + finalize kernels (mc_mincurv_solve_batch)", ALG_BYTES_PER_POINT_K2 * n, "solve")],
                 "c3": [("calc_splines_kernel", 96.0 * n, "splines"),
                        ("5 x (mincurv solve + create_raceline + iqp_new_reftrack + calc_splines): iqp_batch", 5 * ALG_BYTES_PER_POINT_K2 * n, "iqp")],
                 "c5": [("jitter_widths_kernel", 32.0 * n, "jitter"), ("calc_splines_kernel", 96.0 * n, "splines"),
                        ("shortest_path_kernel (mincurv running on the second stream)", ALG_BYTES_PER_POINT_SP * n, "shortest")]}[cfg]
        for nm, bq, key in names:
            ms = tm.mean_ms(key)
            if ms is not None and cfg in ("c2", "c4"):
                ms *= -(-bl // max(W["facts"].get("chunk", bl), 1))          # events are per chunk: per-step time = chunks x mean
            e = _k(nm, bq, ms, bl)
            if e:
                per_kernel.append(e)
        dom = per_kernel[-1]
        roof = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved_gbs"], "peak": hbm_peak, "unit": "GB/s",
                "frac": dom["frac_of_hbm_peak"], "traffic": None, "peak_source": peak_src, "per_kernel": per_kernel}

    iters_mean = float(res["iters"].double().mean().item()) if "iters" in res else None
    line = {
        "metric": METRIC if cfg == "c1" else f"QPs/sec, BASELINE.json config {cfg}", "value": qps, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "step_ms": step_ms, "host_launch_ms": host_step_ms,
        "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"batch {bl} per GPU: " + CONFIGS[cfg]["what"] + f", N={n} points",
                   "baseline_config": cfg, "global_batch": total, "n_points": n, "kappa_bound": KAPPA_BOUND,
                   "w_veh": W_VEH if not hasattr(W["w_veh"], "shape") else "grid 1.6..3.4 m (7 values)",
                   "qps_per_step_per_gpu": W["qps_per_step"],
                   "parallelism": f"batch-sharded x{world}, one all-gather of alpha + status per step on a side stream",
                   "l2": "per-step working set (factor + bands, ~2 MB per QP) exceeds the 126 MB L2; no explicit flush",
                   "solved_ok_fraction": ok_frac, "ipm_iters_mean": iters_mean, **W["facts"]},
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": (W["launches"] * args.steps) if W["launches"] else None,
        "roofline": roof,
    }
    if cfg == "c1" and world == 1:
        line["next_stage"] = velprofile_stage(B_, res, dev)
    if rank == 0 and world == 1 and not args.no_cpu_baseline and cfg == "c1":
        line["cpu_baseline"] = cpu_baseline_dense(n, budget_s=25.0)
        line["cpu_baseline_banded"] = cpu_baseline_banded(n, budget_s=15.0)
    if rank == 0 and args.dump_outputs:
        dump_outputs(res, args.dump_outputs)             # the last timed step's results, written after every measurement
    if world > 1:
        dist.destroy_process_group()
    return line if rank == 0 else None


def streaming_kernel_times(torch, B_, lib, _lib, rt, alpha, n, n_out_max, dev, reps: int = 6):
    """Mean duration [ms] of calc_splines_kernel and create_raceline_kernel: `reps` launches each through the C-ABI, queued
    back to back between two CUDA events, outputs pre-allocated (inputs: the bench batch, larger than L2 together with
    the outputs)."""
    p, s = B_._ptr, B_._stream()
    Bq = rt.shape[0]
    f64 = dict(dtype=torch.float64, device=dev)
    nv, h = torch.empty((Bq, n, 2), **f64), torch.empty((Bq, n), **f64)
    ws = B_._workspace("splines", lib.mc_calc_splines_workspace_bytes(Bq, n), dev)

    def spl():
        _lib.check(lib.mc_calc_splines_batch(Bq, n, None, p(rt), 4, None, 1, None, None, p(nv), p(h), p(ws), ws.numel(), s), "splines")
    o = dict(cx=torch.empty((Bq, n, 4), **f64), cy=torch.empty((Bq, n, 4), **f64), sl=torch.empty((Bq, n), **f64),
             n_out=torch.empty((Bq,), dtype=torch.int32, device=dev), ri=torch.empty((Bq, n_out_max, 2), **f64),
             si=torch.empty((Bq, n_out_max), dtype=torch.int32, device=dev), tv=torch.empty((Bq, n_out_max), **f64),
             ss=torch.empty((Bq, n_out_max), **f64), el=torch.empty((Bq, n_out_max), **f64), psi=torch.empty((Bq, n_out_max), **f64),
             kap=torch.empty((Bq, n_out_max), **f64))

    def rl():
        _lib.check(lib.mc_create_raceline_batch(Bq, n, None, p(rt), 4, p(nv), p(alpha), STEP_INTERP, n_out_max, p(o["cx"]), p(o["cy"]),
                                                p(o["sl"]), p(o["n_out"]), p(o["ri"]), p(o["si"]), p(o["tv"]), p(o["ss"]), p(o["el"]),
                                                p(o["psi"]), p(o["kap"]), p(ws), ws.numel(), s), "raceline")
    out = []
    for fn in (spl, rl):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b) / reps)
    return out[0], out[1]


def pcie_probe(torch, dev) -> dict:
    """Pinned-memory copy bandwidth of this box (256 MB each way, one warm-up): what the e2e figure's copies run at."""
    h = torch.empty(32 * 1024 * 1024, dtype=torch.float64).pin_memory()
    d = torch.empty(h.shape, dtype=torch.float64, device=dev)
    out = {}
    for _ in range(2):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record(); d.copy_(h, non_blocking=True); ev[1].record(); h.copy_(d, non_blocking=True); ev[2].record()
        torch.cuda.synchronize(dev)
        out = {"h2d_gbs": h.numel() * 8 / (ev[0].elapsed_time(ev[1]) * 1e-3) / 1e9, "d2h_gbs": h.numel() * 8 / (ev[1].elapsed_time(ev[2]) * 1e-3) / 1e9}
    return out


def run_e2e(args, W, torch, B_, dev, world, sync_all, dist) -> dict:
    n, bl, cfg = W["n"], W["batch"], W["cfg"]
    n_out_max = W["n_out_max"]
    tm = _Timer(torch)
    if cfg != "c1":
        # sweep / iterative configs: inputs are generated on the device (or are the c1 kind); the e2e figure copies back
        # alpha + status of every step -- what a sweep consumer reads
        host_out = [dict(alpha=torch.empty((bl, W["step"](W["inputs"], tm)["alpha"].shape[1]), dtype=torch.float64).pin_memory(),
                         status=torch.empty((bl,), dtype=torch.int32).pin_memory()) for _ in range(2)]
        d2h = torch.cuda.Stream(device=dev)
        h2d_bytes = int(W["host_in"].numel() * 8) if W["host_in"] is not None else 0
        rt2 = torch.empty_like(W["inputs"]) if W["host_in"] is not None else None
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(args.steps):
            if rt2 is not None:
                rt2.copy_(W["host_in"], non_blocking=True)
            r = W["step"](rt2, tm)
            d2h.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(d2h):
                ncol = min(host_out[k % 2]["alpha"].shape[1], r["alpha"].shape[1])
                host_out[k % 2]["alpha"][:, :ncol].copy_(r["alpha"][:, :ncol], non_blocking=True)
                host_out[k % 2]["status"].copy_(r["status"], non_blocking=True)
                r["alpha"].record_stream(d2h)
                r["status"].record_stream(d2h)
        torch.cuda.current_stream(dev).wait_stream(d2h)
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        d2h_bytes = int(host_out[0]["alpha"].numel() * 8 + host_out[0]["status"].numel() * 4)
        return {"value": W["qps_per_step"] * world * args.steps / (float(ms.item()) * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "api": "batch.jitter_widths_batch / calc_splines_batch / opt_min_curv_batch / iqp_batch / opt_shortest_path_batch"}

    # ---- c1: the public batched API, double-buffered ----
    host_in = W["host_in"]
    h2d, d2h = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    rt_buf = [torch.empty_like(W["inputs"]) for _ in range(2)]
    out_host = [dict(alpha=torch.empty((bl, n), dtype=torch.float64).pin_memory(),
                     kappa=torch.empty((bl, n_out_max), dtype=torch.float64).pin_memory(),
                     raceline=torch.empty((bl, n_out_max, 2), dtype=torch.float64).pin_memory(),
                     n_out=torch.empty((bl,), dtype=torch.int32).pin_memory(),
                     status=torch.empty((bl,), dtype=torch.int32).pin_memory()) for _ in range(2)]
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    cur = torch.cuda.current_stream(dev)

    def upload(k):
        with torch.cuda.stream(h2d):
            h2d.wait_event(ev_free[k % 2])                 # the kernels of step k - 2 are done with this buffer
            rt_buf[k % 2].copy_(host_in, non_blocking=True)
            ev_in[k % 2].record(h2d)

    def one(k):
        if k + 1 < nsteps:
            upload(k + 1)
        cur.wait_event(ev_in[k % 2])
        rt_dev = rt_buf[k % 2]
        cx, cy, nv, h = B_.calc_splines_batch(rt_dev, want_coeffs=False)
        qp = B_.opt_min_curv_batch(rt_dev, nv, h, KAPPA_BOUND, W_VEH, centre_id=W["centre_id"])
        rl = B_.create_raceline_batch(rt_dev, nv, qp["alpha"], STEP_INTERP, n_out_max=n_out_max, with_head_curv=True)
        ev_free[k % 2].record(cur)
        d2h.wait_stream(cur)
        with torch.cuda.stream(d2h):
            oh = out_host[k % 2]
            for key, src in (("alpha", qp["alpha"]), ("kappa", rl["kappa"]), ("raceline", rl["raceline_interp"]),
                             ("n_out", rl["n_out"]), ("status", qp["status"])):
                oh[key].copy_(src, non_blocking=True)
                src.record_stream(d2h)

    # warm-up: enough steps for the allocator's cache to hold every buffer set that is alive at once in steady state (outputs
    # handed to the copy stream are recycled one step later than those of the compute stream)
    for phase_steps in (max(args.warmup, 4), args.steps):
        nsteps = phase_steps
        for e in ev_free:
            e.record(cur)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        upload(0)
        for k in range(nsteps):
            one(k)
        cur.wait_stream(d2h)
        e1.record()
        sync_all()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    oh = out_host[(args.steps - 1) % 2]
    n_out_ok = bool((oh["n_out"] > 0).all().item())
    d2h_bytes = int(sum(t.numel() * t.element_size() for t in out_host[0].values()))
    return {"value": bl * world * args.steps / (float(ms.item()) * 1e-3), "unit": UNIT,
            "h2d_bytes_per_step": int(host_in.numel() * 8), "d2h_bytes_per_step": d2h_bytes,
            "api": "batch.calc_splines_batch -> batch.opt_min_curv_batch -> batch.create_raceline_batch; results copied to "
                   "pinned host memory: alpha, kappa, raceline x/y, n_out, status",
            "copies": "H2D and D2H on their own streams, double-buffered", "all_racelines_fit": n_out_ok,
            "pinned_copy_bandwidth": pcie_probe(torch, dev)}


# ------------------------------------------------------------------------------------------------
def velprofile_stage(B_, res: dict, dev) -> dict:
    """Outside the timed region and not part of `value`: the stage after the path (SURVEY.md 8f-1) on the racelines the
    last step produced -- the reference's lap-time matrix (15 ggv scales x 11 top speeds,
    /root/reference/main_globaltraj.py:77-82, :442-496) for the first 512 racelines in one launch of vel_profile_kernel.
    Reported for information; a failure here is recorded, never raised."""
    import torch
    try:
        g = np.load(os.path.join(ROOT, "tests", "golden", "velprofile.npz"))
        scales = np.linspace(0.3, 1.0, int((1.0 - 0.3) / 0.05) + 1)
        speeds = np.linspace(100.0 / 3.6, 150.0 / 3.6, int((150.0 - 100.0) / 5.0) + 1)
        nb = min(512, res["kappa"].shape[0])
        kap, el, npts = res["kappa"][:nb].contiguous(), res["el"][:nb].contiguous(), res["n_out"][:nb].contiguous()
        args = (kap, el, g["ggv"], g["ax_max_machines"], scales, speeds, float(g["dragcoeff"]), float(g["mass"]))
        B_.lap_time_matrix_batch(*args, n_pts=npts)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        a.record()
        for _ in range(reps):
            ltm = B_.lap_time_matrix_batch(*args, n_pts=npts)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / reps
        profiles = nb * scales.size * speeds.size
        pts = float(npts.double().mean().item())
        return {"stage": "calc_vel_profile + calc_ax_profile + calc_t_profile (lap-time matrix)", "kernel": "vel_profile_kernel",
                "racelines": nb, "variants_per_raceline": int(scales.size * speeds.size), "profiles": profiles,
                "points_per_profile_mean": pts, "ms_per_launch": ms, "profiles_per_s": profiles / (ms * 1e-3),
                "lap_time_s_stock_car_mean": float(ltm[:, -1, -1].mean().item()),
                "note": "includes the launch-side host work of lap_time_matrix_batch (table upload, status check)"}
    except Exception as e:      # informational stage: record, do not fail the bench line
        return {"stage": "calc_vel_profile", "error": f"{type(e).__name__}: {e}"}


# ------------------------------------------------------------------------------------------------
def _oracle_one(rt: np.ndarray) -> float:
    """One reference-style CPU solve of the same path (dense tph restatement + Goldfarb-Idnani)."""
    from oracle import tph_dense as T
    t0 = time.perf_counter()
    path = np.vstack((rt[:, :2], rt[0, :2]))
    cx, cy, A, nv = T.calc_splines(path)
    alpha, _ = T.opt_min_curv(rt, nv, A, KAPPA_BOUND, W_VEH)
    rl = T.create_raceline(rt[:, :2], nv, alpha, STEP_INTERP)
    T.calc_head_curv_an(rl[2], rl[3], rl[4], rl[5])
    return time.perf_counter() - t0


def _oracle_worker(job):
    """One reference-style solve in a worker process with a bounded BLAS pool (several workers share the host cores)."""
    rt, blas_threads = job
    from threadpoolctl import threadpool_limits
    with threadpool_limits(limits=blas_threads):
        return _oracle_one(rt)


def _dense_pool_run(n: int, budget_s: float = None, steps: int = None):
    """THE protocol of the dense CPU arm (used by cpu_baseline of the b200 line and by --impl reference alike): `workers`
    processes solve different QPs of the workload at the same time, each with cores/workers BLAS threads (a single dense
    solve does not scale past ~8 threads: the 4N x 4N inverse is the only threaded part); one step = `workers` QPs in
    flight; `steps` steps, or as many as fit the time budget, after one warm-up step."""
    import multiprocessing as mp
    from oracle import quadprog_gi
    quadprog_gi.build()
    cores = os.cpu_count() or 1
    workers = max(1, min(16, cores // 8))
    if os.environ.get("MC_REF_WORKERS"):                 # override for experiments
        workers = max(1, int(os.environ["MC_REF_WORKERS"]))
    blas_threads = max(1, cores // workers)
    rts = make_inputs(workers, n, seed0=10_000)
    ctx = mp.get_context("spawn")
    with ctx.Pool(workers) as pool:
        jobs = [(rts[i], blas_threads) for i in range(workers)]
        t0 = time.perf_counter()
        pool.map(_oracle_worker, jobs)                   # warm-up step (also sizes the run)
        t_first = time.perf_counter() - t0
        bounded = steps is None
        if bounded:
            steps = max(1, min(1000, int(budget_s / max(t_first, 1e-3)) - 1))
        t0 = time.perf_counter()
        for _ in range(steps):
            pool.map(_oracle_worker, jobs)
        secs = time.perf_counter() - t0
    sample = (f"each step = {workers} QPs of the workload (N={n}) solved concurrently by {workers} processes x {blas_threads} BLAS "
              f"threads through the dense numpy/LAPACK tph restatement (oracle/tph_dense.py) + Goldfarb-Idnani C solver "
              f"(oracle/quadprog_gi.c); {steps} steps timed after 1 warm-up step" +
              (f" (run bounded to ~{budget_s:.0f} s)" if bounded else ""))
    return steps * workers / secs, cores, workers, steps, secs, sample


def cpu_baseline_dense(n: int, budget_s: float = 25.0) -> dict:
    qps, cores, workers, steps, secs, sample = _dense_pool_run(n, budget_s)
    return {"value": qps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}


def _banded_worker(job):
    """QPs of the workload through the banded CPU port (oracle/banded_cpu.c) on ONE core for ~budget seconds."""
    rts, budget_s = job
    from scipy.interpolate import CubicSpline
    from oracle import banded_cpu as BC
    done, t0 = 0, time.perf_counter()
    while True:
        rt = rts[done % len(rts)]
        h = BC.spline_h(rt)
        s = np.concatenate(([0.0], np.cumsum(h)))
        d1 = CubicSpline(s, np.vstack((rt[:, :2], rt[0, :2])), bc_type="periodic").derivative()(s[:-1])
        nv = np.column_stack((d1[:, 1], -d1[:, 0])) / np.linalg.norm(d1, axis=1)[:, None]       # calc_splines' normals
        BC.opt_min_curv_banded(rt, nv, W_VEH, h=h)
        done += 1
        if time.perf_counter() - t0 >= budget_s:
            return done, time.perf_counter() - t0


def cpu_baseline_banded(n: int, budget_s: float = 15.0) -> dict:
    """The fair CPU baseline (SURVEY.md 8d(ii)): the SAME banded O(N b^2) algorithm the GPU runs (periodic-tridiagonal
    splines, band of H from the semiseparable structure, Mehrotra iteration on a bordered band Cholesky) in plain C, one QP
    per host core, all cores busy.  value / the b200 line's value separates "B200" from "algorithm"."""
    import multiprocessing as mp
    from oracle import banded_cpu
    banded_cpu.build()
    cores = os.cpu_count() or 1
    rts = make_inputs(8, n, seed0=10_000)
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        pool.map(_banded_worker, [(rts, 0.2)] * cores)                  # warm-up (imports, page-in)
        t0 = time.perf_counter()
        res = pool.map(_banded_worker, [(rts, budget_s)] * cores)
        wall = time.perf_counter() - t0
    total = sum(r[0] for r in res)
    return {"value": total / wall, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{total} QPs of the workload (N={n}) in {wall:.1f} s: {cores} processes, one QP at a time per core, through "
                      "oracle/banded_cpu.c (periodic-tridiagonal splines via scipy CubicSpline, banded assembly + Mehrotra on a "
                      "bordered band Cholesky: the algorithm of the CUDA path, box-only QP)"}


def run_reference(args) -> dict:
    """Reference arm: the reference-style CPU path (dense numpy/LAPACK tph restatement + Goldfarb-Idnani in C) on ALL host
    cores, with the protocol of _dense_pool_run; --steps timed steps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    n = args.npoints or N_POINTS
    qps, cores, workers, steps, secs, sample = _dense_pool_run(n, steps=args.steps)
    return {"impl": "reference", "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
            "steps": steps, "warmup": 1, "ms_per_step": 1e3 * secs / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"batch {workers} per step: " + CONFIGS["c1"]["what"] + f", N={n} points",
                       "baseline_config": "c1", "n_points": n, "kappa_bound": KAPPA_BOUND, "w_veh": W_VEH, "qps_per_step": workers},
            "cpu_baseline": {"value": qps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c1", choices=sorted(CONFIGS), help="BASELINE.json config (c1 = the headline workload)")
    ap.add_argument("--batch", type=int, default=None, help="QP instances per GPU (default: the config's)")
    ap.add_argument("--npoints", type=int, default=None, help="points per track (default: the config's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's results as DIR/<name>.npy (float64, rank 0, at most 64 MB: a fixed, "
                         "seeded sample of the instances when they do not fit)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 path")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        line = run_reference(args)
    else:
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if args.gpus > 1 and world == 1:
            # convenience: re-launch ourselves under torchrun (a launcher that starts torchrun itself sets WORLD_SIZE)
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                   "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__), "--gpus", str(args.gpus),
                   "--steps", str(args.steps), "--warmup", str(args.warmup), "--config", args.config]
            if args.batch:
                cmd += ["--batch", str(args.batch)]
            if args.npoints:
                cmd += ["--npoints", str(args.npoints)]
            if args.dump_outputs:
                cmd += ["--dump-outputs", os.path.abspath(args.dump_outputs)]
            sys.exit(subprocess.call(cmd))
        line = run_b200(args)
    if line is not None:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
