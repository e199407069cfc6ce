#!/usr/bin/env python3
"""Time curvature's do_smooth solve (pa_smooth, curvature.cpp:328-406) on the north-star hierarchy of bench.py (temp on
3 levels, 512^3 base, ratio 2, 128^3 boxes; 403 M cells) at smoothing_time 1e-7 and 1e-5, on one GPU:

  python scripts/smooth_time.py [--base 512 --box 128] [--times 1e-7 1e-5] [--repeats 3] [--precond jacobi mg] [--profile]

Prints one JSON line per smoothing time: ms per solve from CUDA events (median of `repeats` solves after one warm-up solve,
with the fastest and slowest), BiCGStab iterations, ms per iteration, the achieved bandwidth of an iteration under the bytes
model below as a fraction of the device-to-device copy bandwidth measured in the same run, and the card's name and power
limit read in the same run.

Bytes model of one iteration, per valid cell (8-byte doubles; the slab-wide vector updates also touch the ghost cells and
pads, about 10 % more on 128^3 boxes, which the model leaves out): two operator applications of 16 bytes each (read phi,
write A phi; neighbours come from cache), the vector updates p (32), z = M^-1 p (16), s (24), x (24), z = M^-1 s (16), r (24),
x (24), and the reductions (r0, r) (16), (r0, v) (16), (t, s) (16), (t, t) (8), max |s| (8), max |r| (8).  Ghost fills,
average-down and reflux touch the cells next to box faces only and are left out as well.

--precond jacobi mg times each preconditioner (PA_SMOOTH_PRECOND_*) at every smoothing time; the lines then also carry
"precond" and, for mg, ms per V-cycle step (pa_debug_smooth_vcycle: one V-cycle, one operator application and one max-norm
reduction; (time of 5 steps - time of 0 steps) / 5) and the number of level-0 multigrid levels.  A solve that does not
converge within max_iter (1000) is recorded with "noconv": true and its iteration count.  --profile adds, per smoothing time
and preconditioner, one profiled solve (torch.profiler, CUDA activity) with the device time of every k_sm_* kernel; for mg
also the red-black Gauss-Seidel kernel's bandwidth under the model of 16 bytes per visited cell and colour pass (each pass
visits every valid cell of its level: reads it, and on half of them the right-hand side and the write)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (gen_fields: the benchmark's device-side synthetic fields)
from peleanalysis_b200 import capi, synth  # noqa: E402

BYTES_PER_CELL_ITER = 2 * 16 + (32 + 16 + 24 + 24 + 16 + 24 + 24) + (16 + 16 + 16 + 8 + 8 + 8)


def copy_gbs(nbytes=4 << 30, reps=10):
    a = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    a.fill_(1.0)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del a, b
    torch.cuda.empty_cache()
    return 2 * nbytes / (ms * 1e-3) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", type=int, default=512)
    ap.add_argument("--box", type=int, default=128)
    ap.add_argument("--times", type=float, nargs="+", default=[1e-7, 1e-5])
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--precond", nargs="+", choices=sorted(capi.SMOOTH_PRECONDS), default=None)
    ap.add_argument("--profile", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("smooth_time.py measures on the GPU: no CUDA device")
    dev = 0
    torch.cuda.set_device(dev)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(dev)], capture_output=True, text=True)
    card = q.stdout.strip()
    bw = copy_gbs()
    capi.init(dev)
    stream = torch.cuda.current_stream()
    capi.set_stream(stream.cuda_stream)
    pf = synth.config3(a.base, a.box, fill=False)
    H = capi.Hierarchy(pf.levels)
    cells = H.num_cells
    st = capi.Field(H, 1, 1)
    out = capi.Field(H, 2, 1)
    host = bench.gen_fields(torch, pf.levels, [list(range(len(lv.boxes))) for lv in pf.levels], ["temp"])
    pmin, pmax = float("inf"), -float("inf")
    for l in range(len(pf.levels)):
        st.upload_level(l, 0, host[l][0].numpy())
        pmin, pmax = min(pmin, float(host[l][0].min())), max(pmax, float(host[l][0].max()))
    capi.sync()
    del host
    for t in a.times:
        for pname in (a.precond or ["jacobi"]):
            o = capi.SmoothOpts()
            o.smoothing_time = t
            o.precond = capi.smooth_precond(pname)
            try:
                capi.smooth(st, 0, pmin, pmax, o, out, 0, 1)             # warm-up: tables, work fields, first launches
            except capi.PaError as e:
                if e.code != capi.PA_ERR_NOCONV:
                    raise
            times, its, res, noconv = [], None, None, False
            for _ in range(a.repeats):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                try:
                    it, r = capi.smooth(st, 0, pmin, pmax, o, out, 0, 1)
                except capi.PaError as e:
                    if e.code != capi.PA_ERR_NOCONV:
                        raise
                    it, r, noconv = o.max_iter or 1000, float(str(e).split("max|c - A phi| / max|c| = ")[1].split()[0]), True
                e1.record(stream)
                torch.cuda.synchronize()
                times.append(e0.elapsed_time(e1))
                its, res = it, r
            times.sort()
            ms = times[len(times) // 2]
            per_it = ms / its if its else None
            rec = {"tool": "smooth", "smoothing_time": t, "cells": cells, "ms_per_solve": ms, "ms_min": times[0], "ms_max": times[-1],
                   "iterations": its, "residual": res, "ms_per_iteration": per_it}
            if a.precond is None:
                gbs = BYTES_PER_CELL_ITER * cells / (per_it * 1e-3) / 1e9 if per_it else None
                rec.update({"bytes_per_cell_iteration": BYTES_PER_CELL_ITER, "iteration_gbs": gbs, "copy_gbs_measured": bw,
                            "frac_of_copy": (gbs / bw) if gbs else None, "card": card})
            else:
                rec.update({"precond": pname, "noconv": noconv, "t_over_dx2_finest": t / float(pf.levels[-1].dx[0]) ** 2,
                            "copy_gbs_measured": bw, "card": card})
                if pname == "mg":
                    step_ms = []
                    for n in (0, 5):
                        capi.debug_smooth_vcycle(st, 0, pmin, pmax, o, out, 0, 1, n)
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record(stream)
                        _, nmg = capi.debug_smooth_vcycle(st, 0, pmin, pmax, o, out, 0, 1, n)
                        e1.record(stream)
                        torch.cuda.synchronize()
                        step_ms.append(e0.elapsed_time(e1))
                    rec.update({"ms_per_vcycle_step": (step_ms[1] - step_ms[0]) / 5, "mg_levels": nmg})
            if a.profile:
                rec["kernels"] = profile_solve(st, out, o, pmin, pmax)
                if pname == "mg" and "k_sm_gsrb" in rec["kernels"]:
                    gs = rec["kernels"]["k_sm_gsrb"]
                    visited = gsrb_cells_per_vcycle(pf, rec["mg_levels"]) * 2 * its
                    rec["gsrb_model_gbs"] = 16 * visited / (gs["ms"] * 1e-3) / 1e9
                    rec["gsrb_frac_of_copy"] = rec["gsrb_model_gbs"] / bw
            print(json.dumps(rec), flush=True)


def gsrb_cells_per_vcycle(pf, nmg, nu=2, bottom=16):
    """valid cells the red-black passes of one V-cycle visit: (nu1 + nu2) sweeps of 2 colours on every AMR level above 0 and every
    level-0 multigrid level but the coarsest, `bottom` sweeps on the coarsest"""
    n = 0
    for lv in pf.levels[1:]:
        n += 2 * nu * 2 * sum(int(np.prod(np.array(hi) - np.array(lo) + 1)) for lo, hi in lv.boxes)
    n0 = sum(int(np.prod(np.array(hi) - np.array(lo) + 1)) for lo, hi in pf.levels[0].boxes)
    for k in range(nmg):
        n += (bottom if k == nmg - 1 else 2 * nu) * 2 * (n0 >> (3 * k))
    return n


def profile_solve(st, out, o, pmin, pmax):
    """device time and launches of every k_sm_* kernel in one solve"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        try:
            capi.smooth(st, 0, pmin, pmax, o, out, 0, 1)
        except capi.PaError as e:
            if e.code != capi.PA_ERR_NOCONV:
                raise
        torch.cuda.synchronize()
    k = {}
    for ev in prof.key_averages():
        for name in ("k_sm_gsrb", "k_sm_resid", "k_sm_prolong", "k_sm_apply", "k_sm_reflux", "k_sm_avgdown", "k_sm_lin3", "k_sm_reduce",
                     "k_sm_final", "k_sm_copy", "k_halo", "k_bcfill"):
            if name in ev.key:
                us = getattr(ev, "device_time_total", None)
                if us is None:
                    us = ev.cuda_time_total
                d = k.setdefault(name, {"ms": 0.0, "launches": 0})
                d["ms"] += us / 1e3
                d["launches"] += ev.count
    return k

if __name__ == "__main__":
    main()
