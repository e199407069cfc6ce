#!/usr/bin/env python3
"""Time curvature's do_smooth solve (pa_smooth, curvature.cpp:328-406) on the north-star hierarchy of bench.py (temp on
3 levels, 512^3 base, ratio 2, 128^3 boxes; 403 M cells) at smoothing_time 1e-7 and 1e-5, on one GPU:

  python scripts/smooth_time.py [--base 512 --box 128] [--times 1e-7 1e-5] [--repeats 3]

Prints one JSON line per smoothing time: ms per solve from CUDA events (median of `repeats` solves after one warm-up solve,
with the fastest and slowest), BiCGStab iterations, ms per iteration, the achieved bandwidth of an iteration under the bytes
model below as a fraction of the device-to-device copy bandwidth measured in the same run, and the card's name and power
limit read in the same run.

Bytes model of one iteration, per valid cell (8-byte doubles; the slab-wide vector updates also touch the ghost cells and
pads, about 10 % more on 128^3 boxes, which the model leaves out): two operator applications of 16 bytes each (read phi,
write A phi; neighbours come from cache), the vector updates p (32), z = M^-1 p (16), s (24), x (24), z = M^-1 s (16), r (24),
x (24), and the reductions (r0, r) (16), (r0, v) (16), (t, s) (16), (t, t) (8), max |s| (8), max |r| (8).  Ghost fills,
average-down and reflux touch the cells next to box faces only and are left out as well."""
import argparse
import json
import os
import subprocess
import sys

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
        o = capi.SmoothOpts()
        o.smoothing_time = t
        capi.smooth(st, 0, pmin, pmax, o, out, 0, 1)                 # warm-up: tables, work fields, first launches
        times, its, res = [], None, None
        for _ in range(a.repeats):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            it, r = capi.smooth(st, 0, pmin, pmax, o, out, 0, 1)
            e1.record(stream)
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
            its, res = it, r
        times.sort()
        ms = times[len(times) // 2]
        per_it = ms / its if its else None
        gbs = BYTES_PER_CELL_ITER * cells / (per_it * 1e-3) / 1e9 if per_it else None
        print(json.dumps({"tool": "smooth", "smoothing_time": t, "cells": cells, "ms_per_solve": ms, "ms_min": times[0], "ms_max": times[-1],
                          "iterations": its, "residual": res, "ms_per_iteration": per_it,
                          "bytes_per_cell_iteration": BYTES_PER_CELL_ITER, "iteration_gbs": gbs,
                          "copy_gbs_measured": bw, "frac_of_copy": (gbs / bw) if gbs else None, "card": card}), flush=True)


if __name__ == "__main__":
    main()
