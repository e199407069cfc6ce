#!/usr/bin/env python3
"""Strong scaling of grad and curvature over GPUs with every cross-rank ghost source moved as a packed slab: the north-star
hierarchy of bench.py (temp on 3 levels, 512^3 base, ratio 2, 128^3 boxes) with its boxes spread over the ranks
(pa_sfc_distribute), stencilrun.GradRun / CurvatureRun, slabs moved by NCCL send/recv (nothing peer-mapped).  Run under
torchrun, one process per GPU:

  python -m torch.distributed.run --nproc-per-node N scripts/stencil_scale.py [--base 512 --box 128] [--steps 100] [--repeats 5]
                                                                               [--tools grad curvature]

Prints one JSON line per tool (rank 0): step time from device events (max over ranks; the median of `repeats` timed windows
of `steps` steps each, with the fastest and slowest window), Gcells/s at the median, the time of the exchange alone (a
separate pass), bytes each rank sends per step, the summed output fingerprint (pa_field_hash over the ranks: equal for any
N), and the card's name and power limit read in the same run.  The inputs are generated on the device and are larger than
L2, so every timed step reads them from HBM."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (gen_fields: the benchmark's device-side synthetic fields)
from peleanalysis_b200 import capi, stencilrun, synth  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", type=int, default=512)
    ap.add_argument("--box", type=int, default=128)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--tools", nargs="+", default=["grad", "curvature"], choices=["grad", "curvature"])
    a = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    dev = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
        t = torch.ones(1, device="cuda")
        dist.all_reduce(t)
    capi.init(dev)
    stream = torch.cuda.current_stream()
    capi.set_stream(stream.cuda_stream)
    pf = synth.config3(a.base, a.box, fill=False)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(dev)], capture_output=True, text=True)
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def mx(v, op=None):
        if world == 1:
            return v
        t = torch.tensor([v], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=op or dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, n):
        t0, t1 = ev(), ev()
        t0.record(stream)
        for _ in range(n):
            fn()
        t1.record(stream)
        torch.cuda.synchronize()
        return mx(t0.elapsed_time(t1) / n)

    for tool in a.tools:
        if tool == "grad":
            run = stencilrun.GradRun(capi, pf, ["temp"], upload=False, rank=rank, nranks=world)
            fin, exchanges = run.fin, [(run.exchange, 0)] if run.exchange else []
        else:
            o = capi.CurvOpts()
            run = stencilrun.CurvatureRun(capi, pf, o, "temp", upload=False, rank=rank, nranks=world)
            fin, exchanges = run.state, [(run.op.Xs, 0), (run.op.Xn, 2)] if run.op else []      # S, then the flame normal
        host = bench.gen_fields(torch, pf.levels, run.hier.local_boxes, ["temp"])
        for l in range(run.nlev):
            if run.hier.local_cells[l]:
                capi.check(capi.lib().pa_field_upload_level(fin.f, l, 0, host[l][0].data_ptr()))
        if tool == "curvature":           # the tool's default progMin / progMax: the extremes over every rank's cells
            lo = min([float(h[0].min()) for h in host if h[0].numel()] or [1e300])
            hi = max([float(h[0].max()) for h in host if h[0].numel()] or [-1e300])
            o.prog_min, o.prog_max = -mx(-lo), mx(hi)
        capi.sync()
        del host
        for _ in range(a.warmup):
            run.step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        windows = sorted(timed(run.step, a.steps) for _ in range(a.repeats))
        ms = windows[len(windows) // 2]

        def exchange():
            for x, comp in exchanges:
                x.run(comp)
        xms = timed(exchange, a.steps) if exchanges else 0.0
        sent = 8 * sum(x.soff[-1] for x, _ in exchanges)
        h = run.fout.hash(0)
        if world > 1:
            hs, ss = [None] * world, [None] * world
            dist.all_gather_object(hs, h)
            dist.all_gather_object(ss, sent)
            h = sum(hs) % (1 << 64)
        else:
            ss = [0]
        if rank == 0:
            cells = run.cells()
            print(json.dumps({"workload": "%s on %d GPU(s), packed-slab transport: temp, 3 levels, %d^3 base, ratio 2, %d^3 boxes" % (tool, world, a.base, a.box),
                              "n_gpus": world, "cells": cells, "ms_per_step": ms, "ms_per_step_min": windows[0], "ms_per_step_max": windows[-1],
                              "gcells_per_s": cells / (ms * 1e-3) / 1e9,
                              "exchange_ms_alone": xms, "boxes": [len(lv.boxes) for lv in pf.levels],
                              "bytes_sent_per_rank_per_step": ss, "output_hash": "%016x" % h, "gpu": q.stdout.strip(), "steps": a.steps, "repeats": a.repeats}), flush=True)
        del run, fin, exchanges
        torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
