#!/usr/bin/env python3
"""Strong scaling of filterPlt over GPUs: the filter3 workload of bench.py (box filter, base_fgr 2 -> ghost widths 1/2/4,
max_grid_size 32, temp on 3 levels with a 256^3 base) with its re-chopped boxes spread over the ranks (pa_sfc_distribute);
the FillPatch sources of other ranks move as NCCL send/recv of packed slabs.  Run under torchrun, one process per GPU:

  python -m torch.distributed.run --nproc-per-node N scripts/filter_scale.py [--base 256 --box 64 --mgs 32] [--steps 10]

Prints one JSON line (rank 0): step time from device events (max over ranks), Gcells/s, the per-level exchange / fill /
filter split (device events, a separate pass), bytes each rank sends per step, the summed output fingerprint (pa_field_hash
over the ranks: equal for any N), and the card's name and power limit read in the same run."""
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
from peleanalysis_b200 import capi, filterplt, synth  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", type=int, default=256)
    ap.add_argument("--box", type=int, default=64)
    ap.add_argument("--mgs", type=int, default=32)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
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
    run = filterplt.FilterRun(capi, pf, filter_type=1, base_fgr=2, max_grid_size=a.mgs, upload=False, rank=rank, nranks=world)
    fields = bench.gen_fields(torch, run.levels, run.hier.local_boxes, ["temp"])
    for l in range(run.nlev):
        if run.hier.local_boxes[l]:
            run.fin.upload_level(l, 0, fields[l][0].cpu().numpy())
    capi.sync()
    del fields

    def mx(v):
        if world == 1:
            return v
        t = torch.tensor([v], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ev = lambda: torch.cuda.Event(enable_timing=True)
    for _ in range(a.warmup):
        run.step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0, t1 = ev(), ev()
    t0.record(stream)
    for _ in range(a.steps):
        run.step()
    t1.record(stream)
    torch.cuda.synchronize()
    ms = mx(t0.elapsed_time(t1) / a.steps)
    # split: one more step, events between its phases
    split = []
    for l in range(run.nlev):
        e = [ev() for _ in range(4)]
        e[0].record(stream)
        if run.exchanges:
            run.exchanges[l].run(0)
        e[1].record(stream)
        capi.fill_patch(run.fin, 0, 1, l, run.ngrow[l], 1)
        e[2].record(stream)
        capi.filter_level(run.fin, 0, run.fout, 0, 1, l, 1, run.fgr[l])
        e[3].record(stream)
        torch.cuda.synchronize()
        split.append({"level": l, "ngrow": run.ngrow[l], "exchange_ms": mx(e[0].elapsed_time(e[1])), "fill_ms": mx(e[1].elapsed_time(e[2])),
                      "filter_ms": mx(e[2].elapsed_time(e[3]))})
    h = run.fout.hash(0, 1)
    sent = sum(x.bytes_sent for x in run.exchanges)
    if world > 1:
        hs, ss = [None] * world, [None] * world
        dist.all_gather_object(hs, h)
        dist.all_gather_object(ss, sent)
        h = sum(hs) % (1 << 64)
    else:
        ss = [0]
    if rank == 0:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(dev)], capture_output=True, text=True)
        cells = run.cells()
        print(json.dumps({"workload": "filter3 on %d GPU(s): base %d^3, %d^3 boxes, max_grid_size %d" % (world, a.base, a.box, a.mgs),
                          "n_gpus": world, "cells": cells, "ms_per_step": ms, "gcells_per_s": cells / (ms * 1e-3) / 1e9,
                          "boxes": [len(lv.boxes) for lv in run.levels], "split_max_over_ranks": split,
                          "bytes_sent_per_rank_per_step": ss, "output_hash": "%016x" % h, "gpu": q.stdout.strip(), "steps": a.steps}))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
