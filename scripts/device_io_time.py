#!/usr/bin/env python3
"""Time the device-memory entry points of a field (pa_field_upload_device / pa_field_download_device) against the pinned
host route and the device-resident tools end to end, on one GPU:

  python scripts/device_io_time.py [--out profiles/r09_device_io.jsonl] [--repeats 5] [--hier north_star grad5]

Hierarchies: north_star = bench.py's target hierarchy (temp on 3 levels, 512^3 base, ratio 2, 128^3 boxes; 403 M cells);
grad5 = bench.py's grad5 grids (4 levels, ratios 2/4/2, 128^3 base, 16^3 boxes).  One JSON line per measurement, each with
the card's name and power limit and the device-to-device copy bandwidth (torch copy_ of 4 GiB) read in the same run:

  upload / download     one component of every level from / into one CUDA tensor per box: dense [nz][ny][nx] tensors, and
                        4-component FABs with ng = 1, 2 ghost cells ([4][nz+2ng][ny+2ng][nx+2ng], all 4 components into a
                        4-component field).  Bytes model: 16 B per valid cell and component (read 8, write 8), reported as
                        GB/s and as a fraction of the copy bandwidth.
  host_upload / host_download   the same data through pa_field_upload_level / pa_field_download_level from / into pinned
                        host buffers; rate of the 8 B per cell and component that cross the host link.
  grad_e2e / curv_e2e   GradRun / CurvatureRun from device tensors in to device tensors out: upload_device + step +
                        result_device, beside step alone (the device-resident hot path bench.py measures).

Times are CUDA-event medians over `repeats` runs after one warm-up run, with the fastest and slowest."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from smooth_time import copy_gbs  # noqa: E402
from peleanalysis_b200 import capi, synth  # noqa: E402
from peleanalysis_b200.stencilrun import CurvatureRun, GradRun  # noqa: E402

HIERS = {"north_star": lambda: synth.config3(512, 128, fill=False),
         "grad5": lambda: synth.config5(128, 16, 1, fill=False)}


def timed(fn, repeats, stream):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(min(ts)), float(max(ts))


def dims(box):
    lo, hi = box
    return (hi[2] - lo[2] + 1, hi[1] - lo[1] + 1, hi[0] - lo[0] + 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_device_io.jsonl"))
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--hier", nargs="+", choices=sorted(HIERS), default=["north_star", "grad5"])
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("device_io_time.py measures on the GPU: no CUDA device")
    torch.cuda.set_device(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    card = q.stdout.strip()
    bw = copy_gbs()
    capi.init(0)
    stream = torch.cuda.current_stream()
    capi.set_stream(stream.cuda_stream)
    lines = []

    def emit(**kw):
        kw.update(card=card, copy_gbs=round(bw, 1))
        if "gbs" in kw and kw.get("model") == "16B/cell/comp":
            kw["frac_of_copy"] = round(kw["gbs"] / bw, 3)
        print(json.dumps(kw), flush=True)
        lines.append(kw)

    for hname in a.hier:
        pf = HIERS[hname]()
        H = capi.Hierarchy(pf.levels)
        cells = H.num_cells
        nb = sum(len(lv.boxes) for lv in pf.levels)
        base = dict(hier=hname, cells=cells, boxes=nb)
        gen = torch.Generator(device="cuda").manual_seed(1)
        # dense sources, one tensor per box
        dense = [[torch.rand(dims(b), dtype=torch.float64, device="cuda", generator=gen) for b in lv.boxes] for lv in pf.levels]
        f1 = capi.Field(H, 1, 1)

        def up_dense():
            for l in range(len(pf.levels)):
                f1.upload_level_device(l, 0, dense[l])

        def down_dense():
            for l in range(len(pf.levels)):
                f1.download_level_device(l, 0, dense[l])
        # the same with the pa_array4 records built once (what a C++ caller that keeps its descriptors pays): the C calls only
        pre = [f1._arrays(l, dense[l], 0) for l in range(len(pf.levels))]

        def up_pre():
            for l, (d, n) in enumerate(pre):
                capi.check(capi.lib().pa_field_upload_device(f1.f, l, 0, 1, d, n))

        def down_pre():
            for l, (d, n) in enumerate(pre):
                capi.check(capi.lib().pa_field_download_device(f1.f, l, 0, 1, d, n))
        for what, src, fn in (("upload", "dense", up_dense), ("download", "dense", down_dense),
                              ("upload", "dense_prebuilt", up_pre), ("download", "dense_prebuilt", down_pre)):
            ms, lo, hi = timed(fn, a.repeats, stream)
            emit(**base, what=what, src=src, ncomp=1, ms=round(ms, 3), ms_min=round(lo, 3), ms_max=round(hi, 3),
                 gbs=round(16 * cells / (ms * 1e-3) / 1e9, 1), model="16B/cell/comp")
        # pinned host route, the same component
        host = [capi.PinnedArray(H.local_cells[l]) for l in range(len(pf.levels))]
        for l in range(len(pf.levels)):
            host[l].array[:] = 0.5

        def up_host():
            for l in range(len(pf.levels)):
                f1.upload_level(l, 0, host[l].array)

        def down_host():
            for l in range(len(pf.levels)):
                f1.download_level(l, 0, host[l].array)
        for what, fn in (("host_upload", up_host), ("host_download", down_host)):
            ms, lo, hi = timed(fn, a.repeats, stream)
            emit(**base, what=what, src="pinned", ncomp=1, ms=round(ms, 3), ms_min=round(lo, 3), ms_max=round(hi, 3),
                 gbs=round(8 * cells / (ms * 1e-3) / 1e9, 1), model="8B/cell/comp over the host link")
        for p in host:
            p.free()
        del host
        # 4-component FABs with ghost cells into a 4-component field
        f4 = capi.Field(H, 4, 1)
        for g in (1, 2):
            fabs = [[torch.rand((4,) + tuple(n + 2 * g for n in dims(b)), dtype=torch.float64, device="cuda", generator=gen) for b in lv.boxes]
                    for lv in pf.levels]

            def up_fab():
                for l in range(len(pf.levels)):
                    f4.upload_level_device(l, 0, fabs[l], nghost=g, ncomp=4)

            def down_fab():
                for l in range(len(pf.levels)):
                    f4.download_level_device(l, 0, fabs[l], nghost=g, ncomp=4)
            for what, fn in (("upload", up_fab), ("download", down_fab)):
                ms, lo, hi = timed(fn, a.repeats, stream)
                emit(**base, what=what, src="fab_ng%d" % g, ncomp=4, ms=round(ms, 3), ms_min=round(lo, 3), ms_max=round(hi, 3),
                     gbs=round(16 * 4 * cells / (ms * 1e-3) / 1e9, 1), model="16B/cell/comp")
            del fabs
        del f4
        torch.cuda.empty_cache()
        # the tools end to end from device tensors: upload_device + step + result_device, and step alone
        pf.names = ["temp"]
        o = capi.CurvOpts()
        o.prog_min, o.prog_max = 0.0, 1.0
        for tool, make in (("grad_e2e", lambda: GradRun(capi, pf, names=["temp"], upload=False)),
                           ("curv_e2e", lambda: CurvatureRun(capi, pf, o, upload=False))):
            keep, run = [], None

            def e2e():
                run.upload_device("temp", dense)
                run.step()
                keep[:] = [run.result_device()]
            try:
                run = make()
                ms, lo, hi = timed(e2e, a.repeats, stream)
                ms_step, _, _ = timed(run.step, a.repeats, stream)
            except capi.PaError as e:          # e.g. a hierarchy the tool does not support
                emit(**base, what=tool, error=str(e))
                continue
            emit(**base, what=tool, ms=round(ms, 3), ms_min=round(lo, 3), ms_max=round(hi, 3), ms_step_only=round(ms_step, 3),
                 nout=len(run.out_names))
            del keep, run
            torch.cuda.empty_cache()
        del dense, f1, H
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        for kw in lines:
            fh.write(json.dumps(kw) + "\n")


if __name__ == "__main__":
    main()
