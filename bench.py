#!/usr/bin/env python3
"""bench.py -- benchmark of the grad / curvature stencil path (BASELINE.json metric: Gcells/s over all AMR levels).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

Workloads (--workload; the default, config2, is the configuration the metric is quoted on):
  config2      grad, uniform 512^3, 64 boxes of 128^3, 5 components                         (BASELINE configs[1])
  config4      grad, uniform 1024^3, 512 boxes of 128^3, 1 component                         (BASELINE configs[3])
  target_grad  grad of temp, 3 levels, 512^3 base, ratio 2, 128^3 boxes                      (the north-star target hierarchy)
  target_curv  curvature (default options) on the same hierarchy
  curvature3   curvature, 3 levels, 256^3 base, ratio 2, 64^3 boxes                          (BASELINE configs[2])
  grad5        grad of 12 components, 4 levels (ratios 2/4/2), 128^3 base, 16^3 boxes        (BASELINE configs[4])
  filter3      filterPlt (box filter, base_fgr 2 -> ghost widths 1/2/4, max_grid_size 32) of temp on the configs[2]
               hierarchy: SURVEY 8(f) rank 4, the neighbouring stencil tool (extra only; FP64-pipe-bound, see DESIGN.md 9)

One "step" = one pass of the hot path (ghost fill + c-f fill + stencil kernels) over the synthetic workload:
  value     device-resident inputs -> device-resident outputs, CUDA-event timed, max over ranks
  e2e       the same step through the C ABI with HOST buffers: pinned H2D of the inputs, hot path, D2H of the results
  roofline  the dominant kernel against the measured HBM copy bandwidth of MEASURED_PEAKS.json; bytes = SURVEY 8(d)
            algorithmic bytes (inputs read once + outputs written once)
  cpu_baseline  the compiled reference (oracle/_ref/*.timed.ex, all host cores) on a bounded sample of the workload
  output_hash   order-independent fingerprint of every output bit (pa_field_hash, summed over the ranks): equal for any
            number of GPUs, and compared with tests/golden/bench_hashes.json -- a mismatch makes the run fail (rc 3)
  extras    the other workloads, measured the same way (device-resident; no e2e) and fingerprinted
N > 1 (torchrun, one process per GPU): the boxes of the same workload are distributed over the ranks (strong scaling).
--transport peer (default): every rank maps its peers' slabs through CUDA IPC and the stencil kernels' TMA producer reads
cross-rank neighbour planes / rows in place over NVLink -- no pack, no exchange, no halo kernel.  --transport slab: the
cross-rank ghost cells move as NCCL send/recv of packed slabs between a pack and a fill kernel (what an MPI code does).
--impl reference: the unmodified reference tool (oracle/_ref) on the host cores, on the SAME workload (same grid, same
variables), its hot-path region looped inside one process per variable.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (it may be read-only)

UNIT = "Gcells/s"
HASH_FILE = os.path.join(ROOT, "tests", "golden", "bench_hashes.json")


def metric_name(kind):
    return "Gcells/s (all AMR levels) for " + ("grad" if kind == "grad" else "curvature")


def workload_spec(name):
    """kind, hierarchy builder, differentiated variables, description.  `cells` etc. follow from the hierarchy."""
    from peleanalysis_b200 import synth
    if name == "config2":
        return dict(name=name, kind="grad", build=lambda fill=False: synth.make_hierarchy(512, [], [], 128, list(synth.FIELD_NAMES), fill=fill),
                    names=list(synth.FIELD_NAMES), desc="grad, uniform 512^3, 64 boxes of 128^3, 5 components (BASELINE configs[1])")
    if name == "config4":
        return dict(name=name, kind="grad", build=lambda fill=False: synth.make_hierarchy(1024, [], [], 128, ["temp"], fill=fill),
                    names=["temp"], desc="grad, uniform 1024^3, 512 boxes of 128^3, 1 component (BASELINE configs[3])")
    if name == "config2_small":
        return dict(name=name, kind="grad", build=lambda fill=False: synth.make_hierarchy(256, [], [], 128, list(synth.FIELD_NAMES), fill=fill),
                    names=list(synth.FIELD_NAMES), desc="grad, uniform 256^3, 8 boxes of 128^3, 5 components (smoke-size)")
    if name in ("target_grad", "target_curv"):
        kind = "grad" if name == "target_grad" else "curv"
        return dict(name=name, kind=kind, build=lambda fill=False: synth.config3(512, 128, fill=fill), names=["temp"],
                    desc="%s, 3 levels, 512^3 base, ratio 2, 128^3 boxes (the north-star target hierarchy)" % (
                        "grad of temp" if kind == "grad" else "curvature (default options)"))
    if name == "curvature3":
        return dict(name=name, kind="curv", build=lambda fill=False: synth.config3(256, 64, fill=fill), names=["temp"],
                    desc="curvature (default options), 3 levels, 256^3 base, ratio 2, 64^3 boxes (BASELINE configs[2])")
    if name == "curvature3_small":
        return dict(name=name, kind="curv", build=lambda fill=False: synth.config3(64, 32, fill=fill), names=["temp"],
                    desc="curvature (default options), 3 levels, 64^3 base, ratio 2, 32^3 boxes (smoke-size)")
    if name == "grad5":
        pf0 = synth.config5(128, 16, 12, fill=False)
        return dict(name=name, kind="grad", build=lambda fill=False: synth.config5(128, 16, 12, fill=fill), names=list(pf0.names),
                    desc="grad of 12 components, 4 levels (ratios 2/4/2), 128^3 base, 16^3 boxes (BASELINE configs[4])")
    raise SystemExit("unknown workload " + name)


def config_of(spec, pf):
    """The workload as both arms report it (identical objects: the driver compares them)."""
    cells = sum(l.ncells for l in pf.levels)
    nvar = len(spec["names"])
    per_cell = 40 if spec["kind"] == "grad" else 48
    return {"workload": spec["desc"], "cells": cells, "variables": nvar, "boxes": [len(l.boxes) for l in pf.levels],
            "cache": "inputs + outputs of one step (%.1f GB) exceed the 126 MB L2; no flush needed" % (cells * nvar * per_cell / 1e9)}


# ---------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the compiled, unmodified reference tool on the host cores
# ---------------------------------------------------------------------------------------------------------------
def run_reference(spec, steps, warmup, variables=None, variants=("timed",)):
    """The reference tool (oracle/_ref/{grad3d,curvature3d}.timed.ex = the unmodified sources plus timing probes around
    grad.cpp:151-236 / curvature.cpp:283-791, FillVar's disk read subtracted) on the workload's own plotfile, one process
    per differentiated variable, the probed region repeated warmup + steps times inside the process (PA_TIMED_REPS).
    variants: "timed" = the CPU/OpenMP build on all host cores; "cuda.timed" = the reference's own generic CUDA build
    (oracle/build_ref_cuda.py) on this box's GPU.  Returns {variant: (Gcells/s, seconds per step, cores, per-step list)}, names."""
    from oracle import oracle as O
    from peleanalysis_b200 import plotfile
    if not O.have_ref():
        raise RuntimeError("oracle/_ref is missing (built by __graft_entry__.build() where /root/reference exists)")
    names = list(variables or spec["names"])
    pf = spec["build"](fill=True)
    cells = sum(l.ncells for l in pf.levels)
    base = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    tmp = tempfile.mkdtemp(prefix="pa_ref_", dir=base)
    cores = os.cpu_count() or 1
    res = {}
    try:
        d = os.path.join(tmp, "plt")
        plotfile.write_plotfile(d, pf, clean="remove")
        del pf
        for variant in variants:
            if not os.path.exists(O.ref_exe("%s3d.%s.ex" % ("grad" if spec["kind"] == "grad" else "curvature", variant))):
                res[variant] = None
                continue
            per_step = np.zeros(steps)
            thr = cores if variant == "timed" else 1
            try:
                for v in names:
                    if spec["kind"] == "grad":
                        hot = O.run_ref_timed("grad", d, d + "_out", threads=thr, reps=warmup + steps, variant=variant, gradVar=v)
                    else:
                        hot = O.run_ref_timed("curvature", d, d + "_out", threads=thr, reps=warmup + steps, variant=variant, progressName=v,
                                              progMin=300.0, progMax=1800.0)
                    shutil.rmtree(d + "_out", ignore_errors=True)
                    per_step += np.asarray(hot[warmup:warmup + steps])
            except Exception as e:
                if variant == "timed":
                    raise
                # the secondary (GPU) baseline is optional; keep WHY it is missing (on this pool: the tools fill their MultiFabs
                # from host code, so the reference's CUDA build needs AMReX's managed arena, and cudaMallocManaged fails with
                # CUDA error 999 inside these VMs -- AMReX_Arena.cpp:189; with the default device arena FillVar segfaults)
                msg = [ln for ln in str(e).splitlines() if "rror" in ln or "Segfault" in ln or "Abort" in ln]
                res[variant] = {"unavailable": (msg[0] if msg else str(e).splitlines()[0])[:240]}
                continue
            t = float(per_step.mean())
            res[variant] = (cells * len(names) / t / 1e9, t, thr, per_step.tolist())
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return res, names


def reference_arm(args, spec):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pf = spec["build"](fill=False)
    cfg = config_of(spec, pf)
    del pf
    try:
        res, names = run_reference(spec, args.steps, args.warmup)
        val, t, cores, per_step = res["timed"]
    except Exception as e:  # the oracle always exists; this only triggers on a broken checkout
        print(json.dumps({"impl": "reference", "unavailable": str(e).splitlines()[0][:200]}))
        return
    region = "grad.cpp:151-236" if spec["kind"] == "grad" else "curvature.cpp:283-791"
    line = {
        "impl": "reference", "metric": metric_name(spec["kind"]), "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": cfg,
        "details": {"timed_region": region + " minus FillVar (hot path, host memory to host memory), looped in-process",
                    "step": "one pass over every differentiated variable of the workload (%s): the whole workload, no sampling" % ", ".join(names)},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "reference",
                         "sample": "the whole workload: %d cells x %d variable(s) per step" % (cfg["cells"], len(names))},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = [int(s[0]) for s in self.samples if s[0].isdigit()]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples if len(s) > 2 + i)]
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.samples)}


def gen_fields(torch, levels, local_boxes, names, prob_hi=(1.0, 1.0, 1.0)):
    """Analytic fields (same formulas as peleanalysis_b200.synth) generated on the GPU, returned as pinned host
    tensors in host-concat order: one tensor per component per level."""
    import math
    out = []
    tp = 2.0 * math.pi
    for l, lv in enumerate(levels):
        comps = [[] for _ in names]
        for b in local_boxes[l]:
            lo, hi = lv.boxes[b]
            ax = [(torch.arange(lo[d], hi[d] + 1, device="cuda", dtype=torch.float64) - lv.domain_lo[d] + 0.5) * lv.dx[d] / prob_hi[d] for d in range(3)]
            X, Y, Z = ax[0][None, None, :], ax[1][None, :, None], ax[2][:, None, None]
            r = torch.sqrt((X - 0.5) ** 2 + (Y - 0.5) ** 2 + (Z - 0.5) ** 2)
            for c, n in enumerate(names):
                if n == "temp":
                    v = 300.0 + 750.0 * (1.0 + torch.tanh((0.25 - r) / 0.05)) + 5.0 * torch.sin(tp * X) * torch.cos(2 * tp * Y) + 0.0 * Z
                elif n == "x_velocity":
                    v = torch.sin(tp * X) * torch.cos(tp * Y) * torch.cos(tp * Z)
                elif n == "y_velocity":
                    v = -torch.cos(tp * X) * torch.sin(tp * Y) * torch.cos(tp * Z)
                elif n == "z_velocity":
                    v = 0.3 * torch.sin(2 * tp * Z) * torch.cos(tp * X) + 0.0 * Y
                else:
                    v = 0.05 * (1.0 - torch.tanh((0.25 - r) / 0.05)) + 0.001 * torch.sin(tp * (X + Y + Z))
                comps[c].append(v.reshape(-1))
        lvl = []
        for c in range(len(names)):
            n = sum(int(t.numel()) for t in comps[c])
            host = torch.empty(max(n, 1), dtype=torch.float64, pin_memory=True)[:n]
            if n:
                host.copy_(torch.cat(comps[c]))
            lvl.append(host)
        out.append(lvl)
        torch.cuda.synchronize()
    return out


class Ctx:
    """What every measurement needs: torch, the binding, the rank layout, the stream."""

    def __init__(self, torch, dist, capi, multigpu, rank, world, local_rank, stream, transport, no_links):
        self.torch, self.dist, self.capi, self.multigpu = torch, dist, capi, multigpu
        self.rank, self.world, self.local_rank, self.stream = rank, world, local_rank, stream
        self.transport, self.no_links = transport, no_links
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        self.peak = float(peaks.get("hbm_gbs", 6650.0))
        self.peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md 6.65 TB/s)"
        try:
            self.expected = json.load(open(HASH_FILE))
        except Exception:
            self.expected = {}

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_hash(self, h):
        """wrapping 64-bit sum of the ranks' fingerprints"""
        if self.world == 1:
            return h & (2 ** 64 - 1)
        t = self.torch.tensor([h - 2 ** 64 if h >= 2 ** 63 else h], device="cuda", dtype=self.torch.int64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return int(t.item()) & (2 ** 64 - 1)


DUMP_BYTES = 60_000_000          # --dump-outputs: the values of all files together; with the .npy headers they stay below 64 MB
DUMP_SEED = 20261020


def output_names(spec):
    """Names of the output components in Field order: gx, gy, gz, |grad| per variable, or the five curvature outputs."""
    if spec["kind"] == "grad":
        return ["%s_%s" % (v, k) for v in spec["names"] for k in ("gx", "gy", "gz", "gradmag")]
    v = spec["names"][0]
    return ["Progress", "MeanCurvature_" + v, "FlameNormalX_" + v, "FlameNormalY_" + v, "FlameNormalZ_" + v]


def dump_cells(cells, ncomp):
    """Host-concat indices of the cells --dump-outputs writes: all of them, or a sorted seeded sample within DUMP_BYTES."""
    n = min(cells, DUMP_BYTES // (8 * ncomp))
    return np.arange(cells) if n == cells else np.sort(np.random.default_rng(DUMP_SEED).choice(cells, n, replace=False))


def dump_outputs(spec, H, fout, out_dir):
    """Write every output component of the last step as out_dir/<name>.npy (float64, valid cells in host-concat order:
    levels, boxes, z-y-x).  Workloads larger than DUMP_BYTES keep the same seeded sample of cells in every component, so
    two builds run with the same arguments can be compared value for value."""
    names = output_names(spec)
    idx = dump_cells(H.num_cells, len(names))
    os.makedirs(out_dir, exist_ok=True)
    vals = np.empty((len(names), idx.size))
    off = 0
    for l, lv in enumerate(H.levels):
        for b, (lo, hi) in enumerate(lv.boxes):
            m = (hi[0] - lo[0] + 1) * (hi[1] - lo[1] + 1) * (hi[2] - lo[2] + 1)
            i0, i1 = np.searchsorted(idx, [off, off + m])
            if i1 > i0:
                for c in range(len(names)):
                    vals[c, i0:i1] = fout.download_box(l, b, c).ravel()[idx[i0:i1] - off]
            off += m
    for c, name in enumerate(names):
        np.save(os.path.join(out_dir, name + ".npy"), vals[c])


def measure(cx, spec, steps, warmup, e2e_steps=0, sampler=None, dump_dir=None):
    """Run one workload on the current rank layout.  Returns a dict with the device-resident timing, the dominant kernel's
    share, the optional host-buffer (e2e) timing and the output fingerprint; with dump_dir, also writes the outputs of the
    last timed step there (dump_outputs)."""
    torch, dist, capi, multigpu = cx.torch, cx.dist, cx.capi, cx.multigpu
    rank, world, stream = cx.rank, cx.world, cx.stream
    kind, names = spec["kind"], spec["names"]
    nvar = len(names)
    pf = spec["build"](fill=False)
    t0 = time.perf_counter()
    flags = capi.NO_LINKS if cx.no_links else (capi.PEER_LINKS if (world > 1 and cx.transport == "peer") else 0)
    H = capi.Hierarchy(pf.levels, (1, 1, 1), (0, 0, 0), rank, world, flags=flags)
    hier_s = time.perf_counter() - t0
    cells = H.num_cells
    host_in = gen_fields(torch, pf.levels, H.local_boxes, names)
    nout = 4 * nvar if kind == "grad" else 5
    fin = capi.Field(H, nvar, 1)
    fout = capi.Field(H, nout, 0 if kind == "grad" else 1)
    peer = bool(flags & capi.PEER_LINKS)
    if peer:
        multigpu.map_peers(fin)

    def upload(comps=range(nvar)):
        for l in range(H.nlev):
            if H.local_cells[l]:
                for c in comps:
                    capi.check(capi.lib().pa_field_upload_level(fin.f, l, c, host_in[l][c].data_ptr()))

    upload()
    capi.sync()
    if world > 1:
        dist.barrier()                 # every rank's inputs are resident before anyone reads them in place

    if kind == "grad":
        # whatever the neighbour links do not cover moves as NCCL send/recv of packed slabs (nothing, for peer transport
        # on a uniform grid)
        X = multigpu.SlabExchange(fin, nvar)

        def step(ev=None):
            X.run(0)
            capi.grad(fin, 0, nvar, fout, 0, phases=1)
            if ev is not None:
                ev[0].record(stream)
            capi.grad(fin, 0, nvar, fout, 0, phases=2)
            if ev is not None:
                ev[1].record(stream)
    else:
        lo = min([float(h[0].min()) for h in host_in if h[0].numel()] or [1e300])
        hi = max([float(h[0].max()) for h in host_in if h[0].numel()] or [-1e300])
        if world > 1:
            t = torch.tensor([-lo, hi], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            lo, hi = -float(t[0].item()), float(t[1].item())
        o = capi.CurvOpts()
        o.prog_min, o.prog_max = lo, hi
        if world > 1:
            op = multigpu.Curvature(fin, 0, o, fout, 0)

            def step(ev=None):
                op.run()
        else:
            def step(ev=None):
                capi.curvature(fin, 0, 0, o, fout, 0)

    for _ in range(warmup):
        step()
    cx.barrier()
    if sampler is not None:
        sampler.start()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)] if kind == "grad" else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0, f0 = capi.kernel_launches(), capi.curv_fused_launches()
    e0.record(stream)
    for i in range(steps):
        step(kev[i] if kev else None)
    e1.record(stream)
    cx.barrier()
    launches = capi.kernel_launches() - l0
    fused = capi.curv_fused_launches() - f0
    ms_step = cx.max_over_ranks(e0.elapsed_time(e1)) / steps
    value = cells * nvar / (ms_step * 1e-3) / 1e9
    alg_local = H.algorithmic_bytes(4) * nvar if kind == "grad" else H.algorithmic_bytes(5)      # this rank's boxes
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev])) if kev else e0.elapsed_time(e1) / steps
    res = {"value": value, "ms_per_step": ms_step, "cells": cells, "nvar": nvar, "launches": launches, "hier_build_s": hier_s,
           "alg_bytes_local": alg_local, "kernel_ms": kernel_ms, "local_cells": H.num_local_cells, "flags": flags,
           "boxes": [len(l.boxes) for l in pf.levels], "fused_launches": fused,
           "slab_cells_rank0": (X.roff[-1] // nvar) if kind == "grad" else None}

    # ---- fingerprint of the outputs of the last step ----
    res["output_hash"] = "%016x" % cx.sum_hash(fout.hash(0, nout))
    if dump_dir is not None:
        dump_outputs(spec, H, fout, dump_dir)

    # ---- e2e: host buffers through the C ABI (pinned H2D of inputs, hot path, D2H of all outputs) -------------
    if e2e_steps > 0:
        host_out = [[torch.empty(max(H.local_cells[l], 1), dtype=torch.float64, pin_memory=True)[:H.local_cells[l]] for _ in range(nout)]
                    for l in range(H.nlev)]
        s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()
        ev_end = torch.cuda.Event()

        def download(comps):
            for l in range(H.nlev):
                if H.local_cells[l]:
                    for c in comps:
                        capi.check(capi.lib().pa_field_download_level(fout.f, l, c, host_out[l][c].data_ptr()))

        if kind == "grad":
            # Pipelined by variable over three streams: H2D of variable v+1 (copy engine), hot path of v (SMs) and D2H of v's
            # four outputs (the other copy engine) overlap; PCIe is full duplex, so the step costs ~max(H2D, D2H), not the sum.
            X1 = multigpu.SlabExchange(fin, 1) if not X.empty else None
            ev_up = [torch.cuda.Event() for _ in range(nvar)]
            ev_g = [torch.cuda.Event() for _ in range(nvar)]

            def e2e_step():
                s_up.wait_event(ev_end)             # the previous step's readers (this rank's and the peers') are done
                capi.set_stream(s_up.cuda_stream)
                for v in range(nvar):
                    upload([v])
                    ev_up[v].record(s_up)
                for v in range(nvar):
                    stream.wait_event(ev_up[v])
                    capi.set_stream(stream.cuda_stream)
                    if peer:
                        multigpu.stream_barrier()   # peers' uploads of v landed before this rank's kernel reads them over NVLink
                    if X1 is not None:
                        X1.run(v)
                    capi.grad(fin, v, 1, fout, 4 * v)
                    ev_g[v].record(stream)
                    s_dn.wait_event(ev_g[v])
                    capi.set_stream(s_dn.cuda_stream)
                    download(range(4 * v, 4 * v + 4))
                capi.set_stream(stream.cuda_stream)
                if peer:
                    multigpu.stream_barrier()       # nobody re-uploads while a peer still reads the old data
                ev_end.record(stream)
        else:
            def e2e_step():
                upload()
                if peer:
                    multigpu.stream_barrier()
                step()
                download(range(nout))
                if peer:
                    multigpu.stream_barrier()
                ev_end.record(stream)

        ev_end.record(stream)
        e2e_step()
        cx.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        cx.barrier()
        e2e_s = cx.max_over_ranks((time.perf_counter() - t0) / e2e_steps)
        res["e2e"] = {"value": cells * nvar / e2e_s / 1e9, "unit": UNIT, "h2d_bytes_per_step": H.num_local_cells * nvar * 8,
                      "d2h_bytes_per_step": H.num_local_cells * nout * 8, "s_per_step": e2e_s}
        del host_out
    del fin, fout, host_in
    return res


FILTER3_DESC = "filterPlt of temp (box filter, base_fgr 2: ghost widths 1/2/4; max_grid_size 32), 3 levels, 256^3 base, ratio 2 (SURVEY 8(f) rank 4)"


def measure_filter(cx, steps, warmup, cpu_baseline=True):
    """filterPlt's compute block (filterPlt.cpp:166-221: FillPatch ghost cells + Filter::apply_filter of every level),
    device-resident, single GPU.  value = cells of all levels / step time.  The filter is a dense (2g+1)^3 weighted sum with
    separate multiplies and adds (bit parity with the reference forbids FMA), so for g >= 2 its bound is the FP64 pipe:
    fp64_frac = useful multiply+add operations / time / the MEASURED rate of that instruction mix on this GPU."""
    torch, P = cx.torch, cx.capi
    from peleanalysis_b200 import filterplt, synth
    pf = synth.config3(256, 64, fill=False)
    run = filterplt.FilterRun(P, pf, filter_type=1, base_fgr=2, max_grid_size=32, upload=False)
    names = ["temp"]
    # synthetic field values on the re-chopped grids, generated on the device
    fields = gen_fields(torch, run.levels, run.hier.local_boxes, names)
    for l in range(run.nlev):
        host = fields[l][0].cpu().numpy()
        run.fin.upload_level(l, 0, host)
    P.sync()
    ev = lambda: torch.cuda.Event(enable_timing=True)
    for _ in range(warmup):
        run.step()
    cx.torch.cuda.synchronize()
    l0 = P.kernel_launches()
    a, b = ev(), ev()
    a.record(cx.stream)
    for _ in range(steps):
        run.step()
    b.record(cx.stream)
    torch.cuda.synchronize()
    launches = P.kernel_launches() - l0
    ms = a.elapsed_time(b) / steps
    per_level = []
    for l in range(run.nlev):
        x, y, z = ev(), ev(), ev()
        x.record(cx.stream)
        P.fill_patch(run.fin, 0, 1, l, run.ngrow[l], 1)
        y.record(cx.stream)
        P.filter_level(run.fin, 0, run.fout, 0, 1, l, 1, run.fgr[l])
        z.record(cx.stream)
        torch.cuda.synchronize()
        per_level.append({"level": l, "ngrow": run.ngrow[l], "boxes": len(run.levels[l].boxes), "cells": run.levels[l].ncells,
                          "fill_ms": x.elapsed_time(y), "filter_ms": y.elapsed_time(z)})
    cells = run.cells()
    ops = sum(2.0 * (2 * g + 1) ** 3 * lv.ncells for g, lv in zip(run.ngrow, run.levels))
    peak = P.fp64_rate_gops()
    filt_ms = sum(x["filter_ms"] for x in per_level)
    rec = {"workload": FILTER3_DESC, "value": cells / (ms * 1e-3) / 1e9, "unit": UNIT, "n_gpus": 1, "ms_per_step": ms, "cells": cells,
           "boxes": [len(lv.boxes) for lv in run.levels], "launches_per_step": launches // max(1, steps), "levels": per_level,
           "roofline": {"bound": "fp64 pipe (separate multiply + add, no FMA)", "useful_ops": ops, "achieved": ops / (filt_ms * 1e-3) / 1e9,
                        "peak": peak, "unit": "Gop/s", "frac": ops / (filt_ms * 1e-3) / 1e9 / peak,
                        "peak_source": "measured on this GPU by pa_debug_fp64_rate (8 independent multiply-add chains per thread)",
                        "hbm_frac_level0": (16.0 * run.levels[0].ncells) / (per_level[0]["filter_ms"] * 1e-3) / 1e9 / cx.peak},
           "output_hash": hash_verdict(cx, "filter3", "%016x" % run.fout.hash(0, 1))}
    if cpu_baseline:
        try:
            rec["cpu_baseline"] = filter_reference(steps=2, warmup=1)
        except Exception as e:
            rec["cpu_baseline"] = {"value": None, "sample": "unavailable: " + str(e).splitlines()[0][:160]}
    return rec


def filter_reference(steps, warmup, base=64, mgs_in=32):
    """The reference filterPlt tool's timed build (oracle/_ref/filterPlt3d.timed.ex: probes around filterPlt.cpp:166-221) on
    all host cores.  The filter3 hierarchy has 50 M cells and the reference needs minutes per pass on it (ghost width 4 = 729
    terms per cell), so the baseline runs a bounded sample: the same three-level shape (equal cells per level, same ghost
    widths, same max_grid_size) with a smaller base grid.  Gcells/s is intensive in the grid size."""
    from oracle import oracle as O
    from peleanalysis_b200 import plotfile, synth
    if not os.path.exists(O.ref_exe("filterPlt3d.timed.ex")):
        raise RuntimeError("oracle/_ref/filterPlt3d.timed.ex is missing")
    pf = synth.config3(base, mgs_in, fill=True)
    cells = sum(l.ncells for l in pf.levels)
    basedir = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    tmp = tempfile.mkdtemp(prefix="pa_reff_", dir=basedir)
    cores = os.cpu_count() or 1
    try:
        d = os.path.join(tmp, "plt")
        plotfile.write_plotfile(d, pf, clean="remove")
        hot = O.run_ref_timed("filterPlt", d, os.path.join(tmp, "plt_filtered"), threads=cores, reps=warmup + steps, variables="temp")
        t = float(np.mean(hot[warmup:]))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return {"value": cells / t / 1e9, "unit": UNIT, "cores": cores, "kind": "reference", "hot_path_seconds": t,
            "sample": "filterPlt of temp on a %d^3-base three-level hierarchy (%d cells; the workload's shape, ghost widths and max_grid_size at "
                      "1/%d of its cells); %d timed repetitions of filterPlt.cpp:166-221" % (base, cells, (256 // base) ** 3, steps)}


def hash_verdict(cx, name, h):
    want = cx.expected.get(name)
    return {"value": h, "expected": want, "ok": (want is None or want == h)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="config2")
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--transport", default="peer", choices=["peer", "slab"])
    ap.add_argument("--no-links", action="store_true", help="materialise every ghost cell (reference data flow)")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary workloads")
    ap.add_argument("--only-extra", default=None, help="run just one workload device-resident and print its short record (profiling aid)")
    ap.add_argument("--write-hashes", action="store_true", help="(N=1) record this run's fingerprints in tests/golden/bench_hashes.json")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="(N=1) write the outputs of the last timed step of the workload as DIR/<name>.npy (float64; a fixed seeded "
                         "sample of cells when all of them would exceed %d MB)" % (DUMP_BYTES // 1000000))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    filter_only = args.only_extra == "filter3"
    if args.dump_outputs and (filter_only or args.impl == "reference" or args.gpus > 1):
        ap.error("--dump-outputs covers the grad and curvature workloads of the B200 arm on one GPU")
    spec = workload_spec("config2" if filter_only else (args.only_extra or args.workload))
    if args.impl == "reference":
        return reference_arm(args, spec)

    import torch
    import torch.distributed as dist
    from peleanalysis_b200 import build, capi, multigpu

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    build.build()                       # no-op when the in-tree .so is current
    torch.cuda.set_device(local_rank)
    capi.init(local_rank)               # raises if there is no B200: no CPU fallback
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.current_stream()
    capi.set_stream(stream.cuda_stream)
    cx = Ctx(torch, dist, capi, multigpu, rank, world, local_rank, stream, args.transport, args.no_links)

    def short(name, r):
        per_rank_alg = r["alg_bytes_local"]
        return {"workload": workload_spec(name)["desc"], "value": r["value"], "unit": UNIT, "n_gpus": world, "ms_per_step": r["ms_per_step"],
                "cells": r["cells"], "boxes": r["boxes"], "launches_per_step": r["launches"] // max(1, r["steps"]),
                "algorithmic_bytes": per_rank_alg, "roofline_frac": per_rank_alg / (r["ms_per_step"] * 1e-3) / 1e9 / cx.peak,
                "hier_build_s": r["hier_build_s"], "output_hash": hash_verdict(cx, name, r["output_hash"])}

    if filter_only:
        if world > 1:
            raise SystemExit("filter3 is a single-GPU workload")
        print(json.dumps(measure_filter(cx, args.steps, args.warmup, cpu_baseline=not args.no_cpu_baseline)))
        return
    if args.only_extra:
        r = measure(cx, spec, args.steps, args.warmup, dump_dir=args.dump_outputs)
        r["steps"] = args.steps
        if rank == 0:
            print(json.dumps(short(args.only_extra, r)))
        if world > 1:
            dist.destroy_process_group()
        return

    sampler = ClockSampler(local_rank) if rank == 0 else None
    r = measure(cx, spec, args.steps, args.warmup, e2e_steps=args.e2e_steps, sampler=sampler, dump_dir=args.dump_outputs)
    r["steps"] = args.steps
    if sampler is not None:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    kind, nvar = spec["kind"], len(spec["names"])
    hashes = {args.workload: r["output_hash"]}

    extras = None
    if not args.no_extras:
        extras = {}
        # every N: the strong-scaling workload BASELINE names and the north-star hierarchy (both tools); N = 1 also the rest
        kinds = ["config4", "target_grad", "target_curv"] + (["curvature3", "grad5"] if world == 1 else [])
        for name in kinds:
            if name == args.workload:
                continue
            try:
                x = measure(cx, workload_spec(name), max(5, args.steps // 2), 3)
                x["steps"] = max(5, args.steps // 2)
                extras[name] = short(name, x)
                hashes[name] = x["output_hash"]
            except Exception as e:
                extras[name] = {"error": str(e).splitlines()[0][:200]}
                if world > 1:
                    raise                         # a rank that fails alone would hang the others at the next collective

    if extras is not None and world == 1:
        try:
            extras["filter3"] = measure_filter(cx, max(3, args.steps // 4), 2, cpu_baseline=not args.no_cpu_baseline)
            hashes["filter3"] = extras["filter3"]["output_hash"]["value"]
        except Exception as e:
            extras["filter3"] = {"error": str(e).splitlines()[0][:200]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    if args.write_hashes and world == 1:
        cur = dict(cx.expected)
        cur.update(hashes)
        with open(HASH_FILE, "w") as f:
            json.dump(cur, f, indent=1, sort_keys=True)
        cx.expected = cur

    cpu = None
    ref_gpu = None
    if not args.no_cpu_baseline and world == 1:
        try:
            one = [spec["names"][-2] if args.workload.startswith("config2") else spec["names"][0]]
            res, ran = run_reference(spec, steps=3, warmup=1, variables=one, variants=("timed", "cuda.timed"))
            v, t, cores, _ = res["timed"]
            sample = "%s of %s on the workload's own grid (%d cells), %d of its %d variable(s); 3 timed repetitions of the tool's hot-path region" % (
                "grad" if kind == "grad" else "curvature", ran[0], r["cells"], len(ran), nvar)
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "reference", "hot_path_seconds": t, "sample": sample}
            if isinstance(res.get("cuda.timed"), dict):
                ref_gpu = {"value": None, "unit": UNIT, "kind": "the reference's own CUDA build (oracle/build_ref_cuda.py) on this GPU",
                           "unavailable": res["cuda.timed"]["unavailable"]}
            elif res.get("cuda.timed"):
                gv, gt, _, _ = res["cuda.timed"]
                ref_gpu = {"value": gv, "unit": UNIT, "kind": "the reference's own CUDA build (AMReX ParallelFor backend, USE_CUDA=TRUE CUDA_ARCH=100, "
                           "oracle/build_ref_cuda.py) on this GPU, same probes as cpu_baseline", "hot_path_seconds": gt, "sample": sample}
        except Exception as e:
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference", "sample": "unavailable: " + str(e).splitlines()[0][:160]}

    pf = spec["build"](fill=False)
    cfg = config_of(spec, pf)
    alg_bytes = r["alg_bytes_local"]
    achieved = alg_bytes / (r["kernel_ms"] * 1e-3) / 1e9
    traffic = None
    traffic_src = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "stencil_traffic.json")))
        ent = tj.get(args.workload)
        if isinstance(ent, dict):
            traffic, traffic_src = ent.get("dram_bytes"), ent.get("source")
        if traffic is not None and world > 1:
            traffic = int(traffic * r["local_cells"] / max(r["cells"], 1))
    except Exception:
        pass
    if kind == "grad":
        kname = "k_stencil_tma<MODE_GRAD>" if os.environ.get("PA_STENCIL", "tma") != "simple" else "k_stencil_simple<MODE_GRAD>"
    else:
        kname = "k_curv_fused (whole step: ghost fills + fused kernel + shell pass)" if r["fused_launches"] else "k_stencil_tma<NORMAL_S> + <DIV> (whole step)"
    hv = hash_verdict(cx, args.workload, r["output_hash"])
    line = {
        "metric": metric_name(kind), "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": cfg,
        "details": {"parallelism": ("1 GPU" if world == 1 else "boxes distributed over %d ranks along a (z, y, x) curve; cross-rank ghosts: %s" % (
                        world, "read in place over NVLink (CUDA-IPC peer links, no exchange step)" if r["flags"] & capi.PEER_LINKS
                        else "NCCL send/recv of packed slabs (%s cells/step recv on rank 0)" % r["slab_cells_rank0"])),
                    "ghosts": "materialised (PA_HIER_NO_LINKS)" if args.no_links else "same-level neighbours read in place by the stencil (neighbour links)",
                    "stencil": os.environ.get("PA_STENCIL", "tma"), "hier_build_s": r["hier_build_s"],
                    "row_align_bytes": int(os.environ.get("PA_ROW_ALIGN", "32"))},
        "e2e": r.get("e2e"),
        "gpu_launches": int(r["launches"]),
        "clocks": sampler.summary(),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": cx.peak, "unit": "GB/s", "frac": achieved / cx.peak, "traffic": traffic,
                     "traffic_source": traffic_src, "kernel": kname, "kernel_ms": r["kernel_ms"], "algorithmic_bytes": alg_bytes,
                     "peak_source": cx.peak_src,
                     "step_frac": alg_bytes / (r["ms_per_step"] * 1e-3) / 1e9 / cx.peak},
        "output_hash": hv,
        "cpu_baseline": cpu,
        "ref_gpu_baseline": ref_gpu,
        "extras": extras,
    }
    print(json.dumps(line))
    bad = [n for n, x in [(args.workload, hv)] + [(n, e.get("output_hash", {})) for n, e in (extras or {}).items()] if x and x.get("ok") is False]
    if world > 1:
        dist.destroy_process_group()
    if bad:
        print("output fingerprint mismatch: " + ", ".join(bad), file=sys.stderr)
        sys.exit(3)


if __name__ == "__main__":
    main()
