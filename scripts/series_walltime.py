#!/usr/bin/env python3
"""Wall time of a series of plotfiles (infiles=, host/series.hpp) against one process per file, per tool.

K plotfiles of the tool_walltime.py shape (3 levels, base^3 cells per level, 64^3 boxes) on /dev/shm; the data differ per file
(phase-shifted fields) and the fine grids of every other file are shifted.  For grad, curvature and filterPlt:
  (a) K single-file runs (one process each), (b) one series run, (c) the reference executable per file where it is built,
  and series runs at ngpus=N for every N up to the GPUs present (N > 1).
Every output of (b) must equal the output of (a) byte for byte (the script fails otherwise).  Prints one JSON line per tool
with seconds per file, the series' per-stage means from its verbose lines, and the speed-ups; the first line records the card
name and power limit.
python scripts/series_walltime.py [base=256] [K=8]"""
import filecmp
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402
from peleanalysis_b200 import plotfile, synth  # noqa: E402

base = int(sys.argv[1]) if len(sys.argv) > 1 else 256
K = int(sys.argv[2]) if len(sys.argv) > 2 else 8
HOST = os.path.join(ROOT, "peleanalysis_b200", "host")
TOOLS = (("grad", "grad3d.ref.ex", "grad3d.b200.ex", ["gradVar=temp"], "_gt"),
         ("curvature", "curvature3d.ref.ex", "curvature3d.b200.ex", ["progressName=temp"], "_K"),
         ("filterPlt", "filterPlt3d.ref.ex", "filterPlt3d.b200.ex", ["variables=temp", "max_filter_level=1"], "_filtered"))
env = dict(os.environ, OMP_NUM_THREADS=str(os.cpu_count() or 1))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    if q.returncode != 0 or not q.stdout.strip():
        raise SystemExit("series_walltime: no GPU (nvidia-smi found none); this is a GPU measurement")
    return [ln.strip() for ln in q.stdout.strip().splitlines()]


def series_file(k):
    """config3's hierarchy; odd k: both fine levels shifted (level 1 by 32 cells, level 2 by 64) in x, properly nested"""
    n = base
    q = n // 4
    l1 = [(q * 2, q * 2, q * 2), (q * 2 + n - 1, q * 2 + n - 1, q * 2 + n - 1)]
    l2 = [((q * 2 + n // 4) * 2,) * 3, ((q * 2 + n // 4) * 2 + n - 1,) * 3]
    if k % 2:
        s1, s2 = n // 8, n // 4
        l1 = [(l1[0][0] + s1,) + l1[0][1:], (l1[1][0] + s1,) + l1[1][1:]]
        l2 = [(l2[0][0] + s2,) + l2[0][1:], (l2[1][0] + s2,) + l2[1][1:]]
    pf = synth.make_hierarchy(n, [[tuple(l1)], [tuple(l2)]], [2, 2], 64, ("temp",), fill=False)
    for lv in pf.levels:
        synth.fill_level(lv, pf.names, pf.prob_lo, pf.prob_hi,
                         fn=lambda name, x, y, z, ph: synth.field_values(name, x, y, z, ph, phase=0.37 * k))
    return pf


def run(cmd, cwd):
    t0 = time.time()
    p = subprocess.run(cmd, capture_output=True, text=True, cwd=cwd, env=env)
    dt = time.time() - t0
    if p.returncode != 0:
        raise RuntimeError(" ".join(cmd[:3]) + " ...\n" + p.stdout[-800:] + p.stderr[-800:])
    return dt, p.stdout


def same_tree(a, b):
    fa = sorted(os.path.relpath(os.path.join(r, f), a) for r, _, fs in os.walk(a) for f in fs)
    fb = sorted(os.path.relpath(os.path.join(r, f), b) for r, _, fs in os.walk(b) for f in fs)
    return fa == fb and all(filecmp.cmp(os.path.join(a, f), os.path.join(b, f), shallow=False) for f in fa)


def stage_means(out):
    rows = [tuple(float(v) for v in m.groups()) for m in
            (re.search(r"read (\S+) s, gpu (\S+) s, write (\S+) s, device bytes (\d+)", ln) for ln in out.splitlines()) if m]
    if len(rows) != K:
        raise RuntimeError("expected %d verbose series lines, got %d" % (K, len(rows)))
    return {"read_s": round(sum(r[0] for r in rows) / K, 3), "gpu_s": round(sum(r[1] for r in rows) / K, 3),
            "write_s": round(sum(r[2] for r in rows) / K, 3), "device_bytes": sorted({int(r[3]) for r in rows})}


def main():
    cards = card()
    print(json.dumps({"cards": cards, "base": base, "K": K, "host_cores": os.cpu_count()}), flush=True)
    subprocess.check_call(["make", "-s", "-C", HOST])
    tmp = tempfile.mkdtemp(prefix="pa_series_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        src = os.path.join(tmp, "in")
        os.makedirs(src)
        files = []
        for k in range(K):
            p = os.path.join(src, "plt%05d" % (100 * (k + 1)))
            pf = series_file(k)
            plotfile.write_plotfile(p, pf, clean="remove")
            cells = sum(lv.ncells for lv in pf.levels)
            del pf
            files.append(p)
        for tool, ref, mine, args, suffix in TOOLS:
            exe = os.path.join(HOST, mine)
            rec = {"tool": tool, "files": K, "cells_per_file": cells, "args": args}
            da, db = os.path.join(tmp, "a"), os.path.join(tmp, "b")
            os.makedirs(da)
            os.makedirs(db)
            ta = sum(run([exe, "infile=" + f, *args], da)[0] for f in files)
            tb, out = run([exe, "infiles=" + " ".join(files), "verbose=1", *args], db)
            for f in files:
                o = os.path.basename(f) + suffix
                if not same_tree(os.path.join(da, o), os.path.join(db, o)):
                    raise SystemExit("series_walltime: %s output of %s differs between the single and the series run" % (tool, o))
            rec["outputs_byte_identical"] = True
            rec["single_runs_s_per_file"] = round(ta / K, 3)
            rec["series_s_per_file"] = round(tb / K, 3)
            rec["series_stage_means"] = stage_means(out)
            rec["speedup_series_vs_single"] = round(ta / tb, 2)
            shutil.rmtree(da)
            shutil.rmtree(db)
            ngpu = len(cards)
            for n in range(2, ngpu + 1):
                dn = os.path.join(tmp, "n%d" % n)
                os.makedirs(dn)
                tn, _ = run([exe, "infiles=" + " ".join(files), "ngpus=%d" % n, *args], dn)
                rec["series_ngpus%d_s_per_file" % n] = round(tn / K, 3)
                shutil.rmtree(dn)
            if O.have_ref() and os.path.exists(O.ref_exe(ref)):
                dr = os.path.join(tmp, "r")
                os.makedirs(dr)
                tr = 0.0
                for f in files:
                    extra = [] if tool == "filterPlt" else ["outfile=" + os.path.join(dr, os.path.basename(f) + suffix)]
                    tr += run([O.ref_exe(ref), "infile=" + f, *args, *extra], dr)[0]
                    shutil.rmtree(dr)
                    os.makedirs(dr)
                rec["reference_s_per_file"] = round(tr / K, 3)
                rec["speedup_series_vs_reference"] = round(tr / tb, 2)
                shutil.rmtree(dr)
            else:
                rec["reference_s_per_file"] = "not measured (reference not built)"
            print(json.dumps(rec), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
