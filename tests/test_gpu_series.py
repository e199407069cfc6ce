"""GPU (-m gpu): a series of plotfiles in one run (infiles=, host/series.hpp and mgtools).  Every output of a series run is
byte-identical (Header, Cell_H, every Cell_D file) to the output of a single run on that file; the up-front checks stop a bad
series before anything is written; device memory does not grow from file to file.  tests/test_emu_series.py runs the same
bodies against the emulated library."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from helpers import load_golden
from peleanalysis_b200 import plotfile

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "peleanalysis_b200", "host")
SUFFIX = {"grad": "_gt", "curvature": "_K", "filter": "_filtered"}
TOOL = {"grad": 0, "curvature": 1, "filter": 2}

# (tool, keys): the cases every series is run with
CASES = [
    ("grad", ["gradVar=temp", "Aux_Variables=Y"]),
    ("curvature", ["progressName=temp"]),
    ("curvature", ["progressName=temp", "threshold_prog=1", "threshold_value=0.01", "do_gaussCurv=1"]),
    ("curvature", ["progressName=temp", "do_smooth=1", "smoothing_time=1e-5", "smooth_precond=mg"]),
    ("filter", ["interp_type=0"]),
    ("filter", ["interp_type=1"]),
]
CASE_IDS = ["grad_aux", "curv_default", "curv_threshold_gauss", "curv_smooth_mg", "filter_pc", "filter_linear"]


@pytest.fixture(scope="module")
def exes(gpu):
    import fcntl
    with open(os.path.join(HOST, ".build.lock"), "w") as lk:
        fcntl.flock(lk, fcntl.LOCK_EX)
        subprocess.check_call(["make", "-s", "-C", HOST])
    return os.path.join(HOST, "grad3d.b200.ex"), os.path.join(HOST, "curvature3d.b200.ex"), os.path.join(HOST, "filterPlt3d.b200.ex")


def _with_aux(pf, scale, shift):
    """pf with its temp data remapped (scale, shift) and a second variable Y derived from it"""
    c = pf.comp("temp")
    for lv in pf.levels:
        fabs = []
        for f in lv.fabs:
            t = f[c] * scale + shift
            fabs.append(np.stack([t, 0.25 + 0.5 * np.sin(3.0 * t)]))
        lv.fabs = fabs
    pf.names = ["temp", "Y"]
    return pf


def make_series(d, drop_aux_in=None):
    """Four plotfiles: c3_three_levels, the same grids with other data, c1_corner_sym (two levels) and lshape (ragged fine
    level).  drop_aux_in = index of a file written without the variable Y."""
    specs = [("c3_three_levels", 1.0, 0.0), ("c3_three_levels", 0.8, 0.15), ("c1_corner_sym", 1.1, -0.05), ("lshape", 0.9, 0.05)]
    paths = []
    for i, (name, a, b) in enumerate(specs):
        pf = _with_aux(load_golden(name)[0], a, b)
        if i == drop_aux_in:
            for lv in pf.levels:
                lv.fabs = [f[:1] for f in lv.fabs]
            pf.names = ["temp"]
        p = os.path.join(d, "plt%05d" % (100 * (i + 1)))
        plotfile.write_plotfile(p, pf)
        paths.append(p)
    return paths


def _run(cmd, cwd, env=None):
    p = subprocess.run(cmd, capture_output=True, text=True, cwd=cwd, env=env)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    return p.stdout


def assert_same_tree(a, b):
    """two plotfile directories equal file for file, byte for byte"""
    fa = sorted(os.path.relpath(os.path.join(r, f), a) for r, _, fs in os.walk(a) for f in fs)
    fb = sorted(os.path.relpath(os.path.join(r, f), b) for r, _, fs in os.walk(b) for f in fs)
    assert fa == fb, (a, b)
    assert any(f.endswith("Cell_H") for f in fa) and any("Cell_D_" in f for f in fa)
    for f in fa:
        with open(os.path.join(a, f), "rb") as x, open(os.path.join(b, f), "rb") as y:
            assert x.read() == y.read(), (a, f)


def check_series_identity(exes, tmp_path, tool, keys, ngpus=1, env=None):
    """infiles= over the four files == one infile= run per file, byte for byte"""
    exe = exes[TOOL[tool]]
    src = str(tmp_path / "in")
    os.makedirs(src)
    files = make_series(src)
    single, series = tmp_path / "single", tmp_path / "series"
    os.makedirs(str(single))
    os.makedirs(str(series))
    for f in files:
        _run([exe, "infile=" + f, *keys], cwd=str(single), env=env)
    _run([exe, "infiles=" + " ".join(files), "ngpus=%d" % ngpus, *keys], cwd=str(series), env=env)
    for f in files:
        out = os.path.basename(f) + SUFFIX[tool]
        assert_same_tree(str(single / out), str(series / out))
    assert sorted(os.listdir(str(series))) == sorted(os.listdir(str(single)))


@pytest.mark.parametrize("tool,keys", CASES, ids=CASE_IDS)
def test_series_identical_to_single_runs(exes, tmp_path, tool, keys):
    check_series_identity(exes, tmp_path, tool, keys)


def _ngpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_ngpus() < 2, reason="needs two GPUs in one box")
@pytest.mark.parametrize("tool,keys", [CASES[0], CASES[3], CASES[5]], ids=["grad_aux", "curv_smooth_mg", "filter_linear"])
def test_series_on_two_gpus(exes, tmp_path, tool, keys):
    check_series_identity(exes, tmp_path, tool, keys, ngpus=2)


def check_errors(exes, tmp_path, env=None):
    src = str(tmp_path / "in")
    os.makedirs(src)
    files = make_series(src, drop_aux_in=2)
    wd = str(tmp_path / "wd")
    os.makedirs(wd)

    def fails(exe, *args):
        p = subprocess.run([exe, *args], capture_output=True, text=True, cwd=wd, env=env)
        assert p.returncode != 0, p.stdout
        assert "amrex::Abort" in p.stderr, p.stderr
        return p.stderr

    # a variable missing in the third file: the single run's message, prefixed with that file; nothing written
    err = fails(exes[0], "infiles=" + " ".join(files), "gradVar=temp", "Aux_Variables=Y")
    assert files[2] + ": Unknown auxiliary variable name: Y" in err, err
    err = fails(exes[2], "infiles=" + " ".join(files), "variables=temp Y")
    assert files[2] + ": Variable 'Y' not found in file" in err, err
    err = fails(exes[1], "infiles=" + " ".join(files), "progressName=Y")
    assert files[2] + ": Wrong progress variable name: Y" in err, err
    assert os.listdir(wd) == []
    # keys that name one file
    for k in ("infile=" + files[0], "outfile=x", "transport=slab"):
        fails(exes[0], "infiles=" + files[0], k)
    fails(exes[1], "infiles=" + files[0], "outfile=x")
    fails(exes[2], "infiles=" + files[0], "infile=" + files[1])
    # two inputs with the same root name
    other = os.path.join(str(tmp_path), "other")
    os.makedirs(other)
    dup = os.path.join(other, os.path.basename(files[1]))
    shutil.copytree(files[1], dup)
    err = fails(exes[0], "infiles=" + " ".join([files[0], files[1], dup]))
    assert "both write" in err and os.path.basename(files[1]) + "_gt" in err, err
    assert os.listdir(wd) == []
    # an unreadable header
    err = fails(exes[1], "infiles=" + files[0] + " " + os.path.join(str(tmp_path), "missing"))
    assert "missing: cannot read plotfile" in err, err
    assert os.listdir(wd) == []


def test_series_errors(exes, tmp_path):
    check_errors(exes, tmp_path)


def check_existing_output_renamed(exes, tmp_path, env=None):
    src = str(tmp_path / "in")
    os.makedirs(src)
    files = make_series(src)[:2]
    wd = tmp_path / "wd"
    os.makedirs(str(wd))
    _run([exes[0], "infile=" + files[0], "gradVar=temp"], cwd=str(wd), env=env)
    first = (wd / "plt00100_gt" / "Header").read_bytes()
    (wd / "plt00100_gt" / "marker").write_text("old")
    _run([exes[0], "infiles=" + " ".join(files), "gradVar=temp"], cwd=str(wd), env=env)
    old = [n for n in os.listdir(str(wd)) if n.startswith("plt00100_gt.old.")]
    assert len(old) == 1, os.listdir(str(wd))
    assert (wd / old[0] / "marker").read_text() == "old"
    assert not (wd / "plt00100_gt" / "marker").exists()
    assert (wd / "plt00100_gt" / "Header").read_bytes() == first
    assert (wd / "plt00200_gt").is_dir()


def test_series_renames_existing_output(exes, tmp_path):
    check_existing_output_renamed(exes, tmp_path)


def check_no_device_memory_growth(exes, tmp_path, tool, keys, env=None):
    """six files, 4-6 copies of 1-3 under other names: the device bytes after files 4-6 equal those after files 1-3"""
    src = str(tmp_path / "in")
    os.makedirs(src)
    files = make_series(src)[1:]
    for i, f in enumerate(list(files)):
        c = os.path.join(src, "copy%d" % i)
        shutil.copytree(f, c)
        files.append(c)
    wd = str(tmp_path / "wd")
    os.makedirs(wd)
    out = _run([exes[TOOL[tool]], "infiles=" + " ".join(files), "verbose=1", *keys], cwd=wd, env=env)
    got = {}
    for line in out.splitlines():
        m = re.match(r"\[b200\] series (\d+)/6 .*: read \S+ s, gpu \S+ s, write \S+ s, device bytes (\d+)$", line)
        if m:
            got[int(m.group(1))] = int(m.group(2))
    assert sorted(got) == [1, 2, 3, 4, 5, 6], out
    assert [got[4], got[5], got[6]] == [got[1], got[2], got[3]], got
    return got


@pytest.mark.parametrize("tool,keys", [CASES[0], CASES[2], CASES[3], CASES[5]], ids=["grad_aux", "curv_threshold_gauss", "curv_smooth_mg", "filter_linear"])
def test_series_no_device_memory_growth(exes, tmp_path, tool, keys):
    check_no_device_memory_growth(exes, tmp_path, tool, keys)


def check_device_bytes_binding(capi):
    """pa_debug_device_bytes counts a field's slabs while it lives and drops back to the same value when it is freed"""
    from peleanalysis_b200 import synth
    H = capi.Hierarchy(synth.config1(16, 8).levels)
    keep = capi.Field(H, 1, 1)                       # the hierarchy's device tables exist from here on
    base = capi.device_bytes()
    f = capi.Field(H, 3, 1)
    assert capi.device_bytes() - base >= f.nbytes > 0
    f.free()
    assert capi.device_bytes() == base
    keep.free()


def test_device_bytes_binding(gpu):
    check_device_bytes_binding(gpu)


# ---- mgtools infiles= ----------------------------------------------------------------------------------------------------
MG_CASES = [("grad", ["gradVar=temp", "Aux_Variables=Y"]), ("curvature", ["progressName=temp", "do_smooth=1", "smoothing_time=1e-5"]),
            ("filter", ["interp_type=1"])]


def check_mgtools_series(run_world, tmp_path, tool, keys, worlds):
    """mgtools <tool> infiles= at each world size == single-file world-1 mgtools runs, byte for byte.  run_world(world, args,
    cwd) runs mgtools.run(tool, args) on `world` ranks with working directory cwd."""
    src = str(tmp_path / "in")
    os.makedirs(src)
    files = make_series(src)
    single = str(tmp_path / "single")
    os.makedirs(single)
    for f in files:
        run_world(1, tool, ["infile=" + f] + keys, single)
    for w in worlds:
        wd = str(tmp_path / ("w%d" % w))
        os.makedirs(wd)
        run_world(w, tool, ["infiles=" + " ".join(files)] + keys, wd)
        for f in files:
            out = os.path.basename(f) + SUFFIX[tool]
            assert_same_tree(os.path.join(single, out), os.path.join(wd, out))


def _mgtools_worker(rank, world, port, tool, args, cwd, q):
    import sys
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    os.chdir(cwd)
    from peleanalysis_b200 import mgtools
    try:
        mgtools.run(tool, args, backend="gloo")
        q.put((rank, "ok"))
    except SystemExit as e:
        q.put((rank, str(e)))


def run_world_processes(worker, world, tool, args, cwd):
    """mgtools on `world` spawned ranks (gloo); worker(rank, world, port, tool, args, cwd, queue) is the rank's body"""
    import multiprocessing as mp
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=worker, args=(r, world, port, tool, args, cwd, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=1200) for _ in procs)
    for p in procs:
        p.join(timeout=120)
    assert res == {r: "ok" for r in range(world)}, res


@pytest.mark.parametrize("tool,keys", MG_CASES, ids=["grad_aux", "curv_smooth", "filter_linear"])
def test_mgtools_series(gpu, tmp_path, tool, keys):
    worlds = [1, 2] if _ngpus() >= 2 else [1]
    check_mgtools_series(lambda w, t, a, cwd: run_world_processes(_mgtools_worker, w, t, a, cwd), tmp_path, tool, keys, worlds)
