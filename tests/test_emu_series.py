"""CPU tier: the checks of tests/test_gpu_series.py (a series of plotfiles in one run: infiles= of the three executables and of
mgtools) against the EMULATED library of tests/emu, including ngpus=2 and 3 on emulated GPUs (CUEMU_DEVICES) and mgtools at
world 2 over gloo."""
import fcntl
import importlib.util
import os
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "emu"))

import test_gpu_series as S  # noqa: E402  (the GPU tests' bodies, reused as plain functions)
from test_emu_smooth import emu  # noqa: E402,F401  (fixture: the emulated binding)
from test_emu_tools import emu_exes  # noqa: E402,F401  (fixture: the emulated host executables)

EMU_ENV = dict(os.environ, PA_NORMAL_MATH="fast")


@pytest.fixture(scope="module")
def exes(request):
    """the emulated executables, relinked when series.hpp is newer than they are"""
    import build_emu
    out = os.path.dirname(build_emu.LIB)
    dep = os.path.join(ROOT, "peleanalysis_b200", "host", "series.hpp")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, ".exe_build.lock"), "w") as lk:
        fcntl.flock(lk, fcntl.LOCK_EX)
        for n in ("grad3d.emu.ex", "curvature3d.emu.ex", "filterPlt3d.emu.ex"):
            e = os.path.join(out, n)
            if os.path.exists(e) and os.path.getmtime(e) < os.path.getmtime(dep):
                os.remove(e)
    return request.getfixturevalue("emu_exes")


@pytest.mark.parametrize("tool,keys", S.CASES, ids=S.CASE_IDS)
def test_emulated_series_identical_to_single_runs(exes, tmp_path, tool, keys):
    S.check_series_identity(exes, tmp_path, tool, keys, env=EMU_ENV)


@pytest.mark.parametrize("ngpus", [2, 3])
@pytest.mark.parametrize("tool,keys", [S.CASES[0], S.CASES[3], S.CASES[5]], ids=["grad_aux", "curv_smooth_mg", "filter_linear"])
def test_emulated_series_on_several_gpus(exes, tmp_path, tool, keys, ngpus):
    S.check_series_identity(exes, tmp_path, tool, keys, ngpus=ngpus, env=dict(EMU_ENV, CUEMU_DEVICES=str(ngpus)))


def test_emulated_series_errors(exes, tmp_path):
    S.check_errors(exes, tmp_path, env=EMU_ENV)


def test_emulated_series_renames_existing_output(exes, tmp_path):
    S.check_existing_output_renamed(exes, tmp_path, env=EMU_ENV)


@pytest.mark.parametrize("tool,keys", [S.CASES[0], S.CASES[2], S.CASES[3], S.CASES[5]], ids=["grad_aux", "curv_threshold_gauss", "curv_smooth_mg", "filter_linear"])
def test_emulated_series_no_device_memory_growth(exes, tmp_path, tool, keys):
    S.check_no_device_memory_growth(exes, tmp_path, tool, keys, env=EMU_ENV)


def test_emulated_device_bytes_binding(emu):
    S.check_device_bytes_binding(emu)


def _mgtools_worker(rank, world, port, tool, args, cwd, q):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), PA_NORMAL_MATH="fast")
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.join(HERE, "emu"))
    os.chdir(cwd)
    import build_emu
    from peleanalysis_b200 import capi as product_capi, mgtools
    spec = importlib.util.spec_from_file_location("capi_emulated_series", product_capi.__file__)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    m.LIB_PATH = build_emu.LIB
    try:
        mgtools.run(tool, args, capi=m, backend="gloo", device=0)
        q.put((rank, "ok"))
    except SystemExit as e:
        q.put((rank, str(e)))


@pytest.mark.parametrize("tool,keys", S.MG_CASES, ids=["grad_aux", "curv_smooth", "filter_linear"])
def test_emulated_mgtools_series(emu, tmp_path, tool, keys):
    """world 1 and world 2 (gloo); do_smooth=1 is accepted at world 2 because every file runs on one rank"""
    S.check_mgtools_series(lambda w, t, a, cwd: S.run_world_processes(_mgtools_worker, w, t, a, cwd), tmp_path, tool, keys, [1, 2])


def test_emulated_mgtools_series_errors(tmp_path):
    from peleanalysis_b200 import mgtools, plotfile
    from helpers import load_golden
    d = str(tmp_path / "a" / "plt")
    os.makedirs(os.path.dirname(d))
    plotfile.write_plotfile(d, load_golden("c1_periodic")[0])
    e = str(tmp_path / "b" / "plt")
    os.makedirs(os.path.dirname(e))
    plotfile.write_plotfile(e, load_golden("c1_periodic")[0])
    for args, msg in ((["infiles=" + d, "outfile=x"], "cannot be combined with outfile"),
                      (["infiles=" + d, "infile=" + d], "cannot be combined with infile"),
                      (["infiles=" + d, "transport=slab"], "cannot be combined with transport"),
                      (["infiles=" + d + " " + e], "both write plt_gt"),
                      (["infiles=" + d + " " + str(tmp_path / "missing")], "missing: cannot read plotfile")):
        with pytest.raises(SystemExit) as x:
            mgtools.run("grad", args)
        assert msg in str(x.value), (args, str(x.value))
