"""CPU tier: pa_smooth's multigrid preconditioner with the kernel SOURCES run under the CUDA execution-model emulator of
tests/emu -- the checks of tests/test_gpu_smooth_mg.py, plus `mgtools curvature smooth_precond=mg` at world 1 against the
emulated executable."""
import multiprocessing as mp
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emu"))

import test_gpu_smooth as G  # noqa: E402
import test_gpu_smooth_mg as M  # noqa: E402  (the GPU tests' bodies, reused as plain functions)
from test_emu_smooth import _free_port, _mgtools_worker, emu  # noqa: E402,F401  (fixture: the emulated binding)
from test_emu_tools import emu_exes  # noqa: E402,F401  (fixture: the emulated host executables)


@pytest.mark.parametrize("t", [1e-7, 1e-5])
@pytest.mark.parametrize("name", G.SMOOTH_FIXTURES)
def test_emulated_smooth_mg_fixture(emu, name, t):
    M.check_fixture(emu, name, t)


@pytest.mark.parametrize("ratio", M.STIFF_RATIOS)
@pytest.mark.parametrize("name", M.STIFF_CASES)
def test_emulated_smooth_mg_stiff(emu, name, ratio):
    M.check_stiff(emu, name, ratio)


@pytest.mark.parametrize("name", G.SMOOTH_FIXTURES)
def test_emulated_smooth_mg_iteration_bound(emu, name):
    M.check_iteration_bound(emu, name)


@pytest.mark.parametrize("name,ratio", [(n, r) for n in M.ISOTROPIC for r in (1e0, 1e2, 1e4)] + [(n, 1e0) for n in M.ANISOTROPIC])
def test_emulated_smooth_mg_vcycle(emu, name, ratio):
    M.check_vcycle(emu, name, ratio)


@pytest.mark.parametrize("name,expected", [("c1_periodic", 3), ("np2", 2), ("thin", 4)])
def test_emulated_smooth_mg_levels(emu, name, expected):
    M.check_mg_levels(emu, name, expected)


def test_emulated_smooth_mg_errors(emu):
    M.check_errors(emu)


def test_emulated_smooth_mg_curvature_run(emu):
    M.check_curvature_run(emu)


@pytest.mark.parametrize("name", ["c1_periodic", "c3_three_levels", "c1_corner_sym"])
def test_emulated_curvature_executable_smooth_mg(emu_exes, tmp_path, monkeypatch, name):
    M.check_tool(emu_exes[1], tmp_path, name, monkeypatch)


def test_emulated_curvature_executable_smooth_precond_unknown(emu_exes, tmp_path):
    M.check_tool_bad_precond(emu_exes[1], tmp_path)


def test_emulated_mgtools_smooth_mg(emu_exes, tmp_path):
    """mgtools curvature do_smooth=1 smooth_precond=mg at world 1: the executable's plotfile values, bit for bit"""
    from helpers import load_golden
    from peleanalysis_b200 import plotfile
    pf, z = load_golden("c3_three_levels")
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    args = ["infile=" + d, "progressName=temp", "do_smooth=1", "smoothing_time=1e-5", "smooth_precond=mg"]
    p = G.run_tool(emu_exes[1], d, str(tmp_path), *args[2:], "outfile=" + str(tmp_path / "exe"))
    assert p.returncode == 0, p.stdout + p.stderr
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    pr = ctx.Process(target=_mgtools_worker, args=(0, 1, _free_port(), args + ["outfile=" + str(tmp_path / "mg1")], q))
    pr.start()
    res = dict([q.get(timeout=600)])
    pr.join(timeout=60)
    assert res == {0: "ok"}, res
    a, b = plotfile.read_plotfile(str(tmp_path / "exe")), plotfile.read_plotfile(str(tmp_path / "mg1"))
    assert a.names == b.names
    for n in a.names:
        ka, kb = a.comp(n), b.comp(n)
        for la, lb in zip(a.levels, b.levels):
            for fa, fb in zip(la.fabs, lb.fabs):
                assert np.array_equal(fa[ka].view(np.int64), fb[kb].view(np.int64)), n
