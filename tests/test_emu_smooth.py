"""CPU tier: pa_smooth (curvature's do_smooth, R/Src/curvature.cpp:328-406) with the kernel SOURCES run under the CUDA
execution-model emulator of tests/emu -- the same checks as tests/test_gpu_smooth.py: the golden fixtures against the SciPy
oracle, the error codes, the emulated curvature3d do_smooth=1 and `mgtools curvature do_smooth=1` at world 1 and 2."""
import importlib.util
import multiprocessing as mp
import os
import socket
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emu"))

import test_gpu_smooth as G  # noqa: E402  (the GPU tests' bodies, reused as plain functions)
from test_emu_tools import emu_exes  # noqa: E402,F401  (fixture: the emulated host executables)


@pytest.fixture(scope="module")
def emu():
    import build_emu
    from peleanalysis_b200 import capi as product_capi
    lib = build_emu.build()
    spec = importlib.util.spec_from_file_location("capi_emulated_smooth", product_capi.__file__)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    m.LIB_PATH = lib                     # a private module instance: the product binding itself is untouched
    old = os.environ.get("PA_NORMAL_MATH")
    os.environ["PA_NORMAL_MATH"] = "fast"
    m.init(0)
    yield m
    if old is None:
        os.environ.pop("PA_NORMAL_MATH", None)
    else:
        os.environ["PA_NORMAL_MATH"] = old


@pytest.mark.parametrize("t", [1e-7, 1e-5])
@pytest.mark.parametrize("name", G.SMOOTH_FIXTURES)
def test_emulated_smooth_fixture(emu, name, t):
    G.check_fixture(emu, name, t)


def test_emulated_smooth_zero_time(emu):
    G.check_zero_time(emu)


def test_emulated_smooth_errors(emu):
    G.check_errors(emu)


def test_emulated_smooth_two_ranks(emu):
    G.check_two_ranks(emu)


@pytest.mark.parametrize("name", ["c1_periodic", "c3_three_levels", "c1_corner_sym"])
def test_emulated_curvature_executable_do_smooth(emu_exes, tmp_path, name):
    G.check_tool(emu_exes[1], tmp_path, name)


def test_emulated_curvature_executable_do_smooth_refuses_several_gpus(emu_exes, tmp_path):
    G.check_tool_multi_gpu_abort(emu_exes[1], tmp_path, env={"CUEMU_DEVICES": "2"})


def _mgtools_worker(rank, world, port, args, q):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), PA_NORMAL_MATH="fast")
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.join(HERE, "emu"))
    import build_emu
    from peleanalysis_b200 import capi as product_capi, mgtools
    spec = importlib.util.spec_from_file_location("capi_emulated_smooth", product_capi.__file__)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    m.LIB_PATH = build_emu.LIB
    try:
        mgtools.run("curvature", args, capi=m, backend="gloo", device=0)
        q.put((rank, "ok"))
    except SystemExit as e:
        q.put((rank, str(e)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_emulated_mgtools_do_smooth(emu_exes, tmp_path):
    """mgtools curvature do_smooth=1: at world 1 the same plotfile values as the executable; at world 2 an abort that names
    the one-GPU limitation on every rank"""
    from helpers import load_golden
    from peleanalysis_b200 import plotfile
    pf, z = load_golden("c3_three_levels")
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    p = G.run_tool(emu_exes[1], d, str(tmp_path), "outfile=" + str(tmp_path / "exe"), "do_smooth=1", "smoothing_time=1e-5")
    assert p.returncode == 0, p.stdout + p.stderr
    args = ["infile=" + d, "progressName=temp", "do_smooth=1", "smoothing_time=1e-5"]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    for world, out in ((1, "mg1"), (2, "mg2")):
        port = _free_port()
        procs = [ctx.Process(target=_mgtools_worker, args=(r, world, port, args + ["outfile=" + str(tmp_path / out)], q)) for r in range(world)]
        for pr in procs:
            pr.start()
        res = dict(q.get(timeout=600) for _ in procs)
        for pr in procs:
            pr.join(timeout=60)
        if world == 1:
            assert res == {0: "ok"}, res
        else:
            assert len(res) == 2 and all("runs on one GPU only" in v for v in res.values()), res
    a, b = plotfile.read_plotfile(str(tmp_path / "exe")), plotfile.read_plotfile(str(tmp_path / "mg1"))
    assert a.names == b.names
    for n in a.names:
        ka, kb = a.comp(n), b.comp(n)
        for la, lb in zip(a.levels, b.levels):
            for fa, fb in zip(la.fabs, lb.fabs):
                assert np.array_equal(fa[ka].view(np.int64), fb[kb].view(np.int64)), n
