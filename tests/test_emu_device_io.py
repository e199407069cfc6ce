"""CPU tier: pa_field_upload_device / pa_field_download_device and the runs' upload_device / result_device on the EMULATED
library (tests/emu), in its variant with pointer attributes (tests/emu/build_emu_ptr.py, cuemu_pointer.h): the "device"
arrays are emulated device blocks (cuemu_device_alloc), which its cudaPointerGetAttributes reports as device memory, while
any other address is host memory.  The same bodies as tests/test_gpu_device_io.py, plus the runs at world size 2 over gloo,
and the plain emulated library, which cannot query pointer attributes, refusing the calls."""
import ctypes as C
import importlib.util
import os
import socket
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "emu"))

import test_gpu_device_io as G  # noqa: E402  (the GPU tests' bodies are reused as plain functions)
from helpers import bit_equal, load_golden  # noqa: E402


class _Block:
    def __init__(self, lib, nbytes, device):
        self.lib = lib
        self.ptr = lib.cuemu_device_alloc(max(int(nbytes), 8), device)
        assert self.ptr

    def __del__(self):
        self.lib.cuemu_device_free(self.ptr)


class EmuArray:
    """a float64 array in an emulated device block: numpy view for the test's own reads and writes, __cuda_array_interface__
    for the library; slicing keeps the block alive"""

    def __init__(self, block, arr):
        self.block, self.arr = block, arr

    @property
    def shape(self):
        return self.arr.shape

    @property
    def __cuda_array_interface__(self):
        return {"shape": self.arr.shape, "typestr": "<f8", "strides": self.arr.strides, "data": (self.arr.ctypes.data, False), "version": 3}

    def __getitem__(self, idx):
        return EmuArray(self.block, self.arr[idx])

    def zero_(self):
        self.arr[...] = 0.0
        return self


class EmuBackend:
    def __init__(self, P):
        self.P = P
        L = P.lib()
        L.cuemu_device_alloc.restype, L.cuemu_device_alloc.argtypes = C.c_void_p, [C.c_size_t, C.c_int]
        L.cuemu_device_free.restype, L.cuemu_device_free.argtypes = None, [C.c_void_p]
        self.L = L

    def empty(self, shape, device=-1):
        n = int(np.prod(shape))
        b = _Block(self.L, 8 * n, device)
        arr = np.ctypeslib.as_array((C.c_double * max(n, 1)).from_address(b.ptr))[:n].reshape(shape)
        return EmuArray(b, arr)

    def from_np(self, a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        x = self.empty(a.shape)
        x.arr[...] = a
        return x

    def np(self, x):
        self.P.sync()
        return np.array(x.arr)

    def other_device(self, shape):
        return self.empty(shape, device=1)

    def alloc(self, shape):
        return self.empty(shape)


def _load():
    """private binding and multigpu modules on the emulated library WITH pointer attributes (build_emu_ptr.py)"""
    import build_emu_ptr
    from peleanalysis_b200 import capi as product_capi, multigpu as product_multigpu

    def private(mod, name):
        spec = importlib.util.spec_from_file_location("peleanalysis_b200." + name, mod.__file__)
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        return m
    capi = private(product_capi, "_capi_emulated_dio")
    capi.LIB_PATH = build_emu_ptr.build()
    mg = private(product_multigpu, "_multigpu_emulated_dio")
    mg.capi = capi
    return capi, mg


@pytest.fixture(scope="module")
def emu():
    old = os.environ.get("PA_NORMAL_MATH")
    os.environ["PA_NORMAL_MATH"] = "fast"      # the emulator has no MUFU (tests/test_emu_parity.py)
    m, _ = _load()
    m.init(0)
    yield m
    if old is None:
        os.environ.pop("PA_NORMAL_MATH", None)
    else:
        os.environ["PA_NORMAL_MATH"] = old


@pytest.fixture(scope="module")
def D(emu):
    return EmuBackend(emu)


@pytest.mark.parametrize("name", G.GOLDEN_STENCIL)
def test_emulated_device_upload_matches_host_upload_golden(emu, D, name):
    pf, z = load_golden(name)
    G.check_upload_download(emu, D, pf, tuple(int(v) for v in z["is_per"]), tuple(int(v) for v in z["sym_dir"]))


@pytest.mark.parametrize("name", G.GOLDEN_FILTER)
def test_emulated_device_upload_matches_host_upload_golden_filter(emu, D, name):
    pf, _ = load_golden(name)
    G.check_upload_download(emu, D, pf, (0, 0, 0), ng=2)


def test_emulated_device_upload_mid_size(emu, D):
    from peleanalysis_b200 import synth
    G.check_upload_download(emu, D, synth.config3(base=32, mgs=16, names=("temp", "x_velocity")), grown_boxes=1)


def test_emulated_device_io_errors(emu, D):
    G.check_errors(emu, D)


def test_emulated_pointer_attributes(emu, D):
    """the emulator's cudaPointerGetAttributes: its device blocks (and addresses inside them) are device memory of the device
    they were made on; the library's own pinned host buffers and any other address are host memory"""
    from peleanalysis_b200 import synth
    pf = synth.config1(16, 8)
    H = emu.Hierarchy(pf.levels)
    f = emu.Field(H, 1, 1)
    loc = H.local_boxes[0]
    pinned = emu.PinnedArray(8 * 8 * 8 * 4)
    d = (emu.Array4 * len(loc))()
    for k, b in enumerate(loc):
        d[k] = emu.array4_of(D.from_np(pf.levels[0].fabs[b][0]), pf.levels[0].boxes[b])
    d[len(loc) - 1].p = pinned.ptr.value
    with pytest.raises(emu.PaError) as e:
        emu.check(emu.lib().pa_field_upload_device(f.f, 0, 0, 1, d, len(loc)))
    assert "host memory" in str(e.value)
    pinned.free()


def test_plain_emulated_build_refuses_device_arrays(emu):
    """the emulated library of build_emu.py has no pointer attributes: the device calls fail loudly instead of guessing"""
    import build_emu
    from peleanalysis_b200 import capi as product_capi, synth
    spec = importlib.util.spec_from_file_location("capi_emulated_plain_dio", product_capi.__file__)
    P = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(P)
    P.LIB_PATH = build_emu.build()
    P.init(0)
    pf = synth.config1(16, 8)
    H = P.Hierarchy(pf.levels)
    f = P.Field(H, 1, 1)
    loc = H.local_boxes[0]
    keep = [np.ascontiguousarray(pf.levels[0].fabs[b][0]) for b in loc]
    d = (P.Array4 * len(loc))()
    for k, (a, b) in enumerate(zip(keep, loc)):
        lo, hi = pf.levels[0].boxes[b]
        d[k].p = a.ctypes.data
        d[k].jstride, d[k].kstride, d[k].nstride = a.shape[2], a.shape[2] * a.shape[1], a.size
        d[k].begin[:], d[k].end[:], d[k].ncomp = list(lo), [hi[i] + 1 for i in range(3)], 1
    for fn in (P.lib().pa_field_upload_device, P.lib().pa_field_download_device):
        code = fn(f.f, 0, 0, 1, d, len(loc))
        assert code == P.PA_ERR_UNSUPPORTED and "cannot query pointer attributes" in P.lib().pa_last_error().decode()
    del f, H


def test_emulated_device_io_two_ranks(emu, D):
    from peleanalysis_b200 import synth
    G.check_two_ranks(emu, D, synth.config3(16, 8))


@pytest.mark.parametrize("name", ["c1_periodic", "c1_corner_sym", "c3_three_levels", "ratio4", "mixed_boxes"])
def test_emulated_grad_run_device_route(emu, D, name):
    from peleanalysis_b200.stencilrun import GradRun
    pf, z = load_golden(name)
    G.check_runs(emu, D, GradRun, pf, dict(names=["temp"], is_per=tuple(int(v) for v in z["is_per"]), sym_dir=tuple(int(v) for v in z["sym_dir"])),
                 alloc=D.alloc)


@pytest.mark.parametrize("name,smooth", [("c1_periodic", None), ("c3_threshold", None), ("c1_options", None), ("c3_three_levels", "mg")])
def test_emulated_curvature_run_device_route(emu, D, name, smooth):
    from peleanalysis_b200.stencilrun import CurvatureRun
    pf, z = load_golden(name)
    kw = dict(opts=G.curv_kw(emu, z), progress="temp", is_per=tuple(int(v) for v in z["is_per"]), sym_dir=tuple(int(v) for v in z["sym_dir"]))
    if smooth:
        kw.update(do_smooth=True, smooth_precond=smooth)
    G.check_runs(emu, D, CurvatureRun, pf, kw, alloc=D.alloc)


@pytest.mark.parametrize("name", ["filter_c1", "filter_c3_subset"])
def test_emulated_filter_run_device_route(emu, D, name):
    from cases import FILTER_CASES
    from peleanalysis_b200.filterplt import FilterRun
    builder, opts = FILTER_CASES[name]
    kw = dict(opts)
    if "variables" in kw:
        kw["variables"] = kw["variables"].split()
    G.check_runs(emu, D, FilterRun, builder(), kw, alloc=D.alloc)


# ---- world size 2 over gloo: each rank uploads its own boxes from device arrays; the exchanges are the host route's ----------
def _worker(rank, world, port, ok):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.join(HERE, "emu"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), CUEMU_SEED=str(1 + rank), PA_NORMAL_MATH="fast")
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from test_emu_multirank import _wrap_host
        from peleanalysis_b200.filterplt import FilterRun
        from peleanalysis_b200.stencilrun import CurvatureRun, GradRun
        P, mg = _load()
        P.init(0)
        Dv = EmuBackend(P)
        common = dict(rank=rank, nranks=world, multigpu=mg, wrap=_wrap_host)
        pf, z = load_golden("c3_three_levels")
        G.check_runs(P, Dv, GradRun, pf, dict(names=["temp"], **common), alloc=Dv.alloc)
        o = G.curv_kw(P, z)
        G.check_runs(P, Dv, CurvatureRun, pf, dict(opts=o, progress="temp", **common), alloc=Dv.alloc)
        from cases import FILTER_CASES
        builder, opts = FILTER_CASES["filter_c3"]
        G.check_runs(P, Dv, FilterRun, builder(), dict(opts, **common), alloc=Dv.alloc)
        ok[rank] = 1
    finally:
        dist.destroy_process_group()


def test_emulated_runs_device_route_world2():
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    ok = ctx.Array("i", [0, 0])
    procs = [ctx.Process(target=_worker, args=(r, 2, port, ok)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(900)
    assert list(ok) == [1, 1], [p.exitcode for p in procs]
