"""GPU: fields filled from and read back into device memory (pa_field_upload_device / pa_field_download_device, capi.Array4,
the runs' upload_device / result_device) -- bit-identical to the host route, ghost cells and foreign bytes untouched, every
error path.  The bodies take the binding P and a device-array backend D, so tests/test_emu_device_io.py runs them on the
emulated library with its own "device" blocks."""
import contextlib

import numpy as np
import pytest

from helpers import bit_equal, load_golden

GOLDEN_STENCIL = ["c1_periodic", "c1_walls", "c1_corner_sym", "lshape", "edge_walls", "edge_periodic", "np2", "thin", "mixed_boxes",
                  "ratio4", "c3_three_levels", "c3_threshold", "c1_options"]
GOLDEN_FILTER = ["filter_c1", "filter_c1_corner_gauss", "filter_c3", "filter_c3_pc_samefgr", "filter_c3_subset", "filter_lshape",
                 "filter_ratio4", "filter_np2", "filter_types"]
SENTINEL = -7.25e300
HOST_ROUTE = ("upload_level", "download_level", "upload_fabs", "download_fabs", "upload_box", "download_box")


class TorchBackend:
    """CUDA tensors of the current device"""

    def __init__(self, P):
        import torch
        self.P, self.torch = P, torch

    def from_np(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()

    def empty(self, shape):
        return self.torch.empty(shape, dtype=self.torch.float64, device="cuda")

    def np(self, x):
        self.P.sync()
        self.torch.cuda.synchronize()
        return x.cpu().numpy()

    def other_device(self, shape):
        if self.torch.cuda.device_count() < 2:
            return None
        return self.torch.zeros(shape, dtype=self.torch.float64, device="cuda:1")


@contextlib.contextmanager
def host_route_forbidden(P):
    """every host upload / download entry point of capi.Field raises while the block runs"""
    saved = {n: getattr(P.Field, n) for n in HOST_ROUTE}

    def boom(*a, **k):
        raise AssertionError("the host route was used")
    try:
        for n in HOST_ROUTE:
            setattr(P.Field, n, boom)
        yield
    finally:
        for n, f in saved.items():
            setattr(P.Field, n, f)


def _dims(box):
    lo, hi = box
    return [hi[d] - lo[d] + 1 for d in range(3)]


def _fab_with_ghosts(data, g, slot, ncomp, rng):
    """[ncomp][nz+2g][ny+2g][nx+2g] of random bytes with data in component `slot`'s valid region"""
    nz, ny, nx = data.shape
    F = rng.standard_normal((ncomp, nz + 2 * g, ny + 2 * g, nx + 2 * g))
    F[slot, g:g + nz, g:g + ny, g:g + nx] = data
    return F


def _view_of(D, data, rng):
    """a non-contiguous view with unit x stride: the box inside a bigger array (offset in every direction)"""
    nz, ny, nx = data.shape
    big = rng.standard_normal((nz + 3, ny + 2, nx + 5))
    big[2:2 + nz, 1:1 + ny, 3:3 + nx] = data
    return D.from_np(big)[2:2 + nz, 1:1 + ny, 3:3 + nx]


def check_upload_download(P, D, pf, is_per=(1, 1, 1), sym_dir=(0, 0, 0), ng=1, grown_boxes=3):
    """fingerprints of the device routes == the host upload's; field ghosts keep a sentinel; download_device == download_level
    bit for bit and leaves the destination's other bytes alone"""
    rng = np.random.default_rng(7)
    H = P.Hierarchy(pf.levels, is_per, sym_dir)
    nc = len(pf.names)
    ref = P.Field(H, nc, ng)
    ref.set_val(SENTINEL)
    for c in range(nc):
        ref.upload_fabs(c, [[f[c] for f in lv.fabs] for lv in pf.levels])
    want = ref.hash()
    routes = {"dense": lambda c, fab: (D.from_np(fab[c]), 0),
              "view": lambda c, fab: (_view_of(D, fab[c], rng), 0)}
    for g in (1, 2):
        routes["fab%d" % g] = (lambda g: lambda c, fab: (D.from_np(_fab_with_ghosts(fab[c], g, (c + 1) % 4, 4, rng))[(c + 1) % 4:], g))(g)
    for route, make in routes.items():
        f = P.Field(H, nc, ng)
        f.set_val(SENTINEL)
        for c in range(nc):
            for l, lv in enumerate(pf.levels):
                arrs = [make(c, lv.fabs[b]) for b in H.local_boxes[l]]
                f.upload_level_device(l, c, [a for a, _ in arrs], nghost=arrs[0][1] if arrs else 0)
        assert f.hash() == want, route
        for l, lv in enumerate(pf.levels):
            for b in H.local_boxes[l][:grown_boxes]:
                for c in range(nc):
                    got, exp = f.download_grown(l, b, c), ref.download_grown(l, b, c)
                    assert bit_equal(got, exp), (route, l, b, c)          # valid cells equal, ghost cells still the sentinel
    # all components in one call from one [nc][nz][ny][nx] array per box
    f = P.Field(H, nc, ng)
    for l, lv in enumerate(pf.levels):
        f.upload_level_device(l, 0, [D.from_np(lv.fabs[b]) for b in H.local_boxes[l]], ncomp=nc)
    assert f.hash() == want
    # download: valid cells == download_level; a FAB destination keeps its ghost cells and its other components
    for l, lv in enumerate(pf.levels):
        loc = H.local_boxes[l]
        if not loc:
            continue
        for c in range(nc):
            host = np.empty(H.local_cells[l])
            ref.download_level(l, c, host)
            P.sync()
            dense = [D.empty(tuple(reversed(_dims(lv.boxes[b])))) for b in loc]
            ref.download_level_device(l, c, dense)
            got = np.concatenate([D.np(a).ravel() for a in dense])
            assert bit_equal(got, host), (l, c)
            pre = [rng.standard_normal((3,) + tuple(n + 4 for n in reversed(_dims(lv.boxes[b])))) for b in loc]
            fabs = [D.from_np(p) for p in pre]
            ref.download_level_device(l, c, [F[1:] for F in fabs], nghost=2)
            o = 0
            for b, p, F in zip(loc, pre, fabs):
                nx, ny, nz = _dims(lv.boxes[b])
                exp = p.copy()
                exp[1, 2:2 + nz, 2:2 + ny, 2:2 + nx] = host[o:o + nx * ny * nz].reshape(nz, ny, nx)
                o += nx * ny * nz
                assert bit_equal(D.np(F), exp), (l, c, b)


def check_errors(P, D):
    """every PA_ERR_ARG of the two calls, and array4_of's ValueErrors"""
    import ctypes as C
    from peleanalysis_b200 import synth
    pf = synth.config1(16, 8)
    H = P.Hierarchy(pf.levels)
    f = P.Field(H, 2, 1)
    lv = pf.levels[0]
    loc = H.local_boxes[0]
    arrs = [D.from_np(lv.fabs[b][0]) for b in loc]

    def descs(mod=None):
        d = (P.Array4 * len(loc))()
        for k, (a, b) in enumerate(zip(arrs, loc)):
            d[k] = P.array4_of(a, lv.boxes[b])
        if mod:
            mod(d[0])
        return d

    def expect(msg, call):
        with pytest.raises(P.PaError) as e:
            P.check(call())
        assert e.value.code == -1 and msg in str(e.value), str(e.value)
        e = None                 # no frame <-> traceback cycle: fields must go before their hierarchy
    L = P.lib()
    n = len(loc)
    for fn in (L.pa_field_upload_device, L.pa_field_download_device):
        expect("null field", lambda: fn(None, 0, 0, 1, descs(), n))
        expect("null array list", lambda: fn(f.f, 0, 0, 1, None, n))
        expect("arrays for the", lambda: fn(f.f, 0, 0, 1, descs(), n - 1))
        expect("arrays for the", lambda: fn(f.f, 0, 0, 1, descs(), n + 1))
        expect("null data pointer", lambda: fn(f.f, 0, 0, 1, descs(lambda a: setattr(a, "p", None)), n))
        expect("do not contain the box", lambda: fn(f.f, 0, 0, 1, descs(lambda a: a.begin.__setitem__(1, a.begin[1] + 1)), n))
        expect("do not contain the box", lambda: fn(f.f, 0, 0, 1, descs(lambda a: a.end.__setitem__(2, a.end[2] - 1)), n))
        expect("exceeds the array's", lambda: fn(f.f, 0, 0, 2, descs(), n))
        expect("out of [0, 2)", lambda: fn(f.f, 0, 2, 1, descs(), n))
        expect("out of [0, 2)", lambda: fn(f.f, 0, -1, 1, descs(), n))
        expect("level out of range", lambda: fn(f.f, H.nlev, 0, 1, descs(), n))
        expect("overlap", lambda: fn(f.f, 0, 0, 1, descs(lambda a: setattr(a, "jstride", 7)), n))
        expect("overlap", lambda: fn(f.f, 0, 0, 1, descs(lambda a: setattr(a, "kstride", 8 * 8 - 1)), n))
        expect("overlap", lambda: fn(f.f, 0, 0, 1, descs(lambda a: (setattr(a, "ncomp", 2), setattr(a, "nstride", 100))), n))
        host = np.zeros(8 * 8 * 8)
        expect("pa_field_upload_level", lambda: fn(f.f, 0, 0, 1, descs(lambda a: setattr(a, "p", host.ctypes.data)), n))
        other = D.other_device((8, 8, 8))
        if other is not None:
            expect("memory of device", lambda: fn(f.f, 0, 0, 1, descs(lambda a: setattr(a, "p", P.array4_of(other, lv.boxes[loc[0]]).p)), n))
    # download destinations that overlap: the same array for two boxes
    same = [arrs[0]] * n
    with pytest.raises(P.PaError) as e:
        f.download_level_device(0, 0, same)
    assert "overlap" in str(e.value)
    e = None
    # nothing was written by any rejected call
    f.set_val(1.5)
    P.sync()
    # array4_of: ValueError before any library call
    t = D.from_np(np.zeros((8, 8, 8)))
    for bad in (np.zeros((8, 8, 8)), D.from_np(np.zeros((8, 8)))):
        with pytest.raises(ValueError):
            P.array4_of(bad, lv.boxes[loc[0]])
    with pytest.raises(ValueError):
        P.array4_of(D.from_np(np.zeros((8, 8, 16)))[:, :, ::2], lv.boxes[loc[0]])
    with pytest.raises(ValueError):
        P.array4_of(D.from_np(np.zeros((2, 2, 8, 8, 8))), lv.boxes[loc[0]])
    with pytest.raises(ValueError):
        f.upload_level_device(0, 0, [t] * (n - 1))
    assert C.sizeof(P.Array4) == 8 + 3 * 8 + 6 * 4 + 4 + 4          # pa_array4: pointer, 3 x int64, 6 ints, ncomp (+ padding)


def check_two_ranks(P, D, pf, is_per=(1, 1, 1)):
    """boxes spread over two ranks of one process: each rank passes its own boxes; the ranks' fingerprints add up to the
    one-rank value; the wrong box count is rejected; a level without local boxes is a no-op"""
    H1 = P.Hierarchy(pf.levels, is_per)
    one = P.Field(H1, 1, 1)
    for l, lv in enumerate(pf.levels):
        one.upload_level_device(l, 0, [D.from_np(lv.fabs[b][0]) for b in H1.local_boxes[l]])
    total = 0
    for r in range(2):
        H = P.Hierarchy(pf.levels, is_per, rank=r, nranks=2)
        f = P.Field(H, 1, 1)
        for l, lv in enumerate(pf.levels):
            loc = H.local_boxes[l]
            if 0 < len(loc) < len(lv.boxes):
                with pytest.raises(P.PaError) as e:
                    P.check(P.lib().pa_field_upload_device(f.f, l, 0, 1, f._arrays(l, [D.from_np(lv.fabs[b][0]) for b in loc], 0)[0], len(lv.boxes)))
                assert "boxes this rank owns" in str(e.value)
                e = None
            f.upload_level_device(l, 0, [D.from_np(lv.fabs[b][0]) for b in loc])
        total = (total + f.hash()) % (1 << 64)
    assert total == one.hash()
    # a level none of whose boxes this rank owns
    boxes = [((0, 0, 0), (7, 7, 7))]
    from peleanalysis_b200.plotfile import Level
    lv = Level((0, 0, 0), (7, 7, 7), (0.125,) * 3, boxes)
    H = P.Hierarchy([lv], rank=1, nranks=2, owners=[np.zeros(1, dtype=np.int32)])
    f = P.Field(H, 1, 1)
    P.check(P.lib().pa_field_upload_device(f.f, 0, 0, 1, None, 0))
    P.check(P.lib().pa_field_download_device(f.f, 0, 0, 1, None, 0))


def _device_result_flat(D, res, hier, lev):
    loc = hier.local_boxes[lev]
    if not loc:
        return None
    return np.concatenate([D.np(res[lev][b]).reshape(res[lev][b].shape[0], -1) for b in loc], axis=1)


def check_runs(P, D, run_cls, pf, kw, alloc=None):
    """a run fed by upload_device and read by result_device == the same run through the host route, with every host
    upload / download entry point raising during the device run"""
    host = run_cls(P, pf, **kw)
    host.step()
    P.sync()
    want = [host.download_level(l) for l in range(len(host.levels))]
    res_host = host.result()
    with host_route_forbidden(P):
        dev = run_cls(P, pf, upload=False, **kw)
        for name in dev.names:
            k = pf.comp(name)
            if hasattr(dev, "fgr"):         # filterPlt: the re-chopped grids
                per_level = [[D.from_np(lv.fabs[b][dev.names.index(name)]) for b in dev.hier.local_boxes[l]] for l, lv in enumerate(dev.levels)]
            else:
                per_level = [[D.from_np(lv.fabs[b][k]) for b in dev.hier.local_boxes[l]] for l, lv in enumerate(pf.levels)]
            dev.upload_device(name, per_level)
        dev.step()
        res = dev.result_device(alloc) if alloc else dev.result_device()
        for l in range(len(dev.levels)):
            got = _device_result_flat(D, res, dev.hier, l)
            if got is not None:
                assert bit_equal(got, want[l]), (run_cls.__name__, l)
            for b, a in enumerate(res[l]):
                assert (a is None) == (res_host[l][b] is None)
    return dev


def curv_kw(P, z):
    kw = dict(x.split("=") for x in z["curv_opts"]) if "curv_opts" in z.files else {}
    o = P.CurvOpts()
    o.prog_min, o.prog_max = float(z["prog_min"]), float(z["prog_max"])
    o.do_threshold, o.threshold = int(kw.get("threshold_prog", 0)), float(kw.get("threshold_value", 0.0))
    o.do_gauss, o.do_strain = int(kw.get("do_gaussCurv", 0)), int(kw.get("do_strain", 0))
    o.get_strain_tensor, o.do_velnormal = int(kw.get("getStrainTensor", 0)), int(kw.get("do_velnormal", 0))
    return o


# ---- the GPU tests -------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def D(gpu):
    return TorchBackend(gpu)


def _three_level_128():
    from peleanalysis_b200 import synth
    return synth.config3(base=128, mgs=128, nlev=3)


@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN_STENCIL)
def test_device_upload_matches_host_upload_golden(gpu, D, name):
    pf, z = load_golden(name)
    check_upload_download(gpu, D, pf, tuple(int(v) for v in z["is_per"]), tuple(int(v) for v in z["sym_dir"]))


@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN_FILTER)
def test_device_upload_matches_host_upload_golden_filter(gpu, D, name):
    pf, _ = load_golden(name)
    check_upload_download(gpu, D, pf, (0, 0, 0), ng=2)


@pytest.mark.gpu
@pytest.mark.parametrize("size", ["mid", "three_level_128"])
def test_device_upload_matches_host_upload_large(gpu, D, size):
    from peleanalysis_b200 import synth
    pf = synth.config3(base=64, mgs=16, names=("temp", "x_velocity")) if size == "mid" else _three_level_128()
    check_upload_download(gpu, D, pf, grown_boxes=1)


@pytest.mark.gpu
def test_device_io_errors(gpu, D):
    check_errors(gpu, D)


@pytest.mark.gpu
def test_device_io_two_ranks(gpu, D):
    from peleanalysis_b200 import synth
    check_two_ranks(gpu, D, synth.config3(16, 8))


@pytest.mark.gpu
def test_device_upload_ordered_behind_producer_on_torch_stream(gpu, D):
    """pa_set_stream(torch stream): the upload reads what a torch kernel queued before it on that stream wrote"""
    import torch
    from peleanalysis_b200 import synth
    pf = synth.config3(base=64, mgs=32)
    H = gpu.Hierarchy(pf.levels)
    ref = gpu.Field(H, 1, 1)
    ref.upload_fabs(0, [[f[0] for f in lv.fabs] for lv in pf.levels])
    s = torch.cuda.Stream()
    src = [[D.from_np(lv.fabs[b][0]) for b in H.local_boxes[l]] for l, lv in enumerate(pf.levels)]
    torch.cuda.synchronize()
    f = gpu.Field(H, 1, 1)
    try:
        gpu.set_stream(s.cuda_stream)
        with torch.cuda.stream(s):
            dst = [[torch.empty_like(a) for a in lv] for lv in src]
            torch.cuda._sleep(20_000_000)                 # the producer is still running when the upload is queued
            for lv_d, lv_s in zip(dst, src):
                for a, b in zip(lv_d, lv_s):
                    a.copy_(b)
            for l, arrs in enumerate(dst):
                f.upload_level_device(l, 0, arrs)
        assert f.hash() == ref.hash()
    finally:
        gpu.sync()
        gpu.set_stream(0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c1_periodic", "c1_corner_sym", "c3_three_levels", "ratio4", "mixed_boxes"])
def test_grad_run_device_route(gpu, D, name):
    from peleanalysis_b200.stencilrun import GradRun
    pf, z = load_golden(name)
    check_runs(gpu, D, GradRun, pf, dict(names=["temp"], is_per=tuple(int(v) for v in z["is_per"]), sym_dir=tuple(int(v) for v in z["sym_dir"])))


@pytest.mark.gpu
@pytest.mark.parametrize("name,smooth", [("c1_periodic", None), ("c3_threshold", None), ("c1_options", None), ("mixed_boxes", None),
                                         ("c3_three_levels", "jacobi"), ("c3_three_levels", "mg")])
def test_curvature_run_device_route(gpu, D, name, smooth):
    from peleanalysis_b200.stencilrun import CurvatureRun
    pf, z = load_golden(name)
    kw = dict(opts=curv_kw(gpu, z), progress="temp", is_per=tuple(int(v) for v in z["is_per"]), sym_dir=tuple(int(v) for v in z["sym_dir"]))
    if smooth:
        kw.update(do_smooth=True, smooth_precond=smooth)
    check_runs(gpu, D, CurvatureRun, pf, kw)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["filter_c1", "filter_c3", "filter_c3_subset", "filter_c1_corner_gauss"])
def test_filter_run_device_route(gpu, D, name):
    from cases import FILTER_CASES
    from peleanalysis_b200.filterplt import FilterRun
    builder, opts = FILTER_CASES[name]
    pf = builder()
    kw = dict(opts)
    if "variables" in kw:
        kw["variables"] = kw["variables"].split()
    check_runs(gpu, D, FilterRun, pf, kw)


@pytest.mark.gpu
def test_grad_then_curvature_on_device(gpu, D):
    """grad's |grad T| tensors feed a curvature run directly, never leaving the device"""
    from peleanalysis_b200 import synth
    from peleanalysis_b200.stencilrun import CurvatureRun, GradRun
    pf = synth.config3(32, 16)
    g = GradRun(gpu, pf, names=["temp"], upload=False)
    g.upload_device("temp", [[D.from_np(lv.fabs[b][0]) for b in g.hier.local_boxes[l]] for l, lv in enumerate(pf.levels)])
    g.step()
    mags = g.result_device()
    o = gpu.CurvOpts()
    o.prog_min, o.prog_max = 0.0, 1.0
    c = CurvatureRun(gpu, pf, o, upload=False)
    c.upload_device("temp", [[mags[l][b][3] for b in c.hier.local_boxes[l]] for l in range(len(pf.levels))])
    c.step()
    got = c.result_device()
    host_mag = g.result()
    for l, lv in enumerate(pf.levels):
        for b in c.hier.local_boxes[l]:
            lv.fabs[b] = np.stack([host_mag[l][b][3]] + [lv.fabs[b][k] for k in range(1, lv.fabs[b].shape[0])])
    ref = CurvatureRun(gpu, pf, o)
    ref.step()
    for l in range(len(pf.levels)):
        assert bit_equal(_device_result_flat(D, got, c.hier, l), ref.download_level(l))
