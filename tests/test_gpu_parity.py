"""GPU (-m gpu): the CUDA path, called through the C ABI, against the oracle on the same inputs and against the
golden vectors of the compiled reference.  Bit-exact for everything except GaussianCurvature (pow(x,4): CUDA
libdevice vs glibc), which is held to the 1e-12 relative tolerance BASELINE.json states."""
import os

import numpy as np
import pytest

from cases import CASES
from helpers import bit_equal, fabs_from_flat, flat_from_fabs, load_golden, max_rel
from oracle import oracle as O
from peleanalysis_b200 import synth

pytestmark = pytest.mark.gpu

GAUSS_TOL = 1e-12


def _flat(pf, name):
    c = pf.comp(name)
    return np.concatenate([f[c].ravel() for l in pf.levels for f in l.fabs])


def _set_stencil(stencil):
    """tma: TMA pipeline, CTA shape by tile size (small boxes -> 2 / 4 consumer warps); tma_big: TMA pipeline in the 8 /
    16-warp shapes whatever the tile size; tma_fused: curvature through the fused kernel + shell pass where the hierarchy is
    eligible (PA_CURV_FUSED=1, opt-in; tma_fused3: the later fused kernel); simple: the plain-load kernels; unfused: curvature's
    progress pass as a kernel of its own, then the flame normal from the materialised Progress (PA_CURV_UNFUSED=1)."""
    os.environ["PA_STENCIL"] = "simple" if stencil == "simple" else "tma"
    os.environ["PA_CURV_UNFUSED"] = "1" if stencil == "unfused" else "0"
    os.environ["PA_TMA_SMALL"] = "0" if stencil.startswith("tma_big") else "1"
    os.environ["PA_CURV_FUSED"] = {"tma_fused": "1", "tma_fused3": "3"}.get(stencil, "0")
    os.environ["PA_NORMAL_F3"] = "1" if stencil == "tma_n3" else "0"      # flame normal through curv_f3.cu's kernel without its K part
    os.environ["PA_NORMAL_W"] = "1" if stencil == "tma_nw" else "0"       # ... through the barrier-free kernel of normal_w.cu


def _gpu_grad(capi, pf, is_per, sym, names=("temp",), stencil="tma", flags=0):
    _set_stencil(stencil)
    H = capi.Hierarchy(pf.levels, is_per, sym, flags=flags)
    fin = capi.Field(H, len(names), 1)
    fout = capi.Field(H, 4 * len(names), 0)
    for v, n in enumerate(names):
        fin.upload_fabs(v, [[f[pf.comp(n)] for f in l.fabs] for l in pf.levels])
    capi.grad(fin, 0, len(names), fout, 0)
    capi.sync()
    out = np.stack([flat_from_fabs(fout.download_fabs(c)) for c in range(4 * len(names))])
    return out, H, fin


def _gpu_curv(capi, pf, is_per, sym, pmin, pmax, kw, stencil="tma", flags=0):
    _set_stencil(stencil)
    H = capi.Hierarchy(pf.levels, is_per, sym, flags=flags)
    o = capi.CurvOpts()
    o.prog_min, o.prog_max = pmin, pmax
    o.do_threshold = int(kw.get("threshold_prog", 0))
    o.threshold = float(kw.get("threshold_value", 1e-4))
    o.do_gauss = int(kw.get("do_gaussCurv", 0))
    o.do_strain = int(kw.get("do_strain", 0))
    o.get_strain_tensor = int(kw.get("getStrainTensor", 0))
    o.do_velnormal = int(kw.get("do_velnormal", 0))
    need_vel = o.do_strain or o.do_velnormal
    state = capi.Field(H, 4 if need_vel else 1, 1)
    state.upload_fabs(0, [[f[pf.comp("temp")] for f in l.fabs] for l in pf.levels])
    if need_vel:
        for d, n in enumerate(["x_velocity", "y_velocity", "z_velocity"]):
            state.upload_fabs(1 + d, [[f[pf.comp(n)] for f in l.fabs] for l in pf.levels])
    nout = capi.curvature_num_outputs(o)
    out = capi.Field(H, nout, 1)
    capi.curvature(state, 0, 1, o, out, 0)
    capi.sync()
    return np.stack([flat_from_fabs(out.download_fabs(c)) for c in range(nout)]), o


# "links": same-level neighbours are read in place by the stencil (default); "nolinks": every ghost cell is
# materialised by the halo gather first (PA_HIER_NO_LINKS, the reference's data flow).  Both must be bit-exact.
LINK_MODES = {"links": 0, "nolinks": 2}


@pytest.mark.parametrize("links", list(LINK_MODES))
@pytest.mark.parametrize("stencil", ["tma", "tma_big", "simple"])
@pytest.mark.parametrize("name", [n for n, c in CASES.items() if "grad" in c[3]])
def test_grad_matches_reference_golden(gpu, name, stencil, links):
    pf, z = load_golden(name)
    out, _, _ = _gpu_grad(gpu, pf, tuple(z["is_per"]), tuple(z["sym_dir"]), stencil=stencil, flags=LINK_MODES[links])
    for c, k in enumerate(["gx", "gy", "gz", "mag"]):
        assert bit_equal(out[c], z["grad_" + k]), (name, stencil, k, max_rel(out[c], z["grad_" + k]))


@pytest.mark.parametrize("links", list(LINK_MODES))
@pytest.mark.parametrize("stencil", ["tma", "tma_fused", "tma_fused3", "tma_n3", "tma_nw", "tma_big", "simple"])
@pytest.mark.parametrize("name", [n for n, c in CASES.items() if "curvature" in c[3]])
def test_curvature_matches_reference_golden(gpu, name, stencil, links):
    pf, z = load_golden(name)
    kw = dict(s.split("=") for s in z["curv_opts"]) if len(z["curv_opts"]) else {}
    out, o = _gpu_curv(gpu, pf, tuple(z["is_per"]), tuple(z["sym_dir"]), float(z["prog_min"]), float(z["prog_max"]), kw, stencil,
                       flags=LINK_MODES[links])
    names = ["Progress", "MeanCurvature_temp", "FlameNormalX_temp", "FlameNormalY_temp", "FlameNormalZ_temp"]
    c = 5
    if o.do_gauss:
        assert max_rel(out[c], z["curv_GaussianCurvature_temp"]) <= GAUSS_TOL
        c += 1
    if o.do_strain:
        assert bit_equal(out[c], z["curv_StrainRate_temp"])
        c += 1
        if o.get_strain_tensor:
            for m in range(3):
                for n in range(3):
                    assert bit_equal(out[c], z["curv_ROST_dU%sd%s" % ("xyz"[m], "xyz"[n])]), (m, n)
                    c += 1
    if o.do_velnormal:
        assert bit_equal(out[c], z["curv_VelFlameNormal"])
    for i, n in enumerate(names):
        assert bit_equal(out[i], z["curv_" + n]), (name, stencil, n, max_rel(out[i], z["curv_" + n]))


@pytest.mark.parametrize("name", list(CASES))
def test_ghost_cells_match_oracle(gpu, name):
    """FillBoundary (all layers, corners included) and the c-f / physical face fill, ghost cell by ghost cell."""
    builder, is_per, sym, _, _ = CASES[name]
    pf = builder()
    OH = O.OracleHier(pf, is_per, sym)
    s = _flat(pf, "temp")
    H = gpu.Hierarchy(pf.levels, is_per, sym)
    # (a) plain FillBoundary with 2 ghost layers: copies only; untouched ghosts keep the fill value
    f2 = gpu.Field(H, 1, 2)
    f2.set_val(-7.25)
    f2.upload_fabs(0, [[f[pf.comp("temp")] for f in l.fabs] for l in pf.levels])
    f2.fill_boundary(0, 1, cross=False)
    gpu.sync()
    for l, lv in enumerate(pf.levels):
        src = OH.fb_source_map(l, 2)
        flat_l = [f[pf.comp("temp")].ravel() for f in lv.fabs]
        for b in range(len(lv.boxes)):
            got = f2.download_grown(l, b, 0)
            want = np.full(got.shape, -7.25)
            m = src[b] >= 0
            sb, lin = src[b][m] >> 40, src[b][m] & ((1 << 40) - 1)
            want[m] = np.array([flat_l[int(a)][int(q)] for a, q in zip(sb, lin)])
            want[2:-2, 2:-2, 2:-2] = lv.fabs[b][pf.comp("temp")]
            assert bit_equal(got, want), (name, l, b)
    # (b) the operator's ghost fill (applyBC semantics), face ghost layer
    f1 = gpu.Field(H, 1, 1)
    f1.upload_fabs(0, [[f[pf.comp("temp")] for f in l.fabs] for l in pf.levels])
    f1.fill_ghosts(0, 1)
    gpu.sync()
    for l, lv in enumerate(pf.levels):
        want = OH.filled_fabs(l, s, 1, 0.0)
        for b in range(len(lv.boxes)):
            got = f1.download_grown(l, b, 0)
            w = want[b]
            for sl in [(0, slice(1, -1), slice(1, -1)), (-1, slice(1, -1), slice(1, -1)),
                       (slice(1, -1), 0, slice(1, -1)), (slice(1, -1), -1, slice(1, -1)),
                       (slice(1, -1), slice(1, -1), 0), (slice(1, -1), slice(1, -1), -1)]:
                assert bit_equal(got[sl], w[sl]), (name, l, b, sl)


@pytest.mark.parametrize("case,kw", [
    ("config1", dict(base=64, mgs=32)),
    ("config3", dict(base=64, mgs=16)),
    ("config5", dict(base=32, mgs=8, ncomp=3, ratios=(2, 4, 2))),
    ("lshape", dict(base=32, mgs=16)),
])
@pytest.mark.parametrize("stencil", ["tma", "tma_big"])
def test_midsize_grad_and_curvature_vs_oracle(gpu, case, kw, stencil):
    """Mid-size hierarchies (hundreds of boxes) against the oracle run on the GPU box's host."""
    pf = synth.CASES[case](**kw)
    var = pf.names[0]
    OH = O.OracleHier(pf, (1, 1, 1), (0, 0, 0))
    s = _flat(pf, var)
    want = OH.grad(s)
    _set_stencil(stencil)
    H = gpu.Hierarchy(pf.levels)
    fin, fout = gpu.Field(H, 1, 1), gpu.Field(H, 4, 0)
    fin.upload_fabs(0, [[f[0] for f in l.fabs] for l in pf.levels])
    gpu.grad(fin, 0, 1, fout, 0)
    gpu.sync()
    for c in range(4):
        assert bit_equal(flat_from_fabs(fout.download_fabs(c)), want[c]), (case, c)
    if all(r == 2 for r in OH.ratios):       # the reference's curvature hard-codes ratio 2 (curvature.cpp:445,518)
        pmin, pmax = float(s.min()), float(s.max())
        wk = OH.curvature(s, pmin, pmax)
        o = gpu.CurvOpts()
        o.prog_min, o.prog_max = pmin, pmax
        out = gpu.Field(H, 5, 1)
        gpu.curvature(fin, 0, 0, o, out, 0)
        gpu.sync()
        for c in range(5):
            assert bit_equal(flat_from_fabs(out.download_fabs(c)), wk[c]), (case, "curv", c)


@pytest.mark.parametrize("stencil", ["tma", "tma_big", "simple"])
def test_curvature_degenerate_values(gpu, stencil):
    """Exactly flat regions (0/-1e-14 = -0), gradients around the 1e-250 guard of the shared-reciprocal division, huge and
    sign-alternating values: the flame normal's three IEEE divisions must come out bit-identical to the oracle's a/n."""
    pf = synth.config1(16, 8)
    rng = np.random.default_rng(7)
    for lv in pf.levels:
        for b, ((lo, hi), fab) in enumerate(zip(lv.boxes, lv.fabs)):
            kind = (b + lo[0] // 8) % 4
            shape = fab[0].shape
            if kind == 0:
                fab[0][...] = 0.25                                                     # flat: G = 0 exactly
            elif kind == 1:
                fab[0][...] = rng.uniform(-1, 1, shape) * 10.0 ** rng.integers(-262, -240, shape)   # around the guard
            elif kind == 2:
                fab[0][...] = rng.uniform(-1, 1, shape) * 1e150                        # huge
            else:
                fab[0][...] = np.where(rng.random(shape) < 0.5, 0.0, rng.uniform(-1, 1, shape) * 1e-300)
    s = _flat(pf, "temp")
    OH = O.OracleHier(pf, (1, 1, 1), (0, 0, 0))
    want = OH.curvature(s, 0.0, 1.0)                                                   # progMin 0, progMax 1: c == S
    out, _ = _gpu_curv(gpu, pf, (1, 1, 1), (0, 0, 0), 0.0, 1.0, {}, stencil)
    for c in range(5):
        assert bit_equal(out[c], want[c]), (stencil, c, max_rel(out[c], want[c]))
    # signed zeros too: bit_equal uses ==, which does not tell -0 from +0
    for c in range(5):
        ok = np.isnan(want[c]) | (np.signbit(out[c]) == np.signbit(want[c]))
        bad = np.flatnonzero(~ok)
        assert bad.size == 0, (stencil, c, bad.size, bad[:8], out[c][bad[:8]], want[c][bad[:8]], s[bad[:8]])


def test_multi_variable_grad_equals_single(gpu):
    """The multi-variable extension (config 2's 5 components in one call) gives each variable the single-variable result."""
    pf = synth.config1(32, 16, names=synth.FIELD_NAMES)
    out5, _, _ = _gpu_grad(gpu, pf, (1, 1, 1), (0, 0, 0), names=synth.FIELD_NAMES)
    for v, n in enumerate(synth.FIELD_NAMES):
        one, _, _ = _gpu_grad(gpu, pf, (1, 1, 1), (0, 0, 0), names=(n,))
        assert bit_equal(out5[4 * v:4 * v + 4], one)


def test_full_size_properties_config2(gpu):
    """BASELINE config 2 at full size (512^3, one component resident at a time): the TMA pipeline and the simple
    kernel are two independent implementations and must agree bit for bit; a periodic shift of the input by one
    box shifts the output identically (box indexing / halo wrap); spot boxes equal the oracle on the 128^3
    sub-problem they came from."""
    n, mgs = 512, 128
    pf = synth.config2(n, mgs, names=("temp",))
    H = gpu.Hierarchy(pf.levels)
    fin, fout = gpu.Field(H, 1, 1), gpu.Field(H, 4, 0)
    fabs = [[f[0] for f in pf.levels[0].fabs]]
    fin.upload_fabs(0, fabs)
    res = {}
    for st in ("tma", "simple"):
        os.environ["PA_STENCIL"] = st
        fout.set_val(0.0)
        gpu.grad(fin, 0, 1, fout, 0)
        gpu.sync()
        res[st] = [fout.download_fabs(c)[0] for c in range(4)]
    for c in range(4):
        for a, b in zip(res["tma"][c], res["simple"][c]):
            assert bit_equal(a, b)
    # periodic shift by one box along x: box b's data moves to the box at lo.x + 128 (mod 512)
    boxes = pf.levels[0].boxes
    index = {lo: i for i, (lo, hi) in enumerate(boxes)}
    perm = [index[((lo[0] + mgs) % n, lo[1], lo[2])] for lo, hi in boxes]      # destination of box i
    shifted = [None] * len(boxes)
    for i, dst in enumerate(perm):
        shifted[dst] = fabs[0][i]
    fin.upload_fabs(0, [shifted])
    os.environ["PA_STENCIL"] = "tma"
    gpu.grad(fin, 0, 1, fout, 0)
    gpu.sync()
    for c in range(4):
        got = fout.download_fabs(c)[0]
        for i, dst in enumerate(perm):
            assert bit_equal(got[dst], res["tma"][c][i]), (c, i)
    # checksum of checksums, recorded for the log
    print("config2 temp grad checksum", float(sum(np.sum(a, dtype=np.float64) for a in res["tma"][3])))


def test_fast_math_selftest(gpu):
    """The stencil kernel's branch-free sqrt / reciprocal / flame-normal forms against the plain IEEE operators, on the
    device, over every exponent of their ranges (zeros, denormals, the 1e-14 clamp, overflow).  The library runs the same
    self-test before its first flame-normal launch and uses the branch-free forms only if not one bit differs, so the
    check here is that its decision matches what the self-test says on this device (and, when PA_NORMAL_MATH does not
    force a form, that the branch-free forms are in fact clean)."""
    from peleanalysis_b200 import capi
    bad = 0
    for seed in (1, 0x5EED5EED, 2 ** 63 + 12345):
        b = capi.lib().pa_debug_selftest_math(1 << 26, seed)
        assert b >= 0, capi.lib().pa_last_error()
        bad += b
    pf = synth.config1(16, 8)
    s = _flat(pf, "temp")
    _gpu_curv(gpu, pf, (1, 1, 1), (0, 0, 0), float(s.min()), float(s.max()), {})     # makes the library decide
    mode = capi.lib().pa_debug_normal_math()
    forced = os.environ.get("PA_NORMAL_MATH")
    if forced not in ("fast", "plain"):
        assert mode == (1 if bad else 0), (mode, bad)
    if forced != "plain":
        assert bad == 0, "branch-free forms differ from the IEEE operators in %d results (library fell back: %s)" % (bad, mode == 1)


@pytest.mark.parametrize("name", ["c1_periodic", "c3_three_levels"])
def test_curvature_two_phases_equal_one_call(gpu, name):
    """pa_curvature_phases(1) then (2) == pa_curvature (the split a multi-rank caller puts its exchange into)."""
    builder, is_per, sym, _, _ = CASES[name]
    pf = builder()
    s = _flat(pf, "temp")
    one, o = _gpu_curv(gpu, pf, is_per, sym, float(s.min()), float(s.max()), {})
    H = gpu.Hierarchy(pf.levels, is_per, sym)
    state = gpu.Field(H, 1, 1)
    state.upload_fabs(0, [[f[pf.comp("temp")] for f in l.fabs] for l in pf.levels])
    out = gpu.Field(H, 5, 1)
    gpu.curvature_phases(state, 0, 0, o, out, 0, 1)
    gpu.curvature_phases(state, 0, 0, o, out, 0, 2)
    gpu.sync()
    two = np.stack([flat_from_fabs(out.download_fabs(c)) for c in range(5)])
    assert bit_equal(one, two)


def test_flat_field_takes_the_clamp(gpu):
    """A field with exactly flat regions: G.G = 0 there, nrm = -1e-14 by the clamp, n = -0 (curvature.cpp:467-502) -- the
    branch-free normal decides this without a square root; compare with the oracle bit for bit (signed zeros included)."""
    pf = synth.make_hierarchy(32, [], [], 16, ("temp",))
    for lv in pf.levels:
        for f in lv.fabs:
            f[0] = np.where(f[0] > 900.0, 900.0, f[0])           # plateau: exact zeros in the gradient
    s = _flat(pf, "temp")
    out, o = _gpu_curv(gpu, pf, (1, 1, 1), (0, 0, 0), float(s.min()), float(s.max()), {})
    OH = O.OracleHier(pf, (1, 1, 1), (0, 0, 0))
    want = OH.curvature(s, float(s.min()), float(s.max()))
    assert (want[2:5] == 0).sum() > 1000
    for c in range(5):
        assert bit_equal(out[c], want[c]), c


@pytest.mark.parametrize("name", ["c3_three_levels", "mixed_boxes", "lshape"])
def test_side_stream_overlap_is_bit_exact(gpu, name):
    """PA_STREAM_OVERLAP=1 (opt-in): ghost fill of the refined levels on a side stream while level 0's stencil runs."""
    os.environ["PA_STREAM_OVERLAP"] = "1"
    try:
        test_grad_matches_reference_golden(gpu, name, "tma", "links")
        test_curvature_matches_reference_golden(gpu, name, "tma", "links")
    finally:
        os.environ.pop("PA_STREAM_OVERLAP", None)


def check_wide_ghost_inputs(capi, builder):
    """Input fields with nghost 2 or 3 (the reference allocates nGrow = 2 for curvature): general-layout route (simple
    kernel, unfused progress pass); same bits as the oracle."""
    pf = builder()
    OH = O.OracleHier(pf)
    s = OH.flatten(0)
    want = OH.grad(s)
    pmin, pmax = float(s.min()), float(s.max())
    wk = OH.curvature(s, pmin, pmax)
    _set_stencil("tma")
    for ng in (2, 3):
        H = capi.Hierarchy(pf.levels)
        fin, fout = capi.Field(H, 1, ng), capi.Field(H, 4, 0)
        fin.upload_fabs(0, [[f[0] for f in l.fabs] for l in pf.levels])
        capi.grad(fin, 0, 1, fout, 0)
        capi.sync()
        for c in range(4):
            assert bit_equal(flat_from_fabs(fout.download_fabs(c)), want[c]), (ng, c)
        o = capi.CurvOpts()
        o.prog_min, o.prog_max = pmin, pmax
        out = capi.Field(H, 5, 1)
        capi.curvature(fin, 0, 0, o, out, 0)
        capi.sync()
        for c in range(5):
            assert bit_equal(flat_from_fabs(out.download_fabs(c)), wk[c]), (ng, "curvature", c)


def test_wide_ghost_inputs(gpu):
    check_wide_ghost_inputs(gpu, lambda: synth.config3(16, 8))


@pytest.mark.parametrize("name", list(CASES))
def test_unstaged_bcfill_variant(gpu, name):
    """PA_BCFILL_V2=0: the coarse-fine fill in which every ghost cell gathers its coarse cells itself (the default stages them
    in shared memory) -- the second route to the same bits."""
    os.environ["PA_BCFILL_V2"] = "0"
    try:
        test_ghost_cells_match_oracle(gpu, name)
        if "grad" in CASES[name][3]:
            test_grad_matches_reference_golden(gpu, name, "tma", "links")
        if "curvature" in CASES[name][3]:
            test_curvature_matches_reference_golden(gpu, name, "tma", "links")
    finally:
        os.environ.pop("PA_BCFILL_V2", None)


@pytest.mark.parametrize("base,mgs", [((256, 8, 4), 256), ((1024, 4, 4), 1024), ((7, 5, 3), 8), ((2, 2, 2), 2), ((128, 32, 8), 128)])
def test_extreme_box_shapes(gpu, base, mgs):
    pf = synth.make_hierarchy(base, [], [], mgs, ("temp",))
    OH = O.OracleHier(pf)
    s = OH.flatten(0)
    out, _, _ = _gpu_grad(gpu, pf, (1, 1, 1), (0, 0, 0))
    want = OH.grad(s)
    for c in range(4):
        assert bit_equal(out[c], want[c]), c
    outc, _ = _gpu_curv(gpu, pf, (1, 1, 1), (0, 0, 0), float(s.min()), float(s.max()), {})
    wk = OH.curvature(s, float(s.min()), float(s.max()))
    for c in range(5):
        assert bit_equal(outc[c], wk[c]), ("curvature", c)


def _hmix64(z):
    z = (z + np.uint64(0x9E3779B97F4A7C15)).astype(np.uint64)
    z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)).astype(np.uint64)
    z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)).astype(np.uint64)
    return z ^ (z >> np.uint64(31))


def test_field_hash_matches_its_definition(gpu):
    """pa_field_hash: sum mod 2^64 of mix(bits ^ mix(mix(level, GLOBAL box id, component) + cell)) over the valid cells --
    recomputed here in numpy.  Ghost cells do not enter, the box -> rank map does not enter (global ids)."""
    pf = synth.config1(16, 8, names=("temp", "Y_CH4"))
    H = gpu.Hierarchy(pf.levels)
    f = gpu.Field(H, 2, 1)
    f.set_val(-1.5)
    for c in range(2):
        f.upload_fabs(c, [[x[c] for x in l.fabs] for l in pf.levels])
    want = np.uint64(0)
    with np.errstate(over="ignore"):
        for l, lv in enumerate(pf.levels):
            for g, fab in enumerate(lv.fabs):
                for c in range(2):
                    key = _hmix64(np.array([(l << 56) ^ (g << 16) ^ c], dtype=np.uint64))[0]
                    cells = np.arange(fab[c].size, dtype=np.uint64)
                    bits = np.ascontiguousarray(fab[c]).view(np.uint64).ravel()
                    want = want + _hmix64(bits ^ _hmix64(key + cells)).sum(dtype=np.uint64)
    assert f.hash(0, 2) == int(want)
    assert f.hash(1, 1) != f.hash(0, 1)
    f.fill_ghosts(0, 1)                                    # ghost cells change, the fingerprint does not
    assert f.hash(0, 2) == int(want)


@pytest.mark.parametrize("base,mgs,walls", [(32, 16, True), (96, 96, False), (128, 128, True)])
def test_fused3_strips_match_separate_kernels(gpu, base, mgs, walls):
    """the third fused kernel (x strips of at most 64 cells, one barrier per plane) against the separate kernels, bit for bit,
    threshold clip included: narrow boxes (one strip), 96-wide boxes (two strips of 48) and 128-wide boxes (two of 64)"""
    from peleanalysis_b200 import synth
    pf = synth.config3(base, mgs, nlev=3 if base <= 32 else 2)
    per = (0, 0, 0) if walls else (1, 1, 1)
    kw = dict(threshold_prog=1, threshold_value=0.02)
    n0 = gpu.curv_fused_launches()
    a, _ = _gpu_curv(gpu, pf, per, (0, 0, 0), 300.0, 1800.0, kw, "tma_fused3")
    assert gpu.curv_fused_launches() > n0                      # the fused kernel ran (no silent fallback)
    b, _ = _gpu_curv(gpu, pf, per, (0, 0, 0), 300.0, 1800.0, kw, "tma")
    for c in range(a.shape[0]):
        assert bit_equal(a[c], b[c]), c
    for variant in ("tma_n3", "tma_nw"):                       # the same kernel without its K part / the barrier-free kernel, + MODE_DIV
        n0 = gpu.curv_fused_launches()
        a, _ = _gpu_curv(gpu, pf, per, (0, 0, 0), 300.0, 1800.0, kw, variant)
        assert gpu.curv_fused_launches() > n0
        for c in range(a.shape[0]):
            assert bit_equal(a[c], b[c]), (variant, c)
