"""GPU (-m gpu): the optional outputs of pa_curvature -- GaussianCurvature, StrainRate, the nine ROST components,
VelFlameNormal, and threshold_prog combined with them -- against OracleHier.curvature_ex, at production box sizes (128^3),
on every kernel route, in both link modes, for every state-field layout the C ABI accepts.

Every output is compared bit for bit (signed zeros included) except GaussianCurvature, which is held cell by cell to the
1e-12 relative tolerance of pow(x, 4.0) (CUDA libdevice against glibc), with NaN, +inf and -inf in the same cells.  Every
input component carries seeded noise, so no field is even or odd about a wall and a wrong reflect rule for a velocity
component cannot hide.  Components the call does not own hold a sentinel before the call and must still hold it, ghost
cells included.  The check bodies take the binding P: tests/test_emu_curv_options.py runs them through the emulated library."""
import os
import zlib
from collections import namedtuple

import numpy as np
import pytest

import test_gpu_parity as G
from helpers import bit_equal, flat_from_fabs, max_rel
from oracle import oracle as O
from peleanalysis_b200 import synth
from test_fuzz_parity import random_case

pytestmark = pytest.mark.gpu

GAUSS_TOL = 1e-12
SENTINEL = -7.25e77
VEL = ("x_velocity", "y_velocity", "z_velocity")

# (name, builder, is_per, sym_dir, fused): `fused` says whether every fused / alternative flame-normal kernel takes the
# hierarchy (every box eligible), so that those routes must prove they ran
Case = namedtuple("Case", "name builder is_per sym fused")

OPTION_SETS = {
    "gauss": dict(do_gauss=1),
    "strain": dict(do_strain=1),
    "tensor": dict(do_strain=1, get_strain_tensor=1),
    "veln": dict(do_velnormal=1),
    "all": dict(do_gauss=1, do_strain=1, get_strain_tensor=1, do_velnormal=1),
    "all_thr002": dict(do_gauss=1, do_strain=1, get_strain_tensor=1, do_velnormal=1, do_threshold=1, threshold=0.02),
    "all_thr03": dict(do_gauss=1, do_strain=1, get_strain_tensor=1, do_velnormal=1, do_threshold=1, threshold=0.3),
}
ALL_SETS = ["all", "all_thr002", "all_thr03"]
ROUTES = ["tma", "tma_big", "simple", "unfused", "tma_fused", "tma_fused3", "tma_n3", "tma_nw"]
FUSED_ROUTES = ("tma_fused", "tma_fused3", "tma_n3", "tma_nw")       # each bumps curv_fused_launches() when it runs


def _two_boxes_128():
    """Two 128^3 boxes side by side on level 0, and two on level 1 touching the low x and y domain edges."""
    return synth.make_hierarchy((256, 128, 128), [[((0, 0, 64), (255, 127, 191))]], [2], 128, synth.FIELD_NAMES)


PRODUCTION = [
    Case("c3_128", lambda: synth.config3(128, 128, names=synth.FIELD_NAMES), (1, 0, 0), (0, 0, 1), True),
    Case("two_boxes_128", _two_boxes_128, (0, 1, 0), (1, 0, 0), True),
]
MID = [
    Case("c3_64_walls_sym", lambda: synth.config3(64, 32, names=synth.FIELD_NAMES), (0, 1, 0), (1, 0, 1), True),
    Case("edge_32_walls", lambda: synth.case_edge(32, 16, names=synth.FIELD_NAMES), (0, 0, 0), (0, 0, 0), True),
    Case("lshape_32", lambda: synth.case_lshape(32, 16, names=synth.FIELD_NAMES), (1, 1, 1), (0, 0, 0), True),
    Case("mixed_walls", lambda: synth.case_mixed(names=synth.FIELD_NAMES), (0, 1, 1), (0, 0, 0), True),
    Case("thin", lambda: synth.case_thin(names=synth.FIELD_NAMES), (1, 1, 1), (0, 0, 0), False),
    Case("np2_sym", lambda: synth.case_np2(names=synth.FIELD_NAMES), (1, 0, 1), (0, 1, 0), True),
]
FUZZ_SEEDS = list(range(0, 24, 2))


def fuzz_case(seed):
    """The curvature layouts of test_fuzz_parity.py, with velocity.  Whether the fused kernels take them varies (odd widths,
    2-cell boxes): a fallback to the default kernels is allowed here, and its result is checked all the same."""
    def build():
        pf, _, _ = random_case(1000 + seed, True, names=synth.FIELD_NAMES)
        return pf
    _, is_per, sym = random_case(1000 + seed, True)
    return Case("fuzz%d" % seed, build, is_per, sym, None)


# ---- inputs and the oracle, built once per case (the production cases take seconds on the host) -----------------------------
_CACHE = {}


def add_noise(pf, seed):
    """Seeded noise on every component, scaled to the component's range."""
    rng = np.random.default_rng(seed)
    amp = {"temp": 3.0, "Y_CH4": 1e-4}
    for lv in pf.levels:
        for fab in lv.fabs:
            for c, n in enumerate(pf.names):
                fab[c] += amp.get(n, 0.02) * rng.standard_normal(fab[c].shape)
    return pf


def case_inputs(case, make=None):
    """(pf, s, U, prog_min, prog_max, oracle hierarchy) of a case; `make` replaces builder + noise (degenerate inputs)."""
    if _CACHE.get("key") != case.name:
        _CACHE.clear()
        pf = make() if make else add_noise(case.builder(), zlib.crc32(case.name.encode()))
        OH = O.OracleHier(pf, case.is_per, case.sym)
        s = OH.flatten(pf.comp("temp"))
        U = np.stack([OH.flatten(pf.comp(n)) for n in VEL])
        pmin, pmax = (0.0, 1.0) if make else (float(s.min()), float(s.max()))
        _CACHE.update(key=case.name, inputs=(pf, s, U, pmin, pmax, OH), oracle={})
    return _CACHE["inputs"]


def oracle_outputs(case, thr, make=None):
    """curvature_ex of the case, every optional output; thr None: no threshold_prog"""
    pf, s, U, pmin, pmax, OH = case_inputs(case, make)
    orc = _CACHE["oracle"]
    if thr not in orc:
        orc[thr] = OH.curvature_ex(s, U, pmin, pmax, thr is not None, 1e-4 if thr is None else thr)
    return orc[thr]


def curv_opts(P, opts, pmin, pmax):
    o = P.CurvOpts()
    o.prog_min, o.prog_max = pmin, pmax
    for k, v in opts.items():
        setattr(o, k, v)
    return o


def expected(r, o):
    """[(output name, oracle array)] in the library's output order"""
    w = list(zip(["Progress", "MeanCurvature", "FlameNormalX", "FlameNormalY", "FlameNormalZ"], r["core"]))
    if o.do_gauss:
        w.append(("GaussianCurvature", r["gauss"]))
    if o.do_strain:
        w.append(("StrainRate", r["strain"]))
        if o.get_strain_tensor:
            w += [("ROST_dU%sd%s" % ("xyz"[m], "xyz"[n]), r["rost"][3 * m + n]) for m in range(3) for n in range(3)]
    if o.do_velnormal:
        w.append(("VelFlameNormal", r["veln"]))
    return w


def gauss_mismatch(got, want, tol=GAUSS_TOL):
    """Indices where GaussianCurvature differs: NaN / +inf / -inf not in the same cells, a finite cell off by more than tol
    relative, or a zero of the other sign.  Cell by cell: one NaN must not decide the comparison of the whole field."""
    special = (np.isnan(got) != np.isnan(want)) | ((got == np.inf) != (want == np.inf)) | ((got == -np.inf) != (want == -np.inf))
    fin = np.isfinite(want)
    with np.errstate(invalid="ignore"):
        off = fin & ~(np.abs(got - want) <= tol * np.abs(want))
    zero_sign = fin & (want == 0) & (np.signbit(got) != np.signbit(want))
    return np.flatnonzero(special | off | zero_sign)


def assert_matches(got, want, tag):
    assert len(got) == len(want), (tag, len(got), len(want))
    for g, (name, w) in zip(got, want):
        if name == "GaussianCurvature":
            bad = gauss_mismatch(g, w)
            assert bad.size == 0, (tag, name, bad.size, bad[:6], g[bad[:6]], w[bad[:6]])
        else:
            assert bit_equal(g, w), (tag, name, max_rel(g, w), np.flatnonzero(g.view(np.int64) != w.view(np.int64))[:6])


# ---- one pa_curvature call ---------------------------------------------------------------------------------------------------
# Field layouts of the state and output fields: "plain" is temp, u, v, w (comp_S 0, comp_vel 1) and outputs from component 0;
# "offsets" stores the velocity first and temp last with an unrelated component between them (comp_vel 0, comp_S 4) and
# writes the outputs from component 2 of a field with one spare component after them.
LAYOUTS = {
    "plain": (["temp"] + list(VEL), 0, 0),
    "offsets": (list(VEL) + [None, "temp"], 2, 1),
}


def assert_sentinel(P, f, comps, tag):
    for c in comps:
        for l, lv in enumerate(f.hier.levels):
            for b in range(len(lv.boxes)):
                g = f.download_grown(l, b, c)
                assert bit_equal(g, np.full(g.shape, SENTINEL)), (tag, "component %d was written" % c, l, b, int((g != SENTINEL).sum()))


def run_curvature(P, pf, case, o, route, links="links", ng=1, layout="plain", H=None, state=None, out=None):
    """pa_curvature on `route`; returns the outputs (flat, library order), the hierarchy and both fields.  Checks that the
    call left every component it does not own untouched (sentinel, ghost cells included) and the inputs' valid cells too,
    and that a fused / alternative route ran where the case is eligible for it."""
    G._set_stencil(route)
    names, comp_out, spare = LAYOUTS[layout]
    if H is None:
        H = P.Hierarchy(pf.levels, case.is_per, case.sym, flags=G.LINK_MODES[links])
    if state is None:
        state = P.Field(H, len(names), ng)
        state.set_val(SENTINEL)
        for v, n in enumerate(names):
            if n:
                state.upload_fabs(v, [[f[pf.comp(n)] for f in l.fabs] for l in pf.levels])
    nout = P.curvature_num_outputs(o)
    if out is None:
        out = P.Field(H, comp_out + nout + spare, 1)
    out.set_val(SENTINEL)
    n0 = P.curv_fused_launches()
    P.curvature(state, names.index("temp"), names.index("x_velocity"), o, out, comp_out)
    P.sync()
    ran = P.curv_fused_launches() > n0
    tag = (case.name, route, links, ng, layout)
    if route in FUSED_ROUTES and case.fused:
        assert ran, (tag, "the route's kernel did not run (silent fallback)")
    if route not in FUSED_ROUTES:
        assert not ran, tag
    got = [flat_from_fabs(out.download_fabs(c)) for c in range(comp_out, comp_out + nout)]
    assert_sentinel(P, out, [c for c in range(out.ncomp) if not comp_out <= c < comp_out + nout], tag)
    assert_sentinel(P, state, [v for v, n in enumerate(names) if n is None], tag)
    for v, n in enumerate(names):
        if n:
            assert bit_equal(flat_from_fabs(state.download_fabs(v)), flat_from_fabs([[f[pf.comp(n)] for f in l.fabs] for l in pf.levels])), \
                (tag, "input %s changed" % n)
    return got, H, state, out


# ---- check bodies (P: the binding; the emulator tier runs the same bodies) ----------------------------------------------------
def check_options(P, case, opt_name, route, links="links", ng=1, layout="plain"):
    opts = OPTION_SETS[opt_name]
    pf, s, U, pmin, pmax, _ = case_inputs(case)
    o = curv_opts(P, opts, pmin, pmax)
    got, _, _, _ = run_curvature(P, pf, case, o, route, links, ng, layout)
    want = expected(oracle_outputs(case, opts.get("threshold") if opts.get("do_threshold") else None), o)
    assert_matches(got, want, (case.name, opt_name, route, links, ng, layout))


def check_stream_overlap(P, case, opt_names=("gauss", "tensor", "all")):
    """PA_STREAM_OVERLAP=1 with gauss and strain, no threshold: the case in which DIV's ghost fill of the refined levels runs
    on the side stream, while GAUSS / STRAIN follow on the caller's stream."""
    os.environ["PA_STREAM_OVERLAP"] = "1"
    try:
        for opt_name in opt_names:
            check_options(P, case, opt_name, "tma")
    finally:
        os.environ.pop("PA_STREAM_OVERLAP", None)


REUSE_SEQUENCE = [dict(do_gauss=1), dict(do_strain=1), OPTION_SETS["all_thr002"], dict(do_velnormal=1, do_threshold=1, threshold=0.3), {}]


def check_reuse(P, case, route):
    """One hierarchy and one state field, option sets in sequence: the scratch fields the library keeps on the hierarchy
    (tmpG, tmpH, tmpW) are sized by the first use, and the state's ghost cells hold what the previous call left there."""
    pf, s, U, pmin, pmax, _ = case_inputs(case)
    H = state = out = None
    for opts in REUSE_SEQUENCE:
        o = curv_opts(P, opts, pmin, pmax)
        if out is not None and out.ncomp < P.curvature_num_outputs(o):
            out = None
        got, H, state, out = run_curvature(P, pf, case, o, route, H=H, state=state, out=out)
        want = expected(oracle_outputs(case, opts.get("threshold") if opts.get("do_threshold") else None), o)
        assert_matches(got, want, (case.name, route, "reuse", sorted(opts)))


DEGENERATE = Case("degenerate", None, (1, 1, 1), (0, 0, 0), True)


def _degenerate_inputs():
    """test_curvature_degenerate_values' box kinds for temp (flat, around the 1e-250 guard, +-1e150, +-1e-300 with zeros;
    progMin 0, progMax 1 so that c == S), noisy velocity"""
    pf = synth.config1(16, 8, names=synth.FIELD_NAMES)
    rng = np.random.default_rng(7)
    t = pf.comp("temp")
    for lv in pf.levels:
        for b, ((lo, hi), fab) in enumerate(zip(lv.boxes, lv.fabs)):
            kind = (b + lo[0] // 8) % 4
            shape = fab[t].shape
            if kind == 0:
                fab[t][...] = 0.25
            elif kind == 1:
                fab[t][...] = rng.uniform(-1, 1, shape) * 10.0 ** rng.integers(-262, -240, shape)
            elif kind == 2:
                fab[t][...] = rng.uniform(-1, 1, shape) * 1e150
            else:
                fab[t][...] = np.where(rng.random(shape) < 0.5, 0.0, rng.uniform(-1, 1, shape) * 1e-300)
            for n in VEL:
                fab[pf.comp(n)] += 0.02 * rng.standard_normal(shape)
    return pf


def check_degenerate(P, route, opt_name):
    opts = OPTION_SETS[opt_name]
    pf, s, U, pmin, pmax, _ = case_inputs(DEGENERATE, _degenerate_inputs)
    o = curv_opts(P, opts, pmin, pmax)
    got, _, _, _ = run_curvature(P, pf, DEGENERATE, o, route)
    r = oracle_outputs(DEGENERATE, opts.get("threshold") if opts.get("do_threshold") else None, _degenerate_inputs)
    if opt_name == "all":
        assert np.isnan(r["gauss"]).any()                                       # the inputs reach the special values
    assert_matches(got, expected(r, o), ("degenerate", route, opt_name))


def check_fuzz(P, seed, routes=ROUTES, opt_names=("all", "all_thr03")):
    case = fuzz_case(seed)
    for opt_name in opt_names:
        for route in routes:
            check_options(P, case, opt_name, route)


# ---- the tests ----------------------------------------------------------------------------------------------------------------
def _production_params():
    out = []
    for case in PRODUCTION:
        for opt_name in ALL_SETS:
            out += [(case, opt_name, r, "links") for r in ROUTES]
            out.append((case, opt_name, "tma", "nolinks"))
        out += [(case, opt_name, "tma", "links") for opt_name in ("gauss", "strain", "tensor", "veln")]
    return out


def _mid_params():
    return [(case, opt_name, route, links) for case in MID for opt_name in OPTION_SETS for route in ROUTES for links in G.LINK_MODES]


def _ids(p):
    return "-".join([p[0].name] + list(p[1:]))


@pytest.mark.parametrize("case,opt_name,route,links", _production_params(), ids=[_ids(p) for p in _production_params()])
def test_options_production_boxes(gpu, case, opt_name, route, links):
    check_options(gpu, case, opt_name, route, links)


@pytest.mark.parametrize("case,opt_name,route,links", _mid_params(), ids=[_ids(p) for p in _mid_params()])
def test_options_mid_size(gpu, case, opt_name, route, links):
    check_options(gpu, case, opt_name, route, links)


@pytest.mark.parametrize("seed", FUZZ_SEEDS)
def test_options_fuzzed_hierarchies(gpu, seed):
    check_fuzz(gpu, seed)


LAYOUT_PARAMS = [(case, ng, layout, route) for case in (MID[0], MID[1], MID[5]) for ng in (1, 2, 3) for layout in LAYOUTS
                 for route in (ROUTES if ng == 1 else ["tma", "simple", "unfused"])]


@pytest.mark.parametrize("case,ng,layout,route", LAYOUT_PARAMS, ids=["%s-ng%d-%s-%s" % (c.name, n, l, r) for c, n, l, r in LAYOUT_PARAMS])
def test_options_field_layouts(gpu, case, ng, layout, route):
    """state nghost 1, 2 and 3 (k_velnormal reads the velocity through a layout other than the output's); comp_S / comp_vel
    other than 0 / 1 and comp_out 2, with the components the call does not own checked for stray writes"""
    for opt_name in ("all", "all_thr03"):
        check_options(gpu, case, opt_name, route, ng=ng, layout=layout)


@pytest.mark.parametrize("case", PRODUCTION + MID[:3], ids=lambda c: c.name)
def test_options_stream_overlap(gpu, case):
    check_stream_overlap(gpu, case)


@pytest.mark.parametrize("route", ["tma", "simple", "unfused", "tma_fused", "tma_fused3", "tma_nw"])
@pytest.mark.parametrize("case", [PRODUCTION[0], MID[0], MID[3]], ids=lambda c: c.name)
def test_options_reuse_hierarchy(gpu, case, route):
    check_reuse(gpu, case, route)


@pytest.mark.parametrize("opt_name", ["all", "all_thr03"])
@pytest.mark.parametrize("route", ROUTES)
def test_options_degenerate_values(gpu, route, opt_name):
    check_degenerate(gpu, route, opt_name)
