"""CPU tier: the kernel SOURCES of peleanalysis_b200/csrc, compiled by g++ against the CUDA execution-model emulator of
tests/emu (fibers for threads, mbarrier / bulk-copy / shuffle semantics, deadlock detection), run the same parity
checks as the GPU tests -- same C ABI, same oracle, same golden vectors of the compiled reference.

This is test infrastructure: it checks descriptor use, indexing, the TMA ring's producer/consumer protocol and the
host-side sequencing before any GPU time is spent.  It is NOT a CPU path of the product: the emulated library lives under
tests/emu/_build, only this file loads it (through a private copy of the ctypes binding), and capi.py can open nothing but
lib/libpelestencil_b200.so (tests/test_capi_surface.py).  PTX semantics, the MUFU-seeded sqrt / reciprocal forms and
performance are GPU-only matters (tests/test_gpu_parity.py)."""
import importlib.util
import os
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emu"))

import test_gpu_parity as G  # noqa: E402  (the GPU tests' bodies are reused as plain functions)
from cases import CASES  # noqa: E402


@pytest.fixture(scope="module")
def emu():
    import build_emu
    from peleanalysis_b200 import capi as product_capi
    lib = build_emu.build()
    spec = importlib.util.spec_from_file_location("capi_emulated", product_capi.__file__)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    m.LIB_PATH = lib                     # a private module instance: the product binding itself is untouched
    old = {k: os.environ.get(k) for k in ("PA_NORMAL_MATH", "PA_STENCIL", "PA_TMA_SMALL", "PA_CURV_FUSED", "PA_NORMAL_F3", "PA_NORMAL_W", "PA_CURV_UNFUSED",
                                       "CUEMU_SEED")}
    os.environ["PA_NORMAL_MATH"] = "fast"   # no device self-test: the emulator has no MUFU (sqrt_fast == sqrt there)
    m.init(0)
    yield m
    for k, v in old.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


@pytest.fixture(params=[0, 20261017, -6], ids=["inorder", "shuffled", "starved"])
def schedule(request):
    """inorder: threads run round-robin and async copies land within the round; shuffled: a fresh pseudo-random thread
    order every scheduler round and async copies that land 0-3 rounds late; starved: shuffled, and every round each WARP is
    left out with probability 0.6, so warps drift many instructions apart (protocols whose phase bits alias when one warp
    gets two steps ahead of another hang here -- as one did on the GPU in round 2 -- instead of passing by luck)."""
    os.environ["CUEMU_SEED"] = str(request.param if request.param >= 0 else 31337)
    os.environ["CUEMU_STARVE"] = str(-request.param) if request.param < 0 else "0"
    yield request.param
    os.environ["CUEMU_SEED"] = "0"
    os.environ["CUEMU_STARVE"] = "0"


def _thin_out(schedule, stencil, links):
    """Not the full cross product (the suite has to stay a few minutes): the shuffled schedule matters for the TMA pipeline
    only; materialised ghosts (nolinks) are a property of the fill, not of the CTA shape or of the prefetch warp."""
    if schedule and (stencil == "simple" or links == "nolinks"):
        pytest.skip("combination not in the thinned-out matrix")
    if schedule < 0 and stencil not in ("tma", "tma_fused"):
        pytest.skip("combination not in the thinned-out matrix")       # starved warps matter for the mbarrier protocols only
    if schedule and stencil in ("tma_fused3", "tma_nw"):
        pytest.skip("combination not in the thinned-out matrix")       # block barriers / plain loads only; the cp.async staging is tma_n3's
    if links == "nolinks" and stencil not in ("tma", "tma_fused", "tma_fused3", "tma_n3", "tma_nw", "simple"):
        pytest.skip("combination not in the thinned-out matrix")


GRAD_CASES = [n for n, c in CASES.items() if "grad" in c[3]]
CURV_CASES = [n for n, c in CASES.items() if "curvature" in c[3]]


@pytest.mark.parametrize("links", list(G.LINK_MODES))
@pytest.mark.parametrize("stencil", ["tma", "tma_big", "simple"])
@pytest.mark.parametrize("name", GRAD_CASES)
def test_emulated_grad_matches_reference_golden(emu, schedule, name, stencil, links):
    _thin_out(schedule, stencil, links)
    G.test_grad_matches_reference_golden(emu, name, stencil, links)


@pytest.mark.parametrize("links", list(G.LINK_MODES))
@pytest.mark.parametrize("stencil", ["tma", "tma_fused", "tma_fused3", "tma_n3", "tma_nw", "tma_big", "simple"])
@pytest.mark.parametrize("name", CURV_CASES)
def test_emulated_curvature_matches_reference_golden(emu, schedule, name, stencil, links):
    _thin_out(schedule, stencil, links)
    G.test_curvature_matches_reference_golden(emu, name, stencil, links)


@pytest.mark.parametrize("name", list(CASES))
def test_emulated_ghost_cells_match_oracle(emu, name):
    os.environ["CUEMU_SEED"] = "0"
    G.test_ghost_cells_match_oracle(emu, name)


@pytest.mark.parametrize("stencil", ["tma", "tma_big", "simple"])
def test_emulated_curvature_degenerate_values(emu, stencil):
    os.environ["CUEMU_SEED"] = "0"
    G.test_curvature_degenerate_values(emu, stencil)


def test_emulated_field_hash(emu):
    os.environ["CUEMU_SEED"] = "0"
    G.test_field_hash_matches_its_definition(emu)


def test_emulated_multi_variable_and_phases(emu, schedule):
    G.test_multi_variable_grad_equals_single(emu)
    G.test_curvature_two_phases_equal_one_call(emu, "c1_periodic")
    G.test_flat_field_takes_the_clamp(emu)


@pytest.mark.parametrize("case,kw", [
    ("config3", dict(base=32, mgs=16)),
    ("config5", dict(base=16, mgs=8, ncomp=2, ratios=(2, 4, 2))),
    ("lshape", dict(base=32, mgs=16)),
])
def test_emulated_midsize_vs_oracle(emu, case, kw):
    os.environ["CUEMU_SEED"] = "7"
    try:
        G.test_midsize_grad_and_curvature_vs_oracle(emu, case, kw, "tma")
        G.test_midsize_grad_and_curvature_vs_oracle(emu, case, kw, "tma_fused")
    finally:
        os.environ["CUEMU_SEED"] = "0"


@pytest.mark.parametrize("name", [n for n in CASES if n not in ("c3_threshold", "c1_options")])
def test_emulated_side_stream_runs_late(emu, name):
    """PA_STREAM_OVERLAP=1 (opt-in): the ghost fill of the refined levels runs on a side stream, overlapped with the
    stencil of level 0 (api.cu: fork_side / join_side).  The emulator executes side-stream work either at once -- the
    EARLIEST order the events allow -- or holds it back until something waits for that stream -- the LATEST order.
    Bit-exact results in both say the cross-stream dependencies are all expressed as events."""
    os.environ["CUEMU_SEED"] = "0"
    os.environ["PA_STREAM_OVERLAP"] = "1"
    try:
        for defer in ("0", "1"):
            os.environ["CUEMU_DEFER_SIDE"] = defer
            tools = CASES[name][3]
            if "grad" in tools:
                G.test_grad_matches_reference_golden(emu, name, "tma", "links")
            if "curvature" in tools:
                G.test_curvature_matches_reference_golden(emu, name, "tma", "links")
                if defer == "1":
                    G.test_curvature_matches_reference_golden(emu, name, "simple", "nolinks")
    finally:
        os.environ["CUEMU_DEFER_SIDE"] = "0"
        os.environ.pop("PA_STREAM_OVERLAP", None)


@pytest.mark.parametrize("builder", ["config1", "mixed", "config3"])
def test_emulated_wide_ghost_inputs(emu, builder):
    from peleanalysis_b200 import synth
    os.environ["CUEMU_SEED"] = "0"
    b = {"config1": lambda: synth.config1(16, 8), "mixed": synth.case_mixed, "config3": lambda: synth.config3(16, 8)}[builder]
    G.check_wide_ghost_inputs(emu, b)


@pytest.mark.parametrize("name", list(CASES))
def test_emulated_unstaged_bcfill(emu, name):
    """PA_BCFILL_V2=0: the coarse-fine / wall fill in which every ghost cell gathers its coarse cells itself (the default
    stages them in shared memory) -- ghost cells one by one against the oracle, then both tools against the golden vectors."""
    os.environ["CUEMU_SEED"] = "11"
    os.environ["PA_BCFILL_V2"] = "0"
    try:
        G.test_ghost_cells_match_oracle(emu, name)
        tools = CASES[name][3]
        if "grad" in tools:
            G.test_grad_matches_reference_golden(emu, name, "tma", "links")
        if "curvature" in tools:
            G.test_curvature_matches_reference_golden(emu, name, "tma", "nolinks")
    finally:
        os.environ["CUEMU_SEED"] = "0"
        os.environ.pop("PA_BCFILL_V2", None)


@pytest.mark.parametrize("stencil", ["tma", "tma_fused"])
def test_emulated_full_width_tiles(emu, stencil):
    """128-cell-wide boxes: 64 x-pairs per row, 8 rows per tile -- every one of the 512 pair slots of the big CTA shapes is
    in use (the golden cases have narrow boxes), two boxes side by side in y so that linked y rows and periodic x / z wraps
    onto the box itself occur at full width; a refined 64-wide level on top."""
    from oracle import oracle as O
    from peleanalysis_b200 import synth
    from helpers import bit_equal, flat_from_fabs
    os.environ["CUEMU_SEED"] = "13"
    try:
        pf = synth.make_hierarchy((128, 32, 8), [[((64, 16, 4), (191, 47, 11))]], [2], 128, ("temp",))
        OH = O.OracleHier(pf)
        s = OH.flatten(0)
        out, _, _ = G._gpu_grad(emu, pf, (1, 1, 1), (0, 0, 0), stencil=stencil)
        want = OH.grad(s)
        for c in range(4):
            assert bit_equal(out[c], want[c]), c
        pmin, pmax = float(s.min()), float(s.max())
        outc, _ = G._gpu_curv(emu, pf, (1, 1, 1), (0, 0, 0), pmin, pmax, {}, stencil)
        wk = OH.curvature(s, pmin, pmax)
        for c in range(5):
            assert bit_equal(outc[c], wk[c]), ("curvature", c)
    finally:
        os.environ["CUEMU_SEED"] = "0"


@pytest.mark.parametrize("base,mgs", [((256, 8, 4), 256), ((1024, 4, 4), 1024), ((7, 5, 3), 8), ((2, 2, 2), 2), ((1, 1, 1), 1)])
def test_emulated_extreme_box_shapes(emu, base, mgs):
    """Very wide rows (4 and 1 row per tile), odd tiny boxes, and the one-cell periodic box that is its own neighbour six times."""
    from oracle import oracle as O
    from peleanalysis_b200 import synth
    from helpers import bit_equal
    os.environ["CUEMU_SEED"] = "17"
    try:
        pf = synth.make_hierarchy(base, [], [], mgs, ("temp",))
        OH = O.OracleHier(pf)
        s = OH.flatten(0)
        out, _, _ = G._gpu_grad(emu, pf, (1, 1, 1), (0, 0, 0))
        want = OH.grad(s)
        for c in range(4):
            assert bit_equal(out[c], want[c]), c
        pmin, pmax = float(s.min()), float(s.max())
        if pmin < pmax:
            outc, _ = G._gpu_curv(emu, pf, (1, 1, 1), (0, 0, 0), pmin, pmax, {})
            wk = OH.curvature(s, pmin, pmax)
            for c in range(5):
                assert bit_equal(outc[c], wk[c]), ("curvature", c)
    finally:
        os.environ["CUEMU_SEED"] = "0"


def test_box_side_limit_is_an_error(emu):
    from peleanalysis_b200 import synth
    pf = synth.make_hierarchy((1100, 4, 4), [], [], 2048, ("temp",), fill=False)
    with pytest.raises(emu.PaError) as e:
        emu.Hierarchy(pf.levels)
    assert "1024" in str(e.value)


def test_emulated_recv_slab_has_one_owner(emu):
    """The recv slab is shared by all fields of a hierarchy: once another field packs / receives, the first field's
    "received" mark must be gone, or a ghost fill on it would silently read the other field's data (round-1 advisor finding)."""
    from peleanalysis_b200 import synth
    P = emu
    pf = synth.config1(16, 8)
    H = P.Hierarchy(pf.levels, is_per=(1, 1, 1), rank=0, nranks=2)
    a, b = P.Field(H, 1, 1), P.Field(H, 1, 1)
    L = P.lib()
    P.check(L.pa_exchange_pack(a.f, 0, 1))
    P.check(L.pa_exchange_mark_received(a.f, 0, 1))
    a.fill_ghosts(0, 1)                                   # a's data is in the slab: accepted
    P.check(L.pa_exchange_pack(b.f, 0, 1))                # b's transport will overwrite the slab
    with pytest.raises(P.PaError) as e:
        a.fill_ghosts(0, 1)
    assert e.value.code == -5
    P.check(L.pa_exchange_mark_received(b.f, 0, 1))
    b.fill_ghosts(0, 1)
    P.check(L.pa_exchange_mark_received(a.f, 0, 1))       # marking a again takes the slab away from b
    with pytest.raises(P.PaError):
        b.fill_ghosts(0, 1)


@pytest.mark.parametrize("base,mgs,walls", [(32, 16, True), (72, 72, False)])
def test_emulated_fused3_strips(emu, base, mgs, walls):
    G.test_fused3_strips_match_separate_kernels(emu, base, mgs, walls)
