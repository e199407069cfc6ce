"""CPU tier: the check bodies of tests/test_gpu_curv_options.py -- curvature's optional outputs against
OracleHier.curvature_ex on every kernel route, field layout and option sequence -- run through the emulated library
(tests/emu) on hierarchies shrunk to emulator sizes, plus one case with 128-wide boxes so that the big CTA shapes see
full-width tiles.  This is where indexing and sequencing mistakes show before any GPU time is spent; PTX behaviour and the
B200's own results are the GPU file's."""
import os

import pytest

import test_gpu_curv_options as C
from peleanalysis_b200 import synth
from test_emu_parity import emu  # noqa: F401  (fixture: the emulated library behind a private binding)

Case, F = C.Case, synth.FIELD_NAMES

MID = [
    Case("emu_c3_16_walls_sym", lambda: synth.config3(16, 8, names=F), (0, 1, 0), (1, 0, 1), True),
    Case("emu_edge_16_walls", lambda: synth.case_edge(16, 8, names=F), (0, 0, 0), (0, 0, 0), True),
    Case("emu_lshape_16", lambda: synth.case_lshape(16, 8, names=F), (1, 1, 1), (0, 0, 0), True),
    Case("emu_mixed_walls", lambda: synth.case_mixed(names=F), (0, 1, 1), (0, 0, 0), True),
    Case("emu_thin", lambda: synth.case_thin(names=F), (1, 1, 1), (0, 0, 0), False),
    Case("emu_np2_sym", lambda: synth.make_hierarchy((24, 12, 20), [[((12, 6, 10), (35, 17, 29))]], [2], 12, F,
                                                     prob_hi=(0.7, 0.35, 1.3)), (1, 0, 1), (0, 1, 0), True),
]
# 128-cell-wide boxes (every pair slot of the 8- / 16-warp CTA shapes in use), two side by side in y, a refined 64-wide
# level on top; periodic in x (the box is its own x neighbour), a wall in y, symmetry in z
FULL_WIDTH = Case("emu_full_width", lambda: synth.make_hierarchy((128, 32, 8), [[((64, 16, 4), (191, 47, 11))]], [2], 128, F),
                  (1, 0, 0), (0, 0, 1), True)


@pytest.fixture
def seed():
    """the emulator's in-order schedule for everything but the shuffled runs, which set their own seed"""
    os.environ["CUEMU_SEED"] = "0"
    yield
    os.environ["CUEMU_SEED"] = "0"


@pytest.mark.parametrize("route", C.ROUTES)
@pytest.mark.parametrize("case", MID, ids=lambda c: c.name)
def test_emulated_all_options_every_route(emu, seed, case, route):
    C.check_options(emu, case, "all_thr03", route)


@pytest.mark.parametrize("opt_name", ["gauss", "strain", "tensor", "veln", "all", "all_thr002"])
@pytest.mark.parametrize("case", [MID[0], MID[5]], ids=lambda c: c.name)
def test_emulated_each_option_set(emu, seed, case, opt_name):
    C.check_options(emu, case, opt_name, "tma")


@pytest.mark.parametrize("route", ["tma", "simple", "tma_fused", "tma_nw"])
def test_emulated_options_without_links(emu, seed, route):
    C.check_options(emu, MID[0], "all_thr002", route, "nolinks")


@pytest.mark.parametrize("case", [MID[0], MID[3]], ids=lambda c: c.name)
def test_emulated_options_shuffled_schedule(emu, case):
    """the shuffled schedule matters for the TMA ring's protocol only: the tma route"""
    os.environ["CUEMU_SEED"] = "20261017"
    try:
        C.check_options(emu, case, "all_thr002", "tma")
    finally:
        os.environ["CUEMU_SEED"] = "0"


@pytest.mark.parametrize("route", ["tma", "tma_big", "tma_fused", "tma_fused3", "tma_nw"])
def test_emulated_options_full_width_tiles(emu, seed, route):
    C.check_options(emu, FULL_WIDTH, "all_thr002", route)


LAYOUT_PARAMS = [(1, "offsets", "tma"), (1, "offsets", "tma_fused")] + [(ng, layout, route) for ng in (2, 3) for layout in C.LAYOUTS
                                                                         for route in ("tma", "simple")]


@pytest.mark.parametrize("ng,layout,route", LAYOUT_PARAMS, ids=["ng%d-%s-%s" % p for p in LAYOUT_PARAMS])
def test_emulated_options_field_layouts(emu, seed, ng, layout, route):
    C.check_options(emu, MID[1], "all_thr03", route, ng=ng, layout=layout)


@pytest.mark.parametrize("defer", ["0", "1"])
def test_emulated_options_stream_overlap(emu, seed, defer):
    """side-stream work run at the earliest (0) and the latest (1) point its events allow"""
    os.environ["CUEMU_DEFER_SIDE"] = defer
    try:
        C.check_stream_overlap(emu, MID[0], ("all",))
    finally:
        os.environ["CUEMU_DEFER_SIDE"] = "0"


@pytest.mark.parametrize("route", ["tma", "unfused", "tma_fused"])
def test_emulated_options_reuse_hierarchy(emu, seed, route):
    C.check_reuse(emu, MID[2], route)


@pytest.mark.parametrize("opt_name", ["all", "all_thr03"])
@pytest.mark.parametrize("route", ["tma", "simple", "tma_fused"])
def test_emulated_options_degenerate_values(emu, seed, route, opt_name):
    C.check_degenerate(emu, route, opt_name)


@pytest.mark.parametrize("fseed", C.FUZZ_SEEDS)
def test_emulated_options_fuzzed_hierarchies(emu, seed, fseed):
    C.check_fuzz(emu, fseed, ("tma", "tma_fused3"), ("all_thr03",))
