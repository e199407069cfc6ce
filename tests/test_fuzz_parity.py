"""CPU tier: pseudo-random AMR hierarchies (seeded; box layouts, sizes, refinement ratio, periodicity and wall kinds vary)
through three implementations that must agree bit for bit:
   the compiled, unmodified reference (oracle/_ref, where it was built)  ==  the C restatement (oracle/)
   the C restatement  ==  the CUDA kernel sources under the execution-model emulator (tests/emu), through the C ABI
The golden cases of tests/cases.py were designed around the branches of SURVEY 3.3; these layouts are not designed at all
(ragged neighbours, boxes 2-3 cells thick, fine boxes on domain edges, two refined levels, odd box widths)."""
import os

import numpy as np
import pytest

import test_gpu_parity as G
from helpers import bit_equal, flat_from_fabs, max_rel
from oracle import oracle as O
from peleanalysis_b200 import plotfile, synth
from test_emu_parity import emu  # noqa: F401  (fixture: the emulated library behind a private binding)


def _overlaps(a, b):
    return all(a[0][d] <= b[1][d] and b[0][d] <= a[1][d] for d in range(3))


def _random_boxes(rng, lo, hi, nmax, min_size=2, max_size=10):
    """Up to nmax disjoint boxes inside [lo, hi] (inclusive index box)."""
    out = []
    for _ in range(40):
        if len(out) >= nmax:
            break
        size = [int(rng.integers(min_size, min(max_size, hi[d] - lo[d] + 1) + 1)) for d in range(3)]
        blo = [int(rng.integers(lo[d], hi[d] - size[d] + 2)) for d in range(3)]
        b = (tuple(blo), tuple(blo[d] + size[d] - 1 for d in range(3)))
        if not any(_overlaps(b, o) for o in out):
            out.append(b)
    return out


def random_case(seed, curvature, names=("temp",)):
    rng = np.random.default_rng(seed)
    base = tuple(int(rng.choice([8, 10, 12, 16, 20])) for _ in range(3))
    mgs = int(rng.choice([6, 8, 12, 16, 32]))
    r1 = 2 if curvature else int(rng.choice([2, 2, 4]))          # the reference's curvature hard-codes ratio 2
    is_per = tuple(int(rng.integers(0, 2)) for _ in range(3))
    sym = tuple(int(rng.integers(0, 2)) if not is_per[d] else 0 for d in range(3))
    regions, ratios = [], []

    def refined(boxes, r):
        # chop in COARSE index space, then refine: every fine box stays aligned to the ratio (AMReX blocking factor)
        out = []
        for lo, hi in boxes:
            for plo, phi in synth.chop(lo, hi, max(1, mgs // r)):
                out.append((tuple(v * r for v in plo), tuple((v + 1) * r - 1 for v in phi)))
        return out
    c1 = _random_boxes(rng, (0, 0, 0), tuple(v - 1 for v in base), int(rng.integers(1, 4)))
    regions.append(refined(c1, r1))
    ratios.append(r1)
    if rng.random() < 0.5:
        # a third level: boxes inside one level-1 region, two level-1 cells away from its edge (proper nesting)
        plo, phi = regions[0][int(rng.integers(0, len(regions[0])))]
        ilo, ihi = tuple(v + 2 for v in plo), tuple(v - 2 for v in phi)
        if all(ihi[d] - ilo[d] >= 1 for d in range(3)):
            c2 = _random_boxes(rng, ilo, ihi, int(rng.integers(1, 3)), 2, 6)
            if c2:
                regions.append(refined(c2, 2))
                ratios.append(2)
    prob_hi = (1.0, 1.0, 1.0) if rng.random() < 0.7 else (0.7, 0.35, 1.3)
    pf = synth.make_hierarchy(base, regions, ratios, mgs, names, prob_hi=prob_hi, header_ratio=None)
    return pf, is_per, sym


def _flat(pf):
    return np.concatenate([f[0].ravel() for l in pf.levels for f in l.fabs])


SEEDS = list(range(24))


@pytest.mark.parametrize("seed", SEEDS)
def test_random_hierarchy_emulated_kernels_equal_oracle(emu, seed):  # noqa: F811
    curv = seed % 2 == 0
    pf, is_per, sym = random_case(1000 + seed, curv)
    os.environ["CUEMU_SEED"] = str(seed)
    if seed % 3 == 0:
        os.environ["PA_BCFILL_V2"] = "0"          # every third seed through the unstaged coarse-fine fill
    try:
        OH = O.OracleHier(pf, is_per, sym)
        s = _flat(pf)
        want = OH.grad(s)
        for stencil in ("tma", "simple", "tma_big"):
            out, _, _ = G._gpu_grad(emu, pf, is_per, sym, stencil=stencil)
            for c in range(4):
                assert bit_equal(out[c], want[c]), (seed, stencil, c, max_rel(out[c], want[c]), [l.boxes for l in pf.levels])
        if curv:
            pmin, pmax = float(s.min()), float(s.max())
            wk = OH.curvature(s, pmin, pmax)
            # (the fused / plane-staged / barrier-free kernels take a hierarchy only if every box is eligible -- even width, at
            # least three or four cells -- and hand it to the default kernels otherwise: both outcomes are checked here)
            for stencil in ("tma", "tma_fused", "tma_fused3", "tma_n3", "tma_nw"):
                out, _ = G._gpu_curv(emu, pf, is_per, sym, pmin, pmax, {}, stencil)
                for c in range(5):
                    assert bit_equal(out[c], wk[c]), (seed, "curvature", stencil, c, [l.boxes for l in pf.levels])
    finally:
        os.environ["CUEMU_SEED"] = "0"
        os.environ.pop("PA_BCFILL_V2", None)


@pytest.mark.skipif(not O.have_ref(), reason="oracle/_ref not built (python oracle/build_ref.py)")
@pytest.mark.parametrize("seed", SEEDS[:10])
def test_random_hierarchy_oracle_equals_compiled_reference(tmp_path, seed):
    curv = seed % 2 == 0
    pf, is_per, sym = random_case(1000 + seed, curv)
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    OH = O.OracleHier(pf, is_per, sym)
    s = _flat(pf)
    O.run_ref("grad", d, d + "_gt", gradVar="temp", is_per=list(is_per), sym_dir=list(sym))
    r = plotfile.read_plotfile(d + "_gt")
    want = OH.grad(s)
    for c, n in enumerate(["temp_gx", "temp_gy", "temp_gz", "||gradtemp||"]):
        got = np.concatenate([f[r.comp(n)].ravel() for l in r.levels for f in l.fabs])
        assert bit_equal(got, want[c]), (seed, n, max_rel(got, want[c]), [l.boxes for l in pf.levels])
    if curv:
        O.run_ref("curvature", d, d + "_K", progressName="temp", is_per=list(is_per), sym_dir=list(sym))
        r = plotfile.read_plotfile(d + "_K")
        pmin, pmax = plotfile.file_min_max(d, "temp", len(pf.levels))
        wk = OH.curvature(s, pmin, pmax)
        for c, n in enumerate(["Progress", "MeanCurvature_temp", "FlameNormalX_temp", "FlameNormalY_temp", "FlameNormalZ_temp"]):
            got = np.concatenate([f[r.comp(n)].ravel() for l in r.levels for f in l.fabs])
            assert bit_equal(got, wk[c]), (seed, n, max_rel(got, wk[c]), [l.boxes for l in pf.levels])
