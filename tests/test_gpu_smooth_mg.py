"""B200: pa_smooth with the multigrid preconditioner (PA_SMOOTH_PRECOND_MG) -- the same discrete system as the Jacobi-preconditioned
solve of tests/test_gpu_smooth.py, checked against the SciPy oracle on the golden fixtures, in the stiff regime where Jacobi
runs out of iterations, through the V-cycle on its own (pa_debug_smooth_vcycle), and through curvature3d smooth_precond=mg.
The check bodies take the binding module P so that tests/test_emu_smooth_mg.py runs them under the CPU emulation of the kernels."""
import numpy as np
import pytest

import test_gpu_smooth as G
from helpers import bit_equal, flat_from_fabs
from test_gpu_tools import exes  # noqa: F401  (fixture: the built host executables)

pytestmark = pytest.mark.gpu

TOL_REL = G.TOL_REL
# stiff regime: smoothing_time / dx_finest^2 of these ratios on two fixtures with walls / symmetry and with three levels
STIFF_CASES = ["c3_three_levels", "c1_corner_sym"]
STIFF_RATIOS = [1e2, 1e4]
# Below what Jacobi needs there: under the emulator Jacobi takes 67 / 95 iterations on c3_three_levels and 90 / 125 on
# c1_corner_sym at the two ratios; the multigrid preconditioner takes 5 or 6.
STIFF_MAX_ITER = 30
# MG iterations over smoothing_time / dx_finest^2 from 1e-2 to 1e4 stay at or below MG_ITER_BOUND on the fixtures with cubic
# cells: the emulator measures 1, 3, 5 and 6-7 at the four ratios (one V-cycle reduces the residual 10 to 50 fold after the
# first; BiCGStab applies two per iteration); the bound leaves one or two iterations of room.  On the fixtures with
# anisotropic cells (dx differs by a factor 2 or more between directions) a point Gauss-Seidel smoother damps the error
# poorly along the strongly coupled direction and np2 coarsens only once, so the count grows with smoothing_time there:
# 1, 3-4, 8-11, 12-16 -- still far below Jacobi's, and bounded by MG_ITER_BOUND_ANISO on that range.
ISOTROPIC = ["c1_periodic", "c1_walls", "c1_corner_sym", "c3_three_levels", "lshape", "thin"]
ANISOTROPIC = ["mixed_boxes", "np2"]
MG_ITER_BOUND = 8
MG_ITER_BOUND_ANISO = 20
SWEEP_RATIOS = [1e-2, 1e0, 1e2, 1e4]
# One V-cycle used alone as a stationary iteration, on the fixtures with cubic cells: each of 5 cycles reduces the max-norm
# residual by at least VCYCLE_FACTOR (the emulator measures at most 0.70, on the first cycle at ratio 1e4; 0.22 after it), and
# the 5 together by VCYCLE_MEAN_FACTOR^5 (the emulator's geometric means are 0.02 to 0.2).  Anisotropic cells: ratio 1 only,
# where every cycle gains 14 fold or more; at ratio >= 1e2 the V-cycle alone does not contract there (it stays a useful
# preconditioner: see the iteration counts above).
VCYCLE_FACTOR = 0.75
VCYCLE_MEAN_FACTOR = 0.3
VCYCLE_FLOOR = 1e-12


def _finest_dx2(pf):
    return float(pf.levels[-1].dx[0]) ** 2


def _run(P, pf, is_per, sym, t, pmin, pmax, precond, max_iter=0):
    H = P.Hierarchy(pf.levels, is_per, sym)
    st = P.Field(H, 1, 1)
    out = P.Field(H, 2, 1)
    st.upload_fabs(0, [[f[0] for f in lv.fabs] for lv in pf.levels])
    o = P.SmoothOpts()
    o.smoothing_time = t
    o.max_iter = max_iter
    o.precond = precond
    it, res = P.smooth(st, 0, pmin, pmax, o, out, 0, 1)
    return H, st, it, res, flat_from_fabs(out.download_fabs(0)), flat_from_fabs(out.download_fabs(1))


def check_fixture(P, name, t):
    """MG: phi within 1e-9 max|c| of the oracle, reported residual <= tol_rel, two runs bit-identical, c = Progress bit for bit"""
    from oracle.smooth_oracle import SmoothOracle
    pf, is_per, sym, S, pmin, pmax = G._inputs(name)
    H, st, it, res, c, phi = _run(P, pf, is_per, sym, t, pmin, pmax, P.PA_SMOOTH_PRECOND_MG)
    assert res <= TOL_REL and it >= 1, (it, res)
    _, _, it2, res2, c2, phi2 = _run(P, pf, is_per, sym, t, pmin, pmax, P.PA_SMOOTH_PRECOND_MG)
    assert it2 == it and res2 == res and bit_equal(phi2, phi) and bit_equal(c2, c)
    so = SmoothOracle(pf, is_per, sym)
    ref = so.solve(c, t)
    cmax = np.max(np.abs(c[so.uncovered]))
    assert np.max(np.abs(phi - ref)) <= 1e-9 * cmax, (name, t, np.max(np.abs(phi - ref)) / cmax)
    assert so.residual(c, phi, t) <= 1.01 * TOL_REL * cmax
    o = P.CurvOpts()
    o.prog_min, o.prog_max = pmin, pmax
    out = P.Field(H, 5, 1)
    P.curvature(st, 0, 0, o, out, 0)
    assert bit_equal(flat_from_fabs(out.download_fabs(0)), c)


def check_stiff(P, name, ratio):
    """at smoothing_time = ratio * dx_finest^2 Jacobi needs more than STIFF_MAX_ITER iterations (PA_ERR_NOCONV there, phi left
    as it was), MG converges within them and matches the reference solution"""
    from oracle.smooth_oracle import SmoothOracle
    from smooth_stiff_ref import stiff_solve
    pf, is_per, sym, S, pmin, pmax = G._inputs(name)
    t = ratio * _finest_dx2(pf)
    _, _, itj, _, _, _ = _run(P, pf, is_per, sym, t, pmin, pmax, P.PA_SMOOTH_PRECOND_JACOBI)
    assert itj > STIFF_MAX_ITER, itj
    with pytest.raises(P.PaError) as e:
        _run(P, pf, is_per, sym, t, pmin, pmax, P.PA_SMOOTH_PRECOND_JACOBI, max_iter=STIFF_MAX_ITER)
    assert e.value.code == P.PA_ERR_NOCONV
    _, _, it, res, c, phi = _run(P, pf, is_per, sym, t, pmin, pmax, P.PA_SMOOTH_PRECOND_MG, max_iter=STIFF_MAX_ITER)
    assert it <= MG_ITER_BOUND and res <= TOL_REL, (it, res)
    so = SmoothOracle(pf, is_per, sym)
    ref = stiff_solve(so, c, t)
    cmax = np.max(np.abs(c[so.uncovered]))
    assert np.max(np.abs(phi - ref)) <= 1e-9 * cmax, (name, ratio, np.max(np.abs(phi - ref)) / cmax)


def check_iteration_bound(P, name):
    """MG iterations stay under one bound from smoothing_time / dx_finest^2 = 1e-2 to 1e4"""
    pf, is_per, sym, S, pmin, pmax = G._inputs(name)
    its = []
    for r in SWEEP_RATIOS:
        _, _, it, res, _, _ = _run(P, pf, is_per, sym, r * _finest_dx2(pf), pmin, pmax, P.PA_SMOOTH_PRECOND_MG)
        assert res <= TOL_REL
        its.append(it)
    assert max(its) <= (MG_ITER_BOUND_ANISO if name in ANISOTROPIC else MG_ITER_BOUND), (name, its)


def vcycle(P, name, t, ncycles):
    pf, is_per, sym, S, pmin, pmax = G._inputs(name)
    H = P.Hierarchy(pf.levels, is_per, sym)
    st, out = P.Field(H, 1, 1), P.Field(H, 2, 1)
    st.upload_fabs(0, [[f[0] for f in lv.fabs] for lv in pf.levels])
    o = P.SmoothOpts()
    o.smoothing_time = t
    return P.debug_smooth_vcycle(st, 0, pmin, pmax, o, out, 0, 1, ncycles)


def check_vcycle(P, name, ratio):
    """phi <- phi + B (c - A phi): every cycle reduces the residual by VCYCLE_FACTOR and five by VCYCLE_MEAN_FACTOR^5, until the
    residual reaches the rounding floor"""
    pf, _, _, _, _, _ = G._inputs(name)
    res, nmg = vcycle(P, name, ratio * _finest_dx2(pf), 5)
    assert len(res) == 6 and nmg >= 1 and res[0] > 0.0
    for n in range(1, 6):
        if res[n - 1] > VCYCLE_FLOOR:
            assert res[n] <= VCYCLE_FACTOR * res[n - 1], (name, ratio, list(res))
    assert res[5] <= max(VCYCLE_FLOOR, VCYCLE_MEAN_FACTOR ** 5 * res[0]), (name, ratio, list(res))


def mg_levels_expected(pf):
    """the coarsening rule of level 0, restated: MG level k+1 exists while every box of level k (and the domain) has an even low
    corner and an even length of at least 4 in every direction"""
    lv = pf.levels[0]
    boxes = [(np.array(lo), np.array(hi)) for lo, hi in lv.boxes] + [(np.array(lv.domain_lo), np.array(lv.domain_hi))]
    n = 1
    while all(np.all(lo % 2 == 0) and np.all((hi - lo + 1) % 2 == 0) and np.all(hi - lo + 1 >= 4) for lo, hi in boxes):
        boxes = [(lo // 2, (hi + 1) // 2 - 1) for lo, hi in boxes]
        n += 1
    return n


def check_mg_levels(P, name, expected):
    pf, _, _, _, _, _ = G._inputs(name)
    res, nmg = vcycle(P, name, 1e-5, 0)
    assert nmg == expected == mg_levels_expected(pf), (name, nmg, expected)
    assert len(res) == 1


def check_errors(P):
    pf, is_per, sym, S, pmin, pmax = G._inputs("c1_periodic")
    for bad in (2, -1):
        with pytest.raises(P.PaError) as e:
            _run(P, pf, is_per, sym, 1e-5, pmin, pmax, bad)
        assert e.value.code == -1 and "precond" in str(e.value)
    with pytest.raises(ValueError):
        P.smooth_precond("gmres")
    pf3, is_per3, sym3, S3, pmin3, pmax3 = G._inputs("c3_three_levels")
    H = P.Hierarchy(pf3.levels, is_per3, sym3, rank=0, nranks=2)
    st, out = P.Field(H, 1, 1), P.Field(H, 2, 1)
    o = P.SmoothOpts()
    o.smoothing_time, o.precond = 1e-5, P.PA_SMOOTH_PRECOND_MG
    with pytest.raises(P.PaError) as e:
        P.smooth(st, 0, pmin3, pmax3, o, out, 0, 1)
    assert e.value.code == P.PA_ERR_UNSUPPORTED and "one rank" in str(e.value)


def check_curvature_run(P, name="c3_three_levels", t=1e-5):
    """stencilrun.CurvatureRun(smooth_precond="mg"): phi matches the oracle; an unknown name is refused"""
    from oracle.smooth_oracle import SmoothOracle
    from peleanalysis_b200.stencilrun import CurvatureRun
    pf, is_per, sym, S, pmin, pmax = G._inputs(name)
    o = P.CurvOpts()
    o.prog_min, o.prog_max = pmin, pmax
    run = CurvatureRun(P, pf, o, is_per=is_per, sym_dir=sym, do_smooth=True, smoothing_time=t, smooth_precond="mg")
    run.step()
    assert run.residual <= TOL_REL and run.iterations >= 1
    phi = flat_from_fabs(run.smoothed_progress())
    c = (S - pmin) * (1.0 / (pmax - pmin))
    so = SmoothOracle(pf, is_per, sym)
    ref = so.solve(c, t)
    cmax = np.max(np.abs(c[so.uncovered]))
    assert np.max(np.abs(phi[so.uncovered] - ref[so.uncovered])) <= 1e-9 * cmax
    with pytest.raises(ValueError):
        CurvatureRun(P, pf, o, is_per=is_per, sym_dir=sym, do_smooth=True, smooth_precond="ilu")


def check_tool(exe, tmp_path, name, monkeypatch, t=1e-5):
    """curvature3d do_smooth=1 smooth_precond=mg passes the Jacobi tool test's assertions and names the preconditioner"""
    run_tool = G.run_tool
    seen = []

    def run_mg(exe_, d, cwd, *args):
        p = run_tool(exe_, d, cwd, *args, "smooth_precond=mg")
        seen.append(p.stdout)
        return p
    monkeypatch.setattr(G, "run_tool", run_mg)
    G.check_tool(exe, tmp_path, name, t)
    assert any("precond mg" in s for s in seen)


def check_tool_bad_precond(exe, tmp_path):
    from helpers import load_golden
    from peleanalysis_b200 import plotfile
    pf, z = load_golden("c1_periodic")
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    p = G.run_tool(exe, d, str(tmp_path), "outfile=" + str(tmp_path / "K"), "do_smooth=1", "smooth_precond=ilu")
    assert p.returncode != 0 and "smooth_precond must be jacobi or mg" in p.stdout + p.stderr


# ---- on the B200 -----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("t", [1e-7, 1e-5])
@pytest.mark.parametrize("name", G.SMOOTH_FIXTURES)
def test_smooth_mg_fixture(gpu, name, t):
    check_fixture(gpu, name, t)


@pytest.mark.parametrize("ratio", STIFF_RATIOS)
@pytest.mark.parametrize("name", STIFF_CASES)
def test_smooth_mg_stiff(gpu, name, ratio):
    check_stiff(gpu, name, ratio)


@pytest.mark.parametrize("name", G.SMOOTH_FIXTURES)
def test_smooth_mg_iteration_bound(gpu, name):
    check_iteration_bound(gpu, name)


@pytest.mark.parametrize("name,ratio", [(n, r) for n in ISOTROPIC for r in (1e0, 1e2, 1e4)] + [(n, 1e0) for n in ANISOTROPIC])
def test_smooth_mg_vcycle(gpu, name, ratio):
    check_vcycle(gpu, name, ratio)


@pytest.mark.parametrize("name,expected", [("c1_periodic", 3), ("np2", 2), ("thin", 4)])
def test_smooth_mg_levels(gpu, name, expected):
    check_mg_levels(gpu, name, expected)


def test_smooth_mg_errors(gpu):
    check_errors(gpu)


def test_smooth_mg_curvature_run(gpu):
    check_curvature_run(gpu)


@pytest.mark.parametrize("t", [1e-5, 1e-3])
def test_smooth_mg_mid_size(gpu, t):
    """a 64^3 base with two refined levels: the oracle's operator confirms the residual, and phi agrees with the Jacobi-preconditioned
    solve (and, at 1e-5, with the oracle's own solve; at 1e-3, smoothing_time / dx_finest^2 = 66, it does not reach its tolerance)"""
    from oracle.smooth_oracle import SmoothOracle
    from peleanalysis_b200 import synth
    pf = synth.config3(64, 32)
    S = flat_from_fabs([[f[0] for f in lv.fabs] for lv in pf.levels])
    pmin, pmax = float(S.min()), float(S.max())
    _, _, it, res, c, phi = _run(gpu, pf, (1, 1, 1), (0, 0, 0), t, pmin, pmax, gpu.PA_SMOOTH_PRECOND_MG)
    _, _, itj, resj, _, phij = _run(gpu, pf, (1, 1, 1), (0, 0, 0), t, pmin, pmax, gpu.PA_SMOOTH_PRECOND_JACOBI)
    assert res <= TOL_REL and it <= MG_ITER_BOUND and it < itj, (it, itj)
    so = SmoothOracle(pf, (1, 1, 1), (0, 0, 0))
    cmax = np.max(np.abs(c[so.uncovered]))
    assert so.residual(c, phi, t) <= 1.01 * TOL_REL * cmax
    assert np.max(np.abs(phi - phij)) <= 1e-9 * cmax
    if t <= 1e-5:
        assert np.max(np.abs(phi - so.solve(c, t))) <= 1e-9 * cmax


@pytest.mark.parametrize("name", ["c1_periodic", "c3_three_levels", "c1_corner_sym"])
def test_curvature_executable_smooth_mg(exes, tmp_path, monkeypatch, name):
    check_tool(exes[1], tmp_path, name, monkeypatch)


def test_curvature_executable_smooth_precond_unknown(exes, tmp_path):
    check_tool_bad_precond(exes[1], tmp_path)
