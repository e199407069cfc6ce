"""B200: curvature's do_smooth (R/Src/curvature.cpp:328-406) through pa_smooth -- the composite implicit-diffusion solve
phi - smoothing_time * div(grad phi) = c against the SciPy oracle (oracle/smooth_oracle.py), its error codes, and the
curvature3d.b200.ex do_smooth=1 path.  The check bodies take the binding module P so that tests/test_emu_smooth.py runs them
under the CPU emulation of the kernels."""
import os
import subprocess

import numpy as np
import pytest

from helpers import bit_equal, flat_from_fabs, load_golden
from cases import CASES
from peleanalysis_b200 import plotfile
from test_gpu_tools import exes  # noqa: F401  (fixture: the built host executables)

pytestmark = pytest.mark.gpu

SMOOTH_FIXTURES = ["c1_periodic", "c1_walls", "c1_corner_sym", "c3_three_levels", "lshape", "mixed_boxes", "np2", "thin"]
TOL_REL = 1e-10


def _inputs(name):
    pf, z = load_golden(name)
    _, is_per, sym, _, _ = CASES[name]
    S = flat_from_fabs([[f[0] for f in lv.fabs] for lv in pf.levels])
    return pf, is_per, sym, S, float(S.min()), float(S.max())


def _smooth_run(P, pf, is_per, sym, t, pmin, pmax, max_iter=0):
    H = P.Hierarchy(pf.levels, is_per, sym)
    st = P.Field(H, 1, 1)
    out = P.Field(H, 2, 1)
    st.upload_fabs(0, [[f[0] for f in lv.fabs] for lv in pf.levels])
    o = P.SmoothOpts()
    o.smoothing_time = t
    o.max_iter = max_iter
    it, res = P.smooth(st, 0, pmin, pmax, o, out, 0, 1)
    return H, st, it, res, flat_from_fabs(out.download_fabs(0)), flat_from_fabs(out.download_fabs(1))


def check_fixture(P, name, t):
    """phi within 1e-9 max|c| of the oracle, reported residual <= tol_rel, two runs bit-identical, c bit-identical to
    pa_curvature's Progress"""
    from oracle.smooth_oracle import SmoothOracle
    pf, is_per, sym, S, pmin, pmax = _inputs(name)
    H, st, it, res, c, phi = _smooth_run(P, pf, is_per, sym, t, pmin, pmax)
    assert res <= TOL_REL and it >= 1, (it, res)
    _, _, it2, res2, c2, phi2 = _smooth_run(P, pf, is_per, sym, t, pmin, pmax)
    assert it2 == it and res2 == res and bit_equal(phi2, phi) and bit_equal(c2, c)
    so = SmoothOracle(pf, is_per, sym)
    ref = so.solve(c, t)
    cmax = np.max(np.abs(c[so.uncovered]))
    assert np.max(np.abs(phi - ref)) <= 1e-9 * cmax, (name, t, np.max(np.abs(phi - ref)) / cmax)
    assert so.residual(c, phi, t) <= 1.01 * TOL_REL * cmax
    # Progress of the curvature path, same normalisation: the same bits
    o = P.CurvOpts()
    o.prog_min, o.prog_max = pmin, pmax
    out = P.Field(H, 5, 1)
    P.curvature(st, 0, 0, o, out, 0)
    assert bit_equal(flat_from_fabs(out.download_fabs(0)), c)


def check_zero_time(P, name="c3_three_levels"):
    pf, is_per, sym, S, pmin, pmax = _inputs(name)
    _, _, it, res, c, phi = _smooth_run(P, pf, is_per, sym, 0.0, pmin, pmax)
    assert it == 0 and res == 0.0 and bit_equal(phi, c)


def check_errors(P):
    pf, is_per, sym, S, pmin, pmax = _inputs("c1_periodic")
    o = P.SmoothOpts()
    o.smoothing_time = 1e-5
    # refinement ratio 4
    pf4, z4 = load_golden("ratio4")
    H4 = P.Hierarchy(pf4.levels, (1, 1, 1), (0, 0, 0))
    f4, o4 = P.Field(H4, 1, 1), P.Field(H4, 2, 1)
    with pytest.raises(P.PaError) as e:
        P.smooth(f4, 0, 0.0, 1.0, o, o4, 0, 1)
    assert e.value.code == P.PA_ERR_UNSUPPORTED and "ratio 2" in str(e.value)
    # negative smoothing time
    H = P.Hierarchy(pf.levels, is_per, sym)
    st, out = P.Field(H, 1, 1), P.Field(H, 2, 1)
    st.upload_fabs(0, [[f[0] for f in lv.fabs] for lv in pf.levels])
    on = P.SmoothOpts()
    on.smoothing_time = -1e-5
    with pytest.raises(P.PaError) as e:
        P.smooth(st, 0, pmin, pmax, on, out, 0, 1)
    assert e.value.code == -1
    # one iteration is not enough at t = 1e-5
    o1 = P.SmoothOpts()
    o1.smoothing_time, o1.max_iter = 1e-5, 1
    with pytest.raises(P.PaError) as e:
        P.smooth(st, 0, pmin, pmax, o1, out, 0, 1)
    assert e.value.code == P.PA_ERR_NOCONV and "not converged" in str(e.value)


def check_two_ranks(P):
    pf, is_per, sym, S, pmin, pmax = _inputs("c3_three_levels")
    H = P.Hierarchy(pf.levels, is_per, sym, rank=0, nranks=2)
    st, out = P.Field(H, 1, 1), P.Field(H, 2, 1)
    o = P.SmoothOpts()
    o.smoothing_time = 1e-5
    with pytest.raises(P.PaError) as e:
        P.smooth(st, 0, pmin, pmax, o, out, 0, 1)
    assert e.value.code == P.PA_ERR_UNSUPPORTED and "one rank" in str(e.value)


def run_tool(exe, d, cwd, *args):
    p = subprocess.run([exe, "infile=" + d, "progressName=temp", *args], capture_output=True, text=True, cwd=cwd)
    return p


def check_tool(exe, tmp_path, name, t=1e-5):
    """curvature3d do_smooth=1: SmoothedProgress = the oracle's phi to tolerance; MeanCurvature / FlameNormal* = the C oracle's
    curvature of the tool's own SmoothedProgress with prog_min = 0, prog_max = 1, bit for bit; Progress = the do_smooth=0 run's"""
    from oracle import oracle as O
    from oracle.smooth_oracle import SmoothOracle
    pf, is_per, sym, S, pmin, pmax = _inputs(name)
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    per = "is_per=" + " ".join(str(int(v)) for v in is_per)
    sd = "sym_dir=" + " ".join(str(int(v)) for v in sym)
    p = run_tool(exe, d, str(tmp_path), per, sd, "outfile=" + str(tmp_path / "K1"), "do_smooth=1", "smoothing_time=%r" % t, "verbose=1")
    assert p.returncode == 0, p.stdout + p.stderr
    assert "do_smooth: smoothing_time" in p.stdout
    p0 = run_tool(exe, d, str(tmp_path), per, sd, "outfile=" + str(tmp_path / "K0"))
    assert p0.returncode == 0, p0.stdout + p0.stderr
    r1, r0 = plotfile.read_plotfile(str(tmp_path / "K1")), plotfile.read_plotfile(str(tmp_path / "K0"))

    def flat(r, n):
        k = r.comp(n)
        return flat_from_fabs([[f[k] for f in lv.fabs] for lv in r.levels])
    c = flat(r1, "Progress")
    assert bit_equal(c, flat(r0, "Progress"))
    phi = flat(r1, "SmoothedProgress")
    so = SmoothOracle(pf, is_per, sym)
    ref = so.solve(c, t)
    cmax = np.max(np.abs(c[so.uncovered]))
    assert np.max(np.abs(phi - ref)) <= 1e-9 * cmax
    oh = O.OracleHier(pf, is_per, sym)
    cur = oh.curvature(phi, 0.0, 1.0)
    for k, n in enumerate(["MeanCurvature_temp", "FlameNormalX_temp", "FlameNormalY_temp", "FlameNormalZ_temp"]):
        assert bit_equal(flat(r1, n), cur[k + 1]), n
    # the unsmoothed run still writes zeros there
    assert not np.any(flat(r0, "SmoothedProgress"))


def check_tool_multi_gpu_abort(exe, tmp_path, env=None):
    pf, z = load_golden("c1_periodic")
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    p = subprocess.run([exe, "infile=" + d, "do_smooth=1", "ngpus=2"], capture_output=True, text=True, cwd=str(tmp_path),
                       env=dict(os.environ, **(env or {})))
    assert p.returncode != 0 and "do_smooth=1 runs on one GPU only" in p.stdout + p.stderr


# ---- on the B200 -----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("t", [1e-7, 1e-5])
@pytest.mark.parametrize("name", SMOOTH_FIXTURES)
def test_smooth_fixture(gpu, name, t):
    check_fixture(gpu, name, t)


def test_smooth_zero_time(gpu):
    check_zero_time(gpu)


def test_smooth_errors(gpu):
    check_errors(gpu)


def test_smooth_two_ranks(gpu):
    check_two_ranks(gpu)


def test_smooth_mid_size(gpu):
    """a 64^3 base with two refined levels against the oracle"""
    from oracle.smooth_oracle import SmoothOracle
    from peleanalysis_b200 import synth
    pf = synth.config3(64, 32)
    S = flat_from_fabs([[f[0] for f in lv.fabs] for lv in pf.levels])
    pmin, pmax = float(S.min()), float(S.max())
    t = 1e-5
    _, _, it, res, c, phi = _smooth_run(gpu, pf, (1, 1, 1), (0, 0, 0), t, pmin, pmax)
    assert res <= TOL_REL
    so = SmoothOracle(pf, (1, 1, 1), (0, 0, 0))
    ref = so.solve(c, t)
    cmax = np.max(np.abs(c[so.uncovered]))
    assert np.max(np.abs(phi - ref)) <= 1e-9 * cmax


@pytest.mark.parametrize("name", ["c1_periodic", "c3_three_levels", "c1_corner_sym"])
def test_curvature_executable_do_smooth(exes, tmp_path, name):
    check_tool(exes[1], tmp_path, name)


def test_curvature_executable_do_smooth_refuses_several_gpus(exes, tmp_path):
    check_tool_multi_gpu_abort(exes[1], tmp_path)


@pytest.mark.parametrize("name", ["c1_periodic", "c3_three_levels"])
def test_do_smooth_against_reference(exes, tmp_path, name):
    """curvature3d.b200.ex against the compiled reference tool, do_smooth=1 smoothing_time=1e-5: SmoothedProgress agrees to
    1e-8 relative (an iterative solve: the last bits depend on the iteration history).  Skips where the reference is not built."""
    from oracle import oracle as O
    if not O.have_ref():
        pytest.skip("oracle/_ref/curvature3d.ref.ex not built (oracle/build_ref.py builds it where the reference sources exist)")
    pf, is_per, sym, S, pmin, pmax = _inputs(name)
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    per = " ".join(str(int(v)) for v in is_per)
    p = run_tool(exes[1], d, str(tmp_path), "is_per=" + per, "outfile=" + str(tmp_path / "B"), "do_smooth=1", "smoothing_time=1e-5")
    assert p.returncode == 0, p.stdout + p.stderr
    O.run_ref("curvature", d, str(tmp_path / "R"), progressName="temp", is_per=per, do_smooth=1, smoothing_time=1e-5)
    b, r = plotfile.read_plotfile(str(tmp_path / "B")), plotfile.read_plotfile(str(tmp_path / "R"))

    def flat(x):
        k = x.comp("SmoothedProgress")
        return flat_from_fabs([[f[k] for f in lv.fabs] for lv in x.levels])
    fb, fr = flat(b), flat(r)
    assert np.max(np.abs(fb - fr)) <= 1e-8 * np.max(np.abs(fr))
