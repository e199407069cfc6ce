"""GPU (-m gpu): the C++ drop-in executables (peleanalysis_b200/host) end to end through plotfiles: same keys, same
output names, data bit-identical to the compiled reference's golden vectors; when oracle/_ref travelled to the box,
also compared live with AMReX's own fcompare against the reference executable's output."""
import os
import subprocess

import numpy as np
import pytest

from helpers import bit_equal, load_golden, max_rel
from oracle import oracle as O
from peleanalysis_b200 import plotfile

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "peleanalysis_b200", "host")


@pytest.fixture(scope="module")
def exes(gpu):
    # one make at a time: with pytest-xdist a second worker's relink would otherwise hit "Text file busy" on an
    # executable the first worker is already running
    import fcntl
    with open(os.path.join(HOST, ".build.lock"), "w") as lk:
        fcntl.flock(lk, fcntl.LOCK_EX)
        subprocess.check_call(["make", "-s", "-C", HOST])
    return os.path.join(HOST, "grad3d.b200.ex"), os.path.join(HOST, "curvature3d.b200.ex"), os.path.join(HOST, "filterPlt3d.b200.ex")


def _flat(pf, name):
    c = pf.comp(name)
    return np.concatenate([f[c].ravel() for l in pf.levels for f in l.fabs])


def _run(exe, *args, cwd):
    p = subprocess.run([exe, *args], capture_output=True, text=True, cwd=cwd)
    assert p.returncode == 0, p.stdout + p.stderr
    return p.stdout


@pytest.mark.parametrize("name", ["c1_periodic", "c1_corner_sym", "c3_three_levels", "ratio4"])
def test_grad_executable(exes, tmp_path, name):
    pf, z = load_golden(name)
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    per = " ".join(str(int(v)) for v in z["is_per"])
    sym = " ".join(str(int(v)) for v in z["sym_dir"])
    out = _run(exes[0], "infile=" + d, "gradVar=temp", "is_per=" + per, "sym_dir=" + sym, cwd=str(tmp_path))
    assert "Periodicity assumed for this case: " + per in out
    r = plotfile.read_plotfile(str(tmp_path / "plt_gt"))          # default outfile = <root>_gt in the cwd
    assert r.names == ["temp", "temp_gx", "temp_gy", "temp_gz", "||gradtemp||"]
    assert bit_equal(_flat(r, "temp"), z["in_temp"])
    for k, n in zip(["gx", "gy", "gz", "mag"], r.names[1:]):
        assert bit_equal(_flat(r, n), z["grad_" + k]), (name, n)
    if O.have_ref():
        O.run_ref("grad", d, str(tmp_path / "ref_gt"), gradVar="temp", is_per=list(z["is_per"]), sym_dir=list(z["sym_dir"]))
        p = subprocess.run([O.ref_exe("fcompare.ref.ex"), str(tmp_path / "plt_gt"), str(tmp_path / "ref_gt")], capture_output=True, text=True)
        assert "PLOTFILE AGREE" in p.stdout, p.stdout[-1500:]


def test_grad_executable_aux_and_inputs_file(exes, tmp_path):
    pf, z = load_golden("c1_options")
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    inp = tmp_path / "inputs.grad"
    inp.write_text("infile = %s\noutfile = %s   # comment\ngradVar = temp\nfinestLevel = 0\nis_per = 1 1 0\nAux_Variables = Y_CH4 x_velocity\n" % (d, tmp_path / "o"))
    _run(exes[0], str(inp), cwd=str(tmp_path))
    r = plotfile.read_plotfile(str(tmp_path / "o"))
    assert r.names == ["temp", "Y_CH4", "x_velocity", "temp_gx", "temp_gy", "temp_gz", "||gradtemp||"]
    assert len(r.levels) == 1
    n0 = pf.levels[0].ncells
    assert bit_equal(_flat(r, "Y_CH4"), z["in_Y_CH4"][:n0])
    # unknown aux variable aborts like the reference
    p = subprocess.run([exes[0], "infile=" + d, "Aux_Variables=nope"], capture_output=True, text=True, cwd=str(tmp_path))
    assert p.returncode != 0 and "Unknown auxiliary variable name: nope" in p.stderr


@pytest.mark.parametrize("name", ["c1_periodic", "c3_threshold", "c1_options"])
def test_curvature_executable(exes, tmp_path, name):
    check_curvature_executable(exes, tmp_path, name)


def check_curvature_executable(exes, tmp_path, name, skip=()):
    pf, z = load_golden(name)
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    kw = [str(s) for s in z["curv_opts"]]
    per = " ".join(str(int(v)) for v in z["is_per"])
    _run(exes[1], "infile=" + d, "progressName=temp", "is_per=" + per, "outfile=" + str(tmp_path / "K"), *kw, cwd=str(tmp_path))
    r = plotfile.read_plotfile(str(tmp_path / "K"))
    for key in z.files:
        if not key.startswith("curv_") or key == "curv_opts":
            continue
        n = key[5:]
        if n in skip:
            continue
        got = _flat(r, n)
        if n.startswith("GaussianCurvature"):
            assert max_rel(got, z[key]) <= 1e-12
        else:
            assert bit_equal(got, z[key]), (name, n)
    assert "SmoothedProgress" in r.names and "GaussianCurvature_temp" in r.names


def _ngpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_ngpus() < 2, reason="needs two GPUs in one box (gpurun --gpus 2)")
@pytest.mark.parametrize("name", ["c3_three_levels", "mixed_boxes"])
def test_executables_on_two_gpus(exes, tmp_path, name):
    """ngpus=2: one host thread per GPU in one process (host/multi_gpu.hpp) -- peer links over NVLink by pointer, slab copies
    between the two GPUs, one Cell_D file per GPU; same bits as the golden vectors of the compiled reference."""
    pf, z = load_golden(name)
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    per = " ".join(str(int(v)) for v in z["is_per"])
    sym = " ".join(str(int(v)) for v in z["sym_dir"])
    _run(exes[0], "infile=" + d, "gradVar=temp", "is_per=" + per, "sym_dir=" + sym, "ngpus=2", cwd=str(tmp_path))
    r = plotfile.read_plotfile(str(tmp_path / "plt_gt"))
    for k, n in zip(["gx", "gy", "gz", "mag"], r.names[1:]):
        assert bit_equal(_flat(r, n), z["grad_" + k]), (name, n)
    _run(exes[1], "infile=" + d, "progressName=temp", "is_per=" + per, "sym_dir=" + sym, "ngpus=2", "outfile=" + str(tmp_path / "K"), cwd=str(tmp_path))
    r = plotfile.read_plotfile(str(tmp_path / "K"))
    for n in ["Progress", "MeanCurvature_temp", "FlameNormalX_temp", "FlameNormalY_temp", "FlameNormalZ_temp"]:
        assert bit_equal(_flat(r, n), z["curv_" + n]), (name, n)


# ---- source-level drop-in: the reference tools themselves, operator block replaced by the C-ABI calls ---------------------
def _amrex_exes():
    e = (O.ref_exe("grad3d.b200amrex.ex"), O.ref_exe("curvature3d.b200amrex.ex"))
    return e if all(os.path.exists(x) for x in e) else None


@pytest.fixture(scope="module")
def amrex_exes(gpu):
    e = _amrex_exes()
    if e is None:
        pytest.skip("oracle/_ref/*.b200amrex.ex not built (oracle/build_ref.py builds them where /root/reference exists)")
    return e


@pytest.mark.parametrize("name", ["c1_periodic", "c1_corner_sym", "c3_three_levels"])
def test_amrex_linked_grad(amrex_exes, tmp_path, name):
    """grad.cpp of the reference with lines 171-236 replaced by INTEGRATION.md's block (peleanalysis_b200/host/amrex_glue),
    linked against host-only AMReX + libpelestencil_b200.so: AMReX reads and writes the plotfile, the library computes."""
    test_grad_executable(amrex_exes, tmp_path, name)


@pytest.mark.parametrize("name", ["c1_periodic", "c3_threshold", "c1_options"])
def test_amrex_linked_curvature(amrex_exes, tmp_path, name):
    check_curvature_executable(amrex_exes, tmp_path, name, skip=("SmoothedProgress",))


def test_amrex_linked_curvature_do_smooth(amrex_exes, tmp_path):
    """do_smooth=1: AMReX's own MLMG solve smooths the progress variable on the host (the reference's lines 328-406, untouched),
    the stencil path runs on the smoothed field.  Same solve, same bits in -> AMReX's fcompare agrees with the reference tool."""
    pf, z = load_golden("c1_periodic")
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    per = " ".join(str(int(v)) for v in z["is_per"])
    args = ["infile=" + d, "progressName=temp", "is_per=" + per, "do_smooth=1", "smoothing_time=1.0e-5"]
    env = dict(os.environ, OMP_NUM_THREADS="1")
    p = subprocess.run([amrex_exes[1], *args, "outfile=" + str(tmp_path / "K")], capture_output=True, text=True, cwd=str(tmp_path), env=env)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    q = subprocess.run([O.ref_exe("curvature3d.ref.ex"), *args, "outfile=" + str(tmp_path / "Kref")], capture_output=True, text=True, cwd=str(tmp_path), env=env)
    assert q.returncode == 0, q.stdout[-2000:] + q.stderr[-2000:]
    a, b = plotfile.read_plotfile(str(tmp_path / "K")), plotfile.read_plotfile(str(tmp_path / "Kref"))
    for n in ["Progress", "SmoothedProgress", "MeanCurvature_temp", "FlameNormalX_temp", "FlameNormalY_temp", "FlameNormalZ_temp"]:
        assert bit_equal(_flat(a, n), _flat(b, n)), n


# ---- BASELINE-size parity: the C restatement of the reference's arithmetic (oracle/, bit-exact against the reference's
#      golden vectors in tests/test_oracle_golden.py) on the same hierarchy; also the compiled reference itself where it was built
def _big_tmp():
    import tempfile
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    return tempfile.TemporaryDirectory(prefix="pa_full_", dir=base)


@pytest.mark.parametrize("config", ["configs1_512", "configs4_small_boxes"])
def test_full_size_grad_vs_reference_executable(exes, config):
    """BASELINE configs[1] (uniform 512^3 in 128^3 boxes, one of its variables) and configs[4] (4 levels, ratios 2/4/2,
    128^3 base, 16^3 boxes) at FULL size: every output bit of the B200 tool equals the oracle's; where the reference tool
    was built, it reads the same plotfile and AMReX's own fcompare must print PLOTFILE AGREE."""
    from peleanalysis_b200 import synth
    if config == "configs1_512":
        pf, var = synth.make_hierarchy(512, [], [], 128, ("temp",)), "temp"
    else:
        pf = synth.config5(128, 16, 2)
        var = pf.names[1]
    with _big_tmp() as tmp:
        d = os.path.join(tmp, "plt")
        plotfile.write_plotfile(d, pf)
        OH = O.OracleHier(pf)
        want = OH.grad(OH.flatten(pf.comp(var)))
        del pf
        _run(exes[0], "infile=" + d, "gradVar=" + var, "outfile=" + os.path.join(tmp, "b200"), cwd=tmp)
        for c, n in enumerate([var + "_gx", var + "_gy", var + "_gz", "||grad%s||" % var]):
            got = _flat(plotfile.read_plotfile(os.path.join(tmp, "b200"), comps=[n]), n)
            assert bit_equal(got, want[c]), (config, n, max_rel(got, want[c]))
        del want
        if O.have_ref():
            O.run_ref("grad", d, os.path.join(tmp, "ref"), gradVar=var)
            p = subprocess.run([O.ref_exe("fcompare.ref.ex"), os.path.join(tmp, "b200"), os.path.join(tmp, "ref")], capture_output=True, text=True)
            assert "PLOTFILE AGREE" in p.stdout, p.stdout[-1500:]


def test_full_size_curvature_vs_reference_executable(exes):
    """BASELINE configs[2] at full size (3 levels, 256^3 base, ratio 2, 64^3 boxes): every output the reference initialises
    (it leaves SmoothedProgress and, without do_gaussCurv, GaussianCurvature unset) bit for bit, against the oracle and,
    where it was built, the reference tool."""
    from peleanalysis_b200 import synth
    pf = synth.config3(256, 64)
    names = ["Progress", "MeanCurvature_temp", "FlameNormalX_temp", "FlameNormalY_temp", "FlameNormalZ_temp"]
    with _big_tmp() as tmp:
        d = os.path.join(tmp, "plt")
        plotfile.write_plotfile(d, pf)
        OH = O.OracleHier(pf)
        pmin, pmax = plotfile.file_min_max(d, "temp", len(pf.levels))      # the tool's default progMin / progMax
        want = OH.curvature(OH.flatten(pf.comp("temp")), pmin, pmax)
        del pf
        _run(exes[1], "infile=" + d, "progressName=temp", "outfile=" + os.path.join(tmp, "b200"), cwd=tmp)
        a = plotfile.read_plotfile(os.path.join(tmp, "b200"), comps=names)
        for c, n in enumerate(names):
            assert bit_equal(_flat(a, n), want[c]), (n, max_rel(_flat(a, n), want[c]))
        if O.have_ref():
            O.run_ref("curvature", d, os.path.join(tmp, "ref"), progressName="temp")
            b = plotfile.read_plotfile(os.path.join(tmp, "ref"), comps=names)
            for n in names:
                assert bit_equal(_flat(a, n), _flat(b, n)), n


@pytest.mark.parametrize("name", ["filter_c1", "filter_c1_corner_gauss", "filter_c3", "filter_c3_subset", "filter_c3_pc_samefgr", "filter_ratio4"])
def test_filter_executable(exes, tmp_path, name):
    """filterPlt3d.b200.ex: the reference tool's keys, output name (<root>_filtered in the working directory), re-chopped
    output grids and variable names; data bit-identical to the reference's golden vectors; AMReX's fcompare agrees with the
    reference executable's plotfile."""
    pf, z = load_golden(name)
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    opts = [str(s) for s in z["opts"]]
    out = _run(exes[2], "infile=" + d, *opts, cwd=str(tmp_path))
    assert "FillPatching data..." in out and "Filtering data..." in out
    r = plotfile.read_plotfile(str(tmp_path / "plt_filtered"))
    assert r.names == [str(n) for n in z["out_names"]]
    want_boxes = [tuple(int(v) for v in b) for b in z["out_boxes"]]
    assert [tuple(lo) + tuple(hi) for l in r.levels for lo, hi in l.boxes] == want_boxes
    for n in r.names:
        assert bit_equal(_flat(r, n), z["out_" + n]), (name, n)
    if O.have_ref() and os.path.exists(O.ref_exe("filterPlt3d.ref.ex")):
        os.makedirs(str(tmp_path / "ref"))
        kv = dict(s.split("=", 1) for s in opts)
        O.run_ref("filterPlt", d, str(tmp_path / "ref" / "plt_filtered"), **kv)
        p = subprocess.run([O.ref_exe("fcompare.ref.ex"), str(tmp_path / "plt_filtered"), str(tmp_path / "ref" / "plt_filtered")], capture_output=True, text=True)
        assert "PLOTFILE AGREE" in p.stdout, p.stdout[-1500:]


def test_filter_executable_errors(exes, tmp_path):
    pf, _ = load_golden("filter_c1")
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    p = subprocess.run([exes[2], "infile=" + d, "variables=nope"], capture_output=True, text=True, cwd=str(tmp_path))
    assert p.returncode != 0 and "Variable 'nope' not found in file" in p.stderr
    p = subprocess.run([exes[2], "infile=" + d, "base_fgr=3"], capture_output=True, text=True, cwd=str(tmp_path))
    assert p.returncode != 0 and "even" in p.stderr


def test_grad_executable_several_files_per_level(exes, tmp_path, monkeypatch):
    """the writer's multi-file layout (one writer thread per box range, as VisMF with several writers): forced here, chosen
    automatically for large levels; AMReX's own reader (fcompare) must accept it"""
    monkeypatch.setenv("PA_PLT_NFILES", "3")
    test_grad_executable(exes, tmp_path, "c3_three_levels")
    files = sorted(os.listdir(str(tmp_path / "plt_gt" / "Level_0")))
    assert [f for f in files if f.startswith("Cell_D_")] == ["Cell_D_00000", "Cell_D_00001", "Cell_D_00002"]
