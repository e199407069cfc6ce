"""CPU: plotfile reader/writer round trip and header layout."""
import numpy as np
import pytest

from peleanalysis_b200 import plotfile, synth


def test_roundtrip(tmp_path):
    pf = synth.config1(16, 8, names=("temp", "Y_CH4"))
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf, nfiles_per_level=3)
    r = plotfile.read_plotfile(d)
    assert r.names == ["temp", "Y_CH4"] and r.ref_ratio == [2]
    for a, b in zip(pf.levels, r.levels):
        assert a.boxes == b.boxes and a.dx == b.dx
        for fa, fb in zip(a.fabs, b.fabs):
            assert np.array_equal(fa, fb)
    only = plotfile.read_plotfile(d, comps=["Y_CH4"], finest_level=0)
    assert len(only.levels) == 1 and np.array_equal(only.levels[0].fabs[3][0], pf.levels[0].fabs[3][1])
    lo, hi = plotfile.file_min_max(d, "temp", 2)
    assert lo == min(f[0].min() for l in pf.levels for f in l.fabs)
    assert hi == max(f[0].max() for l in pf.levels for f in l.fabs)


def test_existing_directory_is_renamed_like_the_reference(tmp_path):
    pf = synth.config1(16, 8)
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    plotfile.write_plotfile(d, pf)
    olds = [p.name for p in tmp_path.iterdir() if p.name.startswith("plt.old.")]
    assert len(olds) == 1


def _rewrite_fabs(d, nlev, dtype, grow=0):
    """Rewrite every Cell_D file of a plotfile in another on-disk real format (what `fab.format = NATIVE_32` / a big-endian
    machine / a MultiFab written with ghost cells produce) and fix the offsets in Cell_H."""
    import os
    import re
    nb = np.dtype(dtype).itemsize
    fmt = "(64 11 52 0 1 12 0 1023)" if nb == 8 else "(32 8 23 0 1 9 0 127)"
    order = " ".join(str(i) for i in (range(nb, 0, -1) if np.dtype(dtype).byteorder in "<=|" else range(1, nb + 1)))
    for lev in range(nlev):
        ldir = os.path.join(d, "Level_%d" % lev)
        hpath = os.path.join(ldir, "Cell_H")
        L = open(hpath).read().split("\n")
        nboxes = int(re.findall(r"\d+", L[4])[0])
        p = 5 + nboxes + 1
        nf = int(L[p])
        entries = [L[p + 1 + i].split() for i in range(nf)]
        out = {}
        for i, (tag, fn, off) in enumerate(entries):
            with open(os.path.join(ldir, fn), "rb") as f:
                f.seek(int(off))
                head = f.readline().decode()
                v = [int(x) for x in re.findall(r"-?\d+", head[head.find("((", 5):])]
                lo, hi, nc = v[0:3], v[3:6], v[9]
                n = [hi[k] - lo[k] + 1 for k in range(3)]
                a = np.fromfile(f, "<f8", nc * n[0] * n[1] * n[2]).reshape(nc, n[2], n[1], n[0])
            if grow:
                a = np.pad(a, ((0, 0),) + ((grow, grow),) * 3, constant_values=-12345.0)
                lo, hi = [x - grow for x in lo], [x + grow for x in hi]
            buf = out.setdefault(fn, bytearray())
            entries[i][2] = str(len(buf))
            buf += ("FAB ((8, %s),(%d, (%s)))((%d,%d,%d) (%d,%d,%d) (0,0,0)) %d\n" % (fmt, nb, order, *lo, *hi, nc)).encode()
            buf += a.astype(dtype).tobytes()
        for fn, buf in out.items():
            with open(os.path.join(ldir, fn), "wb") as f:
                f.write(buf)
        for i, e in enumerate(entries):
            L[p + 1 + i] = " ".join(e)
        open(hpath, "w").write("\n".join(L))


@pytest.mark.parametrize("dtype,grow", [("<f4", 0), (">f8", 0), (">f4", 1), ("<f8", 2)])
def test_other_on_disk_formats(tmp_path, dtype, grow):
    """NATIVE_32 / big-endian / grown FABs are converted like AmrData does (RealDescriptor), never misread: the Python reader,
    the C++ reader (through the emulated grad executable) and -- where oracle/_ref exists -- AMReX's own reader in the
    reference executable agree."""
    import os
    import subprocess
    import sys
    pf = synth.config1(16, 8, names=("temp", "Y_CH4"))
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    _rewrite_fabs(d, 2, dtype, grow)
    r = plotfile.read_plotfile(d)
    for a, b in zip(pf.levels, r.levels):
        for fa, fb in zip(a.fabs, b.fabs):
            assert np.array_equal(fa.astype(dtype).astype("<f8"), fb)
    only = plotfile.read_plotfile(d, comps=["Y_CH4"])
    assert np.array_equal(only.levels[1].fabs[2][0], pf.levels[1].fabs[2][1].astype(dtype).astype("<f8"))
    # the C++ reader of the host shells, against AMReX's reader in the reference tool
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
    import build_emu
    from oracle import oracle as O
    lib = build_emu.build()
    out = os.path.dirname(lib)
    host = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "peleanalysis_b200", "host")
    exe = os.path.join(out, "grad3d.fmt.ex")
    srcs = [os.path.join(host, "grad_main.cpp"), os.path.join(host, "plotfile.cpp")]
    import fcntl
    with open(os.path.join(out, ".exe_build.lock"), "w") as lk:      # one build at a time (pytest-xdist workers share the directory)
        fcntl.flock(lk, fcntl.LOCK_EX)
        if not os.path.exists(exe) or any(os.path.getmtime(s) > os.path.getmtime(exe) for s in srcs + [lib]):
            subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", *srcs, "-o", exe + ".tmp", "-L", out, "-lpelestencil_emu", "-Wl,-rpath," + out])
            os.replace(exe + ".tmp", exe)
    env = dict(os.environ, PA_NORMAL_MATH="fast", CUEMU_SEED="0")
    p = subprocess.run([exe, "infile=" + d, "gradVar=temp", "outfile=" + str(tmp_path / "g")], capture_output=True, text=True, env=env, cwd=str(tmp_path))
    assert p.returncode == 0, p.stdout + p.stderr
    g = plotfile.read_plotfile(str(tmp_path / "g"))
    got = np.concatenate([f[g.comp("temp")].ravel() for l in g.levels for f in l.fabs])
    want = np.concatenate([f[0].astype(dtype).astype("<f8").ravel() for l in pf.levels for f in l.fabs])
    assert np.array_equal(got, want)
    # mgtools reads through plotfile.read_boxes: the executable's plotfile, value for value
    import importlib.util
    from peleanalysis_b200 import capi as product_capi, mgtools
    spec = importlib.util.spec_from_file_location("capi_emulated_formats", product_capi.__file__)
    emu = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(emu)
    emu.LIB_PATH = lib
    mgtools.run("grad", ["infile=" + d, "gradVar=temp", "outfile=" + str(tmp_path / "m")], capi=emu, device=0)
    m = plotfile.read_plotfile(str(tmp_path / "m"))
    assert m.names == g.names
    for n in g.names:
        assert np.array_equal(np.concatenate([f[m.comp(n)].ravel() for l in m.levels for f in l.fabs]),
                              np.concatenate([f[g.comp(n)].ravel() for l in g.levels for f in l.fabs])), n
    if O.have_ref():
        O.run_ref("grad", d, str(tmp_path / "gref"), gradVar="temp")
        q = subprocess.run([O.ref_exe("fcompare.ref.ex"), str(tmp_path / "g"), str(tmp_path / "gref")], capture_output=True, text=True)
        assert "PLOTFILE AGREE" in q.stdout, q.stdout[-1500:]


def test_unknown_real_format_is_rejected(tmp_path):
    import os
    pf = synth.config1(16, 8)
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    fn = os.path.join(d, "Level_0", "Cell_D_00000")
    raw = open(fn, "rb").read()
    open(fn, "wb").write(raw.replace(b"(64 11 52 0 1 12 0 1023)", b"(64 15 48 0 1 16 0 16383)", 1))
    with pytest.raises(ValueError) as e:
        plotfile.read_plotfile(d)
    assert "unsupported real format" in str(e.value)
