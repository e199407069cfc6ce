"""AMReX plotfile (HyperCLaw-V1.1 / VisMF v1) reader and writer in NumPy.

Host-side format code shared by the Python tool drivers, tests and bench.  The format follows
what the reference reads and writes through AMReX:
  Header              WriteGenericPlotfileHeader  (amrex/Src/Base/AMReX_PlotFileUtil.cpp:73-155)
  Level_L/Cell_H      VisMF::Header operator<<    (amrex/Src/Base/AMReX_VisMF.cpp:274-336)
  Level_L/Cell_D_nnnnn  per FAB: ASCII "FAB (realdescriptor)(box) ncomp\\n" + raw little-endian
                      doubles, i fastest, component slowest (FABio_binary, AMReX_FArrayBox.cpp:905-912)
Arrays are held as numpy [ncomp, nz, ny, nx] (C order), which is byte-identical to the FAB order.
"""
from __future__ import annotations

import os
import re
import shutil
import time
from dataclasses import dataclass, field
from typing import List, Sequence

import numpy as np

_FAB_DESC = "FAB ((8, (64 11 52 0 1 12 0 1023)),(8, (8 7 6 5 4 3 2 1)))"


@dataclass
class Level:
    """One AMR level: index-space domain, cell size and the FABs (valid region only)."""
    domain_lo: tuple
    domain_hi: tuple
    dx: tuple
    boxes: List[tuple]            # [(lo(3), hi(3)), ...] inclusive cell indices
    fabs: List[np.ndarray] = field(default_factory=list)   # [ncomp, nz, ny, nx] float64 each

    @property
    def ncells(self) -> int:
        return int(sum(np.prod([h - l + 1 for l, h in zip(lo, hi)]) for lo, hi in self.boxes))


@dataclass
class Plotfile:
    names: List[str]
    prob_lo: tuple
    prob_hi: tuple
    ref_ratio: List[int]          # header line (one int per coarse level)
    levels: List[Level]
    time: float = 0.0
    coord: int = 0

    @property
    def finest_level(self) -> int:
        return len(self.levels) - 1

    def comp(self, name: str) -> int:
        return self.names.index(name)


def _fmt17(x: float) -> str:
    """C++ ostream << double with precision(17) in default (%g-like) float format."""
    return "%.17g" % x


def _box_str(lo, hi) -> str:
    return "((%d,%d,%d) (%d,%d,%d) (0,0,0))" % (*lo, *hi)


def unique_old_name(path: str) -> str:
    """AMReX UtilCreateCleanDirectory renames an existing directory to <dir>.old.<unique>
    (amrex/Src/Base/AMReX_Utility.cpp:160-172)."""
    return "%s.old.%d" % (path, int(time.time() * 1e6) % 10**10)


def create_plotfile_dirs(path: str, nlev: int, clean: str = "rename") -> None:
    """`path` and its Level_l directories.  clean='rename' mimics the reference (an existing directory is renamed to
    <path>.old.<unique>); clean='remove' deletes it (benchmarks)."""
    if os.path.lexists(path):
        if clean == "remove":
            shutil.rmtree(path)
        else:
            os.rename(path, unique_old_name(path))
    os.makedirs(path)
    for il in range(nlev):
        os.makedirs(os.path.join(path, "Level_%d" % il))


def write_fab_file(path: str, lev: int, fname: str, level: Level, box_ids: Sequence[int], fabs: Sequence[np.ndarray]) -> list:
    """Level_<lev>/<fname> holding the FABs of the boxes box_ids of `level`; fabs[i] is the data of box box_ids[i], component
    first ([ncomp, nz, ny, nx] or [ncomp, cells]).  Returns one record (lev, box, fname, offset, mins, maxs) per box for
    write_metadata.  No file is created for no boxes."""
    records = []
    if not len(box_ids):
        return records
    with open(os.path.join(path, "Level_%d" % lev, fname), "wb") as f:
        for b, fab in zip(box_ids, fabs):
            lo, hi = level.boxes[b]
            n = (hi[2] - lo[2] + 1, hi[1] - lo[1] + 1, hi[0] - lo[0] + 1)
            assert fab.shape[1:] in (n, (n[0] * n[1] * n[2],)), (fname, b, fab.shape)
            a = np.ascontiguousarray(fab, dtype="<f8").reshape(len(fab), -1)
            off = f.tell()
            f.write(("%s%s %d\n" % (_FAB_DESC, _box_str(lo, hi), a.shape[0])).encode())
            f.write(a.tobytes())
            records.append((lev, b, fname, off, a.min(axis=1).tolist(), a.max(axis=1).tolist()))
    return records


def write_metadata(path: str, pf: Plotfile, records: Sequence[tuple]) -> None:
    """Header (WriteGenericPlotfileHeader, AMReX_PlotFileUtil.cpp:73-155) and every Level_l/Cell_H (VisMF header v1) of `pf`
    (its FABs are not used) from the write_fab_file records of all its boxes."""
    nlev = len(pf.levels)
    with open(os.path.join(path, "Header"), "w") as h:
        h.write("HyperCLaw-V1.1\n%d\n" % len(pf.names))
        for n in pf.names:
            h.write(n + "\n")
        h.write("3\n%s\n%d\n" % (_fmt17(pf.time), nlev - 1))
        h.write("".join(_fmt17(v) + " " for v in pf.prob_lo) + "\n")
        h.write("".join(_fmt17(v) + " " for v in pf.prob_hi) + "\n")
        h.write("".join("%d " % r for r in pf.ref_ratio[: nlev - 1]) + "\n")
        h.write("".join(_box_str(l.domain_lo, l.domain_hi) + " " for l in pf.levels) + "\n")
        h.write("".join("0 " for _ in pf.levels) + "\n")
        for l in pf.levels:
            h.write("".join(_fmt17(v) + " " for v in l.dx) + "\n")
        h.write("%d\n0\n" % pf.coord)
        for il, l in enumerate(pf.levels):
            h.write("%d %d %s\n0\n" % (il, len(l.boxes), _fmt17(pf.time)))
            for lo, hi in l.boxes:
                for d in range(3):
                    # RealBox(b shifted by -domain_lo, dx, prob_lo): lo = plo + dx*lo ; hi = plo + dx*(hi+1)
                    a = pf.prob_lo[d] + l.dx[d] * (lo[d] - l.domain_lo[d])
                    b = pf.prob_lo[d] + l.dx[d] * (hi[d] - l.domain_lo[d] + 1)
                    h.write("%s %s\n" % (_fmt17(a), _fmt17(b)))
            h.write("Level_%d/Cell\n" % il)
    ncomp = len(pf.names)
    for il, l in enumerate(pf.levels):
        nb = len(l.boxes)
        rec = {r[1]: r for r in records if r[0] == il}
        assert len(rec) == nb and all(len(r[4]) == ncomp for r in rec.values()), "level %d: %d of %d boxes written" % (il, len(rec), nb)
        with open(os.path.join(path, "Level_%d" % il, "Cell_H"), "w") as c:
            c.write("1\n1\n%d\n0\n" % ncomp)
            c.write("(%d 0\n" % nb)
            for lo, hi in l.boxes:
                c.write(_box_str(lo, hi) + "\n")
            c.write(")\n")
            c.write("%d\n" % nb)
            for b in range(nb):
                c.write("FabOnDisk: %s %d\n" % rec[b][2:4])
            c.write("\n")
            for k in (4, 5):                                   # mins, maxs
                c.write("%d,%d\n" % (nb, ncomp))
                for b in range(nb):
                    c.write("".join("%.17e," % v for v in rec[b][k]) + "\n")
                c.write("\n")


def write_plotfile(path: str, pf: Plotfile, nfiles_per_level: int = 1, clean: str = "rename") -> None:
    """Write `pf` to directory `path`, box b of a level to file Cell_D_<b mod nfiles_per_level>.  clean: as create_plotfile_dirs."""
    create_plotfile_dirs(path, len(pf.levels), clean)
    records = []
    for il, l in enumerate(pf.levels):
        nf = max(1, min(nfiles_per_level, len(l.boxes)))
        for i in range(nf):
            ids = range(i, len(l.boxes), nf)
            records += write_fab_file(path, il, "Cell_D_%05d" % i, l, ids, [l.fabs[b] for b in ids])
    write_metadata(path, pf, records)


def _ints(s: str) -> List[int]:
    return [int(x) for x in re.findall(r"-?\d+", s)]


def read_header(path: str):
    with open(os.path.join(path, "Header")) as f:
        L = f.read().split("\n")
    p = 0
    version = L[p]; p += 1
    nvar = int(L[p]); p += 1
    names = [L[p + i].strip() for i in range(nvar)]; p += nvar
    dim = int(L[p]); p += 1
    if dim != 3:
        raise ValueError("only 3-D plotfiles are supported (got dim=%d)" % dim)
    tm = float(L[p]); p += 1
    finest = int(L[p]); p += 1
    prob_lo = tuple(float(x) for x in L[p].split()); p += 1
    prob_hi = tuple(float(x) for x in L[p].split()); p += 1
    ref_ratio = _ints(L[p]); p += 1
    d = _ints(L[p]); p += 1
    domains = [(tuple(d[9 * i: 9 * i + 3]), tuple(d[9 * i + 3: 9 * i + 6])) for i in range(finest + 1)]
    p += 1  # level steps
    dxs = []
    for _ in range(finest + 1):
        dxs.append(tuple(float(x) for x in L[p].split())); p += 1
    coord = int(L[p]); p += 1
    p += 1  # "0"
    paths = []
    for lev in range(finest + 1):
        t = L[p].split(); p += 1
        ng = int(t[1])
        p += 1  # step
        p += 3 * ng
        paths.append(L[p].strip()); p += 1
    return dict(version=version, names=names, time=tm, finest=finest, prob_lo=prob_lo, prob_hi=prob_hi,
                ref_ratio=ref_ratio, domains=domains, dx=dxs, coord=coord, paths=paths)


def read_cell_h(path: str, relpath: str):
    with open(os.path.join(path, relpath + "_H")) as f:
        L = f.read().split("\n")
    vers = int(L[0]); ncomp = int(L[2])
    nb = int(L[4].strip("(").split()[0])
    boxes = []
    for i in range(nb):
        v = _ints(L[5 + i])
        boxes.append((tuple(v[0:3]), tuple(v[3:6])))
    p = 5 + nb + 1
    nf = int(L[p]); p += 1
    fod = []
    for i in range(nf):
        t = L[p + i].split()
        fod.append((t[1], int(t[2])))
    p += nf
    mins = maxs = None
    if vers == 1:
        tabs = []
        for _ in range(2):
            while L[p].strip() == "":
                p += 1
            n, m = (int(x) for x in L[p].split(",")); p += 1
            tab = np.array([[float(x) for x in L[p + i].rstrip(",").split(",")] for i in range(n)]).reshape(n, m)
            p += n
            tabs.append(tab)
        mins, maxs = tabs
    return ncomp, boxes, fod, mins, maxs


def parse_fab_header(line: str, where: str = "?"):
    """`FAB ((n, (fmt...)),(m, (byte order...))) ((lo) (hi) (type)) ncomp` -> (numpy dtype, lo, hi, ncomp).  IEEE double or
    single, little- or big-endian (what AmrData converts through RealDescriptor, AMReX_FabConv.cpp); the FAB's own box may be
    the valid box grown by ghost cells.  Anything else raises -- a plotfile is never silently misread."""
    import re
    if not line.startswith("FAB"):
        raise ValueError("not a FAB header in %s: %r" % (where, line[:60]))
    box_at = line.find("((", 5)
    d = [int(x) for x in re.findall(r"-?\d+", line[:box_at])]
    b = [int(x) for x in re.findall(r"-?\d+", line[box_at:])]
    if box_at < 0 or len(b) != 10 or len(d) < 2 or len(d) != 2 + d[0] + d[1 + d[0]]:
        raise ValueError("malformed FAB header in %s: %r" % (where, line))
    fmt, order = d[1:1 + d[0]], d[2 + d[0]:]
    kinds = {(64, 11, 52, 0, 1, 12, 0, 1023): 8, (32, 8, 23, 0, 1, 9, 0, 127): 4}
    nbytes = kinds.get(tuple(fmt))
    if nbytes is None or len(order) != nbytes:
        raise ValueError("unsupported real format in %s (only IEEE double / single): %r" % (where, line[:box_at]))
    if order == list(range(nbytes, 0, -1)):
        dt = "<f%d" % nbytes
    elif order == list(range(1, nbytes + 1)):
        dt = ">f%d" % nbytes
    else:
        raise ValueError("unsupported byte order in %s: %r" % (where, line[:box_at]))
    if b[6:9] != [0, 0, 0]:
        raise ValueError("not a cell-centred FAB in %s" % where)
    return dt, tuple(b[0:3]), tuple(b[3:6]), b[9]


def read_boxes(path: str, lev: int, box_ids: Sequence[int], comp_ids: Sequence[int]) -> List[np.ndarray]:
    """Components comp_ids of the boxes box_ids of level lev: one float64 [len(comp_ids), nz, ny, nx] array per box (its valid
    cells).  Only those FABs and components are read; consecutive components are one read per FAB."""
    hd = read_header(path)
    _, boxes, fod, _, _ = read_cell_h(path, hd["paths"][lev])
    ldir = os.path.dirname(os.path.join(path, hd["paths"][lev]))
    comp_ids = list(comp_ids)
    one_read = bool(comp_ids) and comp_ids == list(range(comp_ids[0], comp_ids[0] + len(comp_ids)))
    out = []
    for b in box_ids:
        (lo, hi), (fn, off) = boxes[b], fod[b]
        with open(os.path.join(ldir, fn), "rb") as f:
            f.seek(off)
            dt, flo, fhi, fnc = parse_fab_header(f.readline().decode("ascii", "replace"), fn)
            base = f.tell()
            if any(flo[d] > lo[d] or fhi[d] < hi[d] for d in range(3)) or max(comp_ids, default=-1) >= fnc:
                raise ValueError("FAB in %s does not cover box %s / components %s" % (fn, (lo, hi), comp_ids))
            m = [fhi[d] - flo[d] + 1 for d in range(3)]
            npts = m[0] * m[1] * m[2]
            sl = tuple(slice(lo[d] - flo[d], hi[d] - flo[d] + 1) for d in (2, 1, 0))
            if one_read:
                f.seek(base + np.dtype(dt).itemsize * npts * comp_ids[0])
                a = np.fromfile(f, dt, npts * len(comp_ids)).reshape(len(comp_ids), m[2], m[1], m[0])[(slice(None),) + sl].astype("<f8")
            else:
                a = np.empty((len(comp_ids), hi[2] - lo[2] + 1, hi[1] - lo[1] + 1, hi[0] - lo[0] + 1))
                for k, c in enumerate(comp_ids):
                    f.seek(base + np.dtype(dt).itemsize * npts * c)
                    a[k] = np.fromfile(f, dt, npts).reshape(m[2], m[1], m[0])[sl]
        out.append(a)
    return out


def read_plotfile(path: str, comps: Sequence[str] | None = None, finest_level: int | None = None,
                  load_data: bool = True) -> Plotfile:
    """Read a plotfile.  comps=None reads every component; otherwise only the named ones, in that order.  load_data=False
    reads the metadata only (levels without FABs)."""
    hd = read_header(path)
    nlev = hd["finest"] + 1 if finest_level is None else min(finest_level, hd["finest"]) + 1
    names = hd["names"] if comps is None else list(comps)
    idx = [hd["names"].index(n) for n in names]
    levels = []
    for lev in range(nlev):
        _, boxes, _, _, _ = read_cell_h(path, hd["paths"][lev])
        fabs = read_boxes(path, lev, range(len(boxes)), idx) if load_data else []
        dlo, dhi = hd["domains"][lev]
        levels.append(Level(dlo, dhi, hd["dx"][lev], boxes, fabs))
    return Plotfile(names, hd["prob_lo"], hd["prob_hi"], hd["ref_ratio"][: nlev - 1], levels, hd["time"], hd["coord"])


def file_min_max(path: str, name: str, nlev: int):
    """min/max of a component over levels from the Cell_H per-FAB tables
    (what AmrData::MinMax over the whole domain returns, amrex/Src/Extern/amrdata/AMReX_AmrData.cpp:1702-1880)."""
    hd = read_header(path)
    c = hd["names"].index(name)
    lo, hi = 1.0e20, -1.0e20
    for lev in range(nlev):
        _, _, _, mins, maxs = read_cell_h(path, hd["paths"][lev])
        lo = min(lo, float(mins[:, c].min()))
        hi = max(hi, float(maxs[:, c].max()))
    return lo, hi
