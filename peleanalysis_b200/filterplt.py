"""filterPlt through the C ABI: the host-side sequence of R/Src/filterPlt.cpp:100-222 on a plotfile.Plotfile.

One Python call per C entry point (capi.py); the compute is the library's CUDA kernels (filter.cu) -- there is no CPU path.
The C++ executable peleanalysis_b200/host/filterPlt3d.b200.ex performs the same sequence on plotfiles on disk; this module
is what the parity tests and bench.py drive.  `P` is the binding module (capi), passed in so the emulated test tier can hand
in its private instance."""
from __future__ import annotations

from typing import List, Optional, Sequence

import numpy as np

from .plotfile import Level, Plotfile
from .stencilrun import download_level


def level_fgr(base_fgr: int, ratios: Sequence[int], same_fgr_all_levels: bool, lev: int) -> int:
    """filter-to-grid ratio of a level (filterPlt.cpp:141-147): the base ratio times the refinement ratios below it, so the
    absolute filter width stays the same, unless same_fgr_all_levels."""
    f = base_fgr
    if not same_fgr_all_levels:
        for l in range(1, lev + 1):
            f *= ratios[l - 1]
    return f


def rechop(P, pf: Plotfile, comps: Sequence[int], max_grid_size: int, nlev: int) -> List[Level]:
    """the plotfile's grids re-chopped to max_grid_size (BoxArray::maxSize, filterPlt.cpp:153) with the selected components"""
    out = []
    for lv in pf.levels[:nlev]:
        boxes, fabs = [], []
        have_data = len(lv.fabs) == len(lv.boxes)          # metadata-only levels (timing runs) carry no FABs
        for b, (lo, hi) in enumerate(lv.boxes):
            for clo, chi in P.boxes_max_size([(lo, hi)], max_grid_size):
                boxes.append((clo, chi))
                if have_data:
                    s = tuple(slice(clo[d] - lo[d], chi[d] - lo[d] + 1) for d in (2, 1, 0))
                    fabs.append(np.ascontiguousarray(lv.fabs[b][(comps,) + s]))
        out.append(Level(lv.domain_lo, lv.domain_hi, lv.dx, boxes, fabs))
    return out


class FilterRun:
    """Device state of one filterPlt run: hierarchy on the re-chopped grids, input field with ghost cells, output field.

    rank / nranks > 1: the re-chopped boxes of every level are spread over the ranks by pa_sfc_distribute, only this rank's
    boxes are uploaded and returned, and every fill is preceded by its slab exchange (multigpu.FillPatchExchange over the
    current torch.distributed group; `multigpu` / `wrap` let tests hand in another binding and host-memory slabs).
    out_names: the filtered variables in file order; download_level(l): this rank's share of level l in that order."""

    def __init__(self, P, pf: Plotfile, filter_type: int = 1, base_fgr: int = 2, same_fgr_all_levels: bool = False,
                 max_grid_size: int = 32, interp_type: int = 1, variables: Optional[Sequence[str]] = None,
                 max_filter_level: int = 1000, upload: bool = True, rank: int = 0, nranks: int = 1, multigpu=None, wrap=None):
        self.P = P
        self.names = list(variables) if variables else list(pf.names)
        comps = [pf.comp(n) for n in self.names]
        self.nlev = min(max_filter_level + 1, len(pf.levels))
        ratios = [(pf.levels[l].domain_hi[0] - pf.levels[l].domain_lo[0] + 1) // (pf.levels[l - 1].domain_hi[0] - pf.levels[l - 1].domain_lo[0] + 1)
                  for l in range(1, len(pf.levels))]
        self.filter_type, self.interp_type = filter_type, interp_type
        self.fgr = [level_fgr(base_fgr, ratios, same_fgr_all_levels, l) for l in range(self.nlev)]
        self.ngrow = [P.filter_weights(filter_type, f)[0] for f in self.fgr]
        self.levels = rechop(P, pf, comps, max_grid_size, self.nlev)
        self.hier = P.Hierarchy(self.levels, is_per=(0, 0, 0), sym_dir=(0, 0, 0), rank=rank, nranks=nranks, flags=P.FILTER_ONLY)
        self.ncomp = len(comps)
        self.fin = P.Field(self.hier, self.ncomp, max(self.ngrow))
        self.fout = P.Field(self.hier, self.ncomp, 0)
        self.out_names = self.names
        self.outputs = [(self.fout, c) for c in range(self.ncomp)]
        self.exchanges = []
        if nranks > 1:
            if multigpu is None:
                from . import multigpu
            kw = {} if wrap is None else {"wrap": wrap}
            self.exchanges = [multigpu.FillPatchExchange(self.fin, self.ncomp, l, self.ngrow[l], interp_type, **kw) for l in range(self.nlev)]
        if upload:
            for c in range(self.ncomp):
                self.fin.upload_fabs(c, [[f[c] for f in lv.fabs] for lv in self.levels])

    def step(self) -> None:
        """[exchange +] ghost fill + filter of every level (filterPlt.cpp:166-221), asynchronous on the library stream"""
        P = self.P
        for l in range(self.nlev):
            if self.exchanges:
                self.exchanges[l].run(0)
            P.fill_patch(self.fin, 0, self.ncomp, l, self.ngrow[l], self.interp_type)
            P.filter_level(self.fin, 0, self.fout, 0, self.ncomp, l, self.filter_type, self.fgr[l])

    def result(self) -> List[List[Optional[np.ndarray]]]:
        """per level, per box: [ncomp][nz][ny][nx] (None for boxes of other ranks)"""
        per_comp = [self.fout.download_fabs(c) for c in range(self.ncomp)]
        return [[np.stack([per_comp[c][l][b] for c in range(self.ncomp)]) if per_comp[0][l][b] is not None else None
                 for b in range(len(lv.boxes))] for l, lv in enumerate(self.levels)]

    def download_level(self, lev: int) -> np.ndarray:
        return download_level(self.P, self.hier, self.outputs, lev)

    def grown_input(self, lev: int, box: int, comp: int) -> np.ndarray:
        """the input FAB with the field's ghost width; only the level's own ngrow layers are filled"""
        return self.fin.download_grown(lev, box, comp)

    def cells(self) -> int:
        return sum(lv.ncells for lv in self.levels)


def filter_plotfile(P, pf: Plotfile, **kw):
    run = FilterRun(P, pf, **kw)
    run.step()
    P.sync()
    return run.names, [(lv.boxes, fabs) for lv, fabs in zip(run.levels, run.result())], run
