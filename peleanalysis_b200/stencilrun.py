"""grad and curvature through the C ABI on a plotfile.Plotfile, on one rank or with the boxes spread over several ranks.

The counterpart of filterplt.FilterRun for the two stencil tools: one Python call per C entry point (capi.py), the compute
is the library's CUDA kernels -- there is no CPU path.  `P` is the binding module (capi), passed in so the emulated test
tier can hand in its private instance.

rank / nranks > 1: the boxes of every level are spread over the ranks by pa_sfc_distribute (capi.Hierarchy), only this
rank's boxes are uploaded and returned, and every ghost fill is preceded by its exchange over the current torch.distributed
group: the width-1 ghost sources owned by another rank than the box they fill (same-level neighbours and the coarse cells
of coarse-fine faces) move as packed slabs (multigpu.SlabExchange, hier.cpp: build_exchange).  Nothing is peer-mapped.
On one rank the calls are exactly capi.grad / capi.curvature."""
from __future__ import annotations

from typing import List, Optional, Sequence

import numpy as np

from .plotfile import Plotfile


class _Run:
    def __init__(self, P, pf: Plotfile, is_per, sym_dir, rank: int, nranks: int, multigpu, wrap):
        self.P, self.pf = P, pf
        self.levels = pf.levels
        self.nlev = len(pf.levels)
        self.hier = P.Hierarchy(pf.levels, is_per, sym_dir, rank=rank, nranks=nranks)
        self.rank, self.nranks = rank, nranks
        if nranks > 1 and multigpu is None:
            from . import multigpu
        self.mg = multigpu
        self.kw = {} if wrap is None else {"wrap": wrap}

    def _upload(self, field, names: Sequence[str]) -> None:
        for c, n in enumerate(names):
            k = self.pf.comp(n)
            field.upload_fabs(c, [[f[k] for f in lv.fabs] for lv in self.levels])

    def _result(self, field, ncomp: int) -> List[List[Optional[np.ndarray]]]:
        """per level, per box: [ncomp][nz][ny][nx] (None for boxes of other ranks)"""
        per_comp = [field.download_fabs(c) for c in range(ncomp)]
        return [[np.stack([per_comp[c][l][b] for c in range(ncomp)]) if per_comp[0][l][b] is not None else None
                 for b in range(len(lv.boxes))] for l, lv in enumerate(self.levels)]

    def cells(self) -> int:
        return self.hier.num_cells


class GradRun(_Run):
    """grad.cpp:151-236 on the variables `names`: input field with one ghost layer, output [gx, gy, gz, |grad|] per variable."""

    def __init__(self, P, pf: Plotfile, names: Optional[Sequence[str]] = None, is_per=(1, 1, 1), sym_dir=(0, 0, 0),
                 upload: bool = True, rank: int = 0, nranks: int = 1, multigpu=None, wrap=None):
        super().__init__(P, pf, is_per, sym_dir, rank, nranks, multigpu, wrap)
        self.names = list(names) if names else [pf.names[0]]
        self.nvar = len(self.names)
        self.fin = P.Field(self.hier, self.nvar, 1)
        self.fout = P.Field(self.hier, 4 * self.nvar, 0)
        self.exchange = self.mg.SlabExchange(self.fin, self.nvar, **self.kw) if nranks > 1 else None
        if upload:
            self._upload(self.fin, self.names)

    def step(self) -> None:
        """[exchange +] ghost fill + gradient of every level, asynchronous on the library stream"""
        if self.exchange is not None:
            self.exchange.run(0)
        self.P.grad(self.fin, 0, self.nvar, self.fout, 0)

    def result(self):
        return self._result(self.fout, 4 * self.nvar)


class CurvatureRun(_Run):
    """curvature.cpp on the progress variable `progress` (and the velocities, when the options need them): state field
    [S, (u, v, w)] with one ghost layer, output in the library's order (Progress, K, n, [Kg], [SR], [ROST], [VN])."""

    VEL = ("x_velocity", "y_velocity", "z_velocity")

    def __init__(self, P, pf: Plotfile, opts, progress: str = "temp", is_per=(1, 1, 1), sym_dir=(0, 0, 0), upload: bool = True,
                 rank: int = 0, nranks: int = 1, multigpu=None, wrap=None):
        super().__init__(P, pf, is_per, sym_dir, rank, nranks, multigpu, wrap)
        self.opts = opts
        self.names = [progress] + (list(self.VEL) if (opts.do_strain or opts.do_velnormal) else [])
        self.state = P.Field(self.hier, len(self.names), 1)
        self.nout = P.curvature_num_outputs(opts)
        self.fout = P.Field(self.hier, self.nout, 1)
        comp_vel = 1 if len(self.names) > 1 else 0
        self.op = self.mg.Curvature(self.state, 0, opts, self.fout, 0, comp_vel=comp_vel, **self.kw) if nranks > 1 else None
        if upload:
            self._upload(self.state, self.names)

    def step(self) -> None:
        """every step of the tool with the exchange each one needs in front of it, asynchronous on the library stream"""
        if self.op is not None:
            self.op.run()
        else:
            self.P.curvature(self.state, 0, 1 if len(self.names) > 1 else 0, self.opts, self.fout, 0)

    def result(self):
        return self._result(self.fout, self.nout)
