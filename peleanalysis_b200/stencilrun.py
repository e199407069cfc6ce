"""grad and curvature through the C ABI on a plotfile.Plotfile, on one rank or with the boxes spread over several ranks.

The counterpart of filterplt.FilterRun for the two stencil tools: one Python call per C entry point (capi.py), the compute
is the library's CUDA kernels -- there is no CPU path.  `P` is the binding module (capi), passed in so the emulated test
tier can hand in its private instance.

rank / nranks > 1: the boxes of every level are spread over the ranks by pa_sfc_distribute (capi.Hierarchy), only this
rank's boxes are uploaded and returned, and every ghost fill is preceded by its exchange over the current torch.distributed
group: the width-1 ghost sources owned by another rank than the box they fill (same-level neighbours and the coarse cells
of coarse-fine faces) move as packed slabs (multigpu.SlabExchange, hier.cpp: build_exchange).  Nothing is peer-mapped
unless peer_links=True: then the hierarchy has PEER_LINKS, every rank maps the others' field slabs (CUDA IPC), and ghost
cells behind a neighbour link are read in place -- the caller must barrier after the upload, and after step() before a
field is freed.  On one rank the calls are exactly capi.grad / capi.curvature.

out_names are the computed outputs' plotfile names in file order; download_level(l) returns this rank's share of level l
in that order."""
from __future__ import annotations

from typing import List, Optional, Sequence

import numpy as np

from .plotfile import Plotfile


def download_level(P, hier, outputs, lev: int) -> np.ndarray:
    """[len(outputs)][this rank's cells of level lev, box after box]: row k is component outputs[k] = (field, comp), zeros
    where outputs[k] is None"""
    out = np.zeros((len(outputs), hier.local_cells[lev]))
    for k, src in enumerate(outputs):
        if src is not None:
            src[0].download_level(lev, src[1], out[k])
            P.sync()
    return out


def upload_device(hier, field, comp: int, arrays_per_level, nghost: int = 0) -> None:
    """arrays_per_level[l]: one CUDA array per box this rank owns on level l (hier.local_boxes[l] order), [nz][ny][nx] or a
    FAB [ncomp][nz][ny][nx] whose component 0 is taken (pick another by slicing), each holding its box grown by nghost cells"""
    for l, arrays in enumerate(arrays_per_level):
        if hier.local_boxes[l] or len(arrays):
            field.upload_level_device(l, comp, arrays, nghost)


def _torch_empty(shape):
    import torch
    return torch.empty(shape, dtype=torch.float64, device="cuda")


def result_device(hier, levels, outputs, alloc=None):
    """per level, per box: a torch CUDA tensor [len(outputs)][nz][ny][nx] (None for boxes of other ranks); row k is
    component outputs[k] = (field, comp), zeros where outputs[k] is None.  Written on the library stream.  alloc(shape) may
    supply other CUDA arrays (sliceable along the first axis, with zero_() on a row)."""
    alloc = alloc or _torch_empty
    res = []
    for l, lv in enumerate(levels):
        row: List[Optional[object]] = [None] * len(lv.boxes)
        loc = hier.local_boxes[l]
        for b in loc:
            lo, hi = lv.boxes[b]
            row[b] = alloc((len(outputs), hi[2] - lo[2] + 1, hi[1] - lo[1] + 1, hi[0] - lo[0] + 1))
        k = 0
        while loc and k < len(outputs):
            if outputs[k] is None:
                for b in loc:
                    row[b][k].zero_()
                k += 1
                continue
            f, c = outputs[k]
            n = 1                  # one call per run of consecutive components of one field
            while k + n < len(outputs) and outputs[k + n] is not None and outputs[k + n][0] is f and outputs[k + n][1] == c + n:
                n += 1
            f.download_level_device(l, c, [row[b][k:k + n] for b in loc], ncomp=n)
            k += n
        res.append(row)
    return res


class _Run:
    def __init__(self, P, pf: Plotfile, is_per, sym_dir, rank: int, nranks: int, multigpu, wrap, peer_links: bool):
        self.P, self.pf = P, pf
        self.levels = pf.levels
        self.nlev = len(pf.levels)
        self.hier = P.Hierarchy(pf.levels, is_per, sym_dir, rank=rank, nranks=nranks, flags=P.PEER_LINKS if peer_links else 0)
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

    def download_level(self, lev: int) -> np.ndarray:
        return download_level(self.P, self.hier, self.outputs, lev)

    def upload_device(self, name: str, arrays_per_level, nghost: int = 0) -> None:
        """input variable `name` from device memory: per level, one CUDA array per box this rank owns (see
        stencilrun.upload_device); no host copy.  Asynchronous on the library stream."""
        if name not in self.names:
            raise ValueError("%r is not an input of this run (%s)" % (name, ", ".join(self.names)))
        upload_device(self.hier, self._input, self.names.index(name), arrays_per_level, nghost)

    def result_device(self, alloc=None):
        """per level, per box: torch CUDA tensor [len(out_names)][nz][ny][nx] in out_names order (zeros in the slots the
        tool does not write; None for boxes of other ranks); no host copy.  Enqueued on the library stream."""
        return result_device(self.hier, self.levels, self.outputs, alloc)

    def cells(self) -> int:
        return self.hier.num_cells


class GradRun(_Run):
    """grad.cpp:151-236 on the variables `names`: input field with one ghost layer, output [gx, gy, gz, |grad|] per variable."""

    def __init__(self, P, pf: Plotfile, names: Optional[Sequence[str]] = None, is_per=(1, 1, 1), sym_dir=(0, 0, 0),
                 upload: bool = True, rank: int = 0, nranks: int = 1, multigpu=None, wrap=None, peer_links: bool = False):
        super().__init__(P, pf, is_per, sym_dir, rank, nranks, multigpu, wrap, peer_links)
        self.names = list(names) if names else [pf.names[0]]
        self.nvar = len(self.names)
        self.fin = P.Field(self.hier, self.nvar, 1)
        self.fout = P.Field(self.hier, 4 * self.nvar, 0)
        self.out_names = [s for v in self.names for s in (v + "_gx", v + "_gy", v + "_gz", "||grad" + v + "||")]
        self.outputs = [(self.fout, k) for k in range(4 * self.nvar)]
        self._input = self.fin
        if peer_links and nranks > 1:
            self.mg.map_peers(self.fin)
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
    [S, (u, v, w)] with one ghost layer, output in the library's order (Progress, K, n, [Kg], [SR], [ROST], [VN]).

    do_smooth (one rank only, curvature.cpp:328-406): the progress variable c is first smoothed by one implicit diffusion
    step of `smoothing_time` (capi.smooth) and the curvature runs on the smoothed phi with prog_min = 0, prog_max = 1.
    smooth_precond picks the solve's preconditioner: "jacobi" (default) or "mg" (a multigrid V-cycle).
    Progress stays c; smoothed_progress() returns phi; `iterations` / `residual` report the last solve.

    The file order of the outputs (curvature.cpp:163-224) has SmoothedProgress and GaussianCurvature slots even when their
    options are off; the reference never writes them then, so download_level returns zeros there."""

    VEL = ("x_velocity", "y_velocity", "z_velocity")

    def __init__(self, P, pf: Plotfile, opts, progress: str = "temp", is_per=(1, 1, 1), sym_dir=(0, 0, 0), upload: bool = True,
                 rank: int = 0, nranks: int = 1, multigpu=None, wrap=None, do_smooth: bool = False, smoothing_time: float = 1.0e-7,
                 smooth_precond: str = "jacobi", peer_links: bool = False):
        precond = P.smooth_precond(smooth_precond)
        if do_smooth and nranks > 1:
            raise ValueError("do_smooth runs on one rank only: the smoothing solve has no multi-rank path")
        super().__init__(P, pf, is_per, sym_dir, rank, nranks, multigpu, wrap, peer_links)
        self.opts = opts
        self.names = [progress] + (list(self.VEL) if (opts.do_strain or opts.do_velnormal) else [])
        self.do_smooth = bool(do_smooth)
        self.iterations, self.residual = 0, 0.0
        nst = len(self.names)
        self.comp_c, self.comp_phi = nst, nst + 1
        if self.do_smooth:
            self.sopts = P.SmoothOpts()
            self.sopts.smoothing_time = smoothing_time
            self.sopts.precond = precond
            self.opts_phi = P.CurvOpts.from_buffer_copy(opts)
            self.opts_phi.prog_min, self.opts_phi.prog_max = 0.0, 1.0
        self.state = P.Field(self.hier, nst + 2 if self.do_smooth else nst, 1)
        self._input = self.state
        self.nout = P.curvature_num_outputs(opts)
        self.fout = P.Field(self.hier, self.nout, 1)
        v = progress
        self.out_names = (["Progress", "SmoothedProgress", "MeanCurvature_" + v] + ["FlameNormal%s_%s" % (a, v) for a in "XYZ"]
                          + ["GaussianCurvature_" + v])
        if opts.do_strain:
            self.out_names.append("StrainRate_" + v)
            if opts.get_strain_tensor:
                self.out_names += ["ROST_dU%sd%s" % (a, b) for a in "xyz" for b in "xyz"]
        if opts.do_velnormal:
            self.out_names.append("VelFlameNormal")
        # the library's order is the file's without SmoothedProgress, and without GaussianCurvature unless do_gauss
        lib = [n for k, n in enumerate(self.out_names) if k != 1 and (k != 6 or opts.do_gauss)]
        src = {n: (self.fout, c) for c, n in enumerate(lib)}
        if self.do_smooth:                       # the curvature's Progress is phi; the tool's Progress is c
            src["SmoothedProgress"], src["Progress"] = src["Progress"], (self.state, self.comp_c)
        self.outputs = [src.get(n) for n in self.out_names]
        comp_vel = 1 if len(self.names) > 1 else 0
        self.op = self.mg.Curvature(self.state, 0, opts, self.fout, 0, comp_vel=comp_vel, **self.kw) if nranks > 1 else None
        if upload:
            self._upload(self.state, self.names)

    def step(self) -> None:
        """every step of the tool with the exchange each one needs in front of it, asynchronous on the library stream"""
        comp_vel = 1 if len(self.names) > 1 else 0
        if self.op is not None:
            self.op.run()
        elif self.do_smooth:
            self.iterations, self.residual = self.P.smooth(self.state, 0, self.opts.prog_min, self.opts.prog_max, self.sopts,
                                                           self.state, self.comp_c, self.comp_phi)
            self.P.curvature(self.state, self.comp_phi, comp_vel, self.opts_phi, self.fout, 0)
        else:
            self.P.curvature(self.state, 0, comp_vel, self.opts, self.fout, 0)

    def result(self):
        res = self._result(self.fout, self.nout)
        if self.do_smooth:                       # the curvature's Progress is phi; the tool's Progress is c
            c = self.state.download_fabs(self.comp_c)
            for l, lv in enumerate(res):
                for b, a in enumerate(lv):
                    if a is not None:
                        a[0] = c[l][b]
        return res

    def smoothed_progress(self):
        """per level, per box: phi [nz][ny][nx] (do_smooth only)"""
        if not self.do_smooth:
            raise ValueError("smoothed_progress() needs do_smooth=True")
        return self.fout.download_fabs(0)
