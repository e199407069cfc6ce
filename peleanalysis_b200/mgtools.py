"""grad / curvature / filterPlt on a plotfile with one process per GPU -- the multi-GPU form of the drop-in executables.

    python -m peleanalysis_b200.mgtools grad      infile=plt00100 [gradVar=temp] [Aux_Variables=a b] [finestLevel=N]
                                                  [is_per=1 1 1] [sym_dir=0 0 0] [outfile=name]
    python -m peleanalysis_b200.mgtools curvature infile=plt00100 [progressName=temp] [progMin=.. progMax=..] [useFileMinMax=1]
                                                  [threshold_prog=0 threshold_value=1e-4] [do_gaussCurv=0] [do_strain=0]
                                                  [getStrainTensor=0] [do_velnormal=0] [Aux_Variables=..] [is_per=..] [sym_dir=..]
    python -m peleanalysis_b200.mgtools filter    infile=plt00100 [variables=a b] [max_filter_level=N] [filter_type=1] [base_fgr=2]
                                                  [same_fgr_all_levels=0] [max_grid_size=32] [interp_type=1]
    python -m torch.distributed.run --nproc-per-node 8 -m peleanalysis_b200.mgtools grad infile=... [transport=peer|slab]
    python -m torch.distributed.run --nproc-per-node 8 -m peleanalysis_b200.mgtools grad infiles=plt00100 plt00200 ... [keys]

infiles= processes a series of plotfiles in one process per rank, so `import torch` and the CUDA context are paid once: at
world size W, rank r takes files r, r+W, ... and runs each as the world-size-1 run of that file on its own GPU (do_smooth
included), with no communication except a final barrier.  Every other key applies to each file; each output has the name a
single run writes by default.  infiles cannot be combined with infile, outfile or transport.

Same keys, same output variable names and the same plotfile format as R/Src/grad.cpp / curvature.cpp / filterPlt.cpp (and
as the C++ shells in host/).  filter spreads the boxes re-chopped to max_grid_size over the ranks; the FillPatch sources of
other ranks move as packed slabs (multigpu.FillPatchExchange).  What an MPI build of the reference does, rank by rank, is
done here process by process, in one per-file body for the three tools: the keys become a run object (stencilrun.GradRun /
CurvatureRun, filterplt.FilterRun) on the plotfile's metadata, which owns the boxes the SFC distribution gives this rank and
does the C-ABI calls on its GPU (cross-rank ghost cells through peer links over NVLink or NCCL slab exchange, multigpu.py);
every rank reads only its boxes from disk (plotfile.read_boxes), writes them to its own Level_l/Cell_D_<rank> file
(plotfile.write_fab_file), and rank 0 writes Header and Cell_H from the gathered per-box (file, offset, min, max) records
(plotfile.write_metadata) -- the layout VisMF produces with one file per rank (AMReX_VisMF.cpp:905-1005).  No compute
happens in Python.
"""
from __future__ import annotations

import os
import sys
from typing import Dict, List, Sequence

import numpy as np

from . import filterplt, plotfile, stencilrun


# ---------------------------------------------------------------------------------------------------------------
def parse_args(argv: Sequence[str]) -> Dict[str, List[str]]:
    """key=value [value ...] tokens, or one inputs file first (amrex::ParmParse conventions: '#' starts a comment)."""
    toks: List[str] = []
    if argv and "=" not in argv[0] and os.path.isfile(argv[0]):
        for line in open(argv[0]):
            toks += line.split("#", 1)[0].replace("=", " = ").split()
        argv = argv[1:]
    for a in argv:
        toks += a.replace("=", " = ").split()
    out: Dict[str, List[str]] = {}
    key = None
    i = 0
    while i < len(toks):
        if i + 1 < len(toks) and toks[i + 1] == "=":
            key = toks[i]
            out[key] = []
            i += 2
        else:
            if key is None:
                raise SystemExit("cannot parse argument '%s'" % toks[i])
            out[key].append(toks[i])
            i += 1
    return out


def _get(pp, key, default, conv=str):
    return conv(pp[key][0]) if key in pp and pp[key] else default


def _ints3(pp, key, default):
    return tuple(int(v) for v in pp[key][:3]) if key in pp else default


def file_root(infile: str) -> str:                      # getFileRoot (grad.cpp:26-31)
    return os.path.basename(infile.rstrip("/"))


class _Dist:
    """torch.distributed if this is a multi-process run (RANK / WORLD_SIZE from torchrun), else a single rank.  solo=True: one
    rank of world size 1 whatever the environment (one file of a series)."""

    def __init__(self, backend: str, device: int, solo: bool = False):
        self.rank = 0 if solo else int(os.environ.get("RANK", "0"))
        self.world = 1 if solo else int(os.environ.get("WORLD_SIZE", "1"))
        self.dist = None
        self.own_group = False
        if self.world > 1:
            import torch
            import torch.distributed as dist
            self.dist = dist
            if backend == "nccl":
                torch.cuda.set_device(device)          # torch's current device = the one the C ABI was initialised on
            if not dist.is_initialized():
                if backend == "nccl":
                    dist.init_process_group(backend, device_id=torch.device("cuda", device))
                else:
                    dist.init_process_group(backend)
                self.own_group = True

    def gather_objects(self, obj):
        if self.dist is None:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()

    def close(self):
        if self.dist is not None and self.own_group:
            self.dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------
def run(tool: str, argv: Sequence[str], capi=None, multigpu=None, wrap=None, backend: str = "nccl", device: int | None = None) -> str:
    """Runs one tool; returns the output plotfile path.  capi / multigpu / wrap exist so that tests can run the same code
    against another build of the C ABI; by default they are the product binding and NCCL."""
    if capi is None:
        from . import capi as _capi
        capi = _capi
    pp = parse_args(argv)
    if "infiles" in pp and tool in ("grad", "curvature", "filter"):
        return _series(tool, pp, capi, backend, device)
    if tool not in ("grad", "curvature", "filter") or "infile" not in pp:
        raise SystemExit(__doc__)
    dev = device if device is not None else int(os.environ.get("LOCAL_RANK", "0"))
    return _run_one(tool, pp, capi, multigpu, wrap, backend, dev, _Dist(backend, dev))


def _series(tool: str, pp, capi, backend: str, device: int | None) -> str:
    """infiles=: this rank's files of the list, each as a world-size-1 run; returns the last output of this rank ('' if none)."""
    infiles = pp.pop("infiles")
    if not infiles:
        raise SystemExit("amrex::Abort::0::infiles needs at least one plotfile !!!")
    for k in ("infile", "outfile", "transport"):
        if k in pp:
            raise SystemExit("amrex::Abort::0::infiles cannot be combined with %s (each file's output has its default name) !!!" % k)
    suffix = {"grad": "_gt", "curvature": "_K", "filter": "_filtered"}[tool]
    seen = {}
    for f in infiles:                                          # before anything is computed: one output name per input
        out = file_root(f) + suffix
        if out in seen:
            raise SystemExit("amrex::Abort::0::infiles: %s and %s both write %s !!!" % (seen[out], f, out))
        seen[out] = f
        try:
            plotfile.read_header(f)
        except Exception as e:                                 # noqa: BLE001  (any unreadable header stops the run up front)
            raise SystemExit("amrex::Abort::0::%s: cannot read plotfile: %s !!!" % (f, e))
    dev = device if device is not None else int(os.environ.get("LOCAL_RANK", "0"))
    D = _Dist(backend, dev)
    out = ""
    try:
        for f in infiles[D.rank::D.world]:
            one = dict(pp)
            one["infile"] = [f]
            out = _run_one(tool, one, capi, None, None, backend, dev, _Dist(backend, dev, solo=True))
    finally:
        D.barrier()
        D.close()
    return out


def _run_one(tool: str, pp, capi, multigpu, wrap, backend: str, dev: int, D: "_Dist") -> str:
    """One plotfile: the keys -> a run object (stencilrun / filterplt) over this rank's boxes; read and upload those boxes,
    step, write them to Level_l/Cell_D_<rank>; rank 0 writes Header and Cell_H from every rank's records."""
    infile = pp["infile"][0]
    pf = plotfile.read_plotfile(infile, finest_level=None if tool == "filter" else _get(pp, "finestLevel", 1000, int), load_data=False)

    def comp(n):
        if n not in pf.names:
            raise SystemExit("amrex::Abort::0::Cannot find %s data in pltfile !!!" % n)
        return pf.comp(n)

    if tool == "filter":                                       # filterPlt.cpp:100-222
        variables = pp.get("variables") or None
        for v in variables or []:
            if v not in pf.names:
                raise SystemExit("Variable '%s' not found in file" % v)
        Run, keep, time = filterplt.FilterRun, [], pf.time
        args = dict(filter_type=_get(pp, "filter_type", 1, int), base_fgr=_get(pp, "base_fgr", 2, int),
                    same_fgr_all_levels=bool(_get(pp, "same_fgr_all_levels", 0, int)), max_grid_size=_get(pp, "max_grid_size", 32, int),
                    interp_type=_get(pp, "interp_type", 1, int), variables=variables, max_filter_level=_get(pp, "max_filter_level", 1000, int))
        outfile = file_root(infile) + "_filtered"
    else:
        for lv in pf.levels:                                   # the reference's dx: the problem extents over the cell count
            lv.dx = tuple((pf.prob_hi[d] - pf.prob_lo[d]) / (lv.domain_hi[d] - lv.domain_lo[d] + 1) for d in range(3))
        aux = pp.get("Aux_Variables", [])
        for a in aux:
            if a not in pf.names:
                raise SystemExit("amrex::Abort::0::Unknown auxiliary variable name: %s !!!" % a)
        args = dict(is_per=_ints3(pp, "is_per", (1, 1, 1)), sym_dir=_ints3(pp, "sym_dir", (0, 0, 0)),
                    peer_links=D.world > 1 and _get(pp, "transport", "peer") == "peer")
        time = 0.0
        if tool == "grad":
            gvars = pp.get("gradVars") or [_get(pp, "gradVar", "temp")]
            for v in gvars:
                comp(v)
            Run, keep = stencilrun.GradRun, gvars + list(aux)
            args["names"] = gvars
            outfile = _get(pp, "outfile", file_root(infile) + "_gt")
        else:
            prog = _get(pp, "progressName", "temp")
            o = capi.CurvOpts()
            o.do_threshold = _get(pp, "threshold_prog", 0, int)
            o.threshold = _get(pp, "threshold_value", 1.0e-4, float)
            o.do_gauss, o.do_strain = _get(pp, "do_gaussCurv", 0, int), _get(pp, "do_strain", 0, int)
            o.get_strain_tensor, o.do_velnormal = _get(pp, "getStrainTensor", 0, int), _get(pp, "do_velnormal", 0, int)
            do_smooth = bool(_get(pp, "do_smooth", 0, int))
            if do_smooth and D.world > 1:
                raise SystemExit("amrex::Abort::0::do_smooth=1 runs on one GPU only: the smoothing solve has no multi-GPU path (run at world size 1) !!!")
            precond = _get(pp, "smooth_precond", "jacobi")
            if precond not in capi.SMOOTH_PRECONDS:
                raise SystemExit("amrex::Abort::0::smooth_precond must be jacobi or mg (got %s) !!!" % precond)
            if _get(pp, "useFileMinMax", 1, int):
                o.prog_min, o.prog_max = plotfile.file_min_max(infile, prog, len(pf.levels))
            else:
                o.prog_min, o.prog_max = _get(pp, "progMin", 1.0e20, float), _get(pp, "progMax", -1.0e20, float)
            if not o.prog_min < o.prog_max:
                raise SystemExit("amrex::Abort::0::progMin must be less than progMax !!!")
            vel = list(stencilrun.CurvatureRun.VEL) if (o.do_strain or o.do_velnormal) else []
            for n in [prog] + vel:
                comp(n)
            Run, keep = stencilrun.CurvatureRun, [prog] + (vel if o.do_strain else []) + list(aux)      # curvature.cpp:163-224
            args.update(opts=o, progress=prog, do_smooth=do_smooth, smoothing_time=_get(pp, "smoothing_time", 1.0e-7, float),
                        smooth_precond=precond)
            outfile = _get(pp, "outfile", file_root(infile) + "_K")

    capi.init(dev)
    if D.world > 1 and backend == "nccl":
        import torch
        capi.set_stream(torch.cuda.current_stream().cuda_stream)
    R = Run(capi, pf, upload=False, rank=D.rank, nranks=D.world, multigpu=multigpu, wrap=wrap, **args)
    fin = R.state if Run is stencilrun.CurvatureRun else R.fin

    # ---- this rank's boxes, each cut from the plotfile box that contains it (every FAB needed is read once), upload -------
    need = sorted({comp(n) for n in R.names + keep})
    row = {pf.names[c]: k for k, c in enumerate(need)}
    host_keep = [None] * R.nlev                                # per level: [len(keep)][local cells], the pass-through data
    for l in range(R.nlev):
        ids, boxes, mine = R.hier.local_boxes[l], pf.levels[l].boxes, R.levels[l].boxes
        if not ids:
            continue
        src = _containing(boxes, mine)
        read = sorted({src[b] for b in ids})
        fabs = dict(zip(read, plotfile.read_boxes(infile, l, read, need)))
        data = np.concatenate([_cut(fabs[src[b]], boxes[src[b]], mine[b]) for b in ids], axis=1)
        for k, n in enumerate(R.names):
            fin.upload_level(l, k, np.ascontiguousarray(data[row[n]]))
            capi.sync()
        host_keep[l] = data[[row[n] for n in keep]]
    D.barrier()                                               # every rank's inputs are resident before anyone reads them in place

    R.step()
    capi.sync()
    D.barrier()                                               # nobody frees a slab a peer may still be reading
    if tool == "curvature" and R.do_smooth and _get(pp, "verbose", 0, int):
        print("do_smooth: smoothing_time = %g, precond %s, %d iterations, max|c - A phi| / max|c| = %g" % (R.sopts.smoothing_time, precond,
                                                                                                          R.iterations, R.residual))

    # ---- pass-through components, then the results -> this rank's Cell_D files; rank 0 writes Header and Cell_H ----------
    if D.rank == 0:
        plotfile.create_plotfile_dirs(outfile, R.nlev)
    D.barrier()
    records = []
    for l in range(R.nlev):
        ids = R.hier.local_boxes[l]
        if not ids:
            continue
        res = np.concatenate((host_keep[l], R.download_level(l)))
        cells = [np.prod(np.subtract(hi, lo) + 1) for lo, hi in (R.levels[l].boxes[b] for b in ids)]
        records += plotfile.write_fab_file(outfile, l, "Cell_D_%05d" % D.rank, R.levels[l], ids, np.split(res, np.cumsum(cells)[:-1], axis=1))
    allrec = [r for part in D.gather_objects(records) for r in part]
    if D.rank == 0:                                           # the reference hard-codes refRatios = 2 (grad.cpp:255, filterPlt.cpp:50)
        out = plotfile.Plotfile(keep + R.out_names, pf.prob_lo, pf.prob_hi, [2] * (R.nlev - 1), R.levels, time, pf.coord)
        plotfile.write_metadata(outfile, out, allrec)
    D.barrier()
    D.close()
    return outfile


def _cut(fab: np.ndarray, fab_box, box) -> np.ndarray:
    """the cells of `box` in `fab` ([ncomp, nz, ny, nx] over fab_box) as [ncomp][cells]"""
    (flo, _), (lo, hi) = fab_box, box
    return fab[(slice(None),) + tuple(slice(lo[d] - flo[d], hi[d] - flo[d] + 1) for d in (2, 1, 0))].reshape(len(fab), -1)


def _containing(outer, inner) -> List[int]:
    """for each box of `inner`, the index of the box of `outer` that contains it; inner lists the boxes inside outer's first
    box first, then those inside its second, ... (a level's own boxes, or the boxes rechop cut from them)"""
    out, b = [], 0
    for lo, hi in inner:
        while not all(outer[b][0][d] <= lo[d] and hi[d] <= outer[b][1][d] for d in range(3)):
            b += 1
        out.append(b)
    return out


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    if not argv:
        raise SystemExit(__doc__)
    out = run(argv[0], argv[1:])
    if int(os.environ.get("RANK", "0")) == 0:
        print("Writing new data to " + out)


if __name__ == "__main__":
    main()
