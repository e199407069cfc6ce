"""grad / curvature on a plotfile with one process per GPU -- the multi-GPU form of the drop-in executables.

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
other ranks move as packed slabs (multigpu.FillPatchExchange).  What an MPI build of the reference does, rank by rank, is done here process by process: every rank reads the
metadata, owns the boxes the SFC distribution gives it, reads only those from disk, runs the C-ABI calls on its GPU (cross-
rank ghost cells through peer links over NVLink or NCCL slab exchange, multigpu.py), writes its own boxes to its own
Level_l/Cell_D_<rank> file, and rank 0 writes Header and Cell_H from the gathered per-box (file, offset, min, max) records --
the layout VisMF produces with one file per rank (AMReX_VisMF.cpp:905-1005).  No compute happens in Python.
"""
from __future__ import annotations

import os
import sys
from typing import Dict, List, Sequence

import numpy as np

from . import plotfile


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


def read_boxes(path: str, hd, lev: int, meta, box_ids: Sequence[int], comp_ids: Sequence[int]) -> np.ndarray:
    """[len(comp_ids)][cells of the given boxes, concatenated] -- only those FABs and components are read from disk."""
    ncomp, boxes, fod, _, _ = meta
    ldir = os.path.dirname(os.path.join(path, hd["paths"][lev]))
    sizes = [int(np.prod([boxes[b][1][d] - boxes[b][0][d] + 1 for d in range(3)])) for b in box_ids]
    out = np.empty((len(comp_ids), sum(sizes)))
    o = 0
    for b, n in zip(box_ids, sizes):
        fn, off = fod[b]
        with open(os.path.join(ldir, fn), "rb") as f:
            f.seek(off)
            dt, flo, fhi, fnc = plotfile.parse_fab_header(f.readline().decode("ascii", "replace"), fn)
            base = f.tell()
            lo, hi = boxes[b]
            m = [fhi[d] - flo[d] + 1 for d in range(3)]
            if any(flo[d] > lo[d] or fhi[d] < hi[d] for d in range(3)) or max(comp_ids) >= fnc:
                raise ValueError("FAB in %s does not cover box %s / component %d" % (fn, boxes[b], max(comp_ids)))
            sl = tuple(slice(lo[d] - flo[d], hi[d] - flo[d] + 1) for d in (2, 1, 0))
            nf = m[0] * m[1] * m[2]
            for k, c in enumerate(comp_ids):
                f.seek(base + np.dtype(dt).itemsize * nf * c)
                out[k, o:o + n] = np.fromfile(f, dt, nf).reshape(m[2], m[1], m[0])[sl].ravel()
        o += n
    return out


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
    if multigpu is None and D.world > 1:
        from . import multigpu as _mg
        multigpu = _mg
    infile = pp["infile"][0]
    hd = plotfile.read_header(infile)
    if tool == "filter":
        return _filter(pp, infile, hd, capi, multigpu, wrap, backend, D, dev)
    nlev = min(_get(pp, "finestLevel", 1000, int), hd["finest"]) + 1
    is_per = _ints3(pp, "is_per", (1, 1, 1))
    sym_dir = _ints3(pp, "sym_dir", (0, 0, 0))
    transport = _get(pp, "transport", "peer")
    names_in = hd["names"]

    def comp(n):
        if n not in names_in:
            raise SystemExit("amrex::Abort::0::Cannot find %s data in pltfile !!!" % n)
        return names_in.index(n)
    aux = pp.get("Aux_Variables", [])
    for a in aux:
        if a not in names_in:
            raise SystemExit("amrex::Abort::0::Unknown auxiliary variable name: %s !!!" % a)
    metas = [plotfile.read_cell_h(infile, hd["paths"][l]) for l in range(nlev)]
    levels = [plotfile.Level(hd["domains"][l][0], hd["domains"][l][1],
                             tuple((hd["prob_hi"][d] - hd["prob_lo"][d]) / (hd["domains"][l][1][d] - hd["domains"][l][0][d] + 1) for d in range(3)),
                             metas[l][1], []) for l in range(nlev)]

    capi.init(dev)
    if D.world > 1 and backend == "nccl":
        import torch
        capi.set_stream(torch.cuda.current_stream().cuda_stream)
    flags = capi.PEER_LINKS if (D.world > 1 and transport == "peer") else 0
    H = capi.Hierarchy(levels, is_per, sym_dir, D.rank, D.world, flags=flags)
    kw = {} if wrap is None else {"wrap": wrap}

    do_smooth = False
    if tool == "grad":
        gvars = pp.get("gradVars") or [_get(pp, "gradVar", "temp")]
        dev_in = [comp(v) for v in gvars]
        keep = gvars + list(aux)
        out_names = keep + [s for v in gvars for s in (v + "_gx", v + "_gy", v + "_gz", "||grad" + v + "||")]
        outfile = _get(pp, "outfile", file_root(infile) + "_gt")
        nv = len(gvars)
        fin, fout = capi.Field(H, nv, 1), capi.Field(H, 4 * nv, 0)
        nres = 4 * nv
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
        so = capi.SmoothOpts()
        so.smoothing_time = _get(pp, "smoothing_time", 1.0e-7, float)
        precond = _get(pp, "smooth_precond", "jacobi")
        if precond not in capi.SMOOTH_PRECONDS:
            raise SystemExit("amrex::Abort::0::smooth_precond must be jacobi or mg (got %s) !!!" % precond)
        so.precond = capi.SMOOTH_PRECONDS[precond]
        if _get(pp, "useFileMinMax", 1, int):
            o.prog_min, o.prog_max = plotfile.file_min_max(infile, prog, nlev)
        else:
            o.prog_min, o.prog_max = _get(pp, "progMin", 1.0e20, float), _get(pp, "progMax", -1.0e20, float)
        if not o.prog_min < o.prog_max:
            raise SystemExit("amrex::Abort::0::progMin must be less than progMax !!!")
        need_vel = bool(o.do_strain or o.do_velnormal)
        vel = ["x_velocity", "y_velocity", "z_velocity"] if need_vel else []
        dev_in = [comp(prog)] + [comp(v) for v in vel]
        keep = [prog] + (vel if o.do_strain else []) + list(aux)          # curvature.cpp:163-224
        v = prog
        out_names = keep + ["Progress", "SmoothedProgress", "MeanCurvature_" + v, "FlameNormalX_" + v, "FlameNormalY_" + v,
                            "FlameNormalZ_" + v, "GaussianCurvature_" + v]
        if o.do_strain:
            out_names.append("StrainRate_" + v)
            if o.get_strain_tensor:
                out_names += ["ROST_dU%sd%s" % (a, b) for a in "xyz" for b in "xyz"]
        if o.do_velnormal:
            out_names.append("VelFlameNormal")
        outfile = _get(pp, "outfile", file_root(infile) + "_K")
        fin = capi.Field(H, len(dev_in) + (2 if do_smooth else 0), 1)     # do_smooth: + c and phi
        nres = capi.curvature_num_outputs(o)
        fout = capi.Field(H, nres, 1)

    # ---- read this rank's boxes, upload ---------------------------------------------------------------------------
    host_keep = []                                             # per level: [len(keep)][local cells], pass-through data
    for l in range(nlev):
        ids = H.local_boxes[l]
        need = sorted(set(dev_in) | {comp(n) for n in keep})
        data = read_boxes(infile, hd, l, metas[l], ids, need) if ids else np.empty((len(need), 0))
        row = {c: k for k, c in enumerate(need)}
        if ids:
            for k, c in enumerate(dev_in):
                fin.upload_level(l, k, np.ascontiguousarray(data[row[c]]))
                capi.sync()
        host_keep.append(np.stack([data[row[comp(n)]] for n in keep]) if keep else np.empty((0, data.shape[1])))
    D.barrier()                                               # every rank's inputs are resident before anyone reads them in place

    # ---- the hot path -----------------------------------------------------------------------------------------------
    if tool == "grad":
        if D.world > 1:
            if flags:
                multigpu.map_peers(fin)
                D.barrier()
            X = multigpu.SlabExchange(fin, nv, **kw)
            X.run(0)
        capi.grad(fin, 0, nv, fout, 0)
    elif D.world > 1:
        op = multigpu.Curvature(fin, 0, o, fout, 0, comp_vel=1, **kw)
        D.barrier()
        op.run()
    elif do_smooth:                                            # curvature.cpp:328-406: curvature of phi, identity normalisation
        cc, cphi = len(dev_in), len(dev_in) + 1
        iters, resid = capi.smooth(fin, 0, o.prog_min, o.prog_max, so, fin, cc, cphi)
        if _get(pp, "verbose", 0, int):
            print("do_smooth: smoothing_time = %g, precond %s, %d iterations, max|c - A phi| / max|c| = %g" % (so.smoothing_time, precond, iters,
                                                                                                              resid))
        o_phi = capi.CurvOpts.from_buffer_copy(o)
        o_phi.prog_min, o_phi.prog_max = 0.0, 1.0
        capi.curvature(fin, cphi, 1, o_phi, fout, 0)
    else:
        capi.curvature(fin, 0, 1, o, fout, 0)
    capi.sync()
    D.barrier()                                               # nobody frees a slab a peer may still be reading

    # ---- results -> per-rank Cell_D files; rank 0 writes Header and Cell_H ----------------------------------------------
    if tool == "curvature":
        # library order: Progress, K, n(3), [Kg], [SR], [ROST 9], [VN]; file order has SmoothedProgress and GaussianCurvature
        # slots that exist even when the options are off (never written by the reference: zeros here)
        res_index = {"Progress": 0, "MeanCurvature_" + v: 1, "FlameNormalX_" + v: 2, "FlameNormalY_" + v: 3, "FlameNormalZ_" + v: 4}
        nxt = 5
        if o.do_gauss:
            res_index["GaussianCurvature_" + v] = nxt
            nxt += 1
        if o.do_strain:
            res_index["StrainRate_" + v] = nxt
            nxt += 1
            if o.get_strain_tensor:
                for a in "xyz":
                    for b in "xyz":
                        res_index["ROST_dU%sd%s" % (a, b)] = nxt
                        nxt += 1
        if o.do_velnormal:
            res_index["VelFlameNormal"] = nxt
        if do_smooth:                                         # the curvature's Progress is phi; the file's Progress is c (in fin)
            res_index["SmoothedProgress"] = res_index.pop("Progress")
    else:
        res_index = {n: k for k, n in enumerate(out_names[len(keep):])}

    if D.rank == 0:
        if os.path.lexists(outfile):
            os.rename(outfile, plotfile.unique_old_name(outfile))          # UtilCreateCleanDirectory (AMReX_Utility.cpp:160-172)
        os.makedirs(outfile)
        for l in range(nlev):
            os.makedirs(os.path.join(outfile, "Level_%d" % l))
    D.barrier()
    ncomp_out = len(out_names)
    records = []                                              # (level, global box, file, offset, mins, maxs)
    for l in range(nlev):
        ids = H.local_boxes[l]
        if not ids:
            continue
        ncell = H.local_cells[l]
        res = np.zeros((ncomp_out, ncell))
        res[:len(keep)] = host_keep[l]
        buf = np.empty(ncell)
        for k, n in enumerate(out_names[len(keep):]):
            if n in res_index:
                fout.download_level(l, res_index[n], buf)
                capi.sync()
                res[len(keep) + k] = buf
            elif do_smooth and n == "Progress":
                fin.download_level(l, len(dev_in), buf)
                capi.sync()
                res[len(keep) + k] = buf
        fn = "Cell_D_%05d" % D.rank
        with open(os.path.join(outfile, "Level_%d" % l, fn), "wb") as f:
            o0 = 0
            for b in ids:
                lo, hi = levels[l].boxes[b]
                n = int(np.prod([hi[d] - lo[d] + 1 for d in range(3)]))
                off = f.tell()
                f.write(("FAB ((8, (64 11 52 0 1 12 0 1023)),(8, (8 7 6 5 4 3 2 1)))%s %d\n" % (plotfile._box_str(lo, hi), ncomp_out)).encode())
                blk = res[:, o0:o0 + n]
                f.write(np.ascontiguousarray(blk, dtype="<f8").tobytes())
                records.append((l, b, fn, off, blk.min(axis=1).tolist(), blk.max(axis=1).tolist()))
                o0 += n
    allrec = [r for part in D.gather_objects(records) for r in part]
    if D.rank == 0:
        _write_metadata(outfile, hd, levels, nlev, out_names, allrec, 0.0)
    D.barrier()
    D.close()
    return outfile


def _filter(pp, infile, hd, capi, multigpu, wrap, backend, D, dev) -> str:
    """filterPlt (filterPlt.cpp:100-222) with this rank's share of the re-chopped boxes."""
    from . import filterplt
    variables = pp.get("variables") or None
    for v in variables or []:
        if v not in hd["names"]:
            raise SystemExit("Variable '%s' not found in file" % v)
    nfile = hd["finest"] + 1
    metas = [plotfile.read_cell_h(infile, hd["paths"][l]) for l in range(nfile)]
    levels = [plotfile.Level(hd["domains"][l][0], hd["domains"][l][1], hd["dx"][l], metas[l][1], []) for l in range(nfile)]
    pf = plotfile.Plotfile(list(hd["names"]), hd["prob_lo"], hd["prob_hi"], hd["ref_ratio"], levels, hd["time"], hd["coord"])
    mgs = _get(pp, "max_grid_size", 32, int)
    capi.init(dev)
    if D.world > 1 and backend == "nccl":
        import torch
        capi.set_stream(torch.cuda.current_stream().cuda_stream)
    kw = {} if wrap is None else {"wrap": wrap}
    R = filterplt.FilterRun(capi, pf, filter_type=_get(pp, "filter_type", 1, int), base_fgr=_get(pp, "base_fgr", 2, int),
                            same_fgr_all_levels=bool(_get(pp, "same_fgr_all_levels", 0, int)), max_grid_size=mgs,
                            interp_type=_get(pp, "interp_type", 1, int), variables=variables,
                            max_filter_level=_get(pp, "max_filter_level", 1000, int), upload=False, rank=D.rank, nranks=D.world,
                            multigpu=multigpu, **kw)
    comps = [hd["names"].index(n) for n in R.names]
    # this rank's output boxes, cut from the plotfile boxes that contain them (only those FABs are read)
    for l in range(R.nlev):
        parent = [b for b, bx in enumerate(levels[l].boxes) for _ in capi.boxes_max_size([bx], mgs)]
        ids = R.hier.local_boxes[l]
        if not ids:
            continue
        host = np.empty((len(comps), R.hier.local_cells[l]))
        o, i = 0, 0
        while i < len(ids):
            pb = parent[ids[i]]
            (lo, hi) = levels[l].boxes[pb]
            data = read_boxes(infile, hd, l, metas[l], [pb], comps).reshape(len(comps), hi[2] - lo[2] + 1, hi[1] - lo[1] + 1, hi[0] - lo[0] + 1)
            while i < len(ids) and parent[ids[i]] == pb:
                clo, chi = R.levels[l].boxes[ids[i]]
                blk = data[(slice(None),) + tuple(slice(clo[d] - lo[d], chi[d] - lo[d] + 1) for d in (2, 1, 0))].reshape(len(comps), -1)
                host[:, o:o + blk.shape[1]] = blk
                o += blk.shape[1]
                i += 1
        for c in range(len(comps)):
            R.fin.upload_level(l, c, np.ascontiguousarray(host[c]))
            capi.sync()
    D.barrier()
    R.step()
    capi.sync()
    D.barrier()
    outfile = file_root(infile) + "_filtered"
    if D.rank == 0:
        if os.path.lexists(outfile):
            os.rename(outfile, plotfile.unique_old_name(outfile))
        os.makedirs(outfile)
        for l in range(R.nlev):
            os.makedirs(os.path.join(outfile, "Level_%d" % l))
    D.barrier()
    records = []
    res = R.result()
    fn = "Cell_D_%05d" % D.rank
    for l in range(R.nlev):
        if not R.hier.local_boxes[l]:
            continue
        with open(os.path.join(outfile, "Level_%d" % l, fn), "wb") as f:
            for b in R.hier.local_boxes[l]:
                lo, hi = R.levels[l].boxes[b]
                blk = res[l][b].reshape(R.ncomp, -1)
                off = f.tell()
                f.write(("FAB ((8, (64 11 52 0 1 12 0 1023)),(8, (8 7 6 5 4 3 2 1)))%s %d\n" % (plotfile._box_str(lo, hi), R.ncomp)).encode())
                f.write(np.ascontiguousarray(blk, dtype="<f8").tobytes())
                records.append((l, b, fn, off, blk.min(axis=1).tolist(), blk.max(axis=1).tolist()))
    allrec = [r for part in D.gather_objects(records) for r in part]
    if D.rank == 0:
        _write_metadata(outfile, hd, R.levels, R.nlev, R.names, allrec, hd["time"])    # ref_ratio 2 (filterPlt.cpp:50)
    D.barrier()
    D.close()
    return outfile


def _write_metadata(outfile, hd, levels, nlev, names, records, time):
    """Header (WriteGenericPlotfileHeader, AMReX_PlotFileUtil.cpp:73-155) and Level_l/Cell_H (VisMF header v1)."""
    f17 = plotfile._fmt17
    with open(os.path.join(outfile, "Header"), "w") as h:
        h.write("HyperCLaw-V1.1\n%d\n" % len(names))
        for n in names:
            h.write(n + "\n")
        h.write("3\n%s\n%d\n" % (f17(time), nlev - 1))
        h.write(" ".join(f17(x) for x in hd["prob_lo"]) + " \n")
        h.write(" ".join(f17(x) for x in hd["prob_hi"]) + " \n")
        h.write(" ".join("2" for _ in range(nlev - 1)) + " \n")          # the reference hard-codes refRatios = 2 (grad.cpp:255)
        h.write(" ".join(plotfile._box_str(lv.domain_lo, lv.domain_hi) for lv in levels) + " \n")
        h.write(" ".join("0" for _ in range(nlev)) + " \n")
        for lv in levels:
            h.write(" ".join(f17(x) for x in lv.dx) + " \n")
        h.write("%d\n0\n" % hd["coord"])
        for l, lv in enumerate(levels):
            h.write("%d %d %s\n0\n" % (l, len(lv.boxes), f17(time)))
            for lo, hi in lv.boxes:
                for d in range(3):
                    h.write("%s %s\n" % (f17(hd["prob_lo"][d] + lv.dx[d] * (lo[d] - lv.domain_lo[d])),
                                         f17(hd["prob_lo"][d] + lv.dx[d] * (hi[d] - lv.domain_lo[d] + 1))))
            h.write("Level_%d/Cell\n" % l)
    for l, lv in enumerate(levels):
        rec = {b: (fn, off, mn, mx) for (ll, b, fn, off, mn, mx) in records if ll == l}
        assert len(rec) == len(lv.boxes), "level %d: %d of %d boxes were written" % (l, len(rec), len(lv.boxes))
        with open(os.path.join(outfile, "Level_%d" % l, "Cell_H"), "w") as c:
            c.write("1\n1\n%d\n0\n(%d 0\n" % (len(names), len(lv.boxes)))
            for lo, hi in lv.boxes:
                c.write(plotfile._box_str(lo, hi) + "\n")
            c.write(")\n%d\n" % len(lv.boxes))
            for b in range(len(lv.boxes)):
                c.write("FabOnDisk: %s %d\n" % (rec[b][0], rec[b][1]))
            c.write("\n")
            for k in (2, 3):
                c.write("%d,%d\n" % (len(lv.boxes), len(names)))
                for b in range(len(lv.boxes)):
                    c.write("".join("%.17e," % x for x in rec[b][k]) + "\n")
                c.write("\n")


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    if not argv:
        raise SystemExit(__doc__)
    out = run(argv[0], argv[1:])
    if int(os.environ.get("RANK", "0")) == 0:
        print("Writing new data to " + out)


if __name__ == "__main__":
    main()
