"""CPU tier, world sizes 2 and 3 over gloo: filterPlt on several ranks.

* The FillPatch exchange plan (hier.cpp: Hier::fill_patch) without kernels: what rank p packs for rank q is, cell for cell
  and in order, what q expects from p, on every level and ghost width 1-6 with both interpolaters; an improperly nested
  hierarchy fails with the same message on every rank.
* End to end under the CUDA execution-model emulator of tests/emu (test infrastructure, see tests/test_emu_parity.py):
  pack kernel, send/recv of the packed slabs, unpack + FillPatch + filter; every rank's output boxes bit-equal to the golden
  vectors of the compiled reference or to the NumPy restatement, every rank's grown input FABs bit-equal to the
  restatement's.  A fill whose recv slab holds another level's or another field's data is refused."""
import ctypes as C
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _spawn(target, world, *args, timeout=900):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    ok = ctx.Array("i", [0] * world)
    procs = [ctx.Process(target=target, args=(r, world, port, ok) + args) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout)
    assert list(ok) == [1] * world, [p.exitcode for p in procs]


def _init(rank, world, port):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), CUEMU_SEED=str(1 + rank))
    dist.init_process_group("gloo", rank=rank, world_size=world)


# ---- the plan ----------------------------------------------------------------------------------------------------------
def _plan_hierarchies():
    from cases import FILTER_CASES
    from peleanalysis_b200 import capi, filterplt, synth
    out = []
    for name in ("filter_c3", "filter_lshape", "filter_ratio4", "filter_c1_corner_gauss"):
        builder, kw = FILTER_CASES[name]
        out.append((name, filterplt.rechop(capi, builder(), [0], kw.get("max_grid_size", 32), 1000)))
    pf = synth.config3(32, 16)
    for mgs in (7, 11, 16):
        out.append(("config3_32_mgs%d" % mgs, filterplt.rechop(capi, pf, [0], mgs, 1000)))
    return out


def _plan_worker(rank, world, port, ok):
    _init(rank, world, port)
    try:
        from peleanalysis_b200 import capi
        capi.lib()
        checked = 0
        for name, levels in _plan_hierarchies():
            rng = np.random.default_rng(len(name) + world)
            # the SFC distribution and a random one (uneven, ranks without boxes on some levels)
            owner_sets = [None, [rng.integers(0, world, len(lv.boxes)) for lv in levels]]
            for owners in owner_sets:
                H = capi.Hierarchy(levels, (0, 0, 0), (0, 0, 0), rank, world, owners=owners, flags=capi.FILTER_ONLY)
                for l in range(len(levels)):
                    for ng in range(1, 7):
                        for it in (0, 1):
                            try:
                                send, recv = H.fill_patch_exchange_ids(l, ng, it, 0), H.fill_patch_exchange_ids(l, ng, it, 1)
                                err = None
                            except capi.PaError as e:
                                send = recv = np.empty(0, dtype=np.int64)
                                err = str(e)
                            got = [None] * world
                            dist.all_gather_object(got, (send, recv, err))
                            errs = {g[2] for g in got}
                            assert len(errs) == 1, (name, l, ng, it, errs)          # one verdict on every rank
                            if err is not None:
                                continue
                            # recv slab of q: blocks by source owner, ascending; send slab of p: blocks by destination, ascending
                            lev_of = lambda ids: ids >> 56
                            box_of = lambda ids: (ids >> 32) & ((1 << 24) - 1)
                            blocks = {}
                            for q in range(world):
                                rq = got[q][1]
                                assert (rq >= 0).all()
                                src = np.array([H.owners[int(a)][int(b)] for a, b in zip(lev_of(rq), box_of(rq))], dtype=np.int64)
                                assert (src != q).all() and (np.diff(src) >= 0).all(), (name, l, ng, it, q)
                                for p in range(world):
                                    blocks[(p, q)] = rq[src == p]
                            for p in range(world):
                                want = np.concatenate([blocks[(p, q)] for q in range(world)])
                                assert np.array_equal(got[p][0], want), (name, l, ng, it, p)
                            assert set(np.unique(lev_of(recv))) <= {l, l - 1}
                            checked += 1
        assert checked > 100
        # one rank alone: nothing to exchange
        H1 = capi.Hierarchy(_plan_hierarchies()[0][1], (0, 0, 0), (0, 0, 0), flags=capi.FILTER_ONLY)
        assert H1.fill_patch_exchange_ids(1, 2, 1, 0).size == 0 and H1.fill_patch_exchange_ids(1, 2, 1, 1).size == 0
        # fine boxes whose ghost region needs coarse cells that level 1 does not cover: the same error on every rank
        from peleanalysis_b200 import synth
        lv = synth.config3(16, 8).levels
        bad = [lv[0], type(lv[1])(lv[1].domain_lo, lv[1].domain_hi, lv[1].dx, lv[1].boxes[:1], []), lv[2]]
        H = capi.Hierarchy(bad, (0, 0, 0), (0, 0, 0), rank, world, flags=capi.FILTER_ONLY)
        with pytest.raises(capi.PaError) as e:
            H.fill_patch_exchange_ids(2, 4, 1, 1)
        assert e.value.code == -1 and "not properly nested" in str(e.value)
        msgs = [None] * world
        dist.all_gather_object(msgs, str(e.value))
        assert len(set(msgs)) == 1
        ok[rank] = 1
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_fill_patch_plan_agrees_between_ranks(palib, world):
    _spawn(_plan_worker, world)


# ---- end to end under the emulator ------------------------------------------------------------------------------------
def _wrap_host(ptr, n):
    return torch.from_numpy(np.ctypeslib.as_array((C.c_double * int(n)).from_address(int(ptr))))


def _e2e_worker(rank, world, port, ok):
    _init(rank, world, port)
    try:
        from test_emu_multirank import _load_emulated
        from cases import FILTER_CASES
        from helpers import bit_equal, load_golden
        from oracle import filter_oracle as FO
        from peleanalysis_b200 import filterplt, synth
        from test_filter_oracle import out_boxes, parse_opts
        import test_gpu_filter as GF
        P, mg = _load_emulated()
        P.init(0)
        bad, received = [], 0

        def run(pf, kw):
            R = filterplt.FilterRun(P, pf, rank=rank, nranks=world, multigpu=mg, wrap=_wrap_host, **kw)
            R.step()
            R.step()                                     # twice: nothing stale may survive in the slabs
            P.sync()
            return R

        def check_grown(tag, R, grown):
            G = max(R.ngrow)
            for l in range(R.nlev):
                g = R.ngrow[l]
                for b in R.hier.local_boxes[l]:
                    for c in range(R.ncomp):
                        q = R.grown_input(l, b, c)
                        q = q[G - g:q.shape[0] - (G - g), G - g:q.shape[1] - (G - g), G - g:q.shape[2] - (G - g)]
                        if not bit_equal(q, grown[l][b][c]):
                            bad.append((tag, "ghost", l, b, c))

        for name in sorted(FILTER_CASES):
            pf, z = load_golden(name)
            kw = parse_opts(z)
            R = run(pf, kw)
            received += sum(x.roff[-1] > 0 for x in R.exchanges)
            assert [lv.boxes for lv in R.levels] == out_boxes(z)
            res = R.result()
            for ci, n in enumerate(R.names):
                want = z["out_" + n]
                o = 0
                for l, lv in enumerate(R.levels):
                    for b, (lo, hi) in enumerate(lv.boxes):
                        m = int(np.prod([hi[d] - lo[d] + 1 for d in range(3)]))
                        if res[l][b] is not None and not bit_equal(res[l][b][ci].ravel(), want[o:o + m]):
                            bad.append((name, n, l, b))
                        o += m
            if name in ("filter_c1_corner_gauss", "filter_c3", "filter_lshape", "filter_ratio4"):
                check_grown(name, R, FO.filter_plotfile(pf, **kw)[2])
        for ftype, fgr, mgs in GF.MIDSIZE:
            pf = synth.config3(32, 16, names=("temp", "Y_CH4"))
            kw = dict(filter_type=ftype, base_fgr=fgr, max_grid_size=mgs)
            _, ref, grown = FO.filter_plotfile(pf, **kw)
            R = run(pf, kw)
            received += sum(x.roff[-1] > 0 for x in R.exchanges)
            for l, ((rb, rf), got) in enumerate(zip(ref, R.result())):
                for b in R.hier.local_boxes[l]:
                    if not bit_equal(got[b], rf[b]):
                        bad.append(("midsize", ftype, fgr, mgs, l, b))
            check_grown("midsize %s" % ((ftype, fgr, mgs),), R, grown)
        assert not bad, bad[:10]
        assert received > 0

        # misuse: the recv slab holds another level's / another field's data
        pf = synth.config3(32, 16, names=("temp", "Y_CH4"))
        R = filterplt.FilterRun(P, pf, rank=rank, nranks=world, multigpu=mg, wrap=_wrap_host, max_grid_size=8)
        other = P.Field(R.hier, R.ncomp, max(R.ngrow))
        X1, X2 = R.exchanges[1], R.exchanges[2]
        X1.run(0)
        if X2.roff[-1] > 0:
            with pytest.raises(P.PaError) as e:
                P.fill_patch(R.fin, 0, R.ncomp, 2, R.ngrow[2], R.interp_type)
            assert e.value.code == -1
        if X1.roff[-1] > 0:
            with pytest.raises(P.PaError) as e:
                P.fill_patch(other, 0, R.ncomp, 1, R.ngrow[1], R.interp_type)
            assert e.value.code == -1
            with pytest.raises(P.PaError):                # fewer components than were exchanged
                P.fill_patch(R.fin, 0, 1, 1, R.ngrow[1], R.interp_type)
            P.fill_patch(R.fin, 0, R.ncomp, 1, R.ngrow[1], R.interp_type)
        dist.barrier()
        X2.run(0)                                         # a new pack: the level-1 mark is gone
        if X1.roff[-1] > 0:
            with pytest.raises(P.PaError):
                P.fill_patch(R.fin, 0, R.ncomp, 1, R.ngrow[1], R.interp_type)
        P.fill_patch(R.fin, 0, R.ncomp, 2, R.ngrow[2], R.interp_type)
        P.sync()
        ok[rank] = 1
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_emulated_filter_on_several_ranks(world):
    _spawn(_e2e_worker, world)


# ---- the tools --------------------------------------------------------------------------------------------------------
from test_emu_tools import emu_exes  # noqa: E402,F401  (module-scoped fixture: the host shells linked to the emulated library)

TOOL_CASES = [("filter_c3", 2), ("filter_c3_subset", 3), ("filter_c1_corner_gauss", 4), ("filter_c3_pc_samefgr", 2)]


def _tool_args(z):
    return [str(x) for x in z["opts"]] if "opts" in z.files else []


def _read_all(path):
    from peleanalysis_b200 import plotfile
    with open(os.path.join(path, "Header")) as f:
        head = f.read()
    r = plotfile.read_plotfile(path)
    return head, r


def _same_plotfile(a, b):
    from helpers import bit_equal
    ha, ra = _read_all(a)
    hb, rb = _read_all(b)
    assert ha == hb
    assert ra.names == rb.names and len(ra.levels) == len(rb.levels)
    for la, lb in zip(ra.levels, rb.levels):
        assert la.boxes == lb.boxes
        for fa, fb in zip(la.fabs, lb.fabs):
            assert bit_equal(fa, fb)


def _one_gpu_tool(exe, name, tmp):
    from helpers import load_golden
    from peleanalysis_b200 import plotfile
    pf, z = load_golden(name)
    d = os.path.join(tmp, "plt_" + name)
    plotfile.write_plotfile(d, pf)
    run = os.path.join(tmp, "one_" + name)
    os.makedirs(run)
    env = dict(os.environ, CUEMU_DEVICES="1")
    p = subprocess.run([exe, "infile=" + d] + _tool_args(z), capture_output=True, text=True, cwd=run, env=env)
    assert p.returncode == 0, p.stdout + p.stderr
    return d, z, os.path.join(run, "plt_%s_filtered" % name), p.stdout


@pytest.mark.parametrize("name,ngpus", TOOL_CASES)
def test_emulated_filter_executable_multi_gpu(emu_exes, tmp_path, name, ngpus):  # noqa: F811
    """filterPlt3d ... ngpus=N (one host thread per emulated GPU): the same plotfile as ngpus=1, header and values; AMReX's
    fcompare agrees with the reference executable where the reference tools are built"""
    exe = emu_exes[2]
    d, z, one, out1 = _one_gpu_tool(exe, name, str(tmp_path))
    run = tmp_path / ("multi_%d" % ngpus)
    run.mkdir()
    env = dict(os.environ, CUEMU_DEVICES=str(ngpus), CUEMU_SEED="5")
    p = subprocess.run([exe, "infile=" + d, "ngpus=%d" % ngpus] + _tool_args(z), capture_output=True, text=True, cwd=str(run), env=env)
    assert p.returncode == 0, p.stdout + p.stderr
    assert p.stdout == out1                                   # the tool's progress messages
    out = str(run / ("plt_%s_filtered" % name))
    _same_plotfile(out, one)
    files = {f for l in range(len(os.listdir(out)) - 1) if os.path.isdir(os.path.join(out, "Level_%d" % l))
             for f in os.listdir(os.path.join(out, "Level_%d" % l))}
    assert len([f for f in files if f.startswith("Cell_D_")]) >= 2
    from oracle import oracle as O
    if O.have_ref():
        q = subprocess.run([O.ref_exe("fcompare.ref.ex"), out, one], capture_output=True, text=True)
        assert "PLOTFILE AGREE" in q.stdout, q.stdout[-1500:]


def _mgtool_worker(rank, world, port, ok, tmp, cases):
    _init(rank, world, port)
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world))
    try:
        from peleanalysis_b200 import mgtools
        from test_emu_multirank import _load_emulated
        capi, mg = _load_emulated()
        for name, d, args in cases:
            run = os.path.join(tmp, "mg_%s" % name)
            if rank == 0:
                os.makedirs(run)
            dist.barrier()
            cwd = os.getcwd()
            os.chdir(run)
            try:
                mgtools.run("filter", ["infile=" + d] + args, capi=capi, multigpu=mg, wrap=_wrap_host, backend="gloo", device=0)
            finally:
                os.chdir(cwd)
            dist.barrier()
        ok[rank] = 1
    finally:
        dist.destroy_process_group()


def test_emulated_mgtools_filter_world2(emu_exes, tmp_path):  # noqa: F811
    """torchrun ... -m peleanalysis_b200.mgtools filter (gloo, emulated library): header, box list and every value equal to the
    single-process executable's output"""
    cases, ones = [], {}
    for name in ("filter_c3", "filter_c3_subset", "filter_lshape"):
        d, z, one, _ = _one_gpu_tool(emu_exes[2], name, str(tmp_path))
        cases.append((name, d, _tool_args(z)))
        ones[name] = one
    _spawn(_mgtool_worker, 2, str(tmp_path), cases)
    for name, one in ones.items():
        out = str(tmp_path / ("mg_%s" % name) / ("plt_%s_filtered" % name))
        _same_plotfile(out, one)
        assert sorted(os.listdir(os.path.join(out, "Level_0"))) == ["Cell_D_00000", "Cell_D_00001", "Cell_H"]
