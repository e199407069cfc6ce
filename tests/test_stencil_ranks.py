"""CPU tier, world sizes 2 and 3 over gloo: grad and curvature on several ranks with every cross-rank ghost source moved as a
packed slab (no peer mapping).

* The width-1 exchange plan (hier.cpp: build_exchange) without kernels: what rank p packs for rank q is, cell for cell and
  in order, what q expects from p, for every grad / curvature fixture and the mid-size hierarchies, with the SFC
  distribution and with random owners.  A level 0 that does not cover the domain fails with the same message on every rank.
* End to end under the CUDA execution-model emulator of tests/emu (test infrastructure, see tests/test_emu_parity.py):
  stencilrun.GradRun / CurvatureRun on several ranks against the same runs on one rank, bit for bit, in every output box
  and in the ghost cells of the input, state and flame-normal fields.  A ghost fill whose recv slab was not marked for
  exactly that field and component range is refused.
* The host executables with transport=slab at ngpus=2, 3, 4 and `mgtools grad` / `curvature` at world 3: the same
  plotfile as the one-GPU tool."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist

from test_fill_patch_exchange import _init, _same_plotfile, _spawn, _wrap_host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

MIDSIZE = [("config3", dict(base=32, mgs=16)), ("config5", dict(base=16, mgs=8, ncomp=2, ratios=(2, 4, 2))), ("lshape", dict(base=32, mgs=16))]


def _hierarchies():
    """(name, plotfile, is_per, sym_dir, tools, curvature options) of every grad / curvature fixture and mid-size hierarchy"""
    from cases import CASES
    from peleanalysis_b200 import synth
    out = [(n, b(), per, sym, tools, kw) for n, (b, per, sym, tools, kw) in sorted(CASES.items())]
    for case, kw in MIDSIZE:
        pf = synth.CASES[case](**kw)
        # the reference's curvature hard-codes ratio 2 (curvature.cpp:445,518): config5 (ratios 2, 4, 2) is a grad case only
        out.append(("midsize_" + case, pf, (1, 1, 1), (0, 0, 0), ("grad",) if case == "config5" else ("grad", "curvature"), {}))
    return out


# ---- the plan ----------------------------------------------------------------------------------------------------------
def _plan_worker(rank, world, port, ok):
    _init(rank, world, port)
    try:
        from peleanalysis_b200 import capi, plotfile, synth
        checked = 0
        for name, pf, is_per, sym, _, _ in _hierarchies():
            rng = np.random.default_rng(len(name) + world)
            for owners in (None, [rng.integers(0, world, len(lv.boxes)) for lv in pf.levels]):
                H = capi.Hierarchy(pf.levels, is_per, sym, rank, world, owners=owners)
                send_ids, want = H.exchange_ids(0), H.exchange_ids(1)
                sc, rc = H.exchange_prefix(1)
                assert sc[rank] == 0 and rc[rank] == 0
                assert sc.sum() == send_ids.size and rc.sum() == want.size
                assert (want >= 0).all() and (send_ids >= 0).all()
                so = np.concatenate([[0], np.cumsum(sc)])
                blocks = [None] * world
                dist.all_gather_object(blocks, [send_ids[so[q]:so[q + 1]] for q in range(world)])
                got = np.concatenate([np.asarray(blocks[p][rank], dtype=np.int64) for p in range(world) if p != rank] or [np.zeros(0, np.int64)])
                assert np.array_equal(got, want), (name, int((got != want).sum()))
                tot = torch.tensor([H.num_local_cells], dtype=torch.int64)
                dist.all_reduce(tot)
                assert int(tot.item()) == H.num_cells
                checked += int(want.size)
        assert checked > 0
        # a level 0 with a hole: every rank refuses the hierarchy with the message one rank gives
        full = synth.make_hierarchy(32, [], [], 8, fill=False).levels[0]
        hole = [plotfile.Level(full.domain_lo, full.domain_hi, full.dx, [b for i, b in enumerate(full.boxes) if i != 27], [])]
        with pytest.raises(capi.PaError) as e1:
            capi.Hierarchy(hole, (1, 1, 1), (0, 0, 0))
        for owners in (None, [np.arange(len(hole[0].boxes)) % world]):
            with pytest.raises(capi.PaError) as e:
                capi.Hierarchy(hole, (1, 1, 1), (0, 0, 0), rank, world, owners=owners)
            msgs = [None] * world
            dist.all_gather_object(msgs, str(e.value))
            assert msgs == [str(e1.value)] * world, msgs
            assert "level 0 does not cover the domain" in msgs[0]
        ok[rank] = 1
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_stencil_exchange_plan_agrees_between_ranks(palib, world):
    _spawn(_plan_worker, world)


# ---- end to end, emulated ----------------------------------------------------------------------------------------------
def _curv_opts(P, pf, kw):
    s = np.concatenate([f[pf.comp("temp")].ravel() for lv in pf.levels for f in lv.fabs])
    o = P.CurvOpts()
    o.prog_min, o.prog_max = float(s.min()), float(s.max())
    o.do_threshold = int(kw.get("threshold_prog", 0))
    o.threshold = float(kw.get("threshold_value", 1.0e-4))
    o.do_gauss, o.do_strain = int(kw.get("do_gaussCurv", 0)), int(kw.get("do_strain", 0))
    o.get_strain_tensor, o.do_velnormal = int(kw.get("getStrainTensor", 0)), int(kw.get("do_velnormal", 0))
    return o


def _e2e_worker(rank, world, port, ok):
    _init(rank, world, port)
    try:
        from helpers import bit_equal
        from peleanalysis_b200 import stencilrun, synth
        from test_emu_multirank import _load_emulated
        P, mg = _load_emulated()
        P.init(0)
        bad, moved = [], 0

        def same_outputs(tag, many, one):
            for l, (rm, r1) in enumerate(zip(many.result(), one.result())):
                for b in many.hier.local_boxes[l]:
                    if not bit_equal(rm[b], r1[b]):
                        bad.append((tag, "out", l, b))

        def same_ghosts(tag, fm, f1, comps):
            for l in range(fm.hier.nlev):
                for b in fm.hier.local_boxes[l]:
                    for c in comps:
                        if not bit_equal(fm.download_grown(l, b, c), f1.download_grown(l, b, c)):
                            bad.append((tag, "ghost", l, b, c))

        for name, pf, is_per, sym, tools, kw in _hierarchies():
            var = pf.names[0]
            if "grad" in tools:
                Rm = stencilrun.GradRun(P, pf, [var], is_per, sym, rank=rank, nranks=world, multigpu=mg, wrap=_wrap_host)
                R1 = stencilrun.GradRun(P, pf, [var], is_per, sym)
                Rm.step()
                Rm.step()                                  # twice: nothing stale may survive in the slabs
                R1.step()
                P.sync()
                same_outputs("grad " + name, Rm, R1)
                moved += 0 if Rm.exchange.empty else 1
                # every width-1 face ghost cell materialised (pa_fill_ghosts), the cross-rank ones from the recv slab
                Rm.exchange.run(0)
                Rm.fin.fill_ghosts(0, 1)
                R1.fin.fill_ghosts(0, 1)
                P.sync()
                same_ghosts("grad " + name, Rm.fin, R1.fin, [0])
            if "curvature" in tools:
                o = _curv_opts(P, pf, kw)
                Cm = stencilrun.CurvatureRun(P, pf, o, "temp", is_per, sym, rank=rank, nranks=world, multigpu=mg, wrap=_wrap_host)
                C1 = stencilrun.CurvatureRun(P, pf, o, "temp", is_per, sym)
                Cm.step()
                Cm.step()
                C1.step()
                P.sync()
                same_outputs("curvature " + name, Cm, C1)
                # ghost cells of the state (S, velocities) and of the final flame normal
                Cm.op.Xs.run(0)
                Cm.state.fill_ghosts(0, 1)
                Cm.op.Xn.run(2)
                Cm.fout.fill_ghosts(2, 3)
                C1.state.fill_ghosts(0, 1)
                C1.fout.fill_ghosts(2, 3)
                if Cm.op.Xv is not None:
                    Cm.op.Xv.run(1)
                    Cm.state.fill_ghosts(1, 3)
                    C1.state.fill_ghosts(1, 3)
                P.sync()
                same_ghosts("curvature " + name, Cm.state, C1.state, range(len(Cm.names)))
                same_ghosts("curvature " + name, Cm.fout, C1.fout, [2, 3, 4])
        assert not bad, bad[:10]
        assert moved >= 8

        # misuse: the recv slab holds another field's or another component range's data, or nothing at all
        pf = synth.config3(32, 16, names=("temp", "Y_CH4"))
        R = stencilrun.GradRun(P, pf, ["temp", "Y_CH4"], rank=rank, nranks=world, multigpu=mg, wrap=_wrap_host)
        other = P.Field(R.hier, 2, 1)
        Xo = mg.SlabExchange(other, 2, _wrap_host)
        assert not R.exchange.empty
        with pytest.raises(P.PaError) as e:                # nothing exchanged yet
            P.grad(R.fin, 0, 2, R.fout, 0)
        assert e.value.code == -5
        R.exchange.run(0)
        with pytest.raises(P.PaError) as e:                # fewer components than were exchanged
            P.grad(R.fin, 0, 1, R.fout, 0)
        assert e.value.code == -5
        with pytest.raises(P.PaError) as e:                # another field
            P.grad(other, 0, 2, R.fout, 0)
        assert e.value.code == -5
        P.grad(R.fin, 0, 2, R.fout, 0)
        dist.barrier()
        Xo.run(0)                                          # a new pack into the shared slabs: the mark of R.fin is gone
        with pytest.raises(P.PaError) as e:
            P.grad(R.fin, 0, 2, R.fout, 0)
        assert e.value.code == -5
        P.grad(other, 0, 2, R.fout, 0)
        o = _curv_opts(P, pf, {})
        C = stencilrun.CurvatureRun(P, pf, o, rank=rank, nranks=world, multigpu=mg, wrap=_wrap_host)
        with pytest.raises(P.PaError) as e:                # the one-call form needs the caller's exchange between its passes
            P.curvature(C.state, 0, 0, o, C.fout, 0)
        assert e.value.code == -4
        P.sync()
        ok[rank] = 1
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_emulated_grad_and_curvature_on_several_ranks(world):
    _spawn(_e2e_worker, world)


# ---- the tools --------------------------------------------------------------------------------------------------------
from test_emu_tools import emu_exes  # noqa: E402,F401  (module-scoped fixture: the host shells linked to the emulated library)

GRAD_TOOL_CASES = [("c3_three_levels", 2), ("mixed_boxes", 3), ("lshape", 4), ("c1_corner_sym", 2), ("edge_walls", 3)]
CURV_TOOL_CASES = [("c1_options", 3), ("c3_threshold", 2), ("mixed_boxes", 4), ("c1_periodic", 2)]


def _tool_args(tool, z):
    per = "is_per=" + " ".join(str(int(v)) for v in z["is_per"])
    sym = "sym_dir=" + " ".join(str(int(v)) for v in z["sym_dir"])
    if tool == "grad":
        return ["gradVar=temp", per, sym]
    return ["progressName=temp", per, sym] + [str(s) for s in z["curv_opts"]]


def _run_tool(exe, d, args, cwd, ngpus, seed="5"):
    os.makedirs(cwd, exist_ok=True)
    env = dict(os.environ, CUEMU_DEVICES=str(ngpus), CUEMU_SEED=seed, PA_NORMAL_MATH="fast")
    p = subprocess.run([exe, "infile=" + d] + args, capture_output=True, text=True, cwd=cwd, env=env)
    assert p.returncode == 0, p.stdout + p.stderr
    return p


@pytest.mark.parametrize("tool,name,ngpus", [("grad",) + c for c in GRAD_TOOL_CASES] + [("curvature",) + c for c in CURV_TOOL_CASES])
def test_emulated_stencil_executables_slab_transport(emu_exes, tmp_path, tool, name, ngpus):  # noqa: F811
    """grad3d / curvature3d ... ngpus=N transport=slab (one host thread per emulated GPU, nothing peer-mapped): the same
    plotfile as ngpus=1, header and values, one Cell_D file per thread.  The tool's verbose report shows that no peer slab
    was mapped and, for grad, that every GPU received exactly what the width-1 plan without peer links sends it."""
    from helpers import load_golden
    from peleanalysis_b200 import capi, plotfile
    exe = emu_exes[0 if tool == "grad" else 1]
    pf, z = load_golden(name)
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    args = _tool_args(tool, z) + ["outfile=out"]
    _run_tool(exe, d, args, str(tmp_path / "one"), 1)
    p = _run_tool(exe, d, args + ["ngpus=%d" % ngpus, "transport=slab", "verbose=1"], str(tmp_path / "many"), ngpus)
    out = str(tmp_path / "many" / "out")
    _same_plotfile(out, str(tmp_path / "one" / "out"))
    assert _cell_files(out) <= {"Cell_D_%05d" % r for r in range(ngpus)} and len(_cell_files(out)) >= 2
    transport, mapped, received = _transport_report(p.stdout)
    assert transport == "slab" and mapped == [0] * ngpus, p.stdout
    if tool == "grad":
        per, sym = tuple(int(v) for v in z["is_per"]), tuple(int(v) for v in z["sym_dir"])
        want = [int(capi.Hierarchy(pf.levels, per, sym, r, ngpus).exchange_prefix(1)[1].sum()) for r in range(ngpus)]
        assert received == want and sum(want) > 0, (received, want)
        # the peer transport of the same run does map the other GPUs' slabs (so the report tells the two apart)
        q = _run_tool(exe, d, args + ["ngpus=%d" % ngpus, "verbose=1"], str(tmp_path / "peer"), ngpus)
        transport, mapped, _ = _transport_report(q.stdout)
        assert transport == "peer" and all(m > 0 for m in mapped), q.stdout
    else:
        assert sum(received) > 0, p.stdout


def _transport_report(stdout):
    """(transport, peer slabs mapped per GPU, doubles received per GPU) from the multi-GPU tools' verbose line"""
    line = [x for x in stdout.splitlines() if x.startswith("[b200] transport=")]
    assert len(line) == 1, stdout
    head, rest = line[0][len("[b200] transport="):].split(":", 1)
    mapped, received = rest.split(";")
    return head, [int(v) for v in mapped.split()[5:]], [int(v) for v in received.split()[6:]]


def _cell_files(out):
    levels = [d for d in os.listdir(out) if d.startswith("Level_")]
    return {f for d in levels for f in os.listdir(os.path.join(out, d)) if f.startswith("Cell_D_")}


def test_emulated_stencil_executables_reject_unknown_transport(emu_exes, tmp_path):  # noqa: F811
    from helpers import load_golden
    from peleanalysis_b200 import plotfile
    pf, z = load_golden("c1_periodic")
    d = str(tmp_path / "plt")
    plotfile.write_plotfile(d, pf)
    for exe in emu_exes[:2]:
        p = subprocess.run([exe, "infile=" + d, "ngpus=2", "transport=nvshmem"], capture_output=True, text=True, cwd=str(tmp_path),
                           env=dict(os.environ, CUEMU_DEVICES="2"))
        assert p.returncode != 0 and "transport must be peer or slab" in p.stdout + p.stderr


def _mgtool_worker(rank, world, port, ok, tmp, cases):
    _init(rank, world, port)
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world))
    try:
        from peleanalysis_b200 import mgtools
        from test_emu_multirank import _load_emulated
        capi, mg = _load_emulated()
        for tool, d, args, out in cases:
            mgtools.run(tool, ["infile=" + d, "transport=slab", "outfile=" + out] + args, capi=capi, multigpu=mg, wrap=_wrap_host,
                        backend="gloo", device=0)
            dist.barrier()
        ok[rank] = 1
    finally:
        dist.destroy_process_group()


def test_emulated_mgtools_grad_and_curvature_world3(emu_exes, tmp_path):  # noqa: F811
    """torchrun ... -m peleanalysis_b200.mgtools grad|curvature transport=slab (gloo, emulated library) at world 3: header,
    box list and every value equal to the single-process executable's output"""
    from helpers import load_golden
    from peleanalysis_b200 import plotfile
    cases, ones = [], {}
    for tool, name in (("grad", "c3_three_levels"), ("grad", "mixed_boxes"), ("curvature", "c1_options"), ("curvature", "c3_threshold")):
        pf, z = load_golden(name)
        d = str(tmp_path / ("plt_" + name))
        if not os.path.exists(d):
            plotfile.write_plotfile(d, pf)
        args = _tool_args(tool, z)
        key = tool + "_" + name
        _run_tool(emu_exes[0 if tool == "grad" else 1], d, args + ["outfile=one"], str(tmp_path / key), 1)
        ones[key] = str(tmp_path / key / "one")
        cases.append((tool, d, args, str(tmp_path / key / "mg")))
    _spawn(_mgtool_worker, 3, str(tmp_path), cases)
    for tool, _, _, out in cases:
        key = os.path.basename(os.path.dirname(out))
        _same_plotfile(out, ones[key])
        assert _cell_files(out) <= {"Cell_D_00000", "Cell_D_00001", "Cell_D_00002"} and len(_cell_files(out)) >= 2
