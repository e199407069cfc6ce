"""grad and curvature with every cross-rank ghost source moved as a packed slab, on B200s: the runners on one rank are the
plain C-ABI calls (no exchange, no extra launch); on two GPUs grad3d.b200.ex / curvature3d.b200.ex ngpus=2 transport=slab
(device-to-device slab copies, nothing peer-mapped) equal the C oracle cell for cell on the full-size hierarchies of the
one-GPU parity tests, and tests/dist_check_grad.py passes under torchrun (NCCL)."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from helpers import bit_equal, load_golden, max_rel
from oracle import oracle as O
from peleanalysis_b200 import plotfile, stencilrun
from test_gpu_tools import _big_tmp, _flat, _ngpus, _run, exes  # noqa: F401  (exes: module-scoped fixture, the host shells)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
two_gpus = pytest.mark.skipif(_ngpus() < 2, reason="needs two GPUs in one box")


def np_concat(arrs):
    return np.concatenate([a.ravel() for a in arrs])


def test_stencil_runners_on_one_rank_are_the_plain_calls(gpu):
    P = gpu
    pf, z = load_golden("c3_three_levels")
    R = stencilrun.GradRun(P, pf, ["temp"])
    assert R.exchange is None
    n0 = P.kernel_launches()
    R.step()
    n1 = P.kernel_launches()
    P.grad(R.fin, 0, 1, R.fout, 0)
    assert P.kernel_launches() - n1 == n1 - n0
    P.sync()
    res = R.result()
    for c, k in enumerate(["gx", "gy", "gz", "mag"]):
        got = [f for lv in res for f in lv]
        assert bit_equal(np_concat([g[c] for g in got]), z["grad_" + k]), k
    o = P.CurvOpts()
    o.prog_min, o.prog_max = float(z["prog_min"]), float(z["prog_max"])
    C = stencilrun.CurvatureRun(P, pf, o)
    assert C.op is None
    C.step()
    P.sync()
    res = C.result()
    for c, n in enumerate(["Progress", "MeanCurvature_temp", "FlameNormalX_temp", "FlameNormalY_temp", "FlameNormalZ_temp"]):
        assert bit_equal(np_concat([f[c] for lv in res for f in lv]), z["curv_" + n]), n


@two_gpus
def test_full_size_grad_on_two_gpus_slab_transport(exes):  # noqa: F811
    """BASELINE configs[1] (uniform 512^3 in 128^3 boxes) and the north-star hierarchy (3 levels, 512^3 base, 128^3 boxes)
    at full size through grad3d.b200.ex ngpus=2 transport=slab: every output bit equals the oracle's"""
    from peleanalysis_b200 import synth
    for pf in (synth.make_hierarchy(512, [], [], 128, ("temp",)), synth.config3(512, 128)):
        with _big_tmp() as tmp:
            d = os.path.join(tmp, "plt")
            plotfile.write_plotfile(d, pf)
            OH = O.OracleHier(pf)
            want = OH.grad(OH.flatten(pf.comp("temp")))
            del pf, OH
            _run(exes[0], "infile=" + d, "gradVar=temp", "ngpus=2", "transport=slab", "outfile=" + os.path.join(tmp, "b200"), cwd=tmp)
            for c, n in enumerate(["temp_gx", "temp_gy", "temp_gz", "||gradtemp||"]):
                got = _flat(plotfile.read_plotfile(os.path.join(tmp, "b200"), comps=[n]), n)
                assert bit_equal(got, want[c]), (n, max_rel(got, want[c]))
            del want


@two_gpus
def test_full_size_curvature_on_two_gpus_slab_transport(exes):  # noqa: F811
    """BASELINE configs[2] at full size (3 levels, 256^3 base, ratio 2, 64^3 boxes) through curvature3d.b200.ex ngpus=2
    transport=slab, default options and threshold_prog: every output the reference initialises, bit for bit with the oracle"""
    from peleanalysis_b200 import synth
    pf = synth.config3(256, 64)
    names = ["Progress", "MeanCurvature_temp", "FlameNormalX_temp", "FlameNormalY_temp", "FlameNormalZ_temp"]
    with _big_tmp() as tmp:
        d = os.path.join(tmp, "plt")
        plotfile.write_plotfile(d, pf)
        OH = O.OracleHier(pf)
        s = OH.flatten(pf.comp("temp"))
        pmin, pmax = plotfile.file_min_max(d, "temp", len(pf.levels))
        del pf
        for k, (extra, thr) in enumerate((([], False), (["threshold_prog=1", "threshold_value=0.01"], True))):
            want = OH.curvature(s, pmin, pmax, do_threshold=thr, threshold=0.01)
            out = os.path.join(tmp, "b200_%d" % k)
            _run(exes[1], "infile=" + d, "progressName=temp", "ngpus=2", "transport=slab", "outfile=" + out, *extra, cwd=tmp)
            a = plotfile.read_plotfile(out, comps=names)
            for c, n in enumerate(names):
                assert bit_equal(_flat(a, n), want[c]), (extra, n, max_rel(_flat(a, n), want[c]))
            del want, a
            shutil.rmtree(out)


@two_gpus
def test_dist_check_grad_on_two_gpus(gpu):
    env = dict(os.environ, PYTHONPATH=ROOT)
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29534", os.path.join(ROOT, "tests", "dist_check_grad.py")], capture_output=True, text=True, env=env)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "0 differ" in p.stdout
