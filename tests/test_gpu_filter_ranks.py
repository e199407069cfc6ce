"""filterPlt on several ranks, on B200s: the FillPatch exchange entries on one rank (offsets zero, pack / mark do nothing),
and on two GPUs filterPlt3d.b200.ex ngpus=2 (device-to-device slab copies) and `mgtools filter` under torchrun (NCCL)
bit-identical to the one-GPU tool."""
import os
import subprocess
import sys

import pytest

from helpers import load_golden
from peleanalysis_b200 import filterplt, plotfile, synth
from test_fill_patch_exchange import _same_plotfile, _tool_args
from test_gpu_tools import exes  # noqa: F401  (module-scoped fixture: the host shells, built with make)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_fill_patch_exchange_on_one_rank_is_empty(gpu):
    P = gpu
    pf, z = load_golden("filter_c3")
    R = filterplt.FilterRun(P, pf, max_grid_size=8)
    for l in range(R.nlev):
        sp, rp, so, ro = P.fill_patch_exchange_buffers(R.fin, R.ncomp, l, R.ngrow[l], 1)
        assert so == [0, 0] and ro == [0, 0]
        n0 = P.kernel_launches()
        P.fill_patch_pack(R.fin, 0, R.ncomp, l, R.ngrow[l], 1)
        P.fill_patch_mark_received(R.fin, 0, R.ncomp, l, R.ngrow[l], 1)
        assert P.kernel_launches() == n0
    assert R.exchanges == []


def _cases(tmp):
    pf, z = load_golden("filter_c3")
    d1 = os.path.join(tmp, "plt_c3")
    plotfile.write_plotfile(d1, pf)
    big = synth.config3(128, 64)
    d2 = os.path.join(tmp, "plt_big")
    plotfile.write_plotfile(d2, big)
    return [(d1, _tool_args(z)), (d2, ["max_grid_size=32"])]


def test_filter_tools_on_two_gpus(gpu, exes, tmp_path):  # noqa: F811
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    for d, args in _cases(str(tmp_path)):
        root = os.path.basename(d)
        runs = {}
        for tag, extra in (("one", []), ("two", ["ngpus=2"])):
            cwd = tmp_path / (tag + root)
            cwd.mkdir()
            p = subprocess.run([exes[2], "infile=" + d] + args + extra, capture_output=True, text=True, cwd=str(cwd))
            assert p.returncode == 0, p.stdout + p.stderr
            runs[tag] = str(cwd / (root + "_filtered"))
        _same_plotfile(runs["two"], runs["one"])
        cwd = tmp_path / ("mg" + root)
        cwd.mkdir()
        env = dict(os.environ, PYTHONPATH=ROOT)
        p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                            "--master-port", "29533", "-m", "peleanalysis_b200.mgtools", "filter", "infile=" + d] + args,
                           capture_output=True, text=True, cwd=str(cwd), env=env)
        assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
        _same_plotfile(str(cwd / (root + "_filtered")), runs["one"])
