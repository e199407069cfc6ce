#!/usr/bin/env python3
"""Run under torchrun (one process per GPU): grad and curvature through stencilrun.GradRun / CurvatureRun on boxes spread
over the ranks (pa_sfc_distribute), every cross-rank ghost source moved as NCCL send/recv of the packed slabs (nothing
peer-mapped), every rank's boxes compared bit for bit with the oracle: grad on every grad fixture and the mid-size
hierarchies, default-option curvature (two steps back to back) on the ratio-2 ones.
  python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29513 tests/dist_check_grad.py"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from cases import CASES  # noqa: E402
from helpers import bit_equal  # noqa: E402
from oracle import oracle as O  # noqa: E402
from peleanalysis_b200 import capi, stencilrun, synth  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    capi.init(dev)
    capi.set_stream(torch.cuda.current_stream().cuda_stream)
    hiers = [(n, b(), per, sym, tools) for n, (b, per, sym, tools, kw) in sorted(CASES.items()) if not kw]
    for case, kw in (("config3", dict(base=64, mgs=16)), ("config5", dict(base=16, mgs=8, ncomp=2, ratios=(2, 4, 2))), ("lshape", dict(base=32, mgs=16))):
        # the reference's curvature hard-codes ratio 2 (curvature.cpp:445,518): config5 (ratios 2, 4, 2) is a grad case only
        hiers.append((case, synth.CASES[case](**kw), (1, 1, 1), (0, 0, 0), ("grad",) if case == "config5" else ("grad", "curvature")))
    bad, n = [], 0
    for name, pf, is_per, sym, tools in hiers:
        OH = O.OracleHier(pf, is_per, sym)
        var = pf.names[0]
        s = OH.flatten(pf.comp(var))
        if "grad" in tools:
            R = stencilrun.GradRun(capi, pf, [var], is_per, sym, rank=rank, nranks=world)
            R.step()
            capi.sync()
            want = [OH.unflatten(g) for g in OH.grad(s)]
            for l, got in enumerate(R.result()):
                for b in R.hier.local_boxes[l]:
                    n += 1
                    if not all(bit_equal(got[b][c], want[c][l][b]) for c in range(4)):
                        bad.append(("grad", name, l, b))
            dist.barrier()
        if "curvature" in tools:
            o = capi.CurvOpts()
            o.prog_min, o.prog_max = float(s.min()), float(s.max())
            R = stencilrun.CurvatureRun(capi, pf, o, var, is_per, sym, rank=rank, nranks=world)
            R.step()
            R.step()
            capi.sync()
            want = [OH.unflatten(k) for k in OH.curvature(s, o.prog_min, o.prog_max)]
            for l, got in enumerate(R.result()):
                for b in R.hier.local_boxes[l]:
                    n += 1
                    if not all(bit_equal(got[b][c], want[c][l][b]) for c in range(5)):
                        bad.append(("curvature", name, l, b))
            dist.barrier()
    tot = torch.tensor([len(bad), n], device="cuda")
    dist.all_reduce(tot)
    if rank == 0:
        print("dist_check_grad world=%d: %d boxes checked, %d differ" % (world, int(tot[1]), int(tot[0])))
    dist.destroy_process_group()
    if int(tot[0]):
        print("rank %d: differing boxes %s" % (rank, bad[:10]))
        sys.exit(1)


if __name__ == "__main__":
    main()
