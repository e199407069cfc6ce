#!/usr/bin/env python3
"""Run under torchrun (one process per GPU): filterPlt on boxes spread over the ranks (pa_sfc_distribute), the FillPatch
sources of other ranks moved as NCCL send/recv of the packed slabs, every rank's boxes compared bit for bit with the NumPy
restatement for every filter type at one odd and one even filter-to-grid ratio.
  python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 tests/dist_check_filter.py"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from helpers import bit_equal  # noqa: E402
from oracle import filter_oracle as FO  # noqa: E402
from peleanalysis_b200 import capi, filterplt, synth  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    capi.init(dev)
    capi.set_stream(torch.cuda.current_stream().cuda_stream)
    pf = synth.config3(32, 16, names=("temp", "Y_CH4"))
    bad, n = [], 0
    for ftype in range(0, 11):
        for fgr in (3, 4):
            if ftype in (1, 2) and fgr % 2:
                continue
            kw = dict(filter_type=ftype, base_fgr=fgr, max_grid_size=8)
            _, ref, _ = FO.filter_plotfile(pf, **kw)
            R = filterplt.FilterRun(capi, pf, rank=rank, nranks=world, **kw)
            R.step()
            capi.sync()
            for l, ((rb, rf), got) in enumerate(zip(ref, R.result())):
                for b in R.hier.local_boxes[l]:
                    n += 1
                    if not bit_equal(got[b], rf[b]):
                        bad.append((ftype, fgr, l, b))
            dist.barrier()
    tot = torch.tensor([len(bad), n], device="cuda")
    dist.all_reduce(tot)
    if rank == 0:
        print("dist_check_filter world=%d: %d boxes checked, %d differ" % (world, int(tot[1]), int(tot[0])))
    dist.destroy_process_group()
    if int(tot[0]):
        print("rank %d: differing boxes %s" % (rank, bad[:10]))
        sys.exit(1)


if __name__ == "__main__":
    main()
