#!/bin/bash
# one GPU session: build, smoke, GPU suite, benchmark, grad / curvature scaling over the packed-slab transport and, where the
# box has several GPUs, tests/dist_check_grad.py
#   bash scripts/gpu_r5_stencil_ranks.sh <output directory>
O=${1:?usage: $0 <output directory>}
mkdir -p "$O"
nvidia-smi -L > $O/gpus.txt 2>&1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv >> $O/gpus.txt 2>&1
NG=$(nvidia-smi -L | wc -l)
timeout 900 python -c "import __graft_entry__ as g; g.build(); g.smoke(); print('smoke ok')" > $O/build_smoke.log 2>&1; echo "build+smoke rc=$?" >> $O/summary.txt
timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider > $O/pytest_gpu.log 2>&1; echo "pytest gpu rc=$?" >> $O/summary.txt
tail -3 $O/pytest_gpu.log >> $O/summary.txt
timeout 600 python bench.py --gpus 1 --steps 10 --warmup 3 > $O/bench_n1.json 2> $O/bench_n1.err; echo "bench rc=$?" >> $O/summary.txt
for N in 1 2 4 8; do
  if [ $N -gt $NG ]; then echo "stencil_scale N=$N not measured: $NG GPU(s) in the box" >> $O/summary.txt; continue; fi
  timeout 600 python -m torch.distributed.run --nproc-per-node $N --master-addr 127.0.0.1 --master-port $((29600+N)) scripts/stencil_scale.py --steps 100 --repeats 5 >> $O/stencil_scale.jsonl 2>> $O/stencil_scale.err; echo "stencil_scale N=$N rc=$?" >> $O/summary.txt
done
for N in 2 4 8; do
  [ $N -le $NG ] || continue
  timeout 600 python -m torch.distributed.run --nproc-per-node $N --master-addr 127.0.0.1 --master-port $((29700+N)) tests/dist_check_grad.py >> $O/dist_check_grad.log 2>&1; echo "dist_check_grad N=$N rc=$?" >> $O/summary.txt
done
cat $O/summary.txt
