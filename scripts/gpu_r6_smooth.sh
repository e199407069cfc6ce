#!/bin/bash
# one GPU session: build, smoke, GPU suite (the do_smooth tests among them), benchmark, do_smooth timing
#   bash scripts/gpu_r6_smooth.sh <output directory>
O=${1:?usage: $0 <output directory>}
mkdir -p "$O"
nvidia-smi -L > $O/gpus.txt 2>&1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv >> $O/gpus.txt 2>&1
timeout 900 python -c "import __graft_entry__ as g; g.build(); g.smoke(); print('smoke ok')" > $O/build_smoke.log 2>&1; echo "build+smoke rc=$?" >> $O/summary.txt
timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider > $O/pytest_gpu.log 2>&1; echo "pytest gpu rc=$?" >> $O/summary.txt
tail -3 $O/pytest_gpu.log >> $O/summary.txt
timeout 600 python bench.py --gpus 1 --steps 10 --warmup 3 > $O/bench_n1.json 2> $O/bench_n1.err; echo "bench rc=$?" >> $O/summary.txt
timeout 900 python scripts/smooth_time.py > $O/smooth_time.jsonl 2> $O/smooth_time.err; echo "smooth_time rc=$?" >> $O/summary.txt
cat $O/summary.txt
