#!/bin/bash
# one GPU session: build, smoke, GPU suite (the multigrid do_smooth tests among them), benchmark with its output fingerprint,
# do_smooth timing of both preconditioners at smoothing_time 1e-7, 1e-5, 1e-4, 1e-3 and one profiled solve of each
#   bash scripts/gpu_r7_smooth_mg.sh <output directory>
O=${1:?usage: $0 <output directory>}
mkdir -p "$O"
nvidia-smi -L > $O/gpus.txt 2>&1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv >> $O/gpus.txt 2>&1
timeout 900 python -c "import __graft_entry__ as g; g.build(); g.smoke(); print('smoke ok')" > $O/build_smoke.log 2>&1; echo "build+smoke rc=$?" >> $O/summary.txt
timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider > $O/pytest_gpu.log 2>&1; echo "pytest gpu rc=$?" >> $O/summary.txt
tail -3 $O/pytest_gpu.log >> $O/summary.txt
timeout 600 python bench.py --gpus 1 --steps 10 --warmup 3 > $O/bench_n1.json 2> $O/bench_n1.err; echo "bench rc=$?" >> $O/summary.txt
python -c "import json,sys; d=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); print('bench output_hash', d['output_hash'])" $O/bench_n1.json >> $O/summary.txt 2>&1
timeout 1200 python scripts/smooth_time.py --times 1e-7 1e-5 1e-4 1e-3 --precond jacobi mg > $O/smooth_time.jsonl 2> $O/smooth_time.err; echo "smooth_time rc=$?" >> $O/summary.txt
timeout 600 python scripts/smooth_time.py --times 1e-5 --precond jacobi mg --repeats 1 --profile > $O/smooth_profile.jsonl 2> $O/smooth_profile.err; echo "smooth_profile rc=$?" >> $O/summary.txt
cat $O/summary.txt
