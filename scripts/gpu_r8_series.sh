#!/bin/bash
# one GPU session: build, smoke, GPU suite (the plotfile-series tests among them), benchmark with its output fingerprint,
# and the series wall-time measurement (scripts/series_walltime.py, K = 8 files of 3 x 256^3 cells)
#   bash scripts/gpu_r8_series.sh <output directory>
O=${1:?usage: $0 <output directory>}
mkdir -p "$O"
nvidia-smi -L > $O/gpus.txt 2>&1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv >> $O/gpus.txt 2>&1
timeout 900 python -c "import __graft_entry__ as g; g.build(); g.smoke(); print('smoke ok')" > $O/build_smoke.log 2>&1; echo "build+smoke rc=$?" >> $O/summary.txt
timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider > $O/pytest_gpu.log 2>&1; echo "pytest gpu rc=$?" >> $O/summary.txt
tail -3 $O/pytest_gpu.log >> $O/summary.txt
timeout 600 python bench.py --gpus 1 --steps 10 --warmup 3 > $O/bench_n1.json 2> $O/bench_n1.err; echo "bench rc=$?" >> $O/summary.txt
python -c "import json,sys; d=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); print('bench output_hash', d['output_hash'])" $O/bench_n1.json >> $O/summary.txt 2>&1
timeout 1500 python scripts/series_walltime.py 256 8 > $O/series_walltime.jsonl 2> $O/series_walltime.err; echo "series_walltime rc=$?" >> $O/summary.txt
cat $O/summary.txt
