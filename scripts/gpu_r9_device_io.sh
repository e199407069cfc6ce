#!/bin/bash
# one GPU session: build, smoke, the device-memory entry point tests, their timing (scripts/device_io_time.py), the
# benchmark with its output fingerprint, then the rest of the GPU suite
#   bash scripts/gpu_r9_device_io.sh <output directory>
O=${1:?usage: $0 <output directory>}
mkdir -p "$O"
nvidia-smi -L > $O/gpus.txt 2>&1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv >> $O/gpus.txt 2>&1
timeout 900 python -c "import __graft_entry__ as g; g.build(); g.smoke(); print('smoke ok')" > $O/build_smoke.log 2>&1; echo "build+smoke rc=$?" >> $O/summary.txt
grep -A3 k_array4_copy peleanalysis_b200/lib/build.log > $O/ptxas_array4.txt 2>&1
timeout 900 python -m pytest tests/test_gpu_device_io.py -q -m gpu -p no:cacheprovider > $O/pytest_device_io.log 2>&1; echo "pytest device_io rc=$?" >> $O/summary.txt
tail -3 $O/pytest_device_io.log >> $O/summary.txt
timeout 900 python scripts/device_io_time.py --out $O/r09_device_io.jsonl > $O/device_io_time.log 2>&1; echo "device_io_time rc=$?" >> $O/summary.txt
timeout 600 python bench.py --gpus 1 --steps 10 --warmup 3 > $O/bench_n1.json 2> $O/bench_n1.err; echo "bench rc=$?" >> $O/summary.txt
python -c "import json,sys; d=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); print('bench output_hash', d['output_hash'])" $O/bench_n1.json >> $O/summary.txt 2>&1
if [ "${FULL:-1}" = 1 ]; then
timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider --deselect tests/test_gpu_device_io.py > $O/pytest_gpu.log 2>&1; echo "pytest gpu rc=$?" >> $O/summary.txt
tail -3 $O/pytest_gpu.log >> $O/summary.txt
fi
cat $O/summary.txt
