#!/bin/bash
# one GPU session: build, smoke, GPU suite, benchmark, multi-rank filter checks and scaling
#   bash scripts/gpu_r4_filter_ranks.sh <output directory>
O=${1:?usage: $0 <output directory>}
mkdir -p "$O"
nvidia-smi -L > $O/gpus.txt 2>&1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv >> $O/gpus.txt 2>&1
NG=$(nvidia-smi -L | wc -l)
timeout 900 python -c "import __graft_entry__ as g; g.build(); g.smoke(); print('smoke ok')" > $O/build_smoke.log 2>&1; echo "build+smoke rc=$?" >> $O/summary.txt
timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider > $O/pytest_gpu.log 2>&1; echo "pytest gpu rc=$?" >> $O/summary.txt
tail -3 $O/pytest_gpu.log >> $O/summary.txt
timeout 600 python bench.py --gpus 1 --steps 10 --warmup 3 > $O/bench_n1.json 2> $O/bench_n1.err; echo "bench rc=$?" >> $O/summary.txt
timeout 600 python bench.py --gpus 1 --steps 10 --warmup 3 --only-extra filter3 --no-cpu-baseline > $O/bench_filter3.json 2> $O/bench_filter3.err; echo "bench filter3 rc=$?" >> $O/summary.txt
for N in 1 2 4 8; do
  [ $N -le $NG ] || continue
  timeout 600 python -m torch.distributed.run --nproc-per-node $N --master-addr 127.0.0.1 --master-port $((29600+N)) scripts/filter_scale.py --steps 20 >> $O/filter_scale.jsonl 2>> $O/filter_scale.err; echo "scale N=$N rc=$?" >> $O/summary.txt
done
for N in 2 4 8; do
  [ $N -le $NG ] || continue
  timeout 600 python -m torch.distributed.run --nproc-per-node $N --master-addr 127.0.0.1 --master-port $((29700+N)) tests/dist_check_filter.py >> $O/dist_check_filter.log 2>&1; echo "dist_check_filter N=$N rc=$?" >> $O/summary.txt
done
for N in 1 8; do
  [ $N -le $NG ] || continue
  timeout 600 python -m torch.distributed.run --nproc-per-node $N --master-addr 127.0.0.1 --master-port $((29800+N)) scripts/filter_scale.py --base 512 --box 128 --mgs 128 --steps 5 >> $O/filter_scale_target.jsonl 2>> $O/filter_scale_target.err; echo "scale target N=$N rc=$?" >> $O/summary.txt
done
cat $O/summary.txt
