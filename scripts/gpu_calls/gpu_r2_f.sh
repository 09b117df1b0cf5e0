#!/usr/bin/env bash
set -u
OUT=gpurun_out; mkdir -p $OUT
timeout 400 python -m pytest tests/test_gpu_kernels.py -m gpu -x -q > $OUT/pytest_f.log 2>&1; tail -3 $OUT/pytest_f.log
for k in 16 8 4 1; do
timeout 300 python bench.py --kernel tc --chains $k --steps 10 --warmup 3 --out $OUT/bench_f.jsonl > $OUT/bench_f_tc$k.log 2>&1; tail -1 $OUT/bench_f_tc$k.log | python -c "
import sys,json
d=json.loads(sys.stdin.readline()); c=d['config']; print(c['chains_per_eval'], round(d['value'],1), d['ms_per_step'], c['timed_seconds'], d['verified'], d['max_rel_err'])"
done
