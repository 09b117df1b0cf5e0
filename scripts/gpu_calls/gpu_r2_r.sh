#!/usr/bin/env bash
# final kernels (early loads, every-CTA-had-theta rule): launch list + one full ncu capture per tensor-core kernel
set -u
OUT=gpurun_out; mkdir -p $OUT
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:fed_ -c 40 --csv --log-file $OUT/launches_r2.csv \
    python bench.py --shards 2 --steps 3 --warmup 3 > $OUT/ncu_launches_r2.log 2>&1
timeout 900 ncu --set full --clock-control none --import-source on -k regex:fed_glm_tc -s 4 -c 1 -f -o $OUT/prof_tc_r2_final \
    python bench.py --shards 2 --steps 2 --warmup 3 > $OUT/ncu_tc_r2.log 2>&1; tail -2 $OUT/ncu_tc_r2.log
timeout 900 ncu --set full --clock-control none --import-source on -k regex:fed_glm_fp8 -s 4 -c 1 -f -o $OUT/prof_fp8_r2_final \
    python bench.py --config fp8 --shards 2 --steps 2 --warmup 3 > $OUT/ncu_fp8_r2.log 2>&1; tail -2 $OUT/ncu_fp8_r2.log
ls -la $OUT/*.ncu-rep
timeout 300 python bench.py --config fp8 --steps 30 --warmup 5 --out $OUT/bench_r.jsonl > $OUT/bench_r_fp8.log 2>&1; tail -1 $OUT/bench_r_fp8.log | cut -c1-160
timeout 300 python bench.py --steps 30 --warmup 5 --out $OUT/bench_r.jsonl > $OUT/bench_r_glm.log 2>&1; tail -1 $OUT/bench_r_glm.log | cut -c1-160
