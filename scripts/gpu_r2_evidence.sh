#!/usr/bin/env bash
# Round-2 evidence on ONE GPU: full GPU test suite, smoke, chain sweep, secondary configs, batching over gRPC,
# launch list and ncu captures of the two tensor-core kernels.
set -u
OUT=gpurun_out; mkdir -p $OUT
timeout 900 python -m pytest tests -m gpu -q > $OUT/pytest_gpu_r2.log 2>&1; tail -4 $OUT/pytest_gpu_r2.log
timeout 300 python __graft_entry__.py --smoke > $OUT/smoke_r2.log 2>&1; tail -4 $OUT/smoke_r2.log
for k in 4 8 16; do
  timeout 300 python bench.py --kernel tc --chains $k --steps 10 --warmup 3 --out $OUT/bench_n1_tc_chains_r2.jsonl > $OUT/bench_ev_c$k.log 2>&1; tail -1 $OUT/bench_ev_c$k.log | cut -c1-160
done
timeout 300 python bench.py --kernel simt --steps 10 --warmup 3 --out $OUT/bench_n1_simt_r2.jsonl > $OUT/bench_ev_simt.log 2>&1; tail -1 $OUT/bench_ev_simt.log | cut -c1-160
timeout 300 python bench.py --config ode --steps 30 --warmup 5 --shards 4 --out $OUT/configs_r2_n1.jsonl > $OUT/bench_ev_ode.log 2>&1; tail -1 $OUT/bench_ev_ode.log | cut -c1-160
timeout 300 python bench.py --config linreg --steps 200 --warmup 20 --out $OUT/configs_r2_n1.jsonl > $OUT/bench_ev_linreg.log 2>&1; tail -1 $OUT/bench_ev_linreg.log | cut -c1-160
timeout 300 python bench.py --config fp8 --steps 30 --warmup 5 --out $OUT/configs_r2_n1.jsonl > $OUT/bench_ev_fp8.log 2>&1; tail -1 $OUT/bench_ev_fp8.log | cut -c1-160
timeout 300 python bench.py --steps 30 --warmup 5 --out $OUT/configs_r2_n1.jsonl > $OUT/bench_ev_glm.log 2>&1; tail -1 $OUT/bench_ev_glm.log | cut -c1-160
timeout 300 python bench.py --impl nccl --steps 10 --warmup 3 --out $OUT/configs_r2_n1.jsonl > $OUT/bench_ev_nccl.log 2>&1; tail -1 $OUT/bench_ev_nccl.log | cut -c1-160
timeout 600 python benchmarks/bench_batching_gpu.py --chains 8 16 --evals 300 --out $OUT/batching_gpu_r2.jsonl > $OUT/batching_ev.log 2>&1; tail -4 $OUT/batching_ev.log | cut -c1-330
timeout 600 python benchmarks/bench_configs.py --out $OUT/configs_misc_r2.jsonl > $OUT/bench_configs_ev.log 2>&1; tail -3 $OUT/bench_configs_ev.log | cut -c1-300
# every launch with its device time, then one full capture per tensor-core kernel
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:fed_ -c 40 --csv --log-file $OUT/launches_r2.csv \
    python bench.py --shards 2 --steps 3 --warmup 3 > $OUT/ncu_launches_r2.log 2>&1
timeout 900 ncu --set full --clock-control none --import-source on -k regex:fed_glm_tc -s 4 -c 1 -f -o $OUT/prof_tc_r2_final \
    python bench.py --shards 2 --steps 2 --warmup 3 > $OUT/ncu_tc_r2.log 2>&1; tail -2 $OUT/ncu_tc_r2.log
timeout 900 ncu --set full --clock-control none --import-source on -k regex:fed_glm_fp8 -s 4 -c 1 -f -o $OUT/prof_fp8_r2_final \
    python bench.py --config fp8 --shards 2 --steps 2 --warmup 3 > $OUT/ncu_fp8_r2.log 2>&1; tail -2 $OUT/ncu_fp8_r2.log
ls -la $OUT/*.ncu-rep
