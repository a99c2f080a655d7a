#!/bin/bash
# round 2: the measurements BENCH.md / profiles/ quote, one GPU, written to build/r2_final/.  tools/r2_final.sh [quick]
set -u
cd "$(dirname "$0")/.."
OUT=build/r2_final
mkdir -p $OUT
NCU="ncu --set full --import-source on --clock-control none -k regex:solve_kernel -s 1 -c 1"
for wl in static4096 mixed4096; do
  timeout 600 $NCU -o $OUT/r2_final_$wl -f python tools/profile_run.py $wl 2 > $OUT/r2_final_ncu_$wl.log 2>&1; echo "ncu $wl rc $?"
  grep EVALS_PER_LAUNCH $OUT/r2_final_ncu_$wl.log
done
timeout 900 $NCU -o $OUT/r2_final_dynamic2048 -f python tools/profile_run.py dynamic8192 2 2048 > $OUT/r2_final_ncu_dynamic2048.log 2>&1; echo "ncu dyn rc $?"
grep EVALS_PER_LAUNCH $OUT/r2_final_ncu_dynamic2048.log
# launch list of the bench command (serialised by the profiler: shares, not durations)
CUDA_LAUNCH_BLOCKING=1 timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $OUT/r2_launches_bench.csv python bench.py --steps 4 --warmup 3 --no-cpu-baseline > $OUT/r2_bench_under_ncu.log 2>&1; echo "launch list rc $?"
python bench.py > $OUT/r2_bench_static4096.json 2> $OUT/r2_bench_static4096.err; echo "bench rc $?"; tail -c 400 $OUT/r2_bench_static4096.json
python bench.py --impl reference --steps 5 --warmup 1 > $OUT/r2_bench_reference.json 2>/dev/null; tail -c 300 $OUT/r2_bench_reference.json
python tools/parity_report.py --gpu --n 512 --n-dynamic 96 --out $OUT/r2_parity_distribution_gpu.json > $OUT/r2_parity_gpu.md 2>&1; tail -8 $OUT/r2_parity_gpu.md
python tools/bench_qnet.py > $OUT/r2_qnet.json 2>/dev/null; cat $OUT/r2_qnet.json
python tools/single_latency.py > $OUT/r2_single_latency.txt 2>/dev/null; cat $OUT/r2_single_latency.txt
python tools/bench_fleet.py 4096 2>/dev/null > $OUT/r2_fleet.json; python tools/bench_fleet.py 16384 2>/dev/null >> $OUT/r2_fleet.json; cut -c1-300 $OUT/r2_fleet.json
python tools/bench_hybrid.py 2>/dev/null > $OUT/r2_hybrid.json; cut -c1-400 $OUT/r2_hybrid.json
