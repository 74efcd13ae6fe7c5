#!/bin/bash
# profiles/capture_ab.sh <tag> — one gpurun call on one B200:
#   1. GPU parity tests  2. the bench line (with e2e and the CPU baseline)  3. A/B of the product against the parent commit's
#      library and the switches of any experiment under trial (build them HERE first: bash profiles/build_prev.sh;
#      python -m rala_b200.build --variants)
#   4. ncu launch list of the same bench command  5. one `ncu --set full` capture of the kernels of one step
# Numbers printed under ncu are never bench values.
set -u
TAG=${1:-r01}
OUT=gpurun_out
mkdir -p $OUT
nvidia-smi --query-gpu=index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap --format=csv -lms 200 > $OUT/clocks_$TAG.csv &
SMI=$!
timeout 900 python -m pytest tests -m gpu -x -q > $OUT/pytest_gpu_$TAG.log 2>&1; echo "pytest rc=$?" >> $OUT/pytest_gpu_$TAG.log
tail -15 $OUT/pytest_gpu_$TAG.log | cut -c1-400
timeout 600 python bench.py > $OUT/bench_$TAG.json 2> $OUT/bench_$TAG.err; echo "bench rc=$?"
tail -3 $OUT/bench_$TAG.err | cut -c1-400
cat $OUT/bench_$TAG.json
timeout 600 python bench.py --ab --steps 100 > $OUT/ab_$TAG.json 2> $OUT/ab_$TAG.err; echo "ab rc=$?"
tail -3 $OUT/ab_$TAG.err | cut -c1-400
cat $OUT/ab_$TAG.json
kill $SMI
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file $OUT/launches_$TAG.csv \
    python bench.py --steps 2 --warmup 3 --no-cpu-baseline --skip-e2e > $OUT/bench_under_ncu_$TAG.log 2>&1
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --cache-control none --csv --log-file $OUT/launches_warm_$TAG.csv \
    python bench.py --steps 2 --warmup 3 --no-cpu-baseline --skip-e2e > $OUT/bench_under_ncu_warm_$TAG.log 2>&1
timeout 900 ncu --set full --clock-control none --import-source on \
    -k regex:'k_classify_events|k_classify_survivors|k_relocate_runs|k_transitive_group|k_transitive_light|k_resolve$|k_fill_csr|k_emit_edges' -s ${2:-18} -c ${3:-9} \
    -o $OUT/prof_$TAG -f python bench.py --steps 1 --warmup 3 --no-cpu-baseline --skip-e2e > $OUT/ncu_full_$TAG.log 2>&1
tail -2 $OUT/ncu_full_$TAG.log | cut -c1-300
ls -la $OUT
