#!/bin/bash
# One GPU-box session: parity tests, both bench arms, the ncu launch list of bench.py and one --set full capture of the
# step's kernels.  Every ncu pass runs only after the same command has exited 0 without ncu.  Outputs: gpurun_out/.
#   gpurun --timeout 2400 -- 'bash tools/gpu_round.sh [tag]'
set -u
TAG=${1:-r2}
OUT=gpurun_out/$TAG
mkdir -p $OUT
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm --format=csv > $OUT/gpu.txt 2>&1

if [ "${SKIP_TESTS:-0}" != "1" ]; then
  timeout 1200 python -m pytest tests -m gpu -x -q > $OUT/pytest.log 2>&1
  echo "pytest rc=$?" >> $OUT/pytest.log
  tail -3 $OUT/pytest.log
fi

timeout 900 python bench.py > $OUT/bench.json 2> $OUT/bench.err; echo "bench rc=$?"
timeout 600 python bench.py --impl reference > $OUT/bench_ref.json 2> $OUT/bench_ref.err; echo "bench_ref rc=$?"
tail -c 1500 $OUT/bench.json

if [ "${SKIP_NCU:-0}" != "1" ]; then
  # launch list of the bench command (short timed regions: a profiling run, its numbers are never bench values)
  timeout 300 python bench.py --steps 2 --warmup 3 > $OUT/bench_short.json 2> $OUT/bench_short.err; rc=$?; echo "short bench rc=$rc"
  if [ $rc -eq 0 ]; then
    timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 4000 --csv --log-file $OUT/launches.csv \
      python bench.py --steps 2 --warmup 3 > $OUT/ncu_launch.log 2>&1; echo "ncu launches rc=$?"
    for W in sph_dg cu_dg; do
      timeout 900 ncu --set full --clock-control none --import-source on -s 40 -c 14 \
        -k regex:'vox_front|knn3_warp|ppf_gather_packed|vox_fill|devox|split6' -o $OUT/full_$W -f \
        python bench.py --only --workload $W --steps 2 --warmup 3 > $OUT/ncu_full_$W.log 2>&1; echo "ncu full $W rc=$?"
      ncu -i $OUT/full_$W.ncu-rep --page raw --csv > $OUT/full_$W.csv 2>/dev/null
    done
  fi
fi
ls -la $OUT
