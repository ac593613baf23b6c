#!/bin/bash
# round 2 A/B: tests on the new library, then the bench for each library given as "name:lib"
mkdir -p gpurun_out
if [ "$RUN_TESTS" != "0" ]; then
timeout 1500 python -m pytest tests -m gpu -q --timeout 600 -x 2>&1 | tail -25 > gpurun_out/ab_tests.log; tail -25 gpurun_out/ab_tests.log
fi
for v in $VARIANTS; do
  name=${v%%:*}; lib=${v#*:}
  if [ "$lib" = "default" ]; then unset MOX_GPU_LIB; else export MOX_GPU_LIB=$PWD/$lib; fi
  timeout 600 python bench.py --steps ${STEPS:-6} --warmup 3 --no-cpu-baseline > gpurun_out/ab_$name.json 2> gpurun_out/ab_$name.err || tail -5 gpurun_out/ab_$name.err
  python scripts/show_bench.py gpurun_out/ab_$name.json $name
done
