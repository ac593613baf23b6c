#!/bin/bash
# one GPU doing the work of one rank of an 8-GPU run: ms/step for each library given as "name:lib" (ideal = full-frame ms / 8)
mkdir -p gpurun_out
for v in $VARIANTS; do
  name=${v%%:*}; lib=${v#*:}
  if [ "$lib" = "default" ]; then unset MOX_GPU_LIB; else export MOX_GPU_LIB=$PWD/$lib; fi
  timeout 600 python bench.py --steps ${STEPS:-20} --warmup 3 --no-cpu-baseline --emulate-world ${EW:-8} > gpurun_out/em_$name.json 2> gpurun_out/em_$name.err || tail -5 gpurun_out/em_$name.err
  python scripts/show_bench.py gpurun_out/em_$name.json $name
done
