#!/bin/bash
# Build libmox.so variants for A/B runs: scripts/build_variant.sh NAME "-DMACRO ..."  ->  variants/NAME.so
# (same flags as the Makefile; the quoted switches are split into words; variants/ is scratch, git-ignored through *.so)
set -e
name=$1; shift
mkdir -p variants
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false -Xcompiler -fPIC,-Wall \
  -Iinclude -Iminimaloptix_b200/csrc -Iminimaloptix_b200/csrc/gpu --expt-relaxed-constexpr $@ \
  -shared -o variants/$name.so minimaloptix_b200/csrc/gpu/*.cu -lcudart 2>&1 | grep -E "error|spill|traverse_wideILb[01]ELb0ELb[01]E|Used" | grep -B0 -A2 "traverse_wideILb" | grep -E "spill|Used" || true
ls -la variants/$name.so
