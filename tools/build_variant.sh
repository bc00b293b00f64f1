#!/bin/bash
# A/B builds of the realignment library with extra -D flags (same ABI; select with LGR_LIBRARY=<file>).
# usage: tools/build_variant.sh NAME [-DFLAG ...]   →  lancet2_b200/csrc/variants/libNAME.so (git-ignored, travels with gpurun)
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
NAME=$1; shift
mkdir -p "$ROOT/lancet2_b200/csrc/variants"
C=$ROOT/lancet2_b200/csrc; H=$ROOT/lancet2_b200/host
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -shared -Xcompiler -fPIC "$@" \
  -o "$C/variants/lib$NAME.so" "$C/lgr_gpu.cu" "$C/lgr_format.o" "$C/lgr_repeat.cu" "$H/gpu_genotyper.cpp" "$H/gpu_repeat.cpp" "$H/adapter_capi.cpp" 2>&1 | grep -v "warning #" | grep -v "^$" || true
ls -la "$C/variants/lib$NAME.so"
