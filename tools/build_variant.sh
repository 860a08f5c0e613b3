#!/bin/bash
# Developer tool: build an instrumented copy of the library into tools/variants/ (git-ignored, travels with gpurun).
#   tools/build_variant.sh tl -DTRQ_STAGE_TIMELINE        ->  tools/variants/libtracer_rq_tl.so   (use with TRQ_LIB=...)
#   tools/build_variant.sh stats -DTRQ_STATS
#   tools/build_variant.sh tail -DTRQ_TAIL_TIMELINE       ->  per-CTA start / queue-exhausted / exit stamps (tools/tail_probe.py)
#   tools/build_variant.sh nopdl -DTRQ_NO_PDL             ->  every trace waits for the previous kernel (tools/pdl_ab.py)
# TRQ_VARIANT_DIR=<dir> puts the library (and its objects) there instead.
set -e
NAME=$1; shift
ROOT=$(cd "$(dirname "$0")/.." && pwd)
C=$ROOT/tracer_b200/csrc
OUT=${TRQ_VARIANT_DIR:-$ROOT/tools/variants}
B=$OUT/build_$NAME
mkdir -p $B
NV="/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-ffp-contract=off,-fno-fast-math --expt-relaxed-constexpr $*"
make -s -C $C >/dev/null
(cd $C && $NV -c trq_api.cu -o $B/trq_api.o && $NV -c bvh_build_gpu.cu -o $B/bvh_build_gpu.o)
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $OUT/libtracer_rq_$NAME.so $B/trq_api.o $B/bvh_build_gpu.o $C/build/bvh_build.o $C/build/morton_build.o $C/build/harness.o $C/build/error.o -lpthread
echo built $OUT/libtracer_rq_$NAME.so
