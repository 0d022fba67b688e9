#!/usr/bin/env bash
# Builds libbgg_b200_trace.so: identical sources, k_ipm compiled with -DBGG_IPM_TRACE (one armed CTA records every
# interior-point iteration, csrc/bgg_ipm_trace.cuh).  Needs the objects of bilevel-gait-gen_b200/build.sh.  Used by
# tests/test_gpu_ipm_trace.py, which builds its own copy when nvcc is present.
# OUT=<path> puts the library elsewhere (default: next to libbgg_b200.so).
set -euo pipefail
cd "$(dirname "$0")/../bilevel-gait-gen_b200"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
ARCH="-gencode arch=compute_100a,code=sm_100a"
COMMON="-O3 -std=c++17 -lineinfo -Xcompiler -fPIC --expt-relaxed-constexpr"
OUT=${OUT:-$(pwd)/libbgg_b200_trace.so}
OBJ=$(mktemp -d)
trap 'rm -rf "$OBJ"' EXIT
$NVCC $ARCH $COMMON -DBGG_IPM_TRACE -maxrregcount=128 -dc -o "$OBJ/bgg_ipm_trace.o" csrc/bgg_ipm.cu
$NVCC $ARCH -shared -o "$OUT" build/bgg_prepare.o build/bgg_condense.o "$OBJ/bgg_ipm_trace.o" build/bgg_finish.o build/bgg_assemble.o build/bgg_gradient.o build/bgg_gait.o build/bgg_qp.o build/bgg_qp_adjoint.o build/bgg_ik.o build/bgg_partials.o build/bgg_capi.o -lcudart
echo "built $OUT"
