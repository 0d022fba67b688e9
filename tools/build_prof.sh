#!/usr/bin/env bash
# Builds gpurun_out-free profiling variant libbgg_b200_prof.so: identical sources, k_ipm compiled with -DBGG_IPM_PROF
# (per-phase clock64 accumulation by thread 0 of CTA 0).  Used only by tools/profile_phases.py.
set -euo pipefail
cd "$(dirname "$0")/../bilevel-gait-gen_b200"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
ARCH="-gencode arch=compute_100a,code=sm_100a"
COMMON="-O3 -std=c++17 -lineinfo -Xcompiler -fPIC --expt-relaxed-constexpr"
$NVCC $ARCH $COMMON -DBGG_IPM_PROF ${EXTRA:-} -maxrregcount=128 -dc -o build/bgg_ipm_prof.o csrc/bgg_ipm.cu
$NVCC $ARCH -shared -o libbgg_b200_prof.so build/bgg_prepare.o build/bgg_condense.o build/bgg_ipm_prof.o build/bgg_finish.o build/bgg_assemble.o build/bgg_gradient.o build/bgg_gait.o build/bgg_qp.o build/bgg_qp_adjoint.o build/bgg_ik.o build/bgg_partials.o build/bgg_capi.o -lcudart
echo built libbgg_b200_prof.so
