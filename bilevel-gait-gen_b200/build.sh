#!/usr/bin/env bash
# Builds libbgg_b200.so (the C-ABI library of include/bgg.h) in-tree for sm_100a.
set -euo pipefail
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
ARCH="-gencode arch=compute_100a,code=sm_100a"
COMMON="-O3 -std=c++17 -lineinfo -Xcompiler -fPIC --expt-relaxed-constexpr -Xptxas -v"
mkdir -p build
# bgg_prepare.cu is compiled without FMA contraction so that exact zeros stay exact (sparsity parity).
$NVCC $ARCH $COMMON -fmad=false -dc -o build/bgg_prepare.o csrc/bgg_prepare.cu 2> build/ptxas_prepare.log
$NVCC $ARCH $COMMON -fmad=false -dc -o build/bgg_condense.o csrc/bgg_condense.cu 2> build/ptxas_condense.log
# chol::factor / chol::solve are __noinline__: cap their registers at the kernel's 2-CTAs-per-SM bound
$NVCC $ARCH $COMMON -maxrregcount=128 -dc -o build/bgg_ipm.o csrc/bgg_ipm.cu 2> build/ptxas_ipm.log
$NVCC $ARCH $COMMON -fmad=false -dc -o build/bgg_finish.o csrc/bgg_finish.cu 2> build/ptxas_finish.log
$NVCC $ARCH $COMMON -fmad=false -dc -o build/bgg_assemble.o csrc/bgg_assemble.cu 2> build/ptxas_assemble.log
$NVCC $ARCH $COMMON -dc -o build/bgg_gradient.o csrc/bgg_gradient.cu 2> build/ptxas_gradient.log
$NVCC $ARCH $COMMON -dc -o build/bgg_gait.o csrc/bgg_gait.cu 2> build/ptxas_gait.log
$NVCC $ARCH $COMMON -dc -o build/bgg_qp.o csrc/bgg_qp.cu 2> build/ptxas_qp.log
$NVCC $ARCH $COMMON -dc -o build/bgg_qp_adjoint.o csrc/bgg_qp_adjoint.cu 2> build/ptxas_qp_adjoint.log
$NVCC $ARCH $COMMON -dc -o build/bgg_ik.o csrc/bgg_ik.cu 2> build/ptxas_ik.log
$NVCC $ARCH $COMMON -fmad=false -dc -o build/bgg_partials.o csrc/bgg_partials.cu 2> build/ptxas_partials.log
$NVCC $ARCH $COMMON -fmad=false -dc -o build/bgg_capi.o csrc/bgg_capi.cu 2> build/ptxas_capi.log
$NVCC $ARCH -shared -o libbgg_b200.so build/bgg_prepare.o build/bgg_condense.o build/bgg_ipm.o build/bgg_finish.o build/bgg_assemble.o build/bgg_gradient.o build/bgg_gait.o build/bgg_qp.o build/bgg_qp_adjoint.o build/bgg_ik.o build/bgg_partials.o build/bgg_capi.o -lcudart
# host shim: the reference's C++ call surface over the C ABI (no CUDA in these translation units) and its test driver
CXX=${CXX:-g++}
$CXX -O2 -std=c++17 -Wall -fPIC -shared -o libmpc_b200.so host/mpc_b200.cpp host/mpc_controller_b200.cpp host/urdf_consts.cpp host/config_parser.cpp -L. -lbgg_b200 -Wl,-rpath,'$ORIGIN'
$CXX -O2 -std=c++17 -Wall -Ihost -o ../tests/cpp/test_shim ../tests/cpp/test_shim.cpp -L. -lmpc_b200 -lbgg_b200 -Wl,-rpath,'$ORIGIN/../../bilevel-gait-gen_b200'
$CXX -O2 -std=c++17 -Wall -Ihost -o ../tests/cpp/test_qp_adjoint ../tests/cpp/test_qp_adjoint.cpp -L. -lmpc_b200 -lbgg_b200 -Wl,-rpath,'$ORIGIN/../../bilevel-gait-gen_b200'
echo "built $(pwd)/libbgg_b200.so $(pwd)/libmpc_b200.so"
