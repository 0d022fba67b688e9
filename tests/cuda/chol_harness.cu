// Test-only entry point around chol::factor + chol::solve (bilevel-gait-gen_b200/csrc/bgg_chol.cuh), for
// tests/test_gpu_linalg.py.  One matrix per CTA, at k_ipm's two block sizes (256 and 512 threads); everything else
// (data, references, tolerances) lives in the test.
// build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -maxrregcount=128 -Xcompiler -fPIC -shared
//        -I bilevel-gait-gen_b200/csrc -o libchol_harness.so tests/cuda/chol_harness.cu
#include <cuda_runtime.h>

#include "bgg_chol.cuh"

namespace {

using namespace bgg::chol;

// A: count block-packed lower triangles of nb block rows (doubles(nb) each), rhs: count vectors of 8 nb.
// Out: the factored K of every CTA as factor() leaves it, the solution vector (all 8 nb entries) and the pivot flag.
template <int kThreads>
__global__ void __launch_bounds__(kThreads, 1) k_chol_harness(const double* __restrict__ A, const double* __restrict__ rhs, int nb,
                                                            double* __restrict__ Kout, double* __restrict__ xout, int* __restrict__ flags) {
    extern __shared__ __align__(16) double sm[];
    const size_t nk = doubles(nb);
    double* K = sm;
    double* v = K + nk;
    double* ys = v + 8 * nb;
    __shared__ int flag;
    const int tid = threadIdx.x, b = blockIdx.x;
    for (size_t i = tid; i < nk; i += kThreads) K[i] = A[b * nk + i];
    for (int i = tid; i < 8 * nb; i += kThreads) v[i] = rhs[static_cast<size_t>(b) * 8 * nb + i];
    __syncthreads();
    factor(K, nb, &flag);
    for (size_t i = tid; i < nk; i += kThreads) Kout[b * nk + i] = K[i];
    solve(K, nb, v, ys);
    for (int i = tid; i < 8 * nb; i += kThreads) xout[static_cast<size_t>(b) * 8 * nb + i] = v[i];
    if (tid == 0) flags[b] = flag;
}

template <int kThreads>
cudaError_t launch(const double* dA, const double* drhs, int nb, int count, double* dK, double* dx, int* dflags) {
    const size_t smem = (doubles(nb) + 8 * nb + 64) * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(k_chol_harness<kThreads>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    k_chol_harness<kThreads><<<count, kThreads, smem>>>(dA, drhs, nb, dK, dx, dflags);
    return cudaGetLastError();
}

}  // namespace

// Host arrays in and out: A and K [count][doubles(nb)], rhs and x [count][8 nb], flags [count].  threads: 256 or 512.
// Returns 0 or a cudaError_t (-1 for bad arguments).
extern "C" int chol_harness_run(int threads, int nb, int count, const double* A, const double* rhs, double* K, double* x, int* flags) {
    if (nb < 1 || count < 1 || (threads != 256 && threads != 512)) return -1;
    const size_t nk = doubles(nb) * count, nv = static_cast<size_t>(8) * nb * count;
    double *dA = nullptr, *drhs = nullptr, *dK = nullptr, *dx = nullptr;
    int* dflags = nullptr;
    cudaError_t e = cudaMalloc(&dA, nk * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&dK, nk * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&drhs, nv * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&dx, nv * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&dflags, count * sizeof(int));
    if (e == cudaSuccess) e = cudaMemcpy(dA, A, nk * sizeof(double), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(drhs, rhs, nv * sizeof(double), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = threads == 256 ? launch<256>(dA, drhs, nb, count, dK, dx, dflags) : launch<512>(dA, drhs, nb, count, dK, dx, dflags);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(K, dK, nk * sizeof(double), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(x, dx, nv * sizeof(double), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(flags, dflags, count * sizeof(int), cudaMemcpyDeviceToHost);
    cudaFree(dA);
    cudaFree(dK);
    cudaFree(drhs);
    cudaFree(dx);
    cudaFree(dflags);
    return static_cast<int>(e);
}
