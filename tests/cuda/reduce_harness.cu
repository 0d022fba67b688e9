// Test-only entry point around bgg::block_reduce_multi (bilevel-gait-gen_b200/csrc/bgg_kernels.cuh), for
// tests/test_gpu_reduce.py.  One CTA per case at k_ipm's two block sizes, the (sums, maxima) shapes k_ipm reduces; every
// thread's result is written out, so the test sees the broadcast too.  The reference (the butterfly per value and the
// cross-warp sum in warp order) lives in the test.
// build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -maxrregcount=128 -Xcompiler -fPIC -shared
//        -I bilevel-gait-gen_b200/csrc -o libreduce_harness.so tests/cuda/reduce_harness.cu
#include <cuda_runtime.h>

#include "bgg_kernels.cuh"

namespace {

// in / out: [count][kThreads][NS + NM]
template <int NS, int NM, int kThreads>
__global__ void __launch_bounds__(kThreads, 1) k_reduce_harness(const double* __restrict__ in, double* __restrict__ out) {
    constexpr int K = NS + NM;
    __shared__ double scratch[K * kThreads / 32];
    const size_t base = (static_cast<size_t>(blockIdx.x) * kThreads + threadIdx.x) * K;
    double v[K];
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] = in[base + k];
    bgg::block_reduce_multi<NS, NM>(v, scratch);
#pragma unroll
    for (int k = 0; k < K; ++k) out[base + k] = v[k];
}

template <int NS, int NM>
cudaError_t launch(int threads, int count, const double* din, double* dout) {
    if (threads == 256) k_reduce_harness<NS, NM, 256><<<count, 256>>>(din, dout);
    else k_reduce_harness<NS, NM, 512><<<count, 512>>>(din, dout);
    return cudaGetLastError();
}

}  // namespace

// Host arrays in and out: [count][threads][ns + nm].  (ns, nm): (4, 4), (3, 0) or (0, 2); threads: 256 or 512.
// Returns 0 or a cudaError_t (-1 for bad arguments).
extern "C" int reduce_harness_run(int ns, int nm, int threads, int count, const double* in, double* out) {
    const bool shape = (ns == 4 && nm == 4) || (ns == 3 && nm == 0) || (ns == 0 && nm == 2);
    if (!shape || count < 1 || (threads != 256 && threads != 512)) return -1;
    const size_t n = static_cast<size_t>(count) * threads * (ns + nm);
    double *din = nullptr, *dout = nullptr;
    cudaError_t e = cudaMalloc(&din, n * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&dout, n * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpy(din, in, n * sizeof(double), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        if (ns == 4) e = launch<4, 4>(threads, count, din, dout);
        else if (ns == 3) e = launch<3, 0>(threads, count, din, dout);
        else e = launch<0, 2>(threads, count, din, dout);
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(out, dout, n * sizeof(double), cudaMemcpyDeviceToHost);
    cudaFree(din);
    cudaFree(dout);
    return static_cast<int>(e);
}
