// bilevel-gait-gen_b200 -- kernel launchers and small device helpers shared by the .cu files.
#pragma once
#include <cuda_runtime.h>

#include "bgg_spline.cuh"
#include "bgg_types.cuh"
#include "bgg_ws.cuh"

namespace bgg {

__device__ void quat_log3(const double q[4], double out[3]);
__device__ void quat_exp3(const double v[3], double q[4]);
__device__ void quat_first_order_normalize(double q[4]);

// block-wide reductions (result broadcast to every thread); `scratch` holds >= 33 doubles of shared memory
__device__ __forceinline__ double warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
enum RedOp { kSum, kMax, kMin };
template <int OP>
__device__ __noinline__ double block_reduce(double v, double* scratch) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = (OP == kSum) ? warp_sum(v) : (OP == kMax ? warp_max(v) : warp_min(v));
    __syncthreads();   // protect scratch from the previous use
    if (lane == 0) scratch[wid] = v;
    __syncthreads();
    if (wid == 0) {
        double x = (lane < nw) ? scratch[lane] : ((OP == kSum) ? 0.0 : (OP == kMax ? -1e300 : 1e300));
        x = (OP == kSum) ? warp_sum(x) : (OP == kMax ? warp_max(x) : warp_min(x));
        if (lane == 0) scratch[32] = x;
    }
    __syncthreads();
    return scratch[32];
}

// One level of the warp reduce-scatter behind block_reduce_multi.  On entry lanes l and l ^ O both hold the partials of
// the same n values, n a power of two (v[j] is value idx + j); lanes without bit O keep the first n / 2 of them, lanes
// with it the rest, and each sends its partner only the half it drops.  Every partial is still combined with lane
// l ^ O's at every level, so value k ends as the 5-level butterfly's result bit for bit (a + b == b + a).  Once one
// value is left per lane the remaining levels are the plain butterfly.  Values idx + j >= NS + NM are padding that no
// real value meets.
template <int NS, int NM, int O, int n>
__device__ __forceinline__ void warp_reduce_scatter(double (&v)[NS + NM], int& idx, int lane) {
    if constexpr (O > 0) {
        constexpr int h = (n + 1) / 2;
        const bool hi = (lane & O) != 0;
        if (hi) idx += (n > 1) ? h : 0;
#pragma unroll
        for (int j = 0; j < h; ++j) {
            const double lo_v = v[j], hi_v = (n > 1 && h + j < NS + NM) ? v[h + j] : 0.0;
            const double keep = (n > 1 && hi) ? hi_v : lo_v;
            const double r = __shfl_xor_sync(0xffffffffu, (n > 1) ? (hi ? lo_v : hi_v) : lo_v, O);
            const bool sum = NM == 0 || (NS > 0 && idx + j < NS);
            v[j] = sum ? keep + r : fmax(keep, r);
        }
        warp_reduce_scatter<NS, NM, O / 2, h>(v, idx, lane);
    }
}
__host__ __device__ constexpr int ceil_log2(int n) { return n <= 1 ? 0 : 1 + ceil_log2((n + 1) / 2); }

// NS sums followed by NM maxima in one pass (one pair of barriers for all of them); scratch >= (NS + NM) doubles per warp.
// Result broadcast to every thread in v.  Sums: the 5-level butterfly within the warp, then warp 0 + warp 1 + ... in
// order -- the same rounding as warp_sum per value, through one reduce-scatter per warp instead of one butterfly per value
// (8 values: 9 double shuffles instead of 40).
template <int NS, int NM>
__device__ __forceinline__ void block_reduce_multi(double (&v)[NS + NM], double* scratch) {   // inlined: v stays in registers
    constexpr int K = NS + NM;
    static_assert(K >= 1 && K <= 32, "one value per lane at most");
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    int idx = 0;   // this lane's v[0] is value idx
    warp_reduce_scatter<NS, NM, 16, (1 << ceil_log2(K))>(v, idx, lane);
    __syncthreads();   // protect scratch from the previous use
    constexpr int rep = (32 >> ceil_log2(K)) - 1;   // lanes that differ only in these bits hold the same value
    if ((lane & rep) == 0 && idx < K) scratch[wid * K + idx] = v[0];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] = scratch[k];
#pragma unroll 1
    for (int w = 1; w < nw; ++w) {
#pragma unroll
        for (int k = 0; k < K; ++k) v[k] = (k < NS) ? v[k] + scratch[w * K + k] : fmax(v[k], scratch[w * K + k]);
    }
}

// kernel launchers (each is asynchronous on `stream`)
void launch_prepare(const Params& P, Instance* inst, const double* state, const double* t0, const double* ee_start,
                    const WsLayout& L, char* ws, int B, cudaStream_t stream);
// bgg_ik.cu: SingleRigidBodyModel::InverseKinematics / MPCController::GetTargetsFromTraj, one thread per problem
void launch_ik(const RobotKin& rk, int count, const double* state, const double* ee_des, const double* joint_guess, double* q, int* status,
               int* iters, cudaStream_t stream);
void launch_targets_from_traj(const Params& P, const RobotKin& rk, const Instance* inst, int B, const double* time, double* q_des, double* v_des,
                              double* force_des, int* status, cudaStream_t stream);
// bgg_partials.cu: one contact time's parameter partials written out (ComputeParamPartialsClarabel), blocks described there
constexpr int kPartHdr = 32;
__host__ __device__ size_t param_partials_doubles(int N, int nu_cap);
void launch_param_partials(const Params& P, const Instance* inst, const WsLayout& L, const char* ws, int b, int ee, int idx, int nu_cap, double* out,
                           double* ut, cudaStream_t stream);
void launch_condense(const Params& P, const WsLayout& L, char* ws, int B, int nu_max, int want, cudaStream_t stream);
void launch_ipm(const Params& P, const WsLayout& L, char* ws, int B, int nu_max, int ns_max, int want, cudaStream_t stream, int sm_count = 0);
// max over the batch of (nu, n_samples) after launch_prepare, written to out[0..1] (device); instances larger than the caps
// are marked for the second pass (WsHeader::pass_state = 2)
void launch_batch_max(const WsLayout& L, char* ws, int B, int* out, int cap_nu, int cap_ns, cudaStream_t stream);
// `want`: the pass_state an instance must have to be processed (0: first pass, 2: second pass for the instances that outgrew the first pass's sizes)
size_t finish_smem_bytes(const WsLayout& L);
bool ipm_two_per_sm(const WsLayout& L, int nu_max, int ns_max);
void launch_finish(const Params& P, Instance* inst, const WsLayout& L, char* ws, int B, int want, cudaStream_t stream);
size_t ipm_smem_bytes(const WsLayout& L);
size_t condense_smem_bytes(const WsLayout& L);

// parity taps
void launch_export_dynamics(const Params& P, const WsLayout& L, char* ws, int B, double* Ad, double* Bd, double* cd,
                            int nu_stride, cudaStream_t stream);

// the reference's sparse QP (CSC, bit-identical sparsity) from the structured form; see csrc/bgg_assemble.cu
void launch_export_csc(const Params& P, const WsLayout& L, const char* ws, int B, int32_t* colptr, int32_t* rowidx, double* val,
                       double* p_diag, double* q, double* ub, int32_t* dims, int n_stride, int m_stride, int nnz_cap,
                       cudaStream_t stream);

// gait gradient (csrc/bgg_gradient.cu); returns -1 when the shared memory it needs exceeds max_smem
int launch_gradient(const Params& P, const Instance* inst, const WsLayout& L, char* ws, int B, int nu_max, int ns_max, int max_smem,
                    cudaStream_t stream);
size_t gradient_smem_bytes(const WsLayout& L, int nu_max, int ns_max);

// gait optimiser outer step (csrc/bgg_gait.cu)
void launch_gait_lp(const Instance* inst, const WsLayout& L, const char* ws, int B, const double* grad, const double* time, double trust,
                    double alpha, double* step, double* xk, double* times, int32_t* status, cudaStream_t stream);
void launch_ls_expand(const Instance* parent, Instance* child, int B, int K, const double* xk, const double* step, const double* state,
                      const double* t0, const double* ee, double* c_state, double* c_t0, double* c_ee, cudaStream_t stream);
void launch_ls_select(Instance* parent, const Instance* child, const WsLayout& L, const char* child_ws, int B, int K, int32_t* best,
                      double* costs, int32_t* quality, cudaStream_t stream);

}  // namespace bgg
