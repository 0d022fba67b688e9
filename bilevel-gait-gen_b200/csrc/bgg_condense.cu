// bilevel-gait-gen_b200 -- kernel 3b: state elimination ("condensing") of the arrow-shaped RTI QP, one CTA per
// instance, everything on chip except the outputs.
//
// The reference's decision vector is z = [x_0 .. x_N | u] with the spline coefficients u entering every node's
// dynamics row (mpc_single_rigid_body.cpp:259-273): a block-bidiagonal state chain with a dense border.  With
//   x_0 = x_init,   x_{k+1} = Ad_k x_k + Bd_k u + cd_k          (rows of AddDynamicsConstraints, :218-265)
// every state is affine in u:  x_k = Phi_k u + phi_k,  Phi_{k+1} = Ad_k Phi_k + Bd_k,  phi_{k+1} = Ad_k phi_k + cd_k.
// The cost (P diagonal: Q per node, Phi at node N, force weight, +1e-3 I; mpc.cpp:542-564,791-802,1090-1095) becomes
//   H = sum_k Phi_k' P_k Phi_k + P_u,     g = sum_k Phi_k' (P_k phi_k + q_k).
// Outputs: H (full symmetric, HBM), g, the two position rows of Phi_k for the foot-box rows (k >= 4), and phi_k.
// Phi_k itself (12 x nu) lives in shared memory only, double buffered; H is accumulated in registers by FP64 tensor-core
// instructions (see k_condense).
#include "bgg_kernels.cuh"

namespace bgg {

__device__ __forceinline__ void cross3d(const double a[3], const double b[3], double o[3]) {
    o[0] = a[1] * b[2] - a[2] * b[1];
    o[1] = a[2] * b[0] - a[0] * b[2];
    o[2] = a[0] * b[1] - a[1] * b[0];
}

// row stride of the Phi buffers: >= nu and = 4 mod 16, so that the DMMA operand loads of lanes (g, t) at
// (4 s + t) * ldp + 8 b + g hit 16 distinct 8-byte banks per half warp
static __host__ __device__ inline int condense_ldp(int nu_cap) { return ((nu_cap + 11) / 16) * 16 + 4; }
static size_t condense_smem_for(int nu_cap) {
    return 8 * (static_cast<size_t>(2 * kNx) * condense_ldp(nu_cap) + nu_cap + 4 * kNx) + sizeof(NodeLin) + 256;
}
size_t condense_smem_bytes(const WsLayout& L) { return condense_smem_for(L.max_nu); }

__device__ __forceinline__ void dmma_c(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__device__ __forceinline__ double lds_c(unsigned addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}

// H = sum_k Phi_k' P_k Phi_k is a symmetric rank-12 update per node: on the FP64 tensor-core path (DMMA) one warp owns
// up to NITEM pairs of block rows (row nb-1-p with nb-p blocks of 8 x 8, row p with p+1: nb + 1 <= 21 blocks) and keeps
// their accumulators in registers across all N + 1 nodes; per node and block three DMMAs (12 = 3 x 4), one
// shared-memory load each (the A operand p_r Phi[r][i] is shared by a row's blocks).  The scalar 16 x 16 thread tiling
// this replaces ran at 6 % of the FP64 peak (440 k cycles per instance for 1.8 MFMA, compiled without FMA contraction).
constexpr int kCondAcc = 21;
// the row pair p = 0 holds nb + 1 blocks; a block past kCondAcc would never be accumulated nor written
static_assert((kMaxSplineVars + 7) / 8 + 1 <= kCondAcc, "k_condense: kCondAcc accumulators do not cover max_spline_vars = kMaxSplineVars");

template <int NITEM>
__global__ void __launch_bounds__(256, (NITEM == 1) ? 2 : 1) k_condense(Params P, WsLayout L, char* __restrict__ ws_base, int cap_nu, int want) {
    const int b = blockIdx.x, tid = threadIdx.x, nth = blockDim.x;
    const int lane = tid & 31, wid = tid >> 5, nwarp = nth >> 5, g = lane >> 2, t = lane & 3;
    char* ws = ws_base + static_cast<size_t>(b) * L.stride;
    WsHeader* Hd = reinterpret_cast<WsHeader*>(ws + L.hdr);
    if (Hd->error || Hd->pass_state != want) return;
    const NodeLin* nodes = reinterpret_cast<const NodeLin*>(ws + L.nodes);
    const double* zprev = reinterpret_cast<const double*>(ws + L.zprev);
    double* Hout = reinterpret_cast<double*>(ws + L.H);
    double* gout = reinterpret_cast<double*>(ws + L.g);
    double* phipos = reinterpret_cast<double*>(ws + L.phipos);
    double* xoff = reinterpret_cast<double*>(ws + L.xoff);

    const int N = P.N, nu = Hd->nu, nf = Hd->nf;
    const int ldp = condense_ldp(cap_nu), nb = (nu + 7) >> 3;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* Phi = reinterpret_cast<double*>(smem_raw);         // [2][12][ldp], columns nu .. ldp-1 stay zero
    double* gs = Phi + 2 * kNx * ldp;                          // [nu]
    double* phi = gs + cap_nu;                                 // [2][12]
    double* pq = phi + 2 * kNx;                                // [2][12]: P_k (diag) and P_k phi_k + q_k
    NodeLin* nl = reinterpret_cast<NodeLin*>(pq + 2 * kNx);
    __shared__ int s_fbase[kNumEE], s_pbase[kNumEE], s_nfv[kNumEE], s_npv[kNumEE];
    __shared__ double s_cc[kNx];
    double cc = 0.0;   // this thread's share of the constant term of the condensed objective

    for (int i = tid; i < 2 * kNx * ldp; i += nth) Phi[i] = 0.0;
    for (int i = tid; i < nu; i += nth) gs[i] = 0.0;
    if (tid < kNx) phi[tid] = zprev[tid];   // phi_0 = tangent(state), the right-hand side of the -x_0 row
    if (tid < kNumEE) {
        s_fbase[tid] = Hd->fbase[tid];
        s_pbase[tid] = Hd->pbase[tid];
        s_nfv[tid] = Hd->nfv[tid];
        s_npv[tid] = Hd->npv[tid];
    }
    // this warp's block rows and accumulators
    int rowA[NITEM], lenA[NITEM], rowB[NITEM], lenB[NITEM];
    double2 acc[NITEM][kCondAcc];
#pragma unroll
    for (int it = 0; it < NITEM; ++it) {
        const int p = wid + it * nwarp;
        const bool on = 2 * p <= nb - 1;
        rowA[it] = on ? nb - 1 - p : 0;
        lenA[it] = on ? nb - p : 0;
        rowB[it] = on ? p : 0;
        lenB[it] = (on && p != nb - 1 - p) ? p + 1 : 0;
#pragma unroll
        for (int u = 0; u < kCondAcc; ++u) acc[it][u] = make_double2(0.0, 0.0);
    }
    const unsigned phi_s = static_cast<unsigned>(__cvta_generic_to_shared(Phi));
    const unsigned pq_s = static_cast<unsigned>(__cvta_generic_to_shared(pq));
    __syncthreads();

    for (int k = 0; k <= N; ++k) {
        double* Pc = Phi + (k & 1) * kNx * ldp;          // Phi_k, row-major [12][ldp]
        double* Pn = Phi + ((k + 1) & 1) * kNx * ldp;    // Phi_{k+1}
        double* fc = phi + (k & 1) * kNx;
        double* fn = phi + ((k + 1) & 1) * kNx;
        if (k < N) {
            const double* src = reinterpret_cast<const double*>(&nodes[k]);
            double* dst = reinterpret_cast<double*>(nl);
            for (int i = tid; i < static_cast<int>(sizeof(NodeLin) / 8); i += nth) dst[i] = src[i];
        }
        if (tid < kNx) {
            const double pk = ((k < N) ? P.Q[tid] : P.Phi[tid]) + 1e-3;
            const double qk = (k < N) ? P.w[tid] : P.Phi_w[tid];
            pq[tid] = pk;
            pq[kNx + tid] = pk * fc[tid] + qk;
            cc += 0.5 * pk * fc[tid] * fc[tid] + qk * fc[tid];
            xoff[k * kNx + tid] = fc[tid];
        }
        __syncthreads();
        // g += Phi_k' (P_k phi_k + q_k) ; foot-box position rows
        for (int i = tid; i < nu; i += nth) {
            double s = 0;
#pragma unroll
            for (int r = 0; r < kNx; ++r) s += Pc[r * ldp + i] * pq[kNx + r];
            gs[i] += s;
            if (k >= kEENodeStart) {
                phipos[static_cast<size_t>((k - kEENodeStart) * 2 + 0) * L.max_nu + i] = Pc[0 * ldp + i];
                phipos[static_cast<size_t>((k - kEENodeStart) * 2 + 1) * L.max_nu + i] = Pc[1 * ldp + i];
            }
        }
        // H += Phi_k' P_k Phi_k : DMMA, accumulators in registers (Phi_0 = 0)
        if (k > 0) {
            const unsigned cur_s = phi_s + 8u * ((k & 1) * kNx * ldp);
#pragma unroll
            for (int it = 0; it < NITEM; ++it) {
                if (lenA[it] == 0) continue;   // warp-uniform
#pragma unroll
                for (int s3 = 0; s3 < 3; ++s3) {
                    const unsigned row_s = cur_s + 8u * ((4 * s3 + t) * ldp);
                    const double pr = lds_c(pq_s + 8u * (4 * s3 + t));
                    const double aA = pr * lds_c(row_s + 8u * (8 * rowA[it] + g));
                    const double aB = (lenB[it] > 0) ? pr * lds_c(row_s + 8u * (8 * rowB[it] + g)) : 0.0;
                    const unsigned pA = row_s + 8u * g, pB = row_s + 8u * (g - 8 * lenA[it]);
                    double b_cur = lds_c((0 < lenA[it]) ? pA : pB);
#pragma unroll
                    for (int u = 0; u < kCondAcc; ++u) {
                        double b_next = 0.0;
                        if (u + 1 < kCondAcc) {
                            const int un = (u + 1 < lenA[it] + lenB[it]) ? u + 1 : 0;   // an empty slot reads a valid address and multiplies by a = 0
                            b_next = lds_c(((un < lenA[it]) ? pA : pB) + 64u * un);
                        }
                        dmma_c(acc[it][u].x, acc[it][u].y, (u < lenA[it]) ? aA : ((u < lenA[it] + lenB[it]) ? aB : 0.0), b_cur);
                        b_cur = b_next;
                    }
                }
            }
        }
        // Phi_{k+1} = Ad_k Phi_k + Bd_k ; phi_{k+1} = Ad_k phi_k + cd_k
        if (k < N) {
            for (int i = tid; i < nu; i += nth) {
                double col[kNx];
#pragma unroll
                for (int r = 0; r < kNx; ++r) col[r] = Pc[r * ldp + i];
#pragma unroll
                for (int r = 0; r < kNx; ++r) {
                    double s = 0;
#pragma unroll
                    for (int q = 0; q < kNx; ++q) s += nl->Ad[r * kNx + q] * col[q];
                    Pn[r * ldp + i] = s;
                }
            }
            if (tid < kNx) {
                double s = nl->cd[tid];
                for (int q = 0; q < kNx; ++q) s += nl->Ad[tid * kNx + q] * fc[q];
                fn[tid] = s;
            }
            __syncthreads();
            // + Bd_k : one thread per (foot, coord, weight); distinct threads touch distinct columns
            if (tid < kNumEE * 3 * 4) {
                const int e = tid / 12, c = (tid / 4) % 3, j = tid % 4;
                if (j < nl->fcnt[e]) {
                    const int col = s_fbase[e] + c * s_nfv[e] + nl->foff[e] + j;
                    const double ec[3] = {c == 0 ? 1.0 : 0.0, c == 1 ? 1.0 : 0.0, c == 2 ? 1.0 : 0.0};
                    double rc[3];
                    cross3d(nl->rel[e], ec, rc);
                    Pn[(3 + c) * ldp + col] += P.dt * nl->fw[e][j];
                    for (int r = 0; r < 3; ++r) Pn[(9 + r) * ldp + col] += P.dt * (rc[r] * nl->fw[e][j]);
                }
            } else if (tid >= 64 && tid < 64 + kNumEE * 2 * 2) {
                const int q = tid - 64, e = q / 4, c = (q / 2) % 2, j = q % 2;
                if (j < nl->pcnt[e]) {
                    const int col = nf + s_pbase[e] + c * s_npv[e] + nl->poff[e] + j;
                    const double ec[3] = {c == 0 ? 1.0 : 0.0, c == 1 ? 1.0 : 0.0, 0.0};
                    double ef[3];
                    cross3d(ec, nl->f[e], ef);
                    for (int r = 0; r < 3; ++r) Pn[(9 + r) * ldp + col] += P.dt * (ef[r] * nl->pw[e][j]);
                }
            }
        }
        __syncthreads();
    }
    if (tid < kNx) s_cc[tid] = cc;
    for (int i = tid; i < nu; i += nth) gout[i] = gs[i];
    __syncthreads();
    if (tid == 0) {
        double tt = 0;
        for (int r = 0; r < kNx; ++r) tt += s_cc[r];
        Hd->cost_const = tt;
    }
    // full symmetric H to HBM (the IPM reads it column-wise, coalesced), straight from the accumulators: the block's
    // own entries and their mirror image; P_u (force weight on force variables, +1e-3 on everything: AddForceCost /
    // AddDiagonalCost) goes on the diagonal.  Off the diagonal blocks H is exactly symmetric (one value, stored twice); inside
    // a diagonal block (i, j) and (j, i) are two roundings of the same sum, (p_r Phi[r][i]) Phi[r][j] and
    // (p_r Phi[r][j]) Phi[r][i], and may differ in the last bits.  Both are what the IPM consumes (the factorisation reads
    // the lower triangle, the residuals H v both), so they are kept as they are: tests/test_gpu_linalg.py bounds each against
    // the long-double sum.
#pragma unroll
    for (int it = 0; it < NITEM; ++it)
#pragma unroll
        for (int u = 0; u < kCondAcc; ++u) {
            if (u >= lenA[it] + lenB[it]) continue;
            const int ib = (u < lenA[it]) ? rowA[it] : rowB[it], jb = (u < lenA[it]) ? u : u - lenA[it];
            const int i = 8 * ib + g, j = 8 * jb + 2 * t;
            double v0 = acc[it][u].x, v1 = acc[it][u].y;
            if (i == j) v0 += ((i < nf) ? P.force_cost : 0.0) + 1e-3;
            if (i == j + 1) v1 += ((i < nf) ? P.force_cost : 0.0) + 1e-3;
            if (i < nu) {
                if (j < nu) Hout[static_cast<size_t>(i) * nu + j] = v0;
                if (j + 1 < nu) Hout[static_cast<size_t>(i) * nu + j + 1] = v1;
                if (ib != jb) {
                    if (j < nu) Hout[static_cast<size_t>(j) * nu + i] = v0;
                    if (j + 1 < nu) Hout[static_cast<size_t>(j + 1) * nu + i] = v1;
                }
            }
        }
}

void launch_condense(const Params& P, const WsLayout& L, char* ws, int B, int nu_max, int want, cudaStream_t stream) {
    int cap = (nu_max + 7) / 8 * 8;
    if (cap > L.max_nu) cap = L.max_nu;
    const size_t smem = condense_smem_for(cap);
    // per device and context, so set on every launch (see launch_ipm)
    cudaFuncSetAttribute(k_condense<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    cudaFuncSetAttribute(k_condense<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    // eight warps own one pair of block rows each up to 16 block rows (nu <= 128), two pairs beyond
    if (cap / 8 <= 16) k_condense<1><<<B, 256, smem, stream>>>(P, L, ws, cap, want);
    else k_condense<2><<<B, 256, smem, stream>>>(P, L, ws, cap, want);
}

// Batch maxima of (nu, n_samples) for the shared-memory sizing of the NEXT solve, and the instances that do not fit the caps THIS
// solve's first pass was launched with (sized from the previous solve, no host round trip): they are marked for the second pass.
__global__ void k_batch_max(WsLayout L, char* __restrict__ ws, int B, int* __restrict__ out, int cap_nu, int cap_ns) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    WsHeader* h = reinterpret_cast<WsHeader*>(ws + static_cast<size_t>(b) * L.stride + L.hdr);
    if (h->error) return;
    atomicMax(&out[0], h->nu);
    atomicMax(&out[1], h->n_samples);
    if (h->nu > cap_nu || h->n_samples > cap_ns) {
        h->pass_state = 2;
        atomicAdd(&out[2], 1);
    }
}

void launch_batch_max(const WsLayout& L, char* ws, int B, int* out, int cap_nu, int cap_ns, cudaStream_t stream) {
    cudaMemsetAsync(out, 0, 3 * sizeof(int), stream);
    k_batch_max<<<(B + 255) / 256, 256, 0, stream>>>(L, ws, B, out, cap_nu, cap_ns);
}

// ---- parity tap: dense Ad [N][12][12], Bd [N][12][nu_stride], cd [N][12] per instance (what the reference holds in
// A_, B_, C_ after mpc_single_rigid_body.cpp:246-248)
__global__ void k_export_dynamics(Params P, WsLayout L, const char* __restrict__ ws_base, double* __restrict__ Ad,
                                  double* __restrict__ Bd, double* __restrict__ cd, int nu_stride) {
    const int b = blockIdx.x, tid = threadIdx.x, nth = blockDim.x;
    const char* ws = ws_base + static_cast<size_t>(b) * L.stride;
    const WsHeader* Hd = reinterpret_cast<const WsHeader*>(ws + L.hdr);
    const NodeLin* nodes = reinterpret_cast<const NodeLin*>(ws + L.nodes);
    const int N = P.N, nf = Hd->nf;
    double* A = Ad + static_cast<size_t>(b) * N * 144;
    double* Bm = Bd + static_cast<size_t>(b) * N * kNx * nu_stride;
    double* c = cd + static_cast<size_t>(b) * N * kNx;
    for (int i = tid; i < N * kNx * nu_stride; i += nth) Bm[i] = 0.0;
    __syncthreads();
    for (int i = tid; i < N * 144; i += nth) A[i] = nodes[i / 144].Ad[i % 144];
    for (int i = tid; i < N * kNx; i += nth) c[i] = nodes[i / kNx].cd[i % kNx];
    for (int i = tid; i < N * kNumEE; i += nth) {
        const int k = i / kNumEE, e = i % kNumEE;
        const NodeLin& nl = nodes[k];
        double* Bk = Bm + static_cast<size_t>(k) * kNx * nu_stride;
        for (int cc = 0; cc < 3; ++cc) {
            const double ec[3] = {cc == 0 ? 1.0 : 0.0, cc == 1 ? 1.0 : 0.0, cc == 2 ? 1.0 : 0.0};
            double rc[3], ef[3];
            cross3d(nl.rel[e], ec, rc);
            cross3d(ec, nl.f[e], ef);
            for (int j = 0; j < nl.fcnt[e]; ++j) {
                const int col = Hd->fbase[e] + cc * Hd->nfv[e] + nl.foff[e] + j;
                Bk[(3 + cc) * nu_stride + col] = P.dt * nl.fw[e][j];
                for (int r = 0; r < 3; ++r) Bk[(9 + r) * nu_stride + col] = P.dt * (rc[r] * nl.fw[e][j]);
            }
            if (cc < 2)
                for (int j = 0; j < nl.pcnt[e]; ++j) {
                    const int col = nf + Hd->pbase[e] + cc * Hd->npv[e] + nl.poff[e] + j;
                    for (int r = 0; r < 3; ++r) Bk[(9 + r) * nu_stride + col] = P.dt * (ef[r] * nl.pw[e][j]);
                }
        }
    }
}

void launch_export_dynamics(const Params& P, const WsLayout& L, char* ws, int B, double* Ad, double* Bd, double* cd,
                            int nu_stride, cudaStream_t stream) {
    k_export_dynamics<<<B, 256, 0, stream>>>(P, L, ws, Ad, Bd, cd, nu_stride);
}

}  // namespace bgg
