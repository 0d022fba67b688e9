// bilevel-gait-gen_b200 -- kernel 4: the QP solve, one CTA per MPC instance, a primal-dual interior-point method on the
// condensed QP
//      min 1/2 u'Hu + g'u   s.t.  C u <= d  (force box, friction pyramid, foot box),   E u = e  (touch-down, foot start)
// The reference's live solver is Clarabel, an interior-point method run to 1e-8 (mpc.h:264, clarabel_interface.cpp:
// 18-27,72-155); an ADMM at OSQP tolerances leaves this ill-conditioned QP 1e-2 away from the optimum (DESIGN.md),
// so the kernel follows the live path, and follows Clarabel's algorithm: the homogeneous self-dual embedding
//      H u + C'z + E'y + g tau = 0 ,  C u + s - d tau = 0 ,  E u - e tau = 0 ,  kappa + g'u + d'z + e'y + u'Hu / tau = 0 ,
//      s o z = mu ,  tau kappa = mu
// with predictor-corrector steps (sigma = (1 - alpha_aff)^3, step fraction 0.99), static regularisation and the
// infeasibility certificate  d'z + e'y < 0, C'z + E'y ~ 0.  Per iteration K = H + eps I + C'WC + E'E/delta with
// W = 1 / (s/z + eps) is assembled from the *structured* rows (never a sparse matrix), factorised once by an
// in-shared-memory block Cholesky and used for three solves: the constant right-hand side (-g ; d ; e), the affine and
// the combined step.  The step is the one of the regularised system (primal-dual proximal form, fixed point = the
// solution of the unregularised QP); oracle/qp_ipm.cpp runs the same iteration on the reference's sparse QP and
// tools/ipm_proto.py holds the numpy prototype both were derived from.
//
// Inequality rows, internal order (m = 6 ns + 2 ne):
//   6 j + 0 :  f_z(tau_j) <= force_bound          6 j + 1 : -f_z(tau_j) <= 0               (mpc.cpp:352-414)
//   6 j + 2..5 : (+-e_x - mu e_z).f <= 0, (+-e_y - mu e_z).f <= 0                          (mpc.cpp:153-209)
//   6 ns + 2 e + 0 : -p_c(k) + w.u_pos <=  hip_c + box_c/2     e = ((k-4)*4 + foot)*2 + c   (mpc_single_rigid_body.cpp:381-443)
//   6 ns + 2 e + 1 :  p_c(k) - w.u_pos <= -(hip_c - box_c/2)
#include <cstdio>
#include <cstdlib>

#include "bgg_kernels.cuh"
#include "bgg_chol.cuh"
#include "bgg_kkt.cuh"
#include "bgg_kkt_mma.cuh"
#include "bgg_l2ops.cuh"
#ifdef BGG_IPM_TRACE
#include "bgg_ipm_trace.cuh"
#endif

namespace bgg {

// Phase clocks (tools/profile_phases.py): compiled in only with -DBGG_IPM_PROF into a separate library, never into
// libbgg_b200.so.  Thread 0 of CTA 0 accumulates clock64() deltas between barrier-delimited phases.
#ifdef BGG_IPM_PROF
__device__ long long g_ipm_prof[32];
#define PROF_DECL __shared__ long long s_prof[32]; long long prof_t = 0; if (threadIdx.x == 0) { for (int i_ = 0; i_ < 32; ++i_) s_prof[i_] = 0; prof_t = clock64(); }
#define PROF(k) do { if (threadIdx.x == 0) { const long long t_ = clock64(); s_prof[k] += t_ - prof_t; prof_t = t_; } } while (0)
#define PROF_DUMP do { if (threadIdx.x == 0 && blockIdx.x == 0) for (int i_ = 0; i_ < 32; ++i_) g_ipm_prof[i_] = s_prof[i_]; } while (0)
#else
#define PROF_DECL
#define PROF(k) do { } while (0)
#define PROF_DUMP do { } while (0)
#endif

// Per-iteration trace (tests/test_gpu_ipm_trace.py): compiled in only with -DBGG_IPM_TRACE into a separate library
// (tools/build_trace.sh), never into libbgg_b200.so.  csrc/bgg_ipm_trace.cuh describes the records.  TRACE(...) statements
// run in the armed CTA only and add barriers there; without the macro they are empty.
#ifdef BGG_IPM_TRACE
#define TRACE(...) do { __VA_ARGS__ } while (0)
#else
#define TRACE(...) do { } while (0)
#endif

namespace {

struct Smem {
    double* K;       // lower triangle in 8 x 8 blocks (csrc/bgg_chol.cuh)
    double *u, *du, *rd, *rhs, *Hu, *x1;             // nu (rd: dual residual rx)
    double *s, *lam, *ds, *dl, *rp, *wv, *d;         // m  (wv: row weights while K is built, then C x1; rp: primal residual rz)
    double *tkc, *ckc;                               // 2(N-3)
    double *nueq, *re, *dnu, *y1, *a3;               // kMaxEq
    double* red;                                     // 72
    double* pw;                                      // [(N-3)*4][2] foot-box position weights
    int *pcnt, *poff;                                // [(N-3)*4]
    Sample* smp;                                     // staged force samples
    ColInfo* col;                                    // [nu] per-variable tables of the K assembly
    const double* phi;                               // position rows: shared memory when they fit, else HBM/L2
    int phi_stride;
};

}  // namespace

// What the operators below need.  They are force-inlined.  Measured on B200 (4096 solves): inlined 37.2 ms; as
// __noinline__ functions (one copy of each in the binary: ncu shows the 0.4 MB kernel stalling on instruction fetch) with
// the context by reference and every field copied to locals 41.1 ms, the same plus __isShared assumptions 39.2 ms,
// context by value 83 ms -- the call boundary costs more than the instruction-cache misses it saves.
struct IpmCtx {
    Smem S;
    const double* Hg;
    const EqRow* eq;
    const int *fbase, *pbase, *nfv, *npv;
    int N, nu, nf, ns, ne, neq, nkc;
    double mu_f;
};

// out[0..m) = C v   (v: nu-vector in shared memory); with eout != nullptr also eout[0..neq) = E v - rhs_scale e, computed by the
// last warp while the others take the samples (no extra barrier)
// kRowsShared: every row vector lives in shared memory (false in the spilled layout, where some are in the workspace)
template <bool kRowsShared, int kThreads>
static __device__ __forceinline__ void ipm_apply_C(const IpmCtx& c, const double* v, double* out, double* eout, double rhs_scale) {
    const Smem S = c.S;
    const int *fbase = c.fbase, *pbase = c.pbase, *nfv = c.nfv, *npv = c.npv;
    __builtin_assume(__isShared(v)); if (kRowsShared) __builtin_assume(__isShared(out)); __builtin_assume(__isShared(S.tkc));
    __builtin_assume(__isShared(S.smp)); __builtin_assume(__isShared(S.pw)); __builtin_assume(__isShared(S.pcnt));
    __builtin_assume(__isShared(S.poff)); __builtin_assume(__isShared(fbase)); __builtin_assume(__isShared(pbase));
    __builtin_assume(__isShared(nfv)); __builtin_assume(__isShared(npv));
    const int tid = threadIdx.x;
    constexpr int nth = kThreads;   // the launch's block size, known at compile time: constant strides
    const int nf = c.nf, ns = c.ns, ne = c.ne, nkc = c.nkc;
    const double mu_f = c.mu_f;
    l2_phi_rows_dot(S.phi, S.phi_stride, nkc, nf, smem_addr(v), smem_addr(S.tkc));   // dense position rows (csrc/bgg_l2ops.cuh)
    #pragma unroll 1
    for (int j = tid; j < ns; j += nth) {
        const Sample& sp = S.smp[j];
        double fv[3];
        for (int cc = 0; cc < 3; ++cc) {
            const double* vv = v + fbase[sp.ee] + cc * nfv[sp.ee] + sp.off;
            double s = 0;
            for (int i = 0; i < sp.cnt; ++i) s += sp.w[i] * vv[i];
            fv[cc] = s;
        }
        double* o = out + 6 * j;
        o[0] = fv[2];
        o[1] = -fv[2];
        o[2] = fv[0] - mu_f * fv[2];
        o[3] = -fv[0] - mu_f * fv[2];
        o[4] = fv[1] - mu_f * fv[2];
        o[5] = -fv[1] - mu_f * fv[2];
    }
    if (eout != nullptr && tid >= nth - 32 && tid - (nth - 32) < c.neq) {
        const EqRow& q = c.eq[tid - (nth - 32)];
        double s = -rhs_scale * q.rhs;
        for (int i = 0; i < q.cnt; ++i) s += q.w[i] * v[q.col[i]];
        eout[tid - (nth - 32)] = s;
    }
    __syncthreads();
    #pragma unroll 1
    for (int e = tid; e < ne; e += nth) {
        const int cc = e & 1, foot = (e >> 1) & 3, kk = e >> 3, kf = kk * 4 + foot;
        const double* vv = v + nf + pbase[foot] + cc * npv[foot] + S.poff[kf];
        double s = -S.tkc[kk * 2 + cc];
        for (int i = 0; i < S.pcnt[kf]; ++i) s += S.pw[2 * kf + i] * vv[i];
        out[6 * ns + 2 * e] = s;
        out[6 * ns + 2 * e + 1] = -s;
    }
    __syncthreads();
}

// out[0..nu) += C' y   (y: m-vector; inactive rows carry y == 0); with ey != nullptr also += escale E' ey (the equality rows
// touch position columns only: the thread that owns the column adds them).  Every output entry is owned by one thread.
template <bool kRowsShared, int kThreads>
static __device__ __forceinline__ void ipm_add_Ct(const IpmCtx& c, const double* y, double* out, const double* ey, double escale) {
    const Smem S = c.S;
    if (kRowsShared) __builtin_assume(__isShared(y)); __builtin_assume(__isShared(out)); __builtin_assume(__isShared(S.ckc));
    __builtin_assume(__isShared(S.smp)); __builtin_assume(__isShared(S.pw)); __builtin_assume(__isShared(S.col));
    __builtin_assume(__isShared(S.poff));
    const int tid = threadIdx.x;
    constexpr int nth = kThreads;
    const int nu = c.nu, nf = c.nf, ns = c.ns, nkc = c.nkc;
    const double mu_f = c.mu_f;
    #pragma unroll 1
    for (int q = tid; q < nkc; q += nth) {
        const int kk = q >> 1, cc = q & 1;
        double s = 0;
        for (int foot = 0; foot < kNumEE; ++foot) {
            const int e = (kk * 4 + foot) * 2 + cc;
            s += y[6 * ns + 2 * e] - y[6 * ns + 2 * e + 1];
        }
        S.ckc[q] = -s;
    }
    __syncthreads();
    l2_phi_cols_dot(S.phi, S.phi_stride, nkc, nf, smem_addr(S.ckc), smem_addr(out));   // dense foot-box rows (csrc/bgg_l2ops.cuh)
    // Two threads per column (nu <= 160 < blockDim / 2 ... else one): the first takes the dense foot-box rows (force
    // column) or the first half of the nodes (position column), the second the sample rows / the second half; the
    // loops run over the column's own sample / node range only (ColInfo, csrc/bgg_kkt.cuh).
    {
        const int half = (2 * nu <= nth) ? 2 : 1;
        #pragma unroll 1
        for (int base = 0; base < half * nu; base += nth) {   // whole warps iterate together: the partner exchange is a shuffle
            const int it = base + tid;
            const bool act = it < half * nu;
            const int col = act ? it / half : 0, part = it % half;
            const ColInfo ci = S.col[col];
            double s = 0;
            if (!act) {
            } else if (col < nf) {
                if (part == 1 || half == 1)
                    #pragma unroll 1
                    for (int j = ci.lo; j < ci.hi; ++j) {
                        const Sample& sp = S.smp[j];
                        const double* yy = y + 6 * j;
                        double coef;
                        if (ci.coord == 2) coef = (yy[0] - yy[1]) - mu_f * (yy[2] + yy[3] + yy[4] + yy[5]);
                        else if (ci.coord == 0) coef = yy[2] - yy[3];
                        else coef = yy[4] - yy[5];
                        s += coef * sp.w[ci.var - sp.off];
                    }
            } else {
                const int mid = (half == 2) ? (ci.lo + ci.hi + 1) / 2 : ci.hi;
                const int k0 = (part == 0) ? ci.lo : mid, k1 = (part == 0) ? mid : ci.hi;
                #pragma unroll 1
                for (int kk = k0; kk < k1; ++kk) {
                    const int kf = kk * 4 + ci.foot, e = kf * 2 + ci.coord;
                    s += (y[6 * ns + 2 * e] - y[6 * ns + 2 * e + 1]) * S.pw[2 * kf + (ci.var - S.poff[kf])];
                }
                if (ey != nullptr && part == 0) {
                    double se = 0;
                    const int grp = ci.foot * 2 + ci.coord;   // an equality row touches the position columns of one (foot, coord) only
                    #pragma unroll 1
                    for (int r = 0; r < c.neq; ++r) {
                        const EqRow& q = c.eq[r];
                        if (q.pad != grp) continue;
                        for (int i = 0; i < q.cnt; ++i)
                            if (q.col[i] == col) se += ey[r] * q.w[i];
                    }
                    s += escale * se;
                }
            }
            if (half == 2) s += __shfl_xor_sync(0xffffffffu, s, 1);   // partner thread: adjacent lane
            if (act && part == 0) out[col] += s;
        }
    }
    __syncthreads();
}

// out[0..nu) = H v, H full symmetric in HBM/L2, read column-wise (coalesced across threads)
static __device__ __forceinline__ void ipm_apply_H(const IpmCtx& c, const double* v, double* out, bool subtract) {
    l2_apply_H(c.Hg, c.nu, smem_addr(v), smem_addr(out), subtract);   // csrc/bgg_l2ops.cuh
}

struct IpmCaps {          // per-launch shared-memory sizing, from the actual maxima over the batch
    int nu, rows, ns, stage_phi, spill, threads;
};
constexpr int kRedDoubles256 = 72, kRedDoubles512 = 136;   // block_reduce_multi: 8 values per warp; chol::solve: 64
// spill: the row vectors s, z (they live in the workspace's slack / lam output arrays from the start), rz and the foot-box
// right-hand sides stay in L2 -- three of the six row vectors on chip instead of six
static size_t ipm_smem_core(int N, int nu, int rows, int ns, bool spill = false, int red = kRedDoubles256) {
    const size_t kc = 2 * (N - 3), eb = 4 * (N - 3);
    return 8 * (chol::doubles(nu / 8) + 6 * nu + (spill ? 3 : 6) * static_cast<size_t>(rows) + (spill ? 0 : 2 * eb * 2) + 2 * kc + 5 * kMaxEq + red + 2 * eb) +
           8 * eb + sizeof(Sample) * static_cast<size_t>(ns) + sizeof(ColInfo) * static_cast<size_t>(nu) + 64;
}
static IpmCaps ipm_caps(const WsLayout& L, int nu_max, int ns_max, bool alone = false) {
    IpmCaps c;
    c.nu = (nu_max + 7) / 8 * 8;
    if (c.nu > L.max_nu) c.nu = L.max_nu;
    c.ns = ns_max < 1 ? 1 : ns_max;
    c.rows = 6 * c.ns + 2 * (L.N - 3) * 8;
    // the KKT assembly stages phi chunks and a per-sample table in the ds / dl vectors (csrc/bgg_kkt_mma.cuh)
    const int scratch = kkt_scratch_doubles(c.nu / 8, c.ns);
    if (2 * c.rows < scratch) c.rows = (scratch + 1) / 2;
    const size_t core = ipm_smem_core(L.N, c.nu, c.rows, c.ns);
    const size_t phi = 8 * static_cast<size_t>(2 * (L.N - 3)) * c.nu;
    // two CTAs per SM when the core fits twice into the 227 KB; the dense position rows are staged on chip only
    // if that does not cost the second CTA
    const size_t half = 112 * 1024;   // + 1 KB static + 1 KB reserved per CTA, twice, inside the SM's 228 KB
    c.spill = 0;
    c.threads = 256;
    if (alone && core <= half) {
        // fewer CTAs than SMs (a single robot's solve): every CTA has an SM to itself, so the room of the second CTA holds the dense
        // position rows (1.58 -> 1.52 ms for one instance; sixteen warps on top of that are slower here: 1.67 ms)
        c.stage_phi = (core + phi <= 225 * 1024) ? 1 : 0;
    } else if (core <= half) c.stage_phi = (core + phi <= half) ? 1 : 0;
    else if (ipm_smem_core(L.N, c.nu, c.rows, c.ns, true) <= half) {
        // N = 50: 1232 rows.  Two CTAs per SM with three row vectors in L2 beat one CTA with everything on chip
        c.spill = 1;
        c.stage_phi = 0;
    } else {
        // K alone leaves no room for a second CTA (nu > 136): one CTA per SM, with sixteen warps instead of eight
        c.threads = 512;
        c.stage_phi = (core + phi + 8 * (kRedDoubles512 - kRedDoubles256) <= 225 * 1024) ? 1 : 0;
    }
    return c;
}
static size_t ipm_smem_for(const WsLayout& L, const IpmCaps& c) {
    return ipm_smem_core(L.N, c.nu, c.rows, c.ns, c.spill != 0, c.threads == 512 ? kRedDoubles512 : kRedDoubles256) +
           (c.stage_phi ? 8 * static_cast<size_t>(2 * (L.N - 3)) * c.nu : 0);
}
bool ipm_two_per_sm(const WsLayout& L, int nu_max, int ns_max) {   // do these maxima leave room for a second CTA on the SM?
    const IpmCaps c = ipm_caps(L, nu_max, ns_max);
    return ipm_smem_for(L, c) <= 112 * 1024;
}
size_t ipm_smem_bytes(const WsLayout& L) {   // worst case for the configured caps (bgg_create's feasibility check)
    return ipm_smem_core(L.N, L.max_nu, L.max_rows, kMaxSamples, false, kRedDoubles512);
}

template <bool kSpill, int kThreads>
__global__ void __launch_bounds__(kThreads, kThreads == 256 ? 2 : 1) k_ipm(Params P, WsLayout L, char* __restrict__ ws_base, int stage_phi, int cap_nu, int cap_rows, int want) {
    const int b = blockIdx.x, tid = threadIdx.x;
    constexpr int nth = kThreads;   // = blockDim.x (launch_ipm)
    char* ws = ws_base + static_cast<size_t>(b) * L.stride;
    WsHeader* Hd = reinterpret_cast<WsHeader*>(ws + L.hdr);
    if (!Hd->error && Hd->pass_state != want) return;   // not this pass's instance (uniform over the CTA)
    if (Hd->error) {   // k_prepare refused the instance: no QP, no iterate (k_finish keeps the previous solution)
        if (tid == 0) {
            Hd->status = kOther;
            Hd->no_iterate = 1;
            Hd->iters = 0;
        }
        return;
    }
    const NodeLin* nodes = reinterpret_cast<const NodeLin*>(ws + L.nodes);
    const Sample* samples = reinterpret_cast<const Sample*>(ws + L.samples);
    const EqRow* eqs = reinterpret_cast<const EqRow*>(ws + L.eq);
    const double* Hg = reinterpret_cast<const double*>(ws + L.H);       // full symmetric nu x nu
    const double* gg = reinterpret_cast<const double*>(ws + L.g);
    const double* phipos = reinterpret_cast<const double*>(ws + L.phipos);
    const double* xoff = reinterpret_cast<const double*>(ws + L.xoff);

    const int N = P.N, nu = Hd->nu, nf = Hd->nf, ns = Hd->n_samples, ne = Hd->n_eebox, neq = Hd->n_eq;
    const int m = 6 * ns + 2 * ne, nkc = 2 * (N - 3), npk = nu * (nu + 1) / 2;
    const double cost_const = Hd->cost_const;
    const double mu_f = P.friction_coef, delta = P.ipm_eq_delta, inv_delta = 1.0 / P.ipm_eq_delta, eps = P.ipm_reg_eps;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    PROF_DECL
    Smem S;
    {
        double* p = reinterpret_cast<double*>(smem_raw);
        S.K = p; p += chol::doubles(cap_nu >> 3);
        S.u = p; p += cap_nu; S.du = p; p += cap_nu; S.rd = p; p += cap_nu;
        S.rhs = p; p += cap_nu; S.Hu = p; p += cap_nu; S.x1 = p; p += cap_nu;
        constexpr bool spill = kSpill;
        if (spill) {   // s and z iterate in the arrays they are reported in; rz and d in the workspace's spill area (L2 resident)
            S.s = reinterpret_cast<double*>(ws + L.slack);
            S.lam = reinterpret_cast<double*>(ws + L.lam);
            S.rp = reinterpret_cast<double*>(ws + L.ipm_spill);
            S.d = S.rp + L.max_rows;
        } else {
            S.s = p; p += cap_rows; S.lam = p; p += cap_rows;
        }
        S.ds = p; p += cap_rows; S.dl = p; p += cap_rows;   // adjacent: the KKT assembly's scratch (csrc/bgg_kkt_mma.cuh)
        if (!spill) { S.rp = p; p += cap_rows; }
        S.wv = p; p += cap_rows;
        if (!spill) { S.d = p; p += 2 * 8 * (N - 3); }   // right-hand sides of the foot-box rows only (force rows: see rhs_of)
        S.tkc = p; p += nkc; S.ckc = p; p += nkc;
        S.nueq = p; p += kMaxEq; S.re = p; p += kMaxEq; S.dnu = p; p += kMaxEq; S.y1 = p; p += kMaxEq; S.a3 = p; p += kMaxEq;
        S.red = p; p += (kThreads == 512 ? kRedDoubles512 : kRedDoubles256);   // block_reduce_multi scratch (8 per warp) / chol::solve scratch (64)
        S.pw = p; p += 2 * 4 * (N - 3);
        S.pcnt = reinterpret_cast<int*>(p);
        S.poff = S.pcnt + 4 * (N - 3);
        p += 4 * (N - 3);
        S.smp = reinterpret_cast<Sample*>(p);
        p += (sizeof(Sample) * static_cast<size_t>(ns) + 7) / 8;
        S.col = reinterpret_cast<ColInfo*>(p);
        p += (sizeof(ColInfo) * static_cast<size_t>(nu) + 7) / 8;
        if (stage_phi) {
            S.phi = p;
            S.phi_stride = nf;
            for (int i = tid; i < nkc * nf; i += nth) p[i] = phipos[static_cast<size_t>(i / nf) * L.max_nu + (i % nf)];
        } else {
            S.phi = phipos;
            S.phi_stride = L.max_nu;
        }
    }
    #pragma unroll 1
    for (int i = tid; i < ns * static_cast<int>(sizeof(Sample) / 8); i += nth)
        reinterpret_cast<double*>(S.smp)[i] = reinterpret_cast<const double*>(samples)[i];
    for (int i = tid; i < 4 * (N - 3); i += nth) {
        const NodeLin& nl = nodes[i / 4 + kEENodeStart];
        const int foot = i & 3;
        S.pcnt[i] = nl.pcnt[foot];
        S.poff[i] = nl.poff[foot];
        S.pw[2 * i] = nl.pw[foot][0];
        S.pw[2 * i + 1] = nl.pw[foot][1];
    }
    __shared__ int s_fbase[kNumEE], s_pbase[kNumEE], s_nfv[kNumEE], s_npv[kNumEE];
    __shared__ int s_flag, s_nitems, s_nwork, s_npos;
    __shared__ KktWork s_work[kMaxKktWork];
    __shared__ int s_sb[kNumEE + 1];   // per-foot sample ranges (samples are stored foot-major)
    __shared__ EqRow s_eq[kMaxEq];
    if (tid < neq) s_eq[tid] = eqs[tid];
    if (tid < kNumEE) {
        s_fbase[tid] = Hd->fbase[tid];
        s_pbase[tid] = Hd->pbase[tid];
        s_nfv[tid] = Hd->nfv[tid];
        s_npv[tid] = Hd->npv[tid];
    }
    #pragma unroll 1
    for (int i = tid; i < 6 * cap_nu; i += nth) S.u[i] = 0.0;   // u du rd rhs Hu x1: the padding up to 8 nb stays zero (chol::solve)
    if (tid == 0) {
        int e = 0;
        s_sb[0] = 0;
        for (int j = 0; j < ns; ++j)
            while (samples[j].ee > e) s_sb[++e] = j;
        while (e < kNumEE) s_sb[++e] = ns;
    }

    // ---- right-hand sides d and the active mask.  Force rows have the fixed pattern (force_bound, 0, 0, 0, 0, 0) per
    // sample; only the foot-box right-hand sides are stored.  A row whose coefficients are all exactly zero (the
    // touch-down sample of a stance) stays out of the iteration: it keeps z == 0, s == 1 and weight 0 throughout, and
    // z > 0 is the active mask everywhere below.
    const double box0 = Hd->ee_box[0] / 2, box1 = Hd->ee_box[1] / 2;
    const double fbound = P.force_bound;
    const int m_force = 6 * ns;
    int m_act = 0;
    #pragma unroll 1
    for (int j = tid; j < ns; j += nth) {
        const bool act = samples[j].active != 0;
        for (int r = 0; r < 6; ++r) {
            S.lam[6 * j + r] = act ? 1.0 : 0.0;
            S.s[6 * j + r] = 1.0;
        }
        m_act += act ? 6 : 0;
    }
    #pragma unroll 1
    for (int e = tid; e < ne; e += nth) {
        const int c = e & 1, foot = (e >> 1) & 3, kk = e >> 3;   // node k = kk + 4
        const double bx = c ? box1 : box0;
        const double off = xoff[(kk + kEENodeStart) * kNx + c];
        S.d[2 * e + 0] = (bx + P.hip_xy[foot][c]) + off;
        S.d[2 * e + 1] = -(-bx + P.hip_xy[foot][c]) - off;
        S.lam[m_force + 2 * e + 0] = 1.0;
        S.lam[m_force + 2 * e + 1] = 1.0;
        S.s[m_force + 2 * e + 0] = 1.0;
        S.s[m_force + 2 * e + 1] = 1.0;
        m_act += 2;
    }
    auto rhs_of = [&](int i) -> double { return (i < m_force) ? ((i % 6 == 0) ? fbound : 0.0) : S.d[i - m_force]; };
    m_act = static_cast<int>(block_reduce<kSum>(static_cast<double>(m_act), S.red) + 0.5);
    kkt_build_colinfo(S.col, nu, nf, N, s_fbase, s_pbase, s_nfv, s_npv, s_sb, S.smp, S.pcnt, S.poff);
    __syncthreads();
    KktItem* kitems = reinterpret_cast<KktItem*>(ws + L.ktab);
    KktPos* kpos = reinterpret_cast<KktPos*>(ws + L.ktab + sizeof(KktItem) * kMaxKktItems);
    kkt_mma_setup(s_work, &s_nwork, (nu + 7) >> 3, kitems, &s_nitems, s_fbase, s_nfv, S.col, S.smp, kpos, &s_npos, nu, nf, s_eq, neq);
    if (s_nitems > kMaxKktItems || s_npos > kMaxKktPos) {   // cannot happen within max_spline_vars = 160; refuse rather than drop terms
        if (tid == 0) {
            Hd->status = kOther;
            Hd->no_iterate = 1;
            Hd->iters = 0;
        }
        return;
    }
    __syncthreads();
    PROF(0);
#ifdef BGG_IPM_TRACE
    const trace::Cfg tr_cfg = trace::g_cfg;
    const bool tr_on = tr_cfg.buf != nullptr && tr_cfg.instance == b;
    int tr_n = 0;
    double* tr = nullptr;   // the current record, or nullptr
    if (tr_on && tid == 0) ++trace::g_cfg.launches;
#endif

    // ------------------------------------------------------------------------------------------------ operators
    IpmCtx ctx;
    ctx.S = S; ctx.Hg = Hg; ctx.eq = s_eq; ctx.fbase = s_fbase; ctx.pbase = s_pbase; ctx.nfv = s_nfv; ctx.npv = s_npv;
    ctx.N = N; ctx.nu = nu; ctx.nf = nf; ctx.ns = ns; ctx.ne = ne; ctx.neq = neq; ctx.nkc = nkc; ctx.mu_f = mu_f;
    auto apply_C = [&](const double* v, double* out, double* eout, double rhs_scale) { PROF(10); ipm_apply_C<!kSpill, kThreads>(ctx, v, out, eout, rhs_scale); PROF(6); };
    auto add_Ct = [&](const double* y, double* out, const double* ey, double escale) { PROF(10); ipm_add_Ct<!kSpill, kThreads>(ctx, y, out, ey, escale); PROF(7); };
    auto apply_H = [&](const double* v, double* out, bool subtract) { PROF(10); ipm_apply_H(ctx, v, out, subtract); PROF(8); };

    // K = H + eps I + C' diag(wv) C + E'E/delta in 8 x 8 blocks in shared memory (csrc/bgg_kkt_mma.cuh), then chol::factor in place.
    const int nb = (nu + 7) >> 3;   // 8 x 8 blocks per side; rows nu .. 8 nb - 1 are padded with the identity
    KktMma km;
    km.K = S.K; km.Hg = Hg; km.phig = phipos; km.phi_ld = L.max_nu; km.nu = nu; km.nf = nf; km.nb = nb; km.ns = ns; km.ne = ne;
    km.neq = neq; km.nkc = nkc; km.wv = S.wv; km.pw = S.pw; km.pcnt = S.pcnt; km.poff = S.poff; km.smp = S.smp; km.eq = s_eq;
    km.col = S.col; km.ckc = S.ckc; km.scratch = S.ds; km.work = s_work; km.nwork = s_nwork; km.items = kitems; km.nitems = s_nitems; km.pos = kpos; km.npos = s_npos;
    km.mu_f = mu_f; km.inv_delta = inv_delta; km.eps = eps;
    // row weight 1 / (s/z + eps), computed where it is used: the slot that holds the weights while K is assembled is
    // overwritten by C x1 right after the factorisation (shared memory: six row vectors, as before the embedding)
    auto wrow = [&](int i) -> double {
        const double zi = S.lam[i];
        return (zi > 0.0) ? zi / (S.s[i] + eps * zi) : 0.0;
    };
    auto build_and_factor = [&]() -> bool {
        PROF(10);
        #pragma unroll 1
        for (int i = tid; i < m; i += nth) S.wv[i] = wrow(i);
        __syncthreads();
        kkt_assemble_mma(km);   // csrc/bgg_kkt_mma.cuh (also writes the identity padding)
        PROF(1);
        TRACE(if (tr != nullptr) {
            trace::put_vec(tr, trace::f_w, S.wv, m);
            trace::put_vec(tr, trace::f_K, S.K, static_cast<int>(chol::doubles(nb)));
            __syncthreads();
        });
        chol::factor(S.K, nb, &s_flag);   // csrc/bgg_chol.cuh: DMMA block Cholesky, diagonal super-blocks inverted
        PROF(3);
        return s_flag == 0;
    };
    // Solve K x = rhs in place (x padded with zeros to 8 nb entries); with `refine`, one step of iterative refinement
    // against K = H + eps I + C'WC + E'E/delta applied matrix-free.  It removes the rounding of the factorisation once W
    // has spread over many decades (block inverses, not substitutions, carry the solves: csrc/bgg_chol.cuh); without it
    // one nearly degenerate instance of the 4096 of config #2 stalls short of the tolerance where the oracle converges
    // (instance 2344; refining only the total direction is not enough: d tau is formed from x1).  The residual
    // rhs - K x accumulates in the copy of rhs.  Scratch: rhs, the ds row vector, dnu.
    auto solve_K = [&](double* x, bool refine) {
        PROF(10);
        if (refine) {
            #pragma unroll 1
            for (int i = tid; i < nu; i += nth) S.rhs[i] = x[i];
        }
        chol::solve(S.K, nb, x, S.red);
        PROF(5);
        if (refine) {
            #pragma unroll 1
            for (int i = tid; i < nu; i += nth) S.rhs[i] -= eps * x[i];
            __syncthreads();
            apply_H(x, S.rhs, true);
            apply_C(x, S.ds, S.dnu, 0.0);
            #pragma unroll 1
            for (int i = tid; i < m; i += nth) S.ds[i] *= -wrow(i);
            __syncthreads();
            add_Ct(S.ds, S.rhs, S.dnu, -inv_delta);
            PROF(10);
            chol::solve(S.K, nb, S.rhs, S.red);
            PROF(5);
            #pragma unroll 1
            for (int i = tid; i < nu; i += nth) x[i] += S.rhs[i];
            __syncthreads();
        }
    };

    double nrm_q = 1.0, nrm_d = 1.0;
    for (int r = 0; r < kNx; ++r) nrm_q = fmax(nrm_q, fmax(fabs(P.w[r]), fabs(P.Phi_w[r])));
    {
        double v = 0;
        #pragma unroll 1
        for (int i = tid; i < m; i += nth)
            if (S.lam[i] > 0.0) v = fmax(v, fabs(rhs_of(i)));
        for (int r = 0; r < neq; ++r) v = fmax(v, fabs(s_eq[r].rhs));
        nrm_d = fmax(1.0, block_reduce<kMax>(v, S.red));
    }
    if (tid < kMaxEq) S.nueq[tid] = 0.0;
    __syncthreads();

    // ------------------------------------------------------------------------------------------------ main loop
    // it == -1 is the starting point (Clarabel's QP initialisation: unit scaling, (u, z, y) from the constant solve, s = -z,
    // s and z shifted into the cone, tau = kappa = 1); it shares the factorisation and constant-solve code with the iterations.
    int it = 0, status = kMaxIter;
    double tau = 1.0, kap = 1.0, mu_first = 0.0;
    double res_p = 0, res_d = 0, gap = 0, gscale = 1, bz = 0, aty_n = 0, zn = 1, pc = 0;
    bool have_point = false;
    int n_refined = 0;
    bool confirm = false;
    for (it = -1; it <= P.ipm_max_iter; ++it) {
        double uHu = 0, rt = 0, mu = 0;
        bool refine_now = false;
        TRACE(if (tr_on) {
            using namespace trace;
            tr = begin_record(tr_cfg, tr_n++);
            put(tr, f_it, it); put(tr, f_threads, kThreads); put(tr, f_spill, kSpill); put(tr, f_stage_phi, stage_phi);
            put(tr, f_cap_nu, cap_nu); put(tr, f_cap_rows, cap_rows); put(tr, f_want, want); put(tr, f_confirm, confirm);
            put(tr, f_N, N); put(tr, f_nu, nu); put(tr, f_nf, nf); put(tr, f_nb, nb); put(tr, f_ns, ns); put(tr, f_ne, ne);
            put(tr, f_m, m); put(tr, f_neq, neq); put(tr, f_m_act, m_act);
            put(tr, f_eps, eps); put(tr, f_delta, delta); put(tr, f_mu_f, mu_f); put(tr, f_tol_feas, P.ipm_tol_feas);
            put(tr, f_tol_gap, P.ipm_tol_gap); put(tr, f_tol_infeas, P.ipm_tol_infeas); put(tr, f_nrm_q, nrm_q);
            put(tr, f_nrm_d, nrm_d); put(tr, f_cost_const, cost_const); put(tr, f_tau, tau); put(tr, f_kap, kap);
            put_vec(tr, f_u, S.u, nu); put_vec(tr, f_s, S.s, m); put_vec(tr, f_z, S.lam, m); put_vec(tr, f_y, S.nueq, neq);
            if (tr != nullptr)
                for (int i = tid; i < m; i += nth) tr[off(f_d) + i] = rhs_of(i);
            __syncthreads();
        });
        if (it >= 0) {
            // residuals  rx = H u + C'z + E'y + g tau ,  rz = C u + s - d tau ,  re = E u - e tau
            apply_H(S.u, S.Hu, false);
            #pragma unroll 1
            for (int i = tid; i < nu; i += nth) S.rd[i] = 0.0;
            __syncthreads();
            add_Ct(S.lam, S.rd, S.nueq, 1.0);
            // rz and re are linear in the iterate: after a step they are updated with the very products the step was built
            // from (below), and evaluated from scratch only at the first iteration and to confirm convergence
            const bool fresh_rz = (it == 0) || confirm;
            if (fresh_rz) apply_C(S.u, S.rp, S.re, tau);
            double r8[8] = {0, 0, 0, 0, 0, 0, 0, 1.0};   // sums: u'Hu, g'u, d'z, s'z ; maxima: |C'z + E'y|, |rx|, |rz|, z
            #pragma unroll 1
            for (int i = tid; i < nu; i += nth) {
                const double gi = gg[i], hu = S.Hu[i], ui = S.u[i], at = S.rd[i];
                r8[0] += ui * hu;
                r8[1] += gi * ui;
                r8[4] = fmax(r8[4], fabs(at));
                const double rx = hu + at + gi * tau;
                S.rd[i] = rx;
                r8[5] = fmax(r8[5], fabs(rx));
            }
            #pragma unroll 1
            for (int i = tid; i < m; i += nth) {
                const double zi = S.lam[i];
                if (zi > 0.0) {
                    const double di = rhs_of(i), rz = fresh_rz ? S.rp[i] + S.s[i] - di * tau : S.rp[i];
                    S.rp[i] = rz;
                    r8[2] += di * zi;
                    r8[3] += S.s[i] * zi;
                    r8[6] = fmax(r8[6], fabs(rz));
                    r8[7] = fmax(r8[7], zi);
                } else {
                    S.rp[i] = 0.0;
                }
            }
            PROF(10);
            block_reduce_multi<4, 4>(r8, S.red);
            PROF(13);
            uHu = r8[0];
            const double gu = r8[1];
            double ey = 0, n_re = 0;
            double yn = 0;
            for (int r = 0; r < neq; ++r) {
                ey += s_eq[r].rhs * S.nueq[r];
                n_re = fmax(n_re, fabs(S.re[r]));
                yn = fmax(yn, fabs(S.nueq[r]));
            }
            bz = r8[2] + ey;
            aty_n = r8[4];
            zn = fmax(r8[7], yn);   // max(1, |z|, |y|) over the duals this form keeps (the dynamics multipliers are eliminated)
            rt = kap + gu + bz + uHu / tau;
            mu = (r8[3] + tau * kap) / (m_act + 1);
            pc = (0.5 * uHu / tau + gu) / tau;
            const double dc = (-bz - 0.5 * uHu / tau) / tau;
            const double n_rp = fmax(r8[6], n_re) / tau, n_rd = r8[5] / tau, n_gap = fabs(pc - dc);
            if (!(n_rp == n_rp) || !(n_rd == n_rd) || !(mu == mu) || !(n_gap == n_gap) || !(tau > 0.0)) {
                status = kOther;   // cannot happen while the step below refuses non-finite directions; the outputs then
                break;             // carry the header of the last finite evaluation
            }
            res_p = n_rp;
            res_d = n_rd;
            gap = n_gap;
            gscale = fmax(1.0, fmin(fabs(pc + cost_const), fabs(dc + cost_const)));   // full objective, as Clarabel's relative gap
            have_point = true;
            TRACE(if (tr != nullptr) {
                using namespace trace;
                put(tr, f_fresh, fresh_rz); put(tr, f_mu, mu); put(tr, f_rt, rt); put(tr, f_uHu, uHu); put(tr, f_res_p, res_p);
                put(tr, f_res_d, res_d); put(tr, f_gap, gap); put(tr, f_gscale, gscale); put(tr, f_bz, bz); put(tr, f_aty_n, aty_n);
                put(tr, f_zn, zn); put(tr, f_pc, pc);
                put_vec(tr, f_Hu, S.Hu, nu); put_vec(tr, f_rx, S.rd, nu); put_vec(tr, f_rz, S.rp, m); put_vec(tr, f_re, S.re, neq);
                __syncthreads();
            });
            if (res_d <= P.ipm_tol_feas * nrm_q && res_p <= P.ipm_tol_feas * nrm_d && gap <= P.ipm_tol_gap * gscale) {
                if (fresh_rz) {
                    status = kSolved;
                    break;
                }
                confirm = true;   // same iterate once more, with the primal residuals evaluated from scratch
                --it;
                continue;
            }
            confirm = false;
            // primal infeasibility certificate (Clarabel's is_primal_infeasible): d'z + e'y < 0 with C'z + E'y ~ 0
            if (bz < -P.ipm_tol_infeas && aty_n <= P.ipm_tol_infeas * zn * (-bz)) {
                status = kPrimalInfeasible;
                break;
            }
            if (it == P.ipm_max_iter) break;
            // refinement of the solves pays for itself only once W = z / s has spread over many decades: it starts when mu
            // has fallen to ipm_refine_mu_frac of its first value; an instance still iterating at ipm_refine_from_iter is a hard
            // one (the batch average is 17 iterations) and gets it from there on
            if (it == 0) mu_first = mu;
            refine_now = P.ipm_refine > 0 && (mu <= P.ipm_refine_mu_frac * mu_first || it >= P.ipm_refine_from_iter);
            n_refined += refine_now ? 1 : 0;
        }
        if (!build_and_factor()) {
            status = kOther;
            break;
        }
        TRACE(trace::put(tr, trace::f_refine, refine_now););

        // Three solves with the one factorisation, one copy of the code: pass 0 the constant right-hand side (-g ; d ; e)
        // -> (x1, C x1, y1); pass 1 the affine step; pass 2 the combined step.  Row vectors while a pass runs: dl holds a2
        // (then dz), ds holds W a2 (then C x2, then ds).
        double den = 1.0, dtau = 0.0, dkap = 0.0, sigma = 0.0, alpha = 0.0, dkdt_aff = 0.0;
        bool bad = false;
#pragma unroll 1
        for (int pass = 0; pass < (it < 0 ? 1 : 3); ++pass) {
            const double scale = (pass == 0) ? 0.0 : (pass == 1 ? 1.0 : 1.0 - sigma);
            double* x = (pass == 0) ? S.x1 : S.du;
            double* tslot = (pass == 0) ? S.wv : S.ds;
            #pragma unroll 1
            for (int i = tid; i < m; i += nth) {
                const double zi = S.lam[i];
                if (!(zi > 0.0)) {
                    S.ds[i] = 0.0;
                    if (pass > 0) S.dl[i] = 0.0;
                    continue;
                }
                const double w = wrow(i);
                if (pass == 0) {
                    S.ds[i] = w * rhs_of(i);
                } else {
                    double d_s = S.s[i] * zi;
                    if (pass == 2) d_s += S.ds[i] * S.dl[i] - sigma * mu;
                    const double a2 = -scale * S.rp[i] + d_s / zi;
                    S.dl[i] = a2;
                    S.ds[i] = w * a2;
                }
            }
            #pragma unroll 1
            for (int i = tid; i < nu; i += nth) x[i] = (pass == 0) ? -gg[i] : -scale * S.rd[i];
            if (tid < neq) S.a3[tid] = (pass == 0) ? s_eq[tid].rhs : -scale * S.re[tid];
            __syncthreads();
            PROF(14);
            add_Ct(S.ds, x, S.a3, inv_delta);
            solve_K(x, refine_now && pass != 1);   // the affine step only steers sigma: not refined
            double* yx = (pass == 0) ? S.y1 : S.dnu;
            apply_C(x, tslot, yx, 0.0);
            if (tid < neq) yx[tid] = (yx[tid] - S.a3[tid]) * inv_delta;
            __syncthreads();
            TRACE(if (tr != nullptr && pass != 1) {
                using namespace trace;
                if (pass == 0) { put_vec(tr, f_x1, S.x1, nu); put_vec(tr, f_cx1, S.wv, m); put_vec(tr, f_y1, S.y1, neq); }
                else { put_vec(tr, f_x2, S.du, nu); put_vec(tr, f_cx2, S.ds, m); put_vec(tr, f_a2, S.dl, m); put_vec(tr, f_y2, S.dnu, neq); }
                __syncthreads();
            });
            if (it < 0) break;
            // g'x, (H u)'x, d'z_x with z_x = W (C x - a2), e'y_x
            double r3[3] = {0, 0, 0};
            #pragma unroll 1
            for (int i = tid; i < nu; i += nth) {
                r3[0] += gg[i] * x[i];
                r3[1] += S.Hu[i] * x[i];
            }
            #pragma unroll 1
            for (int i = tid; i < m; i += nth)
                if (S.lam[i] > 0.0) {
                    const double di = rhs_of(i);
                    r3[2] += di * wrow(i) * (tslot[i] - ((pass == 0) ? di : S.dl[i]));
                }
            PROF(10);
            block_reduce_multi<3, 0>(r3, S.red);
            PROF(13);
            double eyx = 0;
            for (int r = 0; r < neq; ++r) eyx += s_eq[r].rhs * yx[r];
            if (pass == 0) {
                den = kap / tau - r3[0] - r3[2] - eyx + uHu / (tau * tau) - 2.0 * r3[1] / tau;
                continue;
            }
            const double d_kap = (pass == 1) ? kap * tau : kap * tau + dkdt_aff - sigma * mu;
            dtau = (scale * rt - d_kap / tau + r3[0] + r3[2] + eyx + 2.0 * r3[1] / tau) / den;
            dkap = (-d_kap - kap * dtau) / tau;
            // total direction: (du, dz, dy) = (x2, z2, y2) + dtau (x1, z1, y1); ds from the complementarity equation (keeps the
            // relative accuracy of tiny slacks); largest step that keeps s, z, tau, kappa non-negative
            bool nf_local = !(dtau == dtau) || !(dkap == dkap) || fabs(dtau) > 1e300 || fabs(dkap) > 1e300;
            #pragma unroll 1
            for (int i = tid; i < nu; i += nth) {
                const double v = S.du[i] + dtau * S.x1[i];
                S.du[i] = v;
                nf_local |= !(fabs(v) <= 1e300);
            }
            #pragma unroll 1
            for (int i = tid; i < m; i += nth) {
                const double zi = S.lam[i];
                if (!(zi > 0.0)) continue;
                const double a2 = S.dl[i], di = rhs_of(i);
                const double t = S.ds[i] + dtau * S.wv[i];
                const double dzv = wrow(i) * (t - a2 - dtau * di);
                const double dsv = -(a2 + scale * S.rp[i]) - (S.s[i] / zi) * dzv;
                S.dl[i] = dzv;
                S.ds[i] = dsv;
                if (pass == 2) S.wv[i] = t + dsv - di * dtau;   // d rz / d alpha = C du + ds - d dtau (C x1 is not needed any more)
            }
            if (pass == 2 && tid < neq) S.a3[tid] = delta * S.dnu[tid] + dtau * delta * S.y1[tid] - scale * S.re[tid];   // d re / d alpha = E du - e dtau
            if (tid < neq) S.dnu[tid] += dtau * S.y1[tid];
            __syncthreads();
            double amax = 1.0;
            #pragma unroll 1
            for (int i = tid; i < m; i += nth) {
                const double zi = S.lam[i];
                if (!(zi > 0.0)) continue;
                const double dsv = S.ds[i], dzv = S.dl[i];
                nf_local |= !(fabs(dzv) <= 1e300) || !(fabs(dsv) <= 1e300);
                if (dsv < 0.0) amax = fmin(amax, -S.s[i] / dsv);
                if (dzv < 0.0) amax = fmin(amax, -zi / dzv);
            }
            PROF(15);
            amax = block_reduce<kMin>(amax, S.red);
            if (__syncthreads_or(nf_local ? 1 : 0)) {
                bad = true;
                break;
            }
            PROF(13);
            if (dtau < 0.0) amax = fmin(amax, -tau / dtau);
            if (dkap < 0.0) amax = fmin(amax, -kap / dkap);
            if (pass == 1) {
                sigma = (1.0 - amax) * (1.0 - amax) * (1.0 - amax);
                dkdt_aff = dkap * dtau;
            } else {
                alpha = 0.99 * amax;
                TRACE(trace::put(tr, trace::f_amax, amax););
            }
        }
        TRACE(if (tr != nullptr && it >= 0 && !bad) {
            using namespace trace;
            put(tr, f_den, den); put(tr, f_sigma, sigma); put(tr, f_dkdt_aff, dkdt_aff); put(tr, f_dtau, dtau); put(tr, f_dkap, dkap);
            put(tr, f_alpha, alpha);
            put_vec(tr, f_du, S.du, nu); put_vec(tr, f_dz, S.dl, m); put_vec(tr, f_ds, S.ds, m); put_vec(tr, f_dy, S.dnu, neq);
            put_vec(tr, f_drz, S.wv, m); put_vec(tr, f_dre, S.a3, neq);
            __syncthreads();
        });
        if (it < 0) {
            // starting point from the constant solve: u = x1, z = W (C x1 - d) with W = 1 / (1 + eps), s = -z, y = y1
            double mn[2] = {-1e300, -1e300};   // maxima of -s and -z = minus the minima
            #pragma unroll 1
            for (int i = tid; i < m; i += nth)
                if (S.lam[i] > 0.0) {
                    const double zv = (S.wv[i] - rhs_of(i)) / (1.0 + eps);
                    S.dl[i] = zv;
                    mn[0] = fmax(mn[0], zv);    // -s = z
                    mn[1] = fmax(mn[1], -zv);
                }
            block_reduce_multi<0, 2>(mn, S.red);
            const double smin = -mn[0], zmin = -mn[1];
            const double sshift = (smin < 1e-8) ? 1.0 - smin : 0.0, zshift = (zmin < 1e-8) ? 1.0 - zmin : 0.0;
            #pragma unroll 1
            for (int i = tid; i < m; i += nth)
                if (S.lam[i] > 0.0) {
                    const double zv = S.dl[i];
                    S.s[i] = -zv + sshift;
                    S.lam[i] = zv + zshift;   // > 0: stays the active mask
                }
            #pragma unroll 1
            for (int i = tid; i < nu; i += nth) S.u[i] = S.x1[i];
            if (tid < neq) S.nueq[tid] = S.y1[tid];
            __syncthreads();
            continue;
        }
        if (bad) {   // a non-finite direction (breakdown of the factorisation that the pivot test did not catch): keep the last iterate
            status = kOther;
            break;
        }
        #pragma unroll 1
        for (int i = tid; i < nu; i += nth) S.u[i] += alpha * S.du[i];
        #pragma unroll 1
        for (int i = tid; i < m; i += nth)
            if (S.lam[i] > 0.0) {
                S.s[i] += alpha * S.ds[i];
                S.lam[i] += alpha * S.dl[i];
                S.rp[i] += alpha * S.wv[i];
            }
        if (tid < neq) {
            S.nueq[tid] += alpha * S.dnu[tid];
            S.re[tid] += alpha * S.a3[tid];
        }
        tau += alpha * dtau;
        kap += alpha * dkap;
        __syncthreads();
    }
    // Exit without meeting the tolerances (iteration limit or a numerical breakdown): Clarabel's reduced tolerances decide
    // between AlmostSolved (SolvedInacc), AlmostPrimalInfeasible and the plain failure status (reduced_tol_feas 1e-4,
    // reduced_tol_gap 5e-5, reduced_tol_infeas 5e-5).  A breakdown before the first complete residual evaluation stays
    // `Other`, and k_finish then reuses the previous solution.  Same rule as oracle/qp_ipm.cpp.
    if ((status == kMaxIter || status == kOther) && have_point) {
        if (res_d <= 1e-4 * nrm_q && res_p <= 1e-4 * nrm_d && gap <= 5e-5 * gscale) status = kSolvedInacc;
        else if (bz < -5e-5 && aty_n <= 5e-5 * zn * (-bz)) status = kPrimalInfeasibleInacc;
    }
    if (it > P.ipm_max_iter) it = P.ipm_max_iter;
    if (it < 0) it = 0;
    TRACE(trace::put(tr, trace::f_status_exit, status); trace::put(tr, trace::f_iters_exit, it); trace::put(tr, trace::f_refined_exit, n_refined););

    // ------------------------------------------------------------------------------------------------ outputs
    // the de-homogenised point (u, z, s, y) / tau; without a finite evaluation (have_point == false) u = 0 is written
    // and the status (Other) makes k_finish keep the previous solution
    double* uo = reinterpret_cast<double*>(ws + L.u);
    double* lo = reinterpret_cast<double*>(ws + L.lam);
    double* so = reinterpret_cast<double*>(ws + L.slack);
    double* no = reinterpret_cast<double*>(ws + L.nueq);
    const double itau = have_point ? 1.0 / tau : 0.0;
    #pragma unroll 1
    for (int i = tid; i < nu; i += nth) uo[i] = have_point ? S.u[i] * itau : 0.0;
    #pragma unroll 1
    for (int i = tid; i < m; i += nth) {
        const bool act = S.lam[i] > 0.0;
        lo[i] = act ? S.lam[i] * itau : 0.0;
        so[i] = act ? S.s[i] * itau : rhs_of(i);   // inactive rows: slack = d (row is 0 <= d)
    }
    if (tid < neq) no[tid] = S.nueq[tid] * itau;
    PROF(10);
    PROF_DUMP;
    if (tid == 0) {
        Hd->status = status;
        Hd->no_iterate = have_point ? 0 : 1;
        Hd->refined_iters = n_refined;
        Hd->iters = it;
        Hd->prim_res = res_p;
        Hd->dual_res = res_d;
        Hd->gap = gap;
        Hd->qp_cost = pc + cost_const;
    }
    (void)delta;
    (void)npk;
    (void)gscale;
}

void launch_ipm(const Params& P, const WsLayout& L, char* ws, int B, int nu_max, int ns_max, int want, cudaStream_t stream, int sm_count) {
    const IpmCaps c = ipm_caps(L, nu_max, ns_max, B <= sm_count);
    const size_t smem = ipm_smem_for(L, c);
    // the opt-in is per device and context: set on every launch (a second handle on another GPU, or another host thread,
    // must not depend on what an earlier launch configured)
    const void* fn = c.threads == 512 ? reinterpret_cast<const void*>(k_ipm<false, 512>)
                                      : (c.spill ? reinterpret_cast<const void*>(k_ipm<true, 256>) : reinterpret_cast<const void*>(k_ipm<false, 256>));
    cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (getenv("BGG_DEBUG_OCC")) {
        int nblk = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nblk, fn, c.threads, smem);
        fprintf(stderr, "k_ipm: dynamic smem %zu B, caps nu %d rows %d, stage_phi %d, spill %d, threads %d, resident CTAs per SM %d\n", smem, c.nu, c.rows, c.stage_phi, c.spill, c.threads, nblk);
    }
    if (c.threads == 512) k_ipm<false, 512><<<B, 512, smem, stream>>>(P, L, ws, c.stage_phi, c.nu, c.rows, want);
    else if (c.spill) k_ipm<true, 256><<<B, 256, smem, stream>>>(P, L, ws, c.stage_phi, c.nu, c.rows, want);
    else k_ipm<false, 256><<<B, 256, smem, stream>>>(P, L, ws, c.stage_phi, c.nu, c.rows, want);
}

}  // namespace bgg

#ifdef BGG_IPM_PROF
extern "C" int bgg_debug_ipm_prof(long long* out32) {
    int rc = static_cast<int>(cudaMemcpyFromSymbol(out32, bgg::g_ipm_prof, 16 * sizeof(long long)));
    if (rc == 0) rc = static_cast<int>(cudaMemcpyFromSymbol(out32 + 16, bgg::chol::g_chol_prof, 16 * sizeof(long long)));
    if (rc == 0) rc = static_cast<int>(cudaMemcpyFromSymbol(out32 + 24, bgg::g_kkt_prof, 8 * sizeof(long long)));
    const long long zero[16] = {0};
    cudaMemcpyToSymbol(bgg::g_kkt_prof, zero, 8 * sizeof(long long));
    cudaMemcpyToSymbol(bgg::chol::g_chol_prof, zero, sizeof(zero));
    return rc;
}
#endif

#ifdef BGG_IPM_TRACE
// Arm the trace for the CTA of `instance` (its index in the launch's batch) with room for `cap` records; a negative instance
// disarms it.  Every later launch of k_ipm in which that CTA iterates rewrites the records from the first.
extern "C" int bgg_debug_ipm_trace_arm(int instance, int cap) {
    using namespace bgg::trace;
    Cfg c{};
    if (cudaMemcpyFromSymbol(&c, g_cfg, sizeof c) != cudaSuccess) return 1;
    if (c.buf != nullptr) cudaFree(c.buf);
    c = Cfg{};
    c.instance = -1;
    if (instance >= 0 && cap > 0) {
        if (cudaMalloc(&c.buf, sizeof(double) * kRecord * static_cast<size_t>(cap)) != cudaSuccess) return 2;
        c.instance = instance;
        c.cap = cap;
    }
    return cudaMemcpyToSymbol(g_cfg, &c, sizeof c) == cudaSuccess ? 0 : 3;
}

// hdr[0..5) = {doubles per record, fields, records written by the last traced launch, records stored, traced launches},
// then (offset, length) per field; names: the field names, comma-separated.  With recs != nullptr also copies
// min(stored, rec_cap) records.  Waits for the device.
extern "C" int bgg_debug_ipm_trace_fetch(int* hdr, int hdr_cap, char* names, int names_cap, double* recs, int rec_cap) {
    using namespace bgg::trace;
    if (hdr_cap < 5 + 2 * kFields) return 1;
    if (cudaDeviceSynchronize() != cudaSuccess) return 2;
    Cfg c{};
    if (cudaMemcpyFromSymbol(&c, g_cfg, sizeof c) != cudaSuccess) return 3;
    const int stored = c.count < c.cap ? c.count : c.cap;
    hdr[0] = kRecord; hdr[1] = kFields; hdr[2] = c.count; hdr[3] = stored; hdr[4] = c.launches;
    for (int f = 0; f < kFields; ++f) { hdr[5 + 2 * f] = off(f); hdr[6 + 2 * f] = len_of(f); }
#define BGG_TR_NAME(name, len) #name ","
    static const char kNames[] = BGG_IPM_TRACE_FIELDS(BGG_TR_NAME);
#undef BGG_TR_NAME
    if (names_cap < static_cast<int>(sizeof kNames)) return 4;
    for (size_t i = 0; i < sizeof kNames; ++i) names[i] = kNames[i];
    if (recs != nullptr && stored > 0) {
        const int n = stored < rec_cap ? stored : rec_cap;
        if (cudaMemcpy(recs, c.buf, sizeof(double) * kRecord * static_cast<size_t>(n), cudaMemcpyDeviceToHost) != cudaSuccess) return 5;
    }
    return 0;
}
#endif
