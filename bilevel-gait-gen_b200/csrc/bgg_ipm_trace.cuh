// bilevel-gait-gen_b200 -- per-iteration trace of k_ipm, compiled in only with -DBGG_IPM_TRACE into a separate library
// (tools/build_trace.sh), never into libbgg_b200.so.  One armed CTA (the instance index) writes one record per pass of the
// interior-point loop, the starting point (it = -1) and the confirmation re-evaluations included, into a device buffer:
// the launch facts, the iterate at the top of the pass, the residuals as the kernel holds them, the row weights, K after
// the assembly and before the factorisation, the solve vectors, the total direction, the scalars of the step and, in the
// last record, the exit status.  Every field is a run of doubles at a fixed offset inside the record; the offsets, lengths
// and names travel with the records (bgg_debug_ipm_trace_fetch), so a reader needs no copy of this table.
// Fields a record does not reach (a pass that stops at the convergence test has no direction) stay NaN.
#pragma once
#include "bgg_chol.cuh"
#include "bgg_ws.cuh"

namespace bgg {
namespace trace {

constexpr int kNu = kMaxSplineVars;                                   // spline variables
constexpr int kRows = 6 * kMaxSamples + 2 * (kMaxNodes - 3) * 8;      // inequality rows (WsLayout::max_rows at N = kMaxNodes)
constexpr int kEq = kMaxEq;
constexpr int kK = (kMaxSplineVars / 8) * (kMaxSplineVars / 8 + 1) / 2 * 64;   // block-packed lower triangle of K

// name, length.  Integers are stored as doubles.
#define BGG_IPM_TRACE_FIELDS(X)                                                                                              \
    X(it, 1) X(threads, 1) X(spill, 1) X(stage_phi, 1) X(cap_nu, 1) X(cap_rows, 1) X(want, 1) X(confirm, 1) X(fresh, 1)       \
    X(refine, 1) X(N, 1) X(nu, 1) X(nf, 1) X(nb, 1) X(ns, 1) X(ne, 1) X(m, 1) X(neq, 1) X(m_act, 1)                            \
    X(eps, 1) X(delta, 1) X(mu_f, 1) X(tol_feas, 1) X(tol_gap, 1) X(tol_infeas, 1) X(nrm_q, 1) X(nrm_d, 1) X(cost_const, 1)   \
    X(tau, 1) X(kap, 1) X(mu, 1) X(rt, 1) X(uHu, 1) X(res_p, 1) X(res_d, 1) X(gap, 1) X(gscale, 1) X(bz, 1) X(aty_n, 1)       \
    X(zn, 1) X(pc, 1) X(den, 1) X(sigma, 1) X(dkdt_aff, 1) X(dtau, 1) X(dkap, 1) X(amax, 1) X(alpha, 1)                       \
    X(status_exit, 1) X(iters_exit, 1) X(refined_exit, 1)                                                                    \
    X(d, kRows) X(u, kNu) X(s, kRows) X(z, kRows) X(y, kEq) X(Hu, kNu) X(rx, kNu) X(rz, kRows) X(re, kEq) X(w, kRows)         \
    X(K, kK) X(x1, kNu) X(cx1, kRows) X(y1, kEq) X(x2, kNu) X(cx2, kRows) X(a2, kRows) X(y2, kEq)                             \
    X(du, kNu) X(dz, kRows) X(ds, kRows) X(dy, kEq) X(drz, kRows) X(dre, kEq)

enum Field {
#define BGG_TR_ENUM(name, len) f_##name,
    BGG_IPM_TRACE_FIELDS(BGG_TR_ENUM)
#undef BGG_TR_ENUM
    kFields
};
#define BGG_TR_LEN(name, len) len,
__host__ __device__ constexpr int len_of(int f) {
    constexpr int lens[] = {BGG_IPM_TRACE_FIELDS(BGG_TR_LEN)};
    return lens[f];
}
#undef BGG_TR_LEN
__host__ __device__ constexpr int off(int f) {
    int o = 0;
    for (int i = 0; i < f; ++i) o += len_of(i);
    return o;
}
constexpr int kRecord = off(kFields);   // doubles per record

struct Cfg {
    double* buf;      // cap records
    int instance;     // the CTA (instance index) that writes; -1: disarmed
    int cap;
    int count;        // records the last traced launch wrote (may exceed cap: the rest were dropped)
    int launches;     // traced launches since arming
};
__device__ Cfg g_cfg;

// Record n of the armed CTA, every entry set to NaN, or nullptr (not the armed CTA, or the buffer is full).  Uniform over
// the CTA; every thread of it calls this.
__device__ inline double* begin_record(const Cfg& c, int n) {
    if (threadIdx.x == 0) g_cfg.count = n + 1;
    if (n >= c.cap) return nullptr;
    double* r = c.buf + static_cast<size_t>(n) * kRecord;
    for (int i = threadIdx.x; i < kRecord; i += blockDim.x) r[i] = __longlong_as_double(0x7ff8000000000000ll);
    __syncthreads();
    return r;
}
__device__ inline void put(double* rec, int f, double v) {
    if (rec != nullptr && threadIdx.x == 0) rec[off(f)] = v;
}
__device__ inline void put_vec(double* rec, int f, const double* src, int n) {
    if (rec == nullptr) return;
    for (int i = threadIdx.x; i < n; i += blockDim.x) rec[off(f) + i] = src[i];
}

}  // namespace trace
}  // namespace bgg
