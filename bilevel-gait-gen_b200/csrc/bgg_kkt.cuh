// bilevel-gait-gen_b200 -- assembly of the reduced KKT matrix  K = H + sign * C' diag(w) C + E'E / delta  from the
// structured constraint rows, shared by the interior-point kernel (sign = +1, packed lower triangle, every Newton
// iteration) and the adjoint kernel of the gait gradient (sign = -1, dense, once).
//
// Owner-computes: the lower triangle is cut into 4 x 4 tiles, a thread owns a tile and produces every term of its
// sixteen entries before writing them once -- no read-modify-write of shared memory, one barrier for the whole
// assembly, and no work item whose length depends on how many samples a foot happens to have.
//   force x force : H + sum_q ckc[q] phi_q[i] phi_q[j]            (foot-box rows through the condensed position map)
//                     + sum over the samples that cover both variables of M(c_i, c_j) w_i w_j   (force box + pyramid)
//   pos   x force : H - sum over the nodes that use the position variable of om phi_(k,c)[j] pw
//   pos   x pos   : H + sum_k om pw pw  +  touch-down / foot-start rows / delta          (same foot and coordinate only)
// Row order of w: see csrc/bgg_ipm.cu.
#pragma once
#include "bgg_chol.cuh"
#include "bgg_kernels.cuh"

namespace bgg {

struct ColInfo {      // per spline variable: which foot / coordinate / local index, and the contiguous range of
    int16_t lo, hi;   // samples (force variable) or foot-box nodes k - 4 (position variable) whose rows contain it
    int8_t foot, coord;
    int16_t var;
};

struct KktView {
    double* K;                 // output: lower triangle in 8 x 8 blocks (PACKED, csrc/bgg_chol.cuh) or dense row-major with leading dimension ld
    int ld;
    const double* Hg;          // condensed Hessian, full symmetric nu x nu in HBM / L2
    int nu, nf, N, ns, ne, neq, nkc;
    const double* wv;          // row weights, m = 6 ns + 2 ne
    const double* phi;         // position rows of the condensed state map [nkc][phi_stride]
    int phi_stride;
    const double* pw;          // [(N-3)*4][2] foot-box position weights
    const int* pcnt;
    const int* poff;
    const Sample* smp;
    const EqRow* eq;
    const ColInfo* col;        // [nu]
    double* ckc;               // scratch [nkc]
    double mu_f, inv_delta, sign;
    const uint16_t* tile;      // optional tile table (kkt_build_tile_table); nullptr: decode by square root
};

constexpr int kTileTab = 41 * 42 / 2;   // tiles of a 164 x 164 lower triangle (max_spline_vars 160 + padding)
static_assert(kTileTab >= ((kMaxSplineVars + 3) / 4) * ((kMaxSplineVars + 3) / 4 + 1) / 2,
              "kTileTab does not cover the 4 x 4 tiles of kMaxSplineVars force variables");

// (ti << 8) | tl for t = 0 .. side (side + 1) / 2 - 1, tiles enumerated row by row
__device__ inline void kkt_build_tile_table(uint16_t* tab, int side) {
    for (int ti = threadIdx.x; ti < side; ti += blockDim.x)
        for (int tl = 0; tl <= ti; ++tl) {
            const int t = ti * (ti + 1) / 2 + tl;
            if (t < kTileTab) tab[t] = static_cast<uint16_t>((ti << 8) | tl);
        }
}

// Fills ColInfo for every spline variable (once per kernel; the tables do not change between iterations).
__device__ inline void kkt_build_colinfo(ColInfo* col, int nu, int nf, int N, const int* fbase, const int* pbase, const int* nfv,
                                         const int* npv, const int* sb, const Sample* smp, const int* pcnt, const int* poff) {
    for (int i = threadIdx.x; i < nu; i += blockDim.x) {
        ColInfo ci;
        if (i < nf) {
            int e = 0;
            while (e < kNumEE - 1 && i >= fbase[e + 1]) ++e;
            const int loc = i - fbase[e], c = loc / nfv[e], v = loc % nfv[e];
            int lo = sb[e + 1], hi = sb[e];
            for (int s = sb[e]; s < sb[e + 1]; ++s) {
                const int a = v - smp[s].off;
                if (a >= 0 && a < smp[s].cnt) {
                    if (s < lo) lo = s;
                    hi = s + 1;
                }
            }
            if (hi < lo) hi = lo;
            ci.lo = static_cast<int16_t>(lo);
            ci.hi = static_cast<int16_t>(hi);
            ci.foot = static_cast<int8_t>(e);
            ci.coord = static_cast<int8_t>(c);
            ci.var = static_cast<int16_t>(v);
        } else {
            const int pc = i - nf;
            int e = 0;
            while (e < kNumEE - 1 && pc >= pbase[e + 1]) ++e;
            const int loc = pc - pbase[e], c = loc / npv[e], v = loc % npv[e];
            int lo = N - 3, hi = 0;
            for (int kk = 0; kk < N - 3; ++kk) {
                const int kf = kk * kNumEE + e, a = v - poff[kf];
                if (a >= 0 && a < pcnt[kf]) {
                    if (kk < lo) lo = kk;
                    hi = kk + 1;
                }
            }
            if (hi < lo) hi = lo;
            ci.lo = static_cast<int16_t>(lo);
            ci.hi = static_cast<int16_t>(hi);
            ci.foot = static_cast<int8_t>(e);
            ci.coord = static_cast<int8_t>(c);
            ci.var = static_cast<int16_t>(v);
        }
        col[i] = ci;
    }
}

template <bool PACKED>
__device__ __forceinline__ double& kkt_at(const KktView& v, int i, int j) {
    return PACKED ? v.K[chol::at(i, j)] : v.K[static_cast<size_t>(i) * v.ld + j];
}

// Every thread of the CTA must call this; it ends with a barrier.  Only the lower triangle (j <= i) is written.
// Three phases, two internal barriers:
//   1. force x force 4 x 4 register tiles (dense foot-box term + H); the warps that are left without a tile in the
//      last round, and then everybody, take the position rows entry by entry (short loops over the nodes that use the
//      position variable);
//   2. force-sample rows: one work item per (foot, coordinate pair, knot pair, value/derivative pair) -- the only K
//      entries two samples can share belong to the same or to neighbouring knots -- summing over the few samples
//      that contain both variables.
#ifdef BGG_IPM_PROF
static __device__ long long g_kkt_prof[8];
#define KPROF(k) do { if (threadIdx.x == 0 && blockIdx.x == 0) { const long long t_ = clock64(); g_kkt_prof[k] += t_ - kprof_t; kprof_t = t_; } } while (0)
#else
#define KPROF(k) do { } while (0)
#endif

template <bool PACKED>
__device__ void kkt_assemble(const KktView& v, const int* fbase, const int* nfv) {
    const int tid = threadIdx.x, nth = blockDim.x, wid = tid >> 5;
#ifdef BGG_IPM_PROF
    long long kprof_t = clock64();
#endif
    const int nu = v.nu, nf = v.nf, np = nu - nf, m_force = 6 * v.ns;
    for (int q = tid; q < v.nkc; q += nth) {   // weight of the dense (node, coord) row pair, summed over the feet
        const int kk = q >> 1, c = q & 1;
        double s = 0;
        for (int foot = 0; foot < kNumEE; ++foot) {
            const int e = (kk * kNumEE + foot) * 2 + c;
            s += v.wv[m_force + 2 * e] + v.wv[m_force + 2 * e + 1];
        }
        v.ckc[q] = s;
    }
    __syncthreads();
    const int fside = (nf + 3) >> 2;
    const int ntile = fside * (fside + 1) / 2;
    for (int t = tid; t < ntile; t += nth) {
        int ti, tl;   // tile (ti, tl), tl <= ti, row by row
        if (v.tile) {
            ti = v.tile[t] >> 8;
            tl = v.tile[t] & 255;
        } else {
            ti = static_cast<int>((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
            while ((ti + 1) * (ti + 2) / 2 <= t) ++ti;
            while (ti * (ti + 1) / 2 > t) --ti;
            tl = t - ti * (ti + 1) / 2;
        }
        const int i0 = 4 * ti, l0 = 4 * tl;
        double acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int i = i0 + a, j = l0 + b;
                acc[a][b] = (i < nf && j <= i) ? v.Hg[static_cast<size_t>(i) * nu + j] : 0.0;
            }
        for (int q = 0; q < v.nkc; ++q) {
            const double* row = v.phi + static_cast<size_t>(q) * v.phi_stride;
            const double wq = v.sign * v.ckc[q];
            double ra[4], rc[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                ra[k] = (i0 + k < nf) ? wq * row[i0 + k] : 0.0;
                rc[k] = (l0 + k < nf) ? row[l0 + k] : 0.0;
            }
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) acc[a][b] += ra[a] * rc[b];
        }
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int i = i0 + a, j = l0 + b;
                if (i < nf && j <= i) kkt_at<PACKED>(v, i, j) = acc[a][b];
            }
    }
    KPROF(0);
    {
        // position rows: the warps that did not get a tile in the last (partial) round start here right away
        const int rem = ntile % nth;
        int wbusy = (rem + 31) >> 5;
        if (32 * wbusy >= nth) wbusy = 0;
        const int pth = nth - 32 * wbusy;
        if (wid >= wbusy)
            for (int idx = tid - 32 * wbusy; idx < np * nu; idx += pth) {
                const int i = nf + idx / nu, j = idx % nu;
                if (j > i) continue;
                const ColInfo ci = v.col[i];
                const int foot = ci.foot, c = ci.coord;
                double term = 0.0, eq = 0.0;
                if (j < nf) {
                    for (int kk = ci.lo; kk < ci.hi; ++kk) {
                        const int kf = kk * kNumEE + foot, e = kf * 2 + c;
                        const double om = v.wv[m_force + 2 * e] + v.wv[m_force + 2 * e + 1];
                        term -= om * v.phi[static_cast<size_t>(kk * 2 + c) * v.phi_stride + j] * v.pw[2 * kf + (ci.var - v.poff[kf])];
                    }
                } else {
                    const ColInfo cj = v.col[j];
                    if (cj.foot == foot && cj.coord == c) {
                        const int lo = ci.lo > cj.lo ? ci.lo : cj.lo, hi = ci.hi < cj.hi ? ci.hi : cj.hi;
                        for (int kk = lo; kk < hi; ++kk) {
                            const int kf = kk * kNumEE + foot, e = kf * 2 + c;
                            const double om = v.wv[m_force + 2 * e] + v.wv[m_force + 2 * e + 1];
                            term += om * v.pw[2 * kf + (ci.var - v.poff[kf])] * v.pw[2 * kf + (cj.var - v.poff[kf])];
                        }
                        const int grp = foot * 2 + c;   // equality rows of this (foot, coord): E'E / delta
                        for (int r = 0; r < v.neq; ++r) {
                            const EqRow& q = v.eq[r];
                            if (q.pad != grp) continue;
                            const int ai = i - q.col[0], aj = j - q.col[0];
                            if (ai >= 0 && ai < q.cnt && aj >= 0 && aj < q.cnt) eq += q.w[ai] * q.w[aj];
                        }
                    }
                }
                kkt_at<PACKED>(v, i, j) = v.Hg[static_cast<size_t>(i) * nu + j] + v.sign * term + v.inv_delta * eq;
            }
    }
    KPROF(1);
    __syncthreads();
    KPROF(2);
    // force-sample rows
    int ib[kNumEE + 1];
    ib[0] = 0;
#pragma unroll
    for (int e = 0; e < kNumEE; ++e) ib[e + 1] = ib[e] + 30 * nfv[e];   // 5 coordinate pairs x nfv/2 knots x 12
    for (int it = tid; it < ib[kNumEE]; it += nth) {
        int e = 0;
        while (it >= ib[e + 1]) ++e;
        const int nv = nfv[e], nk = nv >> 1, loc = it - ib[e];
        const int cp = loc / (12 * nk), rem = loc % (12 * nk), k1 = rem / 12, bits = rem % 12;
        const int dk = bits >> 2, va = (bits >> 1) & 1, vb = bits & 1;   // dk: 0 same knot, 1 previous, 2 next
        const int c1 = (cp < 3) ? cp : 2, c2 = (cp < 3) ? cp : cp - 3;    // (0,0) (1,1) (2,2) (2,0) (2,1)
        const int k2 = (dk == 0) ? k1 : (dk == 1 ? k1 - 1 : k1 + 1);
        if (k2 < 0 || k2 >= nk) continue;
        const int i = 2 * k1 + va, i2 = 2 * k2 + vb;
        if (c1 == c2 && i2 > i) continue;
        const int row = fbase[e] + c1 * nv + i, colj = fbase[e] + c2 * nv + i2;
        const ColInfo a = v.col[row], b = v.col[colj];
        const int lo = a.lo > b.lo ? a.lo : b.lo, hi = a.hi < b.hi ? a.hi : b.hi;
        double acc = 0.0;
        for (int s = lo; s < hi; ++s) {
            const Sample& sp = v.smp[s];
            const double* w6 = v.wv + 6 * s;
            double m;   // sum_r w_r c_r c_r' over the six rows' coefficient 3-vectors, entry (c1, c2)
            if (cp == 2) m = (w6[0] + w6[1]) + v.mu_f * v.mu_f * (w6[2] + w6[3] + w6[4] + w6[5]);
            else if (cp == 0) m = w6[2] + w6[3];
            else if (cp == 1) m = w6[4] + w6[5];
            else if (cp == 3) m = -v.mu_f * (w6[2] - w6[3]);
            else m = -v.mu_f * (w6[4] - w6[5]);
            acc += m * sp.w[i - sp.off] * sp.w[i2 - sp.off];
        }
        if (hi > lo) kkt_at<PACKED>(v, row, colj) += v.sign * acc;
    }
    KPROF(3);
    __syncthreads();
    KPROF(4);
}

}  // namespace bgg
