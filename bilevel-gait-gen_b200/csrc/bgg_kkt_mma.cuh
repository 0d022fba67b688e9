// bilevel-gait-gen_b200 -- assembly of the interior-point KKT matrix  K = H + C' diag(w) C + E'E / delta  into the
// 8 x 8 block-packed lower triangle of csrc/bgg_chol.cuh, every Newton iteration, on the FP64 tensor-core path.
//
// Same mathematics as kkt_assemble (csrc/bgg_kkt.cuh, still used by the adjoint kernel); what changed is where the time
// went.  Measured (tools/profile_phases.py): of 98 k cycles per assembly 76 k were the force x force tiles -- a 34-step
// loop of dependent loads of the condensed position rows phi from L2 (they do not fit in shared memory next to K at
// two CTAs per SM) -- and 30 k the force-sample items with their run-time div / mod decode.  Here:
//   1. dense part, all of it one product:  K(i, j) = H(i, j) + sum_q A(i, q) phi_q(j)  with
//        A(i, q) = w_q phi_q(i)                      for a force variable i   (w_q: summed weight of the foot-box rows of (node, coord) q)
//        A(i, q) = -om(node, foot_i, coord_i) pw(i)  for a position variable i, q of the same coordinate
//      streamed through shared memory four rows of phi at a time (double buffered, one barrier per chunk; the next
//      chunk travels L2 -> registers while the current one is multiplied), one DMMA per 8 x 8 block of K and chunk, the
//      accumulators of a warp's <= 16 blocks in registers, initialised with the blocks of H;
//   2. sparse part after one barrier, read-modify-write on distinct entries: position x position terms and E'E / delta
//      (a few dozen entries), and the force-sample terms from an item table built once per solve (KktItem: target
//      offset, sample range, coordinate pair, the two weight indices) against a per-iteration 5-vector per sample.
#pragma once
#include "bgg_chol.cuh"
#include "bgg_kkt.cuh"

namespace bgg {

struct KktItem {          // one K entry touched by force-sample rows
    int32_t koff;         // offset inside the block-packed K
    uint8_t lo, mid, hi;  // samples [lo, mid) use weight indices (a1, b1), [mid, hi) use (a2, b2)
    uint8_t cp;           // coordinate pair: 0 xx, 1 yy, 2 zz, 3 zx, 4 zy
    uint8_t a1, b1, a2, b2;
};
static_assert(sizeof(KktItem) == 12, "KktItem is read as three 32-bit words");
static_assert(kMaxSamples <= 255, "sample indices are stored in 8 bits");
constexpr int kMaxKktItems = 1536;

struct KktPos {           // one position x position entry of K (same foot and coordinate): sum_kk om pw_i pw_j + eq / delta
    int32_t koff;
    int16_t lo, hi;       // foot-box nodes kk - 4 that contain both variables
    int16_t vi, vj;       // local indices of the two variables
    int8_t foot, coord;
    int16_t pad;
    double eq;            // sum over the touch-down / foot-start rows of w_i w_j (constant over the solve)
};
static_assert(sizeof(KktPos) == 24, "KktPos layout");
constexpr int kMaxKktPos = 512;

constexpr int kAccMax = 16;   // K blocks per warp and pass

// row stride (doubles) of a staged phi chunk: >= 8 nb and = 4 mod 16, so that the fragment loads of lanes (g, t) at
// t * stride + 8 b + g hit 16 distinct 8-byte banks per half warp
__host__ __device__ inline int kkt_chunk_stride(int nb) { return ((8 * nb + 11) / 16) * 16 + 4; }
// scratch doubles the assembly needs (it lives in the ds / dl row vectors, free while K is being built)
__host__ __device__ inline int kkt_scratch_doubles(int nb, int ns) { return 8 * kkt_chunk_stride(nb) + 5 * ns; }

struct KktWork {          // dense part: two row segments of K blocks for one warp (csrc/bgg_kkt_mma.cuh, kkt_assemble_mma)
    uint8_t rowA, jA0, lenA, rowB, jB0, lenB, pad0, pad1;   // read as two 32-bit words
};
static_assert(sizeof(KktWork) == 8, "KktWork is read as two 32-bit words");
constexpr int kMaxKktWork = 32;
// row segments of at most kAccMax blocks that kkt_mma_setup lists for nb block rows (it drops any beyond kMaxKktWork)
constexpr int kkt_segments(int nb) { return nb <= 0 ? 0 : kkt_segments(nb - 1) + (nb + kAccMax - 1) / kAccMax; }
static_assert(kkt_segments((kMaxSplineVars + 7) / 8) <= kMaxKktWork, "kMaxKktWork does not cover the K blocks of kMaxSplineVars spline variables");

// shared-memory accesses by 32-bit shared-window address: inside kkt_dense_mma nothing is a generic pointer, so the
// compiler neither re-derives the window base per access nor has to assume that a store aliases its arguments
__device__ __forceinline__ double lds64(unsigned addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ unsigned lds32(unsigned addr) {
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts64(unsigned addr, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory"); }
__device__ __forceinline__ void sts128(unsigned addr, double2 v) {
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(addr), "d"(v.x), "d"(v.y) : "memory");
}
__device__ __forceinline__ double2 ldg128(const double* p) {   // H blocks: issued in program order, see kkt_dense_mma
    double2 v;
    asm volatile("ld.global.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ unsigned smem_addr(const void* p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }

struct KktDenseArgs {      // 32-bit shared-window addresses and scalars; passed by value in registers / param space
    unsigned K, wv, pw, poff, col, ckc, buf, work;
    int nwork, nu, nf, nb, nkc, m_force, phi_ld;
    double eps;               // static regularisation added to the diagonal of H
};

// Dense part of the assembly (see the file header), its own function so that its sixteen block accumulators do not
// compete for registers with the interior-point loop around it.  Every thread of the CTA; ends with a barrier.
static __device__ __noinline__ void kkt_dense_mma(const KktDenseArgs a, const double* __restrict__ Hg, const double* __restrict__ phig) {
#ifdef BGG_IPM_PROF
    long long kprof_t = clock64();
#endif
    const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, wid = tid >> 5, nwarp = nth >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int nu = a.nu, nf = a.nf, nb = a.nb, nkc = a.nkc, m_force = a.m_force;
    const int w8 = 8 * nb, stride = kkt_chunk_stride(nb);
    const int nchunk = (nkc + 3) >> 2;
    // chunk staging: this thread's (row, column) slots inside a 4 x w8 chunk
    int srow[3], scol[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int e = tid + k * nth;
        srow[k] = (e < 4 * w8) ? e / w8 : -1;
        scol[k] = e - (e / w8) * w8;
    }
    auto fetch = [&](int ch, double pf[3]) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int q = 4 * ch + srow[k];
            pf[k] = (srow[k] >= 0 && q < nkc && scol[k] < nf) ? phig[static_cast<size_t>(q) * a.phi_ld + scol[k]] : 0.0;
        }
    };
    auto stage = [&](int which, const double pf[3]) {
#pragma unroll
        for (int k = 0; k < 3; ++k)
            if (srow[k] >= 0) sts64(a.buf + 8u * (which * 4 * stride + srow[k] * stride + scol[k]), pf[k]);
    };
    double pf[3];
    for (int round = 0; round * nwarp < a.nwork; ++round) {   // every warp runs every round: the chunk barriers are CTA-wide
        const int item = round * nwarp + wid;
        int rowA = 0, jA0 = 0, lenA = 0, rowB = 0, jB0 = 0, lenB = 0;
        if (item < a.nwork) {
            const unsigned w0 = lds32(a.work + 8u * item), w1 = lds32(a.work + 8u * item + 4u);
            rowA = w0 & 255; jA0 = (w0 >> 8) & 255; lenA = (w0 >> 16) & 255; rowB = w0 >> 24; jB0 = w1 & 255; lenB = (w1 >> 8) & 255;
        }
        const int nslot = lenA + lenB;
        fetch(0, pf);
        // accumulators <- blocks of H: sixteen 16-byte loads issued back to back (clamped addresses, no branch per load; the
        // compiler otherwise turns the guarded loads into sixteen dependent L2 round trips), then the identity padding
        double2 acc[kAccMax];
#pragma unroll
        for (int u = 0; u < kAccMax; ++u) {
            const int uu = (u < nslot) ? u : 0;
            const int ib = (uu < lenA) ? rowA : rowB, jb = (uu < lenA) ? jA0 + uu : jB0 + uu - lenA;
            const int i = min(8 * ib + g, nu - 1), j = min(8 * jb + 2 * t, nu - 2);
            acc[u] = ldg128(Hg + static_cast<size_t>(i) * nu + j);
        }
#pragma unroll
        for (int u = 0; u < kAccMax; ++u) {
            const int uu = (u < nslot) ? u : 0;
            const int ib = (uu < lenA) ? rowA : rowB, jb = (uu < lenA) ? jA0 + uu : jB0 + uu - lenA;
            const int i = 8 * ib + g, j = 8 * jb + 2 * t;
            if (i >= nu) acc[u] = make_double2(i == j ? 1.0 : 0.0, i == j + 1 ? 1.0 : 0.0);
            else if (j >= nu) acc[u] = make_double2(0.0, 0.0);
            if (u >= nslot) acc[u] = make_double2(0.0, 0.0);
        }
        const int iA = 8 * rowA + g, iB = 8 * rowB + g;
        // position variable i: foot, coordinate, node range and local index (ColInfo, 8 bytes)
        auto pos_info = [&](int i, int& lo, int& hi, int& foot, int& coord, int& var) {
            const unsigned c0 = lds32(a.col + 8u * i), c1 = lds32(a.col + 8u * i + 4u);
            lo = static_cast<int16_t>(c0 & 0xffff); hi = static_cast<int16_t>(c0 >> 16);
            foot = static_cast<int8_t>(c1 & 255); coord = static_cast<int8_t>((c1 >> 8) & 255); var = static_cast<int16_t>(c1 >> 16);
        };
        int loA = 0, hiA = 0, footA = 0, coordA = -1, varA = 0, loB = 0, hiB = 0, footB = 0, coordB = -1, varB = 0;
        if (iA >= nf && iA < nu && lenA > 0) pos_info(iA, loA, hiA, footA, coordA, varA);
        if (iB >= nf && iB < nu && lenB > 0) pos_info(iB, loB, hiB, footB, coordB, varB);
        auto a_val = [&](int i, int q, double wq, unsigned row_s, int lo, int hi, int foot, int coord, int var) -> double {
            if (i < nf) return wq * lds64(row_s + 8u * i);
            const int kk = q >> 1, cq = q & 1;
            double av = 0.0;
            if (coord == cq && kk >= lo && kk < hi && q < nkc) {
                const int kf = kk * kNumEE + foot, e = kf * 2 + cq;
                const double om = lds64(a.wv + 8u * (m_force + 2 * e)) + lds64(a.wv + 8u * (m_force + 2 * e + 1));
                const int po = static_cast<int>(lds32(a.poff + 4u * kf));
                av = -om * lds64(a.pw + 8u * (2 * kf + (var - po)));
            }
            return av;
        };
        __syncthreads();   // the previous round's readers are done with the chunk buffers
        stage(0, pf);
        __syncthreads();
        KPROF(5);
        for (int ch = 0; ch < nchunk; ++ch) {
            if (ch + 1 < nchunk) fetch(ch + 1, pf);
            const unsigned row_s = a.buf + 8u * ((ch & 1) * 4 * stride + t * stride);   // row t of the chunk
            const int q = 4 * ch + t;
            const double wq = (q < nkc) ? lds64(a.ckc + 8u * q) : 0.0;
            const double aA = (lenA > 0) ? a_val(iA, q, wq, row_s, loA, hiA, footA, coordA, varA) : 0.0;
            const double aB = (lenB > 0) ? a_val(iB, q, wq, row_s, loB, hiB, footB, coordB, varB) : 0.0;
            const unsigned pA = row_s + 8u * (8 * jA0 + g), pB = row_s + 8u * (8 * (jB0 - lenA) + g);
            // One B operand ahead of the DMMA that uses it, all sixteen slots unconditionally (an empty slot multiplies by a
            // zero A operand and reads a valid address): no branch, no warp-convergence bookkeeping between the DMMAs.
            const double aBz = (lenB > 0) ? aB : 0.0;
            double b_cur = lds64(((0 < lenA) ? pA : pB));
#pragma unroll
            for (int u = 0; u < kAccMax; ++u) {
                double b_next = 0.0;
                if (u + 1 < kAccMax) b_next = lds64(((u + 1 < lenA) ? pA : pB) + 64u * (u + 1));
                chol::dmma(acc[u].x, acc[u].y, (u < lenA) ? aA : aBz, b_cur);
                b_cur = b_next;
            }
            if (ch + 1 < nchunk) stage((ch + 1) & 1, pf);
            __syncthreads();
        }
        KPROF(6);
#pragma unroll
        for (int u = 0; u < kAccMax; ++u)
            if (u < nslot) {
                const int ib = (u < lenA) ? rowA : rowB, jb = (u < lenA) ? jA0 + u : jB0 + u - lenA;
                sts128(a.K + 8u * (chol::blk(ib, jb) + (g << 3) + (t << 1)), acc[u]);
            }
    }
    __syncthreads();
}


struct KktMma {
    double* K;
    const double* Hg;          // condensed Hessian, full symmetric nu x nu in HBM / L2
    const double* phig;        // condensed position rows [nkc][phi_ld] in HBM / L2
    int phi_ld;
    int nu, nf, nb, ns, ne, neq, nkc;
    const double* wv;          // row weights, m = 6 ns + 2 ne
    const double* pw;
    const int* pcnt;
    const int* poff;
    const Sample* smp;
    const EqRow* eq;
    const ColInfo* col;
    double* ckc;               // [nkc]
    double* scratch;           // kkt_scratch_doubles(nb, ns)
    const KktWork* work;       // dense work items, one per warp and round
    int nwork;
    const KktItem* items;      // HBM / L2
    int nitems;
    const KktPos* pos;         // HBM / L2
    int npos;
    double mu_f, inv_delta, eps;
};

// Once per solve: the block map and the item table.  Every thread of the CTA; ends with a barrier.
__device__ inline void kkt_mma_setup(KktWork* work, int* nwork_shared, int nb, KktItem* items, int* nitems_shared, const int* fbase,
                                     const int* nfv, const ColInfo* col, const Sample* smp, KktPos* pos, int* npos_shared, int nu, int nf,
                                     const EqRow* eqrows, int neq) {
    const int tid = threadIdx.x, nth = blockDim.x;
    if (tid == 0) {
        int n = 0;
        if (nb + 1 <= kAccMax) {   // pair row nb-1-p (nb-p blocks) with row p (p+1 blocks): nb + 1 blocks per warp
            for (int p = 0; 2 * p <= nb - 1; ++p) {
                KktWork w;
                w.rowA = static_cast<uint8_t>(nb - 1 - p); w.jA0 = 0; w.lenA = static_cast<uint8_t>(nb - p);
                w.rowB = static_cast<uint8_t>(p); w.jB0 = 0; w.lenB = static_cast<uint8_t>((p == nb - 1 - p) ? 0 : p + 1);
                work[n++] = w;
            }
        } else {                   // row segments of at most kAccMax blocks, packed two to an item: longest first, each with
                                   // the longest remaining segment that still fits (nb = 19: 13 items instead of 22)
            uint8_t srow[kMaxKktWork], sj0[kMaxKktWork], slen[kMaxKktWork];
            bool used[kMaxKktWork];
            int ns = 0;
            for (int len = kAccMax; len >= 1; --len)       // descending by length
                for (int r = nb - 1; r >= 0; --r)
                    for (int j0 = 0; j0 <= r; j0 += kAccMax) {
                        const int l = (r + 1 - j0 < kAccMax) ? r + 1 - j0 : kAccMax;
                        if (l == len && ns < kMaxKktWork) {
                            srow[ns] = static_cast<uint8_t>(r); sj0[ns] = static_cast<uint8_t>(j0); slen[ns] = static_cast<uint8_t>(l);
                            used[ns++] = false;
                        }
                    }
            for (int a = 0; a < ns; ++a) {
                if (used[a]) continue;
                used[a] = true;
                KktWork w;
                w.rowA = srow[a]; w.jA0 = sj0[a]; w.lenA = slen[a];
                w.rowB = 0; w.jB0 = 0; w.lenB = 0;
                for (int c = a + 1; c < ns; ++c)
                    if (!used[c] && slen[a] + slen[c] <= kAccMax) {
                        used[c] = true;
                        w.rowB = srow[c]; w.jB0 = sj0[c]; w.lenB = slen[c];
                        break;
                    }
                work[n++] = w;
            }
        }
        *nwork_shared = n;
    }
    if (tid == 0) {
        *nitems_shared = 0;
        *npos_shared = 0;
    }
    __syncthreads();
    {   // position x position entries: pairs of position variables of the same foot and coordinate
        const int np = nu - nf;
        for (int idx = tid; idx < np * np; idx += nth) {
            const int i = nf + idx / np, j = nf + idx % np;
            if (j > i) continue;
            const ColInfo ci = col[i], cj = col[j];
            if (cj.foot != ci.foot || cj.coord != ci.coord) continue;
            KktPos e;
            e.koff = chol::at(i, j);
            e.lo = ci.lo > cj.lo ? ci.lo : cj.lo;
            e.hi = ci.hi < cj.hi ? ci.hi : cj.hi;
            e.vi = ci.var;
            e.vj = cj.var;
            e.foot = ci.foot;
            e.coord = ci.coord;
            e.pad = 0;
            double eq = 0.0;
            const int grp = ci.foot * 2 + ci.coord;
            for (int r = 0; r < neq; ++r) {
                const EqRow& q = eqrows[r];
                if (q.pad != grp) continue;
                const int ai = i - q.col[0], aj = j - q.col[0];
                if (ai >= 0 && ai < q.cnt && aj >= 0 && aj < q.cnt) eq += q.w[ai] * q.w[aj];
            }
            e.eq = eq;
            if (e.hi <= e.lo && eq == 0.0) continue;
            const int k = atomicAdd(npos_shared, 1);
            if (k < kMaxKktPos) pos[k] = e;
        }
    }
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
        const ColInfo a = col[row], b = col[colj];
        const int lo = a.lo > b.lo ? a.lo : b.lo, hi = a.hi < b.hi ? a.hi : b.hi;
        if (hi <= lo) continue;
        int mid = lo + 1;
        while (mid < hi && smp[mid].off == smp[lo].off) ++mid;
        KktItem item;
        item.koff = chol::at(row, colj);
        item.lo = static_cast<uint8_t>(lo);
        item.mid = static_cast<uint8_t>(mid);
        item.hi = static_cast<uint8_t>(hi);
        item.cp = static_cast<uint8_t>(cp);
        item.a1 = static_cast<uint8_t>(i - smp[lo].off);
        item.b1 = static_cast<uint8_t>(i2 - smp[lo].off);
        const int o2 = (mid < hi) ? smp[mid].off : smp[lo].off;
        item.a2 = static_cast<uint8_t>(i - o2);
        item.b2 = static_cast<uint8_t>(i2 - o2);
        const int idx = atomicAdd(nitems_shared, 1);
        if (idx < kMaxKktItems) items[idx] = item;
    }
    __syncthreads();
}

// Every thread of the CTA (blockDim.x = 256); ends with a barrier.
__device__ inline void kkt_assemble_mma(const KktMma& v) {
    const int tid = threadIdx.x, nth = blockDim.x;
    const int nu = v.nu, nf = v.nf, nb = v.nb, ns = v.ns, nkc = v.nkc, m_force = 6 * v.ns;
    const int stride = kkt_chunk_stride(nb);
#ifdef BGG_IPM_PROF
    long long kprof_t = clock64();
#endif
    double* buf = v.scratch;                 // two chunks of 4 x stride
    double* mcp = v.scratch + 8 * stride;    // [ns][5]
    // ---- per-iteration tables: weight of the dense (node, coord) row pair summed over the feet; per sample the five
    //      distinct entries of  sum_r w_r c_r c_r'  over its six rows (xx, yy, zz, zx, zy)
    for (int q = tid; q < nkc; q += nth) {
        const int kk = q >> 1, c = q & 1;
        double s = 0;
        for (int foot = 0; foot < kNumEE; ++foot) {
            const int e = (kk * kNumEE + foot) * 2 + c;
            s += v.wv[m_force + 2 * e] + v.wv[m_force + 2 * e + 1];
        }
        v.ckc[q] = s;
    }
    for (int s = tid; s < ns; s += nth) {
        const double* w6 = v.wv + 6 * s;
        mcp[5 * s + 0] = w6[2] + w6[3];
        mcp[5 * s + 1] = w6[4] + w6[5];
        mcp[5 * s + 2] = (w6[0] + w6[1]) + v.mu_f * v.mu_f * (w6[2] + w6[3] + w6[4] + w6[5]);
        mcp[5 * s + 3] = -v.mu_f * (w6[2] - w6[3]);
        mcp[5 * s + 4] = -v.mu_f * (w6[4] - w6[5]);
    }
    __syncthreads();
    KPROF(0);
    {
        KktDenseArgs a;
        a.K = smem_addr(v.K); a.wv = smem_addr(v.wv); a.pw = smem_addr(v.pw); a.poff = smem_addr(v.poff); a.col = smem_addr(v.col);
        a.ckc = smem_addr(v.ckc); a.buf = smem_addr(buf); a.work = smem_addr(v.work);
        a.eps = v.eps; a.nwork = v.nwork; a.nu = nu; a.nf = nf; a.nb = nb; a.nkc = nkc; a.m_force = m_force; a.phi_ld = v.phi_ld;
        kkt_dense_mma(a, v.Hg, v.phig);   // ends with a barrier
    }
    KPROF(1);
    KPROF(2);
    // ---- sparse part: position x position (same foot and coordinate only) and E'E / delta, from the entry table
    for (int idx = tid; idx < v.npos; idx += nth) {
        const KktPos e = v.pos[idx];
        double term = 0.0;
        for (int kk = e.lo; kk < e.hi; ++kk) {
            const int kf = kk * kNumEE + e.foot, r = kf * 2 + e.coord;
            const double om = v.wv[m_force + 2 * r] + v.wv[m_force + 2 * r + 1];
            term += om * v.pw[2 * kf + (e.vi - v.poff[kf])] * v.pw[2 * kf + (e.vj - v.poff[kf])];
        }
        v.K[e.koff] += term + v.inv_delta * e.eq;
    }
    KPROF(3);
    // ---- sparse part: force-sample rows
    for (int it = tid; it < v.nitems; it += nth) {
        const KktItem item = v.items[it];
        double acc = 0.0;
        for (int s = item.lo; s < item.mid; ++s) acc += mcp[5 * s + item.cp] * v.smp[s].w[item.a1] * v.smp[s].w[item.b1];
        for (int s = item.mid; s < item.hi; ++s) acc += mcp[5 * s + item.cp] * v.smp[s].w[item.a2] * v.smp[s].w[item.b2];
        v.K[item.koff] += acc;
    }
    __syncthreads();
    // + eps I (static regularisation of the (1,1) block): after the entry tables, which also write the diagonal
    for (int i = tid; i < nu; i += nth) v.K[chol::at(i, i)] += v.eps;
    __syncthreads();
    KPROF(4);
}

}  // namespace bgg
