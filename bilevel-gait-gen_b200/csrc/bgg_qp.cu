// bilevel-gait-gen_b200 -- generic QP solve behind the reference's solver seam: QPInterface::SetupQP / Solve
// (mpc/include/qp/qp_interface.h:30-65) as ClarabelInterface implements it (mpc/qp/clarabel_interface.cpp:29-155):
//      min 1/2 x'Px + q'x   s.t.  A x + s = b ,  s in {0} on the rows flagged equality, s >= 0 on the others
// for a batch of independent QPs that share one sparsity pattern (CSC, as Eigen::SparseMatrix hands it over).  One CTA per
// QP.  Same iteration as k_ipm (csrc/bgg_ipm.cu) -- Clarabel's homogeneous self-dual embedding with static regularisation,
// sigma = (1 - alpha_aff)^3, step fraction 0.99, infeasibility certificate -- but on dense data: this entry point serves the
// small QPs that reach the seam directly (the reference's own 3-variable cross-solver test, test/mpc_test.cpp:857-1005; the
// whole-body QP of controllers/qp_control.cpp has 42 variables), not the MPC QP, whose structure k_ipm exploits.
// Limits: n <= 128 variables (K lives in shared memory), any number of rows.  oracle/qp_ipm.cpp is the CPU restatement.
#include <cstdio>

#include "bgg_kernels.cuh"
#include "bgg_qp_common.cuh"

namespace bgg {


struct QpDims {
    int n, m, mi, me;          // variables, rows, inequality rows kept in the iteration, equality rows
    int nnzP, nnzA;
    size_t stride;             // doubles of workspace per QP
    size_t oA, oP, oV;         // offsets (doubles): dense A_I (mi x n), A_E (me x n) behind it; dense P (n x n); row vectors
};

// workspace per QP (global memory, L2 resident): dense A (rows reordered: inequality rows first), dense P, 7 row vectors
size_t qp_ws_doubles(int n, int mi, int me) { return static_cast<size_t>(mi + me) * n + static_cast<size_t>(n) * n + 7 * static_cast<size_t>(mi) + 8; }
size_t qp_smem_bytes(int n, int me) { return 8 * (static_cast<size_t>(n) * n + 7 * n + 6 * static_cast<size_t>(me > 0 ? me : 1) + 72); }

namespace {

__device__ __forceinline__ double wrow_of(double s, double z, double eps) { return z / (s + eps * z); }

}  // namespace

// in_rows / eq_rows: row indices (device) of the rows kept as inequalities / equalities; all-zero inequality rows are left
// out by the host (they read 0 <= b) and reported with s = b, y = 0.
__global__ void __launch_bounds__(256) k_qp_generic(QpDims D, const int* __restrict__ Pcol, const int* __restrict__ Prow,
                                                    const double* __restrict__ Pval, const int* __restrict__ Acol,
                                                    const int* __restrict__ Arow, const double* __restrict__ Aval,
                                                    const double* __restrict__ qv, const double* __restrict__ bv,
                                                    const int* __restrict__ in_rows, const int* __restrict__ eq_rows,
                                                    const int* __restrict__ row_slot, double* __restrict__ ws_base,
                                                    double* __restrict__ x_out, double* __restrict__ y_out, double* __restrict__ s_out,
                                                    int32_t* __restrict__ status_out, int32_t* __restrict__ iters_out,
                                                    double tol_feas, double tol_gap, double tol_inf, double eps, double delta, int max_iter) {
    const int b = blockIdx.x, tid = threadIdx.x, nth = blockDim.x;
    const int n = D.n, m = D.m, mi = D.mi, me = D.me;
    double* ws = ws_base + static_cast<size_t>(b) * D.stride;
    double* AI = ws + D.oA;                           // mi x n, row major
    double* AE = AI + static_cast<size_t>(mi) * n;    // me x n
    double* Pd = ws + D.oP;                           // n x n (full symmetric)
    double* rv = ws + D.oV;                           // s, z, ds, dz, rz, cx1, bI  (mi each)
    double *S = rv, *Z = rv + mi, *DS = rv + 2 * mi, *DZ = rv + 3 * mi, *RZ = rv + 4 * mi, *CX1 = rv + 5 * mi, *BI = rv + 6 * mi;
    const double* q = qv + static_cast<size_t>(b) * n;
    const double* bb = bv + static_cast<size_t>(b) * m;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* K = reinterpret_cast<double*>(smem_raw);   // n x n, lower triangle used
    double* x = K + static_cast<size_t>(n) * n;
    double *Px = x + n, *rx = Px + n, *x1 = rx + n, *du = x1 + n, *tmp = du + n, *aty = tmp + n;
    const int mec = me > 0 ? me : 1;
    double *y = aty + n, *re = y + mec, *dy = re + mec, *y1 = dy + mec, *a3 = y1 + mec, *bE = a3 + mec;
    double* red = bE + mec;
    __shared__ int s_flag;

    // ---- densify (values of this QP on the shared pattern)
    qp_densify(n, mi, me, Pcol, Prow, Pval + static_cast<size_t>(b) * D.nnzP, Acol, Arow, Aval + static_cast<size_t>(b) * D.nnzA, row_slot, AI, AE, Pd);
    for (int r = tid; r < mi; r += nth) BI[r] = bb[in_rows[r]];
    for (int e = tid; e < me; e += nth) bE[e] = bb[eq_rows[e]];
    __syncthreads();

    // ---- dense operators (thread per output entry; the matrices are L2 resident)
    auto mulP = [&](const double* v, double* out) {
        for (int i = tid; i < n; i += nth) {
            double acc = 0;
            for (int j = 0; j < n; ++j) acc += Pd[static_cast<size_t>(i) * n + j] * v[j];
            out[i] = acc;
        }
        __syncthreads();
    };
    auto mulAI = [&](const double* v, double* out) {    // out[mi] = A_I v
        for (int r = tid; r < mi; r += nth) {
            double acc = 0;
            for (int j = 0; j < n; ++j) acc += AI[static_cast<size_t>(r) * n + j] * v[j];
            out[r] = acc;
        }
        __syncthreads();
    };
    auto mulAE = [&](const double* v, double* out, double rhs_scale) {   // out[me] = A_E v - rhs_scale b_E
        for (int e = tid; e < me; e += nth) {
            double acc = -rhs_scale * bE[e];
            for (int j = 0; j < n; ++j) acc += AE[static_cast<size_t>(e) * n + j] * v[j];
            out[e] = acc;
        }
        __syncthreads();
    };
    auto addAt = [&](const double* yi, const double* ye, double escale, double* out) {   // out[n] += A_I' yi + escale A_E' ye
        for (int j = tid; j < n; j += nth) {
            double acc = 0;
            for (int r = 0; r < mi; ++r) acc += AI[static_cast<size_t>(r) * n + j] * yi[r];
            double ae = 0;
            for (int e = 0; e < me; ++e) ae += AE[static_cast<size_t>(e) * n + j] * ye[e];
            out[j] += acc + escale * ae;
        }
        __syncthreads();
    };
    const double inv_delta = 1.0 / delta;
    auto build_and_factor = [&](bool unit) -> bool {
        // K = P + eps I + A_I' W A_I + A_E' A_E / delta (lower triangle), then an in-place Cholesky
        for (int idx = tid; idx < n * n; idx += nth) {
            const int i = idx / n, j = idx % n;
            if (j > i) continue;
            double acc = Pd[static_cast<size_t>(i) * n + j] + (i == j ? eps : 0.0);
            for (int r = 0; r < mi; ++r) {
                const double w = unit ? 1.0 / (1.0 + eps) : wrow_of(S[r], Z[r], eps);
                acc += w * AI[static_cast<size_t>(r) * n + i] * AI[static_cast<size_t>(r) * n + j];
            }
            double ae = 0;
            for (int e = 0; e < me; ++e) ae += AE[static_cast<size_t>(e) * n + i] * AE[static_cast<size_t>(e) * n + j];
            K[static_cast<size_t>(i) * n + j] = acc + inv_delta * ae;
        }
        if (tid == 0) s_flag = 0;
        __syncthreads();
        for (int k = 0; k < n; ++k) {
            if (tid == 0) {
                const double d = K[static_cast<size_t>(k) * n + k];
                if (!(d > 0.0)) s_flag = 1;
                K[static_cast<size_t>(k) * n + k] = sqrt(d > 0.0 ? d : 1.0);
            }
            __syncthreads();
            const double lkk = K[static_cast<size_t>(k) * n + k];
            for (int i = k + 1 + tid; i < n; i += nth) K[static_cast<size_t>(i) * n + k] /= lkk;
            __syncthreads();
            for (int idx = tid; idx < (n - k - 1) * (n - k - 1); idx += nth) {
                const int i = k + 1 + idx / (n - k - 1), j = k + 1 + idx % (n - k - 1);
                if (j <= i) K[static_cast<size_t>(i) * n + j] -= K[static_cast<size_t>(i) * n + k] * K[static_cast<size_t>(j) * n + k];
            }
            __syncthreads();
        }
        return s_flag == 0;
    };
    auto chol_solve = [&](double* v) {   // in place; one warp runs the two substitutions
        if (tid < 32) {
            for (int i = 0; i < n; ++i) {
                double acc = 0;
                for (int j = tid; j < i; j += 32) acc += K[static_cast<size_t>(i) * n + j] * v[j];
                acc = warp_sum(acc);
                if (tid == 0) v[i] = (v[i] - acc) / K[static_cast<size_t>(i) * n + i];
                __syncwarp();
            }
            for (int i = n - 1; i >= 0; --i) {
                double acc = 0;
                for (int j = i + 1 + tid; j < n; j += 32) acc += K[static_cast<size_t>(j) * n + i] * v[j];
                acc = warp_sum(acc);
                if (tid == 0) v[i] = (v[i] - acc) / K[static_cast<size_t>(i) * n + i];
                __syncwarp();
            }
        }
        __syncthreads();
    };
    auto reduce_sum = [&](double v) { return block_reduce<kSum>(v, red); };
    auto reduce_max = [&](double v) { return block_reduce<kMax>(v, red); };

    for (int i = tid; i < n; i += nth) x[i] = 0.0;
    for (int r = tid; r < mi; r += nth) { S[r] = 1.0; Z[r] = 1.0; }
    for (int e = tid; e < me; e += nth) y[e] = 0.0;
    double nrm_q = 0, nrm_b = 0;
    for (int i = tid; i < n; i += nth) nrm_q = fmax(nrm_q, fabs(q[i]));
    for (int r = tid; r < m; r += nth) nrm_b = fmax(nrm_b, fabs(bb[r]));
    nrm_q = fmax(1.0, reduce_max(nrm_q));
    nrm_b = fmax(1.0, reduce_max(nrm_b));

    int it = 0, status = kMaxIter;
    double tau = 1.0, kap = 1.0, res_p = 0, res_d = 0, gap = 0, gscale = 1, bz = 0, aty_n = 0, zn = 1;
    bool have_point = false;
    for (it = -1; it <= max_iter; ++it) {
        double xPx = 0, rt = 0, mu = 0;
        if (it >= 0) {
            mulP(x, Px);
            for (int i = tid; i < n; i += nth) aty[i] = 0.0;
            __syncthreads();
            addAt(Z, y, 1.0, aty);
            mulAI(x, RZ);
            mulAE(x, re, tau);
            double v0 = 0, v1 = 0, a_n = 0, rx_n = 0;
            for (int i = tid; i < n; i += nth) {
                v0 += x[i] * Px[i];
                v1 += q[i] * x[i];
                a_n = fmax(a_n, fabs(aty[i]));
                rx[i] = Px[i] + aty[i] + q[i] * tau;
                rx_n = fmax(rx_n, fabs(rx[i]));
            }
            double v2 = 0, v3 = 0, rz_n = 0, z_n = 1.0;
            for (int r = tid; r < mi; r += nth) {
                RZ[r] = RZ[r] + S[r] - BI[r] * tau;
                v2 += BI[r] * Z[r];
                v3 += S[r] * Z[r];
                rz_n = fmax(rz_n, fabs(RZ[r]));
                z_n = fmax(z_n, Z[r]);
            }
            for (int e = tid; e < me; e += nth) {
                v2 += bE[e] * y[e];
                rz_n = fmax(rz_n, fabs(re[e]));
            }
            xPx = reduce_sum(v0);
            const double qx = reduce_sum(v1);
            bz = reduce_sum(v2);
            const double sz = reduce_sum(v3);
            aty_n = reduce_max(a_n);
            const double n_rx = reduce_max(rx_n), n_rz = reduce_max(rz_n);
            zn = reduce_max(z_n);
            rt = kap + qx + bz + xPx / tau;
            mu = (sz + tau * kap) / (mi + 1);
            const double pc = (0.5 * xPx / tau + qx) / tau, dc = (-bz - 0.5 * xPx / tau) / tau;
            const double n_rp = n_rz / tau, n_rd = n_rx / tau, n_gap = fabs(pc - dc);
            if (!(n_rp == n_rp) || !(n_rd == n_rd) || !(mu == mu) || !(tau > 0.0)) {
                status = kOther;
                break;
            }
            res_p = n_rp; res_d = n_rd; gap = n_gap;
            gscale = fmax(1.0, fmin(fabs(pc), fabs(dc)));
            have_point = true;
            if (res_d <= tol_feas * nrm_q && res_p <= tol_feas * nrm_b && gap <= tol_gap * gscale) { status = kSolved; break; }
            if (bz < -tol_inf && aty_n <= tol_inf * zn * (-bz)) { status = kPrimalInfeasible; break; }
            if (it == max_iter) break;
        }
        if (!build_and_factor(it < 0)) { status = kOther; break; }
        double den = 1, dtau = 0, dkap = 0, sigma = 0, alpha = 0, dkdt_aff = 0;
        bool bad = false;
        for (int pass = 0; pass < (it < 0 ? 1 : 3); ++pass) {
            const double scale = (pass == 0) ? 0.0 : (pass == 1 ? 1.0 : 1.0 - sigma);
            double* xx = (pass == 0) ? x1 : du;
            double* tslot = (pass == 0) ? CX1 : DS;
            for (int r = tid; r < mi; r += nth) {
                const double w = (it < 0) ? 1.0 / (1.0 + eps) : wrow_of(S[r], Z[r], eps);
                if (pass == 0) {
                    DS[r] = w * BI[r];
                } else {
                    double d_s = S[r] * Z[r];
                    if (pass == 2) d_s += DS[r] * DZ[r] - sigma * mu;
                    const double a2 = -scale * RZ[r] + d_s / Z[r];
                    DZ[r] = a2;
                    DS[r] = w * a2;
                }
            }
            for (int i = tid; i < n; i += nth) xx[i] = (pass == 0) ? -q[i] : -scale * rx[i];
            for (int e = tid; e < me; e += nth) a3[e] = (pass == 0) ? bE[e] : -scale * re[e];
            __syncthreads();
            addAt(DS, a3, inv_delta, xx);
            chol_solve(xx);
            mulAI(xx, tslot);
            double* yx = (pass == 0) ? y1 : dy;
            mulAE(xx, yx, 0.0);
            for (int e = tid; e < me; e += nth) yx[e] = (yx[e] - a3[e]) * inv_delta;
            __syncthreads();
            if (it < 0) break;
            double g0 = 0, g1 = 0, g2 = 0;
            for (int i = tid; i < n; i += nth) { g0 += q[i] * xx[i]; g1 += Px[i] * xx[i]; }
            for (int r = tid; r < mi; r += nth) g2 += BI[r] * wrow_of(S[r], Z[r], eps) * (tslot[r] - ((pass == 0) ? BI[r] : DZ[r]));
            for (int e = tid; e < me; e += nth) g2 += bE[e] * yx[e];
            g0 = reduce_sum(g0); g1 = reduce_sum(g1); g2 = reduce_sum(g2);
            if (pass == 0) {
                den = kap / tau - g0 - g2 + xPx / (tau * tau) - 2.0 * g1 / tau;
                continue;
            }
            const double d_kap = (pass == 1) ? kap * tau : kap * tau + dkdt_aff - sigma * mu;
            dtau = (scale * rt - d_kap / tau + g0 + g2 + 2.0 * g1 / tau) / den;
            dkap = (-d_kap - kap * dtau) / tau;
            int nf_local = !(dtau == dtau) || !(dkap == dkap) || fabs(dtau) > 1e300 || fabs(dkap) > 1e300;
            for (int i = tid; i < n; i += nth) {
                du[i] += dtau * x1[i];
                nf_local |= !(fabs(du[i]) <= 1e300);
            }
            double amax = 1.0;
            for (int r = tid; r < mi; r += nth) {
                const double a2 = DZ[r], t = DS[r] + dtau * CX1[r];
                const double dzv = wrow_of(S[r], Z[r], eps) * (t - a2 - dtau * BI[r]);
                const double dsv = -(a2 + scale * RZ[r]) - (S[r] / Z[r]) * dzv;
                DZ[r] = dzv;
                DS[r] = dsv;
                nf_local |= !(fabs(dzv) <= 1e300) || !(fabs(dsv) <= 1e300);
                if (dsv < 0.0) amax = fmin(amax, -S[r] / dsv);
                if (dzv < 0.0) amax = fmin(amax, -Z[r] / dzv);
            }
            for (int e = tid; e < me; e += nth) dy[e] += dtau * y1[e];
            amax = block_reduce<kMin>(amax, red);
            if (__syncthreads_or(nf_local)) { bad = true; break; }
            if (dtau < 0.0) amax = fmin(amax, -tau / dtau);
            if (dkap < 0.0) amax = fmin(amax, -kap / dkap);
            if (pass == 1) { sigma = (1.0 - amax) * (1.0 - amax) * (1.0 - amax); dkdt_aff = dkap * dtau; }
            else alpha = 0.99 * amax;
        }
        if (it < 0) {   // starting point: (x, z, y) from the constant solve, s = -z, both shifted into the cone
            double mns = 1e300, mnz = 1e300;
            for (int r = tid; r < mi; r += nth) {
                const double zv = (CX1[r] - BI[r]) / (1.0 + eps);
                DZ[r] = zv;
                mns = fmin(mns, -zv);
                mnz = fmin(mnz, zv);
            }
            mns = block_reduce<kMin>(mns, red);
            mnz = block_reduce<kMin>(mnz, red);
            const double sshift = (mns < 1e-8) ? 1.0 - mns : 0.0, zshift = (mnz < 1e-8) ? 1.0 - mnz : 0.0;
            for (int r = tid; r < mi; r += nth) { S[r] = -DZ[r] + sshift; Z[r] = DZ[r] + zshift; }
            for (int i = tid; i < n; i += nth) x[i] = x1[i];
            for (int e = tid; e < me; e += nth) y[e] = y1[e];
            __syncthreads();
            continue;
        }
        if (bad) { status = kOther; break; }
        for (int i = tid; i < n; i += nth) x[i] += alpha * du[i];
        for (int r = tid; r < mi; r += nth) { S[r] += alpha * DS[r]; Z[r] += alpha * DZ[r]; }
        for (int e = tid; e < me; e += nth) y[e] += alpha * dy[e];
        tau += alpha * dtau;
        kap += alpha * dkap;
        __syncthreads();
    }
    if ((status == kMaxIter || status == kOther) && have_point) {
        if (res_d <= 1e-4 * nrm_q && res_p <= 1e-4 * nrm_b && gap <= 5e-5 * gscale) status = kSolvedInacc;
        else if (bz < -5e-5 && aty_n <= 5e-5 * zn * (-bz)) status = kPrimalInfeasibleInacc;
    }
    if (it > max_iter) it = max_iter;
    if (it < 0) it = 0;
    // ---- outputs in the caller's row order: y = multipliers, s = slacks (b - A x on the rows that were left out)
    const double itau = have_point ? 1.0 / tau : 0.0;
    for (int i = tid; i < n; i += nth) x_out[static_cast<size_t>(b) * n + i] = x[i] * itau;
    for (int r = tid; r < m; r += nth) {
        const int slot = row_slot[r];
        double yv = 0.0, sv = 0.0;
        if (slot >= 0) { yv = Z[slot] * itau; sv = S[slot] * itau; }
        else if (slot < -1) { yv = y[-(slot + 2)] * itau; }
        else { sv = bb[r]; }
        y_out[static_cast<size_t>(b) * m + r] = yv;
        s_out[static_cast<size_t>(b) * m + r] = sv;
    }
    if (tid == 0) {
        status_out[b] = status;
        iters_out[b] = it;
    }
}

int launch_qp_generic(int count, int n, int m, int mi, int me, int nnzP, int nnzA, const int* Pcol, const int* Prow, const double* Pval,
                      const int* Acol, const int* Arow, const double* Aval, const double* q, const double* b, const int* in_rows,
                      const int* eq_rows, const int* row_slot, double* ws, double* x, double* y, double* s, int32_t* status, int32_t* iters,
                      double tol_feas, double tol_gap, double tol_inf, double eps, double delta, int max_iter, int max_smem, cudaStream_t stream) {
    QpDims D;
    D.n = n; D.m = m; D.mi = mi; D.me = me; D.nnzP = nnzP; D.nnzA = nnzA;
    D.stride = qp_ws_doubles(n, mi, me);
    D.oA = 0;
    D.oP = static_cast<size_t>(mi + me) * n;
    D.oV = D.oP + static_cast<size_t>(n) * n;
    const size_t smem = qp_smem_bytes(n, me);
    if (smem > static_cast<size_t>(max_smem)) return -1;
    cudaFuncSetAttribute(k_qp_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    k_qp_generic<<<count, 256, smem, stream>>>(D, Pcol, Prow, Pval, Acol, Arow, Aval, q, b, in_rows, eq_rows, row_slot, ws, x, y, s, status, iters,
                                               tol_feas, tol_gap, tol_inf, eps, delta, max_iter);
    return 0;
}

}  // namespace bgg
