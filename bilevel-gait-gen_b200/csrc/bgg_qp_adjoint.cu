// bilevel-gait-gen_b200 -- derivative of the generic QP solve (csrc/bgg_qp.cu) at a primal-dual point: the differential system
// of ClarabelInterface::SetupDerivativeCalcs (mpc/qp/clarabel_interface.cpp:262-602) and the outputs of CalcDerivativeWrtVecs /
// CalcDerivativeWrtMats (:182-260), for a batch of independent QPs of one sparsity pattern.  With G the inequality rows of A,
// Ae the equality rows, lam = y on G's rows and nu = y on Ae's rows, the reference solves (the +D(s) block is its own)
//      [ P    G'D(lam)   Ae' ] [dz  ]      [dx]
//      [ G    D(s)       0   ] [dlam]  = - [0 ]
//      [ Ae   0          0   ] [dnu ]      [0 ]
// and reports dq = dz, db = -dnu, dh = -lam o dlam, dA = dnu x' + nu dz' (equality rows), dG = D(lam) dlam x' + lam dz'
// (inequality rows).  tests/qp_adjoint_ref.py is the CPU restatement.
//
// One CTA per QP.  dlam = -(G dz) / s is eliminated, which leaves the bordered system
//      [ P - G'D(lam/s)G   Ae' ] [dz ]   [-dx]
//      [ Ae                0   ] [dnu] = [ 0 ]
// of size n + me.  It is indefinite, so it is factored in shared memory by LU with partial pivoting (as k_gradient,
// csrc/bgg_gradient.cu, factors the MPC's own system).  lam/s reaches 1e9 - 1e10 on active rows, so the reduced matrix alone
// does not give the unreduced system's accuracy: two steps of iterative refinement follow, with residuals of the unreduced
// operator taken matrix-free and corrections through the same factors.
// Limits: n <= 128 (as the solve) and n + me <= 160: K is (n + me)^2 doubles of shared memory (200 KB at 160).
#include <cstdio>

#include "bgg_kernels.cuh"
#include "bgg_qp_common.cuh"

namespace bgg {

constexpr int kQpAdjMaxDim = 160;   // n + me

struct QpAdjDims {
    int n, m, mi, me, nnzP, nnzA;
    size_t stride;             // doubles of workspace per QP
};

// workspace per QP (global memory): dense A_I (mi x n), A_E (me x n), P (n x n), then lam, s, w = lam/s, dlam, r2 (mi each)
size_t qp_adj_ws_doubles(int n, int mi, int me) { return static_cast<size_t>(mi + me) * n + static_cast<size_t>(n) * n + 5 * static_cast<size_t>(mi) + 8; }
// K (N x N), six vectors of N, N pivot indices
size_t qp_adj_smem_bytes(int n, int me) {
    const size_t N = static_cast<size_t>(n + me);
    return 8 * (N * N + 6 * N) + 4 * N;
}

namespace {
__device__ __forceinline__ bool is_fin(double v) { return fabs(v) <= 1.7976931348623157e308; }
}  // namespace

// Outputs (any may be null): dz [count][n]; dy [count][m] (dlam / dnu in the caller's row order, 0 on dropped rows); db [count][m]
// (-dnu on equality rows, dh = -lam dlam on inequality rows); dA [count][nnzA] on A's pattern; status [count]
// (0 ok, 1 zero / non-finite pivot or non-finite result, 2 s <= 0 on a kept inequality row or a non-finite input).
__global__ void __launch_bounds__(256) k_qp_adjoint(QpAdjDims D, const int* __restrict__ Pcol, const int* __restrict__ Prow,
                                                    const double* __restrict__ Pval, const int* __restrict__ Acol,
                                                    const int* __restrict__ Arow, const double* __restrict__ Aval,
                                                    const int* __restrict__ in_rows, const int* __restrict__ eq_rows,
                                                    const int* __restrict__ row_slot, const double* __restrict__ xv,
                                                    const double* __restrict__ yv, const double* __restrict__ sv,
                                                    const double* __restrict__ dxv, double* __restrict__ ws_base,
                                                    double* __restrict__ dz_out, double* __restrict__ dy_out, double* __restrict__ db_out,
                                                    double* __restrict__ dA_out, int32_t* __restrict__ status_out) {
    const int b = blockIdx.x, tid = threadIdx.x, nth = blockDim.x;
    const int lane = tid & 31;
    const int n = D.n, m = D.m, mi = D.mi, me = D.me, N = n + me;
    double* ws = ws_base + static_cast<size_t>(b) * D.stride;
    double* AI = ws;                                     // mi x n
    double* AE = AI + static_cast<size_t>(mi) * n;       // me x n
    double* Pd = AE + static_cast<size_t>(me) * n;       // n x n
    double *LAM = Pd + static_cast<size_t>(n) * n, *S = LAM + mi, *W = S + mi, *DL = W + mi, *R2 = DL + mi;
    const double* Pv = Pval + static_cast<size_t>(b) * D.nnzP;
    const double* Av = Aval + static_cast<size_t>(b) * D.nnzA;
    const double* x = xv + static_cast<size_t>(b) * n;
    const double* y = yv + static_cast<size_t>(b) * m;
    const double* s = sv + static_cast<size_t>(b) * m;
    const double* dx = dxv + static_cast<size_t>(b) * n;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* K = reinterpret_cast<double*>(smem_raw);     // N x N row major: the bordered matrix, then its LU factors
    double* sol = K + static_cast<size_t>(N) * N;        // [dz | dnu]
    double* cor = sol + N;                               // right-hand side / correction
    double* xs = cor + N;                                // x (n)
    double* nu = xs + N;                                 // nu (me)
    double* t0 = nu + N;                                 // scratch (n)
    double* t1 = t0 + N;
    int* piv = reinterpret_cast<int*>(t1 + N);
    __shared__ int s_flag;

    // ---- inputs: dense copies, the row vectors in slot order, the checks of status 2
    qp_densify(n, mi, me, Pcol, Prow, Pv, Acol, Arow, Av, row_slot, AI, AE, Pd);
    int bad = 0;
    for (int k = tid; k < D.nnzP; k += nth) bad |= !is_fin(Pv[k]);
    for (int k = tid; k < D.nnzA; k += nth) bad |= !is_fin(Av[k]);
    for (int r = tid; r < m; r += nth) bad |= !is_fin(y[r]) || !is_fin(s[r]);
    for (int i = tid; i < n; i += nth) {
        bad |= !is_fin(x[i]) || !is_fin(dx[i]);
        xs[i] = x[i];
    }
    for (int r = tid; r < mi; r += nth) {
        const double lr = y[in_rows[r]], sr = s[in_rows[r]];
        bad |= !(sr > 0.0);
        LAM[r] = lr;
        S[r] = sr;
        W[r] = lr / sr;
    }
    for (int e = tid; e < me; e += nth) nu[e] = y[eq_rows[e]];
    int status = __syncthreads_or(bad) ? 2 : 0;

    // dense products on the workspace (thread per output entry)
    auto mulG = [&](const double* v, double* out, int rows, const double* M) {   // out = M v, M rows x n
        for (int r = tid; r < rows; r += nth) {
            double acc = 0;
            for (int j = 0; j < n; ++j) acc += M[static_cast<size_t>(r) * n + j] * v[j];
            out[r] = acc;
        }
    };
    // forward / back substitution with the LU factors and pivots, in place on a shared vector of N; one warp
    auto lu_solve = [&](double* v) {
        if (tid < 32) {
            if (lane == 0)
                for (int k = 0; k < N; ++k)
                    if (piv[k] != k) { const double t = v[k]; v[k] = v[piv[k]]; v[piv[k]] = t; }
            __syncwarp();
            for (int i = 0; i < N; ++i) {
                double acc = 0;
                for (int j = lane; j < i; j += 32) acc += K[static_cast<size_t>(i) * N + j] * v[j];
                acc = warp_sum(acc);
                if (lane == 0) v[i] -= acc;
                __syncwarp();
            }
            for (int i = N - 1; i >= 0; --i) {
                double acc = 0;
                for (int j = i + 1 + lane; j < N; j += 32) acc += K[static_cast<size_t>(i) * N + j] * v[j];
                acc = warp_sum(acc);
                if (lane == 0) v[i] = (v[i] - acc) / K[static_cast<size_t>(i) * N + i];
                __syncwarp();
            }
        }
        __syncthreads();
    };

    if (status == 0) {
        // ---- K = [P - G'D(w)G, Ae'; Ae, 0], the (1,1) block from its lower triangle
        for (int idx = tid; idx < N * N; idx += nth) {
            const int i = idx / N, j = idx % N;
            if (i < n && j < n) {
                if (j > i) continue;
                double acc = Pd[static_cast<size_t>(i) * n + j];
                for (int r = 0; r < mi; ++r) acc -= W[r] * AI[static_cast<size_t>(r) * n + i] * AI[static_cast<size_t>(r) * n + j];
                K[static_cast<size_t>(i) * N + j] = acc;
                K[static_cast<size_t>(j) * N + i] = acc;
            } else if (i >= n && j < n) {
                K[idx] = AE[static_cast<size_t>(i - n) * n + j];
            } else if (i < n) {
                K[idx] = AE[static_cast<size_t>(j - n) * n + i];
            } else {
                K[idx] = 0.0;
            }
        }
        if (tid == 0) s_flag = 0;
        __syncthreads();
        // ---- LU with partial pivoting, right-looking, in place (multipliers by division: rows that are copies of the pivot row
        // cancel exactly, so a repeated equality row ends in an exact zero pivot)
        for (int k = 0; k < N; ++k) {
            if (tid < 32) {
                double best = -1.0;
                int bi = k, nan_seen = 0;
                for (int i = k + lane; i < N; i += 32) {
                    const double a = fabs(K[static_cast<size_t>(i) * N + k]);
                    nan_seen |= !(a == a);
                    if (a > best) { best = a; bi = i; }
                }
                for (int o = 16; o > 0; o >>= 1) {
                    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
                }
                nan_seen = __any_sync(0xffffffffu, nan_seen);
                if (lane == 0) {
                    piv[k] = bi;
                    if (nan_seen || !(best > 0.0) || !is_fin(best)) s_flag = 1;
                }
            }
            __syncthreads();
            if (s_flag) break;
            const int pk = piv[k];
            if (pk != k)
                for (int j = tid; j < N; j += nth) {
                    const double t = K[static_cast<size_t>(k) * N + j];
                    K[static_cast<size_t>(k) * N + j] = K[static_cast<size_t>(pk) * N + j];
                    K[static_cast<size_t>(pk) * N + j] = t;
                }
            __syncthreads();
            const double dkk = K[static_cast<size_t>(k) * N + k];
            for (int i = k + 1 + tid; i < N; i += nth) K[static_cast<size_t>(i) * N + k] /= dkk;
            __syncthreads();
            const int rem = N - k - 1;
            const int strips = (rem + 7) >> 3;   // thread -> (row, 8-column strip)
            for (int idx = tid; idx < rem * strips; idx += nth) {
                const int i = k + 1 + idx / strips, j0 = k + 1 + 8 * (idx % strips);
                const double l = K[static_cast<size_t>(i) * N + k];
                const int j1 = (j0 + 8 < N) ? j0 + 8 : N;
                for (int j = j0; j < j1; ++j) K[static_cast<size_t>(i) * N + j] -= l * K[static_cast<size_t>(k) * N + j];
            }
            __syncthreads();
        }
        if (s_flag) status = 1;
    }

    if (status == 0) {
        // ---- solve, dlam = -(G dz) / s
        for (int i = tid; i < N; i += nth) sol[i] = (i < n) ? -dx[i] : 0.0;
        __syncthreads();
        lu_solve(sol);
        mulG(sol, DL, mi, AI);
        for (int r = tid; r < mi; r += nth) DL[r] = -DL[r] / S[r];   // same thread, same r: no barrier between
        __syncthreads();
        // ---- iterative refinement against the unreduced operator: residual (r1, r2, r3) of the three block rows at (dz, dlam, dnu);
        // correction dz', dnu' from K with the reduced right-hand side [r1 - G'(w o r2); r3], then dlam' = (r2 - G dz') / s
        for (int step = 0; step < 2; ++step) {
            mulG(sol, R2, mi, AI);
            for (int r = tid; r < mi; r += nth) R2[r] = -(R2[r] + S[r] * DL[r]);
            mulG(sol, t0, n, Pd);
            mulG(sol, t1, me, AE);
            __syncthreads();
            for (int j = tid; j < N; j += nth) {
                if (j < n) {
                    double acc = -dx[j] - t0[j];
                    for (int r = 0; r < mi; ++r) acc -= AI[static_cast<size_t>(r) * n + j] * (LAM[r] * DL[r] + W[r] * R2[r]);
                    for (int e = 0; e < me; ++e) acc -= AE[static_cast<size_t>(e) * n + j] * sol[n + e];
                    cor[j] = acc;
                } else {
                    cor[j] = -t1[j - n];
                }
            }
            __syncthreads();
            lu_solve(cor);
            for (int r = tid; r < mi; r += nth) {
                double acc = 0;
                for (int j = 0; j < n; ++j) acc += AI[static_cast<size_t>(r) * n + j] * cor[j];
                DL[r] += (R2[r] - acc) / S[r];
            }
            for (int i = tid; i < N; i += nth) sol[i] += cor[i];
            __syncthreads();
        }
        int nf = 0;
        for (int i = tid; i < N; i += nth) nf |= !is_fin(sol[i]);
        for (int r = tid; r < mi; r += nth) nf |= !is_fin(DL[r]);
        if (__syncthreads_or(nf)) status = 1;
    }

    // ---- outputs in the caller's row order; zeros unless status 0
    const bool ok = status == 0;
    if (dz_out)
        for (int i = tid; i < n; i += nth) dz_out[static_cast<size_t>(b) * n + i] = ok ? sol[i] : 0.0;
    if (dy_out || db_out)
        for (int r = tid; r < m; r += nth) {
            const int slot = row_slot[r];
            double dyr = 0.0, dbr = 0.0;
            if (ok && slot >= 0) { dyr = DL[slot]; dbr = -LAM[slot] * DL[slot]; }
            else if (ok && slot < -1) { dyr = sol[n - (slot + 2)]; dbr = -dyr; }
            if (dy_out) dy_out[static_cast<size_t>(b) * m + r] = dyr;
            if (db_out) db_out[static_cast<size_t>(b) * m + r] = dbr;
        }
    if (dA_out)
        for (int k = tid; k < D.nnzA; k += nth) {
            int lo = 0, hi = n;   // column of entry k: the last j with Acol[j] <= k
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (Acol[mid] <= k) lo = mid;
                else hi = mid;
            }
            const int slot = row_slot[Arow[k]];
            double v = 0.0;
            if (ok && slot >= 0) v = LAM[slot] * DL[slot] * xs[lo] + LAM[slot] * sol[lo];
            else if (ok && slot < -1) v = sol[n - (slot + 2)] * xs[lo] + nu[-(slot + 2)] * sol[lo];
            dA_out[static_cast<size_t>(b) * D.nnzA + k] = v;
        }
    if (tid == 0 && status_out) status_out[b] = status;
}

int launch_qp_adjoint(int count, int n, int m, int mi, int me, int nnzP, int nnzA, const int* Pcol, const int* Prow, const double* Pval,
                      const int* Acol, const int* Arow, const double* Aval, const int* in_rows, const int* eq_rows, const int* row_slot,
                      const double* x, const double* y, const double* s, const double* dx, double* ws, double* dz, double* dy, double* db,
                      double* dA, int32_t* status, int max_smem, cudaStream_t stream) {
    if (n + me > kQpAdjMaxDim) return -1;
    QpAdjDims D;
    D.n = n; D.m = m; D.mi = mi; D.me = me; D.nnzP = nnzP; D.nnzA = nnzA;
    D.stride = qp_adj_ws_doubles(n, mi, me);
    const size_t smem = qp_adj_smem_bytes(n, me);
    if (smem > static_cast<size_t>(max_smem)) return -1;
    cudaFuncSetAttribute(k_qp_adjoint, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    k_qp_adjoint<<<count, 256, smem, stream>>>(D, Pcol, Prow, Pval, Acol, Arow, Aval, in_rows, eq_rows, row_slot, x, y, s, dx, ws, dz, dy, db, dA,
                                               status);
    return 0;
}

}  // namespace bgg
