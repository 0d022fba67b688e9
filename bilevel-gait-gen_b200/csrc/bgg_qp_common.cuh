// bilevel-gait-gen_b200 -- pieces shared by the generic QP solve (csrc/bgg_qp.cu, k_qp_generic) and its adjoint
// (csrc/bgg_qp_adjoint.cu, k_qp_adjoint): both read the same batch of QPs on one CSC pattern in the same row numbering.
//
// Row slots (classified on the host, csrc/bgg_capi.cu): row_slot[r] >= 0 is the inequality slot of caller row r, < -1 the
// equality slot -(row_slot[r] + 2), -1 an inequality row without any stored entry (it reads 0 + s = b and is left out).
#pragma once

namespace bgg {

// Dense copies of one QP's values on the shared pattern: A_I (mi x n) and A_E (me x n) row major, rows in slot order; P (n x n)
// full symmetric (P is stored as a triangle or as the full matrix: every entry is mirrored, the diagonal once).  Zeroes the three
// blocks first; the caller synchronises before reading them.
__device__ __forceinline__ void qp_densify(int n, int mi, int me, const int* __restrict__ Pcol, const int* __restrict__ Prow,
                                           const double* __restrict__ Pv, const int* __restrict__ Acol, const int* __restrict__ Arow,
                                           const double* __restrict__ Av, const int* __restrict__ row_slot, double* AI, double* AE, double* Pd) {
    const int tid = threadIdx.x, nth = blockDim.x;
    for (size_t i = tid; i < static_cast<size_t>(mi) * n; i += nth) AI[i] = 0.0;
    for (size_t i = tid; i < static_cast<size_t>(me) * n; i += nth) AE[i] = 0.0;
    for (size_t i = tid; i < static_cast<size_t>(n) * n; i += nth) Pd[i] = 0.0;
    __syncthreads();
    for (int j = tid; j < n; j += nth) {
        for (int k = Pcol[j]; k < Pcol[j + 1]; ++k) {
            const int i = Prow[k];
            Pd[static_cast<size_t>(i) * n + j] = Pv[k];
            Pd[static_cast<size_t>(j) * n + i] = Pv[k];
        }
        for (int k = Acol[j]; k < Acol[j + 1]; ++k) {
            const int slot = row_slot[Arow[k]];
            if (slot >= 0) AI[static_cast<size_t>(slot) * n + j] = Av[k];
            else if (slot < -1) AE[static_cast<size_t>(-(slot + 2)) * n + j] = Av[k];
        }
    }
}

}  // namespace bgg
