"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the derivative of a generic QP of the solver seam:
ClarabelInterface::SetupDerivativeCalcs + CalcDerivativeWrtVecs / WrtMats (mpc/qp/clarabel_interface.cpp:262-602, 182-260).

It builds and solves the reference's differential system exactly as oracle/gait_oracle.py::derivative_terms does on the MPC's
QP (the same sparse matrix, the same SuperLU solve, the same empty-row rule), for any QP of bgg_qp_solve_batch's form;
tests/test_oracle_qp_adjoint.py checks that the two agree bit for bit on the MPC's QP.
      [ P    G' D(lam)   Ae' ] [dz  ]      [dx]
      [ G    D(s)        0   ] [dlam]  = - [0 ]        (the reference's own +D(s) block)
      [ Ae   0           0   ] [dnu ]      [0 ]
"""
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla


def _full_symmetric(P):
    """P stored as one triangle -> the full symmetric matrix (diagonal once); a full or diagonal P is used as given."""
    P = sp.csr_matrix(P)
    upper, lower = sp.triu(P, 1).nnz, sp.tril(P, -1).nnz
    if (upper == 0) != (lower == 0):
        return (P + P.T - sp.diags(P.diagonal())).tocsr()
    return P


def qp_adjoint(P, A, is_eq, x, y, s, dx):
    """The derivative of min 1/2 x'Px + q'x, A x + s = b (s = 0 on is_eq rows, s >= 0 elsewhere) at the point (x, y, s) in the
    caller's row order, with loss gradient dx.  G = A[inequality rows], Ae = A[equality rows], lam = y on G's rows, nu = y on
    Ae's rows.  Returns the unknowns (dz, dlam, dnu, and lam, nu, slack as used) and, in the caller's row order, dy (dlam / dnu),
    db (-dnu on equality rows, dh = -lam dlam on inequality rows) and dA on A's pattern (the order of its sorted CSC data):
    dnu_r x_j + nu_r dz_j on an equality row, lam_r dlam_r x_j + lam_r dz_j on an inequality row."""
    A = sp.csr_matrix(A)
    P = _full_symmetric(P)
    is_eq = np.asarray(is_eq, bool)
    ineq, eq = np.flatnonzero(~is_eq), np.flatnonzero(is_eq)
    G, Ae = A[ineq], A[eq]
    x, y, dx = np.asarray(x, float), np.asarray(y, float), np.asarray(dx, float)
    lam, nu, s = y[ineq], y[eq], np.asarray(s, float)[ineq]
    m, n, mi, me = A.shape[0], A.shape[1], len(ineq), len(eq)
    # an inequality row without any stored entry reads 0 + s = b and decouples (dlam = 0); where its slack is exactly 0 a unit
    # diagonal keeps the matrix non-singular without changing any other unknown (derivative_terms' rule)
    empty = np.diff(G.indptr) == 0
    s = np.where(empty & (s == 0.0), 1.0, s)
    M = sp.bmat([[P, (G.T @ sp.diags(lam)), Ae.T],
                 [G, sp.diags(s), None],
                 [Ae, None, None]], format="csc")
    rhs = np.concatenate([dx, np.zeros(mi + me)])
    d = -spla.splu(M).solve(rhs)
    dz, dlam, dnu = d[:n], d[n:n + mi], d[n + mi:]
    dy, db, mult = np.zeros(m), np.zeros(m), np.zeros(m)
    dy[ineq], dy[eq] = dlam, dnu
    db[ineq], db[eq] = -lam * dlam, -dnu
    mult[ineq], mult[eq] = lam * dlam, dnu
    Ac = sp.csc_matrix(A)
    Ac.sort_indices()
    rows, cols = Ac.indices, np.repeat(np.arange(n), np.diff(Ac.indptr))
    dA = mult[rows] * x[cols] + y[rows] * dz[cols]
    return dict(ineq=ineq, eq=eq, lam=lam, nu=nu, slack=s, dz=dz, dlam=dlam, dnu=dnu, dy=dy, db=db, dA=dA)
