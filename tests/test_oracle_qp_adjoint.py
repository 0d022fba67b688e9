"""The generic QP derivative of tests/qp_adjoint_ref.py (the restatement of ClarabelInterface::SetupDerivativeCalcs /
CalcDerivativeWrtVecs / CalcDerivativeWrtMats) against the oracle's derivative chain on the MPC's QP, bit for bit, and against an
independent ground truth.

With strict complementarity the optimum is locally the solution of the equality-constrained KKT system on the active set
(equality rows and the inequality rows with lam > 0).  Differentiating that system gives dq, db and dA exactly:
    [P  Aa'] [dz]     [dx]
    [Aa  0 ] [w ] = - [0 ],    dq = dz,  db_r = -w_r,  dA_rj = w_r x_j + y_r dz_j  on active rows, 0 on the others.
The QPs are built around a chosen optimum with a margin (active lam and inactive s in [0.3, 1], unit rows of A) and the margin is confirmed
from a tight solve.  The reference's 3-variable QP (test/mpc_test.cpp:857-904) is included with its closed-form optimum."""
import numpy as np
import scipy.sparse as sp
import pytest

import common
import gait_oracle as go
import pyoracle as po
import qp_adjoint_ref as qa
import test_oracle_qp

BAR = 1e-5          # relative, at the solver's default tolerance
MARGIN = 1e-2       # active lam and inactive s, measured from a tight solve


def margin_qps(seed, n, me, mi_act, mi_inact, n_empty=0, count=1, interleave=True, density=1.0):
    """`count` QPs on one pattern, each built around a known optimum: x*, nu* (equality rows), lam* in [0.3, 1] on mi_act rows,
    s* in [0.3, 1] on mi_inact rows (A's rows have unit norm), and n_empty inequality rows without a stored entry (b = 0.5).  Rows interleaved at random.
    Returns dict(P list (full), A list, q, b, is_eq, x, y, s, active) with x / y / s / active per QP in the caller's row order."""
    rng = np.random.default_rng(seed)
    mi = mi_act + mi_inact + n_empty
    m = me + mi
    kind = np.array([0] * me + [1] * mi_act + [2] * mi_inact + [3] * n_empty)   # eq, active, inactive, empty
    order = rng.permutation(m) if interleave else np.arange(m)
    kind = kind[order]
    mask = rng.uniform(size=(m, n)) < density
    mask[np.arange(m), rng.integers(0, n, m)] = True          # every row but the empty ones has an entry
    mask[kind == 3] = False
    out = dict(P=[], A=[], q=[], b=[], x=[], y=[], s=[], is_eq=kind == 0, active=(kind == 0) | (kind == 1), kind=kind)
    for _ in range(count):
        M = rng.normal(size=(n, n))
        P = M @ M.T / n + 0.5 * np.eye(n)
        A = np.where(mask, rng.normal(size=(m, n)), 0.0)
        A /= np.maximum(np.linalg.norm(A, axis=1), 1e-300)[:, None]    # unit rows: a well-conditioned active set
        x = rng.normal(size=n)
        y = np.zeros(m)
        y[kind == 0] = rng.normal(size=me)
        y[kind == 1] = rng.uniform(0.3, 1.0, mi_act)
        s = np.zeros(m)
        s[kind == 2] = rng.uniform(0.3, 1.0, mi_inact)
        s[kind == 3] = 0.5
        b = A @ x + s
        q = -P @ x - A.T @ y
        for k, v in (("P", P), ("A", A), ("q", q), ("b", b), ("x", x), ("y", y), ("s", s)):
            out[k].append(v)
    return out


def active_set_truth(P, A, x, y, active, dx):
    """dq, db and dA (dense, m x n) of the equality-constrained KKT system on the active rows."""
    n = P.shape[0]
    Aa = A[active]
    K = np.block([[P, Aa.T], [Aa, np.zeros((len(Aa), len(Aa)))]])
    d = -np.linalg.solve(K, np.concatenate([dx, np.zeros(len(Aa))]))
    dz, w = d[:n], d[n:]
    wf = np.zeros(A.shape[0])
    wf[active] = w
    db = -wf
    dA = np.outer(wf, x) + np.outer(np.where(active, y, 0.0), dz)
    return dz, db, dA


def on_pattern(A, dense):
    """Values of a dense m x n matrix at A's stored entries, in the order of A's sorted CSC data."""
    Ac = sp.csc_matrix(A)
    Ac.sort_indices()
    cols = np.repeat(np.arange(A.shape[1]), np.diff(Ac.indptr))
    return dense[Ac.indices, cols]


def rel_err(got, ref):
    return np.abs(np.asarray(got) - np.asarray(ref)).max(initial=0.0) / max(1.0, np.abs(ref).max(initial=0.0))


def three_variable_qp():
    """The reference's cross-solver QP in Clarabel form (equalities, G x <= ub, -G x <= -lb), its closed-form optimum and the
    multipliers of the active set."""
    P, q = test_oracle_qp.P, test_oracle_qp.q
    A = np.vstack([test_oracle_qp.Aeq, test_oracle_qp.G, -test_oracle_qp.G])
    b = np.concatenate([test_oracle_qp.beq, test_oracle_qp.g_ub, -test_oracle_qp.g_lb])
    is_eq = np.array([1, 1, 0, 0, 0, 0], bool)
    x = test_oracle_qp.exact_solution()
    active = is_eq | (np.abs(A @ x - b) < 1e-9)
    y = np.zeros(6)
    y[active] = np.linalg.lstsq(A[active].T, -(P @ x + q), rcond=None)[0]
    return P, q, A, b, is_eq, x, y, active


def test_three_variable_qp_matches_the_closed_form():
    P, q, A, b, is_eq, x, y, active = three_variable_qp()
    assert np.abs(P @ x + q + A.T @ y).max() < 1e-12 and np.all(y[~is_eq] >= 0)
    r = po.ipm_solve(sp.csc_matrix(P), q, sp.csc_matrix(A), b, is_eq)
    assert r["status"] == 0
    dx = P @ r["x"] + q                                               # Computedx, as the reference passes it
    a = qa.qp_adjoint(sp.csc_matrix(P), sp.csc_matrix(A), is_eq, r["x"], r["y"], r["s"], dx)
    dz, db, dA = active_set_truth(P, A, x, y, active, P @ x + q)
    assert rel_err(a["dz"], dz) <= BAR
    assert rel_err(a["db"], db) <= BAR
    assert rel_err(a["dA"], on_pattern(A, dA)) <= BAR


@pytest.mark.parametrize("n,me,mi_act,mi_inact,n_empty,density", [
    (1, 0, 1, 2, 1, 1.0), (3, 2, 1, 3, 1, 1.0), (12, 3, 4, 16, 2, 0.6), (24, 2, 8, 30, 0, 1.0), (42, 18, 10, 50, 2, 0.5),
])
def test_random_margin_qps_match_the_active_set_truth(n, me, mi_act, mi_inact, n_empty, density):
    Q = margin_qps(100 + n, n, me, mi_act, mi_inact, n_empty, count=3, density=density)
    rng = np.random.default_rng(n)
    for k in range(3):
        P, A, is_eq = Q["P"][k], Q["A"][k], Q["is_eq"]
        tight = po.ipm_solve(sp.csc_matrix(P), Q["q"][k], sp.csc_matrix(A), Q["b"][k], is_eq, tol=1e-12)
        assert tight["status"] == 0
        ineq = ~is_eq & (Q["kind"] != 3)
        act = Q["active"] & ineq
        assert tight["y"][act].min(initial=1.0) >= MARGIN and tight["s"][ineq & ~act].min(initial=1.0) >= MARGIN
        assert np.abs(tight["x"] - Q["x"][k]).max() < 1e-8
        r = po.ipm_solve(sp.csc_matrix(P), Q["q"][k], sp.csc_matrix(A), Q["b"][k], is_eq)
        assert r["status"] == 0
        dx = rng.normal(size=n)
        a = qa.qp_adjoint(sp.csc_matrix(P), sp.csc_matrix(A), is_eq, r["x"], r["y"], r["s"], dx)
        dz, db, dA = active_set_truth(P, A, Q["x"][k], Q["y"][k], Q["active"], dx)
        assert rel_err(a["dz"], dz) <= BAR, rel_err(a["dz"], dz)
        assert rel_err(a["db"], db) <= BAR, rel_err(a["db"], db)
        assert rel_err(a["dA"], on_pattern(A, dA)) <= BAR, rel_err(a["dA"], on_pattern(A, dA))
        # empty inequality rows decouple
        assert np.all(a["dy"][Q["kind"] == 3] == 0.0) and np.all(a["db"][Q["kind"] == 3] == 0.0)


def test_a_triangle_and_the_full_matrix_give_the_same_derivative():
    Q = margin_qps(7, 10, 2, 3, 8, 1)
    P, A, is_eq = Q["P"][0], Q["A"][0], Q["is_eq"]
    r = po.ipm_solve(sp.csc_matrix(P), Q["q"][0], sp.csc_matrix(A), Q["b"][0], is_eq)
    dx = np.arange(10.0)
    full = qa.qp_adjoint(sp.csc_matrix(P), sp.csc_matrix(A), is_eq, r["x"], r["y"], r["s"], dx)
    for tri in (np.triu(P), np.tril(P)):
        t = qa.qp_adjoint(sp.csc_matrix(tri), sp.csc_matrix(A), is_eq, r["x"], r["y"], r["s"], dx)
        for k in ("dz", "dy", "db", "dA"):
            assert np.abs(t[k] - full[k]).max() <= 1e-12 * max(1.0, np.abs(full[k]).max())


def test_generic_restatement_is_the_oracles_derivative_chain_on_the_mpc_qp():
    """On the MPC's QP, qp_adjoint gives bit for bit what oracle/gait_oracle.py::derivative_terms gives (that chain is itself pinned
    to the reference's own derivative code by tests/test_oracle_vs_reference_mpc.py)."""
    from common import wl
    cfg = wl.CONFIGS["a1_configuration"]
    init = np.asarray(cfg["srb_init"], float)
    o = common.make_oracle("a1_configuration")
    o.initial_run(init, wl.EE_NOMINAL.copy())
    o.solve(init, 0.0, wl.EE_NOMINAL.copy(), real_time=True)
    t = go.derivative_terms(o)
    assert t is not None
    qp, sol = t["qp"], o.qp_solution()
    a = qa.qp_adjoint(qp["P"], qp["A"], qp["is_eq"], sol["x"], sol["dual"], sol["slack"], t["dx"])
    for key in ("dz", "dlam", "dnu", "lam", "nu", "slack"):
        assert np.array_equal(a[key], t[key]), key
    assert np.array_equal(a["db"][t["eq"]], t["db"]) and np.array_equal(a["db"][t["ineq"]], t["dh"])
