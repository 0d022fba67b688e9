"""k_qp_adjoint (bgg_qp_adjoint_batch, BatchedMPC.QPAdjoint): the derivative of the generic QP solve, the reference's
ClarabelInterface::SetupDerivativeCalcs / CalcDerivativeWrtVecs / CalcDerivativeWrtMats, on the device.

1. Same point, two implementations: at the oracle's own (x, y, s) the kernel must give what tests/qp_adjoint_ref.py::qp_adjoint
   gives, and (dz, dlam, dnu) must have a small normwise backward error in the unreduced system.  This pins the reference's
   +D(s) block, which the active-set truth below cannot tell from -D(s).
2. Solve, then adjoint, against the active-set truth of tests/test_oracle_qp_adjoint.py.
3. Shapes from n = 1 to n + me = 160, interleaved equality / inequality rows, empty inequality rows, P as a triangle and full.
4. Statuses and refusals; 5. batch independence; 6. the C++ layer (tests/cpp/test_qp_adjoint.cpp)."""
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

import common
import bgg_b200 as bg
import qp_adjoint_ref as qa
import pyoracle as po
from test_oracle_qp_adjoint import BAR, active_set_truth, margin_qps, on_pattern, rel_err, three_variable_qp

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SAME_POINT_BAR = 1e-7        # relative to max(1, |ref|_inf)
BACKWARD_BAR = 1e-10         # normwise backward error of (dz, dlam, dnu) in the unreduced system

# n, me, active and inactive inequality rows, empty inequality rows, density of A's pattern
SHAPES = [(1, 0, 1, 2, 1, 1.0), (3, 2, 1, 3, 1, 1.0), (24, 2, 8, 30, 2, 0.6), (24, 0, 6, 20, 0, 1.0), (42, 18, 10, 50, 2, 0.5),
          (42, 32, 6, 20, 1, 0.5), (127, 2, 30, 60, 1, 0.3), (127, 32, 20, 60, 1, 0.3), (128, 32, 24, 60, 2, 0.3), (128, 0, 30, 90, 0, 0.3)]
WORST = {}


@pytest.fixture(scope="module")
def gpu():
    return common.make_gpu("a1_configuration", 1)


def _p_form(P, form):
    return sp.csc_matrix(np.triu(P) if form == "upper" else P)


def unreduced(P, A, is_eq, y, s):
    """The reference's differential matrix (dense) with the oracle's empty-row rule, unknowns ordered (dz, dlam, dnu)."""
    ineq, eq = np.flatnonzero(~is_eq), np.flatnonzero(is_eq)
    G, Ae = A[ineq], A[eq]
    sI = s[ineq].copy()
    sI[(np.abs(G).sum(axis=1) == 0) & (sI == 0.0)] = 1.0
    n, mi, me = P.shape[0], len(ineq), len(eq)
    M = np.zeros((n + mi + me, n + mi + me))
    M[:n, :n] = P
    M[:n, n:n + mi] = G.T * y[ineq]
    M[:n, n + mi:] = Ae.T
    M[n:n + mi, :n] = G
    M[n:n + mi, n:n + mi] = np.diag(sI)
    M[n + mi:, :n] = Ae
    return M, ineq, eq


def backward_error(P, A, is_eq, y, s, dx, dz, dy):
    M, ineq, eq = unreduced(P, A, is_eq, y, s)
    d = np.concatenate([dz, dy[ineq], dy[eq]])
    rhs = np.concatenate([dx, np.zeros(len(ineq) + len(eq))])
    r = M @ d + rhs
    return np.abs(r).max() / (np.abs(M).sum(axis=1).max() * np.abs(d).max() + np.abs(rhs).max())


def _note(key, v):
    WORST[key] = max(WORST.get(key, 0.0), v)


@pytest.mark.parametrize("form", ["upper", "full"])
@pytest.mark.parametrize("shape", SHAPES, ids=[f"n{s[0]}_me{s[1]}" for s in SHAPES])
def test_same_point_matches_the_oracle_restatement(gpu, shape, form):
    n, me, ma, mn, ne, dens = shape
    Q = margin_qps(1000 + n + me, n, me, ma, mn, ne, count=3, density=dens)
    rng = np.random.default_rng(n + me)
    is_eq, pts, dxs = Q["is_eq"], [], []
    for k in range(3):
        r = po.ipm_solve(sp.csc_matrix(Q["P"][k]), Q["q"][k], sp.csc_matrix(Q["A"][k]), Q["b"][k], is_eq)
        assert r["status"] == 0
        pts.append(r)
        dxs.append(rng.normal(size=n))
    out = gpu.QPAdjoint([_p_form(P, form) for P in Q["P"]], [sp.csc_matrix(A) for A in Q["A"]], is_eq, [p["x"] for p in pts],
                        [p["y"] for p in pts], [p["s"] for p in pts], dxs)
    assert out["status"].tolist() == [0, 0, 0]
    for k in range(3):
        P, A, p = Q["P"][k], Q["A"][k], pts[k]
        ref = qa.qp_adjoint(sp.csc_matrix(P), sp.csc_matrix(A), is_eq, p["x"], p["y"], p["s"], dxs[k])
        for key, got, want in (("dz", out["dz"][k], ref["dz"]), ("dy", out["dy"][k], ref["dy"]), ("db", out["db"][k], ref["db"]),
                               ("dA", out["dA"][k], ref["dA"])):
            e = rel_err(got, want)
            _note("same_point_" + key, e)
            assert e <= SAME_POINT_BAR, (key, k, e)
        eta = backward_error(P, A, is_eq, p["y"], p["s"], dxs[k], out["dz"][k], out["dy"][k])
        _note("backward_error", eta)
        assert eta <= BACKWARD_BAR, (k, eta)
        assert np.all(out["dy"][k][Q["kind"] == 3] == 0.0) and np.all(out["db"][k][Q["kind"] == 3] == 0.0)   # empty rows
    print(f"\n{shape} {form}: worst so far " + ", ".join(f"{k} {v:.2e}" for k, v in sorted(WORST.items())))


@pytest.mark.parametrize("form", ["upper", "full"])
@pytest.mark.parametrize("shape", SHAPES, ids=[f"n{s[0]}_me{s[1]}" for s in SHAPES])
def test_solve_then_adjoint_matches_the_active_set_truth(gpu, shape, form):
    n, me, ma, mn, ne, dens = shape
    Q = margin_qps(2000 + n + me, n, me, ma, mn, ne, count=3, density=dens)
    is_eq = Q["is_eq"]
    Ps, As = [_p_form(P, form) for P in Q["P"]], [sp.csc_matrix(A) for A in Q["A"]]
    sol = gpu.SolveQP(Ps, np.array(Q["q"]), As, np.array(Q["b"]), is_eq)
    assert sol["status"].tolist() == [0, 0, 0]
    dx = np.random.default_rng(n).normal(size=(3, n))
    out = gpu.QPAdjoint(Ps, As, is_eq, sol["x"], sol["y"], sol["s"], dx)
    assert out["status"].tolist() == [0, 0, 0]
    for k in range(3):
        dz, db, dA = active_set_truth(Q["P"][k], Q["A"][k], Q["x"][k], Q["y"][k], Q["active"], dx[k])
        for key, got, want in (("dz", out["dz"][k], dz), ("db", out["db"][k], db), ("dA", out["dA"][k], on_pattern(Q["A"][k], dA))):
            e = rel_err(got, want)
            _note("truth_" + key, e)
            assert e <= BAR, (key, k, e)
    print(f"\n{shape} {form}: worst so far " + ", ".join(f"{k} {v:.2e}" for k, v in sorted(WORST.items())))


def _valid_points(Q):
    """The constructed optimum, moved into the interior (s > 0 on every kept inequality row)."""
    s = [np.where(Q["is_eq"], 0.0, np.maximum(v, 1e-9)) for v in Q["s"]]
    return Q["x"], Q["y"], s


def test_one_batch_mixes_statuses_0_1_and_2(gpu):
    """QP 1 repeats its first equality row (singular: status 1), QP 2 has a kept inequality row with s < 0 (status 2); both get
    exact zeros.  QP 0 is unaffected by its neighbours."""
    n = 10
    Q = margin_qps(5, n, 2, 3, 8, 1, count=3, interleave=True, density=1.0)
    eq_rows = np.flatnonzero(Q["is_eq"])
    Q["A"][1][eq_rows[1]] = Q["A"][1][eq_rows[0]]
    X, Y, S = _valid_points(Q)
    kept = np.flatnonzero(~Q["is_eq"] & (Q["kind"] != 3))
    S[2][kept[0]] = -1e-3
    dx = np.random.default_rng(1).normal(size=(3, n))
    As = [sp.csc_matrix(A) for A in Q["A"]]
    Ps = [sp.csc_matrix(P) for P in Q["P"]]
    out = gpu.QPAdjoint(Ps, As, Q["is_eq"], X, Y, S, dx)
    assert out["status"].tolist() == [0, 1, 2]
    for k in (1, 2):
        for key in ("dz", "dy", "db", "dA"):
            assert np.all(out[key][k] == 0.0), (k, key)
    alone = gpu.QPAdjoint(Ps[0], As[0], Q["is_eq"], X[0], Y[0], S[0], dx[0])
    for key in ("dz", "dy", "db", "dA"):
        assert np.array_equal(alone[key][0], out[key][0])
    # a non-finite input is status 2 as well
    bad = [v.copy() for v in X]
    bad[0][0] = np.nan
    assert gpu.QPAdjoint(Ps, As, Q["is_eq"], bad, Y, S, dx)["status"].tolist() == [2, 1, 2]


def test_refusals(gpu):
    rng = np.random.default_rng(3)
    for n, me, msg in ((128, 33, r"n \+ me <= 160"), (129, 0, "at most 128")):
        m = me + 4
        A = sp.csc_matrix(rng.normal(size=(m, n)))
        is_eq = np.arange(m) < me
        with pytest.raises(bg.BggError, match=msg):
            gpu.QPAdjoint(sp.identity(n, format="csc"), A, is_eq, np.zeros(n), np.zeros(m), np.ones(m), np.ones(n))
    # n + me = 160 exactly is accepted
    n, me = 128, 32
    A = sp.csc_matrix(rng.normal(size=(me + 4, n)))
    is_eq = np.arange(me + 4) < me
    out = gpu.QPAdjoint(sp.identity(n, format="csc"), A, is_eq, np.zeros(n), np.zeros(me + 4), np.ones(me + 4), np.ones(n))
    assert out["status"][0] == 0


def test_a_qp_gives_the_same_bits_alone_and_anywhere_in_a_batch(gpu):
    n, count = 24, 4096
    Q = margin_qps(11, n, 2, 6, 30, 2, count=count, density=0.6)
    X, Y, S = _valid_points(Q)
    dx = np.random.default_rng(2).normal(size=(count, n))
    Ps, As = [sp.csc_matrix(np.triu(P)) for P in Q["P"]], [sp.csc_matrix(A) for A in Q["A"]]
    full = gpu.QPAdjoint(Ps, As, Q["is_eq"], X, Y, S, dx)
    assert np.all(full["status"] == 0)
    perm = np.random.default_rng(3).permutation(count)
    shuffled = gpu.QPAdjoint([Ps[i] for i in perm], [As[i] for i in perm], Q["is_eq"], [X[i] for i in perm], [Y[i] for i in perm],
                             [S[i] for i in perm], dx[perm])
    for key in ("dz", "dy", "db", "dA", "status"):
        assert np.array_equal(shuffled[key], full[key][perm]), key
    for k in (0, 1234, count - 1):
        alone = gpu.QPAdjoint(Ps[k], As[k], Q["is_eq"], X[k], Y[k], S[k], dx[k])
        four = gpu.QPAdjoint([Ps[(k + j) % count] for j in (3, 2, 1, 0)], [As[(k + j) % count] for j in (3, 2, 1, 0)], Q["is_eq"],
                             [X[(k + j) % count] for j in (3, 2, 1, 0)], [Y[(k + j) % count] for j in (3, 2, 1, 0)],
                             [S[(k + j) % count] for j in (3, 2, 1, 0)], dx[[(k + j) % count for j in (3, 2, 1, 0)]])
        for key in ("dz", "dy", "db", "dA", "status"):
            assert np.array_equal(alone[key][0], full[key][k]), (k, key)
            assert np.array_equal(four[key][3], full[key][k]), (k, key)


def test_cpp_layer_on_the_references_three_variable_qp():
    """ClarabelInterface::SetupQP, Solve, Computedx, SetupDerivativeCalcs(dx, 0, 0, qp), CalcDerivativeWrtVecs / WrtMats
    (tests/cpp/test_qp_adjoint.cpp, the adjoint half of test/mpc_test.cpp:857-1004) against the oracle at the same point and the
    closed form; dA / dG are zero off the pattern of A."""
    binary = os.path.join(ROOT, "tests", "cpp", "test_qp_adjoint")
    out = subprocess.run([binary], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    kv = {}
    for line in out.stdout.splitlines():
        parts = line.split()
        if parts:
            kv[parts[0]] = parts[1:]
    assert kv["done"] == ["1"] and kv["throws_before_solve"] == ["1"] and kv["quality"] == ["0"]
    vec = lambda k: np.array([float(v) for v in kv[k]])
    mat = lambda k: np.array([float(v) for v in kv[k][2:]]).reshape(int(kv[k][0]), int(kv[k][1]))
    x, y, s, dx = vec("x"), vec("y"), vec("s"), vec("dx")
    dq, db, dh, dA, dG = vec("dq"), vec("db"), vec("dh"), mat("dA"), mat("dG")
    P, q, A, b, is_eq, xs, ys, active = three_variable_qp()
    assert np.abs(dx - (P @ x + q)).max() < 1e-12
    ref = qa.qp_adjoint(sp.csc_matrix(P), sp.csc_matrix(A), is_eq, x, y, s, dx)
    ineq, eq = np.flatnonzero(~is_eq), np.flatnonzero(is_eq)
    full_ref = np.zeros(A.shape)
    Ac = sp.csc_matrix(A)
    Ac.sort_indices()
    full_ref[Ac.indices, np.repeat(np.arange(3), np.diff(Ac.indptr))] = ref["dA"]
    assert rel_err(dq, ref["dz"]) <= SAME_POINT_BAR
    assert rel_err(db, ref["db"][eq]) <= SAME_POINT_BAR and rel_err(dh, ref["db"][ineq]) <= SAME_POINT_BAR
    assert rel_err(dA, full_ref[eq]) <= SAME_POINT_BAR and rel_err(dG, full_ref[ineq]) <= SAME_POINT_BAR
    assert np.all(dA[A[eq] == 0] == 0.0) and np.all(dG[A[ineq] == 0] == 0.0)
    tz, tb, tA = active_set_truth(P, A, xs, ys, active, P @ xs + q)
    assert rel_err(dq, tz) <= BAR
    assert rel_err(np.concatenate([db, dh]), np.concatenate([tb[eq], tb[ineq]])) <= BAR
    assert rel_err(np.vstack([dA, dG]), np.vstack([tA[eq], tA[ineq]]) * (A[np.concatenate([eq, ineq])] != 0)) <= BAR
