"""The dense building blocks under k_ipm, each against a plain high-precision reference of the same operation:

* condensing (k_condense, csrc/bgg_condense.cu): H, g, the foot-box rows `phipos` and the state offsets `xoff` of the
  condensed QP, against the state elimination redone in np.longdouble from the same instance's dynamics and cost;
* the block Cholesky (csrc/bgg_chol.cuh: chol::factor + chol::solve) through a test-only kernel (tests/cuda/chol_harness.cu)
  at every block count from 1 to 23, at k_ipm's two block sizes, against scipy's factor and residuals in np.longdouble;
* the cap on max_spline_vars that the kernels above are sized for.

The end-to-end parity tests (test_gpu_parity.py) compare minimisers to 1e-4; errors in H or in the factor well below that
bar only cost interior-point iterations, so they are bounded here directly, componentwise where a componentwise bound is
the natural one, against the unit roundoff u = 2^-53 times a small constant.
"""
import os
import shutil
import subprocess

import numpy as np
import pytest

import common
from common import wl

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -53
LD = np.longdouble
C_COND = 32   # condensing: |error| <= C_COND * N * u * (the same sums over absolute values)
C_CHOL = 32   # Cholesky: backward errors <= C_CHOL * n * u


# --------------------------------------------------------------------------------------------------------------------------
# condensing
# --------------------------------------------------------------------------------------------------------------------------

def _condense_reference(Ad, Bd, cd, P_diag, q, phi0, N, nu):
    """State elimination in long double: Phi_{k+1} = Ad_k Phi_k + Bd_k, phi_{k+1} = Ad_k phi_k + cd_k (Phi_0 = 0, phi_0 given),
    H = sum_k Phi_k' P_k Phi_k + P_u, g = sum_k Phi_k' (P_k phi_k + q_k) + q_u -- and the same recursions over absolute values
    (Psi, psi) that bound the rounding errors of any evaluation order."""
    Ad, Bd, cd = Ad.astype(LD), Bd.astype(LD), cd.astype(LD)
    Phi, Psi = np.zeros((N + 1, 12, nu), LD), np.zeros((N + 1, 12, nu), LD)
    phi, psi = np.zeros((N + 1, 12), LD), np.zeros((N + 1, 12), LD)
    phi[0] = phi0
    psi[0] = np.abs(phi[0])
    for k in range(N):
        Phi[k + 1] = Ad[k] @ Phi[k] + Bd[k]
        phi[k + 1] = Ad[k] @ phi[k] + cd[k]
        Psi[k + 1] = np.abs(Ad[k]) @ Psi[k] + np.abs(Bd[k])
        psi[k + 1] = np.abs(Ad[k]) @ psi[k] + np.abs(cd[k])
    ns = 12 * (N + 1)
    Pk, Pu = P_diag[:ns].astype(LD).reshape(N + 1, 12), P_diag[ns:ns + nu].astype(LD)
    qk, qu = q[:ns].astype(LD).reshape(N + 1, 12), q[ns:ns + nu].astype(LD)
    F, A = Phi.reshape(ns, nu), Psi.reshape(ns, nu)
    H = F.T @ (Phi * Pk[:, :, None]).reshape(ns, nu) + np.diag(Pu)
    g = F.T @ (Pk * phi + qk).reshape(ns) + qu
    Hb = A.T @ (Psi * np.abs(Pk)[:, :, None]).reshape(ns, nu) + np.diag(np.abs(Pu))
    gb = A.T @ (np.abs(Pk) * psi + np.abs(qk)).reshape(ns) + np.abs(qu)
    return dict(Phi=Phi, phi=phi, Psi=Psi, psi=psi, H=H, g=g, Hb=Hb, gb=gb, Pk=Pk, Pu=Pu, qk=qk, qu=qu)


def _ratio(err, bound):
    """max err / bound over the entries; an entry with a zero bound must be exact."""
    err, bound = np.asarray(err, LD), np.asarray(bound, LD)
    if np.any((bound == 0) & (err != 0)):
        return np.inf
    nz = bound > 0
    return float(np.max(err[nz] / bound[nz])) if nz.any() else 0.0


def _check_condensed(gpu, b, label, rng):
    """k_condense's outputs for instance b of the last solve against the long-double reference; returns (nb, worst ratios)."""
    N = gpu.N
    sz = gpu.sizes(b)
    assert sz["error"] == 0, (label, b, sz["error"])
    nu, nf = sz["nu"], sz["nf"]
    Ad, Bd, cd = (x[0] for x in gpu.dynamics(b, 1))
    qp = gpu.GetQPData(b, 1, nnz_cap=80000)[0]
    A, ub = qp["A"], qp["ub"]
    ns = 12 * (N + 1)
    assert A.shape[1] == ns + nu
    # the x_0 rows of the QP are -x_0 = ub[:12]: phi_0 is their right-hand side
    assert np.array_equal(A[:12].toarray(), np.hstack([-np.eye(12), np.zeros((12, ns - 12 + nu))])), (label, b)
    phi0 = -ub[:12]
    ref = _condense_reference(Ad, Bd, cd, qp["P_diag"], qp["q"], phi0, N, nu)
    out = gpu.condensed(b)
    H, g, phipos, xoff = out["H"], out["g"], out["phipos"], out["xoff"]
    tol = C_COND * N * U

    # the reference's Phi, phi are the QP's own dynamics rows: [Phi u + phi; u] satisfies them for any u
    u = rng.standard_normal(nu).astype(LD)
    z = np.concatenate([(ref["Phi"] @ u + ref["phi"]).reshape(ns), u])
    Ad_rows = A[:ns].toarray().astype(LD)
    res = Ad_rows @ z - ub[:ns].astype(LD)
    scale = np.abs(Ad_rows) @ np.abs(z) + np.abs(ub[:ns]).astype(LD)
    assert _ratio(np.abs(res), 1e-13 * scale) <= 1.0, (label, b, "the reference recursion does not satisfy the QP's dynamics rows")

    # symmetry: outside the diagonal 8 x 8 blocks one value is stored twice, so exactly; inside them (i, j) and (j, i) are two
    # roundings of the same sum (csrc/bgg_condense.cu), equal up to the rounding bound below
    diag_blk = (np.arange(nu)[:, None] // 8) == (np.arange(nu)[None, :] // 8)
    assert np.array_equal(H[~diag_blk], H.T[~diag_blk]), (label, b, "H is not exactly symmetric outside its diagonal blocks")
    rS = _ratio(np.abs(H.astype(LD) - H.T.astype(LD)), tol * ref["Hb"])
    assert rS <= 1.0, (label, b, f"H - H': difference / bound = {rS:.3g}")
    rH = _ratio(np.abs(H.astype(LD) - ref["H"]), tol * ref["Hb"])
    rg = _ratio(np.abs(g.astype(LD) - ref["g"]), tol * ref["gb"])
    # the bound is far below the entries it bounds: a bound that wide would accept anything
    assert tol * float(ref["Hb"].max()) < 1e-10 * float(np.abs(H).max()), (label, b, "vacuous bound on H")
    assert rH <= 1.0, (label, b, nu, f"H: error / bound = {rH:.3g}")
    assert rg <= 1.0, (label, b, nu, f"g: error / bound = {rg:.3g}")

    # foot-box position rows: rows 0 and 1 of Phi_k, k >= 4; structural zeros (spline variables that enter at later nodes)
    # are exact on both sides, so the zero pattern is compared exactly
    pref, pb = ref["Phi"][4:, :2, :].reshape(2 * (N - 3), nu), ref["Psi"][4:, :2, :].reshape(2 * (N - 3), nu)
    assert np.array_equal(phipos != 0, pref != 0), (label, b, "zero pattern of phipos")
    rp = _ratio(np.abs(phipos.astype(LD) - pref), tol * pb)
    assert rp <= 1.0, (label, b, f"phipos: error / bound = {rp:.3g}")

    # state offsets: phi_k, and phi_0 bit for bit
    assert np.array_equal(xoff[0], phi0), (label, b, "xoff[0] differs from the x_0 right-hand side")
    rx = _ratio(np.abs(xoff.astype(LD) - ref["phi"]), tol * ref["psi"])
    assert rx <= 1.0, (label, b, f"xoff: error / bound = {rx:.3g}")

    # the condensed objective is the sparse one restricted to the dynamics, up to a constant: for random u,
    # 1/2 u'Hu + g'u = f(z(u)) - f(z(0)),  f(z) = 1/2 z'Pz + q'z,  z(u) = [Phi u + phi; u]
    Pd, qd = qp["P_diag"].astype(LD), qp["q"].astype(LD)
    f = lambda zz: LD(0.5) * zz @ (Pd * zz) + qd @ zz
    z0 = np.concatenate([ref["phi"].reshape(ns), np.zeros(nu, LD)])
    for _ in range(3):
        u = rng.standard_normal(nu).astype(LD)
        zu = np.concatenate([(ref["Phi"] @ u + ref["phi"]).reshape(ns), u])
        lhs = LD(0.5) * u @ (H.astype(LD) @ u) + g.astype(LD) @ u
        rhs = f(zu) - f(z0)
        au = np.abs(u)
        bound = tol * (LD(0.5) * au @ (ref["Hb"] @ au) + ref["gb"] @ au)
        assert abs(lhs - rhs) <= bound, (label, b, float(lhs), float(rhs), float(bound))
    return (nu + 7) // 8, dict(H=rH, sym=rS, g=rg, phipos=rp, xoff=rx)


class _Coverage:
    def __init__(self):
        self.nb, self.variant, self.worst = set(), set(), {}

    def add(self, nb, ratios, cap_nb=None):
        """cap_nb: the batch's block count when the launch's cap is known to be the batch maximum (first solve after a reset)."""
        self.nb.add(nb)
        if nb >= 17:
            self.variant.add(2)                      # cap >= nu: k_condense<2>
        elif cap_nb is not None:
            self.variant.add(1 if cap_nb <= 16 else 2)
        for k, v in ratios.items():
            self.worst[k] = max(self.worst.get(k, 0.0), v)

    def report(self, label):
        print(f"{label}: nb covered {sorted(self.nb)}, k_condense<{sorted(self.variant)}>, largest error / bound "
              + ", ".join(f"{k} {v:.3g}" for k, v in sorted(self.worst.items())))


# per-foot scalings of the default trot schedule (lift-off / touch-down every 0.3 s) and start times whose horizons hold
# 122 .. 160 spline variables at N = 20 (found with the oracle; the solve status does not matter: condensing runs first)
_SCHEDULES = [
    ([1.097, 0.991, 0.843, 0.811], 0.00),   # nb 16
    ([0.965, 0.688, 1.032, 0.871], 0.00),   # nb 17
    ([0.850, 0.692, 0.748, 0.887], 0.15),   # nb 19
    ([0.733, 0.869, 0.821, 1.066], 0.20),   # nb 20
    ([0.918, 0.735, 0.620, 0.608], 0.00),   # nb 20 (160, the cap)
    ([1.000, 1.000, 1.000, 1.000], 0.00),   # nb 15
]


def _make(cfg_name, B, states=None, **kw):
    return common.make_gpu(cfg_name, B, states, **kw)


@pytest.mark.parametrize("cfg_name", ["a1_configuration", "a1_config_distr_rejection"])
def test_condensing_first_solve_matches_long_double_reference(cfg_name):
    """First solve of a batch (nu = 120 at N = 20 and N = 50): every output of k_condense within its rounding bound."""
    cfg = wl.CONFIGS[cfg_name]
    B = 4
    states, t0, ee = wl.batched_trot_inputs(cfg, B, seed=7)
    gpu = _make(cfg_name, B, states)
    gpu.GetRealTimeUpdate(states, t0, ee)
    cov, rng = _Coverage(), np.random.default_rng(1)
    nbs = [(gpu.sizes(b)["nu"] + 7) // 8 for b in range(B)]
    for b in range(B):
        nb, r = _check_condensed(gpu, b, cfg_name, rng)
        cov.add(nb, r, cap_nb=max(nbs))
    cov.report(f"{cfg_name} first solve")
    assert 15 in cov.nb


@pytest.mark.parametrize("cfg_name,ticks", [("a1_configuration", 20), ("a1_config_distr_rejection", 30)])
def test_condensing_along_the_closed_loop(cfg_name, ticks):
    """The horizon slides (closed loop on the device: plant = node 1 of the solved trajectory): the QP grows from 15 to 18 and
    19 block rows and back, so both k_condense instantiations run; every tick is checked.  Then the same handle solves a
    smaller QP again after a reset: every entry of the outputs is rewritten at the smaller size."""
    cfg = wl.CONFIGS[cfg_name]
    dt = cfg["integrator_dt"]
    states, t0, ee = wl.disturbance_sweep_inputs(cfg, 1, seed=4)
    gpu = _make(cfg_name, 1, states)
    gpu.upload(states, t0, ee)
    cov, rng = _Coverage(), np.random.default_rng(2)
    for tick in range(ticks):
        if tick:
            gpu.advance_plant(dt)
        gpu.solve_resident()
        gpu.download()
        nb, r = _check_condensed(gpu, 0, f"{cfg_name} tick {tick}", rng)
        cov.add(nb, r, cap_nb=nb if tick == 0 else None)
    big = max(cov.nb)
    assert big >= 17 and min(cov.nb) <= 16, f"the horizon did not change size as expected: nb {sorted(cov.nb)}"
    # larger first, then smaller on the same handle
    if (gpu.sizes(0)["nu"] + 7) // 8 < 17:
        gpu.Reset(1)
        gpu.SetStateTrajectoryWarmStart(states)
        gpu.GetRealTimeUpdate(states, np.array([0.22]), ee)
        nb, r = _check_condensed(gpu, 0, f"{cfg_name} large", rng)
        cov.add(nb, r, cap_nb=nb)
        assert nb >= 17
    gpu.Reset(1)
    gpu.SetStateTrajectoryWarmStart(states)
    gpu.GetRealTimeUpdate(states, t0, ee)
    nb, r = _check_condensed(gpu, 0, f"{cfg_name} after reset", rng)
    cov.add(nb, r, cap_nb=nb)
    assert nb == 15
    cov.report(f"{cfg_name} closed loop")
    assert cov.variant == {1, 2}


def test_condensing_mixed_batch_up_to_the_cap():
    """One batch whose instances follow different contact schedules: 15 .. 20 block rows side by side (nu = 160, the cap,
    included).  The launch is sized from the batch maximum (row stride ldp, cap_nu), so the smaller instances are condensed by
    k_condense<2> with padding columns; then the same handle solves a batch of nu = 120 only (k_condense<1>)."""
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    B = len(_SCHEDULES)
    init = np.asarray(cfg["srb_init"], float)
    states, ee = np.tile(init, (B, 1)), np.tile(wl.EE_NOMINAL, (B, 1, 1))
    base = np.array([0.0, 0.3, 0.6, 0.9, 1.2])
    times = np.array([[base * s for s in sc] for sc, _ in _SCHEDULES])
    t0 = np.array([t for _, t in _SCHEDULES])
    gpu = _make(cfg_name, B, states)
    gpu.UpdateContactTimes(times)
    gpu.GetRealTimeUpdate(states, t0, ee)
    cov, rng = _Coverage(), np.random.default_rng(3)
    nbs = [(gpu.sizes(b)["nu"] + 7) // 8 for b in range(B)]
    print("mixed batch nu:", [gpu.sizes(b)["nu"] for b in range(B)])
    for b in range(B):
        nb, r = _check_condensed(gpu, b, f"mixed batch instance {b}", rng)
        cov.add(nb, r, cap_nb=max(nbs))
    assert max(nbs) == 20 and min(nbs) <= 16, nbs
    assert 160 in [gpu.sizes(b)["nu"] for b in range(B)]
    gpu.Reset(B)
    gpu.SetStateTrajectoryWarmStart(states)
    gpu.GetRealTimeUpdate(states, np.zeros(B), ee)
    for b in range(B):
        nb, r = _check_condensed(gpu, b, f"after the mixed batch, instance {b}", rng)
        cov.add(nb, r, cap_nb=15)
        assert nb == 15
    cov.report("mixed batch")
    assert cov.variant == {1, 2}


# --------------------------------------------------------------------------------------------------------------------------
# max_spline_vars
# --------------------------------------------------------------------------------------------------------------------------

def test_max_spline_vars_above_160_is_refused():
    """k_condense's accumulators, the KKT tile table and the KKT work list are sized for 160 spline variables: bgg_create refuses
    more (168 used to pass its shared-memory check at N = 20 and then lose block (0, 0) of H at 21 block rows)."""
    import bgg_b200 as bg
    cfg = wl.CONFIGS["a1_configuration"]
    kw = dict(**wl.mpc_kwargs(cfg))
    for bad in (168, 176, 184):
        with pytest.raises(bg.BggError, match="160"):
            bg.BatchedMPC(cfg["num_nodes"], cfg["integrator_dt"], wl.robot(), max_spline_vars=bad, **kw)
    m = bg.BatchedMPC(cfg["num_nodes"], cfg["integrator_dt"], wl.robot(), max_spline_vars=160, **kw)
    m.close()


# --------------------------------------------------------------------------------------------------------------------------
# block Cholesky
# --------------------------------------------------------------------------------------------------------------------------

def _doubles(nb):
    return nb * (nb + 1) // 2 * 64


def _harness_path(tmp_dir):
    src = os.path.join(ROOT, "tests", "cuda", "chol_harness.cu")
    prebuilt = os.path.join(ROOT, "tools", "bin", "libchol_harness.so")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        if os.path.exists(prebuilt):
            return prebuilt
        pytest.skip("nvcc not found and the Cholesky harness is not built (python -c 'import __graft_entry__ as g; g.build()')")
    out = os.path.join(tmp_dir, "libchol_harness.so")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-maxrregcount=128", "-Xcompiler", "-fPIC", "-shared",
                    "-I", os.path.join(ROOT, "bilevel-gait-gen_b200", "csrc"), "-o", out, src], check=True)
    return out


@pytest.fixture(scope="module")
def chol(tmp_path_factory):
    import ctypes as C
    lib = C.CDLL(_harness_path(str(tmp_path_factory.mktemp("chol_harness"))))
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    lib.chol_harness_run.argtypes = [C.c_int, C.c_int, C.c_int, dp, dp, dp, dp, ip]

    def run(threads, nb, A_packed, rhs):
        A_packed = np.ascontiguousarray(A_packed, np.float64)
        rhs = np.ascontiguousarray(rhs, np.float64)
        count = A_packed.shape[0]
        K, x, flags = np.zeros_like(A_packed), np.zeros_like(rhs), np.zeros(count, np.int32)
        rc = lib.chol_harness_run(threads, nb, count, A_packed.ctypes.data_as(dp), rhs.ctypes.data_as(dp), K.ctypes.data_as(dp),
                                  x.ctypes.data_as(dp), flags.ctypes.data_as(ip))
        assert rc == 0, f"chol_harness_run: error {rc}"
        return K, x, flags
    return run


def _block_index(nb):
    """(row, col) of every packed entry: block (bi, bj), bj <= bi, at (bi (bi + 1) / 2 + bj) * 64, row-major 8 x 8."""
    rows, cols = np.empty(_doubles(nb), np.int64), np.empty(_doubles(nb), np.int64)
    r8, c8 = np.divmod(np.arange(64), 8)
    for bi in range(nb):
        for bj in range(bi + 1):
            o = (bi * (bi + 1) // 2 + bj) * 64
            rows[o:o + 64], cols[o:o + 64] = 8 * bi + r8, 8 * bj + c8
    return rows, cols


def _pad(A, n):
    """k_ipm's padding: rows and columns nu .. 8 nb - 1 are the identity."""
    nu = A.shape[0]
    out = np.eye(n)
    out[:nu, :nu] = A
    return out


def _spd_well(rng, nu):
    G = rng.standard_normal((nu, nu))
    return np.eye(nu) * 2.0 + 0.5 * (G @ G.T) / nu


def _spd_kkt(rng, nu):
    """H + 1e-10 I + C' diag(w) C: H PSD with eigenvalues spread 1e-2 .. 6e8 (the condensed QP's), w over 1e-8 .. 1e8."""
    Q, _ = np.linalg.qr(rng.standard_normal((nu, nu)))
    lam = np.logspace(-2, np.log10(6e8), nu)
    rng.shuffle(lam)
    H = (Q * lam) @ Q.T
    m = 2 * nu
    C = rng.standard_normal((m, nu)) * (rng.random((m, nu)) < 0.2)
    w = np.logspace(-8, 8, m)
    rng.shuffle(w)
    A = H + 1e-10 * np.eye(nu) + (C.T * w) @ C
    return 0.5 * (A + A.T)


def _tri_inv_ld(X):
    """inverse of a lower-triangular matrix by forward substitution in long double"""
    m = X.shape[0]
    X = X.astype(LD)
    Y = np.zeros((m, m), LD)
    for i in range(m):
        e = np.zeros(m, LD)
        e[i] = 1
        Y[i] = (e - X[i, :i] @ Y[:i]) / X[i, i]
    return Y


def _check_factor(nb, nu, A, Kp, x, rhs, rows, cols, well, label):
    """Everything the packed output of factor() and the vector of solve() promise, for one matrix.  Returns worst ratios."""
    n = 8 * nb
    M = np.zeros((n, n))
    M[rows, cols] = Kp
    ratios = {}
    # diagonal 8 x 8 blocks: explicit zeros above the diagonal
    for bi in range(nb):
        blk = M[8 * bi:8 * bi + 8, 8 * bi:8 * bi + 8]
        assert np.all(np.triu(blk, 1) == 0), (label, bi, "non-zero above the diagonal of a diagonal block")
    import scipy.linalg as sl
    Lref = sl.cholesky(A, lower=True)
    kappa_A = np.linalg.cond(A)
    kappa_ss = 1.0   # largest condition number of a diagonal super-block of the factor
    L = M.astype(LD)
    for s in range(0, n, 64):
        e = min(s + 64, n)
        kappa_ss = max(kappa_ss, np.linalg.cond(Lref[s:e, s:e]))
        if well:
            # X = inv(L_ss): X L_ss = I within c n u |X| |L_ss|, times cond(A) for the forward error of scipy's L_ss itself
            X, Lss = M[s:e, s:e].astype(LD), Lref[s:e, s:e].astype(LD)
            R = np.abs(X @ Lss - np.eye(e - s, dtype=LD))
            ratios["X L = I"] = max(ratios.get("X L = I", 0.0), _ratio(R, C_CHOL * n * U * kappa_A * (np.abs(X) @ np.abs(Lss))))
        L[s:e, s:e] = _tri_inv_ld(M[s:e, s:e])
    # the triangular solves multiply by the inverted super-blocks: where those are ill-conditioned (the KKT-like matrices)
    # the backward errors carry their condition number
    scale = 1.0 if well else kappa_ss
    AL = A.astype(LD)
    # backward error of the factor
    be = np.sqrt(np.sum((L @ L.T - AL) ** 2)) / np.sqrt(np.sum(AL ** 2))
    ratios["factor backward"] = float(be / (C_CHOL * n * U * scale))
    if well:   # forward agreement with scipy's factor (normwise, scaled by the condition number)
        fe = np.sqrt(np.sum((L - Lref.astype(LD)) ** 2)) / np.sqrt(np.sum(Lref.astype(LD) ** 2))
        ratios["factor forward"] = float(fe / (C_CHOL * n * U * kappa_A))
    # solve: normwise backward error in long double; the padding entries stay exactly zero
    assert np.all(x[nu:] == 0), (label, "padding entries of the solution are not zero")
    xl, bl = x.astype(LD), rhs.astype(LD)
    res = np.max(np.abs(AL @ xl - bl))
    nA = np.max(np.sum(np.abs(AL), axis=1))
    ratios["solve backward"] = float(res / (nA * np.max(np.abs(xl)) + np.max(np.abs(bl))) / (C_CHOL * n * U * scale))
    bad = {k: v for k, v in ratios.items() if not v <= 1.0}
    assert not bad, (label, f"cond of the diagonal super-blocks {kappa_ss:.3g}", bad)
    return ratios


_CHOL_WORST = {}


@pytest.mark.parametrize("nb", list(range(1, 24)))
def test_block_cholesky_against_long_double(chol, nb):
    """chol::factor + chol::solve for nb = 1 .. 23 block rows (20: the max_spline_vars cap; 16 / 17: a second / third 64 x 64
    super-block; 21 .. 23: beyond the cap), nu = 8 nb - r, r in {0, 3, 7}, with k_ipm's identity padding: well-conditioned SPD
    and KKT-like matrices (H + 1e-10 I + C' diag(w) C, w over sixteen decades), several different matrices per grid.
    Backward errors of the factor and of the solve <= 32 n u (times the condition number of the inverted diagonal super-blocks
    for the KKT-like matrices: the solves multiply by those inverses), the inverted super-blocks against scipy's factor, the
    forward error on the well-conditioned ones, the pivot flag; 256 and 512 threads bit-identical, a CTA of a grid bit-identical
    to the same matrix launched alone."""
    n = 8 * nb
    rows, cols = _block_index(nb)
    rng = np.random.default_rng(1000 + nb)
    mats, kinds, nus = [], [], []
    for r in (0, 3, 7):
        nu = n - r
        if nu < 1:
            continue
        for well in (True, True, False, False):
            A = _pad(_spd_well(rng, nu) if well else _spd_kkt(rng, nu), n)
            mats.append(A)
            kinds.append(well)
            nus.append(nu)
    packed = np.stack([A[rows, cols] for A in mats])
    rhs = np.zeros((len(mats), n))
    for i, nu in enumerate(nus):
        rhs[i, :nu] = rng.standard_normal(nu)
    K256, x256, f256 = chol(256, nb, packed, rhs)
    K512, x512, f512 = chol(512, nb, packed, rhs)
    assert np.all(f256 == 0) and np.all(f512 == 0), (f256, f512)
    # no block's summation order depends on which warp computes it
    assert np.array_equal(K256, K512) and np.array_equal(x256, x512), "256- and 512-thread results differ"
    one = len(mats) - 1
    K1, x1, _ = chol(256, nb, packed[one:one + 1], rhs[one:one + 1])
    assert np.array_equal(K1[0], K256[one]) and np.array_equal(x1[0], x256[one]), "a CTA of the grid differs from a lone launch"
    failures = []
    for i, A in enumerate(mats):
        try:
            ratios = _check_factor(nb, nus[i], A, K256[i], x256[i], rhs[i], rows, cols, kinds[i], f"nb {nb} matrix {i}")
        except AssertionError as e:
            failures.append(str(e))
            continue
        for k, v in ratios.items():
            key = ("well " if kinds[i] else "kkt ") + k
            _CHOL_WORST[key] = max(_CHOL_WORST.get(key, 0.0), v)
    print(f"nb {nb}: largest error / bound so far " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(_CHOL_WORST.items())))
    assert not failures, failures

    # pivot failure: A = L0 D L0' with D > 0 except D[p] = -1, so the first non-positive pivot is p
    piv = [p for p in (0, 7, 8, 63, 64, n - 1) if p < n]
    pm = []
    for p in piv:
        L0 = np.eye(n) + np.tril(rng.standard_normal((n, n)), -1) * (0.3 / np.sqrt(n))
        d = rng.uniform(1.0, 2.0, n)
        d[p] = -1.0
        pm.append((L0 * d) @ L0.T)
    pp = np.stack([A[rows, cols] for A in pm])
    prhs = np.zeros((len(pm), n))
    _, _, pf256 = chol(256, nb, pp, prhs)
    _, _, pf512 = chol(512, nb, pp, prhs)
    assert pf256.tolist() == [1] * len(piv) and pf512.tolist() == [1] * len(piv), (piv, pf256, pf512)
