"""k_ipm's interior-point iteration, one Newton iteration at a time, against a long-double restatement of the same operations.

A trace build of the library (tools/build_trace.sh: k_ipm compiled with -DBGG_IPM_TRACE, csrc/bgg_ipm_trace.cuh) records,
for one CTA, every pass of the interior-point loop: the iterate, the residuals as the kernel holds them, the row weights,
the assembled K before the factorisation, the solve vectors, the total direction and the step.  The reference is built in
np.longdouble from the same handle's own data: the condensed constraint rows C, d from kernel 3's sparse export, the
condensed H and the foot-box rows phipos, the equality rows E, e.  Condensing is bounded by tests/test_gpu_linalg.py; here
the GPU's own H and phipos are used, so every bound below is about the iteration alone.

The end-to-end tests compare minimisers to 1e-4 and iteration counts to a few steps.  An error in K or in the direction
does not move the fixed point (the residuals are separate code, and the solves are refined against the matrix-free
operators): it only costs iterations, or turns a nearly degenerate instance from Solved into SolvedInacc.  Checked here:

a. the weights w = z / (s + eps z) on active rows, exactly 0 on the rows that are structurally zero (kept out with z = 0);
b. K = H + eps I + C' diag(w) C + E'E / delta, lower triangle, componentwise within c k u of the same sum over absolute
   values; structural zeros exact; the padding rows and columns exactly the identity;
c. the residuals rx, rz, re where they are evaluated from scratch, componentwise; where rz and re are updated incrementally,
   their drift from the fresh residual, against a tenth of the feasibility tolerance they are compared with;
d. the direction: the exact relations of the kernel's Newton system (dz, ds, dy, the kappa equation), dtau recomputed from
   the pass vectors, the normwise backward error of the equation the Cholesky solves carry, and the starting point;
e. the step: amax bit for bit, alpha = 0.99 amax, the next iterate = this one + alpha times the direction (to 1 ulp);
f. the exit status, from the last record's norms and tolerances.

The trace library must return what the production library returns, bit for bit, on the same inputs.
"""
import ctypes as C
import importlib.util
import os
import shutil
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import common
from common import wl

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "bilevel-gait-gen_b200")
U = 2.0 ** -53
LD = np.longdouble
C_SUM = 4      # componentwise: |error| <= C_SUM * k * u * (the same sum over absolute values), k the longest sum
C_SOLVE = 32   # normwise backward error of the solves <= C_SOLVE * n * u (times the super-block condition number unrefined)
DRIFT = 0.1    # incremental rz / re: drift <= DRIFT * ipm_tol_feas * nrm_d * tau
SOLVED, SOLVED_INACC, MAX_ITER, PRIMAL_INF, PRIMAL_INF_INACC, OTHER = 0, 1, 2, 3, 5, 8

# per-foot scalings of the default trot schedule whose horizons hold 15 .. 20 block rows at N = 20 (tests/test_gpu_linalg.py)
_SCHEDULES = [
    ([1.097, 0.991, 0.843, 0.811], 0.00),   # nb 16
    ([0.965, 0.688, 1.032, 0.871], 0.00),   # nb 17
    ([0.850, 0.692, 0.748, 0.887], 0.15),   # nb 19
    ([0.733, 0.869, 0.821, 1.066], 0.20),   # nb 20
    ([0.918, 0.735, 0.620, 0.608], 0.00),   # nb 20 (160, the cap)
    ([1.000, 1.000, 1.000, 1.000], 0.00),   # nb 15
]


# --------------------------------------------------------------------------------------------------------------------------
# the trace library
# --------------------------------------------------------------------------------------------------------------------------

def _trace_lib_path(tmp_dir):
    """BGG_IPM_TRACE_LIB names a library built elsewhere (from modified sources, say); else a fresh build when nvcc is
    present; else the copy build() leaves in tools/bin."""
    given = os.environ.get("BGG_IPM_TRACE_LIB")
    if given:
        return given
    prebuilt = os.path.join(ROOT, "tools", "bin", "libbgg_b200_trace.so")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc) or not os.path.exists(os.path.join(PKG, "build", "bgg_capi.o")):
        if os.path.exists(prebuilt):
            return prebuilt
        pytest.skip("nvcc or the objects of build.sh not found and the trace library is not built "
                    "(python -c 'import __graft_entry__ as g; g.build()')")
    out = os.path.join(tmp_dir, "libbgg_b200_trace.so")
    subprocess.run(["bash", os.path.join(ROOT, "tools", "build_trace.sh")], check=True, env=dict(os.environ, NVCC=nvcc, OUT=out),
                   stdout=subprocess.DEVNULL)
    return out


@pytest.fixture(scope="module")
def tmod(tmp_path_factory):
    """bgg_b200.py loaded a second time, under another name, over the trace library (the production binding keeps its own)."""
    path = _trace_lib_path(str(tmp_path_factory.mktemp("ipm_trace")))
    spec = importlib.util.spec_from_file_location("bgg_b200_trace", os.path.join(PKG, "bgg_b200.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.LIB_PATH = path
    L = mod.lib()
    L.bgg_debug_ipm_trace_arm.argtypes = [C.c_int, C.c_int]
    L.bgg_debug_ipm_trace_fetch.argtypes = [C.POINTER(C.c_int32), C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_double), C.c_int]
    yield mod
    L.bgg_debug_ipm_trace_arm(-1, 0)


class Record:
    """One traced pass of the interior-point loop: scalars as floats, vectors cut to the instance's sizes."""

    def __init__(self, raw, layout):
        self.f = {}
        for name, (o, n) in layout.items():
            self.f[name] = raw[o:o + n]
        sc = {k: float(v[0]) for k, v in self.f.items() if len(v) == 1}
        self.__dict__.update(sc)
        nu, m, neq, nb = int(self.nu), int(self.m), int(self.neq), int(self.nb)
        sizes = dict(nu=nu, rows=m, eq=neq, K=nb * (nb + 1) // 2 * 64)
        for name, v in self.f.items():
            if len(v) > 1:
                kind = ("K" if name == "K" else "nu" if name in ("u", "Hu", "rx", "x1", "x2", "du") else
                        "eq" if name in ("y", "re", "y1", "y2", "dy", "dre") else "rows")
                setattr(self, name, v[:sizes[kind]].copy())


def _fetch(mod):
    L = mod.lib()
    hdr = np.zeros(5 + 2 * 256, np.int32)
    names = C.create_string_buffer(8192)
    ip, dp = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    assert L.bgg_debug_ipm_trace_fetch(hdr.ctypes.data_as(ip), len(hdr), names, 8192, None, 0) == 0
    rec_d, nf, count, stored, launches = (int(v) for v in hdr[:5])
    assert count <= stored, f"the trace buffer held {stored} of {count} records"
    raw = np.zeros((max(stored, 1), rec_d))
    assert L.bgg_debug_ipm_trace_fetch(hdr.ctypes.data_as(ip), len(hdr), names, 8192, raw.ctypes.data_as(dp), stored) == 0
    fields = names.value.decode().rstrip(",").split(",")
    assert len(fields) == nf
    layout = {fields[f]: (int(hdr[5 + 2 * f]), int(hdr[6 + 2 * f])) for f in range(nf)}
    return [Record(raw[r], layout) for r in range(stored)], launches


def _make(mod, cfg_name, B, states, **kw):
    cfg = wl.CONFIGS[cfg_name]
    m = mod.BatchedMPC(cfg["num_nodes"], cfg["integrator_dt"], wl.robot(), **wl.mpc_kwargs(cfg), **kw)
    m.AddQuadraticTrackingCost(wl.target_tangent(cfg), np.asarray(cfg["Q"], float))
    m.Reset(B)
    m.SetStateTrajectoryWarmStart(states)
    return m


# --------------------------------------------------------------------------------------------------------------------------
# the long-double reference of the condensed constraints
# --------------------------------------------------------------------------------------------------------------------------

def _reference(gpu, b):
    """C, d (kernel row order), E, e, the structurally zero rows, H, g of instance b's last solve, in long double.  The
    inequality rows of kernel 3's export are A_x x + A_u u <= ub with x_k = Phi_k u + phi_k: the foot-box rows touch the
    positions p_c(k) only, whose Phi rows are phipos and whose phi rows are xoff."""
    N = gpu.N
    sz = gpu.sizes(b)
    nu, ns, ne, neq = sz["nu"], sz["n_samples"], sz["n_eebox"], sz["n_eq"]
    m, nst = 6 * ns + 2 * ne, 12 * (N + 1)
    qp = gpu.GetQPData(b, 1, nnz_cap=80000)[0]
    A, ub = qp["A"].toarray(), qp["ub"]
    assert A.shape == (nst + m + neq, nst + nu) and qp["num_eq"] == nst + neq and qp["num_ineq"] == m
    cond = gpu.condensed(b)
    H, g, phipos, xoff = (cond[k] for k in ("H", "g", "phipos", "xoff"))
    Ain, uin = A[nst:nst + m], ub[nst:nst + m]
    Ax, Au = Ain[:, :nst].astype(LD), Ain[:, nst:].astype(LD)
    touched = np.nonzero(np.any(Ain[:, :nst] != 0, axis=0))[0]
    assert np.all((touched % 12 < 2) & (touched // 12 >= 4)), "an inequality row touches a state other than a foot-box position"
    Pmap = np.zeros((nst, nu), LD)
    for k in range(4, N + 1):
        for c in range(2):
            Pmap[12 * k + c] = phipos[(k - 4) * 2 + c]
    perm = common.gpu_rows_to_reference_order({"sizes": sz}, N)   # reference inequality row r is kernel row perm[r]
    Cm, Ca, d, da = (np.zeros((m, nu), LD), np.zeros((m, nu), LD), np.zeros(m, LD), np.zeros(m, LD))
    Cm[perm] = Au + Ax @ Pmap
    Ca[perm] = np.abs(Au) + np.abs(Ax) @ np.abs(Pmap)
    d[perm] = uin.astype(LD) - Ax @ xoff.reshape(-1).astype(LD)
    da[perm] = np.abs(uin).astype(LD) + np.abs(Ax) @ np.abs(xoff.reshape(-1)).astype(LD)
    assert not np.any(A[nst + m:, :nst]), "an equality row touches a state"
    E, e = A[nst + m:, nst:].astype(LD), ub[nst + m:].astype(LD)
    return dict(N=N, nu=nu, m=m, neq=neq, nf=sz["nf"], C=Cm, Ca=Ca, d=d, da=da, E=E, e=e, zero=~np.any(Cm != 0, axis=1),
                H=H.astype(LD), g=g.astype(LD), nnz_col=int(np.max(np.sum(Cm != 0, axis=0), initial=0)),
                nnz_row=int(np.max(np.sum(Cm != 0, axis=1), initial=0)))


def _ratio(err, bound):
    """max err / bound; an entry with a zero bound must be exact."""
    err, bound = np.abs(np.asarray(err, LD)), np.asarray(bound, LD)
    if np.any((bound == 0) & (err != 0)):
        return np.inf
    nz = bound > 0
    return float(np.max(err[nz] / bound[nz])) if nz.any() else 0.0


def _ulp(x):
    return np.spacing(np.abs(np.asarray(x, np.float64)))


def _unpack_K(Kp, nb):
    n = 8 * nb
    M = np.full((n, n), np.nan)
    r8, c8 = np.divmod(np.arange(64), 8)
    for bi in range(nb):
        for bj in range(bi + 1):
            o = (bi * (bi + 1) // 2 + bj) * 64
            M[8 * bi + r8, 8 * bj + c8] = Kp[o:o + 64]
    return M


def _superblock_cond(K):
    """largest condition number of a 64 x 64 diagonal super-block of K's Cholesky factor (chol::solve multiplies by their inverses)"""
    import scipy.linalg as sl
    L = sl.cholesky(np.asarray(K, np.float64), lower=True)
    return max(np.linalg.cond(L[s:s + 64, s:s + 64]) for s in range(0, L.shape[0], 64))


# --------------------------------------------------------------------------------------------------------------------------
# the checks
# --------------------------------------------------------------------------------------------------------------------------

class Checker:
    def __init__(self):
        self.worst, self.cov, self.drift = {}, {}, {"rz": 0.0, "re": 0.0}

    def ratio(self, key, r, label):
        self.worst[key] = max(self.worst.get(key, 0.0), r)
        assert r <= 1.0, f"{label}: {key}: error / bound = {r:.3g}"

    def note(self, key, v):
        self.cov.setdefault(key, set()).add(v)

    def report(self):
        print("largest error / bound: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(self.worst.items())))
        print(f"incremental residual drift / (ipm_tol_feas nrm_d tau): rz {self.drift['rz']:.3g}, re {self.drift['re']:.3g}")
        print("coverage: " + "; ".join(f"{k} {sorted(v)}" for k, v in sorted(self.cov.items())))

    # ---------------------------------------------------------------------------------------------------------------
    def check_solve(self, gpu, b, recs, label, status, iters):
        assert recs, f"{label}: nothing traced"
        ref = _reference(gpu, b)
        nu, m, neq = ref["nu"], ref["m"], ref["neq"]
        Cm, Ca, E, Ea, H = ref["C"], ref["Ca"], ref["E"], np.abs(ref["E"]), ref["H"]
        act = ~ref["zero"]
        r0 = recs[0]
        assert r0.it == -1, (label, r0.it)
        assert (int(r0.nu), int(r0.m), int(r0.neq), int(r0.N)) == (nu, m, neq, ref["N"]), label
        self.note("launch <spill, threads> stage_phi want", (int(r0.spill), int(r0.threads), int(r0.stage_phi), int(r0.want)))
        self.note("nb", int(r0.nb))
        self.note("nu", nu)
        eps, delta, inv_delta = r0.eps, r0.delta, 1.0 / r0.delta
        # right-hand sides: the kernel's d against ub + xoff
        self.ratio("d", _ratio(r0.d.astype(LD) - ref["d"], 2 * U * ref["da"]), label)
        k_res = nu + ref["nnz_col"] + neq + 3
        kK = max(ref["nnz_col"], 1) + 2 * neq + 4
        for i, r in enumerate(recs):
            lab = f"{label} record {i} (it {int(r.it)})"
            assert int(r.m_act) == int(act.sum()), lab
            # the structurally zero rows stay out: z = 0, s = 1 throughout
            assert np.all(r.z[ref["zero"]] == 0) and np.all(r.s[ref["zero"]] == 1.0), lab
            assert np.all(r.z[act] > 0) and np.all(r.s[act] > 0), lab
            u, s, z, y = (x.astype(LD) for x in (r.u, r.s, r.z, r.y))
            tau = LD(r.tau)
            if r.it >= 0:
                self._residuals(r, ref, u, s, z, y, tau, k_res, lab)
            if not np.isnan(r.w[0]):
                Kref = self._weights_and_K(r, ref, kK, lab)
                if r.it >= 0:
                    self.note("refined", int(r.refine))
                if not np.isnan(r.x1[0]):
                    self._solves(r, ref, Kref, lab)
            if r.it >= 0 and not np.isnan(r.alpha):
                self._direction_and_step(r, recs[i + 1] if i + 1 < len(recs) else None, ref, lab)
            elif r.it >= 0 and i + 1 < len(recs):
                # no direction: the convergence test passed on updated residuals; the next pass re-evaluates the same iterate
                nx = recs[i + 1]
                assert nx.confirm == 1 and nx.it == r.it and nx.fresh == 1, lab
                for f in ("u", "s", "z", "y", "tau", "kap"):
                    assert np.array_equal(getattr(nx, f), getattr(r, f)), (lab, f)
                self.note("statuses", "confirm step")
        self._start(recs, ref, label)
        self._exit(recs, label, status, iters)

    def _residuals(self, r, ref, u, s, z, y, tau, k_res, lab):
        Cm, Ca, E, H, g, d = ref["C"], ref["Ca"], ref["E"], ref["H"], ref["g"], r.d.astype(LD)
        act = ~ref["zero"]
        rx = H @ u + Cm.T @ z + E.T @ y + g * tau
        rxa = np.abs(H) @ np.abs(u) + Ca.T @ np.abs(z) + np.abs(E).T @ np.abs(y) + np.abs(g) * tau
        rz = Cm @ u + s - d * tau
        rza = Ca @ np.abs(u) + np.abs(s) + np.abs(d) * tau
        re = E @ u - ref["e"] * tau
        rea = np.abs(E) @ np.abs(u) + np.abs(ref["e"]) * tau
        tol = C_SUM * k_res * U
        self.ratio("Hu", _ratio(r.Hu.astype(LD) - H @ u, tol * (np.abs(H) @ np.abs(u))), lab)
        self.ratio("rx", _ratio(r.rx.astype(LD) - rx, tol * rxa), lab)
        assert np.all(r.rz[ref["zero"]] == 0), lab
        # the norms the exit test reads, from the vectors it reads them from (maxima: exact)
        assert r.res_d == np.max(np.abs(r.rx)) / r.tau, lab
        assert r.res_p == max(np.max(np.abs(r.rz[act]), initial=0.0), np.max(np.abs(r.re), initial=0.0)) / r.tau, lab
        if r.fresh:
            self.ratio("rz fresh", _ratio(r.rz[act].astype(LD) - rz[act], tol * rza[act]), lab)
            self.ratio("re fresh", _ratio(r.re.astype(LD) - re, tol * rea), lab)
            self.note("rz", "fresh")
        else:
            scale = LD(r.tol_feas) * LD(r.nrm_d) * tau
            drz = float(np.max(np.abs(r.rz[act].astype(LD) - rz[act]), initial=0) / scale)
            dre = float(np.max(np.abs(r.re.astype(LD) - re), initial=0) / scale)
            self.drift["rz"], self.drift["re"] = max(self.drift["rz"], drz), max(self.drift["re"], dre)
            assert drz <= DRIFT and dre <= DRIFT, f"{lab}: incremental residual drift rz {drz:.3g} re {dre:.3g} of the tolerance"
            self.note("rz", "updated")

    def _weights_and_K(self, r, ref, kK, lab):
        act, eps = ~ref["zero"], r.eps
        z, s = r.z.astype(LD), r.s.astype(LD)
        wref = np.zeros(ref["m"], LD)
        wref[act] = z[act] / (s[act] + LD(eps) * z[act])
        assert np.all(r.w[ref["zero"]] == 0), lab
        self.ratio("w", _ratio(r.w[act].astype(LD) - wref[act], 3 * U * wref[act]), lab)
        nu, nb = ref["nu"], int(r.nb)
        n = 8 * nb
        w = r.w.astype(LD)
        Cm, Ca, E = ref["C"], ref["Ca"], ref["E"]
        Kref = ref["H"] + LD(eps) * np.eye(nu, dtype=LD) + (Cm.T * w) @ Cm + (E.T @ E) / LD(r.delta)
        Kabs = np.abs(ref["H"]) + LD(eps) * np.eye(nu, dtype=LD) + (Ca.T * np.abs(w)) @ Ca + (np.abs(E).T @ np.abs(E)) / LD(r.delta)
        M = _unpack_K(r.K, nb)
        low = np.tril(np.ones((nu, nu), bool))   # the upper triangle of the diagonal 8 x 8 blocks is never read by chol::factor
        tol = C_SUM * kK * U
        assert tol * float(Kabs.max()) < 1e-10 * float(np.abs(M[:nu, :nu][low]).max()), (lab, "vacuous bound on K")
        self.ratio("K", _ratio((M[:nu, :nu].astype(LD) - Kref)[low], tol * Kabs[low]), lab)
        pad = np.eye(n)
        lowall = np.tril(np.ones((n, n), bool))
        padmask = lowall.copy()
        padmask[:nu, :nu] = False
        assert np.array_equal(M[padmask], pad[padmask]), (lab, "K padding is not the identity")
        return Kref

    def _solves(self, r, ref, Kref, lab):
        """Normwise backward error of the equation each solve carries, K x = b, in long double."""
        nu, nb, n = ref["nu"], int(r.nb), 8 * int(r.nb)
        act = ~ref["zero"]
        Cm, Ca, E, Ea, g = ref["C"], ref["Ca"], ref["E"], np.abs(ref["E"]), ref["g"]
        w, d = r.w.astype(LD), r.d.astype(LD)
        Kabs = np.abs(Kref)
        inv_delta = LD(1.0) / LD(r.delta)
        # pass 0: K x1 = -g + C'(w d) + E' e / delta
        x1 = r.x1.astype(LD)
        b1 = -g + Cm.T @ (w * d) + E.T @ ref["e"] * inv_delta
        b1a = np.abs(g) + Ca.T @ np.abs(w * d) + Ea.T @ np.abs(ref["e"]) * inv_delta
        refine = r.it >= 0 and r.refine == 1
        kap_ss = 1.0 if refine else _superblock_cond(Kref)
        bound = C_SOLVE * n * U * kap_ss
        res1 = Kref @ x1 - b1
        nrm1 = np.max(Kabs @ np.abs(x1) + b1a)
        self.ratio("solve x1" + (" refined" if refine else ""), float(np.max(np.abs(res1)) / nrm1) / bound, lab)
        # the constant solve's C x1 and y1 = (E x1 - e) / delta as the kernel formed them
        kr = C_SUM * (ref["nnz_row"] + 2) * U
        self.ratio("C x", _ratio(r.cx1.astype(LD) - Cm @ x1, kr * (Ca @ np.abs(x1))), lab)
        ey = (E @ x1 - ref["e"]) * inv_delta
        self.ratio("E x", _ratio(r.y1.astype(LD) - ey, kr * (Ea @ np.abs(x1) + np.abs(ref["e"])) * inv_delta), lab)
        if r.it < 0 or np.isnan(r.alpha):
            return
        # the total direction: K du = b2 + dtau b1 with b2 = -scale rx + C'(w a2) - scale E' re / delta
        scale = LD(1.0) - LD(r.sigma)
        x2, du, dtau = r.x2.astype(LD), r.du.astype(LD), LD(r.dtau)
        a2 = r.a2.astype(LD)
        b2 = -scale * r.rx.astype(LD) + Cm.T @ (w * a2) - scale * (E.T @ r.re.astype(LD)) * inv_delta
        b2a = scale * np.abs(r.rx.astype(LD)) + Ca.T @ np.abs(w * a2) + scale * (Ea.T @ np.abs(r.re.astype(LD))) * inv_delta
        self.ratio("C x", _ratio(r.cx2.astype(LD) - Cm @ x2, kr * (Ca @ np.abs(x2))), lab)
        # the issue's form of the same equation: (H + eps I) du + C'dz + E'dy + g dtau = -scale rx -- with dz, dy as formed
        lhs = (ref["H"] + LD(r.eps) * np.eye(nu, dtype=LD)) @ du + Cm.T @ r.dz.astype(LD) + E.T @ r.dy.astype(LD) + g * dtau
        res = lhs + scale * r.rx.astype(LD)
        nrm = np.max(Kabs @ (np.abs(x2) + abs(dtau) * np.abs(x1)) + b2a + abs(dtau) * b1a)
        self.ratio("solve du" + (" refined" if refine else ""), float(np.max(np.abs(res)) / nrm) / bound, lab)
        self.ratio("solve K du", float(np.max(np.abs(Kref @ du - b2 - dtau * b1)) / nrm) / bound, lab)

    def _direction_and_step(self, r, nx, ref, lab):
        act = ~ref["zero"]
        m, neq = ref["m"], ref["neq"]
        w, d, s, z = (r.w.astype(LD), r.d.astype(LD), r.s.astype(LD), r.z.astype(LD))
        dtau, tau, kap = LD(r.dtau), LD(r.tau), LD(r.kap)
        scale = LD(1.0) - LD(r.sigma)
        cx1, cx2, a2 = r.cx1.astype(LD), r.cx2.astype(LD), r.a2.astype(LD)
        rz = r.rz.astype(LD)
        # exact relations of the kernel's Newton system, to rounding
        t = cx2 + dtau * cx1
        dz = w * (t - a2 - dtau * d)
        dza = np.abs(w) * (np.abs(cx2) + abs(dtau) * np.abs(cx1) + np.abs(a2) + abs(dtau) * np.abs(d))
        self.ratio("dz", _ratio((r.dz.astype(LD) - dz)[act], 6 * U * dza[act]), lab)
        assert np.all(r.dz[ref["zero"]] == 0) and np.all(r.ds[ref["zero"]] == 0), lab
        dzk = r.dz.astype(LD)
        sz = np.where(act, s / np.where(act, z, 1), 0)
        ds = -(a2 + scale * rz) - sz * dzk
        dsa = np.abs(a2) + scale * np.abs(rz) + sz * np.abs(dzk)
        self.ratio("ds", _ratio((r.ds.astype(LD) - ds)[act], 6 * U * dsa[act]), lab)
        dy = r.y2.astype(LD) + dtau * r.y1.astype(LD)
        self.ratio("dy", _ratio(r.dy.astype(LD) - dy, 3 * U * (np.abs(r.y2.astype(LD)) + abs(dtau) * np.abs(r.y1.astype(LD)))), lab)
        mu, sigma, dkdt = LD(r.mu), LD(r.sigma), LD(r.dkdt_aff)
        d_kap = kap * tau + dkdt - sigma * mu
        dkap = LD(r.dkap)
        self.ratio("kappa equation", _ratio(tau * dkap + kap * dtau + d_kap,
                                            8 * U * (abs(tau * dkap) + abs(kap * dtau) + abs(kap * tau) + abs(dkdt) + abs(sigma * mu))), lab)
        # dtau from the pass vectors: z_x = W (C x - a2), with a2 = d for the constant pass
        g, Hu, uHu, e = ref["g"], r.Hu.astype(LD), LD(r.uHu), ref["e"]
        x1, x2 = r.x1.astype(LD), r.x2.astype(LD)
        zx1 = np.where(act, w * (cx1 - d), 0)
        zx2 = np.where(act, w * (cx2 - a2), 0)
        den_terms = [kap / tau, -(g @ x1), -(d @ zx1), -(e @ r.y1.astype(LD)), uHu / (tau * tau), -2 * (Hu @ x1) / tau]
        den_abs = (kap / tau + np.abs(g) @ np.abs(x1) + np.abs(d) @ np.abs(zx1) + np.abs(e) @ np.abs(r.y1.astype(LD)) + abs(uHu) / tau ** 2
                   + 2 * (np.abs(Hu) @ np.abs(x1)) / tau)
        den = sum(den_terms)
        num_terms = [scale * LD(r.rt), -d_kap / tau, g @ x2, d @ zx2, e @ r.y2.astype(LD), 2 * (Hu @ x2) / tau]
        num_abs = (abs(scale * LD(r.rt)) + abs(d_kap / tau) + np.abs(g) @ np.abs(x2) + np.abs(d) @ np.abs(zx2)
                   + np.abs(e) @ np.abs(r.y2.astype(LD)) + 2 * (np.abs(Hu) @ np.abs(x2)) / tau)
        num = sum(num_terms)
        k = ref["nu"] + m + neq + 6
        self.ratio("den", _ratio(LD(r.den) - den, C_SUM * k * U * den_abs), lab)
        self.ratio("dtau", _ratio(dtau - num / den, C_SUM * k * U * (num_abs + abs(num / den) * den_abs) / abs(den)), lab)
        # the step: the same divisions and minima, so bit for bit
        amax = 1.0
        ds64, dz64 = r.ds[act], r.dz[act]
        neg = ds64 < 0
        if neg.any():
            amax = min(amax, float(np.min(-r.s[act][neg] / ds64[neg])))
        neg = dz64 < 0
        if neg.any():
            amax = min(amax, float(np.min(-r.z[act][neg] / dz64[neg])))
        if r.dtau < 0:
            amax = min(amax, -r.tau / r.dtau)
        if r.dkap < 0:
            amax = min(amax, -r.kap / r.dkap)
        assert r.amax == amax, (lab, r.amax, amax)
        assert r.alpha == 0.99 * r.amax, lab
        if nx is None:
            return
        assert nx.it == r.it + 1 and nx.confirm == 0, lab
        al = LD(r.alpha)

        def step(name, cur, dirn, nxt, mask=None):
            exact = cur.astype(LD) + al * dirn.astype(LD)
            err = np.abs(nxt.astype(LD) - exact)
            ok = err <= LD(0.5) * _ulp(nxt).astype(LD)
            ok |= nxt == cur + r.alpha * dirn   # not fused
            if mask is not None:
                ok |= ~mask
            # where the sum cancels, long double is not exact enough: exact rational arithmetic
            for i in np.nonzero(~ok)[0]:
                ex = Fraction(float(cur[i])) + Fraction(r.alpha) * Fraction(float(dirn[i]))
                e_ulp = abs(Fraction(float(nxt[i])) - ex) / Fraction(float(_ulp(nxt[i])))
                assert e_ulp <= 1, (lab, name, int(i), float(e_ulp))

        step("u", r.u, r.du, nx.u)
        step("s", r.s, r.ds, nx.s, act)
        step("z", r.z, r.dz, nx.z, act)
        step("y", r.y, r.dy, nx.y)
        step("tau", np.array([r.tau]), np.array([r.dtau]), np.array([nx.tau]))
        step("kappa", np.array([r.kap]), np.array([r.dkap]), np.array([nx.kap]))
        if not nx.fresh:
            step("rz", r.rz, r.drz, nx.rz, act)
            step("re", r.re, r.dre, nx.re)

    def _start(self, recs, ref, label):
        """Clarabel's QP initialisation as the kernel states it: u = x1, y = y1, z = W (C x1 - d) with W = 1 / (1 + eps), s = -z,
        both shifted into the cone by 1 - min when their minimum is below 1e-8; tau = kappa = 1."""
        r0 = recs[0]
        if len(recs) < 2:
            return
        r1 = recs[1]
        act = ~ref["zero"]
        assert r1.it == 0 and r1.tau == 1.0 and r1.kap == 1.0, label
        assert np.array_equal(r1.u, r0.x1) and np.array_equal(r1.y, r0.y1), label
        zv = (r0.cx1[act] - r0.d[act]) / (1.0 + r0.eps)
        smin, zmin = float(np.min(-zv)), float(np.min(zv))
        sshift = 1.0 - smin if smin < 1e-8 else 0.0
        zshift = 1.0 - zmin if zmin < 1e-8 else 0.0
        assert np.array_equal(r1.s[act], -zv + sshift) and np.array_equal(r1.z[act], zv + zshift), label
        # the starting weights: z = 1 on the active rows, s = 1
        assert np.all(r0.z[act] == 1.0) and np.all(r0.s == 1.0), label

    def _exit(self, recs, label, status, iters):
        last = recs[-1]
        assert last.status_exit == status and last.iters_exit == iters, (label, last.status_exit, status, last.iters_exit, iters)
        ok = lambda r: (r.res_d <= r.tol_feas * r.nrm_q and r.res_p <= r.tol_feas * r.nrm_d and r.gap <= r.tol_gap * r.gscale)
        infeas = lambda r, t: r.bz < -t and r.aty_n <= t * r.zn * (-r.bz)
        for r in recs[1:-1]:   # every pass but the last went on (converged on updated residuals: a confirm step follows)
            assert not (ok(r) and r.fresh) and (ok(r) or not infeas(r, r.tol_infeas)), (label, int(r.it))
        if last.it < 0 or np.isnan(last.res_p):
            return
        if status == SOLVED:
            assert ok(last) and last.fresh == 1, (label, "Solved on residuals that were not evaluated fresh")
            self.note("statuses", "Solved" + (" after a confirm step" if last.confirm else ""))
        elif status == PRIMAL_INF:
            assert not ok(last) and infeas(last, last.tol_infeas), label
            self.note("statuses", "PrimalInfeasible")
        else:
            assert not ok(last) and not infeas(last, last.tol_infeas), label
            red = last.res_d <= 1e-4 * last.nrm_q and last.res_p <= 1e-4 * last.nrm_d and last.gap <= 5e-5 * last.gscale
            want = SOLVED_INACC if red else (PRIMAL_INF_INACC if infeas(last, 5e-5) else None)
            if want is not None:
                assert status == want, (label, status, want)
            self.note("statuses", {SOLVED_INACC: "SolvedInacc", PRIMAL_INF_INACC: "PrimalInfeasibleInacc"}.get(status, str(status)))


# --------------------------------------------------------------------------------------------------------------------------
# the cases
# --------------------------------------------------------------------------------------------------------------------------

def _same_results(prod, trc, B, out_p, out_t, label):
    """The trace library computes what the production library computes, bit for bit."""
    assert np.array_equal(out_p["status"], out_t["status"]) and np.array_equal(out_p["iters"], out_t["iters"]), label
    for b in range(B):
        sp, st = prod.solution(b), trc.solution(b)
        for k in ("qp_sol", "lam", "slack", "nu_eq"):
            assert np.array_equal(sp[k], st[k]), (label, b, k)


@pytest.fixture(scope="module")
def chk():
    c = Checker()
    yield c
    c.report()


def test_trace_first_and_second_solve_n20(tmod, chk):
    """N = 20, four instances: alone on the device (stage_phi from the spare room), first solve in the second pass (nothing
    speculated yet), the next one in the first pass; nb = 15, paired work list.  Then the same with refinement held back
    (ipm_refine_after = -1) and a batch of 300 (not alone)."""
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    B = 4
    states, t0, ee = wl.batched_trot_inputs(cfg, B, seed=7)
    for kw in ({}, {"ipm_refine_after": -1}):
        prod = common.make_gpu(cfg_name, B, states, **kw)
        outs_p = [prod.GetRealTimeUpdate(states, t0, ee) for _ in range(2)]
        for b in (0, 3):
            trc = _make(tmod, cfg_name, B, states, **kw)
            assert tmod.lib().bgg_debug_ipm_trace_arm(b, 160) == 0
            for k in range(2):
                out = trc.GetRealTimeUpdate(states, t0, ee)
                recs, _ = _fetch(tmod)
                chk.check_solve(trc, b, recs, f"N = 20 {kw} instance {b} solve {k}", int(out["status"][b]), int(out["iters"][b]))
            _same_results(prod, trc, B, outs_p[1], out, f"N = 20 second solve {kw}")
            trc.close()
        # the first solve's results, compared on a handle that solved once
        trc = _make(tmod, cfg_name, B, states, **kw)
        prod2 = common.make_gpu(cfg_name, B, states, **kw)
        _same_results(prod2, trc, B, prod2.GetRealTimeUpdate(states, t0, ee), trc.GetRealTimeUpdate(states, t0, ee), f"N = 20 first {kw}")
        trc.close()
        prod2.close()
        prod.close()
    # a batch of 300: more CTAs than SMs
    B = 300
    states, t0, ee = wl.batched_trot_inputs(cfg, B, seed=9)
    prod = common.make_gpu(cfg_name, B, states)
    out_p = prod.GetRealTimeUpdate(states, t0, ee)
    trc = _make(tmod, cfg_name, B, states)
    assert tmod.lib().bgg_debug_ipm_trace_arm(123, 160) == 0
    out = trc.GetRealTimeUpdate(states, t0, ee)
    _same_results(prod, trc, B, out_p, out, "N = 20 batch of 300")
    recs, _ = _fetch(tmod)
    chk.check_solve(trc, 123, recs, "N = 20 batch of 300 instance 123", int(out["status"][123]), int(out["iters"][123]))
    tmod.lib().bgg_debug_ipm_trace_arm(-1, 0)
    trc.close()
    prod.close()
    launches = chk.cov["launch <spill, threads> stage_phi want"]
    assert {(0, 256, 0, 2), (0, 256, 1, 2), (0, 256, 1, 0)} <= launches, launches
    assert 15 in chk.cov["nb"] and chk.cov["refined"] == {0, 1}


def test_trace_mixed_batch_up_to_the_cap(tmod, chk):
    """One batch with 15 .. 20 block rows (nu = 160, the cap, and nu not a multiple of 8): k_ipm<false, 512>, the segment
    packing of the KKT work list from nb = 16 on, the paired list at nb = 15."""
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    B = len(_SCHEDULES)
    init = np.asarray(cfg["srb_init"], float)
    states, ee = np.tile(init, (B, 1)), np.tile(wl.EE_NOMINAL, (B, 1, 1))
    base = np.array([0.0, 0.3, 0.6, 0.9, 1.2])
    times = np.array([[base * s for s in sc] for sc, _ in _SCHEDULES])
    t0 = np.array([t for _, t in _SCHEDULES])

    def make(mod_make):
        g = mod_make()
        g.UpdateContactTimes(times)
        return g
    prod = make(lambda: common.make_gpu(cfg_name, B, states))
    out_p = prod.GetRealTimeUpdate(states, t0, ee)
    for b in range(B):
        trc = make(lambda: _make(tmod, cfg_name, B, states))
        assert tmod.lib().bgg_debug_ipm_trace_arm(b, 160) == 0
        out = trc.GetRealTimeUpdate(states, t0, ee)
        _same_results(prod, trc, B, out_p, out, "mixed batch")
        recs, _ = _fetch(tmod)
        assert recs[0].threads == 512, "nu = 160 in the batch: k_ipm<false, 512>"
        chk.check_solve(trc, b, recs, f"mixed batch instance {b} (nu {trc.sizes(b)['nu']})", int(out["status"][b]), int(out["iters"][b]))
        trc.close()
    tmod.lib().bgg_debug_ipm_trace_arm(-1, 0)
    prod.close()
    assert {15, 16, 17, 19, 20} <= chk.cov["nb"], chk.cov["nb"]   # nb = 18: the closed loop below
    assert 160 in chk.cov["nu"] and any(n % 8 for n in chk.cov["nu"]), chk.cov["nu"]


def test_trace_gait_opt_n50(tmod, chk):
    """N = 50 (the spill layout, k_ipm<true, 256>): the batch of test_first_solve_matches_oracle at 1e-9, which holds Solved
    and PrimalInfeasible instances."""
    cfg_name = "a1_gait_opt_config"
    cfg = wl.CONFIGS[cfg_name]
    B = 16
    states, t0, ee = wl.batched_trot_inputs(cfg, B, seed=3)
    states[0] = cfg["srb_init"]
    ee[0] = wl.EE_NOMINAL
    kw = dict(ipm_tol=1e-9, ipm_tol_gap=1e-9)
    prod = common.make_gpu(cfg_name, B, states, **kw)
    out_p = prod.GetRealTimeUpdate(states, t0, ee)
    st = out_p["status"]
    picks = [int(np.nonzero(st == SOLVED)[0][0])] + [int(i) for i in np.nonzero(st == PRIMAL_INF)[0][:1]]
    for b in picks:
        trc = _make(tmod, cfg_name, B, states, **kw)
        assert tmod.lib().bgg_debug_ipm_trace_arm(b, 160) == 0
        out = trc.GetRealTimeUpdate(states, t0, ee)
        _same_results(prod, trc, B, out_p, out, "N = 50")
        recs, _ = _fetch(tmod)
        assert recs[0].spill == 1 and recs[0].threads == 256, "N = 50: k_ipm<true, 256>"
        chk.check_solve(trc, b, recs, f"N = 50 instance {b}", int(out["status"][b]), int(out["iters"][b]))
        trc.close()
    tmod.lib().bgg_debug_ipm_trace_arm(-1, 0)
    prod.close()
    assert "PrimalInfeasible" in chk.cov["statuses"], chk.cov["statuses"]


def test_trace_closed_loop_second_pass(tmod, chk):
    """The horizon grows along a closed loop (plant = node 1 of the solved trajectory): at the tick it outgrows the caps the
    solve was speculatively launched with, the instance is picked up by the second pass (want = 2)."""
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    dt = cfg["integrator_dt"]
    states, t0, ee = wl.disturbance_sweep_inputs(cfg, 1, seed=4)
    prod = common.make_gpu(cfg_name, 1, states)
    trc = _make(tmod, cfg_name, 1, states)
    prod.upload(states, t0, ee)
    trc.upload(states, t0, ee)
    assert tmod.lib().bgg_debug_ipm_trace_arm(0, 160) == 0
    wants = []
    for tick in range(20):
        if tick:
            prod.advance_plant(dt)
            trc.advance_plant(dt)
        prod.solve_resident()
        trc.solve_resident()
        out_p, out = prod.download(), trc.download()
        _same_results(prod, trc, 1, out_p, out, f"closed loop tick {tick}")
        recs, _ = _fetch(tmod)
        wants.append((int(recs[0].want), int(recs[0].nb)))
        chk.check_solve(trc, 0, recs, f"closed loop tick {tick}", int(out["status"][0]), int(out["iters"][0]))
    tmod.lib().bgg_debug_ipm_trace_arm(-1, 0)
    trc.close()
    prod.close()
    grown = [i for i in range(1, len(wants)) if wants[i][1] > wants[i - 1][1]]
    assert grown and all(wants[i][0] == 2 for i in grown), wants
    assert any(w == 0 for w, _ in wants[1:]), wants


def test_trace_coverage(chk, capsys):
    """Runs last: what the cases above reached, from the traced launch facts."""
    if not chk.cov:
        pytest.skip("no traced case ran")
    launches = chk.cov["launch <spill, threads> stage_phi want"]
    assert {(s, t) for s, t, _, _ in launches} == {(0, 256), (1, 256), (0, 512)}, launches
    assert {p for _, _, p, _ in launches} == {0, 1} and {w for _, _, _, w in launches} == {0, 2}, launches
    assert {"Solved after a confirm step", "PrimalInfeasible"} <= chk.cov["statuses"], chk.cov["statuses"]
    assert chk.cov["rz"] == {"fresh", "updated"} and chk.cov["refined"] == {0, 1}
    assert set(range(15, 21)) <= chk.cov["nb"], chk.cov["nb"]   # paired work list at 15, segment packing from 16
    with capsys.disabled():
        print()
        chk.report()
