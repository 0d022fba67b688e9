"""ctypes binding over libbgg_b200.so (include/bgg.h) -- the product's Python entry point used by tests and bench.py.

There is no CPU fallback: if the shared library is missing, or no CUDA device is present, construction raises.
Nothing here imports or calls anything under oracle/.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbgg_b200.so")

NX, NX_MAN, NUM_EE = 12, 13, 4
MAX_CONTACTS = 12   # BGG_MAX_CONTACTS
MAX_KNOTS, MAX_NODES = 28, 64
STATUS_NAMES = ["Solved", "SolvedInacc", "MaxIter", "PrimalInfeasible", "DualInfeasible", "PrimalInfeasibleInacc",
                "DualInfeasibleInacc", "Unsolved", "Other"]

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


class BggError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [("num_nodes", C.c_int32), ("max_spline_vars", C.c_int32), ("device", C.c_int32), ("ipm_max_iter", C.c_int32),
                ("ipm_refine", C.c_int32), ("ipm_refine_after", C.c_int32), ("integrator_dt", C.c_double), ("friction_coef", C.c_double),
                ("force_bound", C.c_double), ("swing_height", C.c_double), ("foot_offset", C.c_double),
                ("ee_box_size", C.c_double * 2), ("force_cost", C.c_double), ("ipm_tol_feas", C.c_double),
                ("ipm_tol_gap", C.c_double), ("ipm_eq_delta", C.c_double), ("ipm_reg_eps", C.c_double), ("ipm_tol_infeas", C.c_double)]


class Robot(C.Structure):
    _fields_ = [("mass", C.c_double), ("Ir", C.c_double * 9), ("Ir_inv", C.c_double * 9), ("hip_xy", C.c_double * 8),
                ("gravity", C.c_double * 3)]


class Sizes(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n", "nu", "nf", "np", "n_samples", "n_eebox", "n_eq", "n_td", "m_ineq", "status",
                                         "iters", "ls_iters", "error")] + \
               [("nfv", C.c_int32 * 4), ("npv", C.c_int32 * 4), ("fbase", C.c_int32 * 4), ("pbase", C.c_int32 * 4)] + \
               [(n, C.c_double) for n in ("t0", "alpha", "cost", "prim_res", "dual_res", "gap", "eq_violation", "step_norm",
                                          "merit", "merit_dd")] + [("ee_box", C.c_double * 2), ("qp_cost", C.c_double),
                                                                     ("refined_iters", C.c_int32), ("no_iterate", C.c_int32)]


# numpy view of the POD bgg::Instance / bgg::FootSpline (csrc/bgg_types.cuh)
FOOT_DTYPE = np.dtype([("n", np.int32), ("ttype", np.uint8, MAX_KNOTS), ("ftype", np.uint8, MAX_KNOTS),
                       ("ptype", np.uint8, MAX_KNOTS), ("ztype", np.uint8, MAX_KNOTS), ("t", np.float64, MAX_KNOTS),
                       ("f", np.float64, (3, MAX_KNOTS, 2)), ("p", np.float64, (3, MAX_KNOTS, 2))], align=True)
INSTANCE_DTYPE = np.dtype([("states", np.float64, (MAX_NODES + 1, NX_MAN)), ("foot", FOOT_DTYPE, NUM_EE),
                           ("ee_box", np.float64, 2), ("init_time", np.float64), ("run_count", np.int32),
                           ("pad_", np.int32)], align=True)

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BggError(f"{LIB_PATH} is missing: build it with bilevel-gait-gen_b200/build.sh (no CPU fallback exists)")
        L = C.CDLL(LIB_PATH)
        L.bgg_last_error.restype = C.c_char_p
        L.bgg_measure_fp64_peak.argtypes = [C.c_int, _dp]
        L.bgg_create.argtypes = [C.POINTER(Config), C.POINTER(Robot), C.POINTER(C.c_void_p)]
        L.bgg_destroy.argtypes = [C.c_void_p]
        L.bgg_set_costs.argtypes = [C.c_void_p, _dp, _dp, _dp, _dp]
        L.bgg_batch_reset.argtypes = [C.c_void_p, C.c_int, _dp, C.c_int]
        L.bgg_set_warm_states.argtypes = [C.c_void_p, _dp, C.c_int]
        L.bgg_set_contact_times.argtypes = [C.c_void_p, C.c_int, C.c_int, _dp, C.c_int]
        L.bgg_solve_batch.argtypes = [C.c_void_p, _dp, _dp, _dp, _ip, _ip, _dp, _dp, _dp, C.c_int]
        L.bgg_qp_solve_batch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _ip, _ip, _dp, _ip, _ip, _dp, _dp, _dp, C.POINTER(C.c_uint8),
                                         _dp, _dp, _dp, _ip, _ip]
        L.bgg_qp_adjoint_batch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _ip, _ip, _dp, _ip, _ip, _dp, C.POINTER(C.c_uint8),
                                           _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _ip]
        L.bgg_controller_get_step.argtypes = [C.c_void_p, _dp, _dp, _dp]
        L.bgg_upload_inputs.argtypes = [C.c_void_p, _dp, _dp, _dp]
        L.bgg_solve_resident.argtypes = [C.c_void_p]
        L.bgg_download_results.argtypes = [C.c_void_p, _ip, _ip, _dp, _dp, _dp, C.c_int]
        L.bgg_synchronize.argtypes = [C.c_void_p]
        L.bgg_advance_plant.argtypes = [C.c_void_p, C.c_double]
        L.bgg_param_partials.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, _ip, _ip, _ip, _dp, _ip, _ip, _dp, _dp]
        L.bgg_set_kinematics.argtypes = [C.c_void_p, _dp]
        L.bgg_ik_batch.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp, _ip, _ip]
        L.bgg_targets_from_traj_batch.argtypes = [C.c_void_p, _dp, _dp, _dp, _dp, _ip]
        L.bgg_set_profiling.argtypes = [C.c_void_p, C.c_int]
        L.bgg_last_kernel_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.bgg_kernel_launch_count.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
        L.bgg_event_record.argtypes = [C.c_void_p, C.c_int]
        L.bgg_event_elapsed_ms.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float)]
        L.bgg_get_sizes.argtypes = [C.c_void_p, C.c_int, C.POINTER(Sizes)]
        L.bgg_get_dynamics.argtypes = [C.c_void_p, C.c_int, C.c_int, _dp, _dp, _dp, C.c_int]
        L.bgg_get_condensed.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp]
        L.bgg_export_qp_csc.argtypes = [C.c_void_p, C.c_int, C.c_int, _ip, _ip, _ip, _dp, C.c_int, _dp, _dp, _dp, C.c_int, C.c_int]
        L.bgg_gait_gradient_batch.argtypes = [C.c_void_p, _ip, _ip, _dp]
        L.bgg_optimize_contact_times_batch.argtypes = [C.c_void_p, _dp, C.c_double, C.c_double, _dp, _dp, _dp, _dp, _ip]
        L.bgg_line_search_batch.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp, _dp, _ip, _dp, _ip]
        L.bgg_get_adjoint.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp, _dp]
        L.bgg_get_contact_times.argtypes = [C.c_void_p, C.c_int, C.c_int, _dp, _ip, _ip]
        L.bgg_set_solution.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp, _dp]
        L.bgg_get_solution.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp, _dp]
        L.bgg_instance_bytes.restype = C.c_size_t
        L.bgg_get_instance.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.bgg_set_instance.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.bgg_get_states.argtypes = [C.c_void_p, C.c_int, _dp]
        L.bgg_eval_splines.argtypes = [C.c_void_p, C.c_int, _dp, C.c_int, _dp, _dp]
        _lib = L
    return _lib


def exported_symbols():
    """Names include/bgg.h declares; used by the CPU-side ABI test."""
    return ["bgg_last_error", "bgg_device_count", "bgg_measure_fp64_peak", "bgg_create", "bgg_destroy", "bgg_set_costs", "bgg_batch_reset",
            "bgg_set_warm_states", "bgg_set_contact_times", "bgg_solve_batch", "bgg_qp_solve_batch", "bgg_qp_adjoint_batch", "bgg_controller_tick_batch", "bgg_controller_get_step", "bgg_upload_inputs", "bgg_solve_resident",
            "bgg_download_results", "bgg_synchronize", "bgg_advance_plant", "bgg_param_partials", "bgg_set_kinematics", "bgg_ik_batch", "bgg_targets_from_traj_batch", "bgg_set_profiling", "bgg_last_kernel_ms", "bgg_kernel_launch_count", "bgg_event_record", "bgg_event_elapsed_ms",
            "bgg_get_sizes", "bgg_get_dynamics", "bgg_get_condensed", "bgg_export_qp_csc", "bgg_gait_gradient_batch", "bgg_optimize_contact_times_batch",
            "bgg_line_search_batch", "bgg_get_adjoint",
            "bgg_get_contact_times", "bgg_set_solution", "bgg_get_solution", "bgg_instance_bytes",
            "bgg_get_instance", "bgg_set_instance", "bgg_get_states", "bgg_eval_splines"]


def measure_fp64_peak(device=0):
    v = C.c_double(0.0)
    if lib().bgg_measure_fp64_peak(device, C.byref(v)):
        raise BggError(lib().bgg_last_error().decode())
    return v.value


def _d(a):
    return a.ctypes.data_as(_dp)


def _i(a):
    return a.ctypes.data_as(_ip)


class BatchedMPC:
    """A batch of independent mpc::MPCSingleRigidBody instances living on one B200.

    Method names follow the reference class (mpc/include/mpc.h, mpc_single_rigid_body.h); every array argument has a
    leading batch dimension.
    """

    def __init__(self, num_nodes, integrator_dt, robot, friction_coef=0.5, force_bound=150.0, swing_height=0.075,
                 foot_offset=0.015, ee_box_size=(0.15, 0.15), force_cost=0.0, device=0, max_spline_vars=0,
                 ipm_tol=0.0, ipm_max_iter=0, ipm_refine=0, ipm_tol_gap=0.0, ipm_refine_after=0):
        self.L = lib()
        self.N = num_nodes
        cfg = Config()
        cfg.num_nodes = num_nodes
        cfg.max_spline_vars = max_spline_vars
        self.max_nu = max_spline_vars if max_spline_vars > 0 else 160
        cfg.device = device
        cfg.ipm_max_iter = ipm_max_iter
        cfg.ipm_refine = ipm_refine
        cfg.ipm_refine_after = ipm_refine_after
        cfg.integrator_dt = integrator_dt
        cfg.friction_coef = friction_coef
        cfg.force_bound = force_bound
        cfg.swing_height = swing_height
        cfg.foot_offset = foot_offset
        cfg.ee_box_size[0], cfg.ee_box_size[1] = ee_box_size
        cfg.force_cost = force_cost
        cfg.ipm_tol_feas = ipm_tol
        cfg.ipm_tol_gap = ipm_tol_gap if ipm_tol_gap > 0 else ipm_tol
        cfg.ipm_eq_delta = 0.0
        rb = Robot()
        rb.mass = robot["mass"]
        rb.Ir[:] = np.asarray(robot["Ir"], float).ravel().tolist()
        rb.Ir_inv[:] = np.asarray(robot["Ir_inv"], float).ravel().tolist()
        rb.hip_xy[:] = np.asarray(robot["hip_offsets_xy"], float).ravel().tolist()
        rb.gravity[:] = list(robot["gravity"])
        self.h = C.c_void_p()
        self._chk(self.L.bgg_create(C.byref(cfg), C.byref(rb), C.byref(self.h)))
        self.B = 0

    def _chk(self, rc):
        if rc != 0:
            raise BggError(f"bgg error {rc}: {self.L.bgg_last_error().decode()}")

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.L.bgg_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # --- reference-named setters ---------------------------------------------------------------------------------
    def AddQuadraticTrackingCost(self, state_des_tangent, Q_diag, Phi_diag=None, Phi_w=None):
        q = np.ascontiguousarray(Q_diag, np.float64)
        d = np.ascontiguousarray(state_des_tangent, np.float64)
        phi = None if Phi_diag is None else np.ascontiguousarray(Phi_diag, np.float64)
        pw = None if Phi_w is None else np.ascontiguousarray(Phi_w, np.float64)
        self._chk(self.L.bgg_set_costs(self.h, _d(q), _d(d), None if phi is None else _d(phi), None if pw is None else _d(pw)))

    def Reset(self, batch, contact_times=None):
        self.B = batch
        if contact_times is None:
            self._chk(self.L.bgg_batch_reset(self.h, batch, None, 0))
        else:
            ct = np.ascontiguousarray(contact_times, np.float64)
            assert ct.shape[0] == NUM_EE
            self._chk(self.L.bgg_batch_reset(self.h, batch, _d(ct), ct.shape[1]))

    def SetStateTrajectoryWarmStart(self, states):
        s = np.ascontiguousarray(states, np.float64)
        if s.ndim == 2:
            assert s.shape == (self.B, NX_MAN)
            self._chk(self.L.bgg_set_warm_states(self.h, _d(s), 0))
        else:
            assert s.shape == (self.B, self.N + 1, NX_MAN)
            self._chk(self.L.bgg_set_warm_states(self.h, _d(s), 1))

    def UpdateContactTimes(self, times, first=0):
        t = np.ascontiguousarray(times, np.float64)
        assert t.ndim == 3 and t.shape[1] == NUM_EE
        self._chk(self.L.bgg_set_contact_times(self.h, first, t.shape[0], _d(t), t.shape[2]))

    # --- solves ---------------------------------------------------------------------------------------------------
    def GetRealTimeUpdate(self, state, init_time, ee_start_locations, z_out=None):
        """One RTI solve per instance. Returns dict(status, iters, alpha, cost) of numpy arrays [B]; with z_out (a float64
        array [B][z_stride]) also the decision vectors after the line-search update (MPC::GetQPSolution) in z_out."""
        s, t, e = self._inputs(state, init_time, ee_start_locations)
        st, it = np.zeros(self.B, np.int32), np.zeros(self.B, np.int32)
        al, co = np.zeros(self.B), np.zeros(self.B)
        zp, zs = (None, 0) if z_out is None else (_d(z_out), z_out.shape[1])
        self._chk(self.L.bgg_solve_batch(self.h, _d(s), _d(t), _d(e), _i(st), _i(it), _d(al), _d(co), zp, zs))
        out = dict(status=st, iters=it, alpha=al, cost=co)
        if z_out is not None:
            out["z"] = z_out
        return out

    Solve = GetRealTimeUpdate

    def CreateInitialRun(self, state, ee_start_locations, num_solves=10):
        out = None
        for _ in range(num_solves):   # mpc.cpp:78-90: ten solves at t = 0
            out = self.GetRealTimeUpdate(state, np.zeros(self.B), ee_start_locations)
        return out

    def _inputs(self, state, init_time, ee):
        s = np.ascontiguousarray(state, np.float64)
        t = np.ascontiguousarray(np.broadcast_to(np.asarray(init_time, np.float64), (self.B,)))
        e = np.ascontiguousarray(ee, np.float64)
        if s.shape != (self.B, NX_MAN) or e.shape != (self.B, NUM_EE, 3):
            raise BggError("state must be [B][13] and ee_start_locations [B][4][3]")
        return s, t, e

    def upload(self, state, init_time, ee):
        s, t, e = self._inputs(state, init_time, ee)
        self._chk(self.L.bgg_upload_inputs(self.h, _d(s), _d(t), _d(e)))

    def solve_resident(self):
        self._chk(self.L.bgg_solve_resident(self.h))

    @staticmethod
    def _qp_pattern(P, A, is_eq):
        """CSC pattern and stacked values of a batch of QPs (SolveQP / QPAdjoint): P, A scipy sparse matrices or lists of them."""
        import scipy.sparse as sp
        Ps = P if isinstance(P, (list, tuple)) else [P]
        As = A if isinstance(A, (list, tuple)) else [A]
        Ps = [sp.csc_matrix(p_, dtype=np.float64) for p_ in Ps]
        As = [sp.csc_matrix(a_, dtype=np.float64) for a_ in As]
        for m_ in Ps + As:
            m_.sort_indices()
        pc, pr = np.ascontiguousarray(Ps[0].indptr, np.int32), np.ascontiguousarray(Ps[0].indices, np.int32)
        ac, ar = np.ascontiguousarray(As[0].indptr, np.int32), np.ascontiguousarray(As[0].indices, np.int32)
        pv = np.ascontiguousarray(np.stack([p_.data for p_ in Ps]))
        av = np.ascontiguousarray(np.stack([a_.data for a_ in As]))
        eq = np.ascontiguousarray(np.asarray(is_eq, np.uint8))
        return len(Ps), Ps[0].shape[0], As[0].shape[0], pc, pr, pv, ac, ar, av, eq

    def SolveQP(self, P, q, A, b, is_eq):
        """QPInterface::SetupQP + Solve for a batch of QPs of one sparsity pattern (bgg_qp_solve_batch).  P, A: scipy sparse matrices
        (values of the first QP) or lists of them (one per QP, same pattern); q [count][n], b [count][m]; is_eq [m].
        Returns dict(x, y, s, status, iters)."""
        count, n, m, pc, pr, pv, ac, ar, av, eq = self._qp_pattern(P, A, is_eq)
        q = np.ascontiguousarray(np.asarray(q, np.float64).reshape(count, n))
        b = np.ascontiguousarray(np.asarray(b, np.float64).reshape(count, m))
        x, y, s = np.zeros((count, n)), np.zeros((count, m)), np.zeros((count, m))
        st, it = np.zeros(count, np.int32), np.zeros(count, np.int32)
        self._chk(self.L.bgg_qp_solve_batch(self.h, count, n, m, _i(pc), _i(pr), _d(pv), _i(ac), _i(ar), _d(av), _d(q), _d(b),
                                            eq.ctypes.data_as(C.POINTER(C.c_uint8)), _d(x), _d(y), _d(s), _i(st), _i(it)))
        return dict(x=x, y=y, s=s, status=st, iters=it)

    def QPAdjoint(self, P, A, is_eq, x, y, s, dx):
        """ClarabelInterface::SetupDerivativeCalcs + CalcDerivativeWrtVecs / WrtMats for a batch of QPs of one sparsity pattern
        (bgg_qp_adjoint_batch), at the points x [count][n], y / s [count][m] (normally what SolveQP returned) with loss gradient
        dx [count][n].  P, A, is_eq as in SolveQP.  Returns dict(dz, dy, db [count][m] in the caller's row order, dA [count][nnz(A)] in
        the order of A's sorted CSC data, status [count])."""
        count, n, m, pc, pr, pv, ac, ar, av, eq = self._qp_pattern(P, A, is_eq)
        x = np.ascontiguousarray(np.asarray(x, np.float64).reshape(count, n))
        y = np.ascontiguousarray(np.asarray(y, np.float64).reshape(count, m))
        s = np.ascontiguousarray(np.asarray(s, np.float64).reshape(count, m))
        dx = np.ascontiguousarray(np.asarray(dx, np.float64).reshape(count, n))
        dz, dy, db = np.zeros((count, n)), np.zeros((count, m)), np.zeros((count, m))
        dA, st = np.zeros((count, len(ar))), np.zeros(count, np.int32)
        self._chk(self.L.bgg_qp_adjoint_batch(self.h, count, n, m, _i(pc), _i(pr), _d(pv), _i(ac), _i(ar), _d(av),
                                              eq.ctypes.data_as(C.POINTER(C.c_uint8)), _d(x), _d(y), _d(s), _d(dx), _d(dz), _d(dy),
                                              _d(db), _d(dA), _i(st)))
        return dict(dz=dz, dy=dy, db=db, dA=dA, status=st)

    def download(self, z_out=None):
        st, it = np.zeros(self.B, np.int32), np.zeros(self.B, np.int32)
        al, co = np.zeros(self.B), np.zeros(self.B)
        zp, zs = (None, 0) if z_out is None else (_d(z_out), z_out.shape[1])
        self._chk(self.L.bgg_download_results(self.h, _i(st), _i(it), _d(al), _d(co), zp, zs))
        out = dict(status=st, iters=it, alpha=al, cost=co)
        if z_out is not None:
            out["z"] = z_out
        return out

    def ComputeParamPartialsClarabel(self, b, ee, contact_idx, cap=40000):
        """MPCSingleRigidBody::ComputeParamPartialsClarabel for one contact time of instance b: dense dA, dG and db in the reference's
        numbering, or None when the last solve is not Solved."""
        counts = np.zeros(4, np.int32)
        Ar, Ac, Av = np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap)
        Gr, Gc, Gv = np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap)
        sz = self.sizes(b)
        db = np.zeros(sz["n_eq"] + 12 * (self.N + 1))
        rc = self.L.bgg_param_partials(self.h, b, ee, contact_idx, cap, _i(counts), _i(Ar), _i(Ac), _d(Av), _i(Gr), _i(Gc), _d(Gv), _d(db))
        if rc == 1:
            return None
        self._chk(rc)
        n = sz["n"]
        dA, dG = np.zeros((counts[2], n)), np.zeros((counts[3], n))
        np.add.at(dA, (Ar[:counts[0]], Ac[:counts[0]]), Av[:counts[0]])
        np.add.at(dG, (Gr[:counts[1]], Gc[:counts[1]]), Gv[:counts[1]])
        return dict(dA=dA, dG=dG, db=db[:counts[2]], nnz=(int(counts[0]), int(counts[1])))

    # ---- joint-space targets (SURVEY 8f row 2)
    def SetKinematics(self, robot):
        """robot["legs"]: hip / thigh / calf joint placements + foot frame + joint axes per leg (tests/golden/a1_robot_consts.json)."""
        flat = []
        for leg in robot["legs"]:
            flat += np.asarray(leg["t"], float).ravel().tolist() + np.asarray(leg["R"], float).ravel().tolist() + np.asarray(leg["axis"], float).ravel().tolist()
        k = np.ascontiguousarray(flat, np.float64)
        assert k.size == 228
        self._chk(self.L.bgg_set_kinematics(self.h, _d(k)))

    def InverseKinematics(self, state, ee_des, joint_guess):
        """SingleRigidBodyModel::InverseKinematics for a stack of problems: state [n][13], ee_des [n][4][3], joint_guess [n][12]."""
        st = np.ascontiguousarray(state, np.float64).reshape(-1, 13)
        n = st.shape[0]
        ee = np.ascontiguousarray(ee_des, np.float64).reshape(n, 12)
        g = np.ascontiguousarray(joint_guess, np.float64).reshape(n, 12)
        q, status, iters = np.zeros((n, 19)), np.zeros(n, np.int32), np.zeros((n, 4), np.int32)
        self._chk(self.L.bgg_ik_batch(self.h, n, _d(st), _d(ee), _d(g), _d(q), _i(status), _i(iters)))
        return dict(q=q, status=status, iters=iters)

    def GetTargetsFromTraj(self, time, q_des):
        """MPCController::GetTargetsFromTraj for the whole batch: time scalar or [B], q_des [B][19] (running IK guess)."""
        t = np.ascontiguousarray(np.broadcast_to(np.asarray(time, np.float64), (self.B,)))
        q = np.ascontiguousarray(q_des, np.float64).reshape(self.B, 19).copy()
        v, f, status = np.zeros((self.B, 18)), np.zeros((self.B, 4, 3)), np.zeros(self.B, np.int32)
        self._chk(self.L.bgg_targets_from_traj_batch(self.h, _d(t), _d(q), _d(v), _d(f), _i(status)))
        return dict(q_des=q, v_des=v, force_des=f, status=status)

    def advance_plant(self, dt):
        self._chk(self.L.bgg_advance_plant(self.h, dt))

    def synchronize(self):
        self._chk(self.L.bgg_synchronize(self.h))

    def set_profiling(self, on):
        self._chk(self.L.bgg_set_profiling(self.h, int(on)))

    def last_kernel_ms(self):
        ms = (C.c_float * 4)()
        self._chk(self.L.bgg_last_kernel_ms(self.h, ms))
        return dict(zip(("prepare", "condense", "ipm", "finish"), (float(v) for v in ms)))

    def event_record(self, slot):
        self._chk(self.L.bgg_event_record(self.h, slot))

    def event_elapsed_ms(self, a, b):
        ms = C.c_float()
        self._chk(self.L.bgg_event_elapsed_ms(self.h, a, b, C.byref(ms)))
        return float(ms.value)

    def launch_count(self):
        v = C.c_int64()
        self._chk(self.L.bgg_kernel_launch_count(self.h, C.byref(v)))
        return v.value

    # --- accessors ------------------------------------------------------------------------------------------------
    def sizes(self, b=0):
        s = Sizes()
        self._chk(self.L.bgg_get_sizes(self.h, b, C.byref(s)))
        out = {}
        for name, _t in Sizes._fields_:
            v = getattr(s, name)
            out[name] = list(v) if hasattr(v, "__len__") else v
        return out

    def dynamics(self, first=0, count=1, nu=None):
        nu = nu or self.sizes(first)["nu"]
        Ad = np.zeros((count, self.N, 12, 12))
        Bd = np.zeros((count, self.N, 12, nu))
        cd = np.zeros((count, self.N, 12))
        self._chk(self.L.bgg_get_dynamics(self.h, first, count, _d(Ad), _d(Bd), _d(cd), nu))
        return Ad, Bd, cd

    def condensed(self, b=0):
        nu = self.sizes(b)["nu"]
        H, g = np.zeros((nu, nu)), np.zeros(nu)
        pp, xo = np.zeros((2 * (self.N - 3), nu)), np.zeros((self.N + 1, 12))
        self._chk(self.L.bgg_get_condensed(self.h, b, _d(H), _d(g), _d(pp), _d(xo)))
        return dict(H=H, g=g, phipos=pp, xoff=xo)

    def GetQPData(self, first=0, count=1, nnz_cap=25000):
        """The reference's QP (MPC::GetQPData) of the last solve for instances [first, first+count): a list of dicts with
        scipy csc A (reference sparsity), the diagonal of P, q, ub and the equality / inequality row counts.
        nnz_cap defaults to the reference's own reserve (mpc.cpp:47)."""
        import scipy.sparse as sp
        n_stride = 12 * (self.N + 1) + self.max_nu
        m_stride = 12 * (self.N + 1) + 6 * 160 + 2 * (self.N - 3) * 8 + 16
        dims = np.zeros((count, 6), np.int32)
        cp = np.zeros((count, n_stride + 1), np.int32)
        ri = np.zeros((count, nnz_cap), np.int32)
        va = np.zeros((count, nnz_cap))
        pd, q, ub = np.zeros((count, n_stride)), np.zeros((count, n_stride)), np.zeros((count, m_stride))
        self._chk(self.L.bgg_export_qp_csc(self.h, first, count, _i(dims), _i(cp), _i(ri), _d(va), nnz_cap, _d(pd), _d(q),
                                           _d(ub), n_stride, m_stride))
        out = []
        for k in range(count):
            n, m, nnz, neq, nin, err = (int(v) for v in dims[k])
            if err:
                raise BggError(f"instance {first + k}: export error bits {err}")
            A = sp.csc_matrix((va[k, :nnz].copy(), ri[k, :nnz].copy(), cp[k, :n + 1].copy()), shape=(m, n))
            out.append(dict(A=A, P_diag=pd[k, :n].copy(), q=q[k, :n].copy(), ub=ub[k, :m].copy(), num_eq=neq, num_ineq=nin))
        return out

    # --- gait optimiser -------------------------------------------------------------------------------------------
    def ComputeCostFcnDerivWrtContactTimes(self):
        """MPCController::GaitOpt's derivative chain for the whole batch: returns dict(status [B], n_contacts [B][4],
        dHdtheta: list of per-instance arrays over all contact times, foot-major)."""
        B = self.B
        status, nct = np.zeros(B, np.int32), np.zeros((B, NUM_EE), np.int32)
        dh = np.zeros((B, NUM_EE, MAX_CONTACTS))
        self._chk(self.L.bgg_gait_gradient_batch(self.h, _i(status), _i(nct), _d(dh)))
        grads = [np.concatenate([dh[b, e, :nct[b, e]] for e in range(NUM_EE)]) for b in range(B)]
        return dict(status=status, n_contacts=nct, dHdtheta=grads, raw=dh)

    def OptimizeContactTimes(self, time, dHdtheta=None, trust=1.0, alpha=1.0):
        """GaitOptimizer::OptimizeContactTimes for the whole batch.  dHdtheta: [B][4][MAX_CONTACTS] or None (use the last
        gradient).  Returns dict(step, xk, new_times: [B][4][MAX_CONTACTS]; status [B][4])."""
        B = self.B
        t = np.ascontiguousarray(np.broadcast_to(np.asarray(time, np.float64), (B,)))
        step, xk, nt = (np.zeros((B, NUM_EE, MAX_CONTACTS)) for _ in range(3))
        st = np.zeros((B, NUM_EE), np.int32)
        g = None if dHdtheta is None else np.ascontiguousarray(dHdtheta, np.float64)
        self._chk(self.L.bgg_optimize_contact_times_batch(self.h, _d(t), trust, alpha, None if g is None else _d(g), _d(step), _d(xk),
                                                          _d(nt), _i(st)))
        return dict(step=step, xk=xk, new_times=nt, status=st)

    def LineSearch(self, state, time, ee_start_locations, xk, step, K=10):
        """GaitOptimizer::LineSearch for the whole batch (K = LS_SIZE copies per instance, all solved as one batch)."""
        s, t, e = self._inputs(state, time, ee_start_locations)
        B = self.B
        best, costs, q = np.zeros(B, np.int32), np.zeros((B, K)), np.zeros((B, K), np.int32)
        xk = np.ascontiguousarray(xk, np.float64)
        step = np.ascontiguousarray(step, np.float64)
        self._chk(self.L.bgg_line_search_batch(self.h, K, _d(xk), _d(step), _d(s), _d(t), _d(e), _i(best), _d(costs), _i(q)))
        return dict(best=best, costs=costs, quality=q)

    def adjoint(self, b=0):
        sz = self.sizes(b)
        dz, dlam = np.zeros(sz["n"]), np.zeros(sz["m_ineq"])
        dnu, nu, dnue = np.zeros(12 * (self.N + 1)), np.zeros(12 * (self.N + 1)), np.zeros(sz["n_eq"])
        self._chk(self.L.bgg_get_adjoint(self.h, b, _d(dz), _d(dlam), _d(dnu), _d(dnue), _d(nu)))
        return dict(dz=dz, dlam=dlam, dnu_dyn=dnu, dnu_eq=dnue, nu_dyn=nu, sizes=sz)

    def controller_step(self):
        """The contact-time step of the last GAIT_OPT controller tick (bgg_controller_get_step): dict(step, xk, new_times)."""
        step, xk, nt = (np.zeros((self.B, NUM_EE, MAX_CONTACTS)) for _ in range(3))
        self._chk(self.L.bgg_controller_get_step(self.h, _d(step), _d(xk), _d(nt)))
        return dict(step=step, xk=xk, new_times=nt)

    def GetContactTimes(self, first=0, count=None):
        count = self.B - first if count is None else count
        t = np.zeros((count, NUM_EE, MAX_CONTACTS))
        ty, n = np.zeros((count, NUM_EE, MAX_CONTACTS), np.int32), np.zeros((count, NUM_EE), np.int32)
        self._chk(self.L.bgg_get_contact_times(self.h, first, count, _d(t), _i(ty), _i(n)))
        return t, ty, n

    def solution(self, b=0):
        sz = self.sizes(b)
        qp, z = np.zeros(sz["n"]), np.zeros(sz["n"])
        lam, sl, nu = np.zeros(sz["m_ineq"]), np.zeros(sz["m_ineq"]), np.zeros(sz["n_eq"])
        self._chk(self.L.bgg_get_solution(self.h, b, _d(qp), _d(z), _d(lam), _d(sl), _d(nu)))
        return dict(qp_sol=qp, z=z, lam=lam, slack=sl, nu_eq=nu, sizes=sz)

    def set_solution(self, b, qp_sol=None, z=None, lam=None, slack=None, nu_eq=None):
        arrs = [None if a is None else np.ascontiguousarray(a, np.float64) for a in (qp_sol, z, lam, slack, nu_eq)]
        self._chk(self.L.bgg_set_solution(self.h, b, *[None if a is None else _d(a) for a in arrs]))

    def get_instance(self, b=0):
        assert self.L.bgg_instance_bytes() == INSTANCE_DTYPE.itemsize, (self.L.bgg_instance_bytes(), INSTANCE_DTYPE.itemsize)
        buf = np.zeros(1, dtype=INSTANCE_DTYPE)
        self._chk(self.L.bgg_get_instance(self.h, b, buf.ctypes.data_as(C.c_void_p)))
        return buf[0]

    def set_instance(self, b, inst):
        buf = np.zeros(1, dtype=INSTANCE_DTYPE)
        buf[0] = inst
        self._chk(self.L.bgg_set_instance(self.h, b, buf.ctypes.data_as(C.c_void_p)))

    def GetStates(self, b=0):
        s = np.zeros((self.N + 1, NX_MAN))
        self._chk(self.L.bgg_get_states(self.h, b, _d(s)))
        return s

    def eval_splines(self, b, times):
        t = np.ascontiguousarray(times, np.float64)
        f, p = np.zeros((len(t), NUM_EE, 3)), np.zeros((len(t), NUM_EE, 3))
        self._chk(self.L.bgg_eval_splines(self.h, b, _d(t), len(t), _d(f), _d(p)))
        return f, p
