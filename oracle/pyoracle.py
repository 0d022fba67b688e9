"""TEST INFRASTRUCTURE ONLY -- ctypes bindings over the CPU oracle (oracle/liboracle.so) and, when it has been built,
over the reference's own spline sources compiled here (oracle/_ref/libref_splines.so).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(_HERE, "liboracle.so")
REF_SPLINES_SO = os.path.join(_HERE, "_ref", "libref_splines.so")
REF_MPC_SO = os.path.join(_HERE, "_ref", "libref_mpc.so")   # the reference's own MPC sources over stand-in headers (ref_shim/)
# a checkout of the reference project (bilevel-gait-gen); optional, it is not part of this repository
REF_DIR = os.environ.get("BGG_REFERENCE_DIR", "")

FORCE, POSITION = 0, 1
NO_DERIV, FULL_DERIV, EMPTY = 0, 1, 2
LIFT_OFF, TOUCH_DOWN, INTER = 0, 1, 2

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


def build(force=False):
    """Compile the oracle (and oracle/_ref when BGG_REFERENCE_DIR names the reference's sources). Building the checker is not using it."""
    if force or not os.path.exists(ORACLE_SO):
        subprocess.check_call(["make", "-C", _HERE, "liboracle.so"], stdout=subprocess.DEVNULL)
    if REF_DIR and os.path.isdir(os.path.join(REF_DIR, "mpc", "spline")) and (force or not os.path.exists(REF_SPLINES_SO) or not os.path.exists(REF_MPC_SO)):
        subprocess.check_call(["make", "-C", _HERE, "ref", "REF=" + os.path.abspath(REF_DIR)], stdout=subprocess.DEVNULL)


def _dptr(a):
    return a.ctypes.data_as(_dp)


def _iptr(a):
    return a.ctypes.data_as(_ip)


class OracleError(RuntimeError):
    pass


def _bind_spline_api(lib):
    lib.orc_last_error.restype = C.c_char_p
    lib.orc_spline_create.restype = C.c_void_p
    lib.orc_spline_create.argtypes = [C.c_int, _dp, C.c_int, C.c_int]
    lib.orc_spline_destroy.argtypes = [C.c_void_p]
    lib.orc_spline_clone.restype = C.c_void_p
    lib.orc_spline_clone.argtypes = [C.c_void_p]
    lib.orc_spline_value.restype = C.c_double
    lib.orc_spline_value.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double]
    lib.orc_spline_lin.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, _dp]
    lib.orc_spline_vars_idx.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, _ip, _ip]
    lib.orc_spline_is_force_mutable.argtypes = [C.c_void_p, C.c_double]
    lib.orc_spline_is_in_contact.argtypes = [C.c_void_p, C.c_double]
    lib.orc_spline_add_poly.argtypes = [C.c_void_p, C.c_double]
    lib.orc_spline_remove_poly.argtypes = [C.c_void_p, C.c_double]
    lib.orc_spline_partial.restype = C.c_double
    lib.orc_spline_partial.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int]
    lib.orc_spline_coef_partial.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_double, _dp]
    lib.orc_spline_set_vars.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double]
    lib.orc_spline_set_contact_times.argtypes = [C.c_void_p, _dp, C.c_int]
    lib.orc_spline_num_nodes.argtypes = [C.c_void_p]
    lib.orc_spline_num_contacts.argtypes = [C.c_void_p]
    lib.orc_spline_node_type.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    lib.orc_spline_mutable_nodes.argtypes = [C.c_void_p, C.c_int, C.c_int, _ip]
    lib.orc_spline_times.argtypes = [C.c_void_p, _dp, _ip]
    lib.orc_spline_as_qp_vec.argtypes = [C.c_void_p, C.c_int, C.c_int, _dp]
    lib.orc_spline_total_poly_vars.argtypes = [C.c_void_p, C.c_int, C.c_int]
    for f in ("orc_spline_end_time", "orc_spline_start_time"):
        getattr(lib, f).restype = C.c_double
        getattr(lib, f).argtypes = [C.c_void_p]
    for f in ("orc_spline_next_td", "orc_spline_swing_time"):
        getattr(lib, f).restype = C.c_double
        getattr(lib, f).argtypes = [C.c_void_p, C.c_double]
    lib.orc_spline_set_to_touchdown.argtypes = [C.c_void_p, C.c_double]
    if hasattr(lib, "orc_spline_knots"):
        lib.orc_spline_knots.argtypes = [C.c_void_p, C.c_int, C.c_int, _ip, _dp]
    return lib


_libs = {}


def load(which="oracle"):
    """which: 'oracle' (the restatement) or 'ref' (the reference's own spline sources compiled here)."""
    if which not in _libs:
        path = ORACLE_SO if which == "oracle" else REF_SPLINES_SO
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        _libs[which] = _bind_spline_api(C.CDLL(path))
        if which == "oracle":
            _bind_mpc_api(_libs[which])
    return _libs[which]


def have_ref():
    return os.path.exists(REF_SPLINES_SO)


def have_ref_mpc():
    return os.path.exists(REF_MPC_SO)


_ref_mpc_lib = None


def load_ref_mpc():
    """The reference's own MPC sources compiled here (oracle/Makefile: _ref/libref_mpc.so); same entry-point names as the oracle."""
    global _ref_mpc_lib
    if _ref_mpc_lib is None:
        lib = C.CDLL(REF_MPC_SO, mode=os.RTLD_NOW)
        lib.orc_mpc_last_error.restype = C.c_char_p
        lib.orc_last_error = lib.orc_mpc_last_error
        lib.orc_mpc_create_ref.restype = C.c_void_p
        lib.orc_mpc_create_ref.argtypes = [C.POINTER(_MpcInfo), C.POINTER(_RobotConsts), _dp]
        lib.orc_mpc_destroy.argtypes = [C.c_void_p]
        lib.orc_mpc_set_ipm.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_int, C.c_int]
        lib.orc_mpc_set_costs.argtypes = [C.c_void_p, _dp, _dp, _dp, _dp]
        lib.orc_mpc_set_warm_states.argtypes = [C.c_void_p, _dp]
        lib.orc_mpc_solve.argtypes = [C.c_void_p, _dp, C.c_double, _dp, C.c_int]
        lib.orc_mpc_initial_run.argtypes = [C.c_void_p, _dp, _dp]
        lib.orc_mpc_set_contact_times.argtypes = [C.c_void_p, C.c_int, _dp, C.c_int]
        lib.orc_mpc_sizes.argtypes = [C.c_void_p, _ip]
        lib.orc_mpc_get_A.argtypes = [C.c_void_p, _ip, _ip, _dp]
        lib.orc_mpc_get_P.argtypes = [C.c_void_p, _ip, _ip, _dp]
        lib.orc_mpc_get_vectors.argtypes = [C.c_void_p, _dp, _dp, C.c_char_p]
        lib.orc_mpc_get_prev_qp_sol.argtypes = [C.c_void_p, _dp]
        lib.orc_mpc_get_qp_solution.argtypes = [C.c_void_p, _dp, _dp, _dp, _dp]
        lib.orc_mpc_get_stats.argtypes = [C.c_void_p, _dp]
        lib.orc_mpc_get_states.argtypes = [C.c_void_p, _dp]
        lib.orc_mpc_init_time.restype = C.c_double
        lib.orc_mpc_init_time.argtypes = [C.c_void_p]
        lib.orc_mpc_cost.restype = C.c_double
        lib.orc_mpc_cost.argtypes = [C.c_void_p]
        lib.orc_mpc_force_at.argtypes = [C.c_void_p, C.c_int, C.c_double, _dp]
        lib.orc_mpc_ee_at.argtypes = [C.c_void_p, C.c_int, C.c_double, _dp]
        lib.orc_mpc_num_contacts.argtypes = [C.c_void_p, C.c_int]
        lib.orc_mpc_get_contact_times.argtypes = [C.c_void_p, C.c_int, _dp, _ip]
        lib.orc_mpc_gait_gradient.argtypes = [C.c_void_p, _dp, C.c_int]
        _ref_mpc_lib = lib
    return _ref_mpc_lib


class FootSpline:
    """One foot's contact splines (mpc::EndEffectorSplines). `which` selects restatement or compiled reference."""

    def __init__(self, times, start_in_contact, num_force_polys=3, which="oracle", _handle=None, _owned=True):
        self.lib = load(which)
        self.which = which
        self._owned = _owned
        if _handle is not None:
            self.h = _handle
            return
        t = np.ascontiguousarray(times, dtype=np.float64)
        self.h = self.lib.orc_spline_create(len(t), _dptr(t), int(start_in_contact), num_force_polys)
        if not self.h:
            raise OracleError(self.lib.orc_last_error().decode())

    def __del__(self):
        if getattr(self, "h", None) and self._owned:
            self.lib.orc_spline_destroy(self.h)
            self.h = None

    def clone(self):
        return FootSpline(None, None, which=self.which, _handle=self.lib.orc_spline_clone(self.h))

    def _chk(self, rc):
        if rc < 0:
            raise OracleError(self.lib.orc_last_error().decode())
        return rc

    def value(self, typ, coord, t):
        v = self.lib.orc_spline_value(self.h, typ, coord, t)
        if np.isnan(v):
            raise OracleError(self.lib.orc_last_error().decode())
        return v

    def lin(self, typ, coord, t):
        out = np.zeros(8)
        n = self._chk(self.lib.orc_spline_lin(self.h, typ, coord, t, _dptr(out)))
        return out[:n].copy()

    def vars_idx(self, typ, coord, t):
        i, c = C.c_int(), C.c_int()
        self._chk(self.lib.orc_spline_vars_idx(self.h, typ, coord, t, C.byref(i), C.byref(c)))
        return i.value, c.value

    def is_force_mutable(self, t):
        return bool(self._chk(self.lib.orc_spline_is_force_mutable(self.h, t)))

    def is_in_contact(self, t):
        return bool(self._chk(self.lib.orc_spline_is_in_contact(self.h, t)))

    def add_poly(self, dt):
        self._chk(self.lib.orc_spline_add_poly(self.h, dt))

    def remove_poly(self, t):
        self._chk(self.lib.orc_spline_remove_poly(self.h, t))

    def partial(self, typ, coord, t, time_idx):
        v = self.lib.orc_spline_partial(self.h, typ, coord, t, time_idx)
        if np.isnan(v):
            raise OracleError(self.lib.orc_last_error().decode())
        return v

    def coef_partial(self, typ, coord, t, time_idx, dtwdth=0.0):
        out = np.zeros(8)
        n = self._chk(self.lib.orc_spline_coef_partial(self.h, typ, coord, t, time_idx, dtwdth, _dptr(out)))
        return out[:n].copy()

    def set_vars(self, typ, coord, node, v0, v1):
        self._chk(self.lib.orc_spline_set_vars(self.h, typ, coord, node, v0, v1))

    def set_contact_times(self, times):
        t = np.ascontiguousarray(times, dtype=np.float64)
        self._chk(self.lib.orc_spline_set_contact_times(self.h, _dptr(t), len(t)))

    def num_nodes(self):
        return self.lib.orc_spline_num_nodes(self.h)

    def num_contacts(self):
        return self.lib.orc_spline_num_contacts(self.h)

    def node_type(self, typ, coord, node):
        return self._chk(self.lib.orc_spline_node_type(self.h, typ, coord, node))

    def mutable_nodes(self, typ, coord):
        out = np.zeros(64, dtype=np.int32)
        n = self._chk(self.lib.orc_spline_mutable_nodes(self.h, typ, coord, _iptr(out)))
        return [int(v) for v in out[:n]]

    def times(self):
        out = np.zeros(64)
        n = self.lib.orc_spline_times(self.h, _dptr(out), None)
        return out[:n].copy()

    def time_types(self):
        out = np.zeros(64)
        ty = np.zeros(64, dtype=np.int32)
        n = self.lib.orc_spline_times(self.h, _dptr(out), _iptr(ty))
        return ty[:n].copy()

    def knots(self, typ, coord):
        ty = np.zeros(64, dtype=np.int32)
        va = np.zeros((64, 2))
        n = self.lib.orc_spline_knots(self.h, typ, coord, _iptr(ty), _dptr(va))
        return ty[:n].copy(), va[:n].copy()

    def as_qp_vec(self, typ, coord):
        out = np.zeros(128)
        n = self._chk(self.lib.orc_spline_as_qp_vec(self.h, typ, coord, _dptr(out)))
        return out[:n].copy()

    def total_poly_vars(self, typ, coord):
        return self.lib.orc_spline_total_poly_vars(self.h, typ, coord)

    def end_time(self):
        return self.lib.orc_spline_end_time(self.h)

    def start_time(self):
        return self.lib.orc_spline_start_time(self.h)

    def next_td(self, t):
        return self.lib.orc_spline_next_td(self.h, t)

    def swing_time(self, t):
        return self.lib.orc_spline_swing_time(self.h, t)

    def set_to_touchdown(self, t):
        self._chk(self.lib.orc_spline_set_to_touchdown(self.h, t))


# ----------------------------------------------------------------------------------------------- ADMM + MPC
class AdmmSettings(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("rho", "sigma", "alpha", "eps_abs", "eps_rel", "eps_prim_inf", "eps_dual_inf",
                                           "adaptive_rho_tolerance")] + \
               [(n, C.c_int) for n in ("max_iter", "scaling", "check_termination", "adaptive_rho", "adaptive_rho_interval")]


class _MpcInfo(C.Structure):
    _fields_ = [("num_nodes", C.c_int)] + [(n, C.c_double) for n in (
        "friction_coef", "integrator_dt", "force_bound", "swing_height", "foot_offset", "ee_box_x", "ee_box_y", "force_cost")]


class _RobotConsts(C.Structure):
    _fields_ = [("mass", C.c_double), ("Ir", C.c_double * 9), ("Ir_inv", C.c_double * 9), ("hip_xy", C.c_double * 8),
                ("gravity", C.c_double * 3)]


def _bind_mpc_api(lib):
    lib.orc_admm_default_settings.argtypes = [C.POINTER(AdmmSettings)]
    lib.orc_admm_solve.argtypes = [C.c_int, C.c_int, _ip, _ip, _dp, _dp, _ip, _ip, _dp, _dp, _dp, _dp, _dp,
                                   C.POINTER(AdmmSettings), _dp, _dp, _dp, _dp]
    lib.orc_mpc_create.restype = C.c_void_p
    lib.orc_mpc_create.argtypes = [C.POINTER(_MpcInfo), C.POINTER(_RobotConsts)]
    lib.orc_mpc_destroy.argtypes = [C.c_void_p]
    lib.orc_mpc_clone.restype = C.c_void_p
    lib.orc_mpc_clone.argtypes = [C.c_void_p]
    lib.orc_mpc_select_solver.argtypes = [C.c_void_p, C.c_int]
    lib.orc_mpc_set_ipm.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_int, C.c_int]
    lib.orc_ipm_solve.argtypes = [C.c_int, C.c_int, _ip, _ip, _dp, _dp, _ip, _ip, _dp, _dp, C.c_char_p, C.c_double, C.c_int,
                                  _dp, _dp, _dp, _dp]
    lib.orc_mpc_set_admm.argtypes = [C.c_void_p, C.POINTER(AdmmSettings), C.POINTER(AdmmSettings)]
    lib.orc_mpc_get_admm.argtypes = [C.c_void_p, C.POINTER(AdmmSettings), C.POINTER(AdmmSettings)]
    lib.orc_mpc_set_costs.argtypes = [C.c_void_p, _dp, _dp, _dp, _dp]
    lib.orc_mpc_set_warm_states.argtypes = [C.c_void_p, _dp]
    lib.orc_mpc_assemble.argtypes = [C.c_void_p, _dp, C.c_double, _dp]
    lib.orc_mpc_solve.argtypes = [C.c_void_p, _dp, C.c_double, _dp, C.c_int]
    lib.orc_mpc_initial_run.argtypes = [C.c_void_p, _dp, _dp]
    lib.orc_mpc_set_contact_times.argtypes = [C.c_void_p, C.c_int, _dp, C.c_int]
    lib.orc_mpc_sizes.argtypes = [C.c_void_p, _ip]
    lib.orc_mpc_get_A.argtypes = [C.c_void_p, _ip, _ip, _dp]
    lib.orc_mpc_get_P.argtypes = [C.c_void_p, _ip, _ip, _dp]
    lib.orc_mpc_get_vectors.argtypes = [C.c_void_p, _dp, _dp, C.c_char_p]
    lib.orc_mpc_get_prev_qp_sol.argtypes = [C.c_void_p, _dp]
    lib.orc_mpc_get_qp_solution.argtypes = [C.c_void_p, _dp, _dp, _dp, _dp]
    lib.orc_mpc_get_stats.argtypes = [C.c_void_p, _dp]
    lib.orc_mpc_get_node_dynamics.argtypes = [C.c_void_p, _dp, _dp, _dp]
    lib.orc_mpc_get_states.argtypes = [C.c_void_p, _dp]
    lib.orc_mpc_set_state.argtypes = [C.c_void_p, C.c_int, _dp]
    lib.orc_mpc_foot.restype = C.c_void_p
    lib.orc_mpc_foot.argtypes = [C.c_void_p, C.c_int]
    lib.orc_mpc_init_time.restype = C.c_double
    lib.orc_mpc_init_time.argtypes = [C.c_void_p]
    lib.orc_mpc_cost.restype = C.c_double
    lib.orc_mpc_cost.argtypes = [C.c_void_p]
    lib.orc_mpc_force_at.argtypes = [C.c_void_p, C.c_int, C.c_double, _dp]
    lib.orc_mpc_ee_at.argtypes = [C.c_void_p, C.c_int, C.c_double, _dp]
    lib.orc_mpc_merit.restype = C.c_double
    lib.orc_mpc_merit.argtypes = [C.c_void_p, _dp]
    lib.orc_quat_log3.argtypes = [_dp, _dp]
    lib.orc_quat_exp3.argtypes = [_dp, _dp]


def default_admm_settings():
    s = AdmmSettings()
    load().orc_admm_default_settings(C.byref(s))
    return s


def admm_solve(P, q, A, l, u, x0=None, y0=None, settings=None):
    """OSQP-restatement solve of min 1/2 x'Px+q'x, l<=Ax<=u. P, A: scipy.sparse (any format)."""
    import scipy.sparse as sp
    lib = load()
    P = sp.csc_matrix(P, dtype=np.float64)
    A = sp.csc_matrix(A, dtype=np.float64)
    P.sort_indices()
    A.sort_indices()
    n, m = P.shape[0], A.shape[0]
    q = np.ascontiguousarray(q, dtype=np.float64)
    l = np.ascontiguousarray(l, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    x0 = np.zeros(n) if x0 is None else np.ascontiguousarray(x0, dtype=np.float64)
    y0 = np.zeros(m) if y0 is None else np.ascontiguousarray(y0, dtype=np.float64)
    s = settings or default_admm_settings()
    x, y, z, info = np.zeros(n), np.zeros(m), np.zeros(m), np.zeros(5)
    pc, pr = P.indptr.astype(np.int32), P.indices.astype(np.int32)
    ac, ar = A.indptr.astype(np.int32), A.indices.astype(np.int32)
    pv, av = np.ascontiguousarray(P.data), np.ascontiguousarray(A.data)
    st = lib.orc_admm_solve(n, m, _iptr(pc), _iptr(pr), _dptr(pv), _dptr(q), _iptr(ac), _iptr(ar), _dptr(av), _dptr(l),
                            _dptr(u), _dptr(x0), _dptr(y0), C.byref(s), _dptr(x), _dptr(y), _dptr(z), _dptr(info))
    if st < 0:
        raise OracleError(lib.orc_last_error().decode())
    return dict(x=x, y=y, z=z, status=st, iters=int(info[0]), prim_res=info[1], dual_res=info[2], rho=info[3],
                rho_updates=int(info[4]))


def ipm_solve(P, q, A, b, is_eq, tol=0.0, max_iter=0):
    """Interior-point solve of min 1/2 x'Px+q'x, Ax + s = b, s = 0 on is_eq rows and s >= 0 elsewhere."""
    import scipy.sparse as sp
    lib = load()
    P = sp.csc_matrix(P, dtype=np.float64)
    A = sp.csc_matrix(A, dtype=np.float64)
    P.sort_indices()
    A.sort_indices()
    n, m = P.shape[0], A.shape[0]
    q = np.ascontiguousarray(q, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    eq = np.ascontiguousarray(is_eq, dtype=np.uint8).tobytes()
    x, y, s, info = np.zeros(n), np.zeros(m), np.zeros(m), np.zeros(4)
    pc, pr = P.indptr.astype(np.int32), P.indices.astype(np.int32)
    ac, ar = A.indptr.astype(np.int32), A.indices.astype(np.int32)
    pv, av = np.ascontiguousarray(P.data), np.ascontiguousarray(A.data)
    st = lib.orc_ipm_solve(n, m, _iptr(pc), _iptr(pr), _dptr(pv), _dptr(q), _iptr(ac), _iptr(ar), _dptr(av), _dptr(b), eq,
                           tol, max_iter, _dptr(x), _dptr(y), _dptr(s), _dptr(info))
    if st < 0:
        raise OracleError(lib.orc_last_error().decode())
    return dict(x=x, y=y, s=s, status=st, iters=int(info[0]), prim_res=info[1], dual_res=info[2], gap=info[3])


def load_robot_consts(path):
    import json
    with open(path) as f:
        d = json.load(f)
    return d


class SrbMpc:
    """The oracle's restatement of mpc::MPCSingleRigidBody (live path)."""

    def __init__(self, num_nodes, dt, consts, friction_coef=0.5, force_bound=150.0, swing_height=0.075, foot_offset=0.015,
                 ee_box_size=(0.15, 0.15), force_cost=0.0, _handle=None, which="oracle"):
        """which = "oracle": the restatement (liboracle.so); "ref": the reference's own sources compiled here (libref_mpc.so)."""
        self.which = which
        self.lib = load() if which == "oracle" else load_ref_mpc()
        self.N = num_nodes
        if _handle is not None:
            self.h = _handle
            return
        info = _MpcInfo(num_nodes, friction_coef, dt, force_bound, swing_height, foot_offset, ee_box_size[0], ee_box_size[1], force_cost)
        rc = _RobotConsts()
        rc.mass = consts["mass"]
        rc.Ir[:] = np.asarray(consts["Ir"], dtype=float).ravel().tolist()
        rc.Ir_inv[:] = np.asarray(consts["Ir_inv"], dtype=float).ravel().tolist()
        rc.hip_xy[:] = np.asarray(consts["hip_offsets_xy"], dtype=float).ravel().tolist()
        rc.gravity[:] = list(consts["gravity"])
        if which == "ref":
            # the reference adds its +-0.1 (y) and +0.025 (x) offsets to the raw hip-joint translation itself
            # (single_rigid_body_model.cpp:289-305): hand it the translations of models/a1_description/urdf/a1.urdf
            hip = np.ascontiguousarray(np.asarray(consts["hip_joint_translation"], dtype=float))
            self.h = self.lib.orc_mpc_create_ref(C.byref(info), C.byref(rc), _dptr(hip))
        else:
            self.h = self.lib.orc_mpc_create(C.byref(info), C.byref(rc))
        if not self.h:
            raise OracleError(self.lib.orc_last_error().decode())

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.orc_mpc_destroy(self.h)
            self.h = None

    def clone(self):
        return SrbMpc(self.N, 0, None, _handle=self.lib.orc_mpc_clone(self.h))

    def _chk(self, rc):
        if rc < 0:
            raise OracleError(self.lib.orc_last_error().decode())
        return rc

    def select_solver(self, which):
        """'ipm' (default; the reference's live Clarabel path) or 'admm' (its test-only OSQP path)."""
        self.lib.orc_mpc_select_solver(self.h, 1 if which == "admm" else 0)

    def set_ipm(self, tol_feas=0.0, tol_gap=0.0, max_iter=0, refine=-1):
        self.lib.orc_mpc_set_ipm(self.h, tol_feas, tol_gap, max_iter, refine)

    def set_admm(self, initial=None, real_time=None):
        self.lib.orc_mpc_set_admm(self.h, C.byref(initial) if initial is not None else None,
                                  C.byref(real_time) if real_time is not None else None)

    def get_admm(self):
        a, b = AdmmSettings(), AdmmSettings()
        self.lib.orc_mpc_get_admm(self.h, C.byref(a), C.byref(b))
        return a, b

    def set_costs(self, state_des_tan, Q, Phi=None, Phi_w=None):
        Q = np.ascontiguousarray(Q, dtype=np.float64)
        if Q.ndim == 1:
            Q = np.diag(Q)
        Q = np.ascontiguousarray(Q)
        d = np.ascontiguousarray(state_des_tan, dtype=np.float64)
        Phi = Q if Phi is None else np.ascontiguousarray(Phi, dtype=np.float64)
        Phi_w = (-Q @ d) if Phi_w is None else np.ascontiguousarray(Phi_w, dtype=np.float64)
        Phi_w = np.ascontiguousarray(Phi_w)
        self.lib.orc_mpc_set_costs(self.h, _dptr(d), _dptr(Q), _dptr(Phi), _dptr(Phi_w))

    def set_warm_states(self, states):
        s = np.ascontiguousarray(states, dtype=np.float64)
        assert s.shape == (self.N + 1, 13)
        self.lib.orc_mpc_set_warm_states(self.h, _dptr(s))

    def assemble(self, state, t0, ee_start):
        s = np.ascontiguousarray(state, dtype=np.float64)
        e = np.ascontiguousarray(ee_start, dtype=np.float64)
        self._chk(self.lib.orc_mpc_assemble(self.h, _dptr(s), t0, _dptr(e)))

    def solve(self, state, t0, ee_start, real_time=True):
        s = np.ascontiguousarray(state, dtype=np.float64)
        e = np.ascontiguousarray(ee_start, dtype=np.float64)
        return self._chk(self.lib.orc_mpc_solve(self.h, _dptr(s), t0, _dptr(e), int(real_time)))

    def initial_run(self, state, ee_start):
        s = np.ascontiguousarray(state, dtype=np.float64)
        e = np.ascontiguousarray(ee_start, dtype=np.float64)
        return self._chk(self.lib.orc_mpc_initial_run(self.h, _dptr(s), _dptr(e)))

    def set_contact_times(self, ee, times):
        t = np.ascontiguousarray(times, dtype=np.float64)
        self._chk(self.lib.orc_mpc_set_contact_times(self.h, ee, _dptr(t), len(t)))

    def gait_gradient(self):
        """(which="ref" only) dH/dtheta through the reference's own derivative chain (MPCController::GaitOpt, :518-552);
        None when the last solve was not `Solved`."""
        out = np.zeros(64)
        n = self._chk(self.lib.orc_mpc_gait_gradient(self.h, _dptr(out), 64))
        return out[:n].copy() if n else None

    def adjust_for_current_contacts(self, time, in_contact):
        """MPC::AdjustForCurrentContacts (mpc.cpp:1195-1203)."""
        self.lib.orc_mpc_adjust_for_contacts.argtypes = [C.c_void_p, C.c_double, _ip]
        c = np.ascontiguousarray(in_contact, dtype=np.int32)
        self._chk(self.lib.orc_mpc_adjust_for_contacts(self.h, float(time), _iptr(c)))

    def gait_lp(self, time, grad, solution=None):
        """(which="ref" only, after gait_gradient) GaitOptimizer::OptimizeContactTimes as the reference wrote it.  solution None: returns
        (2, A dense, lb, ub, q) -- the LP the reference built, recorded by the solver stand-in; with a solution (the LP's optimum, OSQP being
        absent): returns (0, A, lb, ub, q, new_times) where new_times are the optimiser's contact times after the step, foot-major."""
        self.lib.orc_mpc_gait_lp.argtypes = [C.c_void_p, C.c_double, _dp, _dp, _ip, _dp, _dp, _dp, _dp, _dp]
        g = np.ascontiguousarray(grad, dtype=np.float64)
        n = len(g)
        m = 2 * n + 12
        dims = np.zeros(2, np.int32)
        A, lb, ub, q, nt = np.zeros((m, n)), np.zeros(m), np.zeros(m), np.zeros(n), np.zeros(n)
        sol = None if solution is None else np.ascontiguousarray(solution, dtype=np.float64)
        rc = self.lib.orc_mpc_gait_lp(self.h, float(time), _dptr(g), None if sol is None else _dptr(sol), _iptr(dims), _dptr(A), _dptr(lb),
                                      _dptr(ub), _dptr(q), _dptr(nt))
        if rc < 0:
            raise OracleError(self.lib.orc_last_error().decode())
        assert (dims[0], dims[1]) == (m, n), dims
        return (rc, A, lb, ub, q) if rc == 2 else (rc, A, lb, ub, q, nt)

    def contact_times(self, ee):
        n = self.lib.orc_mpc_num_contacts(self.h, ee)
        t, ty = np.zeros(n), np.zeros(n, dtype=np.int32)
        self.lib.orc_mpc_get_contact_times(self.h, ee, _dptr(t), _iptr(ty))
        return t, ty

    def sizes(self):
        out = np.zeros(14, dtype=np.int32)
        self.lib.orc_mpc_sizes(self.h, _iptr(out))
        keys = ["n", "m", "nnzA", "nnzP", "num_dyn", "num_force_box", "num_cone", "num_ee_loc", "num_td", "num_start",
                "nf", "np", "num_eq", "num_ineq"]
        return dict(zip(keys, (int(v) for v in out)))

    def qp(self):
        """Assembled QP of the last assemble()/solve(): dict with scipy csc A, P and vectors q, ub, is_eq."""
        import scipy.sparse as sp
        sz = self.sizes()
        n, m = sz["n"], sz["m"]
        ac, ar, av = np.zeros(n + 1, np.int32), np.zeros(sz["nnzA"], np.int32), np.zeros(sz["nnzA"])
        pc, pr, pv = np.zeros(n + 1, np.int32), np.zeros(sz["nnzP"], np.int32), np.zeros(sz["nnzP"])
        self.lib.orc_mpc_get_A(self.h, _iptr(ac), _iptr(ar), _dptr(av))
        self.lib.orc_mpc_get_P(self.h, _iptr(pc), _iptr(pr), _dptr(pv))
        q, ub = np.zeros(n), np.zeros(m)
        eq = C.create_string_buffer(m)
        self.lib.orc_mpc_get_vectors(self.h, _dptr(q), _dptr(ub), eq)
        return dict(A=sp.csc_matrix((av, ar, ac), shape=(m, n)), P=sp.csc_matrix((pv, pr, pc), shape=(n, n)), q=q, ub=ub,
                    is_eq=np.frombuffer(eq.raw, dtype=np.uint8).astype(bool), sizes=sz)

    def prev_qp_sol(self):
        z = np.zeros(self.sizes()["n"])
        self.lib.orc_mpc_get_prev_qp_sol(self.h, _dptr(z))
        return z

    def qp_solution(self):
        sz = self.sizes()
        x, d, s, info = np.zeros(sz["n"]), np.zeros(sz["m"]), np.zeros(sz["m"]), np.zeros(4)
        self.lib.orc_mpc_get_qp_solution(self.h, _dptr(x), _dptr(d), _dptr(s), _dptr(info))
        return dict(x=x, dual=d, slack=s, status=int(info[0]), iters=int(info[1]), prim_res=info[2], dual_res=info[3])

    def stats(self):
        out = np.zeros(10)
        self.lib.orc_mpc_get_stats(self.h, _dptr(out))
        keys = ["alpha", "eq_violation", "step_norm", "cost", "merit", "merit_dd", "status", "qp_iters", "ee_box_x", "ee_box_y"]
        return dict(zip(keys, out.tolist()))

    def node_dynamics(self):
        sz = self.sizes()
        nu = sz["nf"] + sz["np"]
        Ad, Bd, cd = np.zeros((self.N, 12, 12)), np.zeros((self.N, 12, nu)), np.zeros((self.N, 12))
        self.lib.orc_mpc_get_node_dynamics(self.h, _dptr(Ad), _dptr(Bd), _dptr(cd))
        return Ad, Bd, cd

    def states(self):
        s = np.zeros((self.N + 1, 13))
        self.lib.orc_mpc_get_states(self.h, _dptr(s))
        return s

    def set_state(self, node, s):
        s = np.ascontiguousarray(s, dtype=np.float64)
        self.lib.orc_mpc_set_state(self.h, node, _dptr(s))

    def foot(self, ee):
        """Borrowed view of foot `ee`'s spline (invalid after the next solve)."""
        return FootSpline(None, None, which="oracle", _handle=self.lib.orc_mpc_foot(self.h, ee), _owned=False)

    def init_time(self):
        return self.lib.orc_mpc_init_time(self.h)

    def cost(self):
        return self.lib.orc_mpc_cost(self.h)

    def force_at(self, ee, t):
        out = np.zeros(3)
        self.lib.orc_mpc_force_at(self.h, ee, t, _dptr(out))
        return out

    def ee_at(self, ee, t):
        out = np.zeros(3)
        self.lib.orc_mpc_ee_at(self.h, ee, t, _dptr(out))
        return out

    def merit(self, z):
        z = np.ascontiguousarray(z, dtype=np.float64)
        return self.lib.orc_mpc_merit(self.h, _dptr(z))


def quat_log3(q):
    q = np.ascontiguousarray(q, dtype=np.float64)
    out = np.zeros(3)
    load().orc_quat_log3(_dptr(q), _dptr(out))
    return out


def quat_exp3(v):
    v = np.ascontiguousarray(v, dtype=np.float64)
    out = np.zeros(4)
    load().orc_quat_exp3(_dptr(v), _dptr(out))
    return out


# ---- inverse kinematics (leg_kinematics.cpp); `which` = "oracle" or "ref" (the reference's InverseKinematics over the stand-in)
def kin_flat(consts):
    """tests/golden/a1_robot_consts.json["legs"] -> the 228 packed doubles of kin::RobotKin."""
    out = []
    for leg in consts["legs"]:
        out += np.asarray(leg["t"], float).ravel().tolist() + np.asarray(leg["R"], float).ravel().tolist() + np.asarray(leg["axis"], float).ravel().tolist()
    a = np.ascontiguousarray(out, dtype=np.float64)
    assert a.size == 228
    return a


def _bind_kin(lib):
    if getattr(lib, "_kin_bound", False):
        return lib
    lib.orc_kin_exp6.argtypes = [_dp, _dp, _dp]
    lib.orc_kin_log6.argtypes = [_dp, _dp, _dp]
    lib.orc_kin_jlog6.argtypes = [_dp, _dp, _dp]
    lib.orc_kin_fk.argtypes = [_dp, _dp, C.c_int, _dp, _dp, _dp]
    lib.orc_kin_integrate.argtypes = [_dp, _dp, _dp]
    lib.orc_ik.argtypes = [_dp, _dp, _dp, _dp, _dp, _ip]
    lib.orc_mpc_targets_from_traj.argtypes = [C.c_void_p, _dp, C.c_double, C.c_double, C.c_double, _dp, _dp, _dp, _dp]
    lib._kin_bound = True
    return lib


def kin_exp6(nu):
    nu = np.ascontiguousarray(nu, dtype=np.float64)
    R, p = np.zeros((3, 3)), np.zeros(3)
    _bind_kin(load()).orc_kin_exp6(_dptr(nu), _dptr(R), _dptr(p))
    return R, p


def kin_log6(R, p):
    R, p = np.ascontiguousarray(R, dtype=np.float64), np.ascontiguousarray(p, dtype=np.float64)
    out = np.zeros(6)
    _bind_kin(load()).orc_kin_log6(_dptr(R), _dptr(p), _dptr(out))
    return out


def kin_jlog6(R, p):
    R, p = np.ascontiguousarray(R, dtype=np.float64), np.ascontiguousarray(p, dtype=np.float64)
    J = np.zeros((6, 6))
    _bind_kin(load()).orc_kin_jlog6(_dptr(R), _dptr(p), _dptr(J))
    return J


def kin_fk(kin, q, ee=0):
    """World positions [4][3] / rotations [4][3][3] of the foot frames, and the 6 x 18 LOCAL Jacobian of foot `ee`."""
    q = np.ascontiguousarray(q, dtype=np.float64)
    fp, fR, J = np.zeros((4, 3)), np.zeros((4, 3, 3)), np.zeros((6, 18))
    _bind_kin(load()).orc_kin_fk(_dptr(kin), _dptr(q), ee, _dptr(fp), _dptr(fR), _dptr(J))
    return fp, fR, J


def kin_integrate(q, v):
    q, v = np.ascontiguousarray(q, dtype=np.float64), np.ascontiguousarray(v, dtype=np.float64)
    out = np.zeros(19)
    _bind_kin(load()).orc_kin_integrate(_dptr(q), _dptr(v), _dptr(out))
    return out


def ik(kin, state, ee_des, joint_guess, which="oracle"):
    """SingleRigidBodyModel::InverseKinematics.  Returns (status, q[19], iters[4]); status 1 = "IK did not converge."."""
    lib = _bind_kin(load()) if which == "oracle" else load_ref_mpc()
    state = np.ascontiguousarray(state, dtype=np.float64)
    ee = np.ascontiguousarray(ee_des, dtype=np.float64)
    g = np.ascontiguousarray(joint_guess, dtype=np.float64)
    q, it = np.zeros(19), np.zeros(4, np.int32)
    if which == "oracle":
        rc = lib.orc_ik(_dptr(kin), _dptr(state), _dptr(ee), _dptr(g), _dptr(q), _iptr(it))
    else:
        rc = lib.orc_ref_ik(_dptr(kin), _dptr(state), _dptr(ee), _dptr(g), _dptr(q))
    return rc, q, it


def targets_from_traj(mpc, kin, consts, time, dt, q_des):
    """MPCController::GetTargetsFromTraj on the oracle's trajectory.  Returns (status, q_des[19], v_des[18], force_des[4][3])."""
    lib = _bind_kin(mpc.lib)
    q = np.ascontiguousarray(q_des, dtype=np.float64).copy()
    v, f = np.zeros(18), np.zeros((4, 3))
    Ii = np.ascontiguousarray(consts["Ir_inv"], dtype=np.float64)
    rc = lib.orc_mpc_targets_from_traj(mpc.h, _dptr(kin), time, dt, consts["mass"], _dptr(Ii), _dptr(q), _dptr(v), _dptr(f))
    return rc, q, v, f
