"""The oracle's restatement of the MPC hot path against the REFERENCE'S OWN SOURCES compiled here.

oracle/_ref/libref_mpc.so (oracle/Makefile) is built from $BGG_REFERENCE_DIR/mpc/{trajectory, mpc, mpc_single_rigid_body,
rk_integrator, gait_optimizer}.cpp, mpc/models/{model, single_rigid_body_model}.cpp, mpc/qp/{qp_data, qp_interface,
clarabel_interface}.cpp, mpc/spline/*.cpp and utils/sparse_matrix_builder.cpp -- unmodified -- over the stand-in headers of
oracle/ref_shim/ (Eigen containers, pinocchio with injected robot constants, the Clarabel solver = the oracle's restatement
of its algorithm).  So everything the reference computes around the solver runs as the reference wrote it:
spline maintenance, linearisation, Euler discretisation, the six constraint emitters, zero dropping, triplets -> CSC, bound
stacking, status handling and foot-box adaptation, the merit line search, the trajectory update -- and the QP derivative
chain of the gait optimiser.  These tests require the oracle to reproduce it BIT FOR BIT (SURVEY.md section 8 rows a5-a15)
and the gait gradient to 1e-9 (a16-a19; the 1384 x 1384 differential system is factorised by two different LU codes).

Where the reference's sources are absent (BGG_REFERENCE_DIR unset) every test runs against what the reference returned, stored in
tests/golden/reference_outputs.json (common.Recorded: digests of the values in call order; the gait gradient as numbers).
"""
import hashlib
import os

import numpy as np
import pytest

import common
from common import wl

po = pytest.importorskip("pyoracle")
LIVE = po.have_ref_mpc()   # the reference's own sources compiled into oracle/_ref/libref_mpc.so


def _make(cfg_name, which, state, digest=None):
    """which "ref": the reference's compiled code, or the restatement standing in for it when that is absent; wrapped in
    common.Recorded (sharing `digest`) so that what it returns is checked against the stored reference outputs."""
    cfg = wl.CONFIGS[cfg_name]
    src = "ref" if which == "ref" and LIVE else "oracle"
    o = po.SrbMpc(cfg["num_nodes"], cfg["integrator_dt"], wl.robot(), which=src, **wl.mpc_kwargs(cfg))
    o.set_costs(wl.target_tangent(cfg), np.asarray(cfg["Q"], float))
    o.set_warm_states(np.tile(np.asarray(state, float), (cfg["num_nodes"] + 1, 1)))
    return common.Recorded(o, digest) if which == "ref" else o


def _assert_same_qp_bitwise(r, o):
    qr, qo = r.qp(), o.qp()
    assert qr["sizes"] == qo["sizes"]
    assert np.array_equal(qr["A"].indptr, qo["A"].indptr) and np.array_equal(qr["A"].indices, qo["A"].indices), "sparsity differs"
    assert np.array_equal(qr["A"].data, qo["A"].data), f"A values differ by {np.abs(qr['A'].data - qo['A'].data).max():.3e}"
    assert np.array_equal(qr["P"].indptr, qo["P"].indptr) and np.array_equal(qr["P"].indices, qo["P"].indices)
    assert np.array_equal(qr["P"].data, qo["P"].data)
    assert np.array_equal(qr["q"], qo["q"])
    assert np.array_equal(qr["ub"], qo["ub"])
    assert np.array_equal(qr["is_eq"], qo["is_eq"])


def _assert_same_step_bitwise(r, o):
    sr, so = r.stats(), o.stats()
    assert sr == so, (sr, so)     # alpha, eq violation, step norm, cost, merit, merit derivative, status, iterations, foot box
    assert np.array_equal(r.prev_qp_sol(), o.prev_qp_sol())
    assert np.array_equal(r.states(), o.states())
    assert r.init_time() == o.init_time() and r.cost() == o.cost()
    for e in range(4):
        for t in np.linspace(r.init_time(), r.init_time() + 1.0, 7):
            assert np.array_equal(r.force_at(e, t), o.force_at(e, t)) and np.array_equal(r.ee_at(e, t), o.ee_at(e, t))


@pytest.mark.parametrize("cfg_name", ["a1_configuration", "a1_gait_opt_config", "a1_config_distr_rejection"])
def test_rti_step_is_bitwise_the_reference(cfg_name):
    """One RTI step from the nominal state (the reference's own test case, test/mpc_test.cpp:91-101) and from random states:
    assembled QP and everything the step leaves behind, bit for bit."""
    cfg = wl.CONFIGS[cfg_name]
    states, _, ee = wl.batched_trot_inputs(cfg, 4, seed=17)
    states[0] = cfg["srb_init"]
    ee[0] = wl.EE_NOMINAL
    seen = set()
    digest = hashlib.sha256()
    for b in range(4):
        r, o = _make(cfg_name, "ref", states[b], digest), _make(cfg_name, "oracle", states[b])
        for _ in range(3):   # three RTI steps at t = 0 (the start of CreateInitialRun)
            sr = r.solve(states[b], 0.0, ee[b])
            so = o.solve(states[b], 0.0, ee[b])
            assert sr == so
            seen.add(sr)
            _assert_same_qp_bitwise(r, o)
            _assert_same_step_bitwise(r, o)
    assert 0 in seen
    common.check_golden_reference(f"rti_step/{cfg_name}", digest)


def test_receding_horizon_is_bitwise_the_reference():
    """15 closed-loop ticks at N = 20 (t0 advances by dt, the state is the model's own next node, feet from the trajectory):
    knots are appended and dropped, touch-down rows appear and vanish, the QP changes size -- assembly and step stay
    bit-identical to the reference's code at every tick."""
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    init = np.asarray(cfg["srb_init"], float)
    r, o = _make(cfg_name, "ref", init), _make(cfg_name, "oracle", init)
    assert r.initial_run(init, wl.EE_NOMINAL) == o.initial_run(init, wl.EE_NOMINAL)
    _assert_same_step_bitwise(r, o)
    sizes = set()
    state = init.copy()
    for step in range(15):
        t0 = cfg["integrator_dt"] * step
        ee_now = np.array([o.ee_at(e, t0) for e in range(4)])
        assert r.solve(state, t0, ee_now) == o.solve(state, t0, ee_now)
        _assert_same_qp_bitwise(r, o)
        _assert_same_step_bitwise(r, o)
        sizes.add((o.sizes()["n"], o.sizes()["m"]))
        state = o.states()[1].copy()
    assert len(sizes) > 1, "the horizon never changed size"
    common.check_golden_reference("receding_horizon", r.digest)


def test_infeasible_qp_takes_the_reference_path():
    """Feet 10 cm off nominal: the QP is infeasible, ClarabelInterface::Solve throws "Primal infeasible.", Solve() catches it,
    keeps the previous solution and widens the foot box (mpc_single_rigid_body.cpp:115-144).  Same on both sides, bit for bit,
    over three solves (the widened box changes the next QP)."""
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    states, _, ee = wl.batched_trot_inputs(cfg, 12, seed=0)
    ee[:, :, :2] += np.random.default_rng(5).uniform(-0.08, 0.08, (12, 4, 2))
    hit = 0
    digest = hashlib.sha256()
    for b in range(12):
        r, o = _make(cfg_name, "ref", states[b], digest), _make(cfg_name, "oracle", states[b])
        st = [(r.solve(states[b], 0.0, ee[b]), o.solve(states[b], 0.0, ee[b])) for _ in range(3)]
        assert all(a == c for a, c in st), st
        _assert_same_qp_bitwise(r, o)
        _assert_same_step_bitwise(r, o)
        if st[0][0] == 3:
            hit += 1
            assert r.stats()["ee_box_x"] > cfg["ee_box_size"][0]
    assert hit >= 1, "no infeasible instance in this batch"
    common.check_golden_reference("infeasible_qp", digest)


@pytest.mark.parametrize("cfg_name", ["a1_configuration"])
def test_gait_gradient_matches_the_reference_chain(cfg_name):
    """dH/dtheta through the reference's own derivative code -- ClarabelInterface::SetupDerivativeCalcs / CalcDerivativeWrtMats /
    Vecs (clarabel_interface.cpp:182-612), MPCSingleRigidBody::ComputeParamPartialsClarabel (mpc_single_rigid_body.cpp:642-792),
    GaitOptimizer::ModifyQPPartials / ComputeCostFcnDerivWrtContactTimes (gait_optimizer.cpp:92-179, 536-539), called in the
    order of MPCController::GaitOpt (mpc_controller.cpp:518-552) -- against the oracle's restatement (oracle/gait_oracle.py).
    Eigen::SparseLU is a dense LU with partial pivoting here, scipy's SuperLU there: 1e-9 relative."""
    import gait_oracle as go
    cfg = wl.CONFIGS[cfg_name]
    init = np.asarray(cfg["srb_init"], float)
    r, o = _make(cfg_name, "ref", init), _make(cfg_name, "oracle", init)
    assert r.initial_run(init, wl.EE_NOMINAL) == o.initial_run(init, wl.EE_NOMINAL) == 0
    assert r.solve(init, 0.0, wl.EE_NOMINAL) == o.solve(init, 0.0, wl.EE_NOMINAL) == 0
    g_o = go.cost_gradient(o)
    n = len(g_o)
    assert n == sum(len(r.contact_times(e)[0]) for e in range(4))
    tol = 1e-9 * max(1.0, np.abs(g_o).max())
    if LIVE:
        g_live = r.gait_gradient()
        assert g_live is not None
        assert np.abs(g_live[:n] - g_o).max() <= tol, (g_live[:n], g_o)
    if os.environ.get("BGG_RECORD_GOLDEN"):
        common.check_golden_reference(f"gait_gradient/{cfg_name}", (g_live if LIVE else g_o)[:n].tolist())
    g_ref = np.array(common.golden_reference(f"gait_gradient/{cfg_name}"))
    assert len(g_ref) == n and np.abs(g_ref - g_o).max() <= tol, (g_ref, g_o)


@pytest.mark.parametrize("cfg_name", ["a1_configuration", "a1_gait_opt_config"])
def test_contact_time_lp_is_the_one_the_reference_builds(cfg_name):
    """GaitOptimizer::OptimizeContactTimes (gait_optimizer.cpp:185-364: CreatePolytopeConstraint, CreateStartConstraint,
    CreateTrustRegionConstraint, CreateNextNodeConstraints, the zero Hessian, ConvertQPVecToContactTimes) run as the reference wrote
    it.  OSQP is absent, so the solver stand-in records the LP the reference hands over and plays back an injected optimum: the
    restatement's LP (oracle/gait_oracle.py: gait_lp) must be the same matrix and bounds, and the contact times the reference makes of
    the step must be the restatement's (contact_times_for)."""
    import gait_oracle as go
    cfg = wl.CONFIGS[cfg_name]
    init = np.asarray(cfg["srb_init"], float)
    r = _make(cfg_name, "ref", init)
    assert r.initial_run(init, wl.EE_NOMINAL) == 0 and r.solve(init, 0.0, wl.EE_NOMINAL) == 0
    ct = [r.contact_times(e) for e in range(4)]
    n = sum(len(t) for t, _ in ct)
    if LIVE:
        g = r.gait_gradient()
        assert g is not None
        g = g[:n]
    else:
        if os.environ.get("BGG_RECORD_GOLDEN"):
            common.check_golden_reference(f"gait_gradient/{cfg_name}", go.cost_gradient(r._obj).tolist())
        g = np.array(common.golden_reference(f"gait_gradient/{cfg_name}"))
        assert len(g) == n

    def gait_lp(time, grad, solution=None):   # the reference's OptimizeContactTimes, or the restatement in its call shape
        if LIVE:
            out = r.gait_lp(time, grad, solution)
        else:
            A, lb, ub = go.gait_lp(ct, grad, time)
            out = (2, A.toarray(), lb, ub, grad.copy())
            if solution is not None:
                xk_ = np.concatenate([t for t, _ in ct])
                out = (0,) + out[1:] + (np.concatenate(go.contact_times_for(ct, xk_, solution, 1.0)),)
        common._feed(r.digest, out)
        return out

    for time in (0.0, 0.13):
        A_o, lb_o, ub_o = go.gait_lp(ct, g, time)
        rc, A_r, lb_r, ub_r, q_r = gait_lp(time, g)
        assert rc == 2
        assert np.array_equal(A_r, A_o.toarray())
        assert np.array_equal(lb_r, lb_o) and np.array_equal(ub_r, ub_o) and np.array_equal(q_r, g)
    step = go.solve_gait_lp(ct, g, 0.0)
    xk = np.concatenate([t for t, _ in ct])
    rc, _, _, _, _, new_times = gait_lp(0.0, g, step)
    assert rc == 0
    want = np.concatenate(go.contact_times_for(ct, xk, step, 1.0))
    assert np.array_equal(new_times, want), np.abs(new_times - want).max()
    if not LIVE or os.environ.get("BGG_RECORD_GOLDEN"):   # with the live reference, its own gradient (1e-9 from the stored one) feeds the LP
        common.check_golden_reference(f"contact_time_lp/{cfg_name}", r.digest)


def test_adjust_for_current_contacts_is_the_references():
    """MPC::AdjustForCurrentContacts (mpc.cpp:1195-1203): a swing foot reported in contact within 70 ms of its planned touch-down is
    put in contact in the plan (EndEffectorSplines::SetToTouchdown), otherwise nothing changes.  Reference code against the
    restatement: the contact schedules after the call and the whole next RTI step, bit for bit."""
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    init = np.asarray(cfg["srb_init"], float)
    digest = hashlib.sha256()
    for early_by, expect_change in ((0.05, True), (0.15, False)):
        r, o = _make(cfg_name, "ref", init, digest), _make(cfg_name, "oracle", init)
        assert r.initial_run(init, wl.EE_NOMINAL) == o.initial_run(init, wl.EE_NOMINAL) == 0
        before = [r.contact_times(e) for e in range(4)]
        swing = [e for e in range(4) if before[e][1][0] != po.TOUCH_DOWN][0]      # a foot that starts in swing
        t_td = [t for t, ty in zip(*before[swing]) if ty == po.TOUCH_DOWN][0]     # its first planned touch-down
        now = t_td - early_by
        flags = [1 if e == swing else 0 for e in range(4)]
        r.adjust_for_current_contacts(now, flags)
        o.adjust_for_current_contacts(now, flags)
        after_r = [r.contact_times(e) for e in range(4)]
        after_o = [o.contact_times(e) for e in range(4)]
        for e in range(4):
            assert np.array_equal(after_r[e][0], after_o[e][0]) and np.array_equal(after_r[e][1], after_o[e][1])
        changed = not all(np.array_equal(after_r[e][0], before[e][0]) for e in range(4))
        assert changed == expect_change
        ee_now = np.array([o.ee_at(e, now) for e in range(4)])
        state = o.states()[1].copy()
        assert r.solve(state, now, ee_now) == o.solve(state, now, ee_now)
        _assert_same_qp_bitwise(r, o)
        _assert_same_step_bitwise(r, o)
    common.check_golden_reference("adjust_for_current_contacts", digest)
