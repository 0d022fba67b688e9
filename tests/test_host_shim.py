"""The C++ host shim (bilevel-gait-gen_b200/host): the reference's MPC / MPCSingleRigidBody / Trajectory / GaitOptimizer call
surface over the C ABI.  CPU part: the shim library loads and its URDF reader reproduces the robot constants the tests
use; GPU part: tests/cpp/test_shim.cpp (shaped like the reference's test/mpc_test.cpp set-up) against the oracle."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

import common
from common import wl

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "bilevel-gait-gen_b200")
SHIM_SO = os.path.join(PKG, "libmpc_b200.so")
TEST_BIN = os.path.join(ROOT, "tests", "cpp", "test_shim")
# a trimmed A1 model with the reference's joint tree and the fixture's constants, and the three configurations in the reference's
# YAML layout; BGG_REFERENCE_DIR (a checkout of the reference project) substitutes the reference's own files
REF_DIR = os.environ.get("BGG_REFERENCE_DIR", "")
A1_URDF = (os.path.join(REF_DIR, "models", "a1_description", "urdf", "a1.urdf") if REF_DIR else
           os.path.join(ROOT, "tests", "golden", "a1_trimmed.urdf"))
REF_APPS = os.path.join(REF_DIR, "apps") if REF_DIR else os.path.join(ROOT, "tests", "golden", "apps")


def test_shim_library_loads_and_exports_the_urdf_entry_point():
    assert os.path.exists(SHIM_SO), "build it with bilevel-gait-gen_b200/build.sh"
    lib = C.CDLL(SHIM_SO)
    assert hasattr(lib, "bgg_host_robot_consts_from_urdf")
    assert os.path.exists(TEST_BIN)


def test_urdf_reader_matches_the_robot_constants_fixture():
    import bgg_b200 as bg
    lib = C.CDLL(SHIM_SO)
    rb = bg.Robot()
    assert lib.bgg_host_robot_consts_from_urdf(A1_URDF.encode(), C.byref(rb)) == 0
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "a1_robot_consts.json")))
    assert abs(rb.mass - gold["mass"]) < 1e-12
    assert np.abs(np.array(rb.Ir[:]).reshape(3, 3) - np.array(gold["Ir"])).max() < 1e-12
    assert np.abs(np.array(rb.Ir_inv[:]).reshape(3, 3) - np.array(gold["Ir_inv"])).max() < 1e-9
    assert np.abs(np.array(rb.hip_xy[:]).reshape(4, 2) - np.array(gold["hip_offsets_xy"])).max() < 1e-12


def test_urdf_reader_extracts_the_leg_chains_of_the_fixture():
    """host/urdf_consts.cpp: LegKinematicsFromURDF (what the inverse kinematics needs of the model) against tests/golden."""
    lib = C.CDLL(SHIM_SO)
    kin = (C.c_double * 228)()
    assert lib.bgg_host_leg_kinematics_from_urdf(A1_URDF.encode(), kin) == 0
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "a1_robot_consts.json")))
    want = []
    for leg in gold["legs"]:
        want += np.asarray(leg["t"], float).ravel().tolist() + np.asarray(leg["R"], float).ravel().tolist() + np.asarray(leg["axis"], float).ravel().tolist()
    assert np.abs(np.array(kin[:]) - np.array(want)).max() < 1e-15


@pytest.mark.parametrize("name", ["a1_configuration", "a1_gait_opt_config", "a1_config_distr_rejection"])
def test_config_parser_reads_the_reference_yaml_and_pins_the_named_workloads(name):
    """utils::ConfigParser + the MPCInfo fill of test/mpc_test.cpp:46-83 on the reference's own configuration files; the
    values must be the ones bilevel-gait-gen_b200/workloads.py (bench.py, tests) carries for the same name."""
    lib = C.CDLL(SHIM_SO)
    out = (C.c_double * 47)()
    assert lib.bgg_host_parse_config(os.path.join(REF_APPS, name + ".yaml").encode(), out) == 0
    v = list(out)
    cfg = wl.CONFIGS[name]
    assert int(v[0]) == cfg["num_nodes"]
    got = dict(integrator_dt=v[1], friction_coef=v[2], force_bound=v[3], swing_height=v[4], foot_offset=v[5], force_cost=v[8])
    for k, x in got.items():
        assert x == cfg[k], (k, x, cfg[k])
    assert tuple(v[6:8]) == tuple(cfg["ee_box_size"])
    assert v[9:21] == [float(x) for x in cfg["Q"]]
    assert v[21:34] == [float(x) for x in cfg["srb_init"]]
    assert v[34:47] == [float(x) for x in cfg["srb_target"]]


@pytest.mark.gpu
def test_shim_reproduces_the_oracle_on_the_reference_test_setup(tmp_path):
    import gait_oracle as go
    rb = wl.robot()
    consts = [rb["mass"]] + list(np.ravel(rb["Ir"])) + list(np.ravel(rb["Ir_inv"])) + list(np.ravel(rb["hip_offsets_xy"]))
    path = tmp_path / "robot.txt"
    path.write_text(" ".join(repr(float(v)) for v in consts))
    yaml = tmp_path / "cfg.yaml"   # the reference's YAML layout: scalars, strings, multi-line flow sequences, comments
    yaml.write_text("""robot_urdf: "/somewhere/a1.urdf"
collision_frames: ["FL_foot", "FR_foot", "RL_foot", "RR_foot"]    # for pinocchio
init_config: [0., 0., 0.3, 0.0, 0.0, 0.0, 1.0, # base
              -0.02, 0.9, -1.6,       # front left
              0.02, 0.9, -1.6, 0.02, 0.9, -1.6, -0.02, 0.9, -1.6]
friction_coef: 0.5 #0.3
discretization_steps: 1
num_nodes: 20 #30
integrator_dt: 0.05
num_qp: 1
vel_bounds: [10, 10, 10]
joint_bounds_lb: [-0.8, -3.0]
joint_bounds_ub: [0.8, 4.1]
num_switches: 2
force_bound: 150
swing_height: 0.075
ee_box_size: [0.15, 0.15]
run_time_iterations: 6000
foot_offset: 0.015
force_cost: 0.000
""")
    out = subprocess.run([TEST_BIN, str(path), str(yaml)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    kv = {}
    for line in out.stdout.splitlines():
        parts = line.split()
        if parts:
            kv[parts[0]] = parts[1:]
    assert kv["done"] == ["1"], out.stdout
    assert kv["bad_cost_throws"] == ["1"]
    assert kv["initial_quality"] == ["0"] and kv["rt_quality"] == ["0"]
    assert kv["num_decision_vars"] == ["372"] and kv["num_constraints"] == ["1012"]      # SURVEY section 8 size table
    assert kv["qp_rows"] == ["1012"] and kv["qp_cols"] == ["372"]
    assert kv["num_equality"] == ["260"] and kv["num_inequality"] == ["752"]
    assert kv["num_contact_nodes"] == ["5", "5", "5", "5"]
    assert kv["copy_cost_equal"] == ["1"] and kv["derivative_terms"] == ["1"]
    assert kv["yaml_num_nodes"] == ["20"] and kv["yaml_friction"] == ["0.500000"] and kv["yaml_frames"] == ["4"]
    log = open(str(path) + ".log").read().splitlines()
    assert log[0] == "-" * 150 and "MPC Statistics" in log[1] and log[3] == "Number of nodes: 20"
    header = [i for i, l in enumerate(log) if l.startswith("Solve #")][0]
    assert log[header].split()[:4] == ["Solve", "#", "Time", "(ms)"] and len(log[header]) == 150
    rows = log[header + 2:]
    assert len(rows) == 2 and rows[0][:15].strip() == "10" and rows[1][:15].strip() == "11" and "Solved" in rows[0]

    # the solver seam on the reference's own 3-variable QP (test/mpc_test.cpp:857-953): quality, primal within its 1e-4 margin of
    # the closed-form optimum, stationarity with the returned multipliers, and the "Primal infeasible." throw
    import test_oracle_qp
    assert kv["qp3_quality"] == ["0"]
    assert np.abs(np.array([float(v) for v in kv["qp3_x"]]) - test_oracle_qp.exact_solution()).max() < 1e-4
    assert float(kv["qp3_stationarity"][0]) < 1e-6
    assert kv["qp3_infeasible_throws"] == ["1"]
    # AdjustForCurrentContacts: inside the 70 ms window the foot is put in contact, outside it is not (mpc.cpp:1195-1203)
    assert int(kv["adjust_swing_foot"][0]) >= 0 and kv["adjust_near"] == ["1"] and kv["adjust_far"] == ["0"]
    # the reference's "Model Partials" check (test/mpc_test.cpp:113-236) through the C++ layer: real sparse QPPartials against finite
    # differences of the assembled constraints, its DERIV_MARGIN = 1e-4
    assert kv["partials_checked"] == ["16"] and int(kv["partials_nnz"][0]) > 0 and int(kv["partials_nnz"][1]) > 0
    assert float(kv["partials_fd_dyn"][0]) < 1e-4 and float(kv["partials_fd_fb"][0]) < 1e-4 and float(kv["partials_fd_cone"][0]) < 1e-4
    # the MPCCentroidal adapter runs the same solves as the live class
    assert kv["centroidal_vars"] == ["372"] and kv["centroidal_cost_equal"] == ["1"]

    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    init = np.asarray(cfg["srb_init"], float)
    ee = wl.EE_NOMINAL.copy()
    o = common.make_oracle(cfg_name)
    o.initial_run(init, ee)
    o.solve(init, 0.0, ee, real_time=True)
    # the two sides ran 11 solves each from their own trajectories: an entry that is exactly 0.0 on one side can be 1e-20 on
    # the other (bit-exact sparsity on identical inputs is tested in test_gpu_parity.py)
    assert abs(int(kv["qp_nnz"][0]) - o.sizes()["nnzA"]) <= 16
    assert abs(float(kv["cost"][0]) - o.cost()) <= 1e-4 * max(1.0, abs(o.cost()))
    assert abs(float(kv["state1_z"][0]) - o.states()[1][2]) < 1e-6
    assert abs(float(kv["force_ee1_z_t01"][0]) - o.force_at(1, 0.1)[2]) <= 1e-4 * max(1.0, abs(o.force_at(1, 0.1)[2]))
    assert abs(float(kv["ee0_x_t04"][0]) - o.ee_at(0, 0.4)[0]) < 1e-6
    # AdjustForCurrentContacts on the oracle (itself bit-identical to the reference's, tests/test_oracle_vs_reference_mpc.py): the same
    # contact times for the foot that was put in contact early
    foot = int(kv["adjust_swing_foot"][0])
    call_time, times_after = float(kv["adjust_near_times"][0]), np.array([float(v) for v in kv["adjust_near_times"][1:]])
    times_before = np.array([float(v) for v in kv["adjust_before_times"]])
    oa = o.clone()
    oa.adjust_for_current_contacts(call_time, [1 if e == foot else 0 for e in range(4)])
    moved_o = np.flatnonzero(oa.contact_times(foot)[0] != o.contact_times(foot)[0])
    moved = np.flatnonzero(times_after != times_before)
    # (the C++ object has been through the gait step above, its later contact times differ from the oracle's: what is compared is
    # which contact time the call moved and where to)
    assert len(moved) == 1 and np.array_equal(moved, moved_o)
    assert abs(times_after[moved[0]] - oa.contact_times(foot)[0][moved[0]]) < 1e-12
    g_o = go.cost_gradient(o)
    g = np.array([float(v) for v in kv["gradient"]])
    assert np.abs(g - g_o).max() <= 1e-4 * max(1.0, np.abs(g_o).max())
    ct = go.contact_times(o)
    s_o = go.solve_gait_lp(ct, g_o, 0.0)
    s = np.array([float(v) for v in kv["step"]])
    assert np.abs(s - s_o).max() < 1e-6
    xk = np.concatenate([t for t, _ in ct])
    best, costs, q = go.line_search(o, init, 0.0, ee, ct, xk, s_o, ls_size=10)
    assert abs(float(kv["ls_cost_min"][0]) - costs[best]) <= 1e-4 * max(1.0, abs(costs[best]))
