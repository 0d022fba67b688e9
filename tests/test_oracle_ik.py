"""CPU tests of the oracle's inverse-kinematics restatement (oracle/leg_kinematics.cpp; SURVEY 8f row 2).

pinocchio is absent, so the rigid-body formulas are pinned by properties (finite differences, round trips, the converged
configuration reaching its targets) and the IK loop built on them by the reference's own
SingleRigidBodyModel::InverseKinematics (mpc/models/single_rigid_body_model.cpp:314-425) compiled over the stand-in headers."""
import numpy as np
import pytest

import common
from common import wl
import pyoracle as po

NOMINAL_JOINTS = np.array([-0.02, 0.9, -1.6, 0.02, 0.9, -1.6, 0.02, 0.9, -1.6, -0.02, 0.9, -1.6])   # apps/a1_configuration.yaml: init_config


def _kin():
    return po.kin_flat(wl.robot())


def random_problems(n, seed):
    """SRB states near the nominal stance and foot targets near the nominal footholds."""
    rng = np.random.default_rng(seed)
    kin = _kin()
    st = np.zeros((n, 13))
    st[:, :3] = [0.0, 0.0, 0.3] + rng.uniform(-0.03, 0.03, (n, 3))
    st[:, 3:6] = rng.normal(0, 1.0, (n, 3))
    quat = np.concatenate([rng.normal(0, 0.05, (n, 3)), np.ones((n, 1))], axis=1)
    st[:, 6:10] = quat / np.linalg.norm(quat, axis=1, keepdims=True)
    st[:, 10:13] = rng.normal(0, 0.1, (n, 3))
    feet0 = po.kin_fk(kin, np.concatenate([[0, 0, 0.3, 0, 0, 0, 1], NOMINAL_JOINTS]))[0]
    ee = feet0[None] + rng.uniform(-0.04, 0.04, (n, 4, 3))
    ee[:, :, 2] = np.maximum(ee[:, :, 2] - feet0[:, 2].mean(), 0.0)
    guess = NOMINAL_JOINTS[None] + rng.normal(0, 0.05, (n, 12))
    return st, ee, guess


def test_exp6_log6_round_trip_and_rotation_is_orthogonal():
    rng = np.random.default_rng(1)
    for scale in (1e-7, 1e-3, 0.5, 2.0):
        nu = rng.normal(size=6)
        nu *= scale / np.linalg.norm(nu[3:])
        R, p = po.kin_exp6(nu)
        assert np.abs(R @ R.T - np.eye(3)).max() < 1e-14
        assert np.abs(po.kin_log6(R, p) - nu).max() < 1e-12 * max(1.0, scale)


def test_jlog6_is_the_right_jacobian_of_log6():
    rng = np.random.default_rng(2)
    for scale in (1e-6, 0.3, 2.0):
        nu = rng.normal(size=6) * scale
        R, p = po.kin_exp6(nu)
        J, h, fd = po.kin_jlog6(R, p), 1e-6, np.zeros((6, 6))
        for k in range(6):
            d = np.zeros(6)
            d[k] = h
            Rd, pd = po.kin_exp6(d)
            Rm, pm = po.kin_exp6(-d)
            fd[:, k] = (po.kin_log6(R @ Rd, p + R @ pd) - po.kin_log6(R @ Rm, p + R @ pm)) / (2 * h)
        assert np.abs(J - fd).max() < 1e-8


def test_foot_jacobian_is_the_local_velocity_of_the_foot_frame():
    kin = _kin()
    q = np.concatenate([[0.1, -0.2, 0.3, 0.1, 0.05, -0.08, 0.99], NOMINAL_JOINTS + 0.1])
    q[3:7] /= np.linalg.norm(q[3:7])
    h = 1e-6
    for ee in range(4):
        fp, fR, J = po.kin_fk(kin, q, ee)
        fd = np.zeros((6, 18))
        for k in range(18):
            v = np.zeros(18)
            v[k] = h
            pp, Rp, _ = po.kin_fk(kin, po.kin_integrate(q, v), ee)
            pm, Rm, _ = po.kin_fk(kin, po.kin_integrate(q, -v), ee)
            fd[:3, k] = fR[ee].T @ (pp[ee] - pm[ee]) / (2 * h)
            dR = fR[ee].T @ (Rp[ee] - Rm[ee]) / (2 * h)
            fd[3:, k] = [dR[2, 1], dR[0, 2], dR[1, 0]]
        assert np.abs(J - fd).max() < 1e-8
        other = [6 + 3 * e + j for e in range(4) if e != ee for j in range(3)]
        assert np.all(J[:, other] == 0.0)


def test_nominal_stance_matches_the_urdf_geometry():
    """Feet of the nominal configuration: x = hip x + thigh/calf offsets, |y| = hip y + 0.0838, symmetric left / right."""
    feet = po.kin_fk(_kin(), np.concatenate([[0, 0, 0.3, 0, 0, 0, 1], NOMINAL_JOINTS]))[0]
    assert np.allclose(feet[0, [0, 2]], feet[1, [0, 2]], atol=1e-15) and np.isclose(feet[0, 1], -feet[1, 1])
    leg_z = -0.2 * np.cos(0.9) - 0.2 * np.cos(0.9 - 1.6)
    assert np.isclose(feet[0, 2], 0.3 + 0.0838 * np.sin(-0.02) + leg_z * np.cos(-0.02), atol=1e-12)   # hip roll tilts the leg plane


def test_ik_reaches_the_targets_and_keeps_the_body_pose():
    kin = _kin()
    st, ee, guess = random_problems(16, 3)
    for b in range(16):
        rc, q, it = po.ik(kin, st[b], ee[b], guess[b])
        assert rc == 0 and it.max() < 1000 and it.min() > 0
        feet = po.kin_fk(kin, q)[0]
        # each foot was converged to 5e-6 in turn; later feet move the base by less than that
        assert np.abs(feet - ee[b]).max() < 2e-5
        assert np.abs(q[:3] - st[b, :3]).max() < 2e-5 and np.abs(q[3:7] - st[b, 6:10]).max() < 2e-5


def test_ik_reports_non_convergence_like_the_reference_throws():
    kin = _kin()
    st, ee, guess = random_problems(1, 4)
    ee[0, 0] = [2.0, 2.0, 0.0]   # out of reach for the first foot: no foot has succeeded yet, the reference throws
    rc, _, it = po.ik(kin, st[0], ee[0], guess[0])
    assert rc == 1 and it[0] == 1000


def test_restated_ik_loop_equals_the_references_own_code():
    """Against the reference's InverseKinematics compiled into oracle/_ref, or, without it, against its joint angles stored in
    tests/golden/reference_outputs.json."""
    import os
    kin = _kin()
    live = po.have_ref_mpc()
    if live:
        po.load_ref_mpc().orc_ref_ik.argtypes = [po._dp] * 5
    st, ee, guess = random_problems(12, 5)
    ref_q = []
    for b in range(12):
        rc, q, _ = po.ik(kin, st[b], ee[b], guess[b])
        assert rc == 0
        if live:
            rc2, q2, _ = po.ik(kin, st[b], ee[b], guess[b], which="ref")
            assert rc2 == 0
            ref_q.append(q2)
        elif os.environ.get("BGG_RECORD_GOLDEN"):
            q2 = q
        else:
            q2 = np.array(common.golden_reference("ik_joint_angles")[b])
        # same arithmetic except the 9 x 9 solve (the stand-in's ldlt() is an LU inverse): rounding level
        assert np.abs(q - q2).max() < 1e-11
    if os.environ.get("BGG_RECORD_GOLDEN"):
        common.check_golden_reference("ik_joint_angles", [list(map(float, q)) for q in ref_q] if live else
                                      [list(map(float, po.ik(kin, st[b], ee[b], guess[b])[1])) for b in range(12)])
    ee[0, 0] = [2.0, 2.0, 0.0]
    if live:
        assert po.ik(kin, st[0], ee[0], guess[0], which="ref")[0] == 1


def test_targets_from_traj_on_a_solved_trajectory():
    cfg_name = "a1_configuration"
    cfg = wl.CONFIGS[cfg_name]
    states, t0, ee0 = wl.batched_trot_inputs(cfg, 1, seed=0)
    o = common.make_oracle(cfg_name, states[0])
    for _ in range(3):
        o.solve(states[0], 0.0, ee0[0], real_time=True)
    kin, rob, dt = _kin(), wl.robot(), cfg["integrator_dt"]
    q0 = np.concatenate([states[0, :3], states[0, 6:10], NOMINAL_JOINTS])
    for time in (0.0, 0.013, 0.05, 0.12, 0.31):
        rc, q, v, f = po.targets_from_traj(o, kin, rob, time, dt, q0)
        assert rc == 0
        feet = po.kin_fk(kin, q)[0]
        want = np.array([o.ee_at(e, time) for e in range(4)])
        assert np.abs(feet - want).max() < 2e-5
        assert np.allclose(f, np.array([o.force_at(e, time) for e in range(4)]))
        assert np.all(np.abs(v) < 100)   # the reference's "Desired velocity too high!" check
        q0 = q
    assert po.targets_from_traj(o, kin, rob, 10.0, dt, q0)[0] == 3   # beyond the horizon
