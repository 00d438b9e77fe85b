"""SURVEY.md row f-4: the tasks' internal OTG on the device (csrc/osc_otg_kernels.cuh around csrc/osc_otg.h) against the
reference's own JointTask / MotionForceTask with their internal OTG left ON -- the reference's default (JointTask.h:38,
MotionForceTask.h:67): OTG_joints.cpp / OTG_6dof_cartesian.cpp + the vendored Ruckig compiled in place (oracle/_ref/libsai_ref*.so).
Desired states AND torques are compared every cycle."""
import math
import os

import numpy as np
import pytest

from oracle import sai_ref
from tests.osc_testlib import REL_TOL, TASK_POINTS, rel_err, rot_exp, sample_states

def tau_err(tau, ref):
    """relative to the robot's torque scale, with an absolute floor: once a robot sits on its goal the commanded torque is the
    rounding residue of (q - q_desired) times the gains (1e-12 Nm), and a ratio of two such numbers means nothing"""
    scale = np.maximum(np.abs(ref).max(axis=1), 1e-3)
    return (np.abs(tau - ref).max(axis=1) / scale).max()


pytestmark = pytest.mark.gpu
needs_reference_library = pytest.mark.skipif(not sai_ref.available(oriented=True), reason="needs oracle/_ref/libsai_ref_orient.so")
GOLD_OTG = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "otg_joints_reference.npz")


@pytest.fixture(autouse=True)
def reference_default_otg_on():
    from sai_primitives_b200 import batched
    batched.JointTask.DefaultParameters.use_internal_otg = True
    batched.MotionForceTask.DefaultParameters.use_internal_otg = True
    yield


def test_mirror_default_is_the_reference_default():
    import sai_primitives_b200 as sp
    robot = sp.BatchedRobot("panda", 4)
    robot.setQ(np.zeros((4, 7))); robot.setDq(np.zeros((4, 7))); robot.updateModel()
    mft = sp.MotionForceTask(robot, "end-effector"); jt = sp.JointTask(robot)
    assert mft.getInternalOtgEnabled() and jt.getInternalOtgEnabled()
    jt.disableInternalOtg()
    assert not jt.getInternalOtgEnabled()
    with pytest.raises(NotImplementedError):
        jt.enableInternalOtgJerkLimited(1.0, 2.0, 3.0)
    with pytest.raises(Exception):
        jt.enableInternalOtgAccelerationLimited(-1.0, 2.0)     # OTG_joints.cpp:50-54


@needs_reference_library
@pytest.mark.parametrize("robot_name", ["panda", "rrrr"])
def test_joint_task_with_internal_otg(robot_name):
    """config 1 with the reference's default trajectory generation: goal steps in mid-motion (collinear and not), per-joint limits
    changed on the fly, re-initialisation; the state follows the commanded motion so that the torques stay meaningful"""
    import sai_primitives_b200 as sp
    from oracle.sai_ref import RefBatch
    N = 24
    q, dq, _ = sample_states(robot_name, N)
    n = q.shape[1]
    robot = sp.BatchedRobot(robot_name, N)
    robot.setQ(q); robot.setDq(dq); robot.updateModel()
    jt = sp.JointTask(robot)
    ctrl = sp.RobotController(robot, [jt])
    rb = RefBatch(robot_name, N, oriented=True); rb.set_state(q, dq)
    ojt = rb.add_jt(otg=True); rb.finalize()
    rng = np.random.default_rng(3)
    K = 1300      # the last move (0.04 rad at >= 2 rad/s^2) lasts at most 0.29 s
    events = {0: "goal", 200: "goal", 330: "scaled", 500: "limits", 520: "goal", 700: "reinit", 760: "small_goal"}
    goal = q.copy()
    worst_des = worst_tau = 0.0
    for k in range(K):
        ev = events.get(k)
        if ev == "goal":
            goal = q + rng.uniform(-0.7, 0.7, (N, n))
        elif ev == "scaled":
            goal = q + 1.4 * (goal - q)
        elif ev == "small_goal":      # short enough to be finished (and the goal flagged as reached) before the test ends
            goal = jt.getDesiredPosition() + rng.uniform(-0.04, 0.04, (N, n))
        if ev in ("goal", "scaled", "small_goal"):
            jt.setGoalPosition(goal)
            for i in range(N):
                ojt[i].setGoalPosition(goal[i])
        if ev == "limits":
            vmax = rng.uniform(0.5, 1.5, n); amax = rng.uniform(2.0, 7.0, n)
            jt.enableInternalOtgAccelerationLimited(vmax, amax)
            for t in ojt:
                t.enableInternalOtgAccelerationLimited(vmax, amax)
        if ev == "reinit":
            ctrl.reinitializeTasks(); rb.all_controllers.reinitializeTasks()
        ctrl.updateControllerTaskModels()
        tau = ctrl.computeControlTorques()
        ref = rb.cycle()
        des = np.concatenate([jt.getDesiredPosition(), jt.getDesiredVelocity(), 1e-3 * jt.getDesiredAcceleration()], axis=1)
        odes = np.array([np.concatenate([t.getDesiredPosition(), t.getDesiredVelocity(), 1e-3 * t.getDesiredAcceleration()]) for t in ojt])
        worst_des = max(worst_des, np.abs(des - odes).max())
        worst_tau = max(worst_tau, tau_err(tau, ref))
        assert worst_des < 1e-10 and worst_tau < REL_TOL, (k, worst_des, worst_tau)
        # the robots track the desired motion (a perfect inner loop): new state for the next cycle
        q_new = des[:, :n]; dq_new = des[:, n:2 * n]
        robot.setQ(q_new); robot.setDq(dq_new); robot.updateModel(); rb.set_state(q_new, dq_new)
    flags = jt.getInternalOtgFlags()
    assert (flags & sp.capi.OTG_GOAL_REACHED).all() and not (flags & sp.capi.OTG_ERROR).any()
    assert np.abs(jt.getGoalPosition() - goal).max() == 0.0          # the goal fields still hold the user's goals


@needs_reference_library
def test_motion_force_task_with_internal_otg_in_the_flagship_hierarchy():
    """config 2 with the reference's defaults: MotionForceTask (6-dof Cartesian generator, moving reference frame for the
    orientation) + JointTask (joint generator) through RobotController"""
    import sai_primitives_b200 as sp
    from oracle.sai_ref import RefBatch
    N = 32
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    link, pt = TASK_POINTS["panda"]
    comp = (np.eye(3), np.array(pt))
    robot = sp.BatchedRobot("panda", N)
    robot.setQ(q); robot.setDq(dq); robot.updateModel()
    mft = sp.MotionForceTask(robot, link, comp); jt = sp.JointTask(robot)
    ctrl = sp.RobotController(robot, [mft, jt])
    rb = RefBatch("panda", N, oriented=True); rb.set_state(q, dq)
    omft = rb.add_mft(link, comp, otg=True); ojt = rb.add_jt(otg=True); rb.finalize()
    x0, R0 = mft.getCurrentPosition(), mft.getCurrentOrientation()
    rng = np.random.default_rng(9)
    K = 700
    events = {0: "goal", 180: "goal", 320: "goal_vel", 450: "tiny", 520: "param"}
    gx, gR, gv, gw = x0.copy(), R0.copy(), np.zeros((N, 3)), np.zeros((N, 3))
    worst_des = worst_tau = 0.0
    for k in range(K):
        ev = events.get(k)
        if ev in ("goal", "goal_vel"):
            gx = x0 + rng.uniform(-0.1, 0.1, (N, 3)); gR = np.array([R0[i] @ rot_exp(rng.uniform(-0.5, 0.5, 3)) for i in range(N)])
            gv = rng.uniform(-0.04, 0.04, (N, 3)) if ev == "goal_vel" else np.zeros((N, 3))
            gw = rng.uniform(-0.08, 0.08, (N, 3)) if ev == "goal_vel" else np.zeros((N, 3))
            jg = q + rng.uniform(-0.3, 0.3, (N, 7))
            jt.setGoalPosition(jg)
            for i in range(N):
                ojt[i].setGoalPosition(jg[i])
        elif ev == "tiny":          # below the reference's 1e-3 relative threshold: ignored by both
            gx = gx * (1.0 + 2e-4)
        elif ev == "param":         # parametrizeForceMotionSpaces resets the linear goals and the linear half of the generator
            assert mft.parametrizeForceMotionSpaces(1, (0, 0, 1)) is True
            for t in omft:
                assert t.parametrizeForceMotionSpaces(1, (0, 0, 1)) is True
            gx = mft.getGoalPosition(); gv = np.zeros((N, 3))
            assert np.abs(gx - np.array([t.getGoalPosition() for t in omft])).max() < 1e-12
        mft.setGoalPosition(gx); mft.setGoalOrientation(gR); mft.setGoalLinearVelocity(gv); mft.setGoalAngularVelocity(gw)
        for i in range(N):
            t = omft[i]
            t.setGoalPosition(gx[i]); t.setGoalOrientation(gR[i]); t.setGoalLinearVelocity(gv[i]); t.setGoalAngularVelocity(gw[i])
        ctrl.updateControllerTaskModels()
        tau = ctrl.computeControlTorques()
        ref = rb.cycle()
        des = np.concatenate([mft.getDesiredPosition(), mft.getDesiredOrientation().reshape(N, 9), mft.getDesiredLinearVelocity(), mft.getDesiredAngularVelocity(),
                              1e-3 * mft.getDesiredLinearAcceleration(), 1e-3 * mft.getDesiredAngularAcceleration()], axis=1)
        odes = np.array([np.concatenate([t.getDesiredPosition(), t.getDesiredOrientation().reshape(-1), t.getDesiredLinearVelocity(), t.getDesiredAngularVelocity(),
                                         1e-3 * t.getDesiredLinearAcceleration(), 1e-3 * t.getDesiredAngularAcceleration()]) for t in omft])
        worst_des = max(worst_des, np.abs(des - odes).max())
        worst_tau = max(worst_tau, tau_err(tau, ref))
        assert worst_des < 1e-9 and worst_tau < REL_TOL, (k, worst_des, worst_tau)
        assert (robot.status() & sp.capi.STATUS_UNHANDLED).sum() == 0
        q = q + 0.0005 * dq
        robot.setQ(q); robot.updateModel(); rb.set_state(q, dq)
    assert not (mft.getInternalOtgFlags() & sp.capi.OTG_ERROR).any()


def test_otg_on_off_round_trip_keeps_the_goals():
    import sai_primitives_b200 as sp
    N = 8
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    robot = sp.BatchedRobot("panda", N)
    robot.setQ(q); robot.setDq(dq); robot.updateModel()
    jt = sp.JointTask(robot)
    ctrl = sp.RobotController(robot, [jt])
    goal = q + 0.3
    jt.setGoalPosition(goal)
    ctrl.updateControllerTaskModels(); ctrl.computeControlTorques()
    assert np.abs(jt.getDesiredPosition() - q).max() < 1e-3          # one millisecond into the move
    jt.disableInternalOtg()
    assert np.abs(jt.getGoalPosition() - goal).max() == 0.0 and np.abs(jt.getDesiredPosition() - goal).max() == 0.0
    jt.enableInternalOtgAccelerationLimited(math.pi / 3, 2 * math.pi)
    assert np.abs(jt.getGoalPosition() - goal).max() == 0.0 and np.abs(jt.getDesiredPosition() - q).max() < 1e-12


def test_joint_task_otg_reproduces_the_stored_reference_trajectory():
    """tests/golden/otg_joints_reference.npz: the reference's vendored Ruckig under the JointTask defaults (acceleration
    limited, pi/3 rad/s, 2 pi rad/s^2, 1 ms) with goal changes in mid-motion, replayed by the device's JointTask generator
    cycle by cycle (tests/golden/generate_otg_reference.py wrote it)"""
    import sai_primitives_b200 as sp
    d = np.load(GOLD_OTG)
    N, K, n = 3, d["pos"].shape[0], d["q0"].size
    q = np.tile(d["q0"], (N, 1))
    robot = sp.BatchedRobot("panda", N)
    robot.setQ(q); robot.setDq(np.zeros((N, n))); robot.updateModel()
    jt = sp.JointTask(robot)
    ctrl = sp.RobotController(robot, [jt])
    goal_at = {int(s): g for g, s in zip(d["goals"], d["goal_steps"])}
    worst = 0.0
    for k in range(K):
        if k in goal_at:
            jt.setGoalPosition(np.tile(goal_at[k], (N, 1)))
        ctrl.updateControllerTaskModels()
        ctrl.computeControlTorques()
        p, v, a = jt.getDesiredPosition(), jt.getDesiredVelocity(), jt.getDesiredAcceleration()
        worst = max(worst, np.abs(p - d["pos"][k]).max(), np.abs(v - d["vel"][k]).max(), 1e-3 * np.abs(a - d["acc"][k]).max())
        assert worst < 1e-10, (k, worst)
        robot.setQ(p); robot.setDq(v); robot.updateModel()      # the robots track the desired motion
    flags = jt.getInternalOtgFlags()
    assert (flags & sp.capi.OTG_GOAL_REACHED).all() and not (flags & sp.capi.OTG_ERROR).any()
    assert (robot.status() & sp.capi.STATUS_UNHANDLED).sum() == 0
