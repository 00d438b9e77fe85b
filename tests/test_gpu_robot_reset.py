"""Per-robot controller resets (osc_reset_robots): re-initialise (TemplateTask::reInitializeTask) or rebuild (the state the task
constructors leave) the tasks of selected robots of a batch between cycles.  Checked against the reference's control law with one
oracle robot per GPU robot, against twin handles that never reset (unselected robots, bit for bit) and against handles freshly
created at the reset state (construct mode, bit for bit)."""
import os

import numpy as np
import pytest

from tests.osc_testlib import REL_TOL, TASK_POINTS, OracleBatch, rel_err, rng_for, rot_exp, sample_states

gpu = pytest.mark.gpu
REINIT, CONSTRUCT = 0, 1

MFT_FIELDS = list(range(0, 21)) + list(range(40, 46))
JT_FIELDS = list(range(32, 39))


# ---- host-side mask conversion (no device needed)
def test_robot_mask_conversion():
    from sai_primitives_b200.batched import robot_mask
    N = 6
    assert robot_mask(None, N) is None
    m = robot_mask(np.array([True, False, True, False, False, True]), N)
    assert m.dtype == np.int32 and m.flags["C_CONTIGUOUS"] and m.tolist() == [1, 0, 1, 0, 0, 1]
    assert robot_mask([0, 2, 5], N).tolist() == [1, 0, 1, 0, 0, 1]
    assert robot_mask(np.array([5, 5, 0], dtype=np.int64), N).tolist() == [1, 0, 0, 0, 0, 1]
    assert robot_mask([], N).tolist() == [0] * N
    for bad in ([6], [-1], [0, 7], np.zeros(5, bool), np.zeros((2, 3), bool), [0.5, 1.0], [[0, 1]], [True, 2], [2, False],
                np.zeros((0, 3)), np.zeros((0, 3), np.int32)):
        with pytest.raises(ValueError):
            robot_mask(bad, N)


# ---- helpers
def _sp():
    import sai_primitives_b200 as sp
    return sp


def _dev_i32(a):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(torch.device("cuda", 0))
    torch.cuda.synchronize()
    return t


def _snapshot(robot, tasks):
    """every readable per-robot field of every task, the generator flags and the status words"""
    sp = _sp()
    out = []
    for t in tasks:
        fields = MFT_FIELDS if t.task_type == sp.capi.OSC_TASK_MOTION_FORCE else JT_FIELDS
        out += [t._get(f) for f in fields]
        if t.getInternalOtgEnabled():
            out.append(t.getInternalOtgFlags())
    out.append(robot.status())
    return out


def _rows_equal(a, b, rows):
    return all(np.array_equal(x[rows], y[rows]) for x, y in zip(a, b))


def _teleport(q, dq, sel, first_index):
    """new states for the selected rows, drawn from another range of robot indices"""
    q2, dq2, _ = sample_states("panda", len(q), min_sigma_ratio=0.1, first_index=first_index)
    qn, dqn = q.copy(), dq.copy()
    qn[sel], dqn[sel] = q2[sel], dq2[sel]
    return qn, dqn


class Panda2:
    """Panda, full six-dof MotionForceTask + JointTask in its null space (config 2), integral gains on, per-robot goals"""

    GAINS = ((120.0, 22.0, 4.0), (200.0, 28.0, 3.0), (50.0, 14.0, 2.0))

    def __init__(self, q, dq, otg=False, env=None):
        sp = _sp()
        self.N, self.n = q.shape
        link, pt = TASK_POINTS["panda"]
        self.comp = (np.eye(3), np.array(pt))
        old = {k: os.environ.get(k) for k in (env or {})}
        os.environ.update(env or {})
        try:
            self.robot = sp.BatchedRobot("panda", self.N)
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        self.move(q, dq)
        self.mft = sp.MotionForceTask(self.robot, link, self.comp)
        self.jt = sp.JointTask(self.robot)
        if otg:
            self.mft.enableInternalOtgAccelerationLimited(0.3, 2.0, np.pi / 3, 2 * np.pi)
            self.jt.enableInternalOtgAccelerationLimited(np.pi / 3, 2 * np.pi)
        g = self.GAINS
        self.mft.setPosControlGains(*g[0]); self.mft.setOriControlGains(*g[1]); self.jt.setGains(*g[2])
        self.tasks = [self.mft, self.jt]
        self.ctrl = sp.RobotController(self.robot, self.tasks)

    def move(self, q, dq):
        self.q, self.dq = q, dq
        self.robot.setQ(q); self.robot.setDq(dq); self.robot.updateModel()

    def set_goals(self, goals):
        xd, Rd, gq = goals
        self.mft.setGoalPosition(xd); self.mft.setGoalOrientation(Rd); self.jt.setGoalPosition(gq)

    def cycle(self):
        self.ctrl.updateControllerTaskModels()
        return self.ctrl.computeControlTorques()


def _goals(x0, R0, q, stream):
    N = len(q)
    xd = np.zeros((N, 3)); Rd = np.zeros((N, 3, 3)); gq = np.zeros_like(q)
    for i in range(N):
        g = rng_for(i, stream=stream)
        xd[i] = x0[i] + g.uniform(-0.05, 0.05, 3); Rd[i] = R0[i] @ rot_exp(g.uniform(-0.2, 0.2, 3))
        gq[i] = q[i] + g.uniform(-0.2, 0.2, q.shape[1])
    return xd, Rd, gq


def _oracle(q, dq, goals, rows):
    """oracle robots for `rows`, built at state (q, dq) with Panda2's configuration and goals"""
    link, pt = TASK_POINTS["panda"]
    ob = OracleBatch("panda", len(rows)); ob.set_state(q[rows], dq[rows])
    omft = ob.add_mft(link, (np.eye(3), np.array(pt))); ojt = ob.add_jt(); ob.finalize()
    g = Panda2.GAINS
    for r, i in enumerate(rows):
        omft[r].setPosControlGains(*[np.full(3, v) for v in g[0]]); omft[r].setOriControlGains(*[np.full(3, v) for v in g[1]])
        ojt[r].setGains(*[np.full(q.shape[1], v) for v in g[2]])
        if goals is not None:
            omft[r].setGoalPosition(goals[0][i]); omft[r].setGoalOrientation(goals[1][i]); ojt[r].setGoalPosition(goals[2][i])
    return ob, omft, ojt


# ---- 1 and 3: both modes against the oracle
@gpu
@pytest.mark.parametrize("split", ["0", "1"])
@pytest.mark.parametrize("filtered", [True, False])
@pytest.mark.parametrize("mode", [REINIT, CONSTRUCT])
def test_reset_against_the_oracle(mode, filtered, split):
    """Run 20 cycles, teleport a third of the robots, reset them through a device mask, run 20 more.  The oracle's robots call
    reInitializeTask on each task (re-initialise mode: the singularity handler keeps its history) or are built anew at the new
    state (construct mode).  Unfiltered states put robots inside the singularity band, where the two differ."""
    N = 64
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1 if filtered else None)
    c = Panda2(q, dq, env={"SAI_B200_BLEND_SPLIT": split})
    goals = _goals(c.mft.getCurrentPosition(), c.mft.getCurrentOrientation(), q, stream=60)
    c.set_goals(goals)
    ob, omft, ojt = _oracle(q, dq, goals, np.arange(N))
    dt = 0.001
    for k in range(20):
        assert rel_err(c.cycle(), ob.cycle()).max() < REL_TOL, k
        c.move(c.q + dt * c.dq, c.dq); ob.set_state(c.q, c.dq)
    sel = np.zeros(N, bool); sel[::3] = True
    if filtered:
        qn, dqn = _teleport(c.q, c.dq, sel, first_index=5000)
    else:
        q2, dq2, _ = sample_states("panda", N, first_index=5000)
        qn, dqn = c.q.copy(), c.dq.copy(); qn[sel], dqn[sel] = q2[sel], dq2[sel]
    c.move(qn, dqn); ob.set_state(qn, dqn)
    mask = _dev_i32(sel)
    (c.ctrl.reinitializeTasksDevice if mode == REINIT else c.ctrl.resetRobotsDevice)(mask.data_ptr())
    rows = np.flatnonzero(sel)
    om, oj = list(omft), list(ojt)
    if mode == REINIT:
        for i in rows:
            omft[i].reInitializeTask(); ojt[i].reInitializeTask()
        fresh = None
    else:
        fresh, fm, fj = _oracle(qn, dqn, None, rows)
        for r, i in enumerate(rows):
            om[i], oj[i] = fm[r], fj[r]
    gp = c.mft.getGoalPosition(); jgp = c.jt.getGoalPosition()
    assert np.array_equal(gp[sel], c.mft.getCurrentPosition()[sel])
    assert np.abs(jgp[sel] - qn[sel]).max() == 0.0
    assert np.array_equal(gp[~sel], goals[0][~sel]) and np.array_equal(jgp[~sel], goals[2][~sel])
    in_band = 0
    for k in range(20):
        tau = c.cycle()
        ref = ob.cycle()
        if fresh is not None:
            ref[rows] = fresh.cycle()
        st = c.robot.status()
        assert (st & _sp().capi.STATUS_UNHANDLED).sum() == 0
        assert rel_err(tau, ref).max() < REL_TOL, k
        _check_fields(c, om, oj, k)
        in_band += _check_status(st, om, rows)
        c.move(c.q + dt * c.dq, c.dq); ob.set_state(c.q, c.dq)
        if fresh is not None:
            fresh.set_state(c.q[rows], c.dq[rows])
    if not filtered:
        assert in_band > 0   # selected robots went through the singularity handler after their reset


def _attr(t, name, *fallback):
    """an oracle member: an attribute of the numpy restatement, a method of the reference's proxy (the first of the names the
    object has)"""
    for n in (name,) + fallback:
        if hasattr(t, n):
            v = getattr(t, n)
            break
    return np.asarray(v() if callable(v) else v, dtype=np.float64).reshape(-1)


def _close(a, b, what):
    b = np.asarray(b)
    assert np.abs(a - b).max() <= 1e-9 * max(1e-3, np.abs(b).max()), (what, np.abs(a - b).max())


def _check_fields(c, om, oj, k):
    """goals, current pose and integrators of both tasks, every robot, against its oracle robot"""
    cap = _sp().capi
    _close(c.mft._get(cap.MFT_GOAL_POSITION), [_attr(t, "getGoalPosition", "_goal_position") for t in om], ("goal position", k))
    _close(c.mft._get(cap.MFT_GOAL_ORIENTATION), [_attr(t, "getGoalOrientation", "_goal_orientation") for t in om], ("goal orientation", k))
    _close(c.mft._get(cap.MFT_CURRENT_POSITION), [_attr(t, "getCurrentPosition") for t in om], ("current position", k))
    _close(c.mft._get(cap.MFT_CURRENT_ORIENTATION), [_attr(t, "getCurrentOrientation") for t in om], ("current orientation", k))
    _close(c.mft._get(cap.MFT_INTEGRATED_POSITION_ERROR), [_attr(t, "_integrated_position_error") for t in om], ("mft integrator", k))
    _close(c.mft._get(cap.MFT_INTEGRATED_ORIENTATION_ERROR), [_attr(t, "_integrated_orientation_error") for t in om], ("mft ori integrator", k))
    _close(c.jt._get(cap.JT_GOAL_POSITION), [_attr(t, "getGoalPosition", "_goal_position") for t in oj], ("joint goal", k))
    _close(c.jt._get(cap.JT_INTEGRATED_POSITION_ERROR), [_attr(t, "_integrated_position_error") for t in oj], ("joint integrator", k))


def _check_status(st, om, rows):
    """singular-path and joint-strategy status bits against the oracle's singularity handler (the strategy is type 1 when the
    handler's type-1 counter exceeds its type-2 counter); returns how many selected robots were inside the band"""
    cap = _sp().capi
    h = [t._singularity_handler for t in om]
    sing = np.array([len(x._singularity_types) != 0 for x in h])
    c1 = np.array([int(x._type_1_counter) for x in h]); c2 = np.array([int(x._type_2_counter) for x in h])
    t1, t2 = (st & cap.STATUS_TYPE1) != 0, (st & cap.STATUS_TYPE2) != 0
    assert ((st & cap.STATUS_SINGULAR_PATH) != 0)[sing].all()
    assert np.array_equal(t1[sing], (c1 > c2)[sing]) and np.array_equal(t2[sing], (c1 <= c2)[sing])
    assert not (t1 | t2)[~sing].any()
    return int(sing[rows].sum())


# ---- 2: construct mode with closed-loop force, POPC and per-robot configuration
XYZ = [(1, 0, 0), (0, 1, 0), (0, 0, 1)]


def _config3(tasks, r, kp, fdim, clf):
    """robot r's configuration on an oracle MotionForceTask / JointTask pair, in the order the GPU handle gets it"""
    omft, ojt = tasks
    omft.setPosControlGains(kp[r], np.full(3, 20.0), np.full(3, 2.0)); omft.setOriControlGains(np.full(3, 150.0), np.full(3, 22.0), np.full(3, 1.0))
    omft.setForceControlGains(0.8, 12.0, 1.5)
    omft.enablePassivity()
    omft.parametrizeForceMotionSpaces(int(fdim[r]), (0.0, 0.0, 1.0))
    omft.setClosedLoopForceControl(bool(clf[r]))
    omft.setGoalForce(np.array([0.0, 0.0, -5.0]))
    ojt.setGains(np.full(7, 60.0), np.full(7, 12.0), np.full(7, 1.0))


@gpu
def test_construct_with_passivity_against_the_oracle():
    """Config 3 (partial xyz MotionForceTask + JointTask, closed-loop force with POPC and a 512-sample ring, sensed forces of
    ex09), per-robot position gains, per-robot force spaces and closed-loop flags.  After 70 cycles a third of the robots are
    teleported and reset in construct mode; the oracle builds those robots anew at the new state with the same configuration,
    the others carry on.  Torques and the POPC state of every robot are compared on each of the 130 cycles that follow, while
    the sensed-force noise makes the passivity controller engage; gains, spaces and flags survive the reset."""
    from tests.osc_testlib import sensed_ex09
    sp = _sp()
    N = 96
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    link, pt = TASK_POINTS["panda"]
    comp = (np.eye(3), np.array(pt))
    i = np.arange(N)
    kp = np.array([rng_for(r, stream=70).uniform(80, 200, 3) for r in range(N)])
    fdim = np.where(i % 3 != 2, 1, 0).astype(np.int32)
    clf = (fdim == 1) & (i % 4 != 3)
    robot = sp.BatchedRobot("panda", N)
    robot.setQ(q); robot.setDq(dq); robot.updateModel()
    mft = sp.MotionForceTask(robot, link, comp, XYZ, []); jt = sp.JointTask(robot)
    ctrl = sp.RobotController(robot, [mft, jt])
    mft.setPosControlGains(kp, 20.0, 2.0); mft.setOriControlGains(150.0, 22.0, 1.0)
    mft.setForceControlGains(0.8, 12.0, 1.5)
    mft.enablePassivity(512)
    mft.parametrizeForceMotionSpaces(fdim, np.tile([0.0, 0.0, 1.0], (N, 1)))
    mft.setClosedLoopForceControl(clf)
    mft.setGoalForce(np.array([0.0, 0.0, -5.0]))
    jt.setGains(60.0, 12.0, 1.0)

    def oracle(qs, dqs, rows):
        ob = OracleBatch("panda", len(rows)); ob.set_state(qs[rows], dqs[rows])
        om = ob.add_mft(link, comp, XYZ, []); oj = ob.add_jt(); ob.finalize()
        for r, k in enumerate(rows):
            _config3((om[r], oj[r]), k, kp, fdim, clf)
        return ob, om, oj

    ob, om, oj = oracle(q, dq, i)
    dt = 0.001
    om_all = list(om)

    def cycle(k, fresh, rows):
        F, Mo = sensed_ex09(N, k)
        mft.updateSensedForceAndMoment(F, Mo)
        for r in range(N):
            om[r].updateSensedForceAndMoment(F[r], Mo[r])
        if fresh is not None:
            for r, j in enumerate(rows):
                fresh[1][r].updateSensedForceAndMoment(F[j], Mo[j])
        ctrl.updateControllerTaskModels()
        tau = ctrl.computeControlTorques()
        ref = ob.cycle()
        if fresh is not None:
            ref[rows] = fresh[0].cycle()
        assert (robot.status() & sp.capi.STATUS_UNHANDLED).sum() == 0
        assert rel_err(tau, ref).max() < REL_TOL, k
        popc = mft._get(sp.capi.MFT_POPC_STATE)
        pv = [t._POPC_force for t in om_all]
        ref_popc = np.array([[p._passivity_observer_value, p._E_correction, p._Rc, p._vcl_squared_sum] for p in pv])
        assert (np.abs(popc - ref_popc) <= 1e-9 * np.maximum(1.0, np.abs(ref_popc))).all(), k
        return popc

    qk = q.copy()
    for k in range(70):
        cycle(k, None, None)
        qk = qk + dt * dq
        robot.setQ(qk); robot.setDq(dq); robot.updateModel(); ob.set_state(qk, dq)
    g0, s0 = mft.getPosControlGains(), mft.getForceMotionSpaces()
    sel = np.zeros(N, bool); sel[1::3] = True
    rows = np.flatnonzero(sel)
    qn, dqn = _teleport(qk, dq, sel, first_index=17000)
    robot.setQ(qn); robot.setDq(dqn); robot.updateModel(); ob.set_state(qn, dqn)
    ctrl.resetRobots(sel)
    after = mft._get(sp.capi.MFT_POPC_STATE)
    assert np.array_equal(after[sel], np.tile([0.0, 0.0, 1.0, 0.0], (sel.sum(), 1)))
    mft.setGoalForce(np.array([0.0, 0.0, -5.0]))   # the construct reset zeroed the selected robots' goals, as a new task has them
    fresh = oracle(qn, dqn, rows)
    for r, j in enumerate(rows):
        om_all[j] = fresh[1][r]
    engaged = np.zeros(N, bool)
    qk, dqk = qn.copy(), dqn.copy()
    for k in range(70, 200):
        popc = cycle(k, fresh, rows)
        engaged |= popc[:, 2] != 1.0
        qk = qk + dt * dqk
        robot.setQ(qk); robot.setDq(dqk); robot.updateModel(); ob.set_state(qk, dqk); fresh[0].set_state(qk[rows], dqk[rows])
    assert engaged[sel & clf].any() and engaged[~sel & clf].any()   # the passivity controller acted on both groups
    for a, b in zip(mft.getPosControlGains(), g0):
        assert np.array_equal(a, b)
    for a, b in zip(mft.getForceMotionSpaces(), s0):
        assert np.array_equal(np.asarray(a), np.asarray(b))


# ---- 4: unselected robots are untouched
def _build(model, N, q, dq, hier):
    sp = _sp()
    link, pt = TASK_POINTS[model]
    comp = (np.eye(3), np.array(pt))
    robot = sp.BatchedRobot(model, N)
    robot.setQ(q); robot.setDq(dq); robot.updateModel()
    n = robot.dof()
    xyz = [(1, 0, 0), (0, 1, 0), (0, 0, 1)]
    if hier == "mft":
        tasks = [sp.MotionForceTask(robot, link, comp)]
    elif hier == "mft_jt":
        tasks = [sp.MotionForceTask(robot, link, comp), sp.JointTask(robot)]
    elif hier == "jt":
        tasks = [sp.JointTask(robot)]
    elif hier == "partial_jt":
        S = np.zeros((2, n)); S[0, 0] = 1; S[1, n - 1] = 1
        tasks = [sp.JointTask(robot, S, task_name="partial_joint_task"), sp.MotionForceTask(robot, link, comp)]
    else:  # two motion-force tasks
        tasks = [sp.MotionForceTask(robot, link, comp, xyz, [], task_name="position"),
                 sp.MotionForceTask(robot, link, comp, [], xyz, task_name="orientation"), sp.JointTask(robot)]
    for t in tasks:
        if t.task_type == sp.capi.OSC_TASK_JOINT:
            t.enableInternalOtgAccelerationLimited(np.pi / 3, 2 * np.pi)
            t.setGains(60.0, 12.0, 1.5)
        else:
            t.enableInternalOtgAccelerationLimited(0.3, 2.0, np.pi / 3, 2 * np.pi)
            t.setPosControlGains(120.0, 22.0, 3.0); t.setOriControlGains(200.0, 28.0, 2.0)
    ctrl = sp.RobotController(robot, tasks)
    ctrl.enableJointLimitAvoidance(True); ctrl.enableGravityCompensation(True); ctrl.enableTorqueSaturation(True)
    for i, t in enumerate(tasks):
        if t.task_type == sp.capi.OSC_TASK_JOINT:
            k = t.getTaskDof()
            t.setGoalPosition(t.getGoalPosition() + np.array([rng_for(r, stream=80 + i).uniform(-0.2, 0.2, k) for r in range(N)]))
        else:
            t.setGoalPosition(t.getGoalPosition() + np.array([rng_for(r, stream=80 + i).uniform(-0.05, 0.05, 3) for r in range(N)]))
    return robot, tasks, ctrl


@gpu
@pytest.mark.parametrize("mode", [REINIT, CONSTRUCT])
@pytest.mark.parametrize("model,hier", [("panda", "mft_jt"), ("puma_like", "mft"), ("rrrr", "jt"),
                                        ("panda_sliding_base", "partial_jt"), ("panda", "two_mft")])
def test_unselected_robots_are_untouched(model, hier, mode):
    N = 200
    q, dq, _ = sample_states(model, N)
    A = _build(model, N, q, dq, hier)
    B = _build(model, N, q, dq, hier)
    dt = 0.001
    for k in range(5):
        for h in (A, B):
            h[2].updateControllerTaskModels(); h[2].computeControlTorques()
            h[0].setQ(q + dt * (k + 1) * dq); h[0].setDq(dq); h[0].updateModel()
    qk = q + dt * 5 * dq
    sel = np.zeros(N, bool); sel[np.array([rng_for(i, stream=90).random() < 0.3 for i in range(N)])] = True
    q2, dq2, _ = sample_states(model, N, first_index=7000)
    qa, dqa = qk.copy(), dq.copy(); qa[sel], dqa[sel] = q2[sel], dq2[sel]
    A[0].setQ(qa); A[0].setDq(dqa); A[0].updateModel()
    before = _snapshot(A[0], A[1])
    (A[2].reinitializeTasks if mode == REINIT else A[2].resetRobots)(sel)
    after = _snapshot(A[0], A[1])
    assert _rows_equal(before, after, ~sel)
    assert not _rows_equal(before, after, sel)
    for k in range(10):
        ta = (A[2].updateControllerTaskModels(), A[2].computeControlTorques())[1]
        tb = (B[2].updateControllerTaskModels(), B[2].computeControlTorques())[1]
        assert np.array_equal(ta[~sel], tb[~sel]), k
        assert _rows_equal(_snapshot(*A[:2]), _snapshot(*B[:2]), ~sel), k
        qa = qa + dt * dqa; qb = qk + dt * (k + 1) * dq
        qa[~sel] = qb[~sel]
        A[0].setQ(qa); A[0].setDq(dqa); A[0].updateModel(); B[0].setQ(qb); B[0].setDq(dq); B[0].updateModel()


# ---- 5: construct mode equals a new handle
@gpu
@pytest.mark.parametrize("otg", [False, True])
def test_construct_equals_a_new_handle(otg):
    sp = _sp()
    N = 256
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    a = Panda2(q, dq, otg=otg)
    a.set_goals(_goals(a.mft.getCurrentPosition(), a.mft.getCurrentOrientation(), q, stream=61))
    dt = 0.001
    for k in range(10):
        a.cycle(); a.move(a.q + dt * a.dq, a.dq)
    sel = np.zeros(N, bool); sel[::2] = True
    qn, dqn = _teleport(a.q, a.dq, sel, first_index=9000)
    a.move(qn, dqn)
    a.ctrl.resetRobots(sel)
    b = Panda2(qn, dqn, otg=otg)
    goals = _goals(b.mft.getCurrentPosition(), b.mft.getCurrentOrientation(), qn, stream=62)
    a.set_goals(goals); b.set_goals(goals)
    desired = [sp.capi.MFT_DESIRED_POSITION, sp.capi.MFT_DESIRED_ORIENTATION, sp.capi.MFT_DESIRED_LINEAR_VELOCITY]
    for k in range(30):
        ta, tb = a.cycle(), b.cycle()
        assert np.array_equal(ta[sel], tb[sel]), k
        for f in desired:
            assert np.array_equal(a.mft._get(f)[sel], b.mft._get(f)[sel]), (k, f)
        assert np.array_equal(a.jt._get(sp.capi.JT_DESIRED_POSITION)[sel], b.jt._get(sp.capi.JT_DESIRED_POSITION)[sel]), k
        if otg:
            assert np.array_equal(a.mft.getInternalOtgFlags()[sel], b.mft.getInternalOtgFlags()[sel]), k
            assert np.array_equal(a.jt.getInternalOtgFlags()[sel], b.jt.getInternalOtgFlags()[sel]), k
        qn = qn + dt * dqn
        a.move(qn, dqn); b.move(qn, dqn)


# ---- 6: mask forms and edge cases
@gpu
def test_mask_forms_and_edge_cases():
    sp = _sp()
    lib = sp.capi.load_library()
    N = 128
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    hs = [Panda2(q, dq, otg=True) for _ in range(2)]
    for h in hs:
        h.set_goals(_goals(h.mft.getCurrentPosition(), h.mft.getCurrentOrientation(), q, stream=63))
        for k in range(5):
            h.cycle(); h.move(h.q + 0.001 * h.dq, h.dq)
    a, b = hs
    qn, dqn = _teleport(a.q, a.dq, np.arange(N) % 3 == 1, first_index=11000)
    a.move(qn, dqn); b.move(qn, dqn)
    same = lambda: all(np.array_equal(x, y) for x, y in zip(_snapshot(a.robot, a.tasks), _snapshot(b.robot, b.tasks)))
    assert same()
    # an all-zero mask changes nothing, in either mode, host or device
    base = _snapshot(a.robot, a.tasks)
    z = _dev_i32(np.zeros(N))
    a.ctrl.resetRobots(np.zeros(N, bool)); a.ctrl.reinitializeTasks([]); a.ctrl.resetRobotsDevice(z.data_ptr()); a.mft.reInitializeTaskDevice(z.data_ptr())
    assert all(np.array_equal(x, y) for x, y in zip(base, _snapshot(a.robot, a.tasks)))
    # bad arguments fail without writing
    for args in ((5, None, 0, 0), (0, None, 0, 2), (0, None, 2, 0), (-1, None, 0, -1)):
        assert lib.osc_reset_robots(a.robot.handle, *args) == sp.capi.OSC_ERR_INVALID_ARGUMENT
    launches = a.robot.launchCount()
    with pytest.raises(ValueError):
        a.ctrl.resetRobots([0, N])
    with pytest.raises(ValueError):
        a.mft.reInitializeTask(np.ones(N - 1, bool))
    assert a.robot.launchCount() == launches
    assert all(np.array_equal(x, y) for x, y in zip(base, _snapshot(a.robot, a.tasks)))
    # NULL in re-initialise mode is osc_reinitialize_task
    assert lib.osc_reinitialize_task(a.robot.handle, -1) == 0
    b.ctrl.reinitializeTasks()
    assert same()
    # host mask == device mask, bool == indices
    sel = np.arange(N) % 5 == 2
    a.ctrl.resetRobots(sel)
    b.ctrl.resetRobotsDevice(_dev_i32(sel).data_ptr())
    assert same()
    a.ctrl.reinitializeTasks(np.flatnonzero(sel))
    d = _dev_i32(sel * 7)  # any non-zero value selects
    b.ctrl.reinitializeTasksDevice(d.data_ptr())
    assert same()
    # task_id = -1 equals each task in turn
    a.ctrl.reinitializeTasks(sel)
    for t in b.tasks:
        t.reInitializeTask(sel)
    assert same()
    for k in range(3):
        assert np.array_equal(a.cycle(), b.cycle())


# ---- 7: ordering with asynchronous device cycles
def _ordering_run(q, dq, qn, dqn, mask, pipelined, fp32):
    import torch
    sp = _sp()
    c = Panda2(q, dq, env=None if pipelined else {"SAI_B200_NO_PIPELINE": "1"})
    c.set_goals(_goals(c.mft.getCurrentPosition(), c.mft.getCurrentOrientation(), q, stream=64))
    if fp32:
        c.ctrl.setPrecision("fp32")
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a.T)).to(dev)
    d_q, d_dq, d_qn, d_dqn = t(q), t(dq), t(qn), t(dqn)
    d_tau = torch.zeros((7, len(q)), dtype=torch.float64, device=dev)
    taus = []
    torch.cuda.synchronize()
    for k in range(12):
        if k == 6:
            c.robot.setStateDevice(d_qn.data_ptr(), d_dqn.data_ptr())
            c.ctrl.resetRobotsDevice(mask.data_ptr())
        if k in (8, 10):
            c.mft.reInitializeTaskDevice(mask.data_ptr())
        src = (d_q, d_dq) if k < 6 else (d_qn, d_dqn)
        c.ctrl.stepDevice(src[0].data_ptr(), src[1].data_ptr(), d_tau.data_ptr())
        if not pipelined:
            c.robot.sync()
        if k % 3 == 2:
            c.robot.sync()
            taus.append(d_tau.cpu().numpy().copy())
    c.robot.sync()
    return taus + [f for f in _snapshot(c.robot, c.tasks)]


@gpu
@pytest.mark.parametrize("fp32", [False, True])
def test_reset_between_asynchronous_cycles(fp32):
    N = 4096
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    sel = np.zeros(N, bool); sel[np.arange(0, N, 7)] = True
    qn, dqn = _teleport(q, dq, sel, first_index=13000)
    mask = _dev_i32(sel)
    a = _ordering_run(q, dq, qn, dqn, mask, True, fp32)
    b = _ordering_run(q, dq, qn, dqn, mask, False, fp32)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


# ---- 9: closed loop with episode resets
def _episodes(reset, N=256, episodes=3, cycles=100):
    """BatchedSimulation + OTG on: every `cycles` cycles, random robots get a new start state and goal (and, with `reset`, a
    construct reset).  Returns the per-episode start offsets and end errors to the goals and the first-cycle torque norms of the
    teleported robots."""
    sp = _sp()
    link, pt = TASK_POINTS["panda"]
    dt = 0.005
    q, _, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    dq = np.zeros_like(q)
    robot = sp.BatchedRobot("panda", N)
    robot.setQ(q); robot.setDq(dq); robot.updateModel()
    mft = sp.MotionForceTask(robot, link, (np.eye(3), np.array(pt)), loop_timestep=dt)
    jt = sp.JointTask(robot, loop_timestep=dt)
    for t in (mft, jt):
        assert not t.getInternalOtgEnabled()
    mft.enableInternalOtgAccelerationLimited(0.3, 2.0, np.pi / 3, 2 * np.pi)
    jt.enableInternalOtgAccelerationLimited(np.pi / 3, 2 * np.pi)
    ctrl = sp.RobotController(robot, [mft, jt])
    ctrl.enableGravityCompensation(True)
    sim = sp.BatchedSimulation(robot, q, dq, timestep=dt)
    start_x = mft.getCurrentPosition()

    def offsets(e):
        return np.array([rng_for(i, stream=100 + e).uniform(-0.01, 0.01, 3) for i in range(N)])

    goal = start_x + offsets(0)
    mft.setGoalPosition(goal); jt.setGoalPosition(q)
    start_err = np.linalg.norm(goal - start_x, axis=1)
    moved = np.ones(N, bool)
    out = []
    for e in range(episodes):
        first = None
        for k in range(cycles):
            qs, dqs = sim.getJointPositions(), sim.getJointVelocities()
            tau = ctrl.step(qs, dqs)
            if k == 0:
                first = np.linalg.norm(tau - robot.evalModel(link)["g"], axis=1)
            sim.setJointTorques(tau); sim.integrate()
        x = mft.getCurrentPosition()
        out.append((start_err[moved], np.linalg.norm(x - goal, axis=1)[moved], first[moved]))
        # next episode: a random third of the robots start over somewhere else with a new goal
        moved = np.array([rng_for(i, stream=120 + e).random() < 0.33 for i in range(N)])
        qn, _, _ = sample_states("panda", N, min_sigma_ratio=0.1, first_index=20000 + 1000 * e)
        sim.setJointPositions(qn[moved], robots=moved)
        sim.setJointVelocities(np.zeros((int(moved.sum()), 7)), robots=np.flatnonzero(moved))
        robot.setQ(sim.getJointPositions()); robot.setDq(sim.getJointVelocities()); robot.updateModel()
        if reset:
            ctrl.resetRobots(moved)
        x0 = mft.getCurrentPosition()
        goal = goal.copy(); goal[moved] = x0[moved] + offsets(e + 1)[moved]
        mft.setGoalPosition(goal)
        gq = jt.getGoalPosition()
        gq[moved] = sim.getJointPositions()[moved]
        jt.setGoalPosition(gq)
        start_err = np.linalg.norm(goal - x0, axis=1)
    return out


@gpu
def test_closed_loop_episode_resets():
    with_reset = _episodes(True)
    for e, (s, end, _) in enumerate(with_reset):
        print("episode %d: start offset max %.2e m, end error max %.2e m" % (e, s.max(), end.max()))
        assert (end < 3e-4).all(), (e, end.max())   # offsets up to 1.7 cm, every robot within 0.3 mm at the episode's end
    without = _episodes(False)
    # the teleported robots of the loop without the reset start with the generator still where they used to be
    ratio = np.median(without[1][2]) / np.median(with_reset[1][2])
    print("first-cycle torque ratio after a teleport, no reset / construct reset (median over robots): %.1f" % ratio)
    assert ratio > 5.0


# ---- 8: the C++ mirror
@gpu
def test_cpp_mirror_robot_reset(tmp_path):
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = tmp_path / "robot_reset_demo"
    libdir = os.path.join(root, "sai_primitives_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(root, "include"),
                           os.path.join(root, "tests", "cpp", "robot_reset_demo.cpp"), "-o", str(exe),
                           "-L", libdir, "-lsai_b200_osc", "-Wl,-rpath," + libdir])
    N = 64
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    sel = np.arange(N) % 3 == 0
    q2, dq2 = _teleport(q, dq, sel, first_index=15000)
    files = []
    for name, (a, b) in (("s1.bin", (q, dq)), ("s2.bin", (q2, dq2))):
        p = tmp_path / name
        p.write_bytes(np.ascontiguousarray(a.T).tobytes() + np.ascontiguousarray(b.T).tobytes())
        files.append(str(p))
    m = tmp_path / "mask.bin"
    m.write_bytes(sel.astype(np.int32).tobytes())
    out = tmp_path / "tau.bin"
    r = subprocess.run([str(exe), files[0], files[1], str(m), str(N), str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert "0 unhandled" in r.stdout
    tau = np.fromfile(out, dtype=np.float64).reshape(7, N).T
    link, pt = TASK_POINTS["panda"]
    ob = OracleBatch("panda", N); ob.set_state(q, dq)
    omft = ob.add_mft(link, (np.eye(3), np.array(pt))); ojt = ob.add_jt(); ob.finalize()
    for a, b in zip(omft, ojt):
        a.setGoalLinearVelocity((0.01, -0.02, 0.03)); b.setGoalVelocity(np.full(7, 0.1))
    for _ in range(3):
        ob.cycle()
    ob.set_state(q2, dq2)
    for i in np.flatnonzero(sel):
        omft[i].reInitializeTask(); ojt[i].reInitializeTask()
    for _ in range(3):
        ref = ob.cycle()
    assert rel_err(tau, ref).max() < REL_TOL
