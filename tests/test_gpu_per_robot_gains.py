"""Per-robot PID gains (osc_set_gains): every robot of a handle with its own JointTask / MotionForceTask gains, on every
cycle path -- the specialised fused kernels (their per-robot instantiations), the non-specialised and general-hierarchy kernels,
the single and the split blending path -- against the reference's control law with one oracle robot per GPU robot, each given
its own gains through the reference setters.  Integral gains are non-zero throughout, so the integrators carry the per-robot
gains from cycle to cycle."""
import ctypes as C
import os

import numpy as np
import pytest

from tests.osc_testlib import REL_TOL, TASK_POINTS, OracleBatch, rel_err, rng_for, rot_exp, sample_states, sensed_ex09

pytestmark = pytest.mark.gpu


def _mft_gains(N, stream=40):
    """(kp, kv, ki) of position and orientation, [N, 3] each"""
    out = [np.zeros((N, 3)) for _ in range(6)]
    for i in range(N):
        g = rng_for(i, stream=stream)
        out[0][i] = g.uniform(50, 200, 3); out[1][i] = g.uniform(10, 30, 3); out[2][i] = g.uniform(0.5, 5, 3)
        out[3][i] = g.uniform(100, 300, 3); out[4][i] = g.uniform(15, 35, 3); out[5][i] = g.uniform(0.5, 5, 3)
    return out


def _jt_gains(N, k, stream=41):
    kp, kv, ki = np.zeros((N, k)), np.zeros((N, k)), np.zeros((N, k))
    for i in range(N):
        g = rng_for(i, stream=stream)
        kp[i] = g.uniform(20, 100, k); kv[i] = g.uniform(5, 20, k); ki[i] = g.uniform(0.5, 3, k)
    return kp, kv, ki


def _goals(N, x0, R0, q, stream=42):
    xd = np.zeros((N, 3)); Rd = np.zeros((N, 3, 3)); vd = np.zeros((N, 3)); gq = np.zeros_like(q)
    for i in range(N):
        g = rng_for(i, stream=stream)
        xd[i] = x0[i] + g.uniform(-0.05, 0.05, 3); Rd[i] = R0[i] @ rot_exp(g.uniform(-0.2, 0.2, 3)); vd[i] = g.uniform(-0.1, 0.1, 3)
        gq[i] = q[i] + g.uniform(-0.2, 0.2, q.shape[1])
    return xd, Rd, vd, gq


class Config2:
    """Panda, full six-dof MotionForceTask + JointTask in its null space, on the GPU and, for the first `n_oracle` robots, in the
    oracle; gains per robot unless `per_robot` is False; goals drawn per robot index unless given."""

    def __init__(self, q, dq, dec=1, gravity=False, per_robot=True, n_oracle=None, gains=None, goals=None, jt_vel_sat=False, robot_name="panda",
                 jt_per_robot=True):
        import sai_primitives_b200 as sp
        self.sp = sp
        N, n = q.shape
        self.N = N
        link, pt = TASK_POINTS[robot_name]
        comp = (np.eye(3), np.array(pt))
        self.robot = sp.BatchedRobot(robot_name, N)
        self.robot.setQ(q); self.robot.setDq(dq); self.robot.updateModel()
        robot = self.robot
        self.mft = sp.MotionForceTask(robot, link, comp); self.jt = sp.JointTask(robot)
        self.mft.setDynamicDecouplingType(dec); self.jt.setDynamicDecouplingType(dec)
        if jt_vel_sat:
            self.jt.enableVelocitySaturation(0.4)
        self.ctrl = sp.RobotController(robot, [self.mft, self.jt])
        if gravity:
            self.ctrl.enableGravityCompensation(True)
        self.g = gains if gains is not None else (_mft_gains(N) + list(_jt_gains(N, n)))
        if not jt_per_robot:   # the joint task stays in broadcast mode
            self.g[6:9] = [np.full((N, n), v) for v in (60.0, 12.0, 1.0)]
            self.jt.setGains(60.0, 12.0, 1.0)
        if per_robot:
            self.mft.setPosControlGains(*self.g[0:3]); self.mft.setOriControlGains(*self.g[3:6])
            if jt_per_robot:
                self.jt.setGains(*self.g[6:9])
        else:
            self.mft.setPosControlGains(150.0, 22.0, 2.0); self.mft.setOriControlGains(220.0, 30.0, 1.5); self.jt.setGains(60.0, 12.0, 1.0)
        self.goals = goals if goals is not None else _goals(N, self.mft.getCurrentPosition(), self.mft.getCurrentOrientation(), q)
        xd, Rd, vd, gq = self.goals
        self.mft.setGoalPosition(xd); self.mft.setGoalOrientation(Rd); self.mft.setGoalLinearVelocity(vd); self.jt.setGoalPosition(gq)
        self.ob = None
        if n_oracle:
            rows = np.arange(n_oracle)
            self.ob = OracleBatch(robot_name, n_oracle); self.ob.set_state(q[rows], dq[rows])
            self.omft = self.ob.add_mft(link, comp); self.ojt = self.ob.add_jt()
            for r, (a, b) in enumerate(zip(self.omft, self.ojt)):
                a.setDynamicDecouplingType(dec); b.setDynamicDecouplingType(dec)
                if jt_vel_sat:
                    b.enableVelocitySaturation(np.full(n, 0.4))
                g = self.g
                a.setPosControlGains(g[0][r], g[1][r], g[2][r]); a.setOriControlGains(g[3][r], g[4][r], g[5][r])
                b.setGains(g[6][r], g[7][r], g[8][r])
                a.setGoalPosition(xd[r]); a.setGoalOrientation(Rd[r]); a.setGoalLinearVelocity(vd[r]); b.setGoalPosition(gq[r])
            self.ob.finalize()
            if gravity:
                for ctl in self.ob.controllers:
                    ctl.enableGravityCompensation(True)

    def cycle(self):
        self.ctrl.updateControllerTaskModels()
        tau = self.ctrl.computeControlTorques()
        assert (self.robot.status() & self.sp.capi.STATUS_UNHANDLED).sum() == 0
        return tau

    def move(self, q, dq):
        self.robot.setQ(q); self.robot.setDq(dq); self.robot.updateModel()
        if self.ob is not None:
            n = len(self.omft)
            self.ob.set_state(q[:n], dq[:n])


@pytest.mark.parametrize("gravity", [False, True])
@pytest.mark.parametrize("dec", [0, 1, 2])
def test_config2_per_robot_gains_against_the_oracle(dec, gravity):
    """the specialised pure-motion kernel with per-robot position, orientation and joint gains, six cycles, state advancing"""
    N = 256
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    c = Config2(q, dq, dec=dec, gravity=gravity, n_oracle=N)
    for k in range(6):
        tau = c.cycle()
        assert rel_err(tau, c.ob.cycle()).max() < REL_TOL, k
        qk = q + 0.001 * (k + 1) * dq
        c.move(qk, dq)
    kp, kv, ki = c.mft.getPosControlGains()
    assert np.array_equal(kp, c.g[0]) and np.array_equal(kv, c.g[1]) and np.array_equal(ki, c.g[2])
    assert all(np.array_equal(a, b) for a, b in zip(c.jt.getGains(), c.g[6:9]))


@pytest.mark.parametrize("filtered", [True, False])
def test_equal_per_robot_gains_are_the_broadcast_result(filtered):
    """a handle in per-robot mode whose rows all equal the broadcast gains computes what the broadcast handle computes: bit for
    bit on the fast path (same arithmetic, gains from the block instead of the constant bank), within 1e-12 with hand-overs"""
    import sai_primitives_b200 as sp
    N, n = 4096, 7
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1 if filtered else None)
    full = lambda v, k: np.full((N, k), v)
    gains = [full(150.0, 3), full(22.0, 3), full(2.0, 3), full(220.0, 3), full(30.0, 3), full(1.5, 3), full(60.0, n), full(12.0, n), full(1.0, n)]
    a = Config2(q, dq, per_robot=False)
    b = Config2(q, dq, per_robot=True, gains=gains)
    for k in range(4):
        ta, tb = a.cycle(), b.cycle()
        ia = [a.mft._get(sp.capi.MFT_INTEGRATED_POSITION_ERROR), a.mft._get(sp.capi.MFT_INTEGRATED_ORIENTATION_ERROR), a.jt._get(sp.capi.JT_INTEGRATED_POSITION_ERROR)]
        ib = [b.mft._get(sp.capi.MFT_INTEGRATED_POSITION_ERROR), b.mft._get(sp.capi.MFT_INTEGRATED_ORIENTATION_ERROR), b.jt._get(sp.capi.JT_INTEGRATED_POSITION_ERROR)]
        if filtered:
            assert np.array_equal(ta, tb), k
            assert all(np.array_equal(x, y) for x, y in zip(ia, ib)), k
        else:
            assert rel_err(tb, ta).max() < 1e-12, k
            assert all(np.abs(x - y).max() < 1e-15 for x, y in zip(ia, ib)), k
        qk = q + 0.001 * (k + 1) * dq
        a.move(qk, dq); b.move(qk, dq)


def test_gains_follow_the_robot_index():
    """duplicated states with different gains per duplicate: each matches the oracle robot that carries its gains; shuffling
    robots together with their gains shuffles the torques bit for bit"""
    NS, N = 64, 4096
    base_q, base_dq, _ = sample_states("panda", NS, min_sigma_ratio=0.1)
    rng = np.random.default_rng(31)
    pick = rng.integers(0, NS, N)
    q, dq = base_q[pick], base_dq[pick]
    c = Config2(q, dq, n_oracle=NS)     # oracle robots 0..NS-1 carry the states and gains of GPU robots 0..NS-1
    tau = c.cycle()
    assert rel_err(tau[:NS], c.ob.cycle()).max() < REL_TOL
    # duplicates of the same state with their own gains differ from each other
    j = next(i for i in range(1, N) if pick[i] == pick[0])
    assert not np.array_equal(tau[0], tau[j])
    perm = rng.permutation(N)
    d = Config2(q[perm], dq[perm], gains=[g[perm] for g in c.g], goals=[x[perm] for x in c.goals])
    assert np.array_equal(d.cycle(), tau[perm])


def test_one_task_per_robot_the_other_broadcast():
    """the per-robot instantiation of the specialised kernel with the joint task still on its broadcast gains"""
    import sai_primitives_b200 as sp
    N = 256
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    c = Config2(q, dq, n_oracle=N, jt_per_robot=False)
    for k in range(3):
        tau = c.cycle()
        assert rel_err(tau, c.ob.cycle()).max() < REL_TOL, k
        c.move(q + 0.001 * (k + 1) * dq, dq)
    assert c.jt._params().kp[0] == 60.0
    assert np.array_equal(c.jt.getGains()[0], np.full((N, 7), 60.0))


def test_single_blending_kernel_with_per_robot_gains():
    """uniformly sampled states (many robots inside the singularity band: single blending kernel, general path)"""
    N = 256
    q, dq, _ = sample_states("panda", N)
    c = Config2(q, dq, n_oracle=N)
    for k in range(3):
        tau = c.cycle()
        assert rel_err(tau, c.ob.cycle()).max() < REL_TOL, k
        c.move(q + 0.002 * (k + 1) * dq, dq)


def test_split_blending_path_with_per_robot_gains():
    """131,072 uniformly sampled states: the robots the fused kernel hands to the split blending path keep their own gains"""
    import sai_primitives_b200 as sp
    N, NS, K = 131072, 256, 4
    base_q, base_dq, _ = sample_states("panda", NS)
    rng = np.random.default_rng(21)
    pick = rng.integers(0, NS, N); pick[:NS] = np.arange(NS)
    c = Config2(base_q[pick], base_dq[pick], n_oracle=NS)
    lib = sp.capi.load_library()
    counts = (C.c_int32 * 4)()
    for k in range(K):
        tau = c.cycle()
        assert rel_err(tau[:NS], c.ob.cycle()).max() < REL_TOL, k
        assert lib.osc_debug_general_path_counts(c.robot.handle, counts) == 0
        if k > 0 or os.environ.get("SAI_B200_BLEND_SPLIT") == "1":
            cn = np.array(list(counts))
            assert cn[1] + cn[2] > 0.4 * N and cn[3] < 0.02 * N, cn
        qk = base_q + 0.002 * (k + 1) * base_dq
        c.move(qk[pick], base_dq[pick])


def test_config3_per_robot_force_gains_reach_passivity():
    """partial XYZ task, force space dimension 1, closed-loop force control with passivity: per-robot force gains (kv_force
    enters the passivity controller per robot) and position gains, 130 cycles with the ex.09 sensed force"""
    import sai_primitives_b200 as sp
    N, K = 48, 130
    dirs = [(1, 0, 0), (0, 1, 0), (0, 0, 1)]
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1, dirs=np.eye(6)[:, :3])
    link, pt = TASK_POINTS["panda"]
    comp = (np.eye(3), np.array(pt))
    robot = sp.BatchedRobot("panda", N)
    robot.setQ(q); robot.setDq(dq); robot.updateModel()
    mft = sp.MotionForceTask(robot, link, comp, dirs, []); jt = sp.JointTask(robot)
    ctrl = sp.RobotController(robot, [mft, jt])
    ob = OracleBatch("panda", N); ob.set_state(q, dq)
    omft = ob.add_mft(link, comp, dirs, []); ojt = ob.add_jt(); ob.finalize()
    assert mft.parametrizeForceMotionSpaces(1, (0, 0, 1)) is True
    mft.setGoalForce(np.array([0, 0, -5.0])); mft.setClosedLoopForceControl(); mft.enablePassivity()
    kpf = np.array([[rng_for(i, stream=43).uniform(0.3, 1.5)] for i in range(N)])
    kvf = np.array([[rng_for(i, stream=44).uniform(5.0, 20.0)] for i in range(N)])
    kif = np.array([[rng_for(i, stream=45).uniform(0.5, 2.0)] for i in range(N)])
    mft.setForceControlGains(kpf, kvf, kif)
    g = _mft_gains(N)
    mft.setPosControlGains(*g[0:3])
    for i, t in enumerate(omft):
        t.parametrizeForceMotionSpaces(1, (0, 0, 1)); t.setGoalForce((0, 0, -5.0)); t.setClosedLoopForceControl(); t.enablePassivity()
        t.setForceControlGains(kpf[i, 0], kvf[i, 0], kif[i, 0]); t.setPosControlGains(g[0][i], g[1][i], g[2][i])
    for k in range(K):
        F, Mo = sensed_ex09(N, k)
        mft.updateSensedForceAndMoment(F, Mo)
        for i in range(N):
            omft[i].updateSensedForceAndMoment(F[i], Mo[i])
        ctrl.updateControllerTaskModels()
        tau = ctrl.computeControlTorques()
        assert (robot.status() & sp.capi.STATUS_UNHANDLED).sum() == 0
        assert rel_err(tau, ob.cycle()).max() < REL_TOL, k
        q = q + 0.0005 * dq
        robot.setQ(q); robot.updateModel(); ob.set_state(q, dq)
    assert np.array_equal(mft.getForceControlGains()[1], kvf)
    popc = mft._get(sp.capi.MFT_POPC_STATE)
    assert (popc[:, 2] < 1.0).any()            # the passivity controller engaged (Rc < 1) somewhere


@pytest.mark.parametrize("case", ["sliding_base", "joint_velocity_saturation"])
def test_non_specialised_kernels_with_per_robot_gains(case):
    """the non-specialised fused kernel reads the gain blocks at run time: a prismatic first joint (sliding-base Panda), and a
    joint task with velocity saturation (per-robot kv inside its pseudo-inverse)"""
    name = "panda_sliding_base" if case == "sliding_base" else "panda"
    N = 64
    q, dq, _ = sample_states(name, N, min_sigma_ratio=0.1)
    c = Config2(q, dq, n_oracle=N, jt_vel_sat=(case == "joint_velocity_saturation"), robot_name=name)
    for k in range(3):
        tau = c.cycle()
        assert rel_err(tau, c.ob.cycle()).max() < REL_TOL, k
        c.move(q + 0.001 * (k + 1) * dq, dq)


def test_general_hierarchy_with_per_robot_gains():
    """[position task, orientation task, joint task]: the general-hierarchy kernel"""
    import sai_primitives_b200 as sp
    N = 48
    q, dq, _ = sample_states("panda", N)
    link, pt = TASK_POINTS["panda"]
    comp = (np.eye(3), np.array(pt))
    xyz = [(1, 0, 0), (0, 1, 0), (0, 0, 1)]
    robot = sp.BatchedRobot("panda", N)
    robot.setQ(q); robot.setDq(dq); robot.updateModel()
    t1 = sp.MotionForceTask(robot, link, comp, xyz, [], task_name="position")
    t2 = sp.MotionForceTask(robot, link, comp, [], xyz, task_name="orientation")
    jt = sp.JointTask(robot)
    ctrl = sp.RobotController(robot, [t1, t2, jt])
    ob = OracleBatch("panda", N); ob.set_state(q, dq)
    o1 = ob.add_mft(link, comp, xyz, [], name="position"); o2 = ob.add_mft(link, comp, [], xyz, name="orientation")
    oj = ob.add_jt(); ob.finalize()
    g = _mft_gains(N); jg = _jt_gains(N, 7)
    t1.setPosControlGains(*g[0:3]); t2.setOriControlGains(*g[3:6]); jt.setGains(*jg)
    xd, Rd, _, gq = _goals(N, t1.getCurrentPosition(), t1.getCurrentOrientation(), q)
    t1.setGoalPosition(xd); t2.setGoalOrientation(Rd); jt.setGoalPosition(gq)
    for i in range(N):
        o1[i].setPosControlGains(g[0][i], g[1][i], g[2][i]); o2[i].setOriControlGains(g[3][i], g[4][i], g[5][i])
        oj[i].setGains(jg[0][i], jg[1][i], jg[2][i])
        o1[i].setGoalPosition(xd[i]); o2[i].setGoalOrientation(Rd[i]); oj[i].setGoalPosition(gq[i])
    for k in range(3):
        ctrl.updateControllerTaskModels()
        tau = ctrl.computeControlTorques()
        assert rel_err(tau, ob.cycle()).max() < REL_TOL, k


def test_mode_rules_and_validation():
    import sai_primitives_b200 as sp
    N = 16
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    c = Config2(q, dq, per_robot=False)
    mft, jt = c.mft, c.jt
    lib = sp.capi.load_library()
    # broadcast mode: a broadcast setter is what it always was
    mft.setPosControlGains([100.0, 110.0, 120.0], 20.0 * np.ones(3), [1.0, 2.0, 3.0])
    p = mft._params()
    assert list(p.kp_pos) == [100.0, 110.0, 120.0] and list(p.ki_pos) == [1.0, 2.0, 3.0]
    kp, _, _ = mft.getPosControlGains()
    assert kp.shape == (N, 3) and np.array_equal(kp, np.tile([100.0, 110.0, 120.0], (N, 1)))
    # invalid per-robot values change nothing
    g = _mft_gains(N)
    for bad, grp in ((-1.0, "pos"), (np.nan, "pos"), (-1.0, "ori"), (np.nan, "joint")):
        before = (mft.getPosControlGains(), mft.getOriControlGains(), jt.getGains())
        a = g[0].copy(); a[3, 1] = bad
        with pytest.raises(ValueError) as e:
            if grp == "pos":
                mft.setPosControlGains(a, g[1], g[2])
            elif grp == "ori":
                mft.setOriControlGains(a, g[4], g[5])
            else:
                kpj = np.full((N, 7), 50.0); kpj[2, 4] = bad
                jt.setGains(kpj, 14.0, 1.0)
        if bad == -1.0:
            assert ("setPosControlGains" if grp == "pos" else "setOriControlGains") in str(e.value)
        after = (mft.getPosControlGains(), mft.getOriControlGains(), jt.getGains())
        assert all(np.array_equal(x, y) for u, v in zip(before, after) for x, y in zip(u, v))
    kf = np.ones((N, 1)); kf[5, 0] = np.nan
    before = mft.getForceControlGains()
    with pytest.raises(ValueError):
        mft.setForceControlGains(kf, np.ones((N, 1)), np.ones((N, 1)))
    assert all(np.array_equal(x, y) for x, y in zip(before, mft.getForceControlGains()))
    mft.setForceControlGains(-np.ones((N, 1)), np.ones((N, 1)), np.ones((N, 1)))   # any finite value, like the reference
    # bad shapes
    with pytest.raises(ValueError):
        mft.setPosControlGains(np.ones((N, 2)), 1.0, 1.0)
    with pytest.raises(ValueError):
        jt.setGains(np.ones((N + 1, 7)), 1.0, 1.0)
    with pytest.raises(ValueError):
        jt.setGains(np.ones(5), 1.0, 1.0)
    # per-robot position gains, then broadcast orientation gains: position stays per robot
    mft.setPosControlGains(*g[0:3])
    mft.setOriControlGains(210.0, 29.0, 1.0)
    assert np.array_equal(mft.getPosControlGains()[0], g[0])
    assert np.array_equal(mft.getOriControlGains()[0], np.full((N, 3), 210.0))
    # per-robot mode: a broadcast setGains fills every robot
    jt.setGains(*_jt_gains(N, 7))
    jt.setGains(42.0, 13.0, 0.5)
    assert all(np.array_equal(x, np.full((N, 7), v)) for x, v in zip(jt.getGains(), (42.0, 13.0, 0.5)))
    # osc_mft_set_params: a changed gain is refused, unchanged gains pass (read-modify-write setters keep working)
    p = mft._params()
    p.kp_pos[0] += 1.0
    assert lib.osc_mft_set_params(c.robot.handle, mft.task_id, C.byref(p)) == sp.capi.OSC_ERR_STATE
    mft.setDynamicDecouplingType(sp.FULL_DYNAMIC_DECOUPLING)
    assert mft._params().dynamic_decoupling_type == sp.FULL_DYNAMIC_DECOUPLING
    jt.setDynamicDecouplingType(sp.IMPEDANCE)
    pj = jt._params(); pj.kv[0] += 1.0
    assert lib.osc_joint_set_params(c.robot.handle, jt.task_id, C.byref(pj)) == sp.capi.OSC_ERR_STATE
    # reInitializeTask keeps the gains
    mft.reInitializeTask(); jt.reInitializeTask()
    assert np.array_equal(mft.getPosControlGains()[0], g[0])
    assert np.array_equal(jt.getGains()[0], np.full((N, 7), 42.0))
    c.cycle()


def test_gain_writes_between_pipelined_cycles():
    """gains rewritten between back-to-back pipelined cycles: broadcast writes into the gain blocks before every cycle (a fill
    kernel in the handle's stream, no host synchronisation) and per-robot position gains from torch device tensors every fifth
    cycle (device input is validated, which synchronises), 20 cycles of stepDevice.  The torques of every cycle must be
    bit-identical to the same run without cycle pipelining, and follow the oracle on a sample over all 20 cycles."""
    import torch
    N, K, NS = 66000, 20, 32
    base_q, base_dq, _ = sample_states("panda", 1024, min_sigma_ratio=0.1)
    rng = np.random.default_rng(7)
    pick = rng.integers(0, 1024, N); pick[:NS] = np.arange(NS)
    q, dq = base_q[pick], base_dq[pick]
    dev = torch.device("cuda", 0)
    G = _mft_gains(N) + list(_jt_gains(N, 7))
    pos_scale = {k: 1.0 + 0.01 * k for k in range(0, K, 5)}
    d_pos = {k: [torch.from_numpy(np.ascontiguousarray((g * s).T)).to(dev) for g in G[0:3]] for k, s in pos_scale.items()}
    ori = [(200.0 + 5 * k, 25.0 + 0.5 * k, 1.0 + 0.1 * k) for k in range(K)]
    joint = [(50.0 + 2 * k, 14.0 - 0.2 * k, 1.0 + 0.05 * k) for k in range(K)]
    d_q = torch.from_numpy(np.ascontiguousarray(q.T)).to(dev); d_dq = torch.from_numpy(np.ascontiguousarray(dq.T)).to(dev)
    torch.cuda.synchronize()   # the library's stream is not torch's: the device inputs are written before the first cycle

    def run(pipelined, n_oracle=None):
        if not pipelined:
            os.environ["SAI_B200_NO_PIPELINE"] = "1"
        try:
            c = Config2(q, dq, gains=G, n_oracle=n_oracle)
        finally:
            os.environ.pop("SAI_B200_NO_PIPELINE", None)
        taus = [torch.empty((7, N), dtype=torch.float64, device=dev) for _ in range(K)]
        for k in range(K):
            if k in d_pos:
                c.mft.setPosControlGainsDevice(*(t.data_ptr() for t in d_pos[k]))
            c.mft.setOriControlGains(*ori[k])
            c.jt.setGains(*joint[k])
            c.ctrl.stepDevice(d_q.data_ptr(), d_dq.data_ptr(), taus[k].data_ptr())
        c.robot.sync()
        return c, [t.cpu().numpy().T for t in taus]

    c, a = run(True, n_oracle=NS)
    _, b = run(False)
    for k in range(K):
        assert np.array_equal(a[k], b[k]), k
    s = 1.0
    for k in range(K):                  # the oracle robots replay the same gain writes
        s = pos_scale.get(k, s)
        for i in range(NS):
            c.omft[i].setPosControlGains(G[0][i] * s, G[1][i] * s, G[2][i] * s)
            c.omft[i].setOriControlGains(np.full(3, ori[k][0]), np.full(3, ori[k][1]), np.full(3, ori[k][2]))
            c.ojt[i].setGains(np.full(7, joint[k][0]), np.full(7, joint[k][1]), np.full(7, joint[k][2]))
        assert rel_err(a[k][:NS], c.ob.cycle()).max() < REL_TOL, k


def test_fp32_mode_refuses_per_robot_gains():
    import sai_primitives_b200 as sp
    N = 64
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    c = Config2(q, dq)
    c.ctrl.setPrecision("fp32")
    c.ctrl.updateControllerTaskModels()
    with pytest.raises(NotImplementedError):
        c.ctrl.computeControlTorques()
    c.ctrl.setPrecision("fp64")
    c.cycle()


def test_n_robots_equal_to_ncomp_keeps_the_broadcast_reading():
    """with as many robots as components, an (N, 1) array is the (ncomp,) broadcast vector it always was; (N, ncomp) is per robot"""
    N = 3
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    c = Config2(q, dq, per_robot=False)
    col = lambda a, b, c: np.array([[a], [b], [c]])
    c.mft.setPosControlGains(col(100.0, 110.0, 120.0), col(20.0, 21.0, 22.0), col(1.0, 2.0, 3.0))
    assert list(c.mft._params().kp_pos) == [100.0, 110.0, 120.0]
    assert np.array_equal(c.mft.getPosControlGains()[0], np.tile([100.0, 110.0, 120.0], (N, 1)))
    per = np.array([[100.0, 101.0, 102.0], [110.0, 111.0, 112.0], [120.0, 121.0, 122.0]])
    c.mft.setPosControlGains(per, 20.0, 1.0)
    assert np.array_equal(c.mft.getPosControlGains()[0], per)
    c.cycle()
