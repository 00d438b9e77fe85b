"""Per-robot force / moment spaces and closed-loop flags of a MotionForceTask (osc_mft_parametrize_spaces_batched,
osc_mft_set_closed_loop_batched): every robot of a handle in its own contact state, on every cycle path, against the reference's
control law with one oracle robot per GPU robot, each parametrised through its own setters.  Integral gains are non-zero, the
state advances between cycles and every robot gets its own sensed wrench (the ex.09 scenario), so integrators, resets and the
passivity controller carry the per-robot choices from cycle to cycle."""
import numpy as np
import pytest

from tests.osc_testlib import REL_TOL, TASK_POINTS, OracleBatch, oracle_kind, rel_err, rng_for, sample_states, sensed_ex09

pytestmark = pytest.mark.gpu

XYZ = [(1, 0, 0), (0, 1, 0), (0, 0, 1)]


def _unit(v):
    return v / np.linalg.norm(v)


def _modes(N, stream=50):
    """per-robot force dim, moment dim, closed-loop force, closed-loop moment (dealt by index) and axes drawn per robot"""
    i = np.arange(N)
    fdim, mdim = (i % 4).astype(np.int32), ((i // 4) % 4).astype(np.int32)
    clf, clm = ((i // 16) % 2).astype(bool), ((i // 32) % 2).astype(bool)
    fax = np.array([_unit(rng_for(k, stream=stream).normal(size=3)) * (1 + k % 3) for k in range(N)])
    max_ = np.array([_unit(rng_for(k, stream=stream + 1).normal(size=3)) for k in range(N)])
    return fdim, mdim, clf, clm, fax, max_


class Setup:
    """[MotionForceTask (full six-dof, or the partial XYZ task of config 3), JointTask] on the GPU and in the oracle, integral
    gains on, internal OTG off, passivity on"""

    def __init__(self, q, dq, hier="full", dec=1, in_compliant=False, robot_name="panda", oracle=True, passivity=True):
        import sai_primitives_b200 as sp
        self.sp = sp
        N = q.shape[0]
        self.N = N
        link, pt = TASK_POINTS[robot_name]
        comp = (np.eye(3), np.array(pt))
        dirs = () if hier == "full" else (XYZ, [])
        self.robot = sp.BatchedRobot(robot_name, N)
        self.robot.setQ(q); self.robot.setDq(dq); self.robot.updateModel()
        self.mft = sp.MotionForceTask(self.robot, link, comp, *dirs, is_force_motion_parametrization_in_compliant_frame=in_compliant)
        self.jt = sp.JointTask(self.robot)
        self.mft.disableInternalOtg(); self.jt.disableInternalOtg()
        self.ctrl = sp.RobotController(self.robot, [self.mft, self.jt])
        self.tasks = [self.mft]
        self.ob = None
        if oracle:
            self.ob = OracleBatch(robot_name, N); self.ob.set_state(q, dq)
            self.omft = self.ob.add_mft(link, comp, *dirs, in_compliant=in_compliant); self.ojt = self.ob.add_jt(); self.ob.finalize()
        for t in self._all():
            t.setDynamicDecouplingType(dec)
            t.setPosControlGains(120.0, 20.0, 3.0); t.setOriControlGains(180.0, 25.0, 2.0)
            t.setForceControlGains(0.8, 12.0, 1.5); t.setMomentControlGains(0.6, 8.0, 1.0)
            t.setGoalForce(np.array([0, 0, -5.0])); t.setGoalMoment(np.array([0.05, 0, 0]))
            if passivity:
                t.enablePassivity()
        x0 = self.mft.getCurrentPosition()
        self.goal = x0 + np.array([0.02, -0.01, 0.015])
        self.mft.setGoalPosition(self.goal); self.jt.setGoalPosition(q + 0.05)
        if oracle:
            for i in range(N):
                self.omft[i].setGoalPosition(self.goal[i]); self.ojt[i].setGoalPosition(q[i] + 0.05)
            for t in self.ojt:
                t.setGains(60.0, 12.0, 1.0)
        self.jt.setGains(60.0, 12.0, 1.0)

    def _all(self):
        return [self.mft] + (list(self.omft) if self.ob is not None else [])

    def sense(self, k):
        F, Mo = sensed_ex09(self.N, k)
        self.mft.updateSensedForceAndMoment(F, Mo)
        if self.ob is not None:
            for i in range(self.N):
                self.omft[i].updateSensedForceAndMoment(F[i], Mo[i])

    def cycle(self):
        self.ctrl.updateControllerTaskModels()
        tau = self.ctrl.computeControlTorques()
        assert (self.robot.status() & self.sp.capi.STATUS_UNHANDLED).sum() == 0
        return tau

    def move(self, q, dq):
        self.robot.setQ(q); self.robot.setDq(dq); self.robot.updateModel()
        if self.ob is not None:
            self.ob.set_state(q, dq)

    def parametrize(self, fdim, mdim, clf, clm, fax, max_, rows=None):
        """per robot on the GPU, robot by robot in the oracle; returns (GPU was_reset force, moment), oracle's likewise"""
        rf = self.mft.parametrizeForceMotionSpaces(fdim, fax)
        rm = self.mft.parametrizeMomentRotMotionSpaces(mdim, max_)
        self.mft.setClosedLoopForceControl(clf); self.mft.setClosedLoopMomentControl(clm)
        of, om = np.zeros(self.N, bool), np.zeros(self.N, bool)
        if self.ob is not None:
            for i, t in enumerate(self.omft):
                of[i] = t.parametrizeForceMotionSpaces(int(fdim[i]), fax[i])
                om[i] = t.parametrizeMomentRotMotionSpaces(int(mdim[i]), max_[i])
                t.setClosedLoopForceControl(bool(clf[i])); t.setClosedLoopMomentControl(bool(clm[i]))
        return rf, rm, of, om


def _check_observers(s):
    for name in ("sigmaForce", "sigmaPosition", "sigmaMoment", "sigmaOrientation"):
        got = getattr(s.mft, name)()
        ref = np.array([getattr(t, name)() for t in s.omft])
        assert np.abs(got - ref).max() < 1e-12, name


def _check_popc(s):
    if oracle_kind() != "numpy":
        return
    popc = s.mft._get(s.sp.capi.MFT_POPC_STATE)
    rc = np.array([t._POPC_force._Rc for t in s.omft])
    assert np.abs(popc[:, 2] - rc).max() < 1e-9


@pytest.mark.parametrize("in_compliant", [False, True])
@pytest.mark.parametrize("dec", [0, 1, 2])
@pytest.mark.parametrize("hier", ["full", "xyz"])
def test_mixed_batch_against_the_oracle(hier, dec, in_compliant):
    """256 robots, force / moment dimension 0..3 with the robot's own axis, closed loops on and off, dealt per index"""
    N, K = 256, 8
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1, dirs=None if hier == "full" else np.eye(6)[:, :3])
    s = Setup(q, dq, hier=hier, dec=dec, in_compliant=in_compliant)
    fdim, mdim, clf, clm, fax, max_ = _modes(N)
    rf, rm, of, om = s.parametrize(fdim, mdim, clf, clm, fax, max_)
    assert np.array_equal(rf, of) and np.array_equal(rm, om)
    dims, axes, cl = s.mft.getForceMotionSpaces()
    assert np.array_equal(dims, fdim) and np.array_equal(cl, clf)
    one = (fdim == 1) | (fdim == 2)
    assert np.abs(axes[one] - fax[one] / np.linalg.norm(fax[one], axis=1)[:, None]).max() < 1e-15
    for k in range(K):
        s.sense(k)
        tau = s.cycle()
        assert rel_err(tau, s.ob.cycle()).max() < REL_TOL, k
        if k == K - 1:
            _check_observers(s)
            _check_popc(s)
        s.move(q + 0.0005 * (k + 1) * dq, dq)


def _transition_plan(N):
    g = np.random.default_rng(7)
    third = g.permutation(N)[: N // 3]
    normals = np.array([_unit(rng_for(k, stream=60).normal(size=3)) for k in range(N)])
    back = third[: len(third) // 3]               # cycle 12: these return to free motion
    same = third[len(third) // 3: len(third) // 2]        # the same axis again: no reset
    scaled = third[len(third) // 2: 2 * len(third) // 3]  # the same axis scaled: no reset
    tiny = third[2 * len(third) // 3: 5 * len(third) // 6]  # 1e-13 off: no reset
    moved = third[5 * len(third) // 6:]               # 1e-6 off: reset
    return third, normals, back, same, scaled, tiny, moved


def _transitions(s, k, plan, fdim, fax, clf):
    third, normals, back, same, scaled, tiny, moved = plan
    if k == 5:
        fdim[third] = 1; fax[third] = normals[third]; clf[third] = True
        return True
    if k == 12:
        fdim[back] = 0; clf[back] = False
        fax[scaled] = normals[scaled] * 2.5
        fax[tiny] = normals[tiny] * (1 + 1e-13 * np.array([1.0, -1.0, 0.5]))
        fax[moved] = normals[moved] * (1 + 1e-6 * np.array([1.0, -1.0, 0.5]))
        return True
    return False


def test_contact_transitions_against_the_oracle():
    """every robot free; at cycle 5 a random third switch to force dimension 1 along their own normal with closed-loop force
    control; at cycle 12 some switch back, some get the same axis again (as given, or scaled, or 1e-13 off: no reset) and some
    an axis 1e-6 off (reset).  was_reset, goals and integrators per robot against the oracle, 20 cycles."""
    sp_ = pytest.importorskip("sai_primitives_b200")
    N, K = 192, 20
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    s = Setup(q, dq, dec=1)
    plan = _transition_plan(N)
    fdim, fax, clf = np.zeros(N, np.int32), np.tile([0.0, 0.0, 1.0], (N, 1)), np.zeros(N, bool)
    mdim, max_, clm = np.zeros(N, np.int32), np.tile([0.0, 0.0, 1.0], (N, 1)), np.zeros(N, bool)
    for k in range(K):
        if _transitions(s, k, plan, fdim, fax, clf):
            rf, rm, of, om = s.parametrize(fdim, mdim, clf, clm, fax, max_)
            assert np.array_equal(rf, of) and np.array_equal(rm, om), k
            if k == 12:
                _, _, back, same, scaled, tiny, moved = plan
                assert rf[back].all() and rf[moved].all() and not rf[same].any() and not rf[scaled].any() and not rf[tiny].any()
            if oracle_kind() == "numpy":
                gp = s.mft.getGoalPosition()
                assert np.abs(gp - np.array([t._goal_position for t in s.omft])).max() < 1e-14, k
                ip = s.mft._get(sp_.capi.MFT_INTEGRATED_POSITION_ERROR)
                assert np.abs(ip - np.array([t._integrated_position_error for t in s.omft])).max() < 1e-14, k
                iff = s.mft._get(sp_.capi.MFT_INTEGRATED_FORCE_ERROR)
                assert np.abs(iff - np.array([t._integrated_force_error for t in s.omft])).max() < 1e-14, k
        s.sense(k)
        tau = s.cycle()
        assert rel_err(tau, s.ob.cycle()).max() < REL_TOL, k
        if k == K - 1:
            _check_observers(s)
        s.move(q + 0.0005 * (k + 1) * dq, dq)


def test_contact_transitions_with_the_internal_otg():
    """the same transitions with the internal OTG on: robots that were reset match a handle that received the same call
    broadcast (its reset path is covered by the OTG tests), robots that were not reset match a handle that received no call"""
    import sai_primitives_b200 as sp
    N, K = 96, 20
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    lim = (0.3, 2.0, np.pi / 3, 2 * np.pi)
    hs = [Setup(q, dq, oracle=False, passivity=False) for _ in range(3)]   # per robot, broadcast call, no call
    for h in hs:
        h.mft.enableInternalOtgAccelerationLimited(*lim)
    plan = _transition_plan(N)
    third, normals = plan[0], plan[1]
    for k in range(K):
        if k == 5:
            fdim = np.zeros(N, np.int32); fdim[third] = 1
            fax = np.tile([0.0, 0.0, 1.0], (N, 1)); fax[third] = normals[0]
            r = hs[0].mft.parametrizeForceMotionSpaces(fdim, fax)
            assert np.array_equal(r, fdim == 1)
            assert hs[1].mft.parametrizeForceMotionSpaces(1, normals[0]) is True
        for h in hs:
            h.sense(k)
        taus = [h.cycle() for h in hs]
        if k >= 5:
            reset = np.zeros(N, bool); reset[third] = True
            d = [h.mft.getDesiredPosition() for h in hs]
            assert np.array_equal(taus[0][reset], taus[1][reset]) and np.array_equal(d[0][reset], d[1][reset]), k
            assert np.abs(taus[0][~reset] - taus[2][~reset]).max() < 1e-12 * max(1.0, np.abs(taus[2]).max()), k
            assert np.abs(d[0][~reset] - d[2][~reset]).max() < 1e-12, k
        for h in hs:
            h.move(q + 0.0005 * (k + 1) * dq, dq)


@pytest.mark.parametrize("filtered", [True, False])
@pytest.mark.parametrize("hier", ["full", "xyz"])
def test_equal_rows_give_the_broadcast_result(hier, filtered):
    """a per-robot task whose rows all equal a broadcast parametrisation computes the broadcast handle's torques: bit for bit
    on the fused kernels, within 1e-12 with hand-overs (uniformly sampled states: single and split blending paths)"""
    N = 4096
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1 if filtered else None, dirs=None if hier == "full" else np.eye(6)[:, :3])
    a = Setup(q, dq, hier=hier, oracle=False)
    b = Setup(q, dq, hier=hier, oracle=False)
    ax = np.array([0.3, -0.2, 0.9])
    a.mft.parametrizeForceMotionSpaces(1, ax); a.mft.setClosedLoopForceControl(True)
    b.mft.parametrizeForceMotionSpaces(np.ones(N, np.int32), np.tile(ax, (N, 1))); b.mft.setClosedLoopForceControl(np.ones(N, bool))
    a.mft.parametrizeMomentRotMotionSpaces(2, (0, 1, 0))
    b.mft.parametrizeMomentRotMotionSpaces(np.full(N, 2, np.int32), np.tile([0.0, 1.0, 0.0], (N, 1)))
    for k in range(4):
        a.sense(k); b.sense(k)
        ta, tb = a.cycle(), b.cycle()
        if filtered:
            assert np.array_equal(ta, tb), k
        else:
            assert np.abs(ta - tb).max() <= 1e-12 * max(1.0, np.abs(ta).max()), k
        a.move(q + 0.0005 * (k + 1) * dq, dq); b.move(q + 0.0005 * (k + 1) * dq, dq)


def test_broadcast_calls_on_a_per_robot_task():
    """after entering per-robot mode, the broadcast setters apply the same values to every robot, each deciding its own reset"""
    N = 64
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    s = Setup(q, dq)
    fdim = (np.arange(N) % 2).astype(np.int32)
    ax = np.tile([0.0, 0.0, 1.0], (N, 1))
    rf, _, of, _ = s.parametrize(fdim, np.zeros(N, np.int32), np.zeros(N, bool), np.zeros(N, bool), ax, ax)
    assert np.array_equal(rf, of)
    assert s.mft.parametrizeForceMotionSpaces(1, (0, 0, 2.0)) is True     # the dimension-0 robots are reset
    assert s.mft.parametrizeForceMotionSpaces(1, (0, 0, 1.0)) is False    # nobody
    s.mft.setClosedLoopForceControl(True)
    for t in s.omft:
        t.parametrizeForceMotionSpaces(1, (0, 0, 1.0)); t.setClosedLoopForceControl(True)
    dims, _, cl = s.mft.getForceMotionSpaces()
    assert (dims == 1).all() and cl.all()
    assert s.mft._params().force_space_dimension == 1
    for k in range(3):
        s.sense(k)
        assert rel_err(s.cycle(), s.ob.cycle()).max() < REL_TOL, k


def test_sliding_base_non_specialised_kernel():
    N = 64
    q, dq, _ = sample_states("panda_sliding_base", N, min_sigma_ratio=0.1)
    s = Setup(q, dq, robot_name="panda_sliding_base")
    s.parametrize(*_modes(N))
    for k in range(4):
        s.sense(k)
        assert rel_err(s.cycle(), s.ob.cycle()).max() < REL_TOL, k
        s.move(q + 0.0005 * (k + 1) * dq, dq)


def test_uniform_states_rolled_general_path():
    """uniformly sampled states (hand-overs to the blending and general paths) with per-robot gains and spaces together"""
    N = 256
    q, dq, _ = sample_states("panda", N)
    s = Setup(q, dq)
    kp = np.array([[rng_for(i, stream=70).uniform(0.3, 1.5)] for i in range(N)])
    kv = np.array([[rng_for(i, stream=71).uniform(5.0, 20.0)] for i in range(N)])
    ki = np.array([[rng_for(i, stream=72).uniform(0.5, 2.0)] for i in range(N)])
    s.mft.setForceControlGains(kp, kv, ki)
    for i, t in enumerate(s.omft):
        t.setForceControlGains(kp[i, 0], kv[i, 0], ki[i, 0])
    s.parametrize(*_modes(N))
    for k in range(4):
        s.sense(k)
        assert rel_err(s.cycle(), s.ob.cycle()).max() < REL_TOL, k
        s.move(q + 0.002 * (k + 1) * dq, dq)


def test_general_hierarchy_two_motion_force_tasks():
    import sai_primitives_b200 as sp
    N = 48
    q, dq, _ = sample_states("panda", N)
    link, pt = TASK_POINTS["panda"]
    comp = (np.eye(3), np.array(pt))
    robot = sp.BatchedRobot("panda", N)
    robot.setQ(q); robot.setDq(dq); robot.updateModel()
    t1 = sp.MotionForceTask(robot, link, comp, XYZ, [], task_name="position")
    t2 = sp.MotionForceTask(robot, link, comp, [], XYZ, task_name="orientation")
    jt = sp.JointTask(robot)
    for t in (t1, t2, jt):
        t.disableInternalOtg()
    ctrl = sp.RobotController(robot, [t1, t2, jt])
    ob = OracleBatch("panda", N); ob.set_state(q, dq)
    o1 = ob.add_mft(link, comp, XYZ, [], name="position"); o2 = ob.add_mft(link, comp, [], XYZ, name="orientation")
    ob.add_jt(); ob.finalize()
    fdim, mdim, clf, clm, fax, max_ = _modes(N)
    t1.parametrizeForceMotionSpaces(fdim, fax); t1.setClosedLoopForceControl(clf)
    t2.parametrizeMomentRotMotionSpaces(mdim, max_); t2.setClosedLoopMomentControl(clm)
    for t in [t1] + o1 + [t2] + o2:
        t.setPosControlGains(120.0, 20.0, 3.0); t.setOriControlGains(180.0, 25.0, 2.0); t.setGoalForce(np.array([0, 0, -5.0]))
    for i in range(N):
        o1[i].parametrizeForceMotionSpaces(int(fdim[i]), fax[i]); o1[i].setClosedLoopForceControl(bool(clf[i]))
        o2[i].parametrizeMomentRotMotionSpaces(int(mdim[i]), max_[i]); o2[i].setClosedLoopMomentControl(bool(clm[i]))
    for k in range(3):
        F, Mo = sensed_ex09(N, k)
        t1.updateSensedForceAndMoment(F, Mo); t2.updateSensedForceAndMoment(F, Mo)
        for i in range(N):
            o1[i].updateSensedForceAndMoment(F[i], Mo[i]); o2[i].updateSensedForceAndMoment(F[i], Mo[i])
        ctrl.updateControllerTaskModels()
        tau = ctrl.computeControlTorques()
        assert rel_err(tau, ob.cycle()).max() < REL_TOL, k


def test_device_input():
    """dims, axes and flags from torch tensors, was_reset to device: the same result as host input"""
    torch = pytest.importorskip("torch")
    N = 128
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    a, b = Setup(q, dq, oracle=False), Setup(q, dq, oracle=False)
    fdim, mdim, clf, clm, fax, max_ = _modes(N)
    ra = a.mft.parametrizeForceMotionSpaces(fdim, fax)
    a.mft.parametrizeMomentRotMotionSpaces(mdim, max_)
    a.mft.setClosedLoopForceControl(clf); a.mft.setClosedLoopMomentControl(clm)
    dev = torch.device("cuda:0")
    d_fdim = torch.tensor(fdim, dtype=torch.int32, device=dev)
    d_fax = torch.tensor(np.ascontiguousarray(fax.T), dtype=torch.float64, device=dev)
    d_mdim = torch.tensor(mdim, dtype=torch.int32, device=dev)
    d_max = torch.tensor(np.ascontiguousarray(max_.T), dtype=torch.float64, device=dev)
    d_reset = torch.full((N,), -1, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    b.mft.parametrizeForceMotionSpacesDevice(d_fdim.data_ptr(), d_fax.data_ptr(), d_reset.data_ptr())
    b.mft.parametrizeMomentRotMotionSpacesDevice(d_mdim.data_ptr(), d_max.data_ptr())
    b.mft.setClosedLoopForceControlDevice(torch.tensor(clf.astype(np.int32), device=dev).data_ptr())
    b.mft.setClosedLoopMomentControlDevice(torch.tensor(clm.astype(np.int32), device=dev).data_ptr())
    b.robot.sync()
    assert np.array_equal(d_reset.cpu().numpy() != 0, ra)
    for g in ("getForceMotionSpaces", "getMomentRotMotionSpaces"):
        assert all(np.array_equal(x, y) for x, y in zip(getattr(a.mft, g)(), getattr(b.mft, g)()))
    for k in range(2):
        a.sense(k); b.sense(k)
        assert np.array_equal(a.cycle(), b.cycle()), k


def test_validation_leaves_every_robot_as_it_was():
    import sai_primitives_b200 as sp
    torch = pytest.importorskip("torch")
    N = 32
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    s = Setup(q, dq, oracle=False)
    ref = Setup(q, dq, oracle=False)
    modes = _modes(N)
    for h in (s, ref):
        h.mft.parametrizeForceMotionSpaces(modes[0], modes[4]); h.mft.setClosedLoopForceControl(modes[2])
    before = (s.mft.getForceMotionSpaces(), s.mft.getMomentRotMotionSpaces())
    ax = np.tile([0.0, 0.0, 1.0], (N, 1))
    bad = []
    d = np.ones(N, np.int32); d[5] = 4; bad.append((d, ax))
    d = np.ones(N, np.int32); d[7] = -1; bad.append((d, ax))
    a2 = ax.copy(); a2[3] = [1e-3, 0, 0]; bad.append((np.ones(N, np.int32), a2))
    a2 = ax.copy(); a2[9] = [np.nan, 0, 1]; bad.append((np.full(N, 2, np.int32), a2))
    a2 = ax.copy(); a2[11] = [np.inf, 0, 1]; bad.append((np.ones(N, np.int32), a2))
    lib = sp.capi.load_library()
    for dims, axes in bad:
        with pytest.raises(ValueError):
            s.mft.parametrizeForceMotionSpaces(dims, axes)
        d_d = torch.tensor(dims, dtype=torch.int32, device="cuda:0")
        d_a = torch.tensor(np.ascontiguousarray(axes.T), dtype=torch.float64, device="cuda:0")
        torch.cuda.synchronize()
        rc = lib.osc_mft_parametrize_spaces_batched(s.robot.handle, s.mft.task_id, 1, d_d.data_ptr(), d_a.data_ptr(), None, sp.capi.OSC_MEM_DEVICE)
        assert rc == sp.capi.OSC_ERR_INVALID_ARGUMENT
    flags = np.ones(N, np.int32); flags[2] = 2
    rc = lib.osc_mft_set_closed_loop_batched(s.robot.handle, s.mft.task_id, 0, flags.ctypes.data, sp.capi.OSC_MEM_HOST)
    assert rc == sp.capi.OSC_ERR_INVALID_ARGUMENT
    d_f = torch.tensor(flags, device="cuda:0")
    torch.cuda.synchronize()
    rc = lib.osc_mft_set_closed_loop_batched(s.robot.handle, s.mft.task_id, 1, d_f.data_ptr(), sp.capi.OSC_MEM_DEVICE)
    assert rc == sp.capi.OSC_ERR_INVALID_ARGUMENT
    after = (s.mft.getForceMotionSpaces(), s.mft.getMomentRotMotionSpaces())
    for x, y in zip(before, after):
        assert all(np.array_equal(u, v) for u, v in zip(x, y))
    s.sense(0); ref.sense(0)
    assert np.array_equal(s.cycle(), ref.cycle())


def test_fp32_runs_while_every_robot_is_free():
    import sai_primitives_b200 as sp
    N = 256
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    s = Setup(q, dq, oracle=False, passivity=False)
    ref = Setup(q, dq, oracle=False, passivity=False)
    s.mft.parametrizeForceMotionSpaces(np.zeros(N, np.int32), np.zeros((N, 3)))
    s.mft.setClosedLoopForceControl(np.zeros(N, bool))
    s.ctrl.setPrecision("fp32")
    t32, t64 = s.cycle(), ref.cycle()
    assert rel_err(t32, t64).max() < 1e-4
    d = np.zeros(N, np.int32); d[17] = 1
    s.mft.parametrizeForceMotionSpaces(d, np.tile([0.0, 0.0, 1.0], (N, 1)))
    s.ctrl.updateControllerTaskModels()
    with pytest.raises(NotImplementedError):
        s.ctrl.computeControlTorques()
    s.ctrl.setPrecision("fp64")
    s.cycle()


def _needs_reference_library():
    from oracle import sai_ref
    return pytest.mark.skipif(not sai_ref.available(oriented=True), reason="needs oracle/_ref/libsai_ref_orient.so")


@_needs_reference_library()
def test_per_robot_resets_with_the_internal_otg_against_the_reference():
    """config 2 with the reference's defaults (internal OTG on in both tasks): half of the robots switch to force dimension 1
    along their own normal mid-motion; was_reset, desired states and torques against the reference's compiled classes"""
    import sai_primitives_b200 as sp
    from oracle.sai_ref import RefBatch
    N, K, SWITCH = 32, 120, 40
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.1)
    link, pt = TASK_POINTS["panda"]
    comp = (np.eye(3), np.array(pt))
    robot = sp.BatchedRobot("panda", N)
    robot.setQ(q); robot.setDq(dq); robot.updateModel()
    mft = sp.MotionForceTask(robot, link, comp); jt = sp.JointTask(robot)
    ctrl = sp.RobotController(robot, [mft, jt])
    rb = RefBatch("panda", N, oriented=True); rb.set_state(q, dq)
    omft = rb.add_mft(link, comp, otg=True); rb.add_jt(otg=True); rb.finalize()
    gx = mft.getCurrentPosition() + np.random.default_rng(4).uniform(-0.05, 0.05, (N, 3))
    dims = (np.arange(N) % 2).astype(np.int32)
    normals = np.array([_unit(rng_for(k, stream=61).normal(size=3)) for k in range(N)])
    for k in range(K):
        if k == SWITCH:
            r = mft.parametrizeForceMotionSpaces(dims, normals)
            ref = np.array([t.parametrizeForceMotionSpaces(int(dims[i]), normals[i]) for i, t in enumerate(omft)])
            assert np.array_equal(r, ref.astype(bool))
            gx = mft.getGoalPosition()
        mft.setGoalPosition(gx)
        for i in range(N):
            omft[i].setGoalPosition(gx[i])
        ctrl.updateControllerTaskModels()
        tau = ctrl.computeControlTorques()
        assert rel_err(tau, rb.cycle()).max() < REL_TOL, k
        des = mft.getDesiredPosition()
        assert np.abs(des - np.array([t.getDesiredPosition() for t in omft])).max() < 1e-9, k
        q = q + 0.0005 * dq
        robot.setQ(q); robot.updateModel(); rb.set_state(q, dq)
