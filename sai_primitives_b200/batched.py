"""Python host-side mirror of the reference interface for the batched path.

Same class and method names as the reference (JointTask, MotionForceTask,
RobotController; SaiModel's role is played by BatchedRobot), every call forwarding to
the C ABI (capi.py -> libsai_b200_osc.so -> sm_100a kernels).  Per-robot quantities are
numpy arrays of shape [n_robots, ncomp] (a single vector of ncomp values is broadcast to
all robots) or, for zero-copy use, raw device pointers in the SoA layout of the C ABI.

Differences from the reference, by design (BASELINE.json north_star):
  * internal OTG: acceleration-limited, phase-synchronised (the reference's default, JointTask.h:38-42 /
    MotionForceTask.h:67-74) runs batched on the device; the jerk-limited variant is not built and raises.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import capi
from .capi import OscError

FULL_DYNAMIC_DECOUPLING = capi.FULL_DYNAMIC_DECOUPLING
BOUNDED_INERTIA_ESTIMATES = capi.BOUNDED_INERTIA_ESTIMATES
IMPEDANCE = capi.IMPEDANCE


def _check(handle, rc):
    if rc == capi.OSC_OK:
        return
    lib = capi.load_library()
    msg = lib.osc_last_error(handle)
    msg = msg.decode() if msg else ""
    if rc == capi.OSC_ERR_INVALID_ARGUMENT:
        raise ValueError(msg)              # the reference throws std::invalid_argument
    if rc == capi.OSC_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise OscError(rc, msg)


def _int_ptr(a):
    assert a.dtype == np.int32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def _soa(a, n_robots, ncomp):
    """[N, ncomp] (or [ncomp] broadcast) -> contiguous SoA [ncomp, N]"""
    a = np.asarray(a, dtype=np.float64)
    if a.shape == (n_robots, ncomp):
        return np.ascontiguousarray(a.T)
    raise ValueError("expected an array of shape (%d, %d), got %s" % (n_robots, ncomp, a.shape))


def robot_mask(robots, n_robots):
    """The int32 [N] mask of osc_reset_robots for `robots`: None (every robot: no mask), a bool [N] array, or an array of robot
    indices in 0..N-1.  Raises ValueError for anything else, an index out of range included."""
    if robots is None:
        return None
    a = np.asarray(robots)
    if a.dtype == np.bool_:
        if a.shape != (n_robots,):
            raise ValueError("a boolean robot selection must have shape (%d,), got %s" % (n_robots, a.shape))
        return np.ascontiguousarray(a, dtype=np.int32)
    if a.ndim != 1:
        raise ValueError("robots must be a boolean array of shape (%d,) or a 1-D array of robot indices" % n_robots)
    if a.size == 0:
        return np.zeros(n_robots, dtype=np.int32)
    # a list mixing booleans and integers is neither form (numpy would read [True, 2] as the indices [1, 2])
    mixed = not isinstance(robots, np.ndarray) and any(isinstance(x, (bool, np.bool_)) for x in robots)
    if mixed or not np.issubdtype(a.dtype, np.integer):
        raise ValueError("robots must be a boolean array of shape (%d,) or a 1-D array of robot indices" % n_robots)
    if a.min() < 0 or a.max() >= n_robots:
        raise ValueError("robot index out of range [0, %d)" % n_robots)
    mask = np.zeros(n_robots, dtype=np.int32)
    mask[a] = 1
    return mask


def _reset(robot, task_id, robots, mode):
    mask = robot_mask(robots, robot.n_robots)
    ptr = None if mask is None else _int_ptr(mask)
    _check(robot.handle, robot._lib.osc_reset_robots(robot.handle, task_id, ptr, capi.OSC_MEM_HOST, mode))


def _reset_device(robot, task_id, mask_ptr, mode):
    _check(robot.handle, robot._lib.osc_reset_robots(robot.handle, task_id, C.c_void_p(mask_ptr), capi.OSC_MEM_DEVICE, mode))


def registerUrdf(model_name, urdf_file_or_text):
    """SURVEY.md row f-3: make a URDF robot (a serial chain) available under `model_name`, the counterpart of
    `SaiModel(robot_file)` (examples/05-using_robot_controller/05-using_robot_controller.cpp:64).  Accepts a file name
    or the XML text; afterwards `BatchedRobot(model_name, n_robots)` and link names work as for the built-in robots."""
    lib = capi.load_library()
    text = str(urdf_file_or_text)
    if text.lstrip().startswith("<"):
        rc = lib.osc_urdf_register(model_name.encode(), text.encode())
    else:
        rc = lib.osc_urdf_register_file(model_name.encode(), text.encode())
    if rc != 0:
        raise ValueError("URDF [%s]: %s" % (model_name, lib.osc_urdf_last_error().decode()))


class BatchedRobot:
    """N independent copies of one robot model on one CUDA device (the SaiModel of the batch)."""

    def __init__(self, robot_name_or_desc, n_robots, device=0, T_world_robot=None, gravity=None):
        lib = self._lib = capi.load_library()
        if isinstance(robot_name_or_desc, str):
            self.name = robot_name_or_desc
            desc = capi.ModelDesc()
            rc = lib.osc_builtin_model(robot_name_or_desc.encode(), C.byref(desc))
            if rc != capi.OSC_OK:
                raise ValueError("unknown built-in robot model [%s]" % robot_name_or_desc)
        else:
            self.name = None
            desc = robot_name_or_desc
        if T_world_robot is not None:
            R, t = T_world_robot
            desc.R_world_base[:] = list(np.asarray(R, dtype=np.float64).reshape(9))
            desc.t_world_base[:] = list(np.asarray(t, dtype=np.float64).reshape(3))
        if gravity is not None:
            desc.gravity_world[:] = list(np.asarray(gravity, dtype=np.float64).reshape(3))
        self.desc = desc
        self.n_robots = int(n_robots)
        h = C.c_void_p()
        rc = lib.osc_create(C.byref(desc), self.n_robots, int(device), C.byref(h))
        if rc != capi.OSC_OK:
            msg = lib.osc_last_error(None)
            raise OscError(rc, msg.decode() if msg else "osc_create failed")
        self.handle = h
        self._finalized = False
        n = desc.n
        self._q = np.zeros((self.n_robots, n))
        self._dq = np.zeros((self.n_robots, n))

    def close(self):
        if getattr(self, "handle", None):
            self._lib.osc_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def dof(self):
        return int(self.desc.n)

    def setQ(self, q):
        self._q = np.asarray(q, dtype=np.float64).reshape(self.n_robots, self.dof()).copy()

    def setDq(self, dq):
        self._dq = np.asarray(dq, dtype=np.float64).reshape(self.n_robots, self.dof()).copy()

    def updateModel(self):
        """SaiModel::updateModel for the batch: uploads q, dq (the kinematics/dynamics are
        evaluated inside the fused control-cycle kernel)."""
        q = _soa(self._q, self.n_robots, self.dof())
        dq = _soa(self._dq, self.n_robots, self.dof())
        _check(self.handle, self._lib.osc_set_state(self.handle, capi.host_ptr(q), capi.host_ptr(dq), capi.OSC_MEM_HOST))

    def setStateDevice(self, q_ptr, dq_ptr):
        """zero-copy: SoA [n, N] device buffers, borrowed until the next state update"""
        _check(self.handle, self._lib.osc_set_state(self.handle, C.c_void_p(q_ptr), C.c_void_p(dq_ptr), capi.OSC_MEM_DEVICE))

    def linkFrame(self, link_name):
        f = capi.LinkFrame()
        if self.name is None:
            raise ValueError("link lookup by name needs a built-in model")
        rc = self._lib.osc_builtin_link(self.name.encode(), link_name.encode(), C.byref(f))
        if rc != capi.OSC_OK:
            raise ValueError("link [%s] does not exist in robot [%s]" % (link_name, self.name))
        return f

    def evalModel(self, link_name, pos_in_link=(0.0, 0.0, 0.0)):
        """kinematics/dynamics stage on its own: dict(M [N,n,n], J [N,6,n], x [N,3], R [N,3,3], g [N,n])"""
        n, N = self.dof(), self.n_robots
        f = self.linkFrame(link_name)
        pt = (C.c_double * 3)(*[float(v) for v in pos_in_link])
        M = np.zeros((n * n, N)); J = np.zeros((6 * n, N)); x = np.zeros((3, N)); R = np.zeros((9, N)); g = np.zeros((n, N))
        _check(self.handle, self._lib.osc_eval_model(self.handle, -1, C.byref(f), pt, capi.host_ptr(M), capi.host_ptr(J),
                                                     capi.host_ptr(x), capi.host_ptr(R), capi.host_ptr(g), capi.OSC_MEM_HOST))
        return dict(M=M.T.reshape(N, n, n).copy(), J=J.T.reshape(N, 6, n).copy(), x=x.T.copy(),
                    R=R.T.reshape(N, 3, 3).copy(), g=g.T.copy())

    def status(self):
        out = np.zeros(self.n_robots, dtype=np.uint32)
        _check(self.handle, self._lib.osc_get_status(self.handle, out.ctypes.data_as(C.c_void_p), capi.OSC_MEM_HOST))
        return out

    def launchCount(self):
        return int(self._lib.osc_launch_count(self.handle))

    def sync(self):
        _check(self.handle, self._lib.osc_sync(self.handle))

    def enableObservers(self, flag=True):
        """osc_enable_observers: per-cycle refresh of getCurrentLinearVelocity / AngularVelocity / getUnitMassForce (default on)"""
        _check(self.handle, self._lib.osc_enable_observers(self.handle, 1 if flag else 0))

    def setStream(self, cuda_stream_ptr):
        _check(self.handle, self._lib.osc_set_stream(self.handle, C.c_void_p(cuda_stream_ptr)))


class BatchedSimulation:
    """Simulation side of the control loop for N robots (SURVEY.md row f-1), with the method names the reference examples
    use on sai-simulation (examples/05-using_robot_controller/05-using_robot_controller.cpp:223-231): setTimestep,
    setJointTorques, integrate, getJointPositions, getJointVelocities.  Semi-implicit Euler on
    ddq = M^-1 (tau - b - g) of the robot's model; state and torques are robots x dof arrays."""

    def __init__(self, robot: BatchedRobot, q, dq, timestep=0.001):
        self._robot = robot
        self._lib = robot._lib
        n, N = robot.dof(), robot.n_robots
        self._q = np.ascontiguousarray(np.asarray(q, dtype=np.float64).reshape(N, n).T)
        self._dq = np.ascontiguousarray(np.asarray(dq, dtype=np.float64).reshape(N, n).T)
        self._tau = np.zeros((n, N))
        self._dt = float(timestep)

    def setTimestep(self, dt):
        self._dt = float(dt)

    def setJointTorques(self, tau):
        n, N = self._robot.dof(), self._robot.n_robots
        self._tau = np.ascontiguousarray(np.asarray(tau, dtype=np.float64).reshape(N, n).T)

    def integrate(self, substeps=1):
        P = C.POINTER(C.c_double)
        _check(self._robot.handle, self._lib.osc_sim_integrate(self._robot.handle, self._q.ctypes.data_as(P), self._dq.ctypes.data_as(P),
                                                               self._tau.ctypes.data_as(P), self._dt, int(substeps), capi.OSC_MEM_HOST))

    def setJointPositions(self, q, robots=None):
        """sai-simulation's setJointPositions, for every robot ([N, n]) or for the robots selected by `robots` (as in
        RobotController.resetRobots; q is then [N, n] or [len(selected), n])"""
        self._set_rows(self._q, q, robots)

    def setJointVelocities(self, dq, robots=None):
        self._set_rows(self._dq, dq, robots)

    def _set_rows(self, dst, v, robots):
        n, N = self._robot.dof(), self._robot.n_robots
        v = np.asarray(v, dtype=np.float64)
        mask = robot_mask(robots, N)
        sel = np.ones(N, dtype=bool) if mask is None else mask != 0
        if v.shape == (N, n):
            v = v[sel]
        if v.shape != (int(sel.sum()), n):
            raise ValueError("expected an array of shape (%d, %d) or (%d, %d), got %s" % (N, n, int(sel.sum()), n, v.shape))
        dst[:, sel] = v.T

    def getJointPositions(self):
        return self._q.T.copy()

    def getJointVelocities(self):
        return self._dq.T.copy()


class _Task:
    def __init__(self, robot: BatchedRobot, task_name, loop_timestep):
        self._robot = robot
        self._lib = robot._lib
        self._task_name = task_name
        self._loop_timestep = loop_timestep
        self.task_id = -1

    def getTaskName(self):
        return self._task_name

    def getLoopTimestep(self):
        return self._loop_timestep

    def _set(self, field, value):
        N = self._robot.n_robots
        ncomp = self._lib.osc_field_ncomp(self._robot.handle, self.task_id, field)
        if ncomp < 0:
            raise ValueError("unknown field")
        a = np.asarray(value, dtype=np.float64)
        if a.ndim == 1:  # one value for every robot
            if a.size != ncomp:
                raise ValueError("expected %d components, got %d" % (ncomp, a.size))
            flat = np.ascontiguousarray(a)
            rc = self._lib.osc_set_field(self._robot.handle, self.task_id, field, capi.host_ptr(flat), capi.OSC_MEM_HOST, 1)
        else:
            soa = _soa(a.reshape(N, ncomp), N, ncomp)
            rc = self._lib.osc_set_field(self._robot.handle, self.task_id, field, capi.host_ptr(soa), capi.OSC_MEM_HOST, 0)
        _check(self._robot.handle, rc)

    def _get(self, field):
        N = self._robot.n_robots
        ncomp = self._lib.osc_field_ncomp(self._robot.handle, self.task_id, field)
        if ncomp < 0:
            raise ValueError("unknown field")
        out = np.zeros((ncomp, N))
        _check(self._robot.handle, self._lib.osc_get_field(self._robot.handle, self.task_id, field, capi.host_ptr(out), capi.OSC_MEM_HOST))
        return out.T.copy()

    def _set_gains(self, group, ncomp, kp, kv, ki, broadcast_form):
        """osc_set_gains.  Each gain is a scalar or an (ncomp,) vector applied to every robot (what broadcast_form accepts, as
        before per-robot gains existed: any array of 1 or ncomp values), or a 2-D (N, 1) / (N, ncomp) array with one row per robot.
        When one of the three is per robot, the other two are expanded to every robot.  An array of 1 or ncomp values is always
        the broadcast form, as it was before: with N == ncomp robots an (N, 1) array is read as ncomp per-component gains for every
        robot, not as one gain per robot (pass (N, ncomp) then)."""
        N = self._robot.n_robots
        arrs = [np.asarray(x, dtype=np.float64) for x in (kp, kv, ki)]

        def per_robot(a):
            return a.ndim == 2 and a.shape[0] == N and a.shape[1] in (1, ncomp) and a.size not in (1, ncomp)

        if not any(per_robot(a) for a in arrs):
            vals = [np.ascontiguousarray(v, dtype=np.float64) for v in broadcast_form(*arrs)]
            _check(self._robot.handle, self._lib.osc_set_gains(self._robot.handle, self.task_id, group, capi.host_ptr(vals[0]),
                                                              capi.host_ptr(vals[1]), capi.host_ptr(vals[2]), capi.OSC_MEM_HOST, 0))
            return
        soa = []
        for a in arrs:
            if per_robot(a):
                full = np.broadcast_to(a, (N, ncomp))
            elif a.size in (1, ncomp):
                full = np.broadcast_to(a.reshape(1, -1), (N, ncomp))
            else:
                raise ValueError("per-robot gains must have shape (%d, 1) or (%d, %d), or 1 or %d values for every robot; got %s"
                                 % (N, N, ncomp, ncomp, a.shape))
            soa.append(np.ascontiguousarray(full.T))
        _check(self._robot.handle, self._lib.osc_set_gains(self._robot.handle, self.task_id, group, capi.host_ptr(soa[0]),
                                                          capi.host_ptr(soa[1]), capi.host_ptr(soa[2]), capi.OSC_MEM_HOST, 1))

    def _set_gains_device(self, group, kp_ptr, kv_ptr, ki_ptr):
        """per-robot gains from device memory, SoA [ncomp, N] each (zero copy, like BatchedRobot.setStateDevice)"""
        _check(self._robot.handle, self._lib.osc_set_gains(self._robot.handle, self.task_id, group, C.c_void_p(kp_ptr), C.c_void_p(kv_ptr),
                                                          C.c_void_p(ki_ptr), capi.OSC_MEM_DEVICE, 1))

    def _get_gains(self, group, ncomp):
        N = self._robot.n_robots
        out = [np.zeros((ncomp, N)) for _ in range(3)]
        _check(self._robot.handle, self._lib.osc_get_gains(self._robot.handle, self.task_id, group, capi.host_ptr(out[0]),
                                                          capi.host_ptr(out[1]), capi.host_ptr(out[2]), capi.OSC_MEM_HOST))
        return tuple(o.T.copy() for o in out)

    def reInitializeTask(self, robots=None):
        """TemplateTask::reInitializeTask for every robot or for those `robots` selects (a bool [N] array or robot indices)"""
        _reset(self._robot, self.task_id, robots, capi.OSC_RESET_REINITIALIZE)

    def reInitializeTaskDevice(self, mask_ptr):
        """the same with an int32 [N] device mask (non-zero selects), ordered with the cycles in the robot's stream"""
        _reset_device(self._robot, self.task_id, mask_ptr, capi.OSC_RESET_REINITIALIZE)

    # TemplateTask.h:74,82,89 -- [N, n, n], evaluated from the robot's current state
    def _nullspace(self, field):
        n = self._robot.dof()
        return self._get(field).reshape(-1, n, n)

    def getTaskNullspace(self): return self._nullspace(capi.TASK_NULLSPACE)
    def getPreviousTasksNullspace(self): return self._nullspace(capi.TASK_PREVIOUS_NULLSPACE)
    def getTaskAndPreviousNullspace(self): return self._nullspace(capi.TASK_AND_PREVIOUS_NULLSPACE)


class JointTask(_Task):
    """reference src/tasks/JointTask.h: JointTask(robot, name, dt) / JointTask(robot, S, name, dt)"""

    task_type = capi.OSC_TASK_JOINT

    class DefaultParameters:
        """JointTask.h:31-45 (the entries this mirror consults at construction)"""
        use_internal_otg = True
        internal_otg_jerk_limited = False
        otg_max_velocity = math.pi / 3.0
        otg_max_acceleration = 2.0 * math.pi

    def __init__(self, robot: BatchedRobot, joint_selection_matrix=None, task_name="joint_task", loop_timestep=0.001):
        super().__init__(robot, task_name, loop_timestep)
        tid = C.c_int(-1)
        if joint_selection_matrix is None:
            rc = self._lib.osc_add_joint_task(robot.handle, None, 0, loop_timestep, C.byref(tid))
        else:
            S = np.ascontiguousarray(np.atleast_2d(np.asarray(joint_selection_matrix, dtype=np.float64)))
            if S.shape[1] != robot.dof():
                raise ValueError("joint selection matrix size not consistent with robot dof in JointTask constructor")
            rc = self._lib.osc_add_joint_task(robot.handle, capi.host_ptr(S), S.shape[0], loop_timestep, C.byref(tid))
        _check(robot.handle, rc)
        self.task_id = tid.value
        self._task_dof = self._lib.osc_get_task_dof(robot.handle, self.task_id)
        if self.DefaultParameters.use_internal_otg:     # JointTask.cpp:66-80
            self.enableInternalOtgAccelerationLimited(self.DefaultParameters.otg_max_velocity, self.DefaultParameters.otg_max_acceleration)

    def getTaskDof(self):
        return self._task_dof

    def isFullJointTask(self):
        return self._task_dof == self._robot.dof()

    def _params(self):
        p = capi.JointParams()
        _check(self._robot.handle, self._lib.osc_joint_get_params(self._robot.handle, self.task_id, C.byref(p)))
        return p

    def _apply(self, p):
        _check(self._robot.handle, self._lib.osc_joint_set_params(self._robot.handle, self.task_id, C.byref(p)))

    def setGoalPosition(self, v): self._set(capi.JT_GOAL_POSITION, v)
    def setGoalVelocity(self, v): self._set(capi.JT_GOAL_VELOCITY, v)
    def setGoalAcceleration(self, v): self._set(capi.JT_GOAL_ACCELERATION, v)
    def getGoalPosition(self): return self._get(capi.JT_GOAL_POSITION)
    def getGoalVelocity(self): return self._get(capi.JT_GOAL_VELOCITY)
    def getGoalAcceleration(self): return self._get(capi.JT_GOAL_ACCELERATION)
    # JointTask.h:162-176: what the control law tracks (the internal OTG's output when it is on, the goal otherwise)
    def getDesiredPosition(self): return self._get(capi.JT_DESIRED_POSITION)
    def getDesiredVelocity(self): return self._get(capi.JT_DESIRED_VELOCITY)
    def getDesiredAcceleration(self): return self._get(capi.JT_DESIRED_ACCELERATION)

    def setGains(self, kp, kv, ki=0.0):
        """JointTask::setGains; also per robot: (N, 1) or (N, k) arrays (see _Task._set_gains)"""
        k = self._task_dof

        def broadcast_form(kp, kv, ki):
            kp, kv, ki = (np.atleast_1d(x).ravel() for x in (kp, kv, ki))
            if kp.size == 1 and kv.size == 1 and ki.size == 1:
                kp, kv, ki = np.full(k, kp[0]), np.full(k, kv[0]), np.full(k, ki[0])
            if kp.size != k or kv.size != k or ki.size != k:
                raise ValueError("size of gain vectors inconsistent with number of task dofs in JointTask::setGains")
            return kp, kv, ki

        self._set_gains(capi.GAINS_JOINT, k, kp, kv, ki, broadcast_form)

    def setGainsDevice(self, kp_ptr, kv_ptr, ki_ptr):
        """per-robot gains from device memory: SoA [k, N] each"""
        self._set_gains_device(capi.GAINS_JOINT, kp_ptr, kv_ptr, ki_ptr)

    def getGains(self):
        """(kp, kv, ki), each [N, k]"""
        return self._get_gains(capi.GAINS_JOINT, self._task_dof)

    def setDynamicDecouplingType(self, t):
        p = self._params(); p.dynamic_decoupling_type = int(t); self._apply(p)

    def setBoundedInertiaEstimateThreshold(self, thr):
        p = self._params(); p.bie_threshold = float(thr); self._apply(p)

    def enableVelocitySaturation(self, saturation_velocity=math.pi / 3):
        sat = np.atleast_1d(np.asarray(saturation_velocity, dtype=np.float64))
        k = self._task_dof
        if sat.size == 1:
            sat = np.full(k, sat[0])
        if sat.size != k:
            raise ValueError("saturation velocity vector size not consistent with task dof in JointTask::enableVelocitySaturation")
        p = self._params()
        p.use_velocity_saturation = 1
        for a in range(k):
            p.saturation_velocity[a] = sat[a]
        self._apply(p)

    def disableVelocitySaturation(self):
        p = self._params(); p.use_velocity_saturation = 0; self._apply(p)

    def enableInternalOtgAccelerationLimited(self, max_velocity, max_acceleration):
        """JointTask.cpp:358-380: scalars or vectors of task dof"""
        k = self._task_dof
        v = np.atleast_1d(np.asarray(max_velocity, dtype=np.float64)); a = np.atleast_1d(np.asarray(max_acceleration, dtype=np.float64))
        if v.size == 1 and a.size == 1:
            v, a = np.full(k, v[0]), np.full(k, a[0])
        if v.size != k or a.size != k:
            raise ValueError("max velocity or max acceleration vector size not consistent with task dof in JointTask::enableInternalOtgAccelerationLimited")
        v, a = np.ascontiguousarray(v), np.ascontiguousarray(a)
        _check(self._robot.handle, self._lib.osc_joint_enable_internal_otg(self._robot.handle, self.task_id,
               v.ctypes.data_as(C.POINTER(C.c_double)), a.ctypes.data_as(C.POINTER(C.c_double))))

    def enableInternalOtgJerkLimited(self, *a, **k):
        raise NotImplementedError("the jerk-limited internal OTG is not built (OSC_ERR_UNSUPPORTED); use enableInternalOtgAccelerationLimited")

    def disableInternalOtg(self):
        _check(self._robot.handle, self._lib.osc_disable_internal_otg(self._robot.handle, self.task_id))

    def getInternalOtgEnabled(self):
        return self._lib.osc_internal_otg_enabled(self._robot.handle, self.task_id) == 1

    def getInternalOtgFlags(self):
        out = np.zeros(self._robot.n_robots, dtype=np.int32)
        _check(self._robot.handle, self._lib.osc_get_internal_otg_flags(self._robot.handle, self.task_id, out.ctypes.data_as(C.c_void_p), capi.OSC_MEM_HOST))
        return out


class MotionForceTask(_Task):
    """reference src/tasks/MotionForceTask.h:96-110 (both constructors)"""

    task_type = capi.OSC_TASK_MOTION_FORCE

    class DefaultParameters:
        """MotionForceTask.h:40-75 (the entries this mirror consults at construction)"""
        use_internal_otg = True
        internal_otg_jerk_limited = False
        otg_max_linear_velocity = 0.3
        otg_max_linear_acceleration = 2.0
        otg_max_angular_velocity = math.pi / 3
        otg_max_angular_acceleration = 2.0 * math.pi

    def __init__(self, robot: BatchedRobot, link_name, compliant_frame=None,
                 controlled_directions_translation=None, controlled_directions_rotation=None,
                 task_name="motion_force_task", is_force_motion_parametrization_in_compliant_frame=False,
                 loop_timestep=0.001):
        super().__init__(robot, task_name, loop_timestep)
        d = capi.MftDesc()
        d.link = robot.linkFrame(link_name)
        R, t = (np.eye(3), np.zeros(3)) if compliant_frame is None else compliant_frame
        d.compliant_R[:] = list(np.asarray(R, dtype=np.float64).reshape(9))
        d.compliant_t[:] = list(np.asarray(t, dtype=np.float64).reshape(3))
        if controlled_directions_translation is None and controlled_directions_rotation is None:
            d.partial = 0
        else:
            d.partial = 1
            dt_ = list(controlled_directions_translation or [])
            dr_ = list(controlled_directions_rotation or [])
            if len(dt_) > 3 or len(dr_) > 3:
                raise ValueError("at most 3 controlled directions per block")
            d.n_dirs_translation = len(dt_)
            d.n_dirs_rotation = len(dr_)
            for i, v in enumerate(dt_):
                d.dirs_translation[i][:] = [float(x) for x in v]
            for i, v in enumerate(dr_):
                d.dirs_rotation[i][:] = [float(x) for x in v]
        d.force_motion_in_compliant_frame = 1 if is_force_motion_parametrization_in_compliant_frame else 0
        d.loop_timestep = loop_timestep
        tid = C.c_int(-1)
        _check(robot.handle, self._lib.osc_add_motion_force_task(robot.handle, C.byref(d), C.byref(tid)))
        self.task_id = tid.value
        self._link_name = link_name
        if self.DefaultParameters.use_internal_otg:     # MotionForceTask.cpp:170-191
            D = self.DefaultParameters
            self.enableInternalOtgAccelerationLimited(D.otg_max_linear_velocity, D.otg_max_linear_acceleration, D.otg_max_angular_velocity, D.otg_max_angular_acceleration)

    def _params(self):
        p = capi.MftParams()
        _check(self._robot.handle, self._lib.osc_mft_get_params(self._robot.handle, self.task_id, C.byref(p)))
        return p

    def _apply(self, p):
        _check(self._robot.handle, self._lib.osc_mft_set_params(self._robot.handle, self.task_id, C.byref(p)))

    # goals
    def setGoalPosition(self, v): self._set(capi.MFT_GOAL_POSITION, v)
    def setGoalOrientation(self, R):
        R = np.asarray(R, dtype=np.float64)
        self._set(capi.MFT_GOAL_ORIENTATION, R.reshape(-1, 9) if R.ndim == 3 else R.reshape(9))
    def setGoalLinearVelocity(self, v): self._set(capi.MFT_GOAL_LINEAR_VELOCITY, v)
    def setGoalAngularVelocity(self, v): self._set(capi.MFT_GOAL_ANGULAR_VELOCITY, v)
    def setGoalLinearAcceleration(self, v): self._set(capi.MFT_GOAL_LINEAR_ACCELERATION, v)
    def setGoalAngularAcceleration(self, v): self._set(capi.MFT_GOAL_ANGULAR_ACCELERATION, v)
    def setGoalForce(self, v): self._set(capi.MFT_GOAL_FORCE, v)
    def setGoalMoment(self, v): self._set(capi.MFT_GOAL_MOMENT, v)
    def setType1Posture(self, q): self._set(capi.MFT_TYPE1_POSTURE, q)
    # observers
    def getGoalPosition(self): return self._get(capi.MFT_GOAL_POSITION)
    def getGoalOrientation(self): return self._get(capi.MFT_GOAL_ORIENTATION).reshape(-1, 3, 3)
    def getCurrentPosition(self): return self._get(capi.MFT_CURRENT_POSITION)
    def getCurrentOrientation(self): return self._get(capi.MFT_CURRENT_ORIENTATION).reshape(-1, 3, 3)
    def getCurrentLinearVelocity(self): return self._get(capi.MFT_CURRENT_LINEAR_VELOCITY)
    def getCurrentAngularVelocity(self): return self._get(capi.MFT_CURRENT_ANGULAR_VELOCITY)
    def getSensedForceControlWorldFrame(self): return self._get(capi.MFT_SENSED_FORCE_CONTROL_WORLD)
    def getSensedMomentControlWorldFrame(self): return self._get(capi.MFT_SENSED_MOMENT_CONTROL_WORLD)
    def getUnitMassForce(self): return self._get(capi.MFT_UNIT_MASS_FORCE)
    # MotionForceTask.h:268-269, :613-616
    def getPositionError(self): return self._get(capi.MFT_POSITION_ERROR)
    def getOrientationError(self): return self._get(capi.MFT_ORIENTATION_ERROR)
    def sigmaForce(self): return self._get(capi.MFT_SIGMA_FORCE).reshape(-1, 3, 3)
    def sigmaPosition(self): return self._get(capi.MFT_SIGMA_POSITION).reshape(-1, 3, 3)
    def sigmaMoment(self): return self._get(capi.MFT_SIGMA_MOMENT).reshape(-1, 3, 3)
    def sigmaOrientation(self): return self._get(capi.MFT_SIGMA_ORIENTATION).reshape(-1, 3, 3)

    @staticmethod
    def _g3(kp, kv, ki, what):
        kp, kv, ki = (np.atleast_1d(np.asarray(x, dtype=np.float64)) for x in (kp, kv, ki))
        if kp.size == 1 and kv.size == 1 and ki.size == 1:
            return np.full(3, kp[0]), np.full(3, kv[0]), np.full(3, ki[0])
        if kp.size != 3 or kv.size != 3 or ki.size != 3:
            raise ValueError("gains should be of size 1 or 3 in MotionForceTask::%s" % what)
        return kp, kv, ki

    @staticmethod
    def _g1(kp, kv, ki, what):
        vals = [np.asarray(x, dtype=np.float64) for x in (kp, kv, ki)]
        if any(v.size != 1 for v in vals):
            raise ValueError("gains should be scalars in MotionForceTask::%s" % what)
        return [v.reshape(1) for v in vals]

    # MotionForceTask::set*ControlGains; also per robot: (N, 1) or (N, 3) arrays (see _Task._set_gains)
    def setPosControlGains(self, kp, kv, ki=0.0):
        self._set_gains(capi.GAINS_POSITION, 3, kp, kv, ki, lambda a, b, c: self._g3(a, b, c, "setPosControlGains"))

    def setOriControlGains(self, kp, kv, ki=0.0):
        self._set_gains(capi.GAINS_ORIENTATION, 3, kp, kv, ki, lambda a, b, c: self._g3(a, b, c, "setOriControlGains"))

    def setForceControlGains(self, kp, kv, ki):
        self._set_gains(capi.GAINS_FORCE, 1, kp, kv, ki, lambda a, b, c: self._g1(a, b, c, "setForceControlGains"))

    def setMomentControlGains(self, kp, kv, ki):
        self._set_gains(capi.GAINS_MOMENT, 1, kp, kv, ki, lambda a, b, c: self._g1(a, b, c, "setMomentControlGains"))

    # per-robot gains from device memory: SoA [3, N] (position, orientation) or [1, N] (force, moment) each
    def setPosControlGainsDevice(self, kp_ptr, kv_ptr, ki_ptr): self._set_gains_device(capi.GAINS_POSITION, kp_ptr, kv_ptr, ki_ptr)
    def setOriControlGainsDevice(self, kp_ptr, kv_ptr, ki_ptr): self._set_gains_device(capi.GAINS_ORIENTATION, kp_ptr, kv_ptr, ki_ptr)
    def setForceControlGainsDevice(self, kp_ptr, kv_ptr, ki_ptr): self._set_gains_device(capi.GAINS_FORCE, kp_ptr, kv_ptr, ki_ptr)
    def setMomentControlGainsDevice(self, kp_ptr, kv_ptr, ki_ptr): self._set_gains_device(capi.GAINS_MOMENT, kp_ptr, kv_ptr, ki_ptr)

    # (kp, kv, ki), each [N, 3] or [N, 1]
    def getPosControlGains(self): return self._get_gains(capi.GAINS_POSITION, 3)
    def getOriControlGains(self): return self._get_gains(capi.GAINS_ORIENTATION, 3)
    def getForceControlGains(self): return self._get_gains(capi.GAINS_FORCE, 1)
    def getMomentControlGains(self): return self._get_gains(capi.GAINS_MOMENT, 1)

    def setFeedforwardForceGain(self, k):
        p = self._params(); p.kff_force = k; self._apply(p)

    def setFeedforwardmomentGain(self, k):
        p = self._params(); p.kff_moment = k; self._apply(p)

    def setMaxForceControlFeedbackOutput(self, v):
        p = self._params(); p.max_force_control_feedback_output = v; self._apply(p)

    def setMaxMomentControlFeedbackOutput(self, v):
        p = self._params(); p.max_moment_control_feedback_output = v; self._apply(p)

    def enableVelocitySaturation(self, linear_vel_sat=0.3, angular_vel_sat=math.pi / 3):
        p = self._params()
        p.use_velocity_saturation = 1
        p.linear_saturation_velocity = linear_vel_sat
        p.angular_saturation_velocity = angular_vel_sat
        self._apply(p)

    def disableVelocitySaturation(self):
        p = self._params(); p.use_velocity_saturation = 0; self._apply(p)

    def setDynamicDecouplingType(self, t):
        p = self._params(); p.dynamic_decoupling_type = int(t); self._apply(p)

    def setBoundedInertiaEstimateThreshold(self, thr):
        p = self._params(); p.bie_threshold = float(thr); self._apply(p)

    def handleAllSingularitiesAsType1(self, flag):
        p = self._params(); p.enforce_type_1_strategy = 1 if flag else 0; self._apply(p)

    def enableSingularityHandling(self):
        p = self._params(); p.singularity_handling_enabled = 1; self._apply(p)

    def disableSingularityHandling(self):
        p = self._params(); p.singularity_handling_enabled = 0; self._apply(p)

    def setSingularityHandlingBounds(self, s_min, s_max):
        p = self._params(); p.s_min, p.s_max = s_min, s_max; self._apply(p)

    def setSingularityHandlingGains(self, kp_type_1, kv_type_1, kv_type_2):
        p = self._params(); p.kp_type_1, p.kv_type_1, p.kv_type_2 = kp_type_1, kv_type_1, kv_type_2; self._apply(p)

    def _parametrize(self, which, dim, axis, broadcast_fn):
        """A scalar dim with a 3-vector: every robot (returns bool).  dim[N] with axis[N, 3] (or one 3-vector for every robot):
        per robot, osc_mft_parametrize_spaces_batched (returns bool[N], True where the robot was reset)."""
        if np.ndim(dim) == 0:
            ax = (C.c_double * 3)(*[float(x) for x in np.asarray(axis, dtype=np.float64).reshape(3)]); r = C.c_int(0)
            _check(self._robot.handle, broadcast_fn(self._robot.handle, self.task_id, int(dim), ax, C.byref(r)))
            return bool(r.value)
        N = self._robot.n_robots
        dims = np.asarray(dim)
        if dims.shape != (N,) or not np.issubdtype(dims.dtype, np.integer):
            raise ValueError("per-robot dimensions must be an integer array of shape (%d,), got %s %s" % (N, dims.dtype, dims.shape))
        dims = np.ascontiguousarray(dims, dtype=np.int32)
        a = np.asarray(axis, dtype=np.float64)
        if a.shape == (3,):
            a = np.broadcast_to(a, (N, 3))
        axes = _soa(a, N, 3)
        reset = np.zeros(N, dtype=np.int32)
        _check(self._robot.handle, self._lib.osc_mft_parametrize_spaces_batched(self._robot.handle, self.task_id, which, _int_ptr(dims),
                                                                               capi.host_ptr(axes), _int_ptr(reset), capi.OSC_MEM_HOST))
        return reset != 0

    def parametrizeForceMotionSpaces(self, dim, axis=(0.0, 0.0, 0.0)):
        return self._parametrize(0, dim, axis, self._lib.osc_mft_parametrize_force_motion_spaces)

    def parametrizeMomentRotMotionSpaces(self, dim, axis=(0.0, 0.0, 0.0)):
        return self._parametrize(1, dim, axis, self._lib.osc_mft_parametrize_moment_rotmotion_spaces)

    def _parametrize_device(self, which, dims_ptr, axes_ptr, was_reset_ptr):
        _check(self._robot.handle, self._lib.osc_mft_parametrize_spaces_batched(self._robot.handle, self.task_id, which, C.c_void_p(dims_ptr),
                                                                               C.c_void_p(axes_ptr), C.c_void_p(was_reset_ptr or None),
                                                                               capi.OSC_MEM_DEVICE))

    # per robot from device memory: dims int32 [N], axes float64 SoA [3, N], was_reset int32 [N] or 0 (zero copy)
    def parametrizeForceMotionSpacesDevice(self, dims_ptr, axes_ptr, was_reset_ptr=0): self._parametrize_device(0, dims_ptr, axes_ptr, was_reset_ptr)
    def parametrizeMomentRotMotionSpacesDevice(self, dims_ptr, axes_ptr, was_reset_ptr=0): self._parametrize_device(1, dims_ptr, axes_ptr, was_reset_ptr)

    def _set_closed_loop(self, which, flag, broadcast_fn):
        if np.ndim(flag) == 0:
            _check(self._robot.handle, broadcast_fn(self._robot.handle, self.task_id, 1 if flag else 0))
            return
        N = self._robot.n_robots
        f = np.asarray(flag)
        if f.shape != (N,):
            raise ValueError("per-robot closed-loop flags must have shape (%d,), got %s" % (N, f.shape))
        f = np.ascontiguousarray(f.astype(bool), dtype=np.int32)
        _check(self._robot.handle, self._lib.osc_mft_set_closed_loop_batched(self._robot.handle, self.task_id, which, _int_ptr(f), capi.OSC_MEM_HOST))

    def setClosedLoopForceControl(self, flag=True):
        """bool for every robot, or bool[N] per robot"""
        self._set_closed_loop(0, flag, self._lib.osc_mft_set_closed_loop_force_control)

    def setClosedLoopMomentControl(self, flag=True):
        """bool for every robot, or bool[N] per robot"""
        self._set_closed_loop(1, flag, self._lib.osc_mft_set_closed_loop_moment_control)

    # per robot from device memory: int32 [N] of 0 / 1
    def setClosedLoopForceControlDevice(self, flags_ptr):
        _check(self._robot.handle, self._lib.osc_mft_set_closed_loop_batched(self._robot.handle, self.task_id, 0, C.c_void_p(flags_ptr), capi.OSC_MEM_DEVICE))

    def setClosedLoopMomentControlDevice(self, flags_ptr):
        _check(self._robot.handle, self._lib.osc_mft_set_closed_loop_batched(self._robot.handle, self.task_id, 1, C.c_void_p(flags_ptr), capi.OSC_MEM_DEVICE))

    def _get_spaces(self, which):
        N = self._robot.n_robots
        dims, cl = np.zeros(N, dtype=np.int32), np.zeros(N, dtype=np.int32)
        axes = np.zeros((3, N))
        _check(self._robot.handle, self._lib.osc_mft_get_spaces(self._robot.handle, self.task_id, which, _int_ptr(dims), capi.host_ptr(axes),
                                                                _int_ptr(cl), capi.OSC_MEM_HOST))
        return dims, axes.T.copy(), cl != 0

    def getForceMotionSpaces(self):
        """what the kernels use: (dims int32 [N], normalised axes [N, 3], closed-loop force control bool [N])"""
        return self._get_spaces(0)

    def getMomentRotMotionSpaces(self):
        """what the kernels use: (dims int32 [N], normalised axes [N, 3], closed-loop moment control bool [N])"""
        return self._get_spaces(1)

    def enablePassivity(self, ring_capacity=0):
        _check(self._robot.handle, self._lib.osc_mft_enable_passivity(self._robot.handle, self.task_id, 1, int(ring_capacity)))

    def disablePassivity(self):
        _check(self._robot.handle, self._lib.osc_mft_enable_passivity(self._robot.handle, self.task_id, 0, 0))

    def setForceSensorFrame(self, link_name, transformation_in_link):
        if link_name != self._link_name:
            raise ValueError("The link to which is attached the sensor should be the same as the link to which is "
                             "attached the control frame in MotionForceTask::setForceSensorFrame")
        R, t = transformation_in_link
        Rc = (C.c_double * 9)(*np.asarray(R, dtype=np.float64).reshape(9))
        tc = (C.c_double * 3)(*np.asarray(t, dtype=np.float64).reshape(3))
        _check(self._robot.handle, self._lib.osc_mft_set_force_sensor_frame(self._robot.handle, self.task_id, Rc, tc))

    def updateSensedForceAndMoment(self, sensed_force_sensor_frame, sensed_moment_sensor_frame):
        N = self._robot.n_robots
        f = np.asarray(sensed_force_sensor_frame, dtype=np.float64)
        m = np.asarray(sensed_moment_sensor_frame, dtype=np.float64)
        if f.shape == (3,):
            f = np.tile(f, (N, 1))
        if m.shape == (3,):
            m = np.tile(m, (N, 1))
        fs, ms = _soa(f, N, 3), _soa(m, N, 3)
        _check(self._robot.handle, self._lib.osc_mft_update_sensed_force_and_moment(
            self._robot.handle, self.task_id, capi.host_ptr(fs), capi.host_ptr(ms), capi.OSC_MEM_HOST))

    def resetIntegrators(self):
        _check(self._robot.handle, self._lib.osc_mft_reset_integrators(self._robot.handle, self.task_id, 0))

    def resetIntegratorsLinear(self):
        _check(self._robot.handle, self._lib.osc_mft_reset_integrators(self._robot.handle, self.task_id, 1))

    def resetIntegratorsAngular(self):
        _check(self._robot.handle, self._lib.osc_mft_reset_integrators(self._robot.handle, self.task_id, 2))

    def enableInternalOtgAccelerationLimited(self, max_linear_velelocity, max_linear_acceleration, max_angular_velocity, max_angular_acceleration):
        """MotionForceTask.cpp:511-523"""
        _check(self._robot.handle, self._lib.osc_mft_enable_internal_otg(self._robot.handle, self.task_id, float(max_linear_velelocity),
               float(max_linear_acceleration), float(max_angular_velocity), float(max_angular_acceleration)))

    def enableInternalOtgJerkLimited(self, *a, **k):
        raise NotImplementedError("the jerk-limited internal OTG is not built (OSC_ERR_UNSUPPORTED); use enableInternalOtgAccelerationLimited")

    def disableInternalOtg(self):
        _check(self._robot.handle, self._lib.osc_disable_internal_otg(self._robot.handle, self.task_id))

    def getInternalOtgEnabled(self):
        return self._lib.osc_internal_otg_enabled(self._robot.handle, self.task_id) == 1

    def getInternalOtgFlags(self):
        out = np.zeros(self._robot.n_robots, dtype=np.int32)
        _check(self._robot.handle, self._lib.osc_get_internal_otg_flags(self._robot.handle, self.task_id, out.ctypes.data_as(C.c_void_p), capi.OSC_MEM_HOST))
        return out

    # MotionForceTask.h:249-266
    def getDesiredPosition(self): return self._get(capi.MFT_DESIRED_POSITION)
    def getDesiredOrientation(self): return self._get(capi.MFT_DESIRED_ORIENTATION).reshape(-1, 3, 3)
    def getDesiredLinearVelocity(self): return self._get(capi.MFT_DESIRED_LINEAR_VELOCITY)
    def getDesiredAngularVelocity(self): return self._get(capi.MFT_DESIRED_ANGULAR_VELOCITY)
    def getDesiredLinearAcceleration(self): return self._get(capi.MFT_DESIRED_LINEAR_ACCELERATION)
    def getDesiredAngularAcceleration(self): return self._get(capi.MFT_DESIRED_ANGULAR_ACCELERATION)


class RobotController:
    """reference src/RobotController.h:47-87.  use_previous_torques=False reproduces the manual
    `tau = mft.computeTorques() + jt.computeTorques()` of examples/04-task_and_redundancy."""

    def __init__(self, robot: BatchedRobot, tasks, use_previous_torques=True):
        if len(tasks) == 0:
            raise ValueError("RobotController must have at least one task")
        names = []
        for i, t in enumerate(tasks):
            if t._robot is not robot:
                raise ValueError("All tasks must have the same robot model in RobotController")
            if t.getTaskName() in names:
                raise ValueError("Tasks in RobotController must have unique names")
            names.append(t.getTaskName())
            if t.task_id != i:
                raise ValueError("tasks must be given in the order they were created on this robot")
        self._robot = robot
        self._lib = robot._lib
        self._tasks = list(tasks)
        _check(robot.handle, self._lib.osc_finalize_controller(robot.handle, 1 if use_previous_torques else 0))

    def updateControllerTaskModels(self):
        _check(self._robot.handle, self._lib.osc_update_task_models(self._robot.handle))

    def computeControlTorques(self):
        n, N = self._robot.dof(), self._robot.n_robots
        tau = np.zeros((n, N))
        _check(self._robot.handle, self._lib.osc_compute_control_torques(self._robot.handle, capi.host_ptr(tau), capi.OSC_MEM_HOST))
        return tau.T.copy()

    def step(self, q, dq):
        """fused cycle through host buffers: [N, n] in, [N, n] out"""
        n, N = self._robot.dof(), self._robot.n_robots
        qs, dqs = _soa(q, N, n), _soa(dq, N, n)
        tau = np.zeros((n, N))
        _check(self._robot.handle, self._lib.osc_step(self._robot.handle, capi.host_ptr(qs), capi.host_ptr(dqs), capi.host_ptr(tau), capi.OSC_MEM_HOST))
        return tau.T.copy()

    def stepDevice(self, q_ptr, dq_ptr, tau_ptr):
        _check(self._robot.handle, self._lib.osc_step(self._robot.handle, C.c_void_p(q_ptr), C.c_void_p(dq_ptr), C.c_void_p(tau_ptr), capi.OSC_MEM_DEVICE))

    def setPrecision(self, precision):
        """osc_set_precision (no reference counterpart: the reference is double precision): "fp64" (default) or "fp32" -- the optional
        single-precision mode of the fused kernel, for a full six-dof MotionForceTask under pure motion control with or without a
        full JointTask; any other hierarchy raises on the next computeControlTorques while it is on"""
        code = {"fp64": capi.OSC_PRECISION_FP64, "fp32": capi.OSC_PRECISION_FP32}[precision]
        _check(self._robot.handle, self._lib.osc_set_precision(self._robot.handle, code))

    def getPrecision(self):
        return "fp32" if self._lib.osc_get_precision(self._robot.handle) == capi.OSC_PRECISION_FP32 else "fp64"

    def enableGravityCompensation(self, flag):
        _check(self._robot.handle, self._lib.osc_enable_gravity_compensation(self._robot.handle, 1 if flag else 0))

    def enableTorqueSaturation(self, flag):
        _check(self._robot.handle, self._lib.osc_enable_torque_saturation(self._robot.handle, 1 if flag else 0))

    def enableJointLimitAvoidance(self, flag):
        _check(self._robot.handle, self._lib.osc_enable_joint_limit_avoidance(self._robot.handle, 1 if flag else 0))

    def reinitializeTasks(self, robots=None):
        """RobotController::reinitializeTasks for every robot or for those `robots` selects (a bool [N] array or robot indices)"""
        _reset(self._robot, -1, robots, capi.OSC_RESET_REINITIALIZE)

    def reinitializeTasksDevice(self, mask_ptr):
        _reset_device(self._robot, -1, mask_ptr, capi.OSC_RESET_REINITIALIZE)

    def resetRobots(self, robots=None):
        """Episode reset (no reference counterpart): every task of the selected robots goes back to the state it had right after
        construction at the robot's current state -- goals at the current pose, integrators, singularity-handler memory and
        POPC state reset, the internal OTG constructed anew.  Gains, spaces and every other setting stay."""
        _reset(self._robot, -1, robots, capi.OSC_RESET_CONSTRUCT)

    def resetRobotsDevice(self, mask_ptr):
        _reset_device(self._robot, -1, mask_ptr, capi.OSC_RESET_CONSTRUCT)

    def getJointTaskByName(self, name):
        for t in self._tasks:
            if t.getTaskName() == name:
                if t.task_type != capi.OSC_TASK_JOINT:
                    raise ValueError("Task %s is not a JointTask" % name)
                return t
        raise ValueError("Task %s not found" % name)

    def getMotionForceTaskByName(self, name):
        for t in self._tasks:
            if t.getTaskName() == name:
                if t.task_type != capi.OSC_TASK_MOTION_FORCE:
                    raise ValueError("Task %s is not a MotionForceTask" % name)
                return t
        raise ValueError("Task %s not found" % name)
