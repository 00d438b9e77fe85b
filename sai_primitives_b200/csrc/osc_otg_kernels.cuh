// Batched internal OTG of the tasks (SURVEY.md row f-4): one robot per thread around the host/device core osc_otg.h.
//   JointTask::computeTorques        src/tasks/JointTask.cpp:313-319  (_otg->setGoalPositionAndVelocity; update; getNext*)
//   MotionForceTask::computeTorques  src/tasks/MotionForceTask.cpp:394-407
//   reInitializeTask / parametrize*  JointTask.cpp:106, MotionForceTask.cpp:244, :854, :886
// The update kernel runs before the cycle kernel of the same control cycle and leaves the desired state in the goal slots the
// control laws read.  A robot whose goal is reached and unchanged costs four SoA rows of loads; a trajectory is recalculated
// only when the goal (or the limits) changed.
#pragma once
#include "osc_dev_types.h"
#include "osc_math.cuh"
#include "osc_otg.h"

namespace osc {

static_assert(sizeof(otg::Section) == 20 * sizeof(double), "SoA layout of the generator state");
static_assert(offsetof(otg::JointsOtg<8>, flags) == OJ_CORE_DOUBLES * sizeof(double), "SoA layout of the joint generator");
static_assert(offsetof(otg::CartesianOtg, g) + offsetof(otg::JointsOtg<6>, flags) == OC_CORE_DOUBLES * sizeof(double), "SoA layout of the Cartesian generator");

template <class T>
DEVI void otg_load(T& o, const double* st, int64_t NR, int64_t i, int base, int count) {
	double* raw = reinterpret_cast<double*>(&o);
	for (int c = 0; c < count; c++) raw[c] = st[(int64_t)(base + c) * NR + i];
}
template <class T>
DEVI void otg_store(const T& o, double* st, int64_t NR, int64_t i, int base, int count) {
	const double* raw = reinterpret_cast<const double*>(&o);
	for (int c = 0; c < count; c++) st[(int64_t)(base + c) * NR + i] = raw[c];
}

static __device__ __noinline__ void otg_joint_step(const DevJt& t, int64_t NR, int64_t i) {
	const DevOtg& g = t.otg;
	const int k = t.k;
	double gp[OSC_MAX_DOF], gv[OSC_MAX_DOF], tp[OSC_MAX_DOF], tv[OSC_MAX_DOF];
	for (int a = 0; a < k; a++) {
		gp[a] = g.st[(int64_t)(OJ_USER_POS + a) * NR + i];
		gv[a] = g.st[(int64_t)(OJ_USER_VEL + a) * NR + i];
		tp[a] = g.st[(int64_t)(OJ_CORE + a) * NR + i];		  // JointsOtg::target_pos
		tv[a] = g.st[(int64_t)(OJ_CORE + 8 + a) * NR + i];  // JointsOtg::target_vel
	}
	int flags = g.flags[i];
	if ((flags & otg::OTG_GOAL_REACHED) && otg::is_approx(gp, tp, k, 1e-12) && otg::is_approx(gv, tv, k, 1e-12)) return;
	otg::JointsOtg<8> o;
	otg_load(o, g.st, NR, i, OJ_CORE, OJ_CORE_DOUBLES);
	o.flags = flags;
	o.set_goal(k, gp, gv);
	otg::Calculator<8> calc;
	o.update(k, t.dt, g.vmax, g.amax, &calc);
	otg_store(o, g.st, NR, i, OJ_CORE, OJ_CORE_DOUBLES);
	g.flags[i] = o.flags;
	for (int a = 0; a < k; a++) {  // _desired_* = _otg->getNext*()
		t.st[(int64_t)(JC_GOAL_POS + a) * NR + i] = o.out_pos[a];
		t.st[(int64_t)(JC_GOAL_VEL + a) * NR + i] = o.out_vel[a];
		t.st[(int64_t)(JC_GOAL_ACC + a) * NR + i] = o.out_acc[a];
	}
}

static __device__ __noinline__ void otg_cart_write_desired(const DevMft& t, const otg::CartesianOtg& o, int64_t NR, int64_t i) {
	double pos[3], R[9], v[3], w[3], a[3], al[3];
	o.desired(pos, R, v, w, a, al);
	for (int c = 0; c < 3; c++) {
		t.st[(int64_t)(MC_GOAL_POS + c) * NR + i] = pos[c];
		t.st[(int64_t)(MC_GOAL_LINVEL + c) * NR + i] = v[c];
		t.st[(int64_t)(MC_GOAL_ANGVEL + c) * NR + i] = w[c];
		t.st[(int64_t)(MC_GOAL_LINACC + c) * NR + i] = a[c];
		t.st[(int64_t)(MC_GOAL_ANGACC + c) * NR + i] = al[c];
	}
	for (int c = 0; c < 9; c++) t.st[(int64_t)(MC_GOAL_ORI + c) * NR + i] = R[c];
}

static __device__ __noinline__ void otg_cart_step(const DevMft& t, int64_t NR, int64_t i) {
	const DevOtg& g = t.otg;
	double user[24];
	for (int c = 0; c < 18; c++) user[c] = g.st[(int64_t)(OC_USER + c) * NR + i];	// goal position, orientation, linear and angular velocity
	int flags = g.flags[i];
	otg::CartesianOtg o;
	if (flags & otg::OTG_GOAL_REACHED) {
		// unchanged goal: compare against the registered targets only (21 + 6 rows)
		double tgt[27];
		for (int c = 0; c < 21; c++) tgt[c] = g.st[(int64_t)(OC_CORE + c) * NR + i];		 // ref, goal_ori, goal_w
		for (int c = 0; c < 3; c++) {
			tgt[21 + c] = g.st[(int64_t)(OC_CORE + 21 + c) * NR + i];		// target_pos[0..2]
			tgt[24 + c] = g.st[(int64_t)(OC_CORE + 21 + 6 + c) * NR + i];	// target_vel[0..2]
		}
		if (otg::is_approx(user, tgt + 21, 3, 1e-3) && otg::is_approx(user + 12, tgt + 24, 3, 1e-3) && otg::is_approx(tgt + 9, user + 3, 9, 1e-3) &&
			otg::is_approx(tgt + 18, user + 15, 3, 1e-3))
			return;
	}
	otg_load(o, g.st, NR, i, OC_CORE, OC_CORE_DOUBLES);
	o.g.flags = flags;
	o.set_goal_linear(user, user + 12);
	o.set_goal_angular(user + 3, user + 15);
	otg::Calculator<6> calc;
	o.update(t.dt, g.vmax, g.amax, &calc);
	otg_store(o, g.st, NR, i, OC_CORE, OC_CORE_DOUBLES);
	g.flags[i] = o.g.flags;
	otg_cart_write_desired(t, o, NR, i);
}

// Reset of robot i's generator by parametrizeForceMotionSpaces (reInitializeLinear, angular = false) or
// parametrizeMomentRotMotionSpaces (reInitializeAngular) with the generator on: the user's goals of that part become the current
// pose at rest, the generator restarts from there, and the desired state goes into the goal slots.
static __device__ __noinline__ void otg_cart_reinit_part(const DevMft& t, int64_t NR, int64_t i, bool angular) {
	const DevOtg& g = t.otg;
	double x[3], R[9];
	for (int c = 0; c < 3; c++) x[c] = t.st[(int64_t)(MC_CUR_POS + c) * NR + i];
	for (int c = 0; c < 9; c++) R[c] = t.st[(int64_t)(MC_CUR_ORI + c) * NR + i];
	otg::CartesianOtg o;
	otg_load(o, g.st, NR, i, OC_CORE, OC_CORE_DOUBLES);
	o.g.flags = g.flags[i];
	if (!angular) {
		for (int c = 0; c < 3; c++) {
			g.st[(int64_t)(OC_USER + MC_GOAL_POS + c) * NR + i] = x[c];
			g.st[(int64_t)(OC_USER + MC_GOAL_LINVEL + c) * NR + i] = 0.0;
			g.st[(int64_t)(OC_USER + MC_GOAL_LINACC + c) * NR + i] = 0.0;
		}
		o.reinitialize_linear(x);
	} else {
		for (int c = 0; c < 9; c++) g.st[(int64_t)(OC_USER + MC_GOAL_ORI + c) * NR + i] = R[c];
		for (int c = 0; c < 3; c++) {
			g.st[(int64_t)(OC_USER + MC_GOAL_ANGVEL + c) * NR + i] = 0.0;
			g.st[(int64_t)(OC_USER + MC_GOAL_ANGACC + c) * NR + i] = 0.0;
		}
		o.reinitialize_angular(R);
	}
	otg_store(o, g.st, NR, i, OC_CORE, OC_CORE_DOUBLES);
	g.flags[i] = o.g.flags;
	otg_cart_write_desired(t, o, NR, i);
}

// one launch per control cycle when any task has its generator on
__global__ void __launch_bounds__(64) otg_update_kernel(const __grid_constant__ OscProgram P) {
	const int64_t NR = P.n_robots;
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= NR) return;
	for (int task = 0; task < P.n_tasks; task++) {
		if (P.tasks[task].type == OSC_TASK_MOTION_FORCE) {
			const DevMft& t = P.mft[P.tasks[task].index];
			if (t.otg.enabled) otg_cart_step(t, NR, i);
		} else {
			const DevJt& t = P.jt[P.tasks[task].index];
			if (t.otg.enabled) otg_joint_step(t, NR, i);
		}
	}
}

// Task-space position S q of a JointTask (k entries): the goal its reset sets and the position its generator starts from.
template <int N>
DEVI void jt_task_position(const DevJt& t, const double (&q)[N], double pos[OSC_MAX_DOF]) {
	for (int a = 0; a < t.k; a++) {
		double s = 0.0;
#pragma unroll
		for (int j = 0; j < N; j++) s += t.S[a][j] * q[j];
		pos[a] = s;
	}
}

// (Re)initialisation of robot i's joint generator at the task-space position pos (k entries), then the desired state into the
// task's goal slots.  fresh: constructed as enabling it does (JointTask.cpp:372-374), the user's goals become what the task's
// goal slots hold; otherwise _otg->reInitialize of JointTask::reInitializeTask (JointTask.cpp:106): goal := current position,
// zero velocity and acceleration goals.
static __device__ __noinline__ void otg_joint_init(const DevJt& t, int64_t NR, int64_t i, const double* pos, bool fresh) {
	const DevOtg& g = t.otg;
	otg::JointsOtg<8> o;
	if (fresh) {
		for (int c = 0; c < OJ_CORE_DOUBLES; c++) reinterpret_cast<double*>(&o)[c] = 0.0;
		o.flags = 0;
		for (int a = 0; a < OSC_MAX_DOF; a++) {
			g.st[(int64_t)(OJ_USER_POS + a) * NR + i] = t.st[(int64_t)(JC_GOAL_POS + a) * NR + i];
			g.st[(int64_t)(OJ_USER_VEL + a) * NR + i] = t.st[(int64_t)(JC_GOAL_VEL + a) * NR + i];
			g.st[(int64_t)(OJ_USER_ACC + a) * NR + i] = t.st[(int64_t)(JC_GOAL_ACC + a) * NR + i];
		}
	} else {
		otg_load(o, g.st, NR, i, OJ_CORE, OJ_CORE_DOUBLES);
		o.flags = g.flags[i];
		for (int a = 0; a < OSC_MAX_DOF; a++) {
			g.st[(int64_t)(OJ_USER_POS + a) * NR + i] = a < t.k ? pos[a] : 0.0;
			g.st[(int64_t)(OJ_USER_VEL + a) * NR + i] = 0.0;
			g.st[(int64_t)(OJ_USER_ACC + a) * NR + i] = 0.0;
		}
	}
	o.reinitialize(t.k, pos);
	otg_store(o, g.st, NR, i, OJ_CORE, OJ_CORE_DOUBLES);
	g.flags[i] = o.flags;
	for (int a = 0; a < t.k; a++) {
		t.st[(int64_t)(JC_GOAL_POS + a) * NR + i] = o.out_pos[a];
		t.st[(int64_t)(JC_GOAL_VEL + a) * NR + i] = 0.0;
		t.st[(int64_t)(JC_GOAL_ACC + a) * NR + i] = 0.0;
	}
}

// The same for the Cartesian generator at the current pose (x, R): fresh = constructed (MotionForceTask.cpp:514-516) with the
// user's goals := the task's goal slots; otherwise _otg->reInitialize of MotionForceTask::reInitializeTask (:244).
static __device__ __noinline__ void otg_cart_init(const DevMft& t, int64_t NR, int64_t i, const double x[3], const double R[9], bool fresh) {
	const DevOtg& g = t.otg;
	otg::CartesianOtg o;
	if (fresh) {
		for (int c = 0; c < 24; c++) g.st[(int64_t)(OC_USER + c) * NR + i] = t.st[(int64_t)(MC_GOAL_POS + c) * NR + i];
		o.construct(x, R);
	} else {
		otg_load(o, g.st, NR, i, OC_CORE, OC_CORE_DOUBLES);
		o.g.flags = g.flags[i];
		for (int c = 0; c < 24; c++) g.st[(int64_t)(OC_USER + c) * NR + i] = 0.0;
		for (int c = 0; c < 3; c++) g.st[(int64_t)(OC_USER + MC_GOAL_POS + c) * NR + i] = x[c];
		for (int c = 0; c < 9; c++) g.st[(int64_t)(OC_USER + MC_GOAL_ORI + c) * NR + i] = R[c];
		o.reinitialize(x, R);
	}
	otg_store(o, g.st, NR, i, OC_CORE, OC_CORE_DOUBLES);
	g.flags[i] = o.g.flags;
	otg_cart_write_desired(t, o, NR, i);
}

// Generator calls of the host layer other than resets (those are reset_robots_kernel, osc_aux_kernels.cuh):
// mode 0: enabled -- constructed at the current position (and orientation), the user's goals are the task's goal slots;
// mode 1: parametrizeForceMotionSpaces reset -> reInitializeLinear; mode 2: parametrizeMomentRotMotionSpaces reset -> reInitializeAngular;
// mode 3: new limits.
template <int N>
__global__ void otg_init_kernel(const __grid_constant__ OscProgram P, int task, int mode) {
	const int64_t NR = P.n_robots;
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= NR) return;
	if (P.tasks[task].type == OSC_TASK_JOINT) {
		const DevJt& t = P.jt[P.tasks[task].index];
		const DevOtg& g = t.otg;
		if (mode == 3) {  // OTG_joints::setMaxVelocity / setMaxAcceleration / disableJerkLimits (:89-92): the acceleration state is dropped
			for (int a = 0; a < OSC_MAX_DOF; a++) g.st[(int64_t)(OJ_CORE + 32 + a) * NR + i] = 0.0;  // JointsOtg::in_acc
			g.flags[i] |= otg::OTG_DIRTY;
			return;
		}
		double q[N], pos[OSC_MAX_DOF];
		for (int j = 0; j < N; j++) q[j] = P.q[(int64_t)j * NR + i];
		jt_task_position<N>(t, q, pos);
		otg_joint_init(t, NR, i, pos, true);
		return;
	}
	const DevMft& t = P.mft[P.tasks[task].index];
	const DevOtg& g = t.otg;
	if (mode == 3) {  // new limits only (OTG_6dof_cartesian::setMax*): the next update recalculates
		g.flags[i] |= otg::OTG_DIRTY;
		return;
	}
	if (mode == 1 || mode == 2) {
		otg_cart_reinit_part(t, NR, i, mode == 2);
		return;
	}
	double x[3], R[9];
	for (int c = 0; c < 3; c++) x[c] = t.st[(int64_t)(MC_CUR_POS + c) * NR + i];
	for (int c = 0; c < 9; c++) R[c] = t.st[(int64_t)(MC_CUR_ORI + c) * NR + i];
	otg_cart_init(t, NR, i, x, R, true);
}

// generator switched off: the user's goals go back into the slots the control laws read
__global__ void otg_disable_kernel(const __grid_constant__ OscProgram P, int task) {
	const int64_t NR = P.n_robots;
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= NR) return;
	if (P.tasks[task].type == OSC_TASK_JOINT) {
		const DevJt& t = P.jt[P.tasks[task].index];
		for (int a = 0; a < OSC_MAX_DOF; a++) {
			t.st[(int64_t)(JC_GOAL_POS + a) * NR + i] = t.otg.st[(int64_t)(OJ_USER_POS + a) * NR + i];
			t.st[(int64_t)(JC_GOAL_VEL + a) * NR + i] = t.otg.st[(int64_t)(OJ_USER_VEL + a) * NR + i];
			t.st[(int64_t)(JC_GOAL_ACC + a) * NR + i] = t.otg.st[(int64_t)(OJ_USER_ACC + a) * NR + i];
		}
	} else {
		const DevMft& t = P.mft[P.tasks[task].index];
		for (int c = 0; c < 24; c++) t.st[(int64_t)(MC_GOAL_POS + c) * NR + i] = t.otg.st[(int64_t)(OC_USER + c) * NR + i];
	}
}

}  // namespace osc
