// Small per-robot service kernels around the fused cycle: task resets of selected robots from
// their current state, sensed-wrench frame change, the stand-alone kinematics/dynamics export
// used by the parity tests, and SoA component fills/copies.
#pragma once
#include "osc_kindyn.cuh"
#include "osc_otg_kernels.cuh"
#include "osc_tasks.cuh"

namespace osc {

#define ST(comp, c) st[(int64_t)((comp) + (c)) * NR + i]

// value fill of `ncomp` consecutive SoA components (vals in kernel parameter space)
struct FillVals {
	double v[16];
};
__global__ void fill_components_kernel(double* st, int64_t NR, int comp, int ncomp, FillVals vals) {
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= NR) return;
	for (int c = 0; c < ncomp; c++) ST(comp, c) = vals.v[c];
}
__global__ void copy_components_kernel(double* st, int64_t NR, int dst, int src, int ncomp) {
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= NR) return;
	for (int c = 0; c < ncomp; c++) ST(dst, c) = ST(src, c);
}
// Validation of caller values in device memory (osc_set_gains): *bad |= 1 if any of the n values is not finite, |= 2 if any is
// negative.  Grid-stride, one atomic per warp that found something.
__global__ void check_values_kernel(const double* v, int64_t n, int32_t* bad) {
	int32_t f = 0;
	for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
		const double x = v[k];
		if (!isfinite(x)) f |= 1;
		else if (x < 0.0) f |= 2;
	}
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) f |= __shfl_xor_sync(0xffffffffu, f, o);
	if (f && (threadIdx.x & 31) == 0) atomicOr(bad, f);
}
__global__ void fill_int_components_kernel(int32_t* ist, int64_t NR, int comp, int ncomp, int32_t value) {
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= NR) return;
	for (int c = 0; c < ncomp; c++) ist[(int64_t)(comp + c) * NR + i] = value;
}

// MotionForceTask::reInitializeTask (MotionForceTask.cpp:204-245) of robot i at its current pose (x, R).  construct also resets
// what only the constructor resets: the singularity handler / POPC initial state (SingularityHandler.cpp:53-63,
// POPCExplicitForceControl.cpp:10-21).
template <int N>
DEVI void mft_reset_robot(const DevMft& t, const DevModel& model, int64_t NR, int64_t i, const double x[3], const double R[9], bool construct) {
	double* st = t.st;
	for (int c = 0; c < MC_POPC; c++) ST(0, c) = 0.0;  // goals, sensed values, integrators, observers
	store3(st, NR, i, MC_GOAL_POS, x);
	store3(st, NR, i, MC_CUR_POS, x);
#pragma unroll
	for (int k = 0; k < 9; k++) {
		ST(MC_GOAL_ORI, k) = R[k];
		ST(MC_CUR_ORI, k) = R[k];
	}
	if (construct) {
		ST(MC_POPC, 0) = 0.0;
		ST(MC_POPC, 1) = 0.0;
		ST(MC_POPC, 2) = 1.0;  // Rc
		ST(MC_POPC, 3) = 0.0;
		for (int j = 0; j < OSC_MAX_DOF; j++) {
			const double mid = (j < N) ? 0.5 * (model.q_lower[j] + model.q_upper[j]) : 0.0;
			ST(MC_Q_PRIOR, j) = mid;
			ST(MC_DQ_PRIOR, j) = 0.0;
			ST(MC_TYPE2_DIR, j) = 1.0;
		}
		for (int c = 0; c < MI_COUNT; c++) t.ist[(int64_t)c * NR + i] = 0;
		t.ist[(int64_t)MI_POPC_COUNTER * NR + i] = 50;
	}
}

// JointTask::reInitializeTask (JointTask.cpp:91-107) of robot i; pos receives the task-space position (jt_task_position).  The
// constructor does nothing more (JointTask.cpp:45-89).
template <int N>
DEVI void jt_reset_robot(const DevJt& t, int64_t NR, int64_t i, const double (&q)[N], double pos[OSC_MAX_DOF]) {
	double* st = t.st;
	for (int c = 0; c < JC_COUNT; c++) ST(0, c) = 0.0;
	jt_task_position<N>(t, q, pos);
	for (int a = 0; a < t.k; a++) ST(JC_GOAL_POS, a) = pos[a];
}

// osc_reset_robots: the selected robots (mask == null: all; otherwise mask[i] != 0) get the tasks `task` (< 0: every task) reset
// at their current state, in hierarchy order, with the internal generator of a task that has it on (osc_otg_kernels.cuh).
// construct = 0: TemplateTask::reInitializeTask, generator re-initialised; construct = 1: the state right after the task's
// constructor, generator constructed as enabling it does.  Robots that are not selected are not written.
template <int N>
__global__ void reset_robots_kernel(const __grid_constant__ OscProgram P, const int32_t* mask, int task, int construct) {
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const int64_t NR = P.n_robots;
	if (i >= NR) return;
	if (mask && mask[i] == 0) return;
	double q[N];
#pragma unroll
	for (int j = 0; j < N; j++) q[j] = P.q[(int64_t)j * NR + i];
	// poses of the (at most two) motion-force tasks first, so that the kinematics are not live across the resets
	double x[2][3], R[2][9];
	{
		KinDyn<N> kd;
		forward_kinematics<N>(P.model, q, kd);
#pragma unroll
		for (int m = 0; m < 2; m++) {
			const DevMft& t = P.mft[m];
			if (t.st) frame_pose<N>(kd, t.body, t.ctrl_R, t.ctrl_t, x[m], R[m]);
		}
	}
	for (int k = 0; k < P.n_tasks; k++) {
		if (task >= 0 && k != task) continue;
		if (P.tasks[k].type == OSC_TASK_MOTION_FORCE) {
			const int m = P.tasks[k].index;
			const DevMft& t = P.mft[m];
			double xm[3], Rm[9];
#pragma unroll
			for (int c = 0; c < 3; c++) xm[c] = m ? x[1][c] : x[0][c];
#pragma unroll
			for (int c = 0; c < 9; c++) Rm[c] = m ? R[1][c] : R[0][c];
			mft_reset_robot<N>(t, P.model, NR, i, xm, Rm, construct != 0);
			if (t.otg.enabled) otg_cart_init(t, NR, i, xm, Rm, construct != 0);  // MotionForceTask.cpp:244
		} else {
			const DevJt& t = P.jt[P.tasks[k].index];
			double pos[OSC_MAX_DOF];
			jt_reset_robot<N>(t, NR, i, q, pos);
			if (t.otg.enabled) otg_joint_init(t, NR, i, pos, construct != 0);  // JointTask.cpp:106
		}
	}
}

// MotionForceTask::updateSensedForceAndMoment (MotionForceTask.cpp:805-828)
template <int N>
__global__ void sensed_wrench_kernel(const __grid_constant__ OscProgram P, int mft_index, const double* f_sensor,
									 const double* m_sensor) {
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const int64_t NR = P.n_robots;
	if (i >= NR) return;
	const DevMft& t = P.mft[mft_index];
	double* st = t.st;
	double q[N];
#pragma unroll
	for (int j = 0; j < N; j++) q[j] = P.q[(int64_t)j * NR + i];
	KinDyn<N> kd;
	forward_kinematics<N>(P.model, q, kd);
	double x[3], R[9];
	frame_pose<N>(kd, t.body, t.ctrl_R, t.ctrl_t, x, R);
	double fs[3], ms[3];
#pragma unroll
	for (int k = 0; k < 3; k++) {
		fs[k] = f_sensor[(int64_t)k * NR + i];
		ms[k] = m_sensor[(int64_t)k * NR + i];
	}
	store3(st, NR, i, MC_SENSED_F_SENSOR, fs);
	store3(st, NR, i, MC_SENSED_M_SENSOR, ms);
	double f[3], m[3], tmp[3], cr[3];
	mat3_vec(t.cs_R, fs, f);
	mat3_vec(t.cs_R, ms, tmp);
	cross3(t.cs_t, f, cr);
#pragma unroll
	for (int k = 0; k < 3; k++) m[k] = cr[k] + tmp[k];
	double fw[3], mw[3];
	mat3_vec(R, f, fw);
	mat3_vec(R, m, mw);
	store3(st, NR, i, MC_SENSED_F, fw);
	store3(st, NR, i, MC_SENSED_M, mw);
}

// Kinematics/dynamics stage on its own: M, J (6 x n, linear first), x, R, g.
struct EvalOut {
	double *M, *J, *x, *R, *g;
};
template <int N>
__global__ void eval_model_kernel(const __grid_constant__ OscProgram P, osc_link_frame frame, EvalOut out) {
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const int64_t NR = P.n_robots;
	if (i >= NR) return;
	double q[N];
#pragma unroll
	for (int j = 0; j < N; j++) q[j] = P.q[(int64_t)j * NR + i];
	KinDyn<N> kd;
	forward_kinematics<N>(P.model, q, kd);
	mass_matrix<N, true>(P.model, kd);
	double x[3], R[9];
	frame_pose<N>(kd, frame.body, frame.R, frame.t, x, R);
	double JT[N][6];
	point_jacobian_t<N>(P.model, kd, frame.body, x, JT);
	if (out.M)
#pragma unroll
		for (int r = 0; r < N; r++)
#pragma unroll
			for (int c = 0; c < N; c++) out.M[(int64_t)(r * N + c) * NR + i] = kd.M[r][c];
	if (out.J)
#pragma unroll
		for (int r = 0; r < 6; r++)
#pragma unroll
			for (int c = 0; c < N; c++) out.J[(int64_t)(r * N + c) * NR + i] = JT[c][r];
	if (out.x)
#pragma unroll
		for (int k = 0; k < 3; k++) out.x[(int64_t)k * NR + i] = x[k];
	if (out.R)
#pragma unroll
		for (int k = 0; k < 9; k++) out.R[(int64_t)k * NR + i] = R[k];
	if (out.g)
#pragma unroll
		for (int j = 0; j < N; j++) out.g[(int64_t)j * NR + i] = kd.g[j];
}

// ------------------------------------------------------------------------------------------------
// JointLimitAvoidanceTask + the blend of RobotController::computeControlTorques (SURVEY.md row f-2), one robot per
// thread, applied to the torques the cycle kernels left in P.tau:
//   limit status per joint            JointLimitAvoidanceTask::updateLimitStatus          JointLimitAvoidanceTask.cpp:174-243
//   N_constraints = I - M^-1 S^T (S M^-1 S^T)^-1 S   updateTaskModel with N_prec = I      :124-172, RobotController.cpp:71-72
//   avoidance torques per active joint computeTorques                                     :258-421
//   tau <- S^T t + N_constraints^T tau, saturation, gravity                               RobotController.cpp:96-116
// S selects the k joints inside a buffer zone.  Instead of compacting them (run-time indices), the k x k block
// (M^-1)_AA is embedded in an n x n matrix with the identity on the inactive joints; its inverse carries
// (S M^-1 S^T)^-1 on the active block.  Robots with no active joint (the common case) only pay the status test.
DEVI double jla_blend(double z, double z1, double z2, bool negative) {	// computeBlendingCoefficient :16-37
	if (negative) {
		if (z >= z1) return 0.0;
		if (z <= z2) return 1.0;
		return (z1 - z) / (z1 - z2);
	}
	if (z <= z1) return 0.0;
	if (z >= z2) return 1.0;
	return (z - z1) / (z2 - z1);
}

template <int N>
__global__ void __launch_bounds__(128) jla_kernel(const __grid_constant__ OscProgram P, DevJla jp) {
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const int64_t NR = P.n_robots;
	if (i >= NR) return;
	if (P.status[i] & OSC_STATUS_UNHANDLED) return;	 // NaN torques stay NaN
	const DevModel& m = P.model;
	enum { OFF = 0, POS_Z1, POS_Z2, VEL_Z1, VEL_Z2 };
	double q[N], dq[N], tau[N];
	int st[N];
	bool neg[N];
	double lv[N];
	int k = 0;
	const double fmax = 1.7976931348623157e308;
#pragma unroll
	for (int j = 0; j < N; j++) {
		q[j] = P.q[(int64_t)j * NR + i];
		dq[j] = P.dq[(int64_t)j * NR + i];
		tau[j] = P.tau[(int64_t)j * NR + i];
		const bool pos_valid = (m.q_upper[j] - m.q_lower[j]) > 2.0 * jp.position_z1_to_limit;	// verifyValidityPerJoint :95-118
		const bool vel_valid = m.dq_max[j] > 2.0 * jp.velocity_z1_to_limit;
		int s = OFF;
		bool ng = false;
		double v = 0.0;
		if (pos_valid && m.q_upper[j] != fmax) {
			if (q[j] > m.q_upper[j] - jp.position_z1_to_limit) {
				ng = false;
				v = m.q_upper[j];
				s = POS_Z1;
			}
			if (q[j] > m.q_upper[j] - jp.position_z2_to_limit) s = POS_Z2;
		}
		if (pos_valid && m.q_lower[j] != -fmax) {
			if (q[j] < m.q_lower[j] + jp.position_z1_to_limit) {
				ng = true;
				v = m.q_lower[j];
				s = POS_Z1;
			}
			if (q[j] < m.q_lower[j] + jp.position_z2_to_limit) s = POS_Z2;
		}
		if (vel_valid && (s == OFF || ng)) {
			if (dq[j] > m.dq_max[j] - jp.velocity_z1_to_limit) {
				ng = false;
				v = m.dq_max[j];
				s = VEL_Z1;
			}
			if (dq[j] > m.dq_max[j] - jp.velocity_z2_to_limit) s = VEL_Z2;
		}
		if (vel_valid && (s == OFF || !ng)) {
			if (dq[j] < -m.dq_max[j] + jp.velocity_z1_to_limit) {
				ng = true;
				v = -m.dq_max[j];
				s = VEL_Z1;
			}
			if (dq[j] < -m.dq_max[j] + jp.velocity_z2_to_limit) s = VEL_Z2;
		}
		st[j] = s;
		neg[j] = ng;
		lv[j] = v;
		k += (s != OFF) ? 1 : 0;
	}
	if (k == 0 && !P.gravity_comp) return;

	KinDyn<N> kd;
	forward_kinematics<N>(m, q, kd);
	if (P.gravity_comp)
		mass_matrix<N, true>(m, kd);
	else
		mass_matrix<N, false>(m, kd);
	if (k > 0) {
		// avoidance torque of every active joint (:279-412)
		double t[N];
		const double pz1 = jp.position_z1_to_limit, pz2 = jp.position_z2_to_limit, vz1 = jp.velocity_z1_to_limit, vz2 = jp.velocity_z2_to_limit;
#pragma unroll
		for (int j = 0; j < N; j++) {
			const double tl = m.effort[j], cap = tl * jp.max_torque_ratio_vel_limit;
			const double damp = -jp.kv * dq[j];
			double dc = damp;
			dc = dc > cap ? cap : dc;
			dc = dc < -cap ? -cap : dc;
			double out = 0.0;
			if (!neg[j]) {
				if (st[j] == POS_Z1) {
					const double a = jla_blend(q[j], lv[j] - pz1, lv[j] - pz2, false);
					out = (1.0 - a) * tau[j] + a * (tau[j] + damp);
				} else if (st[j] == POS_Z2) {
					const double a = jla_blend(q[j], lv[j] - pz2, lv[j], false);
					out = (1.0 - a) * (tau[j] + damp) + a * (-tl * jp.max_torque_ratio_pos_limit + damp);
				} else if (st[j] == VEL_Z1) {
					const double a = jla_blend(dq[j], lv[j] - vz1, lv[j] - vz2, false);
					out = (1.0 - a) * tau[j] + a * damp;
				} else if (st[j] == VEL_Z2) {
					const double a = jla_blend(dq[j], lv[j] - vz2, lv[j], false);
					out = (1.0 - a) * dc + a * (-a * cap);
				}
			} else {
				if (st[j] == POS_Z1) {
					const double a = jla_blend(q[j], lv[j] + pz1, lv[j] + pz2, true);
					double t1 = tau[j] + damp;
					t1 = t1 > cap ? cap : t1;
					t1 = t1 < -cap ? -cap : t1;
					out = a * tau[j] + (1.0 - a) * t1;	// sic (:344-345)
				} else if (st[j] == POS_Z2) {
					const double a = jla_blend(q[j], lv[j] + pz2, lv[j], true);
					out = (1.0 - a) * (tau[j] + damp) + a * (tl * jp.max_torque_ratio_pos_limit + damp);
				} else if (st[j] == VEL_Z1) {
					const double a = jla_blend(dq[j], lv[j] + vz1, lv[j] + vz2, true);
					out = (1.0 - a) * tau[j] + a * dc;
				} else if (st[j] == VEL_Z2) {
					const double a = jla_blend(dq[j], lv[j] + vz2, lv[j], true);
					out = (1.0 - a) * dc + a * cap;
				}
			}
			t[j] = out;
		}
		// N_constraints^T tau = tau - S^T (S M^-1 S^T)^-1 S M^-1 tau
		double L[N][N], invd[N];
#pragma unroll
		for (int r = 0; r < N; r++)
#pragma unroll
			for (int c = 0; c < N; c++) L[r][c] = kd.M[r][c];
		cholesky_lower<N>(L, invd);
		double y[N];
#pragma unroll
		for (int j = 0; j < N; j++) y[j] = tau[j];
		solve_spd<N>(L, invd, y);
		double B[N][N], invb[N];
#pragma unroll
		for (int a = 0; a < N; a++) {
			double col[N];
#pragma unroll
			for (int r = 0; r < N; r++) col[r] = (r == a) ? 1.0 : 0.0;
			if (st[a] != OFF) solve_spd<N>(L, invd, col);
#pragma unroll
			for (int r = 0; r < N; r++) B[r][a] = (st[a] != OFF && st[r] != OFF) ? col[r] : ((r == a) ? 1.0 : 0.0);
		}
		cholesky_lower<N>(B, invb);
		double z[N];
#pragma unroll
		for (int j = 0; j < N; j++) z[j] = (st[j] != OFF) ? y[j] : 0.0;
		solve_spd<N>(B, invb, z);
#pragma unroll
		for (int j = 0; j < N; j++)
			if (st[j] != OFF) tau[j] = t[j] + tau[j] - z[j];
		if (P.torque_saturation) {
#pragma unroll
			for (int j = 0; j < N; j++) {
				if (tau[j] > m.effort[j])
					tau[j] = m.effort[j];
				else if (tau[j] < -m.effort[j])
					tau[j] = -m.effort[j];
			}
		}
	}
	if (P.gravity_comp) {
#pragma unroll
		for (int j = 0; j < N; j++) tau[j] += kd.g[j];
	}
#pragma unroll
	for (int j = 0; j < N; j++) P.tau[(int64_t)j * NR + i] = tau[j];
}

// ------------------------------------------------------------------------------------------------
// Simulation side of the loop (SURVEY.md row f-1): ddq = M^-1 (tau - b - g), semi-implicit Euler, `substeps` steps of dt
// with the torque held.  q and dq are updated in place.
template <int N>
__global__ void __launch_bounds__(128) sim_integrate_kernel(const __grid_constant__ OscProgram P, double* qio, double* dqio, const double* tau_in,
															 double dt, int substeps) {
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const int64_t NR = P.n_robots;
	if (i >= NR) return;
	double q[N], dq[N], tau[N];
#pragma unroll
	for (int j = 0; j < N; j++) {
		q[j] = qio[(int64_t)j * NR + i];
		dq[j] = dqio[(int64_t)j * NR + i];
		tau[j] = tau_in[(int64_t)j * NR + i];
	}
	for (int s = 0; s < substeps; s++) {
		KinDyn<N> kd;
		forward_kinematics<N>(P.model, q, kd);
		mass_matrix<N, false>(P.model, kd);
		double rhs[N];
		rnea_bias<N>(P.model, kd, dq, rhs);
		double invd[N];
#pragma unroll
		for (int j = 0; j < N; j++) rhs[j] = tau[j] - rhs[j];
		cholesky_lower<N>(kd.M, invd);
		solve_spd<N>(kd.M, invd, rhs);
#pragma unroll
		for (int j = 0; j < N; j++) {
			dq[j] += rhs[j] * dt;
			q[j] += dq[j] * dt;
		}
	}
#pragma unroll
	for (int j = 0; j < N; j++) {
		qio[(int64_t)j * NR + i] = q[j];
		dqio[(int64_t)j * NR + i] = dq[j];
	}
}

// ------------------------------------------------------------------------------------------------
// Test probe for SURVEY.md row a12: K consecutive popc_step calls (the device code the fused kernels inline) on the
// POPC state of every robot of a motion-force task, with caller-supplied inputs (K x 3 each, row major, the same for
// all robots).  tests/test_popc_reference.py feeds it the sequence of tests/golden/popc_reference.npz, whose expected
// outputs were produced by the reference's own POPCExplicitForceControl.cpp.
__global__ void popc_probe_kernel(const __grid_constant__ OscProgram P, int mft_index, int K, const double* fd, const double* fs, const double* vcl,
								   const double* vr, double kv, double kff, double* out) {
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const int64_t NR = P.n_robots;
	if (i >= NR) return;
	const DevMft& t = P.mft[mft_index];
	uint32_t status = 0;
	for (int k = 0; k < K; k++) {
		const double a[3] = {fd[3 * k], fd[3 * k + 1], fd[3 * k + 2]}, b[3] = {fs[3 * k], fs[3 * k + 1], fs[3 * k + 2]};
		const double c[3] = {vcl[3 * k], vcl[3 * k + 1], vcl[3 * k + 2]}, d[3] = {vr[3 * k], vr[3 * k + 1], vr[3 * k + 2]};
		double o[3];
		popc_step(t, NR, i, a, b, c, d, kv, kff, o, status);
		if (i == 0) {
			out[3 * k] = o[0];
			out[3 * k + 1] = o[1];
			out[3 * k + 2] = o[2];
		}
	}
	if (status) P.status[i] |= status;
}

// ------------------------------------------------------------------------------------------------
// FP64 FMA issue-rate probe for the roofline denominator (SURVEY.md 8d asks for a measured FP64 figure next to the
// datasheet one): eight independent DFMA chains per thread in a rolled loop, every SM full.
__global__ void __launch_bounds__(1024) fp64_peak_kernel(double* out, double a, double b, int iters) {
	double x[8];
#pragma unroll
	for (int c = 0; c < 8; c++) x[c] = 1e-3 * threadIdx.x + c;
#pragma unroll 1
	for (int it = 0; it < iters; it++) {
#pragma unroll
		for (int r = 0; r < 16; r++)
#pragma unroll
			for (int c = 0; c < 8; c++) x[c] = fma(x[c], a, b);
	}
	double s = 0.0;
#pragma unroll
	for (int c = 0; c < 8; c++) s += x[c];
	if (s == 12345.678) out[0] = s;	 // never true: keeps the chains alive
}

#undef ST
}  // namespace osc
