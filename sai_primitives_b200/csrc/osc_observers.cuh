// Read-only observers of the task models that the fused cycle kernel never materialises (it works with whitened factors):
//   TemplateTask::getTaskNullspace / getPreviousTasksNullspace / getTaskAndPreviousNullspace   src/tasks/TemplateTask.h:74,82,89
//     (JointTask.h:222-226, MotionForceTask.h:205-209; read by POPCBilateralTeleoperation.cpp:81-92)
//   MotionForceTask::getPositionError / getOrientationError                                    src/tasks/MotionForceTask.cpp:540-546
//   MotionForceTask::sigmaForce / sigmaPosition / sigmaMoment / sigmaOrientation               src/tasks/MotionForceTask.cpp:892-971
// One robot per thread, evaluated on request (osc_get_field) from the handle's current state: the null spaces are those an
// updateControllerTaskModels() at that state produces (RobotController.cpp:68-77), statement by statement like the general
// path (osc_singular.cuh) but without touching any task state.
#pragma once
#include "osc_kindyn.cuh"
#include "osc_singular.cuh"
#include "osc_tasks.cuh"

namespace osc {

enum ObserverKind : int {
	OBS_TASK_NULLSPACE = 0,
	OBS_PREVIOUS_NULLSPACE = 1,
	OBS_TASK_AND_PREVIOUS_NULLSPACE = 2,
	OBS_POSITION_ERROR = 3,
	OBS_ORIENTATION_ERROR = 4,
	OBS_SIGMA_FORCE = 5,
	OBS_SIGMA_POSITION = 6,
	OBS_SIGMA_MOMENT = 7,
	OBS_SIGMA_ORIENTATION = 8,
};

// N of hierarchy entry `task` given N_prec (model part of MotionForceTask::updateTaskModel + SingularityHandler::updateTaskModel
// :75-158, or JointTask::updateTaskModel :218-245)
template <int N>
static __device__ __noinline__ void task_nullspace_one(const OscProgram& P, const KinDyn<N>& kd, const double* Minv, const double* Nprec, int task,
													   double* Nmat) {
	using namespace sg;
	constexpr int n = N;
	const DevModel& mdl = P.model;
	for (int a = 0; a < N * N; a++) Nmat[a] = ((a / N) == (a % N)) ? 1.0 : 0.0;
	if (P.tasks[task].type == OSC_TASK_MOTION_FORCE) {
		const DevMft& t = P.mft[P.tasks[task].index];
		const osc_mft_params& p = t.p;
		const int r = t.rank;
		double x[3], Rc[9];
		frame_pose<N>(kd, t.body, t.ctrl_R, t.ctrl_t, x, Rc);
		double JT0[N][6];
		point_jacobian_t<N>(mdl, kd, t.body, x, JT0);
		double J0[6 * N], J[6 * N];
		for (int j = 0; j < N; j++) {
			double v[3] = {JT0[j][0], JT0[j][1], JT0[j][2]}, w[3] = {JT0[j][3], JT0[j][4], JT0[j][5]};
			if (!t.full) {
				double tv[3], tw[3];
				mat3_vec(t.Pt, v, tv);
				mat3_vec(t.Pr, w, tw);
				for (int k = 0; k < 3; k++) {
					v[k] = tv[k];
					w[k] = tw[k];
				}
			}
			for (int k = 0; k < 3; k++) {
				J0[k * N + j] = v[k];
				J0[(3 + k) * N + j] = w[k];
			}
		}
		mm(J0, 6, n, Nprec, n, J);
		constexpr int K = (N < 6) ? N : 6;
		double U[6 * K], sv[K], V[N * K];
		svd_rows6(J, n, U, sv, V);
		int n_ns = 0, n_s = 0;
		if (sv[0] < p.s_abs_tol) {
			n_s = r;
		} else if (r == 1) {
			n_ns = 1;
		} else {
			n_ns = r;
			for (int c = 1; c < r; c++)
				if (sv[c] / sv[0] < p.s_max) {
					n_ns = c;
					n_s = r - c;
					break;
				}
		}
		double Uns[6 * 6], Vs[N * 6], Jns[6 * N], Lns[36], Nns[N * N];
		for (int a = 0; a < 6; a++)
			for (int c = 0; c < n_ns; c++) Uns[a * n_ns + c] = U[a * K + c];
		for (int a = 0; a < N; a++)
			for (int c = 0; c < n_s; c++) Vs[a * n_s + c] = V[a * K + n_ns + c];
		for (int a = 0; a < N * N; a++) Nns[a] = ((a / N) == (a % N)) ? 1.0 : 0.0;
		if (n_ns > 0) {
			mm_at(Uns, 6, n_ns, J, n, Jns);
			op_space(Jns, n_ns, n, Minv, Lns, Nns);
		}
		if (n_s == 0 || !p.singularity_handling_enabled) {
			for (int a = 0; a < N * N; a++) Nmat[a] = Nns[a];
		} else if (n_ns == 0) {
			for (int a = 0; a < N * N; a++) Nmat[a] = Nprec[a];
		} else {
			double Njs[N * N], T1[6 * N], Jpost[6 * N], Ljs[36];
			mm_at(Vs, n, n_s, Nns, n, T1);
			mm(T1, n_s, n, Nprec, n, Jpost);
			op_space(Jpost, n_s, n, Minv, Ljs, Njs);
			mm(Njs, n, n, Nns, n, Nmat);
		}
	} else {
		const DevJt& jt = P.jt[P.tasks[task].index];
		const int k = jt.k;
		double S[N * N], Jp[N * N];
		for (int a = 0; a < k; a++)
			for (int j = 0; j < N; j++) S[a * N + j] = jt.S[a][j];
		mm(S, k, n, Nprec, n, Jp);
		double Ur[N * N], sr[N];
		int kr = 0;
		if (sqrt(fro2(Jp, k * n)) >= 1e-3) {
			left_svd_gram<N>(Jp, k, n, Ur, sr);
			if (sr[0] >= 1e-3) {
				kr = k;
				for (int c = k - 1; c > 0; c--) {
					if (sr[c] / sr[0] < 1e-3)
						kr--;
					else
						break;
				}
			}
		}
		if (kr > 0) {
			double Ub[N * N], Jr[N * N], Mp[N * N];
			for (int a = 0; a < k; a++)
				for (int c = 0; c < kr; c++) Ub[a * kr + c] = (kr == k) ? ((a == c) ? 1.0 : 0.0) : Ur[a * k + c];
			mm_at(Ub, k, kr, Jp, n, Jr);
			op_space(Jr, kr, n, Minv, Mp, Nmat);
		}
	}
}

// out: ncomp x n_robots (SoA)
template <int N>
__global__ void __launch_bounds__(64) osc_observer_kernel(const __grid_constant__ OscProgram P, int task, int kind, double* out) {
	using namespace sg;
	const int64_t NR = P.n_robots;
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= NR) return;
	if (kind <= OBS_TASK_AND_PREVIOUS_NULLSPACE) {
		double q[N];
		for (int j = 0; j < N; j++) q[j] = P.q[(int64_t)j * NR + i];
		KinDyn<N> kd;
		forward_kinematics<N>(P.model, q, kd);
		mass_matrix<N, false>(P.model, kd);
		double M[N * N], Minv[N * N];
		for (int a = 0; a < N; a++)
			for (int b = 0; b < N; b++) M[a * N + b] = kd.M[a][b];
		spd_inverse(M, N, Minv);
		double Nprec[N * N], Nmat[N * N], Nn[N * N];
		for (int a = 0; a < N * N; a++) Nprec[a] = ((a / N) == (a % N)) ? 1.0 : 0.0;
		for (int tk = 0; tk <= task; tk++) {
			task_nullspace_one<N>(P, kd, Minv, Nprec, tk, Nmat);
			if (tk == task) break;
			mm(Nmat, N, N, Nprec, N, Nn);
			for (int a = 0; a < N * N; a++) Nprec[a] = Nn[a];
		}
		const double* src = Nmat;
		if (kind == OBS_PREVIOUS_NULLSPACE) src = Nprec;
		if (kind == OBS_TASK_AND_PREVIOUS_NULLSPACE) {
			mm(Nmat, N, N, Nprec, N, Nn);
			src = Nn;
		}
		for (int a = 0; a < N * N; a++) out[(int64_t)a * NR + i] = src[a];
		return;
	}
	// motion-force task observers from the state the last computeTorques left (current pose, orientation error) and the goals
	const DevMft& t = P.mft[P.tasks[task].index];
	double R[9];
	for (int k = 0; k < 9; k++) R[k] = t.st[(int64_t)(MC_CUR_ORI + k) * NR + i];
	const int32_t mode = mft_space_mode(t, i);	// this robot's spaces, as the control law reads them
	double af[3], am[3], uf[3], um[3];
	mft_space_axes(t, NR, i, af, am);
	if (t.in_compliant) {
		mat3_vec(R, af, uf);
		mat3_vec(R, am, um);
	} else {
		for (int k = 0; k < 3; k++) {
			uf[k] = af[k];
			um[k] = am[k];
		}
	}
	double Sf[9], Sm[9], Sp[9], So[9];
	sigma_space((mode >> SP_FDIM_SHIFT) & 3, t.Pt, uf, Sf);
	sigma_space((mode >> SP_MDIM_SHIFT) & 3, t.Pr, um, Sm);
	sigma_complement(t.Pt, Sf, Sp);
	sigma_complement(t.Pr, Sm, So);
	if (kind == OBS_POSITION_ERROR || kind == OBS_ORIENTATION_ERROR) {
		double e[3], o[3];
		if (kind == OBS_POSITION_ERROR) {
			for (int k = 0; k < 3; k++) e[k] = t.st[(int64_t)(MC_GOAL_POS + k) * NR + i] - t.st[(int64_t)(MC_CUR_POS + k) * NR + i];
			mat3_vec(Sp, e, o);
		} else {
			for (int k = 0; k < 3; k++) e[k] = t.st[(int64_t)(MC_ORI_ERROR + k) * NR + i];
			mat3_vec(So, e, o);
		}
		for (int k = 0; k < 3; k++) out[(int64_t)k * NR + i] = o[k];
		return;
	}
	const double* S = kind == OBS_SIGMA_FORCE ? Sf : kind == OBS_SIGMA_POSITION ? Sp : kind == OBS_SIGMA_MOMENT ? Sm : So;
	for (int k = 0; k < 9; k++) out[(int64_t)k * NR + i] = S[k];
}

}  // namespace osc
