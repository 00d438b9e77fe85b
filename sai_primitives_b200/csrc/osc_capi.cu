// C ABI of the batched operational-space controller (include/sai_b200_osc.h).
// Thin host layer: owns the device buffers of one handle, validates arguments the way the
// reference does (std::invalid_argument -> OSC_ERR_INVALID_ARGUMENT) and launches the kernels.
// There is no CPU fallback anywhere in this file.
#include <cuda_runtime.h>

#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "osc_dev_types.h"
#include "osc_launch.h"

namespace {

thread_local std::string g_create_error;

struct TaskInfo {
	int type;	 // osc_task_type
	int index;	 // into prog.mft / prog.jt
	double dt;
	double compliant_R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};  // MotionForceTask: compliant frame in the link frame
	double compliant_t[3] = {0, 0, 0};
	osc_link_frame link{};
};

}  // namespace

struct osc_handle {
	int device = 0;
	int64_t NR = 0;
	osc_model_desc model;
	OscProgram prog;
	cudaStream_t own_stream = nullptr, stream = nullptr;
	bool finalized = false;
	bool models_armed = false;
	bool jla_enabled = false;  // RobotController::enableJointLimitAvoidance
	int sig_R = 0;
	bool sig_jt = false;
	std::vector<TaskInfo> tasks;
	int n_mft = 0, n_jt = 0;
	double *d_q = nullptr, *d_dq = nullptr, *d_tau = nullptr;
	uint32_t* d_status = nullptr;
	double *d_fs = nullptr, *d_ms = nullptr;  // staging for sensed wrench (3 x N each)
	int32_t *d_sing_list = nullptr, *d_sing_count = nullptr;
	// cycle pipelining (osc_pipeline.cuh): per-block cycle numbers, general-path completion word, mapped host word
	uint32_t *d_block_epoch = nullptr, *d_general_done = nullptr;
	unsigned long long* d_block_times = nullptr;  // osc_debug_block_times
	int otg_tasks = 0;			  // tasks whose internal OTG is on
	double* d_sim = nullptr;	  // staging of osc_sim_integrate with host buffers (q, dq, tau)
	double* d_scratch = nullptr;  // output of the on-request observers (osc_observers.cuh)
	size_t scratch_doubles = 0;
	int32_t* h_seen = nullptr;	// mapped pinned: hand-over count of the last completed cycle
	int32_t* d_check = nullptr;	// result word of the device-input validation of osc_set_gains and of the per-robot space calls
	// staging of the per-robot space calls with host buffers: axes (3 x N), dims or flags (N) and was_reset / closed_loop (N)
	double* d_space_axes = nullptr;
	int32_t* d_space_ints = nullptr;
	int32_t* d_reset_mask = nullptr;  // staging of osc_reset_robots with a host mask (N)
	int clean_cycles = 0;
	int blend_split = -1;  // split blending path: -1 not decided, 0 off (SAI_B200_BLEND_SPLIT=0 or no memory), 1 allocate when needed, 2 allocated
	int64_t blend_split_min = 0;  // hand-over count (host hint) from which the split path is used
	std::vector<void*> allocations;
	std::string err;
	int64_t launches = 0;
	bool cuda_failed = false;
};

namespace {

int fail(osc_handle* h, int code, const std::string& msg) {
	if (h)
		h->err = msg;
	else
		g_create_error = msg;
	return code;
}

#define CUDA_TRY(h, expr)                                                                         \
	do {                                                                                          \
		cudaError_t e_ = (expr);                                                                  \
		if (e_ != cudaSuccess) {                                                                  \
			(h)->cuda_failed = true;                                                              \
			return fail((h), OSC_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));  \
		}                                                                                         \
	} while (0)

#define ENTER(h)                                                                     \
	do {                                                                             \
		if (!(h)) return fail(nullptr, OSC_ERR_INVALID_ARGUMENT, "null handle");     \
		if ((h)->cuda_failed) return OSC_ERR_CUDA; /* sticky, message kept */         \
		cudaError_t e_ = cudaSetDevice((h)->device);                                 \
		if (e_ != cudaSuccess) return fail((h), OSC_ERR_CUDA, cudaGetErrorString(e_)); \
	} while (0)

template <typename T>
int dev_alloc(osc_handle* h, T** out, size_t count, bool zero) {
	void* p = nullptr;
	CUDA_TRY(h, cudaMalloc(&p, count * sizeof(T)));
	h->allocations.push_back(p);
	if (zero) CUDA_TRY(h, cudaMemsetAsync(p, 0, count * sizeof(T), h->stream));
	*out = (T*)p;
	return OSC_OK;
}

void mat3_mul_h(const double* a, const double* b, double* c) {
	for (int i = 0; i < 3; i++)
		for (int j = 0; j < 3; j++) c[3 * i + j] = a[3 * i] * b[j] + a[3 * i + 1] * b[3 + j] + a[3 * i + 2] * b[6 + j];
}
void mat3_vec_h(const double* a, const double* v, double* o) {
	for (int i = 0; i < 3; i++) o[i] = a[3 * i] * v[0] + a[3 * i + 1] * v[1] + a[3 * i + 2] * v[2];
}
void mat3t_h(const double* a, double* t) {
	for (int i = 0; i < 3; i++)
		for (int j = 0; j < 3; j++) t[3 * i + j] = a[3 * j + i];
}

// Symmetric 3x3 eigen-decomposition by cyclic Jacobi (host, setup only). Eigenvalues descending,
// eigenvectors in the columns of V.
void eig_sym3(const double A_in[9], double w[3], double V[9]) {
	double A[9];
	std::memcpy(A, A_in, sizeof(A));
	const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
	std::memcpy(V, I, sizeof(I));
	for (int sweep = 0; sweep < 60; sweep++) {
		const double off = A[1] * A[1] + A[2] * A[2] + A[5] * A[5];
		if (off < 1e-300) break;
		for (int p = 0; p < 2; p++)
			for (int q = p + 1; q < 3; q++) {
				const double apq = A[3 * p + q];
				if (std::fabs(apq) < 1e-300) continue;
				const double theta = (A[3 * q + q] - A[3 * p + p]) / (2.0 * apq);
				const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
				const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
				for (int k = 0; k < 3; k++) {  // A <- A J
					const double akp = A[3 * k + p], akq = A[3 * k + q];
					A[3 * k + p] = c * akp - s * akq;
					A[3 * k + q] = s * akp + c * akq;
				}
				for (int k = 0; k < 3; k++) {  // A <- J^T A
					const double apk = A[3 * p + k], aqk = A[3 * q + k];
					A[3 * p + k] = c * apk - s * aqk;
					A[3 * q + k] = s * apk + c * aqk;
				}
				for (int k = 0; k < 3; k++) {
					const double vkp = V[3 * k + p], vkq = V[3 * k + q];
					V[3 * k + p] = c * vkp - s * vkq;
					V[3 * k + q] = s * vkp + c * vkq;
				}
			}
	}
	w[0] = A[0];
	w[1] = A[4];
	w[2] = A[8];
	for (int a = 0; a < 2; a++)	 // sort descending
		for (int b = a + 1; b < 3; b++)
			if (w[b] > w[a]) {
				std::swap(w[a], w[b]);
				for (int k = 0; k < 3; k++) std::swap(V[3 * k + a], V[3 * k + b]);
			}
}

// SaiModel::matrixRangeBasis for a 3 x k matrix of direction vectors (tolerance 1e-3, SURVEY Appendix B):
// returns the rank (0 = zero range) and an orthonormal basis in the first `rank` columns of U
// (identity when rank == 3).
int range_basis_3(const double dirs[3][3], int k, double U[9]) {
	const double tol = 1e-3;
	double G[9] = {0};	// D D^T, D = 3 x k
	double fro = 0;
	for (int c = 0; c < k; c++)
		for (int i = 0; i < 3; i++) {
			fro += dirs[c][i] * dirs[c][i];
			for (int j = 0; j < 3; j++) G[3 * i + j] += dirs[c][i] * dirs[c][j];
		}
	std::memset(U, 0, 9 * sizeof(double));
	if (k == 0 || std::sqrt(fro) < tol) return 0;
	double w[3], V[9];
	eig_sym3(G, w, V);
	const double s0 = std::sqrt(std::max(w[0], 0.0));
	if (s0 < tol) return 0;
	const int max_range = k < 3 ? k : 3;
	int rank = max_range;
	for (int i = max_range - 1; i > 0; i--) {
		const double si = std::sqrt(std::max(w[i], 0.0));
		if (si / s0 < tol)
			rank--;
		else
			break;
	}
	if (rank == 3) {
		U[0] = U[4] = U[8] = 1.0;
	} else {
		for (int c = 0; c < rank; c++)
			for (int i = 0; i < 3; i++) U[3 * i + c] = V[3 * i + c];
	}
	return rank;
}

int rank_of(const double* S, int k, int n) {
	std::vector<double> A(S, S + (size_t)k * n);
	int rank = 0;
	std::vector<bool> used(k, false);
	for (int c = 0; c < n && rank < k; c++) {
		int piv = -1;
		double best = 1e-12;
		for (int r = 0; r < k; r++)
			if (!used[r] && std::fabs(A[(size_t)r * n + c]) > best) {
				best = std::fabs(A[(size_t)r * n + c]);
				piv = r;
			}
		if (piv < 0) continue;
		used[piv] = true;
		rank++;
		for (int r = 0; r < k; r++) {
			if (r == piv) continue;
			const double f = A[(size_t)r * n + c] / A[(size_t)piv * n + c];
			for (int cc = c; cc < n; cc++) A[(size_t)r * n + cc] -= f * A[(size_t)piv * n + cc];
		}
	}
	return rank;
}

void build_dev_model(const osc_model_desc& m, DevModel& d) {
	std::memset(&d, 0, sizeof(d));
	d.n = m.n;
	for (int i = 0; i < m.n; i++) {
		d.jtype[i] = m.jtype[i];
		std::memcpy(d.axis[i], m.axis[i], sizeof(double) * 3);
		if (i == 0) {  // fold SaiModel::TRobotBase into the first joint: everything downstream is in world axes
			mat3_mul_h(m.R_world_base, m.R_fix[0], d.R_fix[0]);
			double t[3];
			mat3_vec_h(m.R_world_base, m.t_fix[0], t);
			for (int k = 0; k < 3; k++) d.t_fix[0][k] = m.t_world_base[k] + t[k];
		} else {
			std::memcpy(d.R_fix[i], m.R_fix[i], sizeof(double) * 9);
			std::memcpy(d.t_fix[i], m.t_fix[i], sizeof(double) * 3);
		}
		d.mass[i] = m.mass[i];
		std::memcpy(d.com[i], m.com[i], sizeof(double) * 3);
		const double* I = m.inertia[i];
		d.inertia[i][0] = I[0];
		d.inertia[i][1] = 0.5 * (I[1] + I[3]);
		d.inertia[i][2] = 0.5 * (I[2] + I[6]);
		d.inertia[i][3] = I[4];
		d.inertia[i][4] = 0.5 * (I[5] + I[7]);
		d.inertia[i][5] = I[8];
		d.q_lower[i] = m.q_lower[i];
		d.q_upper[i] = m.q_upper[i];
		d.effort[i] = m.effort[i];
		d.dq_max[i] = m.dq_max[i];
	}
	std::memcpy(d.gravity, m.gravity_world, sizeof(double) * 3);
}

int check_task(osc_handle* h, int task_id, int type) {
	if (task_id < 0 || task_id >= (int)h->tasks.size()) return fail(h, OSC_ERR_INVALID_ARGUMENT, "task id out of range");
	if (type != 0 && h->tasks[task_id].type != type)
		return fail(h, OSC_ERR_INVALID_ARGUMENT, type == OSC_TASK_JOINT ? "task is not a JointTask" : "task is not a MotionForceTask");
	return OSC_OK;
}

bool is_finite(double v) { return std::isfinite(v); }

struct FieldInfo {
	int type;
	int comp;
	int ncomp;
	bool writable;
	bool goal = false;		  // a goal field: lives in the generator's block while the task's internal OTG is on
	int observer = -1;		  // >= 0: osc::ObserverKind evaluated on request (osc_observers.cuh), comp unused
	bool needs_observers = false;  // refreshed by the cycle kernels only while osc_enable_observers is on
};

bool field_info(const osc_handle* h, int task_id, int field, FieldInfo& fi) {
	if (task_id < 0 || task_id >= (int)h->tasks.size()) return false;
	const TaskInfo& t = h->tasks[task_id];
	const int n = h->model.n;
	switch (field) {
		case OSC_TASK_NULLSPACE: fi = {t.type, 0, n * n, false, false, 0}; return true;
		case OSC_TASK_PREVIOUS_NULLSPACE: fi = {t.type, 0, n * n, false, false, 1}; return true;
		case OSC_TASK_AND_PREVIOUS_NULLSPACE: fi = {t.type, 0, n * n, false, false, 2}; return true;
		default: break;
	}
	if (t.type == OSC_TASK_MOTION_FORCE) {
		switch (field) {
			case OSC_MFT_DESIRED_POSITION: fi = {t.type, MC_GOAL_POS, 3, false}; return true;
			case OSC_MFT_DESIRED_ORIENTATION: fi = {t.type, MC_GOAL_ORI, 9, false}; return true;
			case OSC_MFT_DESIRED_LINEAR_VELOCITY: fi = {t.type, MC_GOAL_LINVEL, 3, false}; return true;
			case OSC_MFT_DESIRED_ANGULAR_VELOCITY: fi = {t.type, MC_GOAL_ANGVEL, 3, false}; return true;
			case OSC_MFT_DESIRED_LINEAR_ACCELERATION: fi = {t.type, MC_GOAL_LINACC, 3, false}; return true;
			case OSC_MFT_DESIRED_ANGULAR_ACCELERATION: fi = {t.type, MC_GOAL_ANGACC, 3, false}; return true;
			case OSC_MFT_POSITION_ERROR: fi = {t.type, 0, 3, false, false, 3}; return true;
			case OSC_MFT_ORIENTATION_ERROR: fi = {t.type, 0, 3, false, false, 4, true}; return true;
			case OSC_MFT_SIGMA_FORCE: fi = {t.type, 0, 9, false, false, 5}; return true;
			case OSC_MFT_SIGMA_POSITION: fi = {t.type, 0, 9, false, false, 6}; return true;
			case OSC_MFT_SIGMA_MOMENT: fi = {t.type, 0, 9, false, false, 7}; return true;
			case OSC_MFT_SIGMA_ORIENTATION: fi = {t.type, 0, 9, false, false, 8}; return true;
			case OSC_MFT_GOAL_POSITION: fi = {t.type, MC_GOAL_POS, 3, true, true}; return true;
			case OSC_MFT_GOAL_ORIENTATION: fi = {t.type, MC_GOAL_ORI, 9, true, true}; return true;
			case OSC_MFT_GOAL_LINEAR_VELOCITY: fi = {t.type, MC_GOAL_LINVEL, 3, true, true}; return true;
			case OSC_MFT_GOAL_ANGULAR_VELOCITY: fi = {t.type, MC_GOAL_ANGVEL, 3, true, true}; return true;
			case OSC_MFT_GOAL_LINEAR_ACCELERATION: fi = {t.type, MC_GOAL_LINACC, 3, true, true}; return true;
			case OSC_MFT_GOAL_ANGULAR_ACCELERATION: fi = {t.type, MC_GOAL_ANGACC, 3, true, true}; return true;
			case OSC_MFT_GOAL_FORCE: fi = {t.type, MC_GOAL_FORCE, 3, true}; return true;
			case OSC_MFT_GOAL_MOMENT: fi = {t.type, MC_GOAL_MOMENT, 3, true}; return true;
			case OSC_MFT_CURRENT_POSITION: fi = {t.type, MC_CUR_POS, 3, false}; return true;
			case OSC_MFT_CURRENT_ORIENTATION: fi = {t.type, MC_CUR_ORI, 9, false}; return true;
			case OSC_MFT_CURRENT_LINEAR_VELOCITY: fi = {t.type, MC_CUR_LINVEL, 3, false, false, -1, true}; return true;
			case OSC_MFT_CURRENT_ANGULAR_VELOCITY: fi = {t.type, MC_CUR_ANGVEL, 3, false, false, -1, true}; return true;
			case OSC_MFT_SENSED_FORCE_CONTROL_WORLD: fi = {t.type, MC_SENSED_F, 3, false}; return true;
			case OSC_MFT_SENSED_MOMENT_CONTROL_WORLD: fi = {t.type, MC_SENSED_M, 3, false}; return true;
			case OSC_MFT_UNIT_MASS_FORCE: fi = {t.type, MC_UNIT_MASS_FORCE, 6, false, false, -1, true}; return true;
			case OSC_MFT_INTEGRATED_POSITION_ERROR: fi = {t.type, MC_INT_POS, 3, false}; return true;
			case OSC_MFT_INTEGRATED_ORIENTATION_ERROR: fi = {t.type, MC_INT_ORI, 3, false}; return true;
			case OSC_MFT_INTEGRATED_FORCE_ERROR: fi = {t.type, MC_INT_FORCE, 3, false}; return true;
			case OSC_MFT_INTEGRATED_MOMENT_ERROR: fi = {t.type, MC_INT_MOMENT, 3, false}; return true;
			case OSC_MFT_POPC_STATE: fi = {t.type, MC_POPC, 4, false}; return true;
			case OSC_MFT_TYPE1_POSTURE: fi = {t.type, MC_Q_PRIOR, n, true}; return true;
			default: return false;
		}
	}
	const int k = h->prog.jt[t.index].k;
	switch (field) {
		case OSC_JT_GOAL_POSITION: fi = {t.type, JC_GOAL_POS, k, true, true}; return true;
		case OSC_JT_GOAL_VELOCITY: fi = {t.type, JC_GOAL_VEL, k, true, true}; return true;
		case OSC_JT_GOAL_ACCELERATION: fi = {t.type, JC_GOAL_ACC, k, true, true}; return true;
		case OSC_JT_INTEGRATED_POSITION_ERROR: fi = {t.type, JC_INT, k, false}; return true;
		case OSC_JT_DESIRED_POSITION: fi = {t.type, JC_GOAL_POS, k, false}; return true;
		case OSC_JT_DESIRED_VELOCITY: fi = {t.type, JC_GOAL_VEL, k, false}; return true;
		case OSC_JT_DESIRED_ACCELERATION: fi = {t.type, JC_GOAL_ACC, k, false}; return true;
		default: return false;
	}
}

double* task_state(osc_handle* h, int task_id) {
	const TaskInfo& t = h->tasks[task_id];
	return t.type == OSC_TASK_MOTION_FORCE ? h->prog.mft[t.index].st : h->prog.jt[t.index].st;
}

DevOtg& task_otg(osc_handle* h, int task_id) {
	const TaskInfo& t = h->tasks[task_id];
	return t.type == OSC_TASK_MOTION_FORCE ? h->prog.mft[t.index].otg : h->prog.jt[t.index].otg;
}
// where a field lives: goal fields move into the generator's block while the task's internal OTG is on
double* field_storage(osc_handle* h, int task_id, const FieldInfo& fi) {
	DevOtg& g = task_otg(h, task_id);
	if (fi.goal && g.enabled) {
		const int comp = (fi.type == OSC_TASK_MOTION_FORCE) ? OC_USER + fi.comp : OJ_USER_POS + fi.comp;  // JC_GOAL_POS/VEL/ACC = 0/8/16
		return g.st + (size_t)comp * h->NR;
	}
	return task_state(h, task_id) + (size_t)fi.comp * h->NR;
}

int zero_comps(osc_handle* h, double* st, int comp, int ncomp) {
	const double z[16] = {0};
	CUDA_TRY(h, osc::launch_fill(st, h->NR, comp, ncomp, z, h->stream));
	h->launches++;
	return OSC_OK;
}

}  // namespace

extern "C" {

int osc_abi_version(void) { return OSC_ABI_VERSION; }

const char* osc_last_error(const osc_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int osc_create(const osc_model_desc* model, int64_t n_robots, int device, osc_handle** out) {
	if (!model || !out) return fail(nullptr, OSC_ERR_INVALID_ARGUMENT, "null argument in osc_create");
	*out = nullptr;
	if (model->n < 1 || model->n > OSC_MAX_DOF) return fail(nullptr, OSC_ERR_INVALID_ARGUMENT, "model dof must be in 1..8");
	if (n_robots < 1) return fail(nullptr, OSC_ERR_INVALID_ARGUMENT, "n_robots must be positive");
	for (int i = 0; i < model->n; i++) {
		if (model->jtype[i] != 0 && model->jtype[i] != 1) return fail(nullptr, OSC_ERR_INVALID_ARGUMENT, "joint type must be 0 or 1");
		if (!(model->mass[i] > 0)) return fail(nullptr, OSC_ERR_INVALID_ARGUMENT, "body masses must be positive");
	}
	int count = 0;
	cudaError_t e = cudaGetDeviceCount(&count);
	if (e != cudaSuccess || count == 0)
		return fail(nullptr, OSC_ERR_NO_DEVICE,
					std::string("no CUDA device available (this library has no CPU fallback): ") +
						(e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
	if (device < 0 || device >= count) return fail(nullptr, OSC_ERR_INVALID_ARGUMENT, "device index out of range");
	osc_handle* h = new osc_handle();
	h->device = device;
	h->NR = n_robots;
	h->model = *model;
	std::memset(&h->prog, 0, sizeof(h->prog));
	build_dev_model(*model, h->prog.model);
	h->prog.n_robots = n_robots;
	h->prog.use_prev_torques = 1;
	auto cleanup = [&](int code) {
		std::string msg = h->err;
		osc_destroy(h);
		g_create_error = msg;
		return code;
	};
	if (cudaSetDevice(device) != cudaSuccess) return cleanup(fail(h, OSC_ERR_CUDA, "cudaSetDevice failed"));
	if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess)
		return cleanup(fail(h, OSC_ERR_CUDA, "cudaStreamCreate failed"));
	h->stream = h->own_stream;
	const size_t n = (size_t)model->n;
	int rc;
	// q and dq staging buffers are one allocation, so that host state that is contiguous too ([q; dq]) crosses PCIe in
	// a single copy (h2d_state below)
	if ((rc = dev_alloc(h, &h->d_q, 2 * n * n_robots, true)) != OSC_OK) return cleanup(rc);
	h->d_dq = h->d_q + n * n_robots;
	if ((rc = dev_alloc(h, &h->d_tau, n * n_robots, true)) != OSC_OK) return cleanup(rc);
	if ((rc = dev_alloc(h, &h->d_status, (size_t)n_robots, true)) != OSC_OK) return cleanup(rc);
	h->prog.q = h->d_q;
	h->prog.dq = h->d_dq;
	h->prog.tau = h->d_tau;
	h->prog.status = h->d_status;
	if ((rc = dev_alloc(h, &h->d_sing_list, (size_t)n_robots, true)) != OSC_OK) return cleanup(rc);
	if ((rc = dev_alloc(h, &h->d_sing_count, (size_t)2, true)) != OSC_OK) return cleanup(rc);
	h->prog.sing_list = h->d_sing_list;
	h->prog.sing_count = h->d_sing_count;
	h->prog.sing_parity = 0;
	// SAI_B200_NO_PIPELINE=1 (measurements only): every cycle waits for the whole previous grid, as before
	const char* nopipe = getenv("SAI_B200_NO_PIPELINE");
	if (!(nopipe && nopipe[0] == '1')) {
		const size_t blocks = ((size_t)n_robots + osc::kCycleBlock - 1) / osc::kCycleBlock;
		if ((rc = dev_alloc(h, &h->d_block_epoch, blocks, true)) != OSC_OK) return cleanup(rc);
		if ((rc = dev_alloc(h, &h->d_general_done, (size_t)4, true)) != OSC_OK) return cleanup(rc);
		if (cudaHostAlloc((void**)&h->h_seen, sizeof(int32_t), cudaHostAllocMapped) != cudaSuccess) return cleanup(fail(h, OSC_ERR_CUDA, "cudaHostAlloc failed"));
		*h->h_seen = 0;	 // matches general_done[2] == 0: the device rewrites the word only when the count changes
		int32_t* d_seen = nullptr;
		if (cudaHostGetDevicePointer((void**)&d_seen, h->h_seen, 0) != cudaSuccess) return cleanup(fail(h, OSC_ERR_CUDA, "cudaHostGetDevicePointer failed"));
		h->prog.block_epoch = h->d_block_epoch;
		h->prog.general_done = h->d_general_done;
		h->prog.host_seen = d_seen;
	}
	h->prog.epoch = 0;
	h->prog.write_observers = 1;  // like the reference: every computeTorques refreshes the observers
	*out = h;
	return OSC_OK;
}

int osc_destroy(osc_handle* h) {
	if (!h) return OSC_OK;
	cudaSetDevice(h->device);
	if (h->own_stream) cudaStreamSynchronize(h->own_stream);
	if (h->stream && h->stream != h->own_stream) cudaStreamSynchronize(h->stream);
	for (void* p : h->allocations) cudaFree(p);
	if (h->h_seen) cudaFreeHost(h->h_seen);
	if (h->own_stream) cudaStreamDestroy(h->own_stream);
	delete h;
	return OSC_OK;
}

int osc_set_stream(osc_handle* h, void* cuda_stream) {
	ENTER(h);
	CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
	return OSC_OK;
}

int osc_sync(osc_handle* h) {
	ENTER(h);
	CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	return OSC_OK;
}

int64_t osc_num_robots(const osc_handle* h) { return h ? h->NR : 0; }
int osc_dof(const osc_handle* h) { return h ? h->model.n : 0; }
int64_t osc_launch_count(const osc_handle* h) { return h ? h->launches : 0; }

// host q, dq -> the handle's staging buffers: one copy when the caller's arrays are adjacent, else two
static cudaError_t h2d_state(osc_handle* h, const double* q, const double* dq) {
	const size_t count = (size_t)h->model.n * h->NR;
	if (dq == q + count) return cudaMemcpyAsync(h->d_q, q, 2 * count * sizeof(double), cudaMemcpyHostToDevice, h->stream);
	cudaError_t e = cudaMemcpyAsync(h->d_q, q, count * sizeof(double), cudaMemcpyHostToDevice, h->stream);
	if (e != cudaSuccess) return e;
	return cudaMemcpyAsync(h->d_dq, dq, count * sizeof(double), cudaMemcpyHostToDevice, h->stream);
}

int osc_set_state(osc_handle* h, const double* q, const double* dq, int mem_kind) {
	ENTER(h);
	if (!q || !dq) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null state pointer");
	const size_t bytes = (size_t)h->model.n * h->NR * sizeof(double);
	if (mem_kind == OSC_MEM_HOST) {
		CUDA_TRY(h, h2d_state(h, q, dq));
		// the caller may reuse its (pageable) buffers as soon as we return
		CUDA_TRY(h, cudaStreamSynchronize(h->stream));
		h->prog.q = h->d_q;
		h->prog.dq = h->d_dq;
	} else if (mem_kind == OSC_MEM_DEVICE) {
		// device state is borrowed (zero copy) until the next osc_set_state / osc_step
		h->prog.q = q;
		h->prog.dq = dq;
	} else {
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	}
	return OSC_OK;
}

int osc_add_joint_task(osc_handle* h, const double* selection, int k, double loop_timestep, int* task_id) {
	ENTER(h);
	if (h->finalized) return fail(h, OSC_ERR_STATE, "controller already finalized");
	if ((int)h->tasks.size() >= OSC_MAX_TASKS || h->n_jt >= 2) return fail(h, OSC_ERR_UNSUPPORTED, "too many tasks");
	const int n = h->model.n;
	DevJt& t = h->prog.jt[h->n_jt];
	std::memset(&t, 0, sizeof(t));
	if (!selection) {
		t.k = n;
		t.full = 1;
		for (int a = 0; a < n; a++) t.S[a][a] = 1.0;
	} else {
		if (k < 1 || k > n)
			return fail(h, OSC_ERR_INVALID_ARGUMENT,
						"joint selection matrix size not consistent with robot dof in JointTask constructor");
		if (rank_of(selection, k, n) != k)
			return fail(h, OSC_ERR_INVALID_ARGUMENT, "joint selection matrix is not full rank in JointTask constructor");
		t.k = k;
		bool ident = (k == n);
		for (int a = 0; a < k; a++)
			for (int j = 0; j < n; j++) {
				t.S[a][j] = selection[(size_t)a * n + j];
				if (t.S[a][j] != ((a == j) ? 1.0 : 0.0)) ident = false;
			}
		t.full = ident ? 1 : 0;
	}
	if (!(loop_timestep > 0)) return fail(h, OSC_ERR_INVALID_ARGUMENT, "loop timestep must be positive");
	t.dt = loop_timestep;
	osc_joint_default_params(&t.p);
	int rc = dev_alloc(h, &t.st, (size_t)JC_COUNT * h->NR, true);
	if (rc != OSC_OK) return rc;
	{
		TaskInfo ti;
		ti.type = OSC_TASK_JOINT;
		ti.index = h->n_jt;
		ti.dt = loop_timestep;
		h->tasks.push_back(ti);
	}
	h->prog.tasks[h->tasks.size() - 1] = DevTask{OSC_TASK_JOINT, h->n_jt};
	h->prog.n_tasks = (int)h->tasks.size();
	CUDA_TRY(h, osc::launch_reset_robots(h->prog, nullptr, (int)h->tasks.size() - 1, 1, h->stream));
	h->launches++;
	h->n_jt++;
	if (task_id) *task_id = (int)h->tasks.size() - 1;
	return OSC_OK;
}

int osc_add_motion_force_task(osc_handle* h, const osc_mft_desc* desc, int* task_id) {
	ENTER(h);
	if (!desc) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null descriptor");
	if (h->finalized) return fail(h, OSC_ERR_STATE, "controller already finalized");
	if ((int)h->tasks.size() >= OSC_MAX_TASKS || h->n_mft >= 2) return fail(h, OSC_ERR_UNSUPPORTED, "too many tasks");
	const int n = h->model.n;
	if (desc->link.body < -1 || desc->link.body >= n) return fail(h, OSC_ERR_INVALID_ARGUMENT, "link body index out of range");
	if (!(desc->loop_timestep > 0)) return fail(h, OSC_ERR_INVALID_ARGUMENT, "loop timestep must be positive");
	DevMft& t = h->prog.mft[h->n_mft];
	std::memset(&t, 0, sizeof(t));
	t.body = desc->link.body;
	mat3_mul_h(desc->link.R, desc->compliant_R, t.ctrl_R);
	double tt[3];
	mat3_vec_h(desc->link.R, desc->compliant_t, tt);
	for (int k = 0; k < 3; k++) t.ctrl_t[k] = desc->link.t[k] + tt[k];
	const double I3[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
	std::memcpy(t.cs_R, I3, sizeof(I3));
	double Ut[9] = {0}, Ur[9] = {0};
	int rt, rr;
	if (!desc->partial) {
		rt = rr = 3;
		std::memcpy(Ut, I3, sizeof(I3));
		std::memcpy(Ur, I3, sizeof(I3));
	} else {
		if (desc->n_dirs_translation < 0 || desc->n_dirs_translation > 3 || desc->n_dirs_rotation < 0 || desc->n_dirs_rotation > 3)
			return fail(h, OSC_ERR_INVALID_ARGUMENT, "at most 3 controlled directions per block");
		if (desc->n_dirs_translation == 0 && desc->n_dirs_rotation == 0)
			return fail(h, OSC_ERR_INVALID_ARGUMENT,
						"controlled_directions_translation and controlled_directions_rotation cannot both be empty in "
						"MotionForceTask::MotionForceTask");
		rt = range_basis_3(desc->dirs_translation, desc->n_dirs_translation, Ut);
		rr = range_basis_3(desc->dirs_rotation, desc->n_dirs_rotation, Ur);
		if (rt + rr == 0)
			return fail(h, OSC_ERR_INVALID_ARGUMENT,
						"controlled_directions_translation and controlled_directions_rotation cannot both be empty in "
						"MotionForceTask::MotionForceTask");
	}
	t.pos_range = rt;
	t.ori_range = rr;
	t.rank = rt + rr;
	t.full = (rt == 3 && rr == 3) ? 1 : 0;
	for (int c = 0; c < rt; c++)
		for (int i = 0; i < 3; i++) t.B[i][c] = Ut[3 * i + c];
	for (int c = 0; c < rr; c++)
		for (int i = 0; i < 3; i++) t.B[3 + i][rt + c] = Ur[3 * i + c];
	for (int i = 0; i < 3; i++)
		for (int j = 0; j < 3; j++) {
			double st_ = 0, sr_ = 0;
			for (int c = 0; c < rt; c++) st_ += Ut[3 * i + c] * Ut[3 * j + c];
			for (int c = 0; c < rr; c++) sr_ += Ur[3 * i + c] * Ur[3 * j + c];
			t.Pt[3 * i + j] = st_;
			t.Pr[3 * i + j] = sr_;
		}
	t.in_compliant = desc->force_motion_in_compliant_frame ? 1 : 0;
	t.dt = desc->loop_timestep;
	osc_mft_default_params(&t.p);
	int rc;
	if ((rc = dev_alloc(h, &t.st, (size_t)MC_COUNT * h->NR, true)) != OSC_OK) return rc;
	if ((rc = dev_alloc(h, &t.ist, (size_t)MI_COUNT * h->NR, true)) != OSC_OK) return rc;
	{
		TaskInfo ti;
		ti.type = OSC_TASK_MOTION_FORCE;
		ti.index = h->n_mft;
		ti.dt = desc->loop_timestep;
		std::memcpy(ti.compliant_R, desc->compliant_R, sizeof(ti.compliant_R));
		std::memcpy(ti.compliant_t, desc->compliant_t, sizeof(ti.compliant_t));
		ti.link = desc->link;
		h->tasks.push_back(ti);
	}
	h->prog.tasks[h->tasks.size() - 1] = DevTask{OSC_TASK_MOTION_FORCE, h->n_mft};
	h->prog.n_tasks = (int)h->tasks.size();
	CUDA_TRY(h, osc::launch_reset_robots(h->prog, nullptr, (int)h->tasks.size() - 1, 1, h->stream));
	h->launches++;
	h->n_mft++;
	if (task_id) *task_id = (int)h->tasks.size() - 1;
	return OSC_OK;
}

int osc_finalize_controller(osc_handle* h, int use_previous_torques) {
	ENTER(h);
	if (h->finalized) return fail(h, OSC_ERR_STATE, "controller already finalized");
	if (h->tasks.empty()) return fail(h, OSC_ERR_INVALID_ARGUMENT, "RobotController must have at least one task");
	bool closed = false;
	for (size_t i = 0; i < h->tasks.size(); i++) {
		if (h->tasks[i].dt != h->tasks[0].dt)
			return fail(h, OSC_ERR_INVALID_ARGUMENT, "All tasks must have the same loop timestep in RobotController");
		if (closed)
			return fail(h, OSC_ERR_INVALID_ARGUMENT,
						"task cannot be added to the controller because it is in the nullspace of a full joint task");
		if (h->tasks[i].type == OSC_TASK_JOINT && h->prog.jt[h->tasks[i].index].k == h->model.n) closed = true;
	}
	// hierarchy signatures with a specialised fast kernel: [JT full], [MFT], [MFT, JT full]; anything else runs on the
	// general-hierarchy kernel
	int R = 0;
	bool jt = false;
	bool ok = true;
	if (h->tasks.size() == 1) {
		if (h->tasks[0].type == OSC_TASK_MOTION_FORCE)
			R = h->prog.mft[0].rank;
		else {
			jt = true;
			ok = h->prog.jt[0].full != 0;
		}
	} else if (h->tasks.size() == 2 && h->tasks[0].type == OSC_TASK_MOTION_FORCE && h->tasks[1].type == OSC_TASK_JOINT &&
			   h->prog.jt[0].full) {
		R = h->prog.mft[0].rank;
		jt = true;
	} else {
		ok = false;
	}
	if (!ok) {  // partial joint tasks, several motion-force tasks, ...: the general-hierarchy kernel
		R = -1;
		jt = false;
	}
	if (!osc::cycle_signature_available(h->model.n, R, jt))
		return fail(h, OSC_ERR_UNSUPPORTED, "no kernel compiled for this robot dof (see OSC_CYCLE_DOFS in csrc/osc_launch.h)");
	h->sig_R = R;
	h->sig_jt = jt;
	h->prog.use_prev_torques = use_previous_torques ? 1 : 0;
	h->finalized = true;
	return OSC_OK;
}

int osc_num_tasks(const osc_handle* h) { return h ? (int)h->tasks.size() : 0; }
int osc_get_task_type(const osc_handle* h, int task_id) {
	if (!h || task_id < 0 || task_id >= (int)h->tasks.size()) return OSC_ERR_INVALID_ARGUMENT;
	return h->tasks[task_id].type;
}
int osc_get_task_dof(const osc_handle* h, int task_id) {
	if (!h || task_id < 0 || task_id >= (int)h->tasks.size()) return OSC_ERR_INVALID_ARGUMENT;
	const TaskInfo& t = h->tasks[task_id];
	return t.type == OSC_TASK_JOINT ? h->prog.jt[t.index].k : h->prog.mft[t.index].rank;
}

int osc_mft_default_params(osc_mft_params* p) {
	if (!p) return OSC_ERR_INVALID_ARGUMENT;
	std::memset(p, 0, sizeof(*p));
	for (int k = 0; k < 3; k++) {  // MotionForceTask.h:44-49
		p->kp_pos[k] = 100.0;
		p->kv_pos[k] = 20.0;
		p->ki_pos[k] = 0.0;
		p->kp_ori[k] = 200.0;
		p->kv_ori[k] = 28.3;
		p->ki_ori[k] = 0.0;
	}
	p->kp_force = 0.7;	// :50-58
	p->kv_force = 10.0;
	p->ki_force = 1.3;
	p->kp_moment = 0.7;
	p->kv_moment = 10.0;
	p->ki_moment = 1.3;
	p->kff_force = 0.95;
	p->kff_moment = 0.95;
	p->max_force_control_feedback_output = 20.0;
	p->max_moment_control_feedback_output = 10.0;
	p->linear_saturation_velocity = 0.3;  // :64-66
	p->angular_saturation_velocity = M_PI / 3;
	p->bie_threshold = 0.1;
	p->s_min = 6e-3;  // MotionForceTask.cpp:197
	p->s_max = 6e-2;
	p->kp_type_1 = 50;	// SingularityHandler.cpp:10-20
	p->kv_type_1 = 14;
	p->kv_type_2 = 5;
	p->s_abs_tol = 1e-3;
	p->type_1_tol = 0.5;
	p->type_2_torque_ratio = 1e-2;
	p->type_2_angle_threshold = 5 * M_PI / 180;
	p->perturb_step_size = 5;
	p->buffer_size = 200;
	p->dynamic_decoupling_type = OSC_BOUNDED_INERTIA_ESTIMATES;
	p->singularity_handling_enabled = 1;
	return OSC_OK;
}

int osc_mft_get_params(const osc_handle* h, int task_id, osc_mft_params* p) {
	if (!h || !p) return OSC_ERR_INVALID_ARGUMENT;
	if (check_task(const_cast<osc_handle*>(h), task_id, OSC_TASK_MOTION_FORCE) != OSC_OK) return OSC_ERR_INVALID_ARGUMENT;
	*p = h->prog.mft[h->tasks[task_id].index].p;
	return OSC_OK;
}

int osc_mft_set_params(osc_handle* h, int task_id, const osc_mft_params* p) {
	ENTER(h);
	if (!p) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null params");
	int rc = check_task(h, task_id, OSC_TASK_MOTION_FORCE);
	if (rc != OSC_OK) return rc;
	DevMft& t = h->prog.mft[h->tasks[task_id].index];
	const osc_mft_params& c = t.p;
	for (int k = 0; k < 3; k++) {
		if (p->kp_pos[k] < 0 || p->kv_pos[k] < 0 || p->ki_pos[k] < 0)
			return fail(h, OSC_ERR_INVALID_ARGUMENT, "all gains should be positive or zero in MotionForceTask::setPosControlGains");
		if (p->kp_ori[k] < 0 || p->kv_ori[k] < 0 || p->ki_ori[k] < 0)
			return fail(h, OSC_ERR_INVALID_ARGUMENT, "all gains should be positive or zero in MotionForceTask::setOriControlGains");
	}
	if (p->use_velocity_saturation && (p->linear_saturation_velocity <= 0 || p->angular_saturation_velocity <= 0))
		return fail(h, OSC_ERR_INVALID_ARGUMENT,
					"Velocity saturation values should be strictly positive or zero in MotionForceTask::enableVelocitySaturation");
	if (p->bie_threshold < 0) return fail(h, OSC_ERR_INVALID_ARGUMENT, "bounded inertia estimate threshold must not be negative");
	if (p->dynamic_decoupling_type < 0 || p->dynamic_decoupling_type > 2)
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "Dynamic decoupling type not recognized");
	if (p->buffer_size < 1 || p->buffer_size > OSC_HIST_MAX)
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "singularity history buffer size must be in 1..256");
	if (p->force_space_dimension != c.force_space_dimension || p->moment_space_dimension != c.moment_space_dimension ||
		std::memcmp(p->force_or_motion_axis, c.force_or_motion_axis, sizeof(c.force_or_motion_axis)) != 0 ||
		std::memcmp(p->moment_or_rotmotion_axis, c.moment_or_rotmotion_axis, sizeof(c.moment_or_rotmotion_axis)) != 0)
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "force/moment spaces must be changed with osc_mft_parametrize_*");
	if (p->closed_loop_force_control != c.closed_loop_force_control || p->closed_loop_moment_control != c.closed_loop_moment_control)
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "closed loop flags must be changed with osc_mft_set_closed_loop_*");
	if (p->passivity_enabled != c.passivity_enabled)
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "passivity must be changed with osc_mft_enable_passivity");
	if (t.gains && std::memcmp(p, &c, GAIN_COUNT * sizeof(double)) != 0)
		return fail(h, OSC_ERR_STATE, "this task's gains are per robot: change them with osc_set_gains");
	t.p = *p;
	return OSC_OK;
}

// ---- force / moment spaces and closed-loop flags, broadcast and per robot ----
namespace {
const char* space_dim_msg(bool moment) {
	return moment ? "Moment space dimension should be between 0 and 3 in MotionForceTask::parametrizeMomentRotMotionSpaces"
				  : "Force space dimension should be between 0 and 3 in MotionForceTask::parametrizeForceMotionSpaces";
}
const char* space_axis_msg(bool moment) {
	return moment ? "Moment or rot motion axis should be a non singular vector in MotionForceTask::parametrizeMomentRotMotionSpaces"
				  : "Force or motion axis should be a non singular vector in MotionForceTask::parametrizeForceMotionSpaces";
}
int32_t space_summary(const osc_mft_params& p) {
	return (p.force_space_dimension ? SPS_FORCE_DIM : 0) | (p.moment_space_dimension ? SPS_MOMENT_DIM : 0) |
		   (p.closed_loop_force_control ? SPS_CL_FORCE : 0) | (p.closed_loop_moment_control ? SPS_CL_MOMENT : 0);
}
void set_summary_bit(DevMft& t, int32_t bit, bool on) { t.space_any = (t.space_any & ~bit) | (on ? bit : 0); }
// The first per-robot call on a task: its space block, every robot as the broadcast parameters say.  There is no way back.
int space_block(osc_handle* h, DevMft& t) {
	if (t.space_mode) return OSC_OK;
	int32_t* mode = nullptr;
	double* axes = nullptr;
	int rc = dev_alloc(h, &mode, (size_t)h->NR, false);
	if (rc != OSC_OK) return rc;
	if ((rc = dev_alloc(h, &axes, (size_t)SP_AXES_COUNT * h->NR, false)) != OSC_OK) return rc;
	const osc_mft_params& p = t.p;
	const double v[SP_AXES_COUNT] = {p.force_or_motion_axis[0], p.force_or_motion_axis[1], p.force_or_motion_axis[2],
									 p.moment_or_rotmotion_axis[0], p.moment_or_rotmotion_axis[1], p.moment_or_rotmotion_axis[2]};
	CUDA_TRY(h, osc::launch_fill_int(mode, h->NR, 0, 1,
									 space_mode_word(p.force_space_dimension, p.moment_space_dimension, p.closed_loop_force_control != 0,
													 p.closed_loop_moment_control != 0),
									 h->stream));
	CUDA_TRY(h, osc::launch_fill(axes, h->NR, 0, SP_AXES_COUNT, v, h->stream));
	h->launches += 2;
	t.space_mode = mode;
	t.space_axes = axes;
	t.space_any = space_summary(p);
	return OSC_OK;
}
int space_staging(osc_handle* h) {
	if (h->d_space_axes) return OSC_OK;
	int rc = dev_alloc(h, &h->d_space_axes, (size_t)3 * h->NR, false);
	if (rc != OSC_OK) return rc;
	return dev_alloc(h, &h->d_space_ints, (size_t)2 * h->NR, false);
}
// h->d_check, cleared in stream order
int clear_check_word(osc_handle* h) {
	if (!h->d_check) {
		int rc = dev_alloc(h, &h->d_check, 1, false);
		if (rc != OSC_OK) return rc;
	}
	CUDA_TRY(h, cudaMemsetAsync(h->d_check, 0, sizeof(int32_t), h->stream));
	return OSC_OK;
}
// SpaceCheck bits of per-robot values in device memory (dims / axes or flags); synchronises the stream
int check_spaces_device(osc_handle* h, const int32_t* dims, const double* axes, const int32_t* flags, int32_t* f) {
	int rc = clear_check_word(h);
	if (rc != OSC_OK) return rc;
	CUDA_TRY(h, osc::launch_check_spaces(dims, axes, flags, h->NR, h->d_check, h->stream));
	h->launches++;
	CUDA_TRY(h, cudaMemcpyAsync(f, h->d_check, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
	CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	return OSC_OK;
}
}  // namespace

static int parametrize_common(osc_handle* h, int task_id, int dim, const double axis[3], bool moment, int* was_reset) {
	int rc = check_task(h, task_id, OSC_TASK_MOTION_FORCE);
	if (rc != OSC_OK) return rc;
	const int idx = h->tasks[task_id].index;
	DevMft& t = h->prog.mft[idx];
	if (dim < 0 || dim > 3) return fail(h, OSC_ERR_INVALID_ARGUMENT, space_dim_msg(moment));
	int32_t& cur_dim = moment ? t.p.moment_space_dimension : t.p.force_space_dimension;
	double* cur_axis = moment ? t.p.moment_or_rotmotion_axis : t.p.force_or_motion_axis;
	bool reset = dim != cur_dim;
	if (dim == 1 || dim == 2) {
		if (!axis) return fail(h, OSC_ERR_INVALID_ARGUMENT, "axis required for dimension 1 or 2");
		double a[3];
		if (space_normalize(axis, a) < 1e-2) return fail(h, OSC_ERR_INVALID_ARGUMENT, space_axis_msg(moment));
		reset = reset || !space_axis_is_approx(a, cur_axis);
		for (int k = 0; k < 3; k++) cur_axis[k] = a[k];
	}
	cur_dim = dim;
	if (t.space_mode) {
		// per-robot spaces: the same values for every robot, each robot decides its own reset; *was_reset: any robot was reset
		set_summary_bit(t, moment ? SPS_MOMENT_DIM : SPS_FORCE_DIM, dim != 0);
		if ((rc = clear_check_word(h)) != OSC_OK) return rc;
		const double none[3] = {0, 0, 0};
		CUDA_TRY(h, osc::launch_apply_spaces(h->prog, idx, moment ? 1 : 0, nullptr, nullptr, dim, axis ? axis : none, nullptr, h->d_check, h->stream));
		h->launches++;
		int32_t any = 0;
		CUDA_TRY(h, cudaMemcpyAsync(&any, h->d_check, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
		CUDA_TRY(h, cudaStreamSynchronize(h->stream));
		if (was_reset) *was_reset = any ? 1 : 0;
		return OSC_OK;
	}
	if (reset && t.otg.enabled) {
		// the same resets with the internal OTG on: goals and generator together (_otg->reInitializeLinear / Angular, :854, :886)
		CUDA_TRY(h, osc::launch_otg_init(h->prog, task_id, moment ? 2 : 1, h->stream));
		h->launches++;
		if ((rc = zero_comps(h, t.st, moment ? MC_INT_ORI : MC_INT_POS, 3)) != OSC_OK) return rc;
		if ((rc = zero_comps(h, t.st, moment ? MC_INT_MOMENT : MC_INT_FORCE, 3)) != OSC_OK) return rc;
	} else if (reset) {
		if (!moment) {	// MotionForceTask.cpp:850-856
			CUDA_TRY(h, osc::launch_copy(t.st, h->NR, MC_GOAL_POS, MC_CUR_POS, 3, h->stream));
			h->launches++;
			if ((rc = zero_comps(h, t.st, MC_GOAL_LINVEL, 3)) != OSC_OK) return rc;
			if ((rc = zero_comps(h, t.st, MC_GOAL_LINACC, 3)) != OSC_OK) return rc;
			if ((rc = zero_comps(h, t.st, MC_INT_POS, 3)) != OSC_OK) return rc;
			if ((rc = zero_comps(h, t.st, MC_INT_FORCE, 3)) != OSC_OK) return rc;
		} else {  // :882-888
			CUDA_TRY(h, osc::launch_copy(t.st, h->NR, MC_GOAL_ORI, MC_CUR_ORI, 9, h->stream));
			h->launches++;
			if ((rc = zero_comps(h, t.st, MC_GOAL_ANGVEL, 3)) != OSC_OK) return rc;
			if ((rc = zero_comps(h, t.st, MC_GOAL_ANGACC, 3)) != OSC_OK) return rc;
			if ((rc = zero_comps(h, t.st, MC_INT_ORI, 3)) != OSC_OK) return rc;
			if ((rc = zero_comps(h, t.st, MC_INT_MOMENT, 3)) != OSC_OK) return rc;
		}
	}
	if (was_reset) *was_reset = reset ? 1 : 0;
	return OSC_OK;
}

int osc_mft_parametrize_force_motion_spaces(osc_handle* h, int task_id, int dim, const double axis[3], int* was_reset) {
	ENTER(h);
	return parametrize_common(h, task_id, dim, axis, false, was_reset);
}
int osc_mft_parametrize_moment_rotmotion_spaces(osc_handle* h, int task_id, int dim, const double axis[3], int* was_reset) {
	ENTER(h);
	return parametrize_common(h, task_id, dim, axis, true, was_reset);
}

int osc_mft_reset_integrators(osc_handle* h, int task_id, int which) {
	ENTER(h);
	int rc = check_task(h, task_id, OSC_TASK_MOTION_FORCE);
	if (rc != OSC_OK) return rc;
	DevMft& t = h->prog.mft[h->tasks[task_id].index];
	if (which == 0 || which == 1) {
		if ((rc = zero_comps(h, t.st, MC_INT_POS, 3)) != OSC_OK) return rc;
		if ((rc = zero_comps(h, t.st, MC_INT_FORCE, 3)) != OSC_OK) return rc;
	}
	if (which == 0 || which == 2) {
		if ((rc = zero_comps(h, t.st, MC_INT_ORI, 3)) != OSC_OK) return rc;
		if ((rc = zero_comps(h, t.st, MC_INT_MOMENT, 3)) != OSC_OK) return rc;
	}
	return OSC_OK;
}

static int set_closed_loop_common(osc_handle* h, int task_id, int enabled, bool moment) {
	int rc = check_task(h, task_id, OSC_TASK_MOTION_FORCE);
	if (rc != OSC_OK) return rc;
	const int idx = h->tasks[task_id].index;
	DevMft& t = h->prog.mft[idx];
	int32_t& cur = moment ? t.p.closed_loop_moment_control : t.p.closed_loop_force_control;
	const bool changed = (cur != 0) != (enabled != 0);
	cur = enabled ? 1 : 0;
	if (t.space_mode) {
		// per-robot flags: every robot gets the flag, a robot whose flag changes gets its integrators zeroed
		set_summary_bit(t, moment ? SPS_CL_MOMENT : SPS_CL_FORCE, enabled != 0);
		CUDA_TRY(h, osc::launch_set_closed_loop(h->prog, idx, moment ? 1 : 0, nullptr, enabled ? 1 : 0, h->stream));
		h->launches++;
		return OSC_OK;
	}
	return changed ? osc_mft_reset_integrators(h, task_id, moment ? 2 : 1) : OSC_OK;
}
int osc_mft_set_closed_loop_force_control(osc_handle* h, int task_id, int enabled) {
	ENTER(h);
	return set_closed_loop_common(h, task_id, enabled, false);
}
int osc_mft_set_closed_loop_moment_control(osc_handle* h, int task_id, int enabled) {
	ENTER(h);
	return set_closed_loop_common(h, task_id, enabled, true);
}

int osc_mft_parametrize_spaces_batched(osc_handle* h, int task_id, int which, const int32_t* dims, const double* axes, int32_t* was_reset,
									   int mem_kind) {
	ENTER(h);
	int rc = check_task(h, task_id, OSC_TASK_MOTION_FORCE);
	if (rc != OSC_OK) return rc;
	if (which != 0 && which != 1) return fail(h, OSC_ERR_INVALID_ARGUMENT, "which must be 0 (force / motion) or 1 (moment / rot motion)");
	if (!dims || !axes) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null dims or axes");
	if (mem_kind != OSC_MEM_HOST && mem_kind != OSC_MEM_DEVICE) return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	const bool moment = which == 1, host = mem_kind == OSC_MEM_HOST;
	const int idx = h->tasks[task_id].index;
	DevMft& t = h->prog.mft[idx];
	const int64_t NR = h->NR;
	// every value is checked before anything is written
	int32_t f = 0;
	if (host) {
		for (int64_t i = 0; i < NR; i++)
			f |= (dims[i] == 1 || dims[i] == 2) ? space_check(dims[i], axes[i], axes[NR + i], axes[2 * NR + i]) : space_check(dims[i], 0, 0, 0);
	} else if ((rc = check_spaces_device(h, dims, axes, nullptr, &f)) != OSC_OK) {
		return rc;
	}
	if (f & SPC_BAD_DIM) return fail(h, OSC_ERR_INVALID_ARGUMENT, space_dim_msg(moment));
	if (f & SPC_BAD_AXIS) return fail(h, OSC_ERR_INVALID_ARGUMENT, space_axis_msg(moment));
	if ((rc = space_block(h, t)) != OSC_OK) return rc;
	const int32_t* d_dims = dims;
	const double* d_axes = axes;
	int32_t* d_reset = was_reset;
	if (host) {
		if ((rc = space_staging(h)) != OSC_OK) return rc;
		CUDA_TRY(h, cudaMemcpyAsync(h->d_space_ints, dims, (size_t)NR * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
		CUDA_TRY(h, cudaMemcpyAsync(h->d_space_axes, axes, (size_t)3 * NR * sizeof(double), cudaMemcpyHostToDevice, h->stream));
		d_dims = h->d_space_ints;
		d_axes = h->d_space_axes;
		d_reset = was_reset ? h->d_space_ints + NR : nullptr;
	}
	const double none[3] = {0, 0, 0};
	CUDA_TRY(h, osc::launch_apply_spaces(h->prog, idx, moment ? 1 : 0, d_dims, d_axes, 0, none, d_reset, nullptr, h->stream));
	h->launches++;
	set_summary_bit(t, moment ? SPS_MOMENT_DIM : SPS_FORCE_DIM, (f & SPC_NONZERO) != 0);
	if (host) {
		if (was_reset) CUDA_TRY(h, cudaMemcpyAsync(was_reset, d_reset, (size_t)NR * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
		CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	}
	return OSC_OK;
}

int osc_mft_set_closed_loop_batched(osc_handle* h, int task_id, int which, const int32_t* enabled, int mem_kind) {
	ENTER(h);
	int rc = check_task(h, task_id, OSC_TASK_MOTION_FORCE);
	if (rc != OSC_OK) return rc;
	if (which != 0 && which != 1) return fail(h, OSC_ERR_INVALID_ARGUMENT, "which must be 0 (force) or 1 (moment)");
	if (!enabled) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null flags");
	if (mem_kind != OSC_MEM_HOST && mem_kind != OSC_MEM_DEVICE) return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	const bool moment = which == 1, host = mem_kind == OSC_MEM_HOST;
	const int idx = h->tasks[task_id].index;
	DevMft& t = h->prog.mft[idx];
	const int64_t NR = h->NR;
	int32_t f = 0;
	if (host) {
		for (int64_t i = 0; i < NR; i++) f |= closed_loop_check(enabled[i]);
	} else if ((rc = check_spaces_device(h, nullptr, nullptr, enabled, &f)) != OSC_OK) {
		return rc;
	}
	if (f & SPC_BAD_FLAG) return fail(h, OSC_ERR_INVALID_ARGUMENT, "closed loop flags must be 0 or 1");
	if ((rc = space_block(h, t)) != OSC_OK) return rc;
	const int32_t* d_flags = enabled;
	if (host) {
		if ((rc = space_staging(h)) != OSC_OK) return rc;
		CUDA_TRY(h, cudaMemcpyAsync(h->d_space_ints, enabled, (size_t)NR * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
		d_flags = h->d_space_ints;
	}
	CUDA_TRY(h, osc::launch_set_closed_loop(h->prog, idx, moment ? 1 : 0, d_flags, 0, h->stream));
	h->launches++;
	set_summary_bit(t, moment ? SPS_CL_MOMENT : SPS_CL_FORCE, (f & SPC_NONZERO) != 0);
	if (host) CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	return OSC_OK;
}

int osc_mft_get_spaces(osc_handle* h, int task_id, int which, int32_t* dims, double* axes, int32_t* closed_loop, int mem_kind) {
	ENTER(h);
	int rc = check_task(h, task_id, OSC_TASK_MOTION_FORCE);
	if (rc != OSC_OK) return rc;
	if (which != 0 && which != 1) return fail(h, OSC_ERR_INVALID_ARGUMENT, "which must be 0 (force / motion) or 1 (moment / rot motion)");
	if (mem_kind != OSC_MEM_HOST && mem_kind != OSC_MEM_DEVICE) return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	const int idx = h->tasks[task_id].index;
	const int64_t NR = h->NR;
	if (mem_kind == OSC_MEM_DEVICE) {
		CUDA_TRY(h, osc::launch_get_spaces(h->prog, idx, which, dims, axes, closed_loop, h->stream));
		h->launches++;
		return OSC_OK;
	}
	if ((rc = space_staging(h)) != OSC_OK) return rc;
	int32_t* d_dims = dims ? h->d_space_ints : nullptr;
	int32_t* d_cl = closed_loop ? h->d_space_ints + NR : nullptr;
	double* d_axes = axes ? h->d_space_axes : nullptr;
	CUDA_TRY(h, osc::launch_get_spaces(h->prog, idx, which, d_dims, d_axes, d_cl, h->stream));
	h->launches++;
	if (dims) CUDA_TRY(h, cudaMemcpyAsync(dims, d_dims, (size_t)NR * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
	if (closed_loop) CUDA_TRY(h, cudaMemcpyAsync(closed_loop, d_cl, (size_t)NR * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
	if (axes) CUDA_TRY(h, cudaMemcpyAsync(axes, d_axes, (size_t)3 * NR * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
	CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	return OSC_OK;
}

int osc_mft_enable_passivity(osc_handle* h, int task_id, int enabled, int ring_capacity) {
	ENTER(h);
	int rc = check_task(h, task_id, OSC_TASK_MOTION_FORCE);
	if (rc != OSC_OK) return rc;
	DevMft& t = h->prog.mft[h->tasks[task_id].index];
	if (enabled) {
		if (!t.ring) {
			const int cap = ring_capacity > 0 ? ring_capacity : 1024;
			if (cap < 256) return fail(h, OSC_ERR_INVALID_ARGUMENT, "POPC ring capacity must be at least 256 (window is 250)");
			if ((rc = dev_alloc(h, &t.ring, (size_t)cap * h->NR, true)) != OSC_OK) return rc;
			t.ring_capacity = cap;
		}
		t.p.passivity_enabled = 1;
	} else {
		// POPCExplicitForceControl::disable() re-initialises (POPCExplicitForceControl.cpp:25-28)
		t.p.passivity_enabled = 0;
		const double init[4] = {0.0, 0.0, 1.0, 0.0};
		CUDA_TRY(h, osc::launch_fill(t.st, h->NR, MC_POPC, 4, init, h->stream));
		CUDA_TRY(h, osc::launch_fill_int(t.ist, h->NR, MI_POPC_COUNTER, 1, 50, h->stream));
		CUDA_TRY(h, osc::launch_fill_int(t.ist, h->NR, MI_RING_HEAD, 2, 0, h->stream));
		h->launches += 3;
	}
	return OSC_OK;
}

int osc_mft_set_force_sensor_frame(osc_handle* h, int task_id, const double R_in_link[9], const double t_in_link[3]) {
	ENTER(h);
	int rc = check_task(h, task_id, OSC_TASK_MOTION_FORCE);
	if (rc != OSC_OK) return rc;
	if (!R_in_link || !t_in_link) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null sensor frame");
	const TaskInfo& ti = h->tasks[task_id];
	DevMft& t = h->prog.mft[ti.index];
	// _T_control_to_sensor = compliant_frame.inverse() * transformation_in_link  (MotionForceTask.cpp:802)
	double Rct[9];
	mat3t_h(ti.compliant_R, Rct);
	mat3_mul_h(Rct, R_in_link, t.cs_R);
	const double d[3] = {t_in_link[0] - ti.compliant_t[0], t_in_link[1] - ti.compliant_t[1], t_in_link[2] - ti.compliant_t[2]};
	mat3_vec_h(Rct, d, t.cs_t);
	return OSC_OK;
}

int osc_mft_update_sensed_force_and_moment(osc_handle* h, int task_id, const double* force_sensor_frame,
										   const double* moment_sensor_frame, int mem_kind) {
	ENTER(h);
	int rc = check_task(h, task_id, OSC_TASK_MOTION_FORCE);
	if (rc != OSC_OK) return rc;
	if (!force_sensor_frame || !moment_sensor_frame) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null sensed wrench pointer");
	const double *f = force_sensor_frame, *m = moment_sensor_frame;
	if (mem_kind == OSC_MEM_HOST) {
		if (!h->d_fs) {
			if ((rc = dev_alloc(h, &h->d_fs, (size_t)3 * h->NR, false)) != OSC_OK) return rc;
			if ((rc = dev_alloc(h, &h->d_ms, (size_t)3 * h->NR, false)) != OSC_OK) return rc;
		}
		const size_t bytes = (size_t)3 * h->NR * sizeof(double);
		CUDA_TRY(h, cudaMemcpyAsync(h->d_fs, f, bytes, cudaMemcpyHostToDevice, h->stream));
		CUDA_TRY(h, cudaMemcpyAsync(h->d_ms, m, bytes, cudaMemcpyHostToDevice, h->stream));
		CUDA_TRY(h, cudaStreamSynchronize(h->stream));
		f = h->d_fs;
		m = h->d_ms;
	} else if (mem_kind != OSC_MEM_DEVICE) {
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	}
	CUDA_TRY(h, osc::launch_sensed_wrench(h->prog, h->tasks[task_id].index, f, m, h->stream));
	h->launches++;
	return OSC_OK;
}

int osc_joint_default_params(osc_joint_params* p) {
	if (!p) return OSC_ERR_INVALID_ARGUMENT;
	std::memset(p, 0, sizeof(*p));
	for (int i = 0; i < OSC_MAX_DOF; i++) {	 // JointTask.h:32-44
		p->kp[i] = 50.0;
		p->kv[i] = 14.0;
		p->ki[i] = 0.0;
		p->saturation_velocity[i] = M_PI / 3.0;
	}
	p->bie_threshold = 0.1;
	p->dynamic_decoupling_type = OSC_BOUNDED_INERTIA_ESTIMATES;
	return OSC_OK;
}

int osc_joint_get_params(const osc_handle* h, int task_id, osc_joint_params* p) {
	if (!h || !p) return OSC_ERR_INVALID_ARGUMENT;
	if (check_task(const_cast<osc_handle*>(h), task_id, OSC_TASK_JOINT) != OSC_OK) return OSC_ERR_INVALID_ARGUMENT;
	*p = h->prog.jt[h->tasks[task_id].index].p;
	return OSC_OK;
}

int osc_joint_set_params(osc_handle* h, int task_id, const osc_joint_params* p) {
	ENTER(h);
	if (!p) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null params");
	int rc = check_task(h, task_id, OSC_TASK_JOINT);
	if (rc != OSC_OK) return rc;
	DevJt& t = h->prog.jt[h->tasks[task_id].index];
	for (int a = 0; a < t.k; a++) {
		if (p->kp[a] < 0 || p->kv[a] < 0 || p->ki[a] < 0)
			return fail(h, OSC_ERR_INVALID_ARGUMENT, "gains must be positive or zero in JointTask::setGains");
		if (p->use_velocity_saturation && p->saturation_velocity[a] <= 0)
			return fail(h, OSC_ERR_INVALID_ARGUMENT, "saturation velocity must be positive in JointTask::enableVelocitySaturation");
	}
	if (p->dynamic_decoupling_type < 0 || p->dynamic_decoupling_type > 2)
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "Dynamic decoupling type not recognized in JointTask::updateTaskModel");
	if (t.gains) {
		for (int a = 0; a < t.k; a++)
			if (p->kp[a] != t.p.kp[a] || p->kv[a] != t.p.kv[a] || p->ki[a] != t.p.ki[a])
				return fail(h, OSC_ERR_STATE, "this task's gains are per robot: change them with osc_set_gains");
	}
	t.p = *p;
	if (t.p.bie_threshold < 0) t.p.bie_threshold = 0;  // JointTask.h:372-378
	return OSC_OK;
}

// ---- per-robot gains (osc_set_gains / osc_get_gains) ----
// The first GAIN_COUNT doubles of both parameter structs have the layout of the gain block (GainComp).
static_assert(offsetof(osc_mft_params, kp_pos) == 0 && offsetof(osc_mft_params, kp_ori) == MG_KP_ORI * sizeof(double) &&
				  offsetof(osc_mft_params, kp_force) == MG_KP_FORCE * sizeof(double) &&
				  offsetof(osc_mft_params, ki_moment) == MG_KI_MOMENT * sizeof(double),
			  "osc_mft_params gains out of step with GainComp");
static_assert(offsetof(osc_joint_params, kp) == JG_KP * sizeof(double) && offsetof(osc_joint_params, kv) == JG_KV * sizeof(double) &&
				  offsetof(osc_joint_params, ki) == JG_KI * sizeof(double),
			  "osc_joint_params gains out of step with GainComp");

namespace {
struct GainGroup {
	double* params;	 // first GAIN_COUNT doubles of the task's broadcast parameters
	double** block;	 // the task's gain-block pointer
	int comp[3];	 // first block component of kp, kv, ki
	int ncomp;
	bool nonneg;	 // gains must be >= 0 (joint, position, orientation)
	const char* msg;
};
int gain_group(osc_handle* h, int task_id, int group, GainGroup& g) {
	if (group < OSC_GAINS_JOINT || group > OSC_GAINS_MOMENT) return fail(h, OSC_ERR_INVALID_ARGUMENT, "unknown gain group");
	int rc = check_task(h, task_id, group == OSC_GAINS_JOINT ? OSC_TASK_JOINT : OSC_TASK_MOTION_FORCE);
	if (rc != OSC_OK) return rc;
	const int idx = h->tasks[task_id].index;
	if (group == OSC_GAINS_JOINT) {
		DevJt& t = h->prog.jt[idx];
		g = {reinterpret_cast<double*>(&t.p), &t.gains, {JG_KP, JG_KV, JG_KI}, t.k, true, "gains must be positive or zero in JointTask::setGains"};
		return OSC_OK;
	}
	DevMft& t = h->prog.mft[idx];
	g.params = reinterpret_cast<double*>(&t.p);
	g.block = &t.gains;
	switch (group) {
		case OSC_GAINS_POSITION:
			g = {g.params, g.block, {MG_KP_POS, MG_KV_POS, MG_KI_POS}, 3, true, "all gains should be positive or zero in MotionForceTask::setPosControlGains"};
			break;
		case OSC_GAINS_ORIENTATION:
			g = {g.params, g.block, {MG_KP_ORI, MG_KV_ORI, MG_KI_ORI}, 3, true, "all gains should be positive or zero in MotionForceTask::setOriControlGains"};
			break;
		case OSC_GAINS_FORCE:
			g = {g.params, g.block, {MG_KP_FORCE, MG_KV_FORCE, MG_KI_FORCE}, 1, false, "force control gains must be finite"};
			break;
		default:
			g = {g.params, g.block, {MG_KP_MOMENT, MG_KV_MOMENT, MG_KI_MOMENT}, 1, false, "moment control gains must be finite"};
	}
	return OSC_OK;
}
// 0: all finite (and >= 0 where required), else the message's error
int check_gain_values(osc_handle* h, const GainGroup& g, int32_t flags) {
	if (flags & 1) return fail(h, OSC_ERR_INVALID_ARGUMENT, g.nonneg ? std::string(g.msg) + " (non-finite value)" : std::string(g.msg));
	if ((flags & 2) && g.nonneg) return fail(h, OSC_ERR_INVALID_ARGUMENT, g.msg);
	return OSC_OK;
}
int32_t host_value_flags(const double* v, size_t n) {
	int32_t f = 0;
	for (size_t k = 0; k < n; k++) {
		if (!std::isfinite(v[k])) f |= 1;
		else if (v[k] < 0.0) f |= 2;
	}
	return f;
}
}  // namespace

int osc_set_gains(osc_handle* h, int task_id, int group, const double* kp, const double* kv, const double* ki, int mem_kind, int per_robot) {
	ENTER(h);
	GainGroup g;
	int rc = gain_group(h, task_id, group, g);
	if (rc != OSC_OK) return rc;
	if (!kp || !kv || !ki) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null gains");
	if (mem_kind != OSC_MEM_HOST && mem_kind != OSC_MEM_DEVICE) return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	const double* src[3] = {kp, kv, ki};
	const int64_t NR = h->NR;
	if (!per_robot) {
		if (mem_kind != OSC_MEM_HOST) return fail(h, OSC_ERR_INVALID_ARGUMENT, "broadcast values must be in host memory");
		int32_t f = 0;
		for (int a = 0; a < 3; a++) f |= host_value_flags(src[a], (size_t)g.ncomp);
		if ((rc = check_gain_values(h, g, f)) != OSC_OK) return rc;
		for (int a = 0; a < 3; a++) {
			if (*g.block) {
				CUDA_TRY(h, osc::launch_fill(*g.block, NR, g.comp[a], g.ncomp, src[a], h->stream));
				h->launches++;
			} else {
				std::memcpy(g.params + g.comp[a], src[a], (size_t)g.ncomp * sizeof(double));
			}
		}
		return OSC_OK;
	}
	// per robot: every value is checked before anything is written
	const size_t n = (size_t)g.ncomp * (size_t)NR;
	int32_t f = 0;
	if (mem_kind == OSC_MEM_HOST) {
		for (int a = 0; a < 3; a++) f |= host_value_flags(src[a], n);
	} else {
		if (!h->d_check) {
			rc = dev_alloc(h, &h->d_check, 1, false);
			if (rc != OSC_OK) return rc;
		}
		CUDA_TRY(h, cudaMemsetAsync(h->d_check, 0, sizeof(int32_t), h->stream));
		for (int a = 0; a < 3; a++) {
			CUDA_TRY(h, osc::launch_check_values(src[a], (int64_t)n, h->d_check, h->stream));
			h->launches++;
		}
		CUDA_TRY(h, cudaMemcpyAsync(&f, h->d_check, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
		CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	}
	if ((rc = check_gain_values(h, g, f)) != OSC_OK) return rc;
	if (!*g.block) {
		// entering per-robot mode: every group of the block starts from the current broadcast values
		double* blk = nullptr;
		rc = dev_alloc(h, &blk, (size_t)GAIN_COUNT * NR, false);
		if (rc != OSC_OK) return rc;
		CUDA_TRY(h, osc::launch_fill(blk, NR, 0, 16, g.params, h->stream));
		CUDA_TRY(h, osc::launch_fill(blk, NR, 16, GAIN_COUNT - 16, g.params + 16, h->stream));
		h->launches += 2;
		*g.block = blk;
	}
	for (int a = 0; a < 3; a++)
		CUDA_TRY(h, cudaMemcpyAsync(*g.block + (size_t)g.comp[a] * NR, src[a], n * sizeof(double),
									mem_kind == OSC_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, h->stream));
	if (mem_kind == OSC_MEM_HOST) CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	return OSC_OK;
}

int osc_get_gains(osc_handle* h, int task_id, int group, double* kp, double* kv, double* ki, int mem_kind) {
	ENTER(h);
	GainGroup g;
	int rc = gain_group(h, task_id, group, g);
	if (rc != OSC_OK) return rc;
	if (!kp || !kv || !ki) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null output");
	if (mem_kind != OSC_MEM_HOST && mem_kind != OSC_MEM_DEVICE) return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	double* dst[3] = {kp, kv, ki};
	const int64_t NR = h->NR;
	const size_t n = (size_t)g.ncomp * (size_t)NR;
	for (int a = 0; a < 3; a++) {
		if (*g.block) {
			CUDA_TRY(h, cudaMemcpyAsync(dst[a], *g.block + (size_t)g.comp[a] * NR, n * sizeof(double),
										mem_kind == OSC_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, h->stream));
		} else if (mem_kind == OSC_MEM_DEVICE) {
			CUDA_TRY(h, osc::launch_fill(dst[a], NR, 0, g.ncomp, g.params + g.comp[a], h->stream));
			h->launches++;
		} else {
			for (int c = 0; c < g.ncomp; c++)
				for (int64_t i = 0; i < NR; i++) dst[a][(size_t)c * NR + i] = g.params[g.comp[a] + c];
		}
	}
	if (mem_kind == OSC_MEM_HOST) CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	return OSC_OK;
}

int osc_field_ncomp(const osc_handle* h, int task_id, int field) {
	FieldInfo fi;
	if (!h || !field_info(h, task_id, field, fi)) return OSC_ERR_INVALID_ARGUMENT;
	return fi.ncomp;
}

int osc_set_field(osc_handle* h, int task_id, int field, const double* data, int mem_kind, int broadcast) {
	ENTER(h);
	FieldInfo fi;
	if (!field_info(h, task_id, field, fi)) return fail(h, OSC_ERR_INVALID_ARGUMENT, "unknown field for this task");
	if (!fi.writable) return fail(h, OSC_ERR_INVALID_ARGUMENT, "field is read-only");
	if (!data) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null data");
	double* dst = field_storage(h, task_id, fi);
	if (broadcast) {
		if (mem_kind != OSC_MEM_HOST) return fail(h, OSC_ERR_INVALID_ARGUMENT, "broadcast values must be in host memory");
		for (int c = 0; c < fi.ncomp; c++)
			if (!is_finite(data[c])) return fail(h, OSC_ERR_INVALID_ARGUMENT, "non-finite value");
		CUDA_TRY(h, osc::launch_fill(dst, h->NR, 0, fi.ncomp, data, h->stream));
		h->launches++;
		return OSC_OK;
	}
	const size_t bytes = (size_t)fi.ncomp * h->NR * sizeof(double);
	if (mem_kind == OSC_MEM_HOST) {
		CUDA_TRY(h, cudaMemcpyAsync(dst, data, bytes, cudaMemcpyHostToDevice, h->stream));
		CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	} else if (mem_kind == OSC_MEM_DEVICE) {
		CUDA_TRY(h, cudaMemcpyAsync(dst, data, bytes, cudaMemcpyDeviceToDevice, h->stream));
	} else {
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	}
	return OSC_OK;
}

int osc_get_field(osc_handle* h, int task_id, int field, double* out, int mem_kind) {
	ENTER(h);
	FieldInfo fi;
	if (!field_info(h, task_id, field, fi)) return fail(h, OSC_ERR_INVALID_ARGUMENT, "unknown field for this task");
	if (!out) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null output");
	if (fi.needs_observers && !h->prog.write_observers)
		return fail(h, OSC_ERR_STATE, "this field is refreshed by the cycle kernels only while osc_enable_observers(h, 1) is in effect");
	const double* src = field_storage(h, task_id, fi);
	const size_t bytes = (size_t)fi.ncomp * h->NR * sizeof(double);
	if (fi.observer >= 0) {
		if (!h->finalized) return fail(h, OSC_ERR_STATE, "controller not finalized");
		if (h->scratch_doubles < (size_t)fi.ncomp * h->NR) {
			double* p = nullptr;
			int rc = dev_alloc(h, &p, (size_t)OSC_MAX_DOF * OSC_MAX_DOF * h->NR, false);
			if (rc != OSC_OK) return rc;
			h->d_scratch = p;
			h->scratch_doubles = (size_t)OSC_MAX_DOF * OSC_MAX_DOF * h->NR;
		}
		CUDA_TRY(h, osc::launch_observer(h->prog, task_id, fi.observer, h->d_scratch, h->stream));
		h->launches++;
		src = h->d_scratch;
	}
	if (mem_kind == OSC_MEM_HOST) {
		CUDA_TRY(h, cudaMemcpyAsync(out, src, bytes, cudaMemcpyDeviceToHost, h->stream));
		CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	} else if (mem_kind == OSC_MEM_DEVICE) {
		CUDA_TRY(h, cudaMemcpyAsync(out, src, bytes, cudaMemcpyDeviceToDevice, h->stream));
	} else {
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	}
	return OSC_OK;
}

int osc_reinitialize_task(osc_handle* h, int task_id) { return osc_reset_robots(h, task_id, nullptr, OSC_MEM_DEVICE, OSC_RESET_REINITIALIZE); }

int osc_reset_robots(osc_handle* h, int task_id, const int32_t* robot_mask, int mem_kind, int mode) {
	ENTER(h);
	if (task_id >= (int)h->tasks.size()) return fail(h, OSC_ERR_INVALID_ARGUMENT, "task id out of range");
	if (mode != OSC_RESET_REINITIALIZE && mode != OSC_RESET_CONSTRUCT) return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad reset mode");
	if (mem_kind != OSC_MEM_HOST && mem_kind != OSC_MEM_DEVICE) return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	const int32_t* mask = robot_mask;
	if (robot_mask && mem_kind == OSC_MEM_HOST) {
		if (!h->d_reset_mask) {
			int rc = dev_alloc(h, &h->d_reset_mask, (size_t)h->NR, false);
			if (rc != OSC_OK) return rc;
		}
		CUDA_TRY(h, cudaMemcpyAsync(h->d_reset_mask, robot_mask, (size_t)h->NR * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
		mask = h->d_reset_mask;
	}
	CUDA_TRY(h, osc::launch_reset_robots(h->prog, mask, task_id, mode == OSC_RESET_CONSTRUCT ? 1 : 0, h->stream));
	h->launches++;
	return OSC_OK;
}

// ---- internal OTG (osc_otg_kernels.cuh)
static int otg_enable_common(osc_handle* h, int task_id, int dim, const double* vmax, const double* amax) {
	DevOtg& g = task_otg(h, task_id);
	for (int a = 0; a < dim; a++) {
		if (!(vmax[a] > 0.0) || !is_finite(vmax[a])) return fail(h, OSC_ERR_INVALID_ARGUMENT, "max velocity cannot be 0 or negative in any directions in OTG_joints::setMaxVelocity");
		if (!(amax[a] > 0.0) || !is_finite(amax[a])) return fail(h, OSC_ERR_INVALID_ARGUMENT, "max acceleration cannot be 0 or negative in any directions in OTG_joints::setMaxAcceleration");
	}
	const bool is_mft = h->tasks[task_id].type == OSC_TASK_MOTION_FORCE;
	if (!g.st) {
		int rc = dev_alloc(h, &g.st, (size_t)(is_mft ? OC_COUNT : OJ_COUNT) * h->NR, true);
		if (rc != OSC_OK) return rc;
		if ((rc = dev_alloc(h, &g.flags, (size_t)h->NR, true)) != OSC_OK) return rc;
	}
	for (int a = 0; a < OSC_MAX_DOF; a++) {
		g.vmax[a] = a < dim ? vmax[a] : 1.0;
		g.amax[a] = a < dim ? amax[a] : 1.0;
	}
	const bool was_on = g.enabled != 0;
	g.enabled = 1;
	// off -> on: the generator restarts at the current position (JointTask.cpp:372-374, MotionForceTask.cpp:514-516) and the
	// user's goals stay; already on: new limits only (OTG_joints.cpp:44-92)
	CUDA_TRY(h, osc::launch_otg_init(h->prog, task_id, was_on ? 3 : 0, h->stream));
	h->launches++;
	if (!was_on) h->otg_tasks++;
	return OSC_OK;
}
int osc_joint_enable_internal_otg(osc_handle* h, int task_id, const double* max_velocity, const double* max_acceleration) {
	ENTER(h);
	int rc = check_task(h, task_id, OSC_TASK_JOINT);
	if (rc != OSC_OK) return rc;
	if (!max_velocity || !max_acceleration) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null limits");
	return otg_enable_common(h, task_id, h->prog.jt[h->tasks[task_id].index].k, max_velocity, max_acceleration);
}
int osc_mft_enable_internal_otg(osc_handle* h, int task_id, double max_linear_velocity, double max_linear_acceleration, double max_angular_velocity,
								double max_angular_acceleration) {
	ENTER(h);
	int rc = check_task(h, task_id, OSC_TASK_MOTION_FORCE);
	if (rc != OSC_OK) return rc;
	const double v[6] = {max_linear_velocity, max_linear_velocity, max_linear_velocity, max_angular_velocity, max_angular_velocity, max_angular_velocity};
	const double a[6] = {max_linear_acceleration, max_linear_acceleration, max_linear_acceleration, max_angular_acceleration, max_angular_acceleration,
						 max_angular_acceleration};
	return otg_enable_common(h, task_id, 6, v, a);
}
int osc_disable_internal_otg(osc_handle* h, int task_id) {
	ENTER(h);
	if (task_id < 0 || task_id >= (int)h->tasks.size()) return fail(h, OSC_ERR_INVALID_ARGUMENT, "task id out of range");
	DevOtg& g = task_otg(h, task_id);
	if (!g.enabled) return OSC_OK;
	CUDA_TRY(h, osc::launch_otg_disable(h->prog, task_id, h->stream));
	h->launches++;
	g.enabled = 0;
	h->otg_tasks--;
	return OSC_OK;
}
int osc_internal_otg_enabled(const osc_handle* h, int task_id) {
	if (!h || task_id < 0 || task_id >= (int)h->tasks.size()) return OSC_ERR_INVALID_ARGUMENT;
	return task_otg(const_cast<osc_handle*>(h), task_id).enabled ? 1 : 0;
}
int osc_get_internal_otg_flags(osc_handle* h, int task_id, int32_t* flags_out, int mem_kind) {
	ENTER(h);
	if (task_id < 0 || task_id >= (int)h->tasks.size()) return fail(h, OSC_ERR_INVALID_ARGUMENT, "task id out of range");
	if (!flags_out) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null output");
	DevOtg& g = task_otg(h, task_id);
	if (!g.enabled) return fail(h, OSC_ERR_STATE, "internal OTG is not enabled on this task");
	const size_t bytes = (size_t)h->NR * sizeof(int32_t);
	CUDA_TRY(h, cudaMemcpyAsync(flags_out, g.flags, bytes, mem_kind == OSC_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, h->stream));
	if (mem_kind == OSC_MEM_HOST) CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	return OSC_OK;
}

int osc_enable_gravity_compensation(osc_handle* h, int enabled) {
	ENTER(h);
	h->prog.gravity_comp = enabled ? 1 : 0;
	return OSC_OK;
}
int osc_enable_torque_saturation(osc_handle* h, int enabled) {
	ENTER(h);
	h->prog.torque_saturation = enabled ? 1 : 0;
	return OSC_OK;
}
int osc_enable_joint_limit_avoidance(osc_handle* h, int enabled) {
	ENTER(h);
	h->jla_enabled = enabled != 0;
	return OSC_OK;
}

int osc_set_precision(osc_handle* h, int precision) {
	ENTER(h);
	if (precision != OSC_PRECISION_FP64 && precision != OSC_PRECISION_FP32) return fail(h, OSC_ERR_INVALID_ARGUMENT, "precision must be OSC_PRECISION_FP64 or OSC_PRECISION_FP32");
	if (precision == OSC_PRECISION_FP32 && !osc::cycle_f32_dof(h->model.n))
		return fail(h, OSC_ERR_UNSUPPORTED, "FP32 mode: no single-precision kernel compiled for this robot dof");
	h->prog.precision_fp32 = (precision == OSC_PRECISION_FP32) ? 1 : 0;
	return OSC_OK;
}

int osc_get_precision(osc_handle* h) {
	ENTER(h);
	return h->prog.precision_fp32 ? OSC_PRECISION_FP32 : OSC_PRECISION_FP64;
}

int osc_debug_general_path_counts(osc_handle* h, int32_t* out4) {
	ENTER(h);
	if (!out4) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null output");
	for (int k = 0; k < 4; k++) out4[k] = -1;
	if (!h->prog.blend_counts) return OSC_OK;  // the split blending path has not been used by this handle
	CUDA_TRY(h, cudaMemcpyAsync(out4, h->prog.blend_counts + 4, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
	CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	return OSC_OK;
}

int osc_debug_block_times(osc_handle* h, int enabled, unsigned long long* out, int64_t out_capacity) {
	ENTER(h);
	const size_t blocks = ((size_t)h->NR + osc::kCycleBlock - 1) / osc::kCycleBlock;
	const size_t words = blocks * 8 * 2;
	if (out) {	// read back: [cycle & 7][block][start, end] in globaltimer nanoseconds
		if (!h->d_block_times) return fail(h, OSC_ERR_STATE, "block times were not enabled");
		if (out_capacity < (int64_t)words) return fail(h, OSC_ERR_INVALID_ARGUMENT, "output too small");
		CUDA_TRY(h, cudaMemcpyAsync(out, h->d_block_times, words * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
		CUDA_TRY(h, cudaStreamSynchronize(h->stream));
		return (int)blocks;
	}
	if (enabled && !h->d_block_times) {
		int rc = dev_alloc(h, &h->d_block_times, words, true);
		if (rc != OSC_OK) return rc;
	}
	h->prog.block_times = enabled ? h->d_block_times : nullptr;
	return (int)blocks;
}

int osc_enable_observers(osc_handle* h, int enabled) {
	ENTER(h);
	h->prog.write_observers = enabled ? 1 : 0;
	return OSC_OK;
}

int osc_shard_range(int64_t n_robots, int rank, int world, int64_t* first, int64_t* count) {
	if (n_robots < 0 || world <= 0 || rank < 0 || rank >= world || !first || !count) return OSC_ERR_INVALID_ARGUMENT;
	// robot i belongs to shard floor(i * world / n_robots): shard r starts at ceil(r * n_robots / world)
	const int64_t lo = (rank * n_robots + world - 1) / world, hi = ((rank + 1) * n_robots + world - 1) / world;
	*first = lo;
	*count = hi - lo;
	return OSC_OK;
}

int osc_update_task_models(osc_handle* h) {
	ENTER(h);
	if (!h->finalized) return fail(h, OSC_ERR_STATE, "controller not finalized");
	h->models_armed = true;
	return OSC_OK;
}

static int run_cycle(osc_handle* h, double* tau_out, int mem_kind, bool sync_host = true) {
	if (!h->finalized) return fail(h, OSC_ERR_STATE, "controller not finalized");
	if (!tau_out) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null torque output");
	if (mem_kind != OSC_MEM_HOST && mem_kind != OSC_MEM_DEVICE) return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	// scheduling hint only (any grid size is correct): after a few cycles without hand-overs a handful of general-path blocks
	// is launched instead of a grid that covers the machine
	if (h->h_seen) {
		const int32_t seen = *(volatile int32_t*)h->h_seen;
		h->clean_cycles = (seen == 0) ? h->clean_cycles + 1 : 0;
		h->prog.general_grid_small = h->clean_cycles >= 4 ? 1 : 0;
		// Flagship hierarchy with MANY robots on the general path (more than the single blending kernel holds in a wave and
		// a half): run it as the three kernels of the split blending path (osc_blend.cuh), which keep their speed beyond one
		// wave.  The scratch block (1.3 KB per robot for seven joints) is allocated the first time that happens.
		// SAI_B200_BLEND_SPLIT=0: never (osc_blend_kernel alone);  =1: always, from the first cycle on (tests).
		if (h->blend_split == -1) {
			const char* e = getenv("SAI_B200_BLEND_SPLIT");
			h->blend_split = (h->sig_R == 6 && h->prog.mft[0].full) ? ((e && e[0] == '0') ? 0 : 1) : 0;
			h->blend_split_min = (e && e[0] == '1') ? 0 : 49152;
		}
		const bool many = h->blend_split > 0 && (int64_t)seen >= h->blend_split_min && (seen > 0 || h->blend_split_min == 0);
		if (many && h->blend_split == 1) {
			const size_t cap = (size_t)h->NR, doubles = (size_t)blend_scratch_doubles(h->model.n);
			void *a = nullptr, *b = nullptr, *c = nullptr;
			if (cudaMalloc(&a, cap * doubles * sizeof(double)) == cudaSuccess && cudaMalloc(&b, cap * 4 * sizeof(int32_t)) == cudaSuccess &&
				cudaMalloc(&c, 8 * sizeof(int32_t)) == cudaSuccess && cudaMemsetAsync(c, 0, 8 * sizeof(int32_t), h->stream) == cudaSuccess) {
				h->allocations.push_back(a);
				h->allocations.push_back(b);
				h->allocations.push_back(c);
				h->prog.blend_scratch = (double*)a;
				h->prog.blend_lists = (int32_t*)b;
				h->prog.blend_counts = (int32_t*)c;
				h->prog.blend_cap = (int64_t)cap;
				h->blend_split = 2;
			} else {  // no room: stay with the single kernel
				cudaGetLastError();
				if (a) cudaFree(a);
				if (b) cudaFree(b);
				if (c) cudaFree(c);
				h->blend_split = 0;
			}
		}
		h->prog.blend_split_on = (many && h->blend_split == 2) ? 1 : 0;
	}
	// The program the cycle kernels run.  RobotController.cpp:96-116: the avoidance blend comes after the task torques (and their
	// saturation) and before gravity compensation, so with joint-limit avoidance the cycle kernels leave gravity to its kernel.
	OscProgram prog = h->prog;
	if (h->jla_enabled) prog.gravity_comp = 0;
	// decided before anything is launched or counted: a refused cycle leaves the models armed and the epoch as they were
	const osc::CyclePlan plan = osc::plan_cycle(prog, h->model.n, h->sig_R, h->sig_jt);
	if (plan.error != OSC_OK) return fail(h, plan.error, plan.message);
	h->prog.tau = prog.tau = (mem_kind == OSC_MEM_DEVICE) ? tau_out : h->d_tau;
	h->prog.update_models = prog.update_models = h->models_armed ? 1 : 0;
	h->models_armed = false;
	prog.epoch = ++h->prog.epoch;
	cudaError_t e;
	if (h->otg_tasks > 0) {	 // the tasks' internal OTG produces this cycle's desired state first (JointTask.cpp:313-319, MotionForceTask.cpp:394-407)
		CUDA_TRY(h, osc::launch_otg_update(h->prog, h->stream));
		h->launches += 1;
	}
	e = osc::launch_cycle(h->model.n, h->sig_R, h->sig_jt, plan, prog, h->stream);
	if (e == cudaSuccess && h->jla_enabled) {
		e = osc::launch_jla(h->prog, h->stream);
		if (e == cudaSuccess) h->launches += 1;
	}
	if (e == cudaErrorNotSupported) return fail(h, OSC_ERR_UNSUPPORTED, "no kernel compiled for this hierarchy signature");
	CUDA_TRY(h, e);
	h->launches += plan.launches;
	h->prog.sing_parity ^= 1;
	if (mem_kind == OSC_MEM_HOST) {
		CUDA_TRY(h, cudaMemcpyAsync(tau_out, h->d_tau, (size_t)h->model.n * h->NR * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
		if (sync_host) CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	}
	return OSC_OK;
}

int osc_compute_control_torques(osc_handle* h, double* tau_out, int mem_kind) {
	ENTER(h);
	return run_cycle(h, tau_out, mem_kind);
}

static int step_impl(osc_handle* h, const double* q, const double* dq, double* tau_out, int mem_kind, bool sync_host);

int osc_step(osc_handle* h, const double* q, const double* dq, double* tau_out, int mem_kind) {
	ENTER(h);
	return step_impl(h, q, dq, tau_out, mem_kind, true);
}

int osc_step_async(osc_handle* h, const double* q, const double* dq, double* tau_out, int mem_kind) {
	ENTER(h);
	return step_impl(h, q, dq, tau_out, mem_kind, false);
}

static int step_impl(osc_handle* h, const double* q, const double* dq, double* tau_out, int mem_kind, bool sync_host) {
	if (!h->finalized) return fail(h, OSC_ERR_STATE, "controller not finalized");
	if (!q || !dq) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null state pointer");
	const size_t bytes = (size_t)h->model.n * h->NR * sizeof(double);
	if (mem_kind == OSC_MEM_HOST) {
		CUDA_TRY(h, h2d_state(h, q, dq));
		h->prog.q = h->d_q;
		h->prog.dq = h->d_dq;
	} else if (mem_kind == OSC_MEM_DEVICE) {
		h->prog.q = q;
		h->prog.dq = dq;
	} else {
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	}
	h->models_armed = true;
	return run_cycle(h, tau_out, mem_kind, sync_host);
}

int osc_debug_popc_sequence(osc_handle* h, int task_id, int n_steps, const double* fd, const double* fs, const double* vcl, const double* vr,
							double kv_force, double kff_force, double* out) {
	ENTER(h);
	int rc = check_task(h, task_id, OSC_TASK_MOTION_FORCE);
	if (rc != OSC_OK) return rc;
	if (n_steps < 1 || !fd || !fs || !vcl || !vr || !out) return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad argument");
	const int idx = h->tasks[task_id].index;
	if (!h->prog.mft[idx].p.passivity_enabled || !h->prog.mft[idx].ring) return fail(h, OSC_ERR_STATE, "passivity is not enabled on this task");
	const size_t bytes = (size_t)3 * n_steps * sizeof(double);
	double* d = nullptr;
	CUDA_TRY(h, cudaMalloc(&d, 5 * bytes));
	const double* src[4] = {fd, fs, vcl, vr};
	cudaError_t e = cudaSuccess;
	for (int k = 0; k < 4 && e == cudaSuccess; k++) e = cudaMemcpyAsync(d + (size_t)k * 3 * n_steps, src[k], bytes, cudaMemcpyHostToDevice, h->stream);
	if (e == cudaSuccess)
		e = osc::launch_popc_probe(h->prog, idx, n_steps, d, d + (size_t)3 * n_steps, d + (size_t)6 * n_steps, d + (size_t)9 * n_steps, kv_force, kff_force,
								   d + (size_t)12 * n_steps, h->stream);
	if (e == cudaSuccess) e = cudaMemcpyAsync(out, d + (size_t)12 * n_steps, bytes, cudaMemcpyDeviceToHost, h->stream);
	if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
	cudaFree(d);
	CUDA_TRY(h, e);
	h->launches += 1;
	return OSC_OK;
}

int osc_measure_fp64_peak(osc_handle* h, double seconds, double* tflops_out) {
	ENTER(h);
	if (!tflops_out || !(seconds > 0.0)) return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad argument");
	CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	CUDA_TRY(h, osc::measure_fp64_peak(seconds, tflops_out, h->stream));
	return OSC_OK;
}

int osc_sim_integrate(osc_handle* h, double* q, double* dq, const double* tau, double dt, int substeps, int mem_kind) {
	ENTER(h);
	if (!q || !dq || !tau) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null pointer");
	if (!(dt > 0.0) || substeps < 1) return fail(h, OSC_ERR_INVALID_ARGUMENT, "timestep must be positive and substeps >= 1");
	const size_t bytes = (size_t)h->model.n * h->NR * sizeof(double);
	if (mem_kind == OSC_MEM_DEVICE) {
		CUDA_TRY(h, osc::launch_sim_integrate(h->prog, q, dq, tau, dt, substeps, h->stream));
	} else if (mem_kind == OSC_MEM_HOST) {
		// the simulation has its own staging buffers: the controller's state (osc_set_state) and its last torques are separate
		// objects in the reference too (sai-simulation vs SaiModel) and must survive this call
		if (!h->d_sim) {
			int rc = dev_alloc(h, &h->d_sim, 3 * (size_t)h->model.n * h->NR, false);
			if (rc != OSC_OK) return rc;
		}
		double *sq = h->d_sim, *sdq = h->d_sim + (size_t)h->model.n * h->NR, *stau = h->d_sim + 2 * (size_t)h->model.n * h->NR;
		CUDA_TRY(h, cudaMemcpyAsync(sq, q, bytes, cudaMemcpyHostToDevice, h->stream));
		CUDA_TRY(h, cudaMemcpyAsync(sdq, dq, bytes, cudaMemcpyHostToDevice, h->stream));
		CUDA_TRY(h, cudaMemcpyAsync(stau, tau, bytes, cudaMemcpyHostToDevice, h->stream));
		CUDA_TRY(h, osc::launch_sim_integrate(h->prog, sq, sdq, stau, dt, substeps, h->stream));
		CUDA_TRY(h, cudaMemcpyAsync(q, sq, bytes, cudaMemcpyDeviceToHost, h->stream));
		CUDA_TRY(h, cudaMemcpyAsync(dq, sdq, bytes, cudaMemcpyDeviceToHost, h->stream));
		CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	} else {
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	}
	h->launches += 1;
	return OSC_OK;
}

int osc_get_status(osc_handle* h, uint32_t* flags_out, int mem_kind) {
	ENTER(h);
	if (!flags_out) return fail(h, OSC_ERR_INVALID_ARGUMENT, "null output");
	const size_t bytes = (size_t)h->NR * sizeof(uint32_t);
	if (mem_kind == OSC_MEM_HOST) {
		CUDA_TRY(h, cudaMemcpyAsync(flags_out, h->d_status, bytes, cudaMemcpyDeviceToHost, h->stream));
		CUDA_TRY(h, cudaStreamSynchronize(h->stream));
	} else if (mem_kind == OSC_MEM_DEVICE) {
		CUDA_TRY(h, cudaMemcpyAsync(flags_out, h->d_status, bytes, cudaMemcpyDeviceToDevice, h->stream));
	} else {
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	}
	return OSC_OK;
}

int osc_eval_model(osc_handle* h, int task_id, const osc_link_frame* frame, const double point[3], double* M, double* J,
				   double* x, double* R, double* g, int mem_kind) {
	ENTER(h);
	osc_link_frame f;
	if (task_id >= 0) {
		int rc = check_task(h, task_id, OSC_TASK_MOTION_FORCE);
		if (rc != OSC_OK) return rc;
		const DevMft& t = h->prog.mft[h->tasks[task_id].index];
		f.body = t.body;
		std::memcpy(f.R, t.ctrl_R, sizeof(f.R));
		std::memcpy(f.t, t.ctrl_t, sizeof(f.t));
	} else {
		if (!frame) return fail(h, OSC_ERR_INVALID_ARGUMENT, "frame required when task_id < 0");
		if (frame->body < -1 || frame->body >= h->model.n) return fail(h, OSC_ERR_INVALID_ARGUMENT, "link body index out of range");
		f = *frame;
		if (point) {
			double tt[3];
			mat3_vec_h(frame->R, point, tt);
			for (int k = 0; k < 3; k++) f.t[k] = frame->t[k] + tt[k];
		}
	}
	const int n = h->model.n;
	const size_t NR = (size_t)h->NR;
	double *dM = M, *dJ = J, *dx = x, *dR = R, *dg = g;
	double* scratch = nullptr;
	if (mem_kind == OSC_MEM_HOST) {
		const size_t total = (size_t)(n * n + 6 * n + 3 + 9 + n) * NR;
		CUDA_TRY(h, cudaMalloc((void**)&scratch, total * sizeof(double)));
		dM = scratch;
		dJ = dM + (size_t)n * n * NR;
		dx = dJ + (size_t)6 * n * NR;
		dR = dx + 3 * NR;
		dg = dR + 9 * NR;
	} else if (mem_kind != OSC_MEM_DEVICE) {
		return fail(h, OSC_ERR_INVALID_ARGUMENT, "bad mem_kind");
	}
	cudaError_t e = osc::launch_eval_model(h->prog, f, dM, dJ, dx, dR, dg, h->stream);
	h->launches++;
	if (e == cudaSuccess && mem_kind == OSC_MEM_HOST) {
		struct {
			double* dst;
			const double* src;
			size_t comps;
		} cp[5] = {{M, dM, (size_t)n * n}, {J, dJ, (size_t)6 * n}, {x, dx, 3}, {R, dR, 9}, {g, dg, (size_t)n}};
		for (auto& c : cp)
			if (c.dst && e == cudaSuccess)
				e = cudaMemcpyAsync(c.dst, c.src, c.comps * NR * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
		if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
	}
	if (scratch) cudaFree(scratch);
	CUDA_TRY(h, e);
	return OSC_OK;
}

}  // extern "C"
