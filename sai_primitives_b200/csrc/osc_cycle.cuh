// The fused control-cycle kernel: one robot per thread, FP64, no tensor cores.
//
//   kinematics/dynamics -> MotionForceTask model + torque -> JointTask model + torque
//   -> RobotController stacking (previous-torque feed-forward, saturation, gravity)
//
// Reference path being replaced (one launch == these calls for N robots):
//   SaiModel::updateModel                               examples/05-...cpp:143-145
//   RobotController::updateControllerTaskModels         src/RobotController.cpp:68-77
//     MotionForceTask::updateTaskModel                  src/tasks/MotionForceTask.cpp:247-268
//       SingularityHandler::updateTaskModel             src/tasks/SingularityHandler.cpp:75-228
//     JointTask::updateTaskModel                        src/tasks/JointTask.cpp:218-283
//   RobotController::computeControlTorques              src/RobotController.cpp:79-118
//     MotionForceTask::computeTorques                   src/tasks/MotionForceTask.cpp:270-509
//       SingularityHandler::computeTorques              src/tasks/SingularityHandler.cpp:297-309
//     JointTask::computeTorques                         src/tasks/JointTask.cpp:285-356
//
// Algebra (DESIGN.md section 4, validated on the CPU by tests/test_algebra_proto.py):
// with M = L L^T every task Jacobian is whitened, X = L^-1 J^T, so that
// J M^-1 J^T = X^T X and the dynamically consistent null space becomes the orthogonal
// complement of range(X).  A Householder QR of X gives Lambda = (R^T R)^-1 and, through
// its reflectors, an orthonormal basis Q_perp of that complement; a full joint task in
// the null space is then  tau = L Q_perp G^-1 W^T(.)  with  W = L^-T Q_perp, G = W^T W.
// The bounded-inertia variant M_BIE = M + diag(d) is a rank-one update M + h h^T whenever a single
// diagonal entry is clamped (always the case for the Panda: SURVEY.md Appendix D), handled by
// Sherman-Morrison on the factors already at hand; several clamped entries take the general route.
// When the null space is one-dimensional (the flagship: seven joints under a six-dof pure-motion task) the specialised
// kernel needs neither X nor the QR: the null vector n of J_t and the Cholesky factor of G = J_t J_t^T give the task
// torque and the joint task in closed form (RANK1 below, tests/test_rank_one_tail.py).
// No singular value decomposition is needed on this (non-singular) branch: the branch
// decision uses the sound spectral test in osc_math.cuh; robots that fail it are handed to the
// general-path kernel (osc_singular.cuh) through a compacted list.
#pragma once
#include "osc_kindyn.cuh"
#include "osc_launch.h"
#include "osc_pipeline.cuh"
#include "osc_tasks.cuh"

namespace osc {

#ifndef OSC_MIN_BLOCKS
#define OSC_MIN_BLOCKS 1
#endif

// M_BIE = M + diag(d),  d_i = max(thr - M_ii, 0).  Returns the number of clamped entries k; for k == 1 the update is
// the rank-one matrix  delta e e^T  (e = indicator of the clamped entry, delta = sum(d)), which needs no square root.
template <int N>
DEVI int bie_shift(const double (&Mdiag)[N], double thr, double (&d)[N], double& delta) {
	int k = 0;
	delta = 0.0;
#pragma unroll
	for (int j = 0; j < N; j++) {
		const double dj = thr - Mdiag[j];
		d[j] = (dj > 0.0) ? dj : 0.0;
		delta += d[j];
		k += (dj > 0.0) ? 1 : 0;
	}
	return k;
}

// Cholesky of M_BIE re-assembled from M = L L^T (the lower triangle of M is overwritten by its factor):
// general route for two or more clamped entries.
template <int N>
DEVI void bie_cholesky_from_factor(const double (&L)[N][N], const double (&d)[N], double (&Lb)[N][N], double (&invdb)[N]) {
#pragma unroll
	for (int r = 0; r < N; r++)
#pragma unroll
		for (int c = 0; c <= r; c++) {
			double s = 0.0;
#pragma unroll
			for (int k = 0; k <= c; k++) s += L[r][k] * L[c][k];
			Lb[r][c] = (r == c) ? s + d[r] : s;
		}
	cholesky_lower<N>(Lb, invdb);
}

// Dynamic shared memory of the fused kernel, in doubles per thread: the body orientations (9 N) between the forward
// pass and the mass matrix, then the Cholesky factor with its reciprocal diagonal (kSmFactor) followed by the N x R
// reduced Jacobian columns and the gravity vector.
template <int N>
constexpr int kSmFactor = N * (N + 1) / 2 + N;
template <int N, int R, unsigned V>
constexpr int cycle_smem_doubles() {
	constexpr bool SPEC = V & CV_SPEC, MOTION = V & CV_MOTION;
	// rolled kinematics layout (osc_kindyn.cuh); factor and Jacobian columns fit underneath, the staged goals of the
	// motion-force task (30) go behind the Jacobian columns, those of the joint task (6 N) later take their place
	if (SPEC) {
		int d = 15 * N;
		if (MOTION && kSmFactor<N> + N * R + 30 > d) d = kSmFactor<N> + N * R + 30;
		if (kSmFactor<N> + 6 * N > d) d = kSmFactor<N> + 6 * N;
		return d;
	}
	return (9 * N > kSmFactor<N> + N * R + N) ? 9 * N : kSmFactor<N> + N * R + N;
}
static_assert(kSmFactor<8> + 8 * 6 <= 15 * 8 && kSmFactor<8> <= 9 * 8, "rolled layout: the Jacobian columns must not run into live joint data");

template <bool NARROW>
struct IndexType {
	using type = int64_t;
};
template <>
struct IndexType<true> {
	using type = uint32_t;
};

// phase barrier of the kernel body: the specialisation (instruction stream inside the cache, no spills to fence) runs
// without them
#if defined(OSC_TRACE)
#define OSC_LS_K() OSC_LS()
#else
#define OSC_LS_K()      \
	do {                 \
		if constexpr (!SPEC) OSC_LS(); \
	} while (0)
#endif

DEVI void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }


// y = B^T v: the six world-frame components of a task vector reduced to the R coordinates of the task range
// (identity for a full task)
template <int R, bool FULL>
DEVI void reduce_task_vector(const DevMft& t, const double (&v6)[6], double (&y)[R]) {
#pragma unroll
	for (int a = 0; a < R; a++) {
		if constexpr (FULL) {
			y[a] = v6[a < 6 ? a : 0];
		} else {
			double s = 0.0;
#pragma unroll
			for (int k = 0; k < 6; k++) s += t.B[k][a] * v6[k];
			y[a] = s;
		}
	}
}

// One bulk prefetch (cp.async.bulk.prefetch.L2) per state component for the robots of block `blk`: they are contiguous
// in every component row, so thread k asks for row k of the list below -- one instruction per thread instead of one
// prefetch per thread and component.  MG > 0 (per-robot gains): also the first MG rows of the motion-force task's gain block
// and the joint task's 3 N gain rows (at most 2 N + 31 + 4 N + 24 + 3 N = 127 rows for eight joints).  SP (the instantiations
// without MOTION, whose control law reads the per-robot spaces): also the motion-force task's space block when it has one, last,
// so that in the one case with more rows than threads (eight joints and per-robot gains) only some of its rows go unrequested.
template <int N, int R, bool HAS_JT, int MG = 0, bool SP = false>
DEVI void prefetch_block_rows(const OscProgram& P, uint64_t blk) {
	const uint64_t nrl = (uint64_t)P.n_robots;
	const uint64_t b0 = blk * blockDim.x;
	if (b0 >= nrl) return;
	const uint32_t cnt = (uint32_t)((nrl - b0 < (uint64_t)blockDim.x) ? (nrl - b0) : (uint64_t)blockDim.x);
	int k = threadIdx.x;
	const char* row = nullptr;
	uint32_t esz = 8;
	if (k < N) {
		row = (const char*)(P.q + (uint64_t)k * nrl);
	} else if ((k -= N) < N) {
		row = (const char*)(P.dq + (uint64_t)k * nrl);
	} else {
		k -= N;
		if constexpr (R > 0) {
			const DevMft& t = P.mft[0];
			if (k >= 0 && k < 24) row = (const char*)(t.st + (uint64_t)k * nrl);
			else if (k >= 24 && k < 30) row = (const char*)(t.st + (uint64_t)(MC_INT_POS + k - 24) * nrl);
			else if (k == 30) { row = (const char*)(t.ist + (uint64_t)MI_N_TYPES * nrl); esz = 4; }
			k -= 31;
		}
		if constexpr (HAS_JT || R == 0) {
			const DevJt& jt = P.jt[0];
			if (k >= 0 && k < 4 * N) {
				const int grp = k / N, c = k - grp * N;
				const int comp = (grp == 0 ? JC_GOAL_POS : grp == 1 ? JC_GOAL_VEL : grp == 2 ? JC_GOAL_ACC : JC_INT) + c;
				row = (const char*)(jt.st + (uint64_t)comp * nrl);
			}
			if constexpr (MG > 0 || SP) k -= 4 * N;
		}
		if constexpr (MG > 0 && R > 0) {
			if (k >= 0 && k < MG && P.mft[0].gains) row = (const char*)(P.mft[0].gains + (uint64_t)k * nrl);
			k -= MG;
		}
		if constexpr (MG > 0 && HAS_JT) {
			if (k >= 0 && k < 3 * N && P.jt[0].gains) {
				const int grp = k / N, c = k - grp * N;
				row = (const char*)(P.jt[0].gains + (uint64_t)((grp == 0 ? JG_KP : grp == 1 ? JG_KV : JG_KI) + c) * nrl);
			}
			if constexpr (SP) k -= 3 * N;
		}
		if constexpr (SP && R > 0) {
			if (k == 0 && P.mft[0].space_mode) {
				row = (const char*)P.mft[0].space_mode;
				esz = 4;
			} else if (k >= 1 && k <= SP_AXES_COUNT && P.mft[0].space_axes) {
				row = (const char*)(P.mft[0].space_axes + (uint64_t)(k - 1) * nrl);
			}
		}
	}
	if (row) {
		// 16-byte granules strictly inside [first robot, last robot] of the row: nothing outside the caller's buffer is named
		const uint64_t a0 = (uint64_t)(row + b0 * esz);
		const uint64_t a = (a0 + 15) & ~(uint64_t)15;
		const uint64_t end = a0 + (uint64_t)cnt * esz;
		const uint32_t bytes = (end > a) ? (uint32_t)((end - a) & ~(uint64_t)15) : 0u;
		if (bytes) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a), "r"(bytes) : "memory");
	}
}

// Hand-over to the split blending path: the scratch block of list slot `slot` (BlendLayout, osc_blend.cuh) receives the
// state, the pose of the control frame, gravity, the factor of M and the Jacobian columns staged in shared memory (their Gram
// matrix did not survive the non-singularity test: the classification kernel forms it again).  Only lanes that hand a robot
// over get here.
template <int N>
DEVI void park_for_blend(const OscProgram& P, int slot, int64_t i, const double (&q)[N], const double x[3], const double Rc[9], const double (&Mdiag)[N],
						 const double (&grav)[N], const SmTri<N, kCycleBlock>& Ls, const double* Js) {
	using BL = BlendLayout<N>;
	const int64_t cap = P.blend_cap, NR = P.n_robots;
	gdouble* S = P.blend_scratch + slot;
	constexpr int sms = kCycleBlock;
#pragma unroll
	for (int j = 0; j < N; j++) {
		S[(int64_t)(BL::Q + j) * cap] = q[j];
		S[(int64_t)(BL::DQ + j) * cap] = P.dq[(int64_t)j * NR + i];
		S[(int64_t)(BL::MDIAG + j) * cap] = Mdiag[j];
		S[(int64_t)(BL::GRAV + j) * cap] = grav[j];
		S[(int64_t)(BL::INVD + j) * cap] = Ls.invd(j);
#pragma unroll
		for (int c = 0; c <= j; c++) S[(int64_t)(BL::LL + j * (j + 1) / 2 + c) * cap] = Ls.L(j, c);
#pragma unroll
		for (int a = 0; a < 6; a++) S[(int64_t)(BL::JT0 + j * 6 + a) * cap] = Js[(size_t)(j * 6 + a) * sms];
	}
#pragma unroll
	for (int k = 0; k < 3; k++) S[(int64_t)(BL::X + k) * cap] = x[k];
#pragma unroll
	for (int k = 0; k < 9; k++) S[(int64_t)(BL::RC + k) * cap] = Rc[k];
}

// Signature <N, R, HAS_JT>:  R = rank of a leading MotionForceTask (0: none), HAS_JT = a full JointTask closes the hierarchy.
// V: the flag word (CV_* bits, osc_launch.h, which also lists the instantiated words and their legal combinations).
// Dynamic shared memory: cycle_smem_doubles<N, R, V>() doubles per thread,
// element e of thread t at  sm[e * blockDim.x + t]  (conflict-free, 8-byte interleave).
//
// FULL: the motion-force task controls all six directions (B = I).
// SPEC is the specialisation for the default configuration of the flagship hierarchy (cycle_spec_eligible()
// in osc_launch.h states the conditions: every joint revolute about its local z axis, pure motion control, no
// velocity saturation, FULL or BOUNDED_INERTIA decoupling).  Everything those conditions rule out is
// compiled out, which brings the kernel from 223 KB to under 128 KB of code: beyond that size the instruction stream
// no longer stays in the SM's instruction cache between blocks and every 256-byte line costs a round trip to L2
// (profiles/r01_ifetch.md).  Robots whose bounded-inertia update has rank two or more leave through the general path.
// GRAV (with SPEC only): gravity compensation compiled in; the non-specialised instantiations test the run-time flag.
// MOTION (with SPEC only): the motion-force task is a full task under pure motion control, so only the two PID
// laws are compiled in and its goals are staged through shared memory.  SPEC without MOTION keeps the general control
// law (partial tasks, force / moment spaces, closed loops, POPC) on top of the same rolled kinematics.
// PARK (full six-dof task only): hand-overs also leave kinematics and dynamics in the scratch block of the split blending path
// (osc_blend.cuh); a separate instantiation, because compiled into the kernel of the headline it costs 6 registers and 0.7 %.
// PRG (with SPEC, or for a JointTask alone): a task of the launch carries per-robot PID gains (osc_set_gains), read from its gain block in global
// memory (a task without a block: its parameters); the instantiations without it read the broadcast parameters (SPEC) or test
// the block pointer at run time (the others).
template <int N, int R, bool HAS_JT, unsigned V>
__global__ void __launch_bounds__(kCycleBlock, OSC_MIN_BLOCKS) osc_cycle_kernel(const __grid_constant__ OscProgram P) {
	constexpr bool FULL = V & CV_FULL, SPEC = V & CV_SPEC, GRAV = V & CV_GRAV, MOTION = V & CV_MOTION, PARK = V & CV_PARK, PRG = V & CV_PRG;
	extern __shared__ double sm[];
	// Programmatic dependent launch on both sides: the general-path kernel of this cycle may be scheduled into whatever
	// the last wave leaves free (it waits for this grid to complete before it reads the hand-over list), and this kernel
	// may itself have been scheduled while the general-path kernel of the previous cycle was still running: it waits for
	// it below, after the prefetches.
	asm volatile("griddepcontrol.launch_dependents;");
#if defined(OSC_TRACE)
	if (threadIdx.x == 0) s_trace_k = 0;
	OSC_LS_K();
#endif
	// element index type of the state blocks: 32 bits in the specialisation (the launcher checks the sizes)
	using IDX = typename IndexType<SPEC>::type;
	const IDX NR = (IDX)P.n_robots;
	const IDX i_raw = (IDX)blockIdx.x * blockDim.x + threadIdx.x;

	// Every thread of the block walks the whole kernel (the phase barriers below need all of them): threads past the
	// end of the batch and robots handed to the general path keep computing on valid data but touch no state.
	bool alive = i_raw < NR;
	const IDX i = alive ? i_raw : NR - 1;
	const DevModel& mdl = P.model;
	double* smt = sm + threadIdx.x;
	constexpr int sms = kCycleBlock;  // the launcher always uses kCycleBlock threads per block

	// Warm L2 with this robot's inputs and task state (goals, integrators) before anything else: a first-touch DRAM miss
	// in the middle of the control law cannot be hidden with two warps per scheduler, and a block that was scheduled
	// while the previous kernel of the stream is still running (programmatic dependent launch) uses the wait for it.
	// Prefetches are safe ahead of griddepcontrol.wait: they only move lines into L2, which stays coherent.
	// where the control laws read the gains: a JointTask alone (R = 0) has a per-robot instantiation like the specialised kernels,
	// the other non-specialised instantiations test the block pointer at run time
	constexpr int G = PRG ? GAINS_ROBOT : (SPEC || R == 0) ? GAINS_BCAST : GAINS_ANY;
	// task tail of a one-dimensional null space (the flagship: a 7-joint robot under a six-dof pure-motion task) built from
	// the null vector of J_t instead of a Householder QR.  Every other signature keeps the QR route; in the specialisation
	// without MOTION (general control law) the new tail would push the kernel, already at 255 registers, into more spills.
	constexpr bool RANK1 = SPEC && MOTION && FULL && HAS_JT && R > 1 && N - R == 1;
#ifndef OSC_NO_PREFETCH
	if constexpr (PRG)
		prefetch_block_rows<N, R, HAS_JT, MOTION ? MG_KP_FORCE : GAIN_COUNT, !MOTION>(P, blockIdx.x);
	else
		prefetch_block_rows<N, R, HAS_JT, 0, !MOTION>(P, blockIdx.x);
#endif
	grid_dependency_wait(P);
	stamp_block(P, 0);
	if (!P.block_epoch && i_raw == 0 && P.sing_count) P.sing_count[P.sing_parity ^ 1] = 0;
	bool handed_over = false;
	double q[N];
#pragma unroll
	for (int j = 0; j < N; j++) q[j] = P.q[(IDX)j * NR + i];
	KinDynS<N> kd;
	if constexpr (SPEC) {
#if defined(OSC_TRACE)
		OSC_LS_K();
#endif
		forward_kinematics_rolled<N>(mdl, q, smt, sms);
#if defined(OSC_TRACE)
		OSC_LS_K();
#endif
	} else
		forward_kinematics_s<N, false>(mdl, q, kd, smt, sms);

	double tau[N];
	double gvec_out[N];	 // gravity vector of the specialisation (GRAV), added after the saturation
#pragma unroll
	for (int j = 0; j < N; j++) tau[j] = gvec_out[j] = 0.0;
	uint32_t status = 0;

	if constexpr (R == 0) {
		// ---- a full JointTask alone: N_prec = I, range = I:  tau = M qdd_d + M_mod t   (JointTask.cpp:348-355)
		if (!SPEC && P.gravity_comp)
			mass_matrix_s<N, true, SPEC>(mdl, kd, smt, sms);
		else
			mass_matrix_s<N, false, SPEC>(mdl, kd, smt, sms);
		const DevJt& t = P.jt[0];
		const osc_joint_params& p = t.p;
		double pid[N], acc[N];
#pragma unroll
		for (int j = 0; j < N; j++) pid[j] = acc[j] = 0.0;
		wait_previous_cycle(P);	 // first access to task state
		if (alive) {
			double dq[N];
#pragma unroll
			for (int j = 0; j < N; j++) dq[j] = P.dq[(IDX)j * NR + i];
			joint_control_law<N, N, false, IDX, G>(t, NR, i, q, dq, pid, acc);
		}
#pragma unroll
		for (int r = 0; r < N; r++) {
			double s = 0.0;
#pragma unroll
			for (int c = 0; c < N; c++) {
				const double m = (c <= r) ? kd.M[r][c] : kd.M[c][r];
				double mod;
				if (p.dynamic_decoupling_type == OSC_FULL_DYNAMIC_DECOUPLING)
					mod = m;
				else if (p.dynamic_decoupling_type == OSC_BOUNDED_INERTIA_ESTIMATES)
					mod = (r == c && m < p.bie_threshold) ? p.bie_threshold : m;
				else
					mod = (r == c) ? 1.0 : 0.0;
				s += m * acc[c] + mod * pid[c];
			}
			tau[r] += s;
		}
	} else {
		const DevMft& t = P.mft[0];
		const osc_mft_params& p = t.p;
		double x[3], Rc[9];
		if constexpr (SPEC)
			frame_pose_rolled<N>(t.body, t.ctrl_R, t.ctrl_t, x, Rc, smt, sms);
		else
			frame_pose_s<N>(kd, t.body, t.ctrl_R, t.ctrl_t, x, Rc, smt, sms);

		// ---- dynamics first: M (composite rigid bodies), M = L L^T in place.  The body orientations in shared memory
		// are dead after this, the factor takes their place; only diag(M) is kept for the bounded-inertia variant.
		double dqr[N];	// joint velocities for the Jacobian pass below, requested early
		if constexpr (SPEC) {
			mass_matrix_rolled<N, GRAV>(mdl, smt, sms);
			if constexpr (GRAV) {
#pragma unroll
				for (int j = 0; j < N; j++) gvec_out[j] = smt[(size_t)(9 * j + 8) * sms];
			}
#if defined(OSC_TRACE)
			OSC_LS_K();
#endif
#pragma unroll
			for (int j = 0; j < N; j++) dqr[j] = P.dq[(IDX)j * NR + i];
#pragma unroll
			for (int r = 0; r < N; r++)
#pragma unroll
				for (int c = 0; c <= r; c++) kd.M[r][c] = smt[(size_t)(9 * r + c) * sms];
		} else if (P.gravity_comp) {
			mass_matrix_s<N, true, false>(mdl, kd, smt, sms);
#pragma unroll
			for (int j = 0; j < N; j++) smt[(size_t)(kSmFactor<N> + N * R + j) * sms] = kd.g[j];
		} else {
			mass_matrix_s<N, false, false>(mdl, kd, smt, sms);
		}
		double Mdiag[N];
		SmTri<N, kCycleBlock> Ls{smt};
		{
			double invd[N];
#pragma unroll
			for (int j = 0; j < N; j++) Mdiag[j] = kd.M[j][j];
			cholesky_lower<N>(kd.M, invd);
			Ls.store(kd.M, invd);
		}
		OSC_LS_K();

		// ---- one pass over the Jacobian columns: G = J_t J_t^T, the task velocity J0 dq, and the reduced columns
		// staged in shared memory behind the factor (the joint axes and origins are dead after this loop)
		double* Js = smt + (size_t)kSmFactor<N> * sms;
		double v[3] = {0, 0, 0}, w[3] = {0, 0, 0};
		double Cg[R][R], invc[R];  // RANK1: G = J_t J_t^T = C C^T
		{
			double G[R][R];
#pragma unroll
			for (int a = 0; a < R; a++)
#pragma unroll
				for (int b = 0; b < R; b++) G[a][b] = 0.0;
			if constexpr (SPEC) {
				// rolled: axis, origin and velocity of joint j from shared memory
				static_assert(!MOTION || (R == 6 && FULL), "pure motion control is specialised for the full six-dof task");
				const int nb = t.body + 1;	// joints beyond the task body do not move it
#pragma unroll 1
				for (int j = 0; j < N; j++) {
					const double* ap = smt + (size_t)(kSmAxes<N> + 6 * j) * sms;
					const double a3[3] = {ap[0], ap[1 * sms], ap[2 * sms]};
					const double d[3] = {x[0] - ap[3 * sms], x[1] - ap[4 * sms], x[2] - ap[5 * sms]};
					const double mk = (j < nb) ? 1.0 : 0.0;
					const double dqj = dqr[0];	// rotate the register file: no run-time register index
#pragma unroll
					for (int k = 0; k + 1 < N; k++) dqr[k] = dqr[k + 1];
					double c6[6], cr[R];
					cross3(a3, d, c6);
					c6[0] *= mk;
					c6[1] *= mk;
					c6[2] *= mk;
					c6[3] = a3[0] * mk;
					c6[4] = a3[1] * mk;
					c6[5] = a3[2] * mk;
#pragma unroll
					for (int k = 0; k < 3; k++) {
						v[k] += c6[k] * dqj;
						w[k] += c6[3 + k] * dqj;
					}
					reduce_task_vector<R, FULL>(t, c6, cr);
					double* Jj = Js + (size_t)(j * R) * sms;
#pragma unroll
					for (int a = 0; a < R; a++) Jj[a * sms] = cr[a];
#pragma unroll
					for (int a = 0; a < R; a++)
#pragma unroll
						for (int b = 0; b <= a; b++) G[a][b] += cr[a] * cr[b];
				}
			}
			wait_previous_cycle(P);	 // first access to task state (nothing above reads anything a control cycle writes)
			if constexpr (MOTION) mft_stage_goals(t, NR, i, smt + (size_t)(kSmFactor<N> + N * R) * sms, sms);
#pragma unroll
			for (int j = 0; j < (SPEC ? 0 : N); j++) {
				double c6[6], cr[R];
				jacobian_column<N, false>(mdl, kd, t.body, x, j, c6);
				const double dqj = P.dq[(IDX)j * NR + i];
#pragma unroll
				for (int k = 0; k < 3; k++) {
					v[k] += c6[k] * dqj;
					w[k] += c6[3 + k] * dqj;
				}
				reduce_task_vector<R, FULL>(t, c6, cr);
#pragma unroll
				for (int a = 0; a < R; a++) Js[(j * R + a) * sms] = cr[a];
#pragma unroll
				for (int a = 0; a < R; a++)
#pragma unroll
					for (int b = 0; b <= a; b++) G[a][b] += cr[a] * cr[b];
			}
			OSC_LS_K();
#pragma unroll
			for (int a = 0; a < R; a++)
#pragma unroll
				for (int b = a + 1; b < R; b++) G[a][b] = G[b][a];
			// Branch decision of SingularityHandler::updateTaskModel (:83-105), taken before any task state is touched:
			// robots that are not provably non-singular are appended (warp-aggregated) to the list of the general-path
			// kernel and leave this kernel.
			bool leave;
			if constexpr (RANK1)
				leave = !sound_nonsingular_gram_factor<R>(G, p.s_max, p.s_abs_tol, Cg, invc);
			else
				leave = !sound_nonsingular_gram<R>(G, p.s_max, p.s_abs_tol);
			if constexpr (SPEC) {
				// the specialisation carries the rank-zero and rank-one bounded-inertia updates only
				double hh[N], dd;
				if (p.dynamic_decoupling_type == OSC_BOUNDED_INERTIA_ESTIMATES && bie_shift<N>(Mdiag, p.bie_threshold, hh, dd) >= 2) leave = true;
				if constexpr (HAS_JT) {
					const osc_joint_params& jp0 = P.jt[0].p;
					if (jp0.dynamic_decoupling_type == OSC_BOUNDED_INERTIA_ESTIMATES && bie_shift<N>(Mdiag, jp0.bie_threshold, hh, dd) >= 2)
						leave = true;
				}
			}
			const bool flagged = alive && leave;
			const unsigned m = __ballot_sync(0xffffffffu, flagged);
			if (flagged) {
				const int lane = threadIdx.x & 31;
				const int leader = __ffs(m) - 1;
				int base = 0;
				if (lane == leader) {
					// the list of this parity was last read by the general-path kernel two cycles ago; the scratch block of the split
					// blending path is not double-buffered: the previous cycle's general path must be through with it
					if (P.general_done) {
						const uint32_t need = P.epoch - ((PARK && P.blend_split_on) ? 1u : 2u);
						while ((int32_t)(ld_acquire_u32(P.general_done) - need) < 0) __nanosleep(256);
					}
					base = atomicAdd(&P.sing_count[P.sing_parity], __popc(m));
				}
				base = __shfl_sync(m, base, leader);
				const int slot = base + __popc(m & ((1u << lane) - 1u));
				P.sing_list[slot] = (int32_t)i;
				if constexpr (PARK) {
					// split blending path (osc_blend.cuh): leave what is already known about this robot in its scratch block
					if (P.blend_split_on) {
						double gv[N];
#pragma unroll
						for (int j = 0; j < N; j++) {
							if constexpr (SPEC)
								gv[j] = gvec_out[j];
							else
								gv[j] = P.gravity_comp ? smt[(size_t)(kSmFactor<N> + N * R + j) * sms] : 0.0;
						}
						park_for_blend<N>(P, slot, (int64_t)i, q, x, Rc, Mdiag, gv, Ls, Js);
					}
				}
				alive = false;	// the general-path kernel owns this robot from here on
				handed_over = true;
			}
		}
		// classifySingularity with an empty singular range clears the handler memory (:239-245); only robots that
		// were singular at the previous update have anything to clear
		if (alive && P.update_models && t.ist[(IDX)MI_N_TYPES * NR + i] != 0) {
			t.ist[(IDX)MI_N_TYPES * NR + i] = 0;
			t.ist[(IDX)MI_T1_COUNTER * NR + i] = 0;
			t.ist[(IDX)MI_T2_COUNTER * NR + i] = 0;
			t.ist[(IDX)MI_HIST_HEAD * NR + i] = 0;
			t.ist[(IDX)MI_HIST_SIZE * NR + i] = 0;
		}

		OSC_LS_K();
		double yf[R], yF[R];
		bool has_F;
		{
			double fstar[6] = {0, 0, 0, 0, 0, 0}, F[6] = {0, 0, 0, 0, 0, 0};
			has_F = true;
			if (alive)
				has_F = mft_control_law<MOTION, IDX, G>(t, NR, i, x, Rc, v, w, P.write_observers != 0, fstar, F, status,
												MOTION ? smt + (size_t)(kSmFactor<N> + N * R) * sms : nullptr, sms);
			reduce_task_vector<R, FULL>(t, fstar, yf);
			reduce_task_vector<R, FULL>(t, F, yF);
		}
		OSC_LS_K();

		if constexpr (RANK1) {
			// ---- one-dimensional null space (N - R = 1, DESIGN.md section 4).  With G = J_t J_t^T = C C^T (factored with
			// the branch test), column k of the projector I - J_t^T G^-1 J_t is parallel to the null vector n of J_t; the
			// column with the largest diagonal entry 1 - |C^-1 J_k|^2 (at least 1/N) is taken.  The scale of n is free.
			double ub[R], pbest = 0.0;
			int kb = 0;
#pragma unroll
			for (int k = 0; k < N; k++) {
				double u[R];
#pragma unroll
				for (int a = 0; a < R; a++) u[a] = Js[(k * R + a) * sms];
				solve_lower<R>(Cg, invc, u);
				double pk = 1.0;
#pragma unroll
				for (int a = 0; a < R; a++) pk -= u[a] * u[a];
				const bool better = (k == 0) || pk > pbest;
				pbest = better ? pk : pbest;
				kb = better ? k : kb;
#pragma unroll
				for (int a = 0; a < R; a++) ub[a] = better ? u[a] : ub[a];
			}
			solve_lower_t<R>(Cg, invc, ub);	 // G^-1 J_kb
			// v = J_t^T G^-1 f, the minimum-norm solution of J_t v = f: no component along n (impedance decoupling: J_t^T f)
			const int dec = p.dynamic_decoupling_type;
			if (dec != OSC_IMPEDANCE) solve_spd<R>(Cg, invc, yf);
			double nv[N], tv[N];
#pragma unroll
			for (int j = 0; j < N; j++) {
				double sn = (j == kb) ? 1.0 : 0.0, sv = 0.0, sF = 0.0;
#pragma unroll
				for (int a = 0; a < R; a++) {
					const double c = Js[(j * R + a) * sms];
					sn -= c * ub[a];
					sv += c * yf[a];
					sF += c * yF[a];
				}
				nv[j] = sn;
				tv[j] = sv;
				if (has_F) tau[j] += sF;
			}
			// the Jacobian columns are dead: their slots receive the joint task's goals, integrator and q, dq, requested now
			// and read after the task torque below
			joint_stage_goals<N>(P.jt[0], P.q, P.dq, NR, i, smt + (size_t)kSmFactor<N> * sms, sms);
			OSC_LS_K();
			// tau_task = J_t^T Lambda_b f = M_b v - M_b n (n . M_b v) / (n . M_b n),  M_b = M + diag(d): the two projectors
			// M_b^-1 J_t^T Lambda_b J_t and n (n^T M_b n)^-1 n^T M_b are M_b-orthogonal and add up to I
			double Mn[N], Mv[N], dm[N], dsum;
			Ls.mul_llt(nv, Mn);
			Ls.mul_llt(tv, Mv);
			if (dec == OSC_BOUNDED_INERTIA_ESTIMATES)
				bie_shift<N>(Mdiag, p.bie_threshold, dm, dsum);
			else {
#pragma unroll
				for (int j = 0; j < N; j++) dm[j] = 0.0;
			}
			double Mbn[N], nMbv = 0.0, nMbn = 0.0;
#pragma unroll
			for (int j = 0; j < N; j++) {
				Mv[j] += dm[j] * tv[j];
				Mbn[j] = Mn[j] + dm[j] * nv[j];
				nMbv += nv[j] * Mv[j];
				nMbn += nv[j] * Mbn[j];
			}
			const double cf = div_nz(nMbv, nMbn);
#pragma unroll
			for (int j = 0; j < N; j++) tau[j] += (dec == OSC_IMPEDANCE) ? tv[j] : Mv[j] - Mbn[j] * cf;
			OSC_LS_K();

			// ---- joint task in the null space, s = n . M n, m = M^-1 n:
			//   tau_jt = M n [ (n . qdd_d - m . tau_task) / (n . n) + (n . pid) / ((n . n) h) ]
			// h = 1 under full decoupling; with one clamped entry e of M_b = M + delta e e^T, h = 1 - delta n_e^2 / (s (1 + delta mu)),
			// mu = |L^-1 e|^2; impedance decoupling: (n . pid) / s
			const DevJt& jt = P.jt[0];
			const osc_joint_params& jp = jt.p;
			double m[N];
#pragma unroll
			for (int j = 0; j < N; j++) m[j] = nv[j];
			Ls.solve_lower(m);
			Ls.solve_lower_t(m);
			double pid[N], acc[N];
#pragma unroll
			for (int j = 0; j < N; j++) pid[j] = acc[j] = 0.0;
			if (alive) joint_control_law_staged<N, IDX, G>(jt, NR, i, smt + (size_t)kSmFactor<N> * sms, sms, pid, acc);
			double nn = 0.0, s = 0.0, mm = 0.0, na = 0.0, np = 0.0, mt = 0.0;
#pragma unroll
			for (int j = 0; j < N; j++) {
				nn += nv[j] * nv[j];
				s += nv[j] * Mn[j];
				mm += Mn[j] * Mn[j];
				na += nv[j] * acc[j];
				np += nv[j] * pid[j];
				mt += m[j] * tau[j];
			}
			// ||N_prec||_F^2 = (n . n)(M n . M n) / s^2 must stay < 1e6 for the reference's 1e-3 range tolerance
			if (!(nn * mm < 1.0e6 * (s * s))) status |= OSC_STATUS_UNHANDLED;
			const double inn = rcp_nz(nn);
			double zp = inn;
			const int jdec = jp.dynamic_decoupling_type;
			if (jdec == OSC_IMPEDANCE)
				zp = rcp_nz(s);
			else if (jdec == OSC_BOUNDED_INERTIA_ESTIMATES) {
				double hj[N], dj;
				if (bie_shift<N>(Mdiag, jp.bie_threshold, hj, dj) == 1) {
					double g[N], ne = 0.0, mu = 0.0;
#pragma unroll
					for (int j = 0; j < N; j++) {
						g[j] = (hj[j] > 0.0) ? 1.0 : 0.0;
						ne += (hj[j] > 0.0) ? nv[j] : 0.0;
					}
					Ls.solve_lower(g);
#pragma unroll
					for (int j = 0; j < N; j++) mu += g[j] * g[j];
					zp = div_nz(inn, 1.0 - dj * ne * ne * rcp_nz(s * (1.0 + dj * mu)));
				}
			}
			const double zc = (na - (P.use_prev_torques ? mt : 0.0)) * inn + np * zp;
#pragma unroll
			for (int j = 0; j < N; j++) tau[j] += Mn[j] * zc;
		} else {
			// ---- X = L^-1 J_t^T row by row (row r needs column r of J only), operands from shared memory
			double X[N][R];
	#pragma unroll
			for (int r = 0; r < N; r++) {
				double cr[R];
	#pragma unroll
				for (int a = 0; a < R; a++) cr[a] = Js[(r * R + a) * sms];
	#pragma unroll
				for (int k = 0; k < r; k++) {
					const double l = Ls.L(r, k);
	#pragma unroll
					for (int a = 0; a < R; a++) cr[a] -= l * X[k][a];
				}
				const double inv = Ls.invd(r);
	#pragma unroll
				for (int a = 0; a < R; a++) X[r][a] = cr[a] * inv;
			}
			// the Jacobian columns are dead: their slots receive the joint task's goals, integrator and q, dq, requested now
			// and read after the factorisation below
			if constexpr (SPEC && HAS_JT) joint_stage_goals<N>(P.jt[0], P.q, P.dq, NR, i, smt + (size_t)kSmFactor<N> * sms, sms);
			OSC_LS_K();
			// bounded inertia estimates: M_BIE = M + diag(d); with one clamped entry: M + delta e e^T,
			// g = L^-1 e, mu = g.g, z = J M^-1 e = X^T g
			const int dec = p.dynamic_decoupling_type;
			int kclamp = 0;
			double z[R], mu = 0.0, delta = 0.0;
			double h[N];
			if (dec == OSC_BOUNDED_INERTIA_ESTIMATES) {
				kclamp = bie_shift<N>(Mdiag, p.bie_threshold, h, delta);
				if (kclamp == 1) {
					double g[N];
	#pragma unroll
					for (int j = 0; j < N; j++) g[j] = (h[j] > 0.0) ? 1.0 : 0.0;
					Ls.solve_lower(g);
	#pragma unroll
					for (int j = 0; j < N; j++) mu += g[j] * g[j];
	#pragma unroll
					for (int a = 0; a < R; a++) {
						double s = 0.0;
	#pragma unroll
						for (int j = 0; j < N; j++) s += X[j][a] * g[j];
						z[a] = s;
					}
				}
			}
			OSC_LS_K();
			double vhead[R], beta[R], rinv[R];
			householder_qr<N, R, 0>(X, vhead, beta, rinv);
			OSC_LS_K();

			if (dec == OSC_FULL_DYNAMIC_DECOUPLING || (dec == OSC_BOUNDED_INERTIA_ESTIMATES && kclamp == 0)) {
				solve_rtr<N, R, 0>(X, rinv, yf);
			} else if (dec == OSC_BOUNDED_INERTIA_ESTIMATES && kclamp == 1) {
				// (A - delta z z^T / (1 + delta mu))^-1 y = A^-1 y + (A^-1 z) (z . A^-1 y) delta / ((1 + delta mu) - delta z . A^-1 z)
				double sz[R];
	#pragma unroll
				for (int a = 0; a < R; a++) sz[a] = z[a];
				solve_rtr<N, R, 0>(X, rinv, sz);
				solve_rtr<N, R, 0>(X, rinv, yf);
				double zs = 0.0, zt = 0.0;
	#pragma unroll
				for (int a = 0; a < R; a++) {
					zs += z[a] * sz[a];
					zt += z[a] * yf[a];
				}
				const double f = delta * zt / ((1.0 + delta * mu) - delta * zs);
	#pragma unroll
				for (int a = 0; a < R; a++) yf[a] += sz[a] * f;
			}
			else if (!SPEC && dec == OSC_BOUNDED_INERTIA_ESTIMATES) {
				// general route (two or more clamped entries): A_b = W^T W, W = L_b^-1 J_t^T with J_t^T = L Q [R; 0]
				double Lf[N][N], Lb[N][N], invdb[N];
	#pragma unroll
				for (int r = 0; r < N; r++)
	#pragma unroll
					for (int c = 0; c <= r; c++) Lf[r][c] = Ls.L(r, c);
				bie_cholesky_from_factor<N>(Lf, h, Lb, invdb);
				double Wb[N][R];
	#pragma unroll
				for (int a = 0; a < R; a++) {
					double e[N], col[N];
	#pragma unroll
					for (int j = 0; j < N; j++) e[j] = (j <= a) ? X[j][a] : 0.0;  // column a of [R; 0]
					apply_q<N, R, 0>(X, vhead, beta, e);
					mul_lower<N>(Lf, e, col);
					solve_lower<N>(Lb, invdb, col);
	#pragma unroll
					for (int j = 0; j < N; j++) Wb[j][a] = col[j];
				}
				double Ab[R][R], invda[R];
	#pragma unroll
				for (int a = 0; a < R; a++)
	#pragma unroll
					for (int b = 0; b <= a; b++) {
						double s = 0.0;
	#pragma unroll
						for (int j = 0; j < N; j++) s += Wb[j][a] * Wb[j][b];
						Ab[a][b] = s;
					}
				cholesky_lower<R>(Ab, invda);
				solve_spd<R>(Ab, invda, yf);
			}  // IMPEDANCE: Lambda_modified = I
			OSC_LS_K();
			// tau_task = J_t^T y = L Q [R y; 0]
			{
				if (has_F) {
	#pragma unroll
					for (int a = 0; a < R; a++) yf[a] += yF[a];
				}
				double e[N], lt[N];
	#pragma unroll
				for (int r = 0; r < N; r++) {
					double s = 0.0;
					if (r < R) {
	#pragma unroll
						for (int a = r; a < R; a++) s += X[r][a] * yf[a];
					}
					e[r] = s;
				}
				apply_q<N, R, 0>(X, vhead, beta, e);
				Ls.mul_lower(e, lt);
	#pragma unroll
				for (int j = 0; j < N; j++) tau[j] += lt[j];
			}

			if constexpr (HAS_JT) {
				const DevJt& jt = P.jt[0];
				const osc_joint_params& jp = jt.p;
				constexpr int Mn = N - R;  // dimension of the remaining null space
				if constexpr (Mn == 0) {
					status |= OSC_STATUS_ZERO_RANGE;  // JointTask.cpp:234-239, 302-306
				} else {
					double pid[N], acc[N];
	#pragma unroll
					for (int j = 0; j < N; j++) pid[j] = acc[j] = 0.0;
					if constexpr (SPEC) {
						if (alive) joint_control_law_staged<N, IDX, G>(jt, NR, i, smt + (size_t)kSmFactor<N> * sms, sms, pid, acc);
					} else if (alive) {
						double qj[N], dqj[N];  // re-read (L2 hot) rather than kept live across the task above
	#pragma unroll
						for (int j = 0; j < N; j++) {
							qj[j] = P.q[(IDX)j * NR + i];
							dqj[j] = P.dq[(IDX)j * NR + i];
						}
						joint_control_law<N, N, SPEC>(jt, NR, i, qj, dqj, pid, acc);
					}
			OSC_LS_K();
					// Q_perp = H_1..H_R [0; I],  W = L^-T Q_perp,  K = L Q_perp
					double Qp[N][Mn], W[N][Mn], K[N][Mn];
	#pragma unroll
					for (int a = 0; a < Mn; a++) {
						double e[N];
	#pragma unroll
						for (int j = 0; j < N; j++) e[j] = (j == R + a) ? 1.0 : 0.0;
						apply_q<N, R, 0>(X, vhead, beta, e);
						double k[N];
						Ls.mul_lower(e, k);
	#pragma unroll
						for (int j = 0; j < N; j++) Qp[j][a] = e[j];
						Ls.solve_lower_t(e);
	#pragma unroll
						for (int j = 0; j < N; j++) {
							W[j][a] = e[j];
							K[j][a] = k[j];
						}
					}
					double G[Mn][Mn], invg[Mn];
					double nrm_chk = 0.0;
	#pragma unroll
					for (int a = 0; a < Mn; a++)
	#pragma unroll
						for (int b = 0; b <= a; b++) {
							double s = 0.0, kk = 0.0;
	#pragma unroll
							for (int j = 0; j < N; j++) {
								s += W[j][a] * W[j][b];
								kk += K[j][a] * K[j][b];
							}
							G[a][b] = s;
							nrm_chk += (a == b) ? s * kk : 2.0 * s * kk;
						}
					// ||N_prec||_F^2 = tr(G K^T K) must stay < 1e6 for the reference's 1e-3 range tolerance
					if (!(nrm_chk < 1.0e6)) status |= OSC_STATUS_UNHANDLED;
					cholesky_lower<Mn>(G, invg);
			OSC_LS_K();
					// u = W^T (qdd_d - M^-1 tau_prec)
					double rhs[N];
					if (P.use_prev_torques) {
	#pragma unroll
						for (int j = 0; j < N; j++) rhs[j] = tau[j];
						Ls.solve_lower(rhs);
						Ls.solve_lower_t(rhs);
	#pragma unroll
						for (int j = 0; j < N; j++) rhs[j] = acc[j] - rhs[j];
					} else {
	#pragma unroll
						for (int j = 0; j < N; j++) rhs[j] = acc[j];
					}
					double z1[Mn], z2[Mn];
	#pragma unroll
					for (int a = 0; a < Mn; a++) {
						double s1 = 0.0, s2 = 0.0;
	#pragma unroll
						for (int j = 0; j < N; j++) {
							s1 += W[j][a] * rhs[j];
							s2 += W[j][a] * pid[j];
						}
						z1[a] = s1;
						z2[a] = s2;
					}
					solve_spd<Mn>(G, invg, z1);
					const int jdec = jp.dynamic_decoupling_type;
					if (jdec == OSC_FULL_DYNAMIC_DECOUPLING) {
						solve_spd<Mn>(G, invg, z2);
					} else if (jdec == OSC_BOUNDED_INERTIA_ESTIMATES) {
						solve_spd<Mn>(G, invg, z2);
						double hj[N], dj = 0.0;
						const int kj = bie_shift<N>(Mdiag, jp.bie_threshold, hj, dj);
						if (kj == 1) {
							// H = K^T M_b^-1 K = I - delta c c^T / (1 + delta mu),  c = Q_perp^T L^-1 e;
							// H^-1 z = z + c (c . z) delta / ((1 + delta mu) - delta c . c)
							double g[N];
	#pragma unroll
							for (int j = 0; j < N; j++) g[j] = (hj[j] > 0.0) ? 1.0 : 0.0;
							Ls.solve_lower(g);
							double muj = 0.0;
	#pragma unroll
							for (int j = 0; j < N; j++) muj += g[j] * g[j];
							double c[Mn], cc = 0.0, cz = 0.0;
	#pragma unroll
							for (int a = 0; a < Mn; a++) {
								double s = 0.0;
	#pragma unroll
								for (int j = 0; j < N; j++) s += Qp[j][a] * g[j];
								c[a] = s;
								cc += s * s;
								cz += s * z2[a];
							}
							const double f = dj * cz / ((1.0 + dj * muj) - dj * cc);
	#pragma unroll
							for (int a = 0; a < Mn; a++) z2[a] += c[a] * f;
						}
						else if (!SPEC && kj >= 2) {
							double Lf[N][N], Lb[N][N], invdb[N];
	#pragma unroll
							for (int r = 0; r < N; r++)
	#pragma unroll
								for (int c = 0; c <= r; c++) Lf[r][c] = Ls.L(r, c);
							bie_cholesky_from_factor<N>(Lf, hj, Lb, invdb);
							double Z[N][Mn];
	#pragma unroll
							for (int a = 0; a < Mn; a++) {
								double col[N];
	#pragma unroll
								for (int j = 0; j < N; j++) col[j] = K[j][a];
								solve_lower<N>(Lb, invdb, col);
	#pragma unroll
								for (int j = 0; j < N; j++) Z[j][a] = col[j];
							}
							double H[Mn][Mn], invh[Mn];
	#pragma unroll
							for (int a = 0; a < Mn; a++)
	#pragma unroll
								for (int b = 0; b <= a; b++) {
									double s = 0.0;
	#pragma unroll
									for (int j = 0; j < N; j++) s += Z[j][a] * Z[j][b];
									H[a][b] = s;
								}
							cholesky_lower<Mn>(H, invh);
							solve_spd<Mn>(H, invh, z2);
						}
					}  // IMPEDANCE: z2 = W^T t
	#pragma unroll
					for (int j = 0; j < N; j++) {
						double s = 0.0;
	#pragma unroll
						for (int a = 0; a < Mn; a++) s += K[j][a] * (z1[a] + z2[a]);
						tau[j] += s;
					}
				}
			}
		}
	}

#if defined(OSC_TRACE)
	OSC_LS_K();
#endif
	// RobotController::computeControlTorques tail (RobotController.cpp:86-116)
	if (P.torque_saturation) {
#pragma unroll
		for (int j = 0; j < N; j++) {
			if (tau[j] > mdl.effort[j])
				tau[j] = mdl.effort[j];
			else if (tau[j] < -mdl.effort[j])
				tau[j] = -mdl.effort[j];
		}
	}
	if constexpr (SPEC && GRAV && R > 0) {
#pragma unroll
		for (int j = 0; j < N; j++) tau[j] += gvec_out[j];
	}
	if (!SPEC && P.gravity_comp) {
#pragma unroll
		for (int j = 0; j < N; j++) {
			if constexpr (R == 0)
				tau[j] += kd.g[j];
			else
				tau[j] += smt[(size_t)(kSmFactor<N> + N * R + j) * sms];
		}
	}
	if (status & OSC_STATUS_UNHANDLED) {
#pragma unroll
		for (int j = 0; j < N; j++) tau[j] = __longlong_as_double(0x7ff8000000000000LL);
	}
	if (alive) {
#pragma unroll
		for (int j = 0; j < N; j++) P.tau[(IDX)j * NR + i] = tau[j];
		P.status[i] = status;
	}
	publish_cycle(P, handed_over);
	stamp_block(P, 1);
}

}  // namespace osc
