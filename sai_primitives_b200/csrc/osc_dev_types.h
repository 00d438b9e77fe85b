// Device-side program description shared by the host layer (osc_capi.cu) and the kernels.
// One OscProgram is passed to every kernel as a __grid_constant__ parameter, so its
// members are served from the constant bank (warp-uniform broadcast reads).
#pragma once
#include <math.h>
#include <stdint.h>

#include "../../include/sai_b200_osc.h"

// element type of the arrays in global memory (inputs, task state, torques): FP64 also in the single-precision
// instantiation of the kernels (gen_fp32.py rewrites `double`, not this)
typedef double gdouble;

// ---- SoA component layout of the per-robot MotionForceTask state block ----
enum MftComp : int {
	MC_GOAL_POS = 0,	  // 3
	MC_GOAL_ORI = 3,	  // 9
	MC_GOAL_LINVEL = 12,  // 3
	MC_GOAL_ANGVEL = 15,  // 3
	MC_GOAL_LINACC = 18,  // 3
	MC_GOAL_ANGACC = 21,  // 3
	MC_GOAL_FORCE = 24,	  // 3
	MC_GOAL_MOMENT = 27,  // 3
	MC_SENSED_F = 30,	  // 3  control point, world axes
	MC_SENSED_M = 33,	  // 3
	MC_SENSED_F_SENSOR = 36,
	MC_SENSED_M_SENSOR = 39,
	MC_INT_POS = 42,
	MC_INT_ORI = 45,
	MC_INT_FORCE = 48,
	MC_INT_MOMENT = 51,
	MC_CUR_POS = 54,	 // 3
	MC_CUR_ORI = 57,	 // 9
	MC_CUR_LINVEL = 66,	 // 3
	MC_CUR_ANGVEL = 69,	 // 3
	MC_UNIT_MASS_FORCE = 72, // 6
	MC_ORI_ERROR = 78,	 // 3
	MC_POPC = 81,		 // 4: PO, E_correction, Rc, sum vcl^2
	MC_Q_PRIOR = 85,	 // OSC_MAX_DOF
	MC_DQ_PRIOR = 93,	 // OSC_MAX_DOF
	MC_TYPE2_DIR = 101,	 // OSC_MAX_DOF
	MC_COUNT = 109
};

// int32 state components of a MotionForceTask
enum MftIntComp : int {
	MI_POPC_COUNTER = 0,
	MI_RING_HEAD = 1,  // index of the oldest sample
	MI_RING_SIZE = 2,
	MI_T1_COUNTER = 3,
	MI_T2_COUNTER = 4,
	MI_HIST_HEAD = 5,
	MI_HIST_SIZE = 6,
	MI_N_TYPES = 7,	   // number of singular directions classified last update
	MI_TYPES = 8,	   // 2 bits per direction
	MI_HIST_BITS = 9,  // 8 words = 256 bits (bit = 1: type-1 entry)
	MI_COUNT = 17
};

enum JtComp : int { JC_GOAL_POS = 0, JC_GOAL_VEL = 8, JC_GOAL_ACC = 16, JC_INT = 24, JC_COUNT = 32 };

// SoA layout of a task's per-robot gain block (osc_set_gains), GAIN_COUNT x N.  A MotionForceTask uses every component, a
// JointTask of dof k the components JG_KP.. JG_KP + k - 1 and the same of JG_KV, JG_KI.
enum GainComp : int {
	MG_KP_POS = 0, MG_KV_POS = 3, MG_KI_POS = 6,  // 3 each
	MG_KP_ORI = 9, MG_KV_ORI = 12, MG_KI_ORI = 15,
	MG_KP_FORCE = 18, MG_KV_FORCE = 19, MG_KI_FORCE = 20,
	MG_KP_MOMENT = 21, MG_KV_MOMENT = 22, MG_KI_MOMENT = 23,
	JG_KP = 0, JG_KV = 8, JG_KI = 16,  // OSC_MAX_DOF each
	GAIN_COUNT = 24
};

// Per-robot force / moment spaces of a MotionForceTask (osc_mft_parametrize_spaces_batched): one mode word per robot
// (bits 0-1 force space dimension, 2-3 moment space dimension, 4 closed-loop force, 5 closed-loop moment) and the
// normalised axes, SoA SP_AXES_COUNT x N (force / motion axis in rows 0-2, moment / rot-motion axis in rows 3-5).
// A word of 0 is pure motion control.
enum SpaceBits : int32_t { SP_FDIM_SHIFT = 0, SP_MDIM_SHIFT = 2, SP_CL_FORCE = 16, SP_CL_MOMENT = 32, SP_AXES_COUNT = 6 };
// host-side OR over the robots of a task (DevMft::space_any)
enum SpaceSummary : int32_t { SPS_FORCE_DIM = 1, SPS_MOMENT_DIM = 2, SPS_CL_FORCE = 4, SPS_CL_MOMENT = 8 };
#if defined(__CUDACC__)
#define OSC_HD __host__ __device__ inline
#else
#define OSC_HD inline
#endif
OSC_HD int32_t space_mode_word(int fdim, int mdim, bool cl_force, bool cl_moment) {
	return (int32_t)((fdim << SP_FDIM_SHIFT) | (mdim << SP_MDIM_SHIFT) | (cl_force ? SP_CL_FORCE : 0) | (cl_moment ? SP_CL_MOMENT : 0));
}
// Sums of squares without fused multiply-adds, so that the host and the kernels normalise an axis and take a reset decision
// bit for bit alike (a broadcast call and a per-robot call with the same values give the same stored axes).
OSC_HD double sq3_rn(double x, double y, double z) {
#if defined(__CUDA_ARCH__)
	return __dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z));
#else
	return x * x + y * y + z * z;
#endif
}
// |axis|, and the normalised axis in u (MotionForceTask.cpp:838, :868)
OSC_HD double space_normalize(const double axis[3], double u[3]) {
	const double nrm = sqrt(sq3_rn(axis[0], axis[1], axis[2]));
	for (int k = 0; k < 3; k++) u[k] = axis[k] / nrm;
	return nrm;
}
// the reset rule of parametrizeForceMotionSpaces / parametrizeMomentRotMotionSpaces (MotionForceTask.cpp:845, :877): the new
// normalised axis a is Eigen's isApprox to the stored axis b, |a - b|^2 <= 1e-24 min(|a|^2, |b|^2) with |a| = 1
OSC_HD bool space_axis_is_approx(const double a[3], const double b[3]) {
	const double d2 = sq3_rn(a[0] - b[0], a[1] - b[1], a[2] - b[2]), b2 = sq3_rn(b[0], b[1], b[2]);
	return d2 <= 1e-24 * (b2 < 1.0 ? b2 : 1.0);
}
// Validation of per-robot values (SpaceCheck bits; SPC_NONZERO feeds the host's summary): a space dimension in 0..3 and, for
// dimension 1 or 2, a finite axis of norm >= 1e-2; a closed-loop flag 0 or 1.
enum SpaceCheck : int32_t { SPC_BAD_DIM = 1, SPC_BAD_AXIS = 2, SPC_BAD_FLAG = 4, SPC_NONZERO = 8 };
OSC_HD int32_t space_check(int32_t dim, double a0, double a1, double a2) {
	if (dim < 0 || dim > 3) return SPC_BAD_DIM;
	if (dim == 0) return 0;
	if (dim == 3) return SPC_NONZERO;
	// x - x is 0 for a finite x and NaN for an infinite or NaN one
	const bool finite = (a0 - a0) == 0.0 && (a1 - a1) == 0.0 && (a2 - a2) == 0.0;
	const double axis[3] = {a0, a1, a2};
	double u[3];
	return (finite && space_normalize(axis, u) >= 1e-2) ? SPC_NONZERO : SPC_BAD_AXIS;
}
OSC_HD int32_t closed_loop_check(int32_t flag) { return flag == 0 ? 0 : flag == 1 ? SPC_NONZERO : SPC_BAD_FLAG; }

#define OSC_HIST_MAX 256

struct DevModel {
	int32_t n;
	int32_t jtype[OSC_MAX_DOF];
	double axis[OSC_MAX_DOF][3];
	double R_fix[OSC_MAX_DOF][9];  // joint 0 has the world<-base transform folded in
	double t_fix[OSC_MAX_DOF][3];
	double mass[OSC_MAX_DOF];
	double com[OSC_MAX_DOF][3];
	double inertia[OSC_MAX_DOF][6];	 // xx xy xz yy yz zz
	double q_lower[OSC_MAX_DOF], q_upper[OSC_MAX_DOF], effort[OSC_MAX_DOF], dq_max[OSC_MAX_DOF];
	double gravity[3];	// world frame
};

// Internal OTG of one task (osc_otg.h / osc_otg_kernels.cuh).  While enabled, the task's goal slots (JC_GOAL_* / MC_GOAL_*)
// hold the DESIRED state the generator produced for this cycle -- the control laws read nothing else -- and the goals the user
// sets live in the generator's own block.
enum OtgJointComp : int { OJ_USER_POS = 0, OJ_USER_VEL = 8, OJ_USER_ACC = 16, OJ_CORE = 24, OJ_CORE_DOUBLES = 226, OJ_COUNT = 250 };
enum OtgCartComp : int { OC_USER = 0 /* 24, same order as MC_GOAL_POS .. MC_GOAL_ANGACC */, OC_CORE = 24, OC_CORE_DOUBLES = 191, OC_COUNT = 215 };
struct DevOtg {
	int32_t enabled;
	int32_t pad;
	double vmax[OSC_MAX_DOF], amax[OSC_MAX_DOF];  // motion-force task: linear x 3, angular x 3
	double* st;		 // OJ_COUNT / OC_COUNT x N
	int32_t* flags;	 // N (otg::OtgFlags)
};

struct DevMft {
	int32_t body;
	int32_t rank, pos_range, ori_range;
	int32_t full;		   // partial-task projection is the identity
	int32_t in_compliant;  // force/motion spaces parametrised in the compliant frame
	int32_t ring_capacity;
	double ctrl_R[9], ctrl_t[3];  // compliant frame expressed in the body frame
	double B[6][6];				  // orthonormal basis of the task range, 6 x rank (columns)
	double Pt[9], Pr[9];		  // translation / rotation selection projectors
	double cs_R[9], cs_t[3];	  // control frame -> sensor frame
	double dt;
	osc_mft_params p;
	double* st;	   // MC_COUNT x N
	int32_t* ist;  // MI_COUNT x N
	double* ring;  // ring_capacity x N (or null)
	double* gains;	// per-robot PID gains, GAIN_COUNT x N (osc_set_gains); null: every robot uses those of p
	// per-robot spaces and closed-loop flags (SpaceBits); null: every robot uses those of p
	int32_t* space_mode;  // N
	double* space_axes;	  // SP_AXES_COUNT x N
	int32_t space_any;	  // SpaceSummary over the robots, kept by the host while space_mode is set
	DevOtg otg;
};

struct DevJt {
	int32_t k;
	int32_t full;  // selection is the identity
	double S[OSC_MAX_DOF][OSC_MAX_DOF];
	double dt;
	osc_joint_params p;
	double* st;	 // JC_COUNT x N
	double* gains;	// per-robot PID gains, GAIN_COUNT x N (osc_set_gains); null: every robot uses those of p
	DevOtg otg;
};

// JointLimitAvoidanceTask parameters (JointLimitAvoidanceTask.h:26-35; the reference has no setters for them)
struct DevJla {
	double kv;
	double position_z1_to_limit, position_z2_to_limit;
	double velocity_z1_to_limit, velocity_z2_to_limit;
	double max_torque_ratio_pos_limit, max_torque_ratio_vel_limit;
};

struct DevTask {
	int32_t type;  // osc_task_type
	int32_t index; // index into mft[] / jt[]
};

// scratch block of the split blending path (osc_blend.cuh): doubles per list slot, and where each quantity sits
constexpr int blend_scratch_doubles(int n) { return 11 * n + n * (n + 1) / 2 + 55; }
template <int N>
struct BlendLayout {
	// written by the fused kernel when it hands the robot over (park_for_blend, osc_cycle.cuh): state, pose, gravity, M = L L^T
	// and the Jacobian (transposed);  written by the classification kernel: U, SIG, ALPHA
	static constexpr int Q = 0, DQ = Q + N, LL = DQ + N, INVD = LL + N * (N + 1) / 2, MDIAG = INVD + N, JT0 = MDIAG + N, U = JT0 + 6 * N,
						 SIG = U + 36, ALPHA = SIG + 6, X = ALPHA + 1, RC = X + 3, GRAV = RC + 9, COUNT = GRAV + N;
};
static_assert(BlendLayout<OSC_MAX_DOF>::COUNT == blend_scratch_doubles(OSC_MAX_DOF) && BlendLayout<4>::COUNT == blend_scratch_doubles(4),
			  "blend_scratch_doubles out of step with BlendLayout");

struct OscProgram {
	DevModel model;
	int32_t n_tasks;
	DevTask tasks[OSC_MAX_TASKS];
	DevMft mft[2];
	DevJt jt[2];
	int32_t use_prev_torques;
	int32_t gravity_comp;
	int32_t torque_saturation;
	int32_t update_models;	// this launch follows an updateControllerTaskModels()
	int32_t write_observers;
	int64_t n_robots;
	const double* q;   // n x N
	const double* dq;  // n x N
	double* tau;	   // n x N
	uint32_t* status;  // N
	// robots that need the singular (SVD) path this cycle: compacted list + two counters used alternately
	// (the fast kernel of cycle c fills count[c & 1] and clears count[(c + 1) & 1])
	int32_t* sing_list;	  // N
	int32_t* sing_count;  // 2
	int32_t sing_parity;
	// Cycle pipelining (osc_cycle.cuh, "cross-cycle dependencies"): consecutive cycles of one handle depend on each other
	// robot by robot only, so the fused kernel of cycle c + 1 waits for ITS OWN block of cycle c instead of the whole grid.
	uint32_t* block_epoch;	 // one word per block of the fused kernel: (cycle number << 1) | handed-robots-over bit
	uint32_t* general_done;	 // [0] cycle number the general-path kernel has completed, [1] its block completion counter, [2] count last sent to host_seen
	int32_t* host_seen;		 // mapped host word: hand-over count of the last completed cycle (a scheduling hint for the host)
	uint32_t epoch;			 // cycle number of this launch (31 bits used)
	unsigned long long* block_times;  // measurement aid (osc_debug_block_times): globaltimer at block start / end, 8 cycles deep; normally null
	int32_t general_grid_small;	 // host hint: the last cycles handed nothing over, a handful of general-path blocks is enough
	// split blending path (osc_blend.cuh): scratch block, variant lists [4][blend_cap] and their counters; null until needed
	double* blend_scratch;	// blend_scratch_doubles(n) x blend_cap
	int32_t* blend_lists;
	int32_t* blend_counts;	// [0..3] list counters, [4..7] those of the last cycle (osc_debug_general_path_counts)
	int64_t blend_cap;
	int32_t blend_split_on;	 // host decision for this cycle (the hint says many robots are on the general path)
	int32_t precision_fp32;	 // osc_set_precision: the fused kernel of the flagship hierarchy runs in single precision
};
