// Per-robot force / moment spaces and closed-loop flags of a MotionForceTask (osc_mft_parametrize_spaces_batched,
// osc_mft_set_closed_loop_batched, osc_mft_get_spaces): validation of device input, the per-robot parametrisation with the
// reference's resets, and the read-back.  One robot per thread.
//   MotionForceTask::parametrizeForceMotionSpaces     src/tasks/MotionForceTask.cpp:830-858
//   MotionForceTask::parametrizeMomentRotMotionSpaces :860-890
//   MotionForceTask::setClosedLoopForceControl / setClosedLoopMomentControl :973-986
#pragma once
#include "osc_dev_types.h"
#include "osc_otg_kernels.cuh"
#include "osc_tasks.cuh"

namespace osc {

// OR over the robots of space_check (dims != null: dims N, axes SoA 3 x N) or closed_loop_check (flags != null) into *out.
// Grid-stride, one atomic per warp that found something.
__global__ void check_spaces_kernel(const int32_t* dims, const double* axes, const int32_t* flags, int64_t NR, int32_t* out) {
	int32_t f = 0;
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < NR; i += (int64_t)gridDim.x * blockDim.x) {
		if (dims) {
			const int32_t d = dims[i];
			// the axis of a robot of dimension 0 or 3 is not read (the caller may leave it unset)
			f |= (d == 1 || d == 2) ? space_check(d, axes[i], axes[NR + i], axes[2 * NR + i]) : space_check(d, 0.0, 0.0, 0.0);
		}
		if (flags) f |= closed_loop_check(flags[i]);
	}
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) f |= __shfl_xor_sync(0xffffffffu, f, o);
	if (f && (threadIdx.x & 31) == 0) atomicOr(out, f);
}

// Arguments of the per-robot parametrisation: per-robot values (dims != null) or the same values for every robot.
struct SpaceArgs {
	const int32_t* dims;  // N, validated
	const double* axes;	  // SoA 3 x N, read for robots of dimension 1 or 2
	int32_t dim;		  // dims == null: every robot's dimension and axis (not normalised)
	double axis[3];
	int32_t* was_reset;	 // N or null
	int32_t* any_reset;	 // |= 1 if a robot was reset, or null
};

// what parametrize* does to robot i's task object (moment = 0: force / motion space, 1: moment / rot-motion space)
__global__ void apply_spaces_kernel(const __grid_constant__ OscProgram P, int mft_index, int moment, const SpaceArgs a) {
	const int64_t NR = P.n_robots;
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= NR) return;
	const DevMft& t = P.mft[mft_index];
	const int shift = moment ? SP_MDIM_SHIFT : SP_FDIM_SHIFT;
	const int32_t mode = t.space_mode[i];
	const int32_t dim = a.dims ? a.dims[i] : a.dim;
	bool reset = dim != ((mode >> shift) & 3);
	if (dim == 1 || dim == 2) {	 // dimension 0 or 3: the stored axis stays as it was
		double in[3], u[3], cur[3];
		double* ax = t.space_axes + (moment ? 3 : 0) * NR;
		for (int k = 0; k < 3; k++) {
			in[k] = a.dims ? a.axes[k * NR + i] : a.axis[k];
			cur[k] = ax[k * NR + i];
		}
		space_normalize(in, u);
		reset = reset || !space_axis_is_approx(u, cur);
		for (int k = 0; k < 3; k++) ax[k * NR + i] = u[k];
	}
	t.space_mode[i] = (mode & ~(3 << shift)) | (dim << shift);
	auto S = [&](int comp) -> gdouble& { return t.st[(int64_t)comp * NR + i]; };	 // component comp of robot i
	if (reset) {
		if (t.otg.enabled) {  // _otg->reInitializeLinear / reInitializeAngular (:854, :886): goals and generator together
			otg_cart_reinit_part(t, NR, i, moment != 0);
		} else if (!moment) {  // :850-856
			for (int k = 0; k < 3; k++) {
				S(MC_GOAL_POS + k) = S(MC_CUR_POS + k);
				S(MC_GOAL_LINVEL + k) = 0.0;
				S(MC_GOAL_LINACC + k) = 0.0;
			}
		} else {  // :882-888
			for (int k = 0; k < 9; k++) S(MC_GOAL_ORI + k) = S(MC_CUR_ORI + k);
			for (int k = 0; k < 3; k++) {
				S(MC_GOAL_ANGVEL + k) = 0.0;
				S(MC_GOAL_ANGACC + k) = 0.0;
			}
		}
		for (int k = 0; k < 3; k++) {
			S((moment ? MC_INT_ORI : MC_INT_POS) + k) = 0.0;
			S((moment ? MC_INT_MOMENT : MC_INT_FORCE) + k) = 0.0;
		}
		if (a.any_reset) atomicOr(a.any_reset, 1);
	}
	if (a.was_reset) a.was_reset[i] = reset ? 1 : 0;
}

// setClosedLoopForceControl / setClosedLoopMomentControl of robot i (flags != null: flags[i], else `flag` for every robot): a
// robot whose flag changes gets its linear (force) or angular (moment) integrators zeroed
__global__ void set_closed_loop_kernel(const __grid_constant__ OscProgram P, int mft_index, int moment, const int32_t* flags, int32_t flag) {
	const int64_t NR = P.n_robots;
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= NR) return;
	const DevMft& t = P.mft[mft_index];
	const int32_t bit = moment ? SP_CL_MOMENT : SP_CL_FORCE;
	const int32_t mode = t.space_mode[i];
	const bool on = (flags ? flags[i] : flag) != 0;
	if (((mode & bit) != 0) == on) return;
	t.space_mode[i] = mode ^ bit;
	auto S = [&](int comp) -> gdouble& { return t.st[(int64_t)comp * NR + i]; };
	for (int k = 0; k < 3; k++) {
		S((moment ? MC_INT_ORI : MC_INT_POS) + k) = 0.0;
		S((moment ? MC_INT_MOMENT : MC_INT_FORCE) + k) = 0.0;
	}
}

// what the control laws use for robot i; any output may be null
__global__ void get_spaces_kernel(const __grid_constant__ OscProgram P, int mft_index, int moment, int32_t* dims, double* axes, int32_t* closed_loop) {
	const int64_t NR = P.n_robots;
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= NR) return;
	const DevMft& t = P.mft[mft_index];
	const int32_t mode = mft_space_mode(t, i);
	if (dims) dims[i] = (mode >> (moment ? SP_MDIM_SHIFT : SP_FDIM_SHIFT)) & 3;
	if (closed_loop) closed_loop[i] = (mode & (moment ? SP_CL_MOMENT : SP_CL_FORCE)) ? 1 : 0;
	if (axes) {
		double af[3], am[3];
		mft_space_axes(t, NR, i, af, am);
		for (int k = 0; k < 3; k++) axes[k * NR + i] = moment ? am[k] : af[k];
	}
}

}  // namespace osc
