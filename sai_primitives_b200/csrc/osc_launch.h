// Host-callable launch wrappers around the templated kernels (implemented in the .cu files).
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>

#include "osc_dev_types.h"

namespace osc {

#ifndef OSC_CYCLE_BLOCK
#define OSC_CYCLE_BLOCK 128
#endif
constexpr int kCycleBlock = OSC_CYCLE_BLOCK;

// robot dofs the fused cycle kernel is instantiated for (one translation unit each, see Makefile)
#ifdef OSC_TUNE_DOF7_ONLY  // tuning builds (tools/tune.sh): the Panda kernels only
#define OSC_CYCLE_DOFS(X) X(7)
#else
#define OSC_CYCLE_DOFS(X) X(4) X(6) X(7) X(8)
#endif

// Fused control cycle for hierarchy signature (n, R, has_jt): R = rank of a leading MotionForceTask (0: none),
// has_jt = a full JointTask closes the hierarchy; R < 0 selects the general-hierarchy kernel.
// cudaErrorNotSupported when the dof is not compiled in (OSC_CYCLE_DOFS).
cudaError_t launch_cycle(int n, int R, bool has_jt, const OscProgram& P, cudaStream_t stream);
bool cycle_signature_available(int n, int R, bool has_jt);
// the general path of this launch runs as the three kernels of the split blending path (osc_blend.cuh) instead of osc_blend_kernel:
// flagship hierarchy, pipelined handle, and the host hint says that many robots are on the general path (osc_capi.cu, run_cycle)
inline bool blend_split_selected(const OscProgram& P) {
	return P.blend_split_on && !P.precision_fp32 && P.blend_scratch != nullptr && P.general_done != nullptr && !P.general_grid_small && P.n_tasks >= 1 && P.tasks[0].type == OSC_TASK_MOTION_FORCE &&
		   P.mft[0].full && P.mft[0].rank == 6;
}

// smallest eigenvalue of a symmetric 3 x 3 matrix (xx xy xz yy yz zz), trigonometric closed form
inline double min_eig_sym3(const double* I) {
	const double a = I[0], b = I[3], c = I[5], d = I[1], e = I[2], f = I[4];
	const double p1 = d * d + e * e + f * f;
	const double q = (a + b + c) / 3.0;
	if (p1 == 0.0) return std::min(a, std::min(b, c));
	const double p2 = (a - q) * (a - q) + (b - q) * (b - q) + (c - q) * (c - q) + 2.0 * p1;
	const double p = std::sqrt(p2 / 6.0);
	const double B[6] = {(a - q) / p, d / p, e / p, (b - q) / p, f / p, (c - q) / p};
	double r = 0.5 * (B[0] * (B[3] * B[5] - B[4] * B[4]) - B[1] * (B[1] * B[5] - B[4] * B[2]) + B[2] * (B[1] * B[4] - B[3] * B[2]));
	r = std::max(-1.0, std::min(1.0, r));
	const double phi = std::acos(r) / 3.0;
	return q + 2.0 * p * std::cos(phi + 2.0 * 3.14159265358979323846 / 3.0);
}

// Every robot of the motion-force task is under pure motion control of a full task without velocity saturation, so the
// MOTION instantiations, which never read the per-robot space block, compute what the general control law would: no force or
// moment space and both loops open -- the task's parameters, or with per-robot spaces (osc_mft_parametrize_spaces_batched)
// the host's summary over the robots.
inline bool mft_pure_motion(const DevMft& t) {
	const osc_mft_params& p = t.p;
	const bool free = t.space_mode ? t.space_any == 0
								   : (p.force_space_dimension == 0 && p.moment_space_dimension == 0 && !p.closed_loop_force_control &&
									  !p.closed_loop_moment_control);
	return t.full && free && !p.use_velocity_saturation;
}

// Conditions under which the specialised instantiation (SPEC, osc_cycle.cuh) computes the same thing as the general one.
// *motion: the motion-force task additionally is a full task under pure motion control (the MOTION flag of the kernel)
inline bool cycle_spec_eligible(const OscProgram& P, bool has_jt, bool* motion) {
	const DevModel& m = P.model;
	for (int j = 0; j < m.n; j++)
		if (m.jtype[j] != 0 || m.axis[j][0] != 0.0 || m.axis[j][1] != 0.0 || m.axis[j][2] != 1.0) return false;
	if (P.mft[0].body < 0) return false;
	if ((unsigned long long)P.n_robots * (unsigned long long)MC_COUNT >= (1ull << 32)) return false;  // 32-bit element indices
	// The specialisation carries the bounded-inertia update of rank <= 1 only (robots needing more are handed to the
	// general path one by one, which is correct but slow): require that at most one diagonal entry of M can ever fall
	// below the threshold.  M_jj >= sum over the bodies the joint moves of their smallest principal moment of inertia.
	{
		double thr = 0.0;
		if (P.mft[0].p.dynamic_decoupling_type == OSC_BOUNDED_INERTIA_ESTIMATES) thr = std::max(thr, P.mft[0].p.bie_threshold);
		if (has_jt && P.jt[0].p.dynamic_decoupling_type == OSC_BOUNDED_INERTIA_ESTIMATES) thr = std::max(thr, P.jt[0].p.bie_threshold);
		double lb = 0.0;
		int may_clamp = 0;
		for (int j = m.n - 1; j >= 0; j--) {
			lb += min_eig_sym3(m.inertia[j]);
			if (lb < thr) may_clamp++;
		}
		if (may_clamp > 1) return false;
	}
	// IMPEDANCE decoupling needs no code of its own (Lambda_modified = I: the solves are skipped); velocity saturation of the
	// motion-force task is part of the general control law, which the structural specialisation (MOTION = false) keeps
	*motion = mft_pure_motion(P.mft[0]);
	if (has_jt) {
		const DevJt& j = P.jt[0];
		if (!j.full || j.p.use_velocity_saturation) return false;  // the staged joint control law has no velocity saturation
	}
	return true;
}

// Per-robot PID gains (osc_set_gains): a leading task of the hierarchy has a gain block.
inline bool cycle_per_robot_gains(const OscProgram& P, bool has_jt) {
	return (P.n_tasks >= 1 && P.tasks[0].type == OSC_TASK_MOTION_FORCE && P.mft[0].gains != nullptr) || (has_jt && P.jt[0].gains != nullptr);
}
// With per-robot gains, the specialised fused kernel of signature R (spec, motion: cycle_spec_eligible) has an instantiation that
// reads them (PRG): the pure-motion full six-dof task and the three-direction task.  Otherwise the launch takes the
// non-specialised kernel, which tests the gain-block pointers at run time.
inline bool cycle_prg_specialised(int R, bool spec, bool motion) { return spec && ((R == 6 && motion) || R == 3); }

// The optional single-precision mode (osc_cycle_f32.cu): the fused kernel of [full six-dof MotionForceTask under pure motion
// control (+ full JointTask)] computed in FP32 on the FP64 state in global memory; robots it hands over continue on the FP64
// general path.  cudaErrorNotSupported for a dof that is not compiled in (fused_f32_available).
cudaError_t launch_cycle_fused_f32(int n, bool has_jt, const OscProgram& P, cudaStream_t stream);
bool fused_f32_available(int n);
cudaError_t launch_popc_probe(const OscProgram& P, int mft_index, int K, const double* fd, const double* fs, const double* vcl, const double* vr,
							  double kv, double kff, double* out, cudaStream_t stream);
cudaError_t measure_fp64_peak(double seconds, double* tflops, cudaStream_t stream);
cudaError_t launch_sim_integrate(const OscProgram& P, double* q, double* dq, const double* tau, double dt, int substeps, cudaStream_t stream);
cudaError_t launch_jla(const OscProgram& P, cudaStream_t stream);
// internal OTG of the tasks (osc_otg_kernels.cuh): per-cycle update, (re)initialisation (mode 0 whole task, 1 linear part,
// 2 angular part, 3 limits changed; fresh = generator constructed), switch-off
cudaError_t launch_otg_update(const OscProgram& P, cudaStream_t stream);
cudaError_t launch_otg_init(const OscProgram& P, int task, int mode, int fresh, cudaStream_t stream);
cudaError_t launch_otg_disable(const OscProgram& P, int task, cudaStream_t stream);
// read-only observers (osc_observers.cuh): kind = ObserverKind, task = position in the hierarchy, out = ncomp x N (SoA)
cudaError_t launch_observer(const OscProgram& P, int task, int kind, double* out, cudaStream_t stream);
cudaError_t launch_reinit_mft(const OscProgram& P, int mft_index, int full_init, cudaStream_t stream);
cudaError_t launch_reinit_jt(const OscProgram& P, int jt_index, cudaStream_t stream);
cudaError_t launch_sensed_wrench(const OscProgram& P, int mft_index, const double* f, const double* m, cudaStream_t stream);
cudaError_t launch_eval_model(const OscProgram& P, const osc_link_frame& frame, double* M, double* J, double* x, double* R,
							  double* g, cudaStream_t stream);
cudaError_t launch_fill(double* st, int64_t NR, int comp, int ncomp, const double* vals, cudaStream_t stream);
cudaError_t launch_copy(double* st, int64_t NR, int dst, int src, int ncomp, cudaStream_t stream);
// *bad |= 1: some of the n values is not finite, |= 2: some is negative (*bad is not cleared)
cudaError_t launch_check_values(const double* v, int64_t n, int32_t* bad, cudaStream_t stream);
// per-robot force / moment spaces (osc_space_kernels.cuh).  check: *out |= SpaceCheck bits over the n robots (dims / axes and
// flags may each be null).  apply: parametrize* per robot (dims == null: dim and axis for every robot).  moment: 0 force, 1 moment.
cudaError_t launch_check_spaces(const int32_t* dims, const double* axes, const int32_t* flags, int64_t n, int32_t* out, cudaStream_t stream);
cudaError_t launch_apply_spaces(const OscProgram& P, int mft_index, int moment, const int32_t* dims, const double* axes, int dim,
								const double axis[3], int32_t* was_reset, int32_t* any_reset, cudaStream_t stream);
cudaError_t launch_set_closed_loop(const OscProgram& P, int mft_index, int moment, const int32_t* flags, int flag, cudaStream_t stream);
cudaError_t launch_get_spaces(const OscProgram& P, int mft_index, int moment, int32_t* dims, double* axes, int32_t* closed_loop, cudaStream_t stream);
cudaError_t launch_fill_int(int32_t* ist, int64_t NR, int comp, int ncomp, int32_t value, cudaStream_t stream);

}  // namespace osc
