// Host-callable launch wrappers around the templated kernels (implemented in the .cu files).
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstddef>
#include <iterator>

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
// robot dofs the single-precision fused kernel is instantiated for (osc_cycle_f32.cu)
#define OSC_F32_DOFS(X) X(7)
#define OSC_F32_IS(m) || n == m
inline bool cycle_f32_dof(int n) { return false OSC_F32_DOFS(OSC_F32_IS); }
#undef OSC_F32_IS

// Flag word V of the fused cycle kernel osc_cycle_kernel<N, R, HAS_JT, V> (osc_cycle.cuh, which states what each flag compiles in).
constexpr unsigned CV_FULL = 1u << 0;	 // the motion-force task controls all six directions (B = I)
constexpr unsigned CV_SPEC = 1u << 1;	 // specialisation for the default configuration (cycle_spec_eligible)
constexpr unsigned CV_GRAV = 1u << 2;	 // gravity compensation compiled in
constexpr unsigned CV_MOTION = 1u << 3;	 // the motion-force task is under pure motion control (mft_pure_motion)
constexpr unsigned CV_PARK = 1u << 4;	 // hand-overs are parked for the split blending path
constexpr unsigned CV_PRG = 1u << 5;	 // per-robot PID gains read from the tasks' gain blocks
constexpr unsigned CV_F32 = 1u << 6;	 // in a plan only: the single-precision instantiation (osc_cycle_f32.cu) of the word without it
constexpr bool cycle_word_legal(int R, unsigned v) {
	return (!(v & (CV_MOTION | CV_GRAV)) || (v & CV_SPEC)) && (!(v & CV_PRG) || (v & CV_SPEC) || R == 0) &&
		   (!(v & CV_PARK) || (R == 6 && (v & CV_FULL)));
}

// The instantiated fused kernels: one flag word each, per signature class.  The planner (plan_cycle) only produces listed words.
constexpr unsigned kCycleWordsR6[] = {
	0,	// partial task
	CV_FULL, CV_FULL | CV_PARK,
	CV_FULL | CV_SPEC, CV_FULL | CV_SPEC | CV_GRAV, CV_FULL | CV_SPEC | CV_PARK, CV_FULL | CV_SPEC | CV_GRAV | CV_PARK,
	CV_FULL | CV_SPEC | CV_MOTION, CV_FULL | CV_SPEC | CV_MOTION | CV_GRAV, CV_FULL | CV_SPEC | CV_MOTION | CV_PARK,
	CV_FULL | CV_SPEC | CV_MOTION | CV_GRAV | CV_PARK,
	CV_FULL | CV_SPEC | CV_MOTION | CV_PRG, CV_FULL | CV_SPEC | CV_MOTION | CV_PRG | CV_GRAV, CV_FULL | CV_SPEC | CV_MOTION | CV_PRG | CV_PARK,
	CV_FULL | CV_SPEC | CV_MOTION | CV_PRG | CV_GRAV | CV_PARK,
};
constexpr unsigned kCycleWordsR3[] = {0, CV_SPEC, CV_SPEC | CV_GRAV, CV_SPEC | CV_PRG, CV_SPEC | CV_GRAV | CV_PRG};
constexpr unsigned kCycleWordsR0[] = {0, CV_PRG};  // a JointTask alone
constexpr unsigned kCycleWordsOther[] = {0};
constexpr unsigned kCycleWordsF32[] = {CV_FULL | CV_SPEC | CV_MOTION, CV_FULL | CV_SPEC | CV_MOTION | CV_GRAV};  // R = 6, OSC_F32_DOFS
struct CycleWordList {
	const unsigned* word;
	size_t count;
};
// the list of signature class R (f32: of the single-precision instantiations)
constexpr CycleWordList cycle_words(int R, bool f32 = false) {
	return f32		 ? CycleWordList{kCycleWordsF32, std::size(kCycleWordsF32)}
		   : R == 6 ? CycleWordList{kCycleWordsR6, std::size(kCycleWordsR6)}
		   : R == 3 ? CycleWordList{kCycleWordsR3, std::size(kCycleWordsR3)}
		   : R == 0 ? CycleWordList{kCycleWordsR0, std::size(kCycleWordsR0)}
					: CycleWordList{kCycleWordsOther, std::size(kCycleWordsOther)};
}
constexpr bool cycle_words_legal(int R, bool f32 = false) {
	const CycleWordList L = cycle_words(R, f32);
	for (size_t k = 0; k < L.count; k++)
		if (!cycle_word_legal(R, L.word[k]) || (L.word[k] & CV_F32)) return false;
	return true;
}
static_assert(cycle_words_legal(6) && cycle_words_legal(3) && cycle_words_legal(0) && cycle_words_legal(1) && cycle_words_legal(6, true),
			  "fused kernel flags: MOTION and GRAV require SPEC, PRG requires SPEC or R = 0, PARK requires R = 6 and FULL");

// Launches the fused cycle kernel K over the robots of P: kCycleBlock threads per block, `smem` bytes of dynamic shared memory,
// programmatic stream serialization with the general-path kernels before and after it.  The shared-memory attribute is set
// once per device: function attributes belong to the device's context.  Atomic flags: host threads driving different handles
// may get here at the same time (setting the attribute twice is harmless, a torn read of a plain bool is not defined).
template <auto K, typename Program>
cudaError_t launch_fused_kernel(const Program& P, int smem, cudaStream_t stream) {
	static std::atomic<bool> configured[64];
	int dev = 0;
	cudaGetDevice(&dev);
	if (dev < 0 || dev >= 64 || !configured[dev].load(std::memory_order_acquire)) {
		cudaError_t e = cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
		if (e != cudaSuccess) return e;
		if (dev >= 0 && dev < 64) configured[dev].store(true, std::memory_order_release);
	}
	cudaLaunchConfig_t cfg{};
	cfg.gridDim = dim3((unsigned)((P.n_robots + kCycleBlock - 1) / kCycleBlock));
	cfg.blockDim = dim3(kCycleBlock);
	cfg.dynamicSmemBytes = smem;
	cfg.stream = stream;
	cudaLaunchAttribute attr[1];
	attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
	attr[0].val.programmaticStreamSerializationAllowed = 1;
	cfg.attrs = attr;
	cfg.numAttrs = 1;
	return cudaLaunchKernelEx(&cfg, K, P);
}

// The kernels one control cycle launches (plan_cycle): the fused kernel, then the general path for the robots it hands over.
enum class GeneralPath {
	None,		  // a JointTask alone: nothing is handed over
	Singular,	  // osc_singular_kernel
	Blend,		  // osc_blend_kernel (full six-dof task)
	BlendSplit,	  // the three kernels of the split blending path (osc_blend.cuh)
	Generic,	  // general hierarchy (R < 0): osc_generic_kernel for every robot, no fused kernel
};
struct CyclePlan {
	unsigned fused = 0;	 // flag word of the fused kernel, in the list of its signature class (cycle_words)
	GeneralPath general = GeneralPath::None;
	int launches = 0;			  // kernels launched
	int error = OSC_OK;			  // OSC_ERR_UNSUPPORTED: the cycle is refused with `message`
	const char* message = nullptr;
};

// Fused control cycle for hierarchy signature (n, R, has_jt): R = rank of a leading MotionForceTask (0: none),
// has_jt = a full JointTask closes the hierarchy; R < 0 selects the general-hierarchy kernel.  Launches what `plan` names.
// cudaErrorNotSupported when the dof is not compiled in (OSC_CYCLE_DOFS) or the plan refuses the cycle.
cudaError_t launch_cycle(int n, int R, bool has_jt, const CyclePlan& plan, const OscProgram& P, cudaStream_t stream);
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

// The kernels of one control cycle of hierarchy signature (n, R, has_jt) on program P, or its refusal.
inline CyclePlan plan_cycle(const OscProgram& P, int n, int R, bool has_jt) {
	CyclePlan c;
	bool motion = false;
	const bool spec = (R == 6 || R == 3) && cycle_spec_eligible(P, has_jt, &motion);
	// the single-precision mode has the fused kernel of the pure-motion full six-dof task only
	if (P.precision_fp32 && !(R == 6 && P.mft[0].full && spec && motion && cycle_f32_dof(n)))
		c.message = "FP32 mode covers a full six-dof MotionForceTask under pure motion control (alone or with a full JointTask) on an all-revolute-z chain only";
	else if (P.precision_fp32 && (P.mft[0].gains || P.mft[1].gains || P.jt[0].gains || P.jt[1].gains))
		c.message = "FP32 mode: the kernels have no single-precision form with per-robot gains (osc_set_gains)";
	if (c.message) {
		c.error = OSC_ERR_UNSUPPORTED;
		return c;
	}
	const bool prg = cycle_per_robot_gains(P, has_jt), prg_spec = prg && cycle_prg_specialised(R, spec, motion);
	const unsigned grav = P.gravity_comp ? CV_GRAV : 0u;
	const bool split = R == 6 && blend_split_selected(P);
	if (R == 6 && P.mft[0].full) {
		// with many robots on the general path the hand-overs also park their kinematics and dynamics
		c.fused = CV_FULL | (split ? CV_PARK : 0u);
		if (spec && (prg_spec || !prg)) c.fused |= CV_SPEC | grav | (motion ? CV_MOTION : 0u) | (prg_spec ? CV_PRG : 0u);
	} else if (R == 3 && spec) {
		c.fused = CV_SPEC | grav | (prg_spec ? CV_PRG : 0u);
	} else if (R == 0 && prg) {
		c.fused = CV_PRG;
	}
	if (P.precision_fp32) c.fused |= CV_F32;
	c.general = R < 0	 ? GeneralPath::Generic
				: R == 0 ? GeneralPath::None
				: split	 ? GeneralPath::BlendSplit
				: (R == 6 && P.mft[0].full) ? GeneralPath::Blend
											: GeneralPath::Singular;
	c.launches = (R <= 0) ? 1 : split ? 4 : 2;
	return c;
}

// The optional single-precision mode (osc_cycle_f32.cu): the fused kernel of [full six-dof MotionForceTask under pure motion
// control (+ full JointTask)] computed in FP32 on the FP64 state in global memory; robots it hands over continue on the FP64
// general path.  `word`: a plan's fused word.  cudaErrorNotSupported for a dof (OSC_F32_DOFS) or word that is not compiled in.
cudaError_t launch_cycle_fused_f32(int n, bool has_jt, unsigned word, const OscProgram& P, cudaStream_t stream);
cudaError_t launch_popc_probe(const OscProgram& P, int mft_index, int K, const double* fd, const double* fs, const double* vcl, const double* vr,
							  double kv, double kff, double* out, cudaStream_t stream);
cudaError_t measure_fp64_peak(double seconds, double* tflops, cudaStream_t stream);
cudaError_t launch_sim_integrate(const OscProgram& P, double* q, double* dq, const double* tau, double dt, int substeps, cudaStream_t stream);
cudaError_t launch_jla(const OscProgram& P, cudaStream_t stream);
// internal OTG of the tasks (osc_otg_kernels.cuh): per-cycle update, (re)initialisation (mode 0 enabled: generator constructed,
// 1 linear part, 2 angular part, 3 limits changed), switch-off
cudaError_t launch_otg_update(const OscProgram& P, cudaStream_t stream);
cudaError_t launch_otg_init(const OscProgram& P, int task, int mode, cudaStream_t stream);
cudaError_t launch_otg_disable(const OscProgram& P, int task, cudaStream_t stream);
// read-only observers (osc_observers.cuh): kind = ObserverKind, task = position in the hierarchy, out = ncomp x N (SoA)
cudaError_t launch_observer(const OscProgram& P, int task, int kind, double* out, cudaStream_t stream);
// task resets of the robots selected by mask (device int32 x N, != 0 selects; null: every robot), task < 0: every task, in one
// launch (reset_robots_kernel, osc_aux_kernels.cuh).  construct = 0: reInitializeTask; 1: the state the constructor leaves
cudaError_t launch_reset_robots(const OscProgram& P, const int32_t* mask, int task, int construct, cudaStream_t stream);
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
