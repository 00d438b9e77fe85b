// The host-side plan of a control cycle (csrc/osc_launch.h) for tests/test_cycle_plan.py: the declared fused-kernel lists, and
// the kernels plan_cycle chooses for programs built from a set of conditions.
#include "../../sai_primitives_b200/csrc/osc_launch.h"
#include <cstring>

// CV_* bits in declaration order (FULL, SPEC, GRAV, MOTION, PARK, PRG, F32)
extern "C" void cycle_bits(unsigned* out) {
	const unsigned bits[7] = {osc::CV_FULL, osc::CV_SPEC, osc::CV_GRAV, osc::CV_MOTION, osc::CV_PARK, osc::CV_PRG, osc::CV_F32};
	std::memcpy(out, bits, sizeof(bits));
}

// the declared list of signature class R (f32: of the single-precision kernels) into out[16]; returns its length
extern "C" int cycle_words(int R, int f32, unsigned* out) {
	const osc::CycleWordList L = osc::cycle_words(R, f32 != 0);
	for (size_t k = 0; k < L.count && k < 16; k++) out[k] = L.word[k];
	return (int)L.count;
}

// Conditions of a program for plan(), as bits of `cond` (a hierarchy of signature (n, R, has_jt) on an all-revolute-z chain
// that the specialised kernel covers, unless a condition says otherwise).
enum Cond {
	C_FULL = 1,				// the motion-force task controls all six directions (with R = 6 only)
	C_OFF_AXIS = 2,			// a joint not about its local z axis
	C_TWO_CLAMPED = 4,		// two diagonal entries of M may fall below the bounded-inertia threshold
	C_FORCE = 8,			// force space of dimension one
	C_CLOSED_LOOP = 16,		// closed-loop force control
	C_VEL_SAT = 32,			// velocity saturation of the motion-force task
	C_MFT_GAINS = 64,		// gain block on the motion-force task
	C_JT_GAINS = 128,		// gain block on the joint task
	C_GRAVITY = 256,		// gravity compensation
	C_SPLIT_HINT = 512,		// the host hint says many robots are on the general path
	C_SCRATCH = 1024,		// the scratch block of the split blending path is allocated
	C_FP32 = 2048,			// single-precision mode
};

// plan_cycle for the program of (n, R, has_jt, cond): R > 0 a leading MotionForceTask of rank R, R == 0 a JointTask alone,
// R < 0 a general hierarchy led by a six-dof MotionForceTask.  Returns the plan's error code and, in *message, its message.
extern "C" int plan(int n, int R, int has_jt, int cond, unsigned* word, int* general, int* launches, const char** message) {
	OscProgram P;
	std::memset(&P, 0, sizeof(P));
	static double block[1];
	static uint32_t done[4];
	P.model.n = n;
	for (int j = 0; j < n; j++) {
		P.model.axis[j][2] = 1.0;
		P.model.inertia[j][0] = P.model.inertia[j][3] = P.model.inertia[j][5] = 0.3;
	}
	if (cond & C_OFF_AXIS) P.model.axis[1][2] = 0.0, P.model.axis[1][0] = 1.0;
	P.n_robots = 65536;
	if (R == 0) {
		P.n_tasks = 1;
		P.tasks[0].type = OSC_TASK_JOINT;
	} else {
		P.n_tasks = has_jt ? 2 : 1;
		P.tasks[0].type = OSC_TASK_MOTION_FORCE;
		P.tasks[1].type = OSC_TASK_JOINT;
		P.mft[0].rank = R > 0 ? R : 6;
		P.mft[0].full = (P.mft[0].rank == 6 && (cond & C_FULL)) ? 1 : 0;
	}
	P.mft[0].body = n - 1;
	P.mft[0].p.dynamic_decoupling_type = OSC_BOUNDED_INERTIA_ESTIMATES;
	P.mft[0].p.bie_threshold = (cond & C_TWO_CLAMPED) ? 0.7 : 0.1;
	P.mft[0].p.force_space_dimension = (cond & C_FORCE) ? 1 : 0;
	P.mft[0].p.closed_loop_force_control = (cond & C_CLOSED_LOOP) ? 1 : 0;
	P.mft[0].p.use_velocity_saturation = (cond & C_VEL_SAT) ? 1 : 0;
	P.jt[0].full = 1;
	P.jt[0].p.dynamic_decoupling_type = OSC_BOUNDED_INERTIA_ESTIMATES;
	P.jt[0].p.bie_threshold = 0.1;
	if (cond & C_MFT_GAINS) P.mft[0].gains = block;
	if (cond & C_JT_GAINS) P.jt[0].gains = block;
	P.gravity_comp = (cond & C_GRAVITY) ? 1 : 0;
	P.general_done = done;
	P.blend_split_on = (cond & C_SPLIT_HINT) ? 1 : 0;
	P.blend_scratch = (cond & C_SCRATCH) ? block : nullptr;
	P.precision_fp32 = (cond & C_FP32) ? 1 : 0;
	const osc::CyclePlan c = osc::plan_cycle(P, n, R, has_jt != 0);
	*word = c.fused;
	*general = (int)c.general;
	*launches = c.launches;
	*message = c.message;
	return c.error;
}
