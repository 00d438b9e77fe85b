// Host-side decisions of the launcher (csrc/osc_launch.h) about per-robot gains, for tests/test_gain_selection.py: when a
// launch counts as one with per-robot gains, and which specialised signatures have an instantiation that reads them.
#include "../../sai_primitives_b200/csrc/osc_launch.h"
#include <cstring>

// bit 0: cycle_per_robot_gains(P, has_jt) for a [MotionForceTask, JointTask] program with gain blocks on the tasks named by
// `blocks` (bit 0 motion-force task, bit 1 joint task); `jt_first`: a JointTask leads the hierarchy instead
extern "C" int per_robot_case(int blocks, int has_jt, int jt_first) {
	OscProgram P;
	std::memset(&P, 0, sizeof(P));
	static double block[1];
	P.n_tasks = 2;
	P.tasks[0].type = jt_first ? OSC_TASK_JOINT : OSC_TASK_MOTION_FORCE;
	P.tasks[1].type = jt_first ? OSC_TASK_MOTION_FORCE : OSC_TASK_JOINT;
	if (blocks & 1) P.mft[0].gains = block;
	if (blocks & 2) P.jt[0].gains = block;
	return osc::cycle_per_robot_gains(P, has_jt != 0) ? 1 : 0;
}

extern "C" int prg_specialised(int R, int spec, int motion) { return osc::cycle_prg_specialised(R, spec != 0, motion != 0) ? 1 : 0; }
