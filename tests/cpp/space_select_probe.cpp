// Host-side pieces of the per-robot force / moment spaces (csrc/osc_dev_types.h, csrc/osc_launch.h), for
// tests/test_space_selection.py: the pure-motion decision that selects the MOTION kernels, the reset rule shared by the host
// and the kernels, the mode word and the validation of per-robot values.
#include "../../sai_primitives_b200/csrc/osc_launch.h"
#include <cstring>

// mft_pure_motion for a full (or partial) task with the given broadcast parameters and, when `block` is set, a space block
// whose host summary is `summary`
extern "C" int pure_motion(int block, int summary, int fdim, int mdim, int clf, int clm, int full, int vel_sat) {
	static int32_t word[1];
	static double axes[6];
	DevMft t;
	std::memset(&t, 0, sizeof(t));
	t.full = full;
	t.p.force_space_dimension = fdim;
	t.p.moment_space_dimension = mdim;
	t.p.closed_loop_force_control = clf;
	t.p.closed_loop_moment_control = clm;
	t.p.use_velocity_saturation = vel_sat;
	if (block) {
		t.space_mode = word;
		t.space_axes = axes;
		t.space_any = summary;
	}
	return osc::mft_pure_motion(t) ? 1 : 0;
}

extern "C" int axis_is_approx(const double* a, const double* b) { return space_axis_is_approx(a, b) ? 1 : 0; }
extern "C" double normalize(const double* axis, double* u) { return space_normalize(axis, u); }
extern "C" int mode_word(int fdim, int mdim, int clf, int clm) { return space_mode_word(fdim, mdim, clf != 0, clm != 0); }
extern "C" int check_space(int dim, double a0, double a1, double a2) { return space_check(dim, a0, a1, a2); }
extern "C" int check_flag(int flag) { return closed_loop_check(flag); }
