// Control laws of the two task types, one robot per thread.
//   mft_control_law   MotionForceTask::computeTorques() up to the call into the singularity handler
//                     (reference src/tasks/MotionForceTask.cpp:278-491)
//   popc_step         POPCExplicitForceControl::computePassivitySaturatedForce
//                     (reference src/helper_modules/POPCExplicitForceControl.cpp:30-96)
//   joint_control_law JointTask::computeTorques() up to the range-space mapping
//                     (reference src/tasks/JointTask.cpp:294-346)
#pragma once
#include "osc_dev_types.h"
#include "osc_math.cuh"

namespace osc {

// IDX is int64_t in general; the SPEC instantiation of the fused kernel uses uint32_t (host check: every state block has
// fewer than 2^32 elements), which halves the integer work per access.
#define ST(comp, c) st[(decltype(NR))((comp) + (c)) * NR + i]

template <typename IDX>
DEVI void load3(const gdouble* st, IDX NR, IDX i, int comp, double v[3]) {
	v[0] = ST(comp, 0);
	v[1] = ST(comp, 1);
	v[2] = ST(comp, 2);
}
template <typename IDX>
DEVI void store3(gdouble* st, IDX NR, IDX i, int comp, const double v[3]) {
	ST(comp, 0) = v[0];
	ST(comp, 1) = v[1];
	ST(comp, 2) = v[2];
}

// SaiModel::orientationError(desired, current) = -1/2 sum_i Rc[:,i] x Rd[:,i]
DEVI void orientation_error(const double Rd[9], const double Rc[9], double e[3]) {
	e[0] = e[1] = e[2] = 0.0;
#pragma unroll
	for (int k = 0; k < 3; k++) {
		const double c[3] = {Rc[k], Rc[3 + k], Rc[6 + k]};
		const double d[3] = {Rd[k], Rd[3 + k], Rd[6 + k]};
		double x[3];
		cross3(c, d, x);
		e[0] -= 0.5 * x[0];
		e[1] -= 0.5 * x[1];
		e[2] -= 0.5 * x[2];
	}
}

// sigma projector of MotionForceTask::sigmaForce / sigmaMoment (MotionForceTask.cpp:892-966):
//   dim 0: 0;  1: P u u^T P^T;  2: P (I - u u^T) P^T;  3: P      with u = Rsel * axis
DEVI void sigma_space(int dim, const double P[9], const double u[3], double S[9]) {
	if (dim == 0) {
#pragma unroll
		for (int k = 0; k < 9; k++) S[k] = 0.0;
	} else if (dim == 3) {
#pragma unroll
		for (int k = 0; k < 9; k++) S[k] = P[k];
	} else {
		double Pu[3];
		mat3_vec(P, u, Pu);
		if (dim == 1) {
#pragma unroll
			for (int r = 0; r < 3; r++)
#pragma unroll
				for (int c = 0; c < 3; c++) S[3 * r + c] = Pu[r] * Pu[c];
		} else {
			double PPt[9];
			mat3_mul_bt(P, P, PPt);
#pragma unroll
			for (int r = 0; r < 3; r++)
#pragma unroll
				for (int c = 0; c < 3; c++) S[3 * r + c] = PPt[3 * r + c] - Pu[r] * Pu[c];
		}
	}
}
// sigmaPosition / sigmaOrientation: P (I - S) P^T  (MotionForceTask.cpp:927-930, 968-971)
DEVI void sigma_complement(const double P[9], const double S[9], double C[9]) {
	double ImS[9], T[9];
#pragma unroll
	for (int k = 0; k < 9; k++) ImS[k] = ((k % 4 == 0) ? 1.0 : 0.0) - S[k];
	mat3_mul(P, ImS, T);
	mat3_mul_bt(T, P, C);
}

// POPC step on the state of robot i.  fd, fs, vcl, vr are already sigma_force-projected.
template <typename IDX>
DEVI void popc_step(const DevMft& t, IDX NR, IDX i, const double fd[3], const double fs[3], const double vcl[3],
					const double vr[3], double kv, double kff, double out[3], uint32_t& status) {
	gdouble* st = t.st;
	int32_t* ist = t.ist;
	if (!t.p.passivity_enabled) {
#pragma unroll
		for (int k = 0; k < 3; k++) out[k] = vcl[k] - kv * vr[k];
		return;
	}
	const double dt = t.dt;
	double PO = ST(MC_POPC, 0), Ecorr = ST(MC_POPC, 1), Rc = ST(MC_POPC, 2), vsum = ST(MC_POPC, 3);
	int32_t counter = ist[(int64_t)MI_POPC_COUNTER * NR + i];
	int32_t head = ist[(int64_t)MI_RING_HEAD * NR + i];
	int32_t size = ist[(int64_t)MI_RING_SIZE * NR + i];
	const int32_t cap = t.ring_capacity;
	double Fcmd[3];
#pragma unroll
	for (int k = 0; k < 3; k++) Fcmd[k] = kff * fd[k] + Rc * vcl[k] - kv * vr[k];
	const double vc2 = dot3(vcl, vcl);
	const double fdiff[3] = {fs[0] - fd[0], fs[1] - fd[1], fs[2] - fd[2]};
	const double power = (dot3(fdiff, vcl) - dot3(Fcmd, vr)) * dt;
	PO += power;
	// push
	if (size == cap) {
		// Ring full (the reference queue is unbounded: it only shrinks while the observer total is positive, :49-61).  The oldest
		// sample leaves the way the reference will eventually pop it: a positive sample is subtracted from the observer.  For
		// samples <= 0 this is exactly what the reference does later (they are popped without touching the observer), so only a
		// positive sample that is more than `capacity` cycles old while the observer has stayed <= 0 all along is forgotten early.
		// From then on the passivity controller's Rc differs from the reference's (tests/test_popc_reference.py measures by how
		// much); the status bit says that parity is lost.  A ring as long as the longest active episode never gets here.
		const double front = t.ring[(int64_t)head * NR + i];
		if (front > 0.0) PO -= front;
		head = (head + 1) % cap;
		size--;
		status |= OSC_STATUS_POPC_OVERFLOW;
	}
	t.ring[(int64_t)((head + size) % cap) * NR + i] = power;
	size++;
	const int32_t window = 250;		// POPCExplicitForceControl.h:37
	const int32_t max_counter = 50; // POPCExplicitForceControl.h:38
	if (PO + Ecorr > 0.0) {
		while (size > window) {
			const double front = t.ring[(int64_t)head * NR + i];
			if (PO + Ecorr > front) {
				if (front > 0.0) PO -= front;
				head = (head + 1) % cap;
				size--;
			} else {
				break;
			}
		}
	}
	if (counter <= 0) {
		counter = max_counter;
		const double old_Rc = Rc;
		if (PO + Ecorr < 0.0) {
			Rc = 1.0 + (PO + Ecorr) / (vsum * dt);
			if (Rc > 1.0) Rc = 1.0;
			if (Rc < 0.0) Rc = 0.0;
		} else {
			Rc = (1.0 + (0.1 * max_counter - 1.0) * Rc) / (double)(0.1 * max_counter);
		}
		Ecorr += (1.0 - old_Rc) * vsum * dt;
		vsum = 0.0;
	}
	counter--;
	vsum += vc2;
#pragma unroll
	for (int k = 0; k < 3; k++) out[k] = Rc * vcl[k] - kv * vr[k];
	ST(MC_POPC, 0) = PO;
	ST(MC_POPC, 1) = Ecorr;
	ST(MC_POPC, 2) = Rc;
	ST(MC_POPC, 3) = vsum;
	ist[(int64_t)MI_POPC_COUNTER * NR + i] = counter;
	ist[(int64_t)MI_RING_HEAD * NR + i] = head;
	ist[(int64_t)MI_RING_SIZE * NR + i] = size;
}

// Where a control law reads its PID gains: the task's broadcast parameters (GAINS_BCAST); its per-robot gain block
// (GAINS_ROBOT: osc_set_gains, GainComp layout), loaded into registers once per robot -- or, for a task of the launch that has
// no block, its parameters (one uniform branch); or, per use, whichever of the two the block pointer says (GAINS_ANY: the
// non-specialised and general-path kernels).
enum GainSrc : int { GAINS_BCAST = 0, GAINS_ROBOT = 1, GAINS_ANY = 2 };
// pb: the task's parameters, whose first GAIN_COUNT values have the block's layout (checked in osc_capi.cu)
template <int G, typename IDX>
DEVI void load_gain_block(const gdouble* blk, const double* pb, IDX NR, IDX i, int c0, int nc, double* g) {
	if constexpr (G == GAINS_ROBOT) {
		if (blk) {
#pragma unroll
			for (int c = 0; c < nc; c++) g[c] = blk[(IDX)(c0 + c) * NR + i];
		} else {
#pragma unroll
			for (int c = 0; c < nc; c++) g[c] = pb[c0 + c];
		}
	}
}
// gain `member[k]` (block component comp + k) of robot i
#define OSC_GAIN(member, comp, k)                                                     \
	(G == GAINS_BCAST	? p.member[k]                                                  \
	 : G == GAINS_ROBOT ? kg[(comp) + (k)]                                             \
						: (t.gains ? t.gains[(IDX)((comp) + (k)) * NR + i] : p.member[k]))
#define OSC_GAIN1(member, comp)                                          \
	(G == GAINS_BCAST	? p.member                                        \
	 : G == GAINS_ROBOT ? kg[comp]                                        \
						: (t.gains ? t.gains[(IDX)(comp) * NR + i] : p.member))

// Force / moment spaces and closed-loop flags of robot i (SpaceBits): its row of the per-robot space block
// (osc_mft_parametrize_spaces_batched), or, for a task without one, its parameters.
template <typename IDX>
DEVI int32_t mft_space_mode(const DevMft& t, IDX i) {
	const osc_mft_params& p = t.p;
	return t.space_mode ? t.space_mode[i]
						: space_mode_word(p.force_space_dimension, p.moment_space_dimension, p.closed_loop_force_control != 0, p.closed_loop_moment_control != 0);
}
// the force / motion and moment / rot-motion axes of robot i as parametrised (compliant frame or world axes)
template <typename IDX>
DEVI void mft_space_axes(const DevMft& t, IDX NR, IDX i, double af[3], double am[3]) {
	const osc_mft_params& p = t.p;
#pragma unroll
	for (int k = 0; k < 3; k++) {
		af[k] = t.space_axes ? t.space_axes[(IDX)k * NR + i] : p.force_or_motion_axis[k];
		am[k] = t.space_axes ? t.space_axes[(IDX)(3 + k) * NR + i] : p.moment_or_rotmotion_axis[k];
	}
}

DEVI void scale_to_norm(double v[3], double maxn) {
	const double n = sqrt(dot3(v, v));
	if (n > maxn) {
		const double s = maxn / n;
		v[0] *= s;
		v[1] *= s;
		v[2] *= s;
	}
}
// pseudo-inverse of a diagonal gain entry (SaiModel::computePseudoInverse of a diagonal matrix)
DEVI double pinv_gain(double k) { return (k > 1e-6) ? 1.0 / k : 0.0; }

// x, R: pose of the compliant frame in the world; v_in, w_in: J0 dq of the full (unprojected) Jacobian.
// Outputs the unit-mass force f* and the force-related terms F (world axes, 6 each); returns false when F is
// identically zero (pure motion control of a full task), so that callers can skip it.
// MOTION: the task is known (host check: mft_pure_motion) to be a full task under pure motion control without velocity
// saturation, so only the two PID laws are compiled in.
// sg != nullptr: the 24 goal components and the two motion integrators (30 doubles, components MC_GOAL_POS.. then
// MC_INT_POS, MC_INT_ORI) were staged into shared memory (element e at sg[e * sgs]) by mft_stage_goals.
template <typename IDX>
DEVI void mft_stage_goals(const DevMft& t, IDX NR, IDX i, double* sg, int sgs) {
	const gdouble* st = t.st;
#pragma unroll
	for (int c = 0; c < 24; c++) cp_async8(sg + c * sgs, &ST(MC_GOAL_POS, c));
#pragma unroll
	for (int c = 0; c < 6; c++) cp_async8(sg + (24 + c) * sgs, &ST(MC_INT_POS, c));
}
// G: where the gains come from (GainSrc).
template <bool MOTION = false, typename IDX = int64_t, int G = GAINS_ANY>
DEVI bool mft_control_law(const DevMft& t, IDX NR, IDX i, const double x[3], const double R[9], const double v_in[3],
						  const double w_in[3], bool write_observers, double fstar[6], double F[6], uint32_t& status,
						  const double* sg = nullptr, int sgs = 0) {
	gdouble* st = t.st;
	const osc_mft_params& p = t.p;
	const double dt = t.dt;
	// per-robot gains: requested first (the fused kernel prefetched their rows into L2); pure motion control reads the motion ones only
	double kg[GAIN_COUNT];
	load_gain_block<G>(t.gains, reinterpret_cast<const double*>(&p), NR, i, 0, MOTION ? MG_KP_FORCE : GAIN_COUNT, kg);
	double v[3] = {v_in[0], v_in[1], v_in[2]}, w[3] = {w_in[0], w_in[1], w_in[2]};
	if (!MOTION && !t.full) {	// _jacobian = P * J0  (MotionForceTask.cpp:280-282, 293-298)
		double tv[3], tw[3];
		mat3_vec(t.Pt, v, tv);
		mat3_vec(t.Pr, w, tw);
#pragma unroll
		for (int k = 0; k < 3; k++) {
			v[k] = tv[k];
			w[k] = tw[k];
		}
	}
	double xd[3], Rd[9], vd[3], wd[3], ad[3], ald[3];
	if (MOTION && sg) {
		cp_async_wait_all();
#pragma unroll
		for (int k = 0; k < 3; k++) {
			xd[k] = sg[(MC_GOAL_POS + k) * sgs];
			vd[k] = sg[(MC_GOAL_LINVEL + k) * sgs];
			wd[k] = sg[(MC_GOAL_ANGVEL + k) * sgs];
			ad[k] = sg[(MC_GOAL_LINACC + k) * sgs];
			ald[k] = sg[(MC_GOAL_ANGACC + k) * sgs];
		}
#pragma unroll
		for (int k = 0; k < 9; k++) Rd[k] = sg[(MC_GOAL_ORI + k) * sgs];
	} else {
		load3(st, NR, i, MC_GOAL_POS, xd);
#pragma unroll
		for (int k = 0; k < 9; k++) Rd[k] = ST(MC_GOAL_ORI, k);
		load3(st, NR, i, MC_GOAL_LINVEL, vd);
		load3(st, NR, i, MC_GOAL_ANGVEL, wd);
		load3(st, NR, i, MC_GOAL_LINACC, ad);
		load3(st, NR, i, MC_GOAL_ANGACC, ald);
	}

	double ori_err_goal[3];
	orientation_error(Rd, R, ori_err_goal);	 // :291-292 (desired == goal with OTG off)

	// Pure motion control of a full task (no force/moment space, open loop): every sigma is 0 or the identity
	// (MotionForceTask.cpp:892-971), the force-related terms vanish and only the two PID laws remain.  MOTION: known for every
	// robot (host check); otherwise decided per robot from its mode word (a word of 0 is pure motion control).
	const int32_t mode = MOTION ? 0 : mft_space_mode(t, i);
	if (MOTION || (t.full && mode == 0)) {
		double Ip[3], Io[3];
		if (MOTION && sg) {
#pragma unroll
			for (int k = 0; k < 3; k++) {
				Ip[k] = sg[(24 + k) * sgs];
				Io[k] = sg[(27 + k) * sgs];
			}
		} else {
			load3(st, NR, i, MC_INT_POS, Ip);
			load3(st, NR, i, MC_INT_ORI, Io);
		}
#pragma unroll
		for (int k = 0; k < 3; k++) {
			const double ex = x[k] - xd[k];
			Ip[k] += ex * dt;
			Io[k] += ori_err_goal[k] * dt;
			if (MOTION || !p.use_velocity_saturation) {
				fstar[k] = ad[k] - OSC_GAIN(kp_pos, MG_KP_POS, k) * ex - OSC_GAIN(kv_pos, MG_KV_POS, k) * (v[k] - vd[k]) - OSC_GAIN(ki_pos, MG_KI_POS, k) * Ip[k];
				fstar[3 + k] = ald[k] - OSC_GAIN(kp_ori, MG_KP_ORI, k) * ori_err_goal[k] - OSC_GAIN(kv_ori, MG_KV_ORI, k) * (w[k] - wd[k]) - OSC_GAIN(ki_ori, MG_KI_ORI, k) * Io[k];
			}
			F[k] = 0.0;
			F[3 + k] = 0.0;
		}
		if (!MOTION && p.use_velocity_saturation) {
			double vdes[3], wdes[3];
#pragma unroll
			for (int k = 0; k < 3; k++) {
				const double kvi = pinv_gain(OSC_GAIN(kv_pos, MG_KV_POS, k)), kwi = pinv_gain(OSC_GAIN(kv_ori, MG_KV_ORI, k));
				vdes[k] = -OSC_GAIN(kp_pos, MG_KP_POS, k) * kvi * (x[k] - xd[k]) - OSC_GAIN(ki_pos, MG_KI_POS, k) * kvi * Ip[k];
				wdes[k] = -OSC_GAIN(kp_ori, MG_KP_ORI, k) * kwi * ori_err_goal[k] - OSC_GAIN(ki_ori, MG_KI_ORI, k) * kwi * Io[k];
			}
			scale_to_norm(vdes, p.linear_saturation_velocity);
			scale_to_norm(wdes, p.angular_saturation_velocity);
#pragma unroll
			for (int k = 0; k < 3; k++) {
				fstar[k] = ad[k] - OSC_GAIN(kv_pos, MG_KV_POS, k) * (v[k] - vdes[k]);
				fstar[3 + k] = ald[k] - OSC_GAIN(kv_ori, MG_KV_ORI, k) * (w[k] - wdes[k]);
			}
		}
		store3(st, NR, i, MC_INT_POS, Ip);
		store3(st, NR, i, MC_INT_ORI, Io);
		store3(st, NR, i, MC_CUR_POS, x);
#pragma unroll
		for (int k = 0; k < 9; k++) ST(MC_CUR_ORI, k) = R[k];
		if (write_observers) {
			store3(st, NR, i, MC_CUR_LINVEL, v);
			store3(st, NR, i, MC_CUR_ANGVEL, w);
			store3(st, NR, i, MC_ORI_ERROR, ori_err_goal);
#pragma unroll
			for (int k = 0; k < 6; k++) ST(MC_UNIT_MASS_FORCE, k) = fstar[k];
		}
		return false;
	}

	if constexpr (MOTION) return false;
	// selection matrices
	const double I3[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
	const bool cl_force = (mode & SP_CL_FORCE) != 0, cl_moment = (mode & SP_CL_MOMENT) != 0;
	double uf[3], um[3];
	{
		double af[3], am[3];
		mft_space_axes(t, NR, i, af, am);
		if (t.in_compliant) {
			mat3_vec(R, af, uf);
			mat3_vec(R, am, um);
		} else {
#pragma unroll
			for (int k = 0; k < 3; k++) {
				uf[k] = af[k];
				um[k] = am[k];
			}
		}
	}
	double Sf[9], Sm[9], Sp[9], So[9];
	sigma_space((mode >> SP_FDIM_SHIFT) & 3, t.Pt, uf, Sf);
	sigma_space((mode >> SP_MDIM_SHIFT) & 3, t.Pr, um, Sm);
	sigma_complement(t.Pt, Sf, Sp);
	sigma_complement(t.Pr, Sm, So);

	double gf_raw[3] = {0, 0, 0}, gm_raw[3] = {0, 0, 0}, gf[3], gm[3];
	const bool any_force = mode != 0;
	if (any_force) {
		load3(st, NR, i, MC_GOAL_FORCE, gf_raw);
		load3(st, NR, i, MC_GOAL_MOMENT, gm_raw);
	}
	if (t.in_compliant) {  // getGoalForce / getGoalMoment :755-769
		mat3_vec(R, gf_raw, gf);
		mat3_vec(R, gm_raw, gm);
	} else {
#pragma unroll
		for (int k = 0; k < 3; k++) {
			gf[k] = gf_raw[k];
			gm[k] = gm_raw[k];
		}
	}

	double force_fb[3], moment_fb[3];
	// ---- force ----  :327-354
	if (cl_force) {
		double fs[3], If[3], e[3], se[3];
		load3(st, NR, i, MC_SENSED_F, fs);
		load3(st, NR, i, MC_INT_FORCE, If);
#pragma unroll
		for (int k = 0; k < 3; k++) e[k] = fs[k] - gf[k];
		mat3_vec(Sf, e, se);
#pragma unroll
		for (int k = 0; k < 3; k++) If[k] += se[k] * dt;
		store3(st, NR, i, MC_INT_FORCE, If);
		double pre[3], fb[3];
#pragma unroll
		for (int k = 0; k < 3; k++) pre[k] = -OSC_GAIN1(kp_force, MG_KP_FORCE) * e[k] - OSC_GAIN1(ki_force, MG_KI_FORCE) * If[k];
		mat3_vec(Sf, pre, fb);
		scale_to_norm(fb, p.max_force_control_feedback_output);
		double a_fd[3], a_fs[3], a_vcl[3], a_vr[3];
		mat3_vec(Sf, gf, a_fd);
		mat3_vec(Sf, fs, a_fs);
		mat3_vec(Sf, fb, a_vcl);
		mat3_vec(Sf, v, a_vr);
		popc_step(t, NR, i, a_fd, a_fs, a_vcl, a_vr, OSC_GAIN1(kv_force, MG_KV_FORCE), p.kff_force, force_fb, status);
	} else {
		double pre[3] = {-OSC_GAIN1(kv_force, MG_KV_FORCE) * v[0], -OSC_GAIN1(kv_force, MG_KV_FORCE) * v[1], -OSC_GAIN1(kv_force, MG_KV_FORCE) * v[2]};
		mat3_vec(Sf, pre, force_fb);
	}
	// ---- moment ----  :357-383
	if (cl_moment) {
		double ms[3], Im[3], e[3], se[3];
		load3(st, NR, i, MC_SENSED_M, ms);
		load3(st, NR, i, MC_INT_MOMENT, Im);
#pragma unroll
		for (int k = 0; k < 3; k++) e[k] = ms[k] - gm[k];
		mat3_vec(Sm, e, se);
#pragma unroll
		for (int k = 0; k < 3; k++) Im[k] += se[k] * dt;
		store3(st, NR, i, MC_INT_MOMENT, Im);
		double pre[3], mb[3];
#pragma unroll
		for (int k = 0; k < 3; k++) pre[k] = -OSC_GAIN1(kp_moment, MG_KP_MOMENT) * e[k] - OSC_GAIN1(ki_moment, MG_KI_MOMENT) * Im[k];
		mat3_vec(Sm, pre, mb);
		scale_to_norm(mb, p.max_moment_control_feedback_output);
#pragma unroll
		for (int k = 0; k < 3; k++) pre[k] = mb[k] - OSC_GAIN1(kv_moment, MG_KV_MOMENT) * w[k];
		mat3_vec(Sm, pre, moment_fb);
	} else {
		double pre[3] = {-OSC_GAIN1(kv_moment, MG_KV_MOMENT) * w[0], -OSC_GAIN1(kv_moment, MG_KV_MOMENT) * w[1], -OSC_GAIN1(kv_moment, MG_KV_MOMENT) * w[2]};
		mat3_vec(Sm, pre, moment_fb);
	}

	// ---- linear motion ----  :409-437
	double Ip[3], ex[3], sex[3];
	load3(st, NR, i, MC_INT_POS, Ip);
#pragma unroll
	for (int k = 0; k < 3; k++) ex[k] = x[k] - xd[k];
	mat3_vec(Sp, ex, sex);
#pragma unroll
	for (int k = 0; k < 3; k++) Ip[k] += sex[k] * dt;
	store3(st, NR, i, MC_INT_POS, Ip);
	double pos_force[3];
	if (p.use_velocity_saturation) {
		double vdes[3];
#pragma unroll
		for (int k = 0; k < 3; k++) {
			const double kvi = pinv_gain(OSC_GAIN(kv_pos, MG_KV_POS, k));
			vdes[k] = -OSC_GAIN(kp_pos, MG_KP_POS, k) * kvi * sex[k] - OSC_GAIN(ki_pos, MG_KI_POS, k) * kvi * Ip[k];
		}
		scale_to_norm(vdes, p.linear_saturation_velocity);
		double pre[3];
#pragma unroll
		for (int k = 0; k < 3; k++) pre[k] = ad[k] - OSC_GAIN(kv_pos, MG_KV_POS, k) * (v[k] - vdes[k]);
		mat3_vec(Sp, pre, pos_force);
	} else {
		double pre[3];
#pragma unroll
		for (int k = 0; k < 3; k++)
			pre[k] = ad[k] - OSC_GAIN(kp_pos, MG_KP_POS, k) * ex[k] - OSC_GAIN(kv_pos, MG_KV_POS, k) * (v[k] - vd[k]) - OSC_GAIN(ki_pos, MG_KI_POS, k) * Ip[k];
		mat3_vec(Sp, pre, pos_force);
	}
	// ---- angular motion ----  :439-468
	double Io[3], eo[3];
	load3(st, NR, i, MC_INT_ORI, Io);
	mat3_vec(So, ori_err_goal, eo);
#pragma unroll
	for (int k = 0; k < 3; k++) Io[k] += eo[k] * dt;
	store3(st, NR, i, MC_INT_ORI, Io);
	double ori_force[3];
	if (p.use_velocity_saturation) {
		double wdes[3];
#pragma unroll
		for (int k = 0; k < 3; k++) {
			const double kvi = pinv_gain(OSC_GAIN(kv_ori, MG_KV_ORI, k));
			wdes[k] = -OSC_GAIN(kp_ori, MG_KP_ORI, k) * kvi * eo[k] - OSC_GAIN(ki_ori, MG_KI_ORI, k) * kvi * Io[k];
		}
		scale_to_norm(wdes, p.angular_saturation_velocity);
		double pre[3];
#pragma unroll
		for (int k = 0; k < 3; k++) pre[k] = ald[k] - OSC_GAIN(kv_ori, MG_KV_ORI, k) * (w[k] - wdes[k]);
		mat3_vec(So, pre, ori_force);
	} else {
		double pre[3];
#pragma unroll
		for (int k = 0; k < 3; k++)
			pre[k] = ald[k] - OSC_GAIN(kp_ori, MG_KP_ORI, k) * eo[k] - OSC_GAIN(kv_ori, MG_KV_ORI, k) * (w[k] - wd[k]) - OSC_GAIN(ki_ori, MG_KI_ORI, k) * Io[k];
		mat3_vec(So, pre, ori_force);
	}
	// ---- assemble ----  :470-491
	double ff_f[3], ff_m[3];
	mat3_vec(Sf, gf, ff_f);
	mat3_vec(Sm, gm, ff_m);
	if (cl_force) {	 // keyed on the force flag only (:484-487)
#pragma unroll
		for (int k = 0; k < 3; k++) {
			ff_f[k] *= p.kff_force;
			ff_m[k] *= p.kff_moment;
		}
	}
#pragma unroll
	for (int k = 0; k < 3; k++) {
		fstar[k] = pos_force[k];
		fstar[3 + k] = ori_force[k];
		F[k] = force_fb[k] + ff_f[k];
		F[3 + k] = moment_fb[k] + ff_m[k];
	}
	// observers the reference keeps as members (_current_*, _orientation_error, _unit_mass_force)
	store3(st, NR, i, MC_CUR_POS, x);
#pragma unroll
	for (int k = 0; k < 9; k++) ST(MC_CUR_ORI, k) = R[k];
	if (write_observers) {
		store3(st, NR, i, MC_CUR_LINVEL, v);
		store3(st, NR, i, MC_CUR_ANGVEL, w);
		store3(st, NR, i, MC_ORI_ERROR, ori_err_goal);
#pragma unroll
		for (int k = 0; k < 6; k++) ST(MC_UNIT_MASS_FORCE, k) = fstar[k];
	}
	(void)I3;
	return true;
}

// JointTask PID in task coordinates: returns t (pid "torques") and the desired acceleration.
// e = S q - q_d etc.  (JointTask.cpp:299-346; Appendix C8: saturation loop uses the task dof)
// staged variant: goals (position, velocity, acceleration), integrator, q and dq of the robot, 6 N doubles, copied to
// shared memory ahead of time (element e at sg[e * sgs])
template <int N, typename IDX>
DEVI void joint_stage_goals(const DevJt& t, const gdouble* qg, const gdouble* dqg, IDX NR, IDX i, double* sg, int sgs) {
	const gdouble* st = t.st;
#pragma unroll
	for (int a = 0; a < N; a++) {
		cp_async8(sg + a * sgs, &ST(JC_GOAL_POS, a));
		cp_async8(sg + (N + a) * sgs, &ST(JC_GOAL_VEL, a));
		cp_async8(sg + (2 * N + a) * sgs, &ST(JC_GOAL_ACC, a));
		cp_async8(sg + (3 * N + a) * sgs, &ST(JC_INT, a));
		cp_async8(sg + (4 * N + a) * sgs, qg + (IDX)a * NR + i);
		cp_async8(sg + (5 * N + a) * sgs, dqg + (IDX)a * NR + i);
	}
}
// full joint task without velocity saturation from the staged copy (the SPEC instantiation)
template <int N, typename IDX, int G = GAINS_ANY>
DEVI void joint_control_law_staged(const DevJt& t, IDX NR, IDX i, const double* sg, int sgs, double (&pid)[N], double (&acc)[N]) {
	gdouble* st = t.st;
	const osc_joint_params& p = t.p;
	double kg[GAIN_COUNT];
	load_gain_block<G>(t.gains, reinterpret_cast<const double*>(&p), NR, i, JG_KP, N, kg + JG_KP);
	load_gain_block<G>(t.gains, reinterpret_cast<const double*>(&p), NR, i, JG_KV, N, kg + JG_KV);
	load_gain_block<G>(t.gains, reinterpret_cast<const double*>(&p), NR, i, JG_KI, N, kg + JG_KI);
	cp_async_wait_all();
	double I[N];
#pragma unroll
	for (int a = 0; a < N; a++) {
		const double e = sg[(4 * N + a) * sgs] - sg[a * sgs];
		acc[a] = sg[(2 * N + a) * sgs];
		I[a] = sg[(3 * N + a) * sgs] + e * t.dt;
		pid[a] = -OSC_GAIN(kp, JG_KP, a) * e - OSC_GAIN(kv, JG_KV, a) * (sg[(5 * N + a) * sgs] - sg[(N + a) * sgs]) - OSC_GAIN(ki, JG_KI, a) * I[a];
	}
#pragma unroll
	for (int a = 0; a < N; a++) ST(JC_INT, a) = I[a];
}

template <int N, int K, bool SPEC = false, typename IDX = int64_t, int G = GAINS_ANY>  // SPEC: full selection, no velocity saturation (host check)
DEVI void joint_control_law(const DevJt& t, IDX NR, IDX i, const double (&q)[N], const double (&dq)[N],
							double (&pid)[K], double (&acc)[K]) {
	gdouble* st = t.st;
	const osc_joint_params& p = t.p;
	double kg[GAIN_COUNT];
	load_gain_block<G>(t.gains, reinterpret_cast<const double*>(&p), NR, i, JG_KP, K, kg + JG_KP);
	load_gain_block<G>(t.gains, reinterpret_cast<const double*>(&p), NR, i, JG_KV, K, kg + JG_KV);
	load_gain_block<G>(t.gains, reinterpret_cast<const double*>(&p), NR, i, JG_KI, K, kg + JG_KI);
	// all loads first, all stores last: the compiler cannot prove that the integrator stores do not alias the
	// following goal loads, and would otherwise serialise one memory round trip per task coordinate
	double gp[K], gv[K], I[K];
#pragma unroll
	for (int a = 0; a < K; a++) {
		gp[a] = ST(JC_GOAL_POS, a);
		gv[a] = ST(JC_GOAL_VEL, a);
		acc[a] = ST(JC_GOAL_ACC, a);
		I[a] = ST(JC_INT, a);
	}
#pragma unroll
	for (int a = 0; a < K; a++) {
		double pos, vel;
		if (SPEC || t.full) {
			pos = q[a];
			vel = dq[a];
		} else {
			pos = 0.0;
			vel = 0.0;
#pragma unroll
			for (int j = 0; j < N; j++) {
				pos += t.S[a][j] * q[j];
				vel += t.S[a][j] * dq[j];
			}
		}
		const double e = pos - gp[a];
		I[a] += e * t.dt;
		if (!SPEC && p.use_velocity_saturation) {
			const double kvi = pinv_gain(OSC_GAIN(kv, JG_KV, a));
			double vdes = -OSC_GAIN(kp, JG_KP, a) * kvi * e - OSC_GAIN(ki, JG_KI, a) * kvi * I[a];
			if (vdes > p.saturation_velocity[a])
				vdes = p.saturation_velocity[a];
			else if (vdes < -p.saturation_velocity[a])
				vdes = -p.saturation_velocity[a];
			pid[a] = -OSC_GAIN(kv, JG_KV, a) * (vel - vdes);
		} else {
			pid[a] = -OSC_GAIN(kp, JG_KP, a) * e - OSC_GAIN(kv, JG_KV, a) * (vel - gv[a]) - OSC_GAIN(ki, JG_KI, a) * I[a];
		}
	}
#pragma unroll
	for (int a = 0; a < K; a++) ST(JC_INT, a) = I[a];
}

// Same law with a run-time task dimension (general hierarchies, osc_singular.cuh)
template <int N>
static __device__ __noinline__ void joint_control_law_rt(const DevJt& t, int64_t NR, int64_t i, const double (&q)[N], const double (&dq)[N], int k,
														  double* pid, double* acc) {
	gdouble* st = t.st;
	const osc_joint_params& p = t.p;
	constexpr int G = GAINS_ANY;
	using IDX = int64_t;
	double* kg = nullptr;  // unused with GAINS_ANY
	for (int a = 0; a < k; a++) {
		double pos = 0.0, vel = 0.0;
		for (int j = 0; j < N; j++) {
			pos += t.S[a][j] * q[j];
			vel += t.S[a][j] * dq[j];
		}
		const double e = pos - ST(JC_GOAL_POS, a);
		const double vd = ST(JC_GOAL_VEL, a);
		acc[a] = ST(JC_GOAL_ACC, a);
		double I = ST(JC_INT, a);
		I += e * t.dt;
		ST(JC_INT, a) = I;
		if (p.use_velocity_saturation) {
			const double kvi = pinv_gain(OSC_GAIN(kv, JG_KV, a));
			double vdes = -OSC_GAIN(kp, JG_KP, a) * kvi * e - OSC_GAIN(ki, JG_KI, a) * kvi * I;
			if (vdes > p.saturation_velocity[a])
				vdes = p.saturation_velocity[a];
			else if (vdes < -p.saturation_velocity[a])
				vdes = -p.saturation_velocity[a];
			pid[a] = -OSC_GAIN(kv, JG_KV, a) * (vel - vdes);
		} else {
			pid[a] = -OSC_GAIN(kp, JG_KP, a) * e - OSC_GAIN(kv, JG_KV, a) * (vel - vd) - OSC_GAIN(ki, JG_KI, a) * I;
		}
	}
}

#undef OSC_GAIN
#undef OSC_GAIN1
#undef ST
}  // namespace osc
