#include "osc_aux_kernels.cuh"
#include "osc_observers.cuh"
#include "osc_otg_kernels.cuh"
#include "osc_space_kernels.cuh"
#include "osc_launch.h"

namespace osc {

static inline dim3 grid_for(int64_t n, int block) { return dim3((unsigned)((n + block - 1) / block)); }

#define DISPATCH_N(n, CALL)                  \
	switch (n) {                             \
		case 1: { constexpr int N_ = 1; CALL; } break; \
		case 2: { constexpr int N_ = 2; CALL; } break; \
		case 3: { constexpr int N_ = 3; CALL; } break; \
		case 4: { constexpr int N_ = 4; CALL; } break; \
		case 5: { constexpr int N_ = 5; CALL; } break; \
		case 6: { constexpr int N_ = 6; CALL; } break; \
		case 7: { constexpr int N_ = 7; CALL; } break; \
		case 8: { constexpr int N_ = 8; CALL; } break; \
		default: return cudaErrorInvalidValue;         \
	}

cudaError_t launch_reset_robots(const OscProgram& P, const int32_t* mask, int task, int construct, cudaStream_t stream) {
	DISPATCH_N(P.model.n, (reset_robots_kernel<N_><<<grid_for(P.n_robots, 128), 128, 0, stream>>>(P, mask, task, construct)));
	return cudaGetLastError();
}
cudaError_t launch_popc_probe(const OscProgram& P, int mft_index, int K, const double* fd, const double* fs, const double* vcl, const double* vr,
							  double kv, double kff, double* out, cudaStream_t stream) {
	popc_probe_kernel<<<grid_for(P.n_robots, 128), 128, 0, stream>>>(P, mft_index, K, fd, fs, vcl, vr, kv, kff, out);
	return cudaGetLastError();
}
cudaError_t measure_fp64_peak(double seconds, double* tflops, cudaStream_t stream) {
	int dev = 0, sms = 0;
	cudaGetDevice(&dev);
	cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
	double* out = nullptr;
	cudaError_t e = cudaMalloc(&out, sizeof(double));
	if (e != cudaSuccess) return e;
	cudaEvent_t e0, e1;
	cudaEventCreate(&e0);
	cudaEventCreate(&e1);
	const int grid = sms * 2, block = 1024, iters = 2048;	// 2 x 32 warps per SM
	const double flop_per_launch = 2.0 * 128.0 * iters * (double)grid * block;
	double best = 0.0, spent = 0.0;
	for (int rep = 0; rep < 10000 && spent < seconds; rep++) {
		cudaEventRecord(e0, stream);
		fp64_peak_kernel<<<grid, block, 0, stream>>>(out, 1.0000001, 1e-9, iters);
		cudaEventRecord(e1, stream);
		e = cudaEventSynchronize(e1);
		if (e != cudaSuccess) break;
		float ms = 0.f;
		cudaEventElapsedTime(&ms, e0, e1);
		spent += ms * 1e-3;
		const double t = flop_per_launch / (ms * 1e-3) / 1e12;
		if (spent > 0.5 * seconds && t > best) best = t;	// the second half: clocks have settled under load
	}
	cudaEventDestroy(e0);
	cudaEventDestroy(e1);
	cudaFree(out);
	*tflops = best;
	return e == cudaSuccess ? cudaGetLastError() : e;
}
cudaError_t launch_sim_integrate(const OscProgram& P, double* q, double* dq, const double* tau, double dt, int substeps, cudaStream_t stream) {
	DISPATCH_N(P.model.n, (sim_integrate_kernel<N_><<<grid_for(P.n_robots, 128), 128, 0, stream>>>(P, q, dq, tau, dt, substeps)));
	return cudaGetLastError();
}
cudaError_t launch_jla(const OscProgram& P, cudaStream_t stream) {
	DevJla jp;	// JointLimitAvoidanceTask.h:26-35
	jp.kv = 20.0;
	jp.position_z1_to_limit = 9.0 * 3.14159265358979323846 / 180.0;
	jp.position_z2_to_limit = 6.0 * 3.14159265358979323846 / 180.0;
	jp.velocity_z1_to_limit = 0.5;
	jp.velocity_z2_to_limit = 0.3;
	jp.max_torque_ratio_pos_limit = 1.0;
	jp.max_torque_ratio_vel_limit = 0.05;
	DISPATCH_N(P.model.n, (jla_kernel<N_><<<grid_for(P.n_robots, 128), 128, 0, stream>>>(P, jp)));
	return cudaGetLastError();
}
cudaError_t launch_otg_update(const OscProgram& P, cudaStream_t stream) {
	otg_update_kernel<<<grid_for(P.n_robots, 64), 64, 0, stream>>>(P);
	return cudaGetLastError();
}
cudaError_t launch_otg_init(const OscProgram& P, int task, int mode, cudaStream_t stream) {
	DISPATCH_N(P.model.n, (otg_init_kernel<N_><<<grid_for(P.n_robots, 64), 64, 0, stream>>>(P, task, mode)));
	return cudaGetLastError();
}
cudaError_t launch_otg_disable(const OscProgram& P, int task, cudaStream_t stream) {
	otg_disable_kernel<<<grid_for(P.n_robots, 64), 64, 0, stream>>>(P, task);
	return cudaGetLastError();
}
cudaError_t launch_observer(const OscProgram& P, int task, int kind, double* out, cudaStream_t stream) {
	DISPATCH_N(P.model.n, (osc_observer_kernel<N_><<<grid_for(P.n_robots, 64), 64, 0, stream>>>(P, task, kind, out)));
	return cudaGetLastError();
}
cudaError_t launch_sensed_wrench(const OscProgram& P, int mft_index, const double* f, const double* m, cudaStream_t stream) {
	DISPATCH_N(P.model.n, (sensed_wrench_kernel<N_><<<grid_for(P.n_robots, 128), 128, 0, stream>>>(P, mft_index, f, m)));
	return cudaGetLastError();
}
cudaError_t launch_eval_model(const OscProgram& P, const osc_link_frame& frame, double* M, double* J, double* x, double* R,
							  double* g, cudaStream_t stream) {
	EvalOut out{M, J, x, R, g};
	DISPATCH_N(P.model.n, (eval_model_kernel<N_><<<grid_for(P.n_robots, 128), 128, 0, stream>>>(P, frame, out)));
	return cudaGetLastError();
}
cudaError_t launch_fill(double* st, int64_t NR, int comp, int ncomp, const double* vals, cudaStream_t stream) {
	if (ncomp > 16) return cudaErrorInvalidValue;
	FillVals v;
	for (int c = 0; c < 16; c++) v.v[c] = (c < ncomp) ? vals[c] : 0.0;
	fill_components_kernel<<<grid_for(NR, 256), 256, 0, stream>>>(st, NR, comp, ncomp, v);
	return cudaGetLastError();
}
cudaError_t launch_copy(double* st, int64_t NR, int dst, int src, int ncomp, cudaStream_t stream) {
	copy_components_kernel<<<grid_for(NR, 256), 256, 0, stream>>>(st, NR, dst, src, ncomp);
	return cudaGetLastError();
}
cudaError_t launch_check_values(const double* v, int64_t n, int32_t* bad, cudaStream_t stream) {
	const int64_t want = (n + 255) / 256;
	check_values_kernel<<<(unsigned)(want < 1024 ? (want > 0 ? want : 1) : 1024), 256, 0, stream>>>(v, n, bad);
	return cudaGetLastError();
}
cudaError_t launch_check_spaces(const int32_t* dims, const double* axes, const int32_t* flags, int64_t n, int32_t* out, cudaStream_t stream) {
	const int64_t want = (n + 255) / 256;
	check_spaces_kernel<<<(unsigned)(want < 1024 ? (want > 0 ? want : 1) : 1024), 256, 0, stream>>>(dims, axes, flags, n, out);
	return cudaGetLastError();
}
cudaError_t launch_apply_spaces(const OscProgram& P, int mft_index, int moment, const int32_t* dims, const double* axes, int dim,
								const double axis[3], int32_t* was_reset, int32_t* any_reset, cudaStream_t stream) {
	SpaceArgs a{dims, axes, dim, {axis[0], axis[1], axis[2]}, was_reset, any_reset};
	apply_spaces_kernel<<<grid_for(P.n_robots, 64), 64, 0, stream>>>(P, mft_index, moment, a);
	return cudaGetLastError();
}
cudaError_t launch_set_closed_loop(const OscProgram& P, int mft_index, int moment, const int32_t* flags, int flag, cudaStream_t stream) {
	set_closed_loop_kernel<<<grid_for(P.n_robots, 256), 256, 0, stream>>>(P, mft_index, moment, flags, flag);
	return cudaGetLastError();
}
cudaError_t launch_get_spaces(const OscProgram& P, int mft_index, int moment, int32_t* dims, double* axes, int32_t* closed_loop, cudaStream_t stream) {
	get_spaces_kernel<<<grid_for(P.n_robots, 256), 256, 0, stream>>>(P, mft_index, moment, dims, axes, closed_loop);
	return cudaGetLastError();
}
cudaError_t launch_fill_int(int32_t* ist, int64_t NR, int comp, int ncomp, int32_t value, cudaStream_t stream) {
	fill_int_components_kernel<<<grid_for(NR, 256), 256, 0, stream>>>(ist, NR, comp, ncomp, value);
	return cudaGetLastError();
}

}  // namespace osc
