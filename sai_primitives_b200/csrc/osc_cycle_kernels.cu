// Instantiations of the fused cycle kernel, one translation unit per robot dof (OSC_INST_N)
// so that nvcc compiles them in parallel.
#include "osc_cycle.cuh"
#include "osc_singular.cuh"
#include "osc_blend.cuh"
#include "osc_launch.h"
#include <algorithm>
#include <atomic>
#include <cmath>
#if defined(OSC_TRACE)
#include <cstdio>
#include <cstdlib>
#include <vector>
#endif

#ifndef OSC_INST_N
#error "compile with -DOSC_INST_N=<dof>"
#endif

// OSC_ONLY_R=<r> (tuning builds only): instantiate just the [MotionForceTask rank r, JointTask] kernel
#ifndef OSC_ONLY_R
#define OSC_ONLY_R 0
#endif

namespace osc {

// multiprocessors of the current device (cached per device)
static int sm_count() {
	static std::atomic<int> cached[64];
	int dev = 0;
	cudaGetDevice(&dev);
	if (dev < 0 || dev >= 64) dev = 0;
	int v = cached[dev].load(std::memory_order_relaxed);
	if (v == 0) {
		cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
		if (v <= 0) v = 148;
		cached[dev].store(v, std::memory_order_relaxed);
	}
	return v;
}

template <int N, int R, bool JT, bool FULL, bool SPEC = false, bool GRAV = false, bool MOTION = SPEC, bool PARK = false, bool PRG = false>
static cudaError_t launch_variant(const OscProgram& P, cudaStream_t stream) {
	const unsigned grid = (unsigned)((P.n_robots + kCycleBlock - 1) / kCycleBlock);
	constexpr int smem = cycle_smem_doubles<N, R, SPEC, MOTION>() * kCycleBlock * (int)sizeof(double);
	// per device: function attributes belong to the device's context.  Atomic flags: host threads driving different handles
	// may get here at the same time (setting the attribute twice is harmless, a torn read of a plain bool is not defined).
	static std::atomic<bool> configured[64];
	int dev = 0;
	cudaGetDevice(&dev);
	if (dev < 0 || dev >= 64 || !configured[dev].load(std::memory_order_acquire)) {
		cudaError_t e = cudaFuncSetAttribute(osc_cycle_kernel<N, R, JT, FULL, SPEC, GRAV, MOTION, PARK, PRG>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
		if (e != cudaSuccess) return e;
		if (dev >= 0 && dev < 64) configured[dev].store(true, std::memory_order_release);
	}
#if defined(OSC_TRACE)
	static unsigned long long* d_trace = nullptr;
	const size_t tbytes = (size_t)grid * 32 * 2 * sizeof(unsigned long long);
	if (!d_trace) {
		cudaMalloc(&d_trace, (size_t)1 << 26);
		cudaMemcpyToSymbol(g_trace, &d_trace, sizeof(d_trace));
	}
	cudaMemsetAsync(d_trace, 0, tbytes, stream);
#endif
	{
		cudaLaunchConfig_t cfg{};
		cfg.gridDim = dim3(grid);
		cfg.blockDim = dim3(kCycleBlock);
		cfg.dynamicSmemBytes = smem;
		cfg.stream = stream;
		cudaLaunchAttribute attr[1];
		attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
		attr[0].val.programmaticStreamSerializationAllowed = 1;
		cfg.attrs = attr;
		cfg.numAttrs = 1;
		cudaError_t e = cudaLaunchKernelEx(&cfg, osc_cycle_kernel<N, R, JT, FULL, SPEC, GRAV, MOTION, PARK, PRG>, P);
		if (e != cudaSuccess) return e;
	}
#if defined(OSC_TRACE)
	if (const char* path = getenv("OSC_TRACE_FILE")) {
		cudaStreamSynchronize(stream);
		std::vector<unsigned long long> hbuf(tbytes / sizeof(unsigned long long));
		cudaMemcpy(hbuf.data(), d_trace, tbytes, cudaMemcpyDeviceToHost);
		if (FILE* f = fopen(path, "ab")) {
			unsigned long long hdr[2] = {0x4f53435452414345ull, (unsigned long long)grid};
			fwrite(hdr, sizeof(hdr), 1, f);
			fwrite(hbuf.data(), 1, tbytes, f);
			fclose(f);
		}
	}
#endif
	return cudaGetLastError();
}

template <int N, int R, bool JT>
static cudaError_t launch_one(const OscProgram& P, cudaStream_t stream) {
	cudaError_t e0;
	if constexpr (R == 6) {
		bool motion = false;
		const bool spec = cycle_spec_eligible(P, JT, &motion);
		// with many robots on the general path the hand-overs also park their kinematics and dynamics for the split blending path
		const bool park = P.mft[0].full && blend_split_selected(P);
		const bool prg = cycle_per_robot_gains(P, JT);
		if (P.precision_fp32) {
			// optional single-precision mode: only the specialised pure-motion kernel has an FP32 instantiation (osc_cycle_f32.cu)
			if (!(P.mft[0].full && spec && motion)) return cudaErrorNotSupported;
			e0 = launch_cycle_fused_f32(N, JT, P, stream);
		} else if (!P.mft[0].full)
			e0 = launch_variant<N, R, JT, false>(P, stream);
		else if (prg && cycle_prg_specialised(R, spec, motion)) {
			// per-robot gains: the pure-motion specialisation has its own instantiations (the others test the pointer at run time)
			if (!park)
				e0 = P.gravity_comp ? launch_variant<N, R, JT, true, true, true, true, false, true>(P, stream)
									: launch_variant<N, R, JT, true, true, false, true, false, true>(P, stream);
			else
				e0 = P.gravity_comp ? launch_variant<N, R, JT, true, true, true, true, true, true>(P, stream)
									: launch_variant<N, R, JT, true, true, false, true, true, true>(P, stream);
		} else if (prg && !park)
			e0 = launch_variant<N, R, JT, true>(P, stream);
		else if (prg)
			e0 = launch_variant<N, R, JT, true, false, false, false, true>(P, stream);
		else if (spec && motion && !park)
			e0 = P.gravity_comp ? launch_variant<N, R, JT, true, true, true>(P, stream) : launch_variant<N, R, JT, true, true, false>(P, stream);
		else if (spec && motion)
			e0 = P.gravity_comp ? launch_variant<N, R, JT, true, true, true, true, true>(P, stream) : launch_variant<N, R, JT, true, true, false, true, true>(P, stream);
		else if (spec && !park)	// full task with force / moment control or velocity saturation
			e0 = P.gravity_comp ? launch_variant<N, R, JT, true, true, true, false>(P, stream) : launch_variant<N, R, JT, true, true, false, false>(P, stream);
		else if (spec)
			e0 = P.gravity_comp ? launch_variant<N, R, JT, true, true, true, false, true>(P, stream) : launch_variant<N, R, JT, true, true, false, false, true>(P, stream);
		else if (!park)
			e0 = launch_variant<N, R, JT, true>(P, stream);
		else
			e0 = launch_variant<N, R, JT, true, false, false, false, true>(P, stream);
	} else if constexpr (R == 3) {
		// the other common shape: three controlled directions (position only, or a planar task), any control law
		bool motion = false;
		const bool spec = cycle_spec_eligible(P, JT, &motion);
		if (spec && cycle_per_robot_gains(P, JT) && cycle_prg_specialised(R, spec, motion))
			e0 = P.gravity_comp ? launch_variant<N, R, JT, false, true, true, false, false, true>(P, stream)
								: launch_variant<N, R, JT, false, true, false, false, false, true>(P, stream);
		else if (spec)
			e0 = P.gravity_comp ? launch_variant<N, R, JT, false, true, true, false>(P, stream) : launch_variant<N, R, JT, false, true, false, false>(P, stream);
		else
			e0 = launch_variant<N, R, JT, false>(P, stream);
	} else if constexpr (R == 0) {
		// a JointTask alone: per-robot gains have their own instantiation, the broadcast one reads the parameters
		e0 = cycle_per_robot_gains(P, JT) ? launch_variant<N, R, JT, false, false, false, false, false, true>(P, stream) : launch_variant<N, R, JT, false>(P, stream);
	} else {
		e0 = launch_variant<N, R, JT, false>(P, stream);
	}
	if (e0 != cudaSuccess) return e0;
	if constexpr (R > 0) {
#ifdef OSC_TUNE_SKIP_GENERAL
		return e0;	// tuning builds only: measure what the second launch costs when the hand-over list is empty
#endif
		// The general path for the robots the fast kernel handed over (usually none or few).  One block per SM,
		// grid-stride over the compacted list; launched with programmatic stream serialization so that its launch
		// latency overlaps the tail of the fast kernel (it waits on griddepcontrol.wait before reading the list).
		const long long want = (P.n_robots + 63) / 64;
		cudaLaunchConfig_t cfg{};
		const long long cover = (long long)sm_count() * OSC_GENERIC_MIN_BLOCKS;
		cfg.gridDim = dim3((unsigned)(P.general_grid_small ? 1 : (want < cover ? want : cover)));
		cfg.blockDim = dim3(64);
		cfg.dynamicSmemBytes = 0;
		cfg.stream = stream;
		cudaLaunchAttribute attr[1];
		attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
		attr[0].val.programmaticStreamSerializationAllowed = 1;
		cfg.attrs = attr;
		cfg.numAttrs = 1;
		if constexpr (R == 6) {
			// flagship hierarchy: unrolled blending path (osc_blend.cuh), general path only as its fallback
			if (P.mft[0].full && blend_split_selected(P)) {
				// hand-overs are expected (host hint): prefix / variants / fallback as three kernels, each grid-stride over
				// its list with as many blocks as the device holds at once
				const bool motion = mft_pure_motion(P.mft[0]);
				constexpr int vsmem = kBlendSmem ? blend_smem_doubles<N>() * kBlendBlock * (int)sizeof(double) : 0;
				static_assert(vsmem <= 48 * 1024, "variants kernel: dynamic shared memory beyond the default limit");
				static std::atomic<int> per_sm[64][3];
				int dev = 0;
				cudaGetDevice(&dev);
				int occ[3] = {0, 0, 0};
				for (int k = 0; k < 3; k++) {
					occ[k] = (dev >= 0 && dev < 64) ? per_sm[dev][k].load(std::memory_order_acquire) : 0;
					if (occ[k] == 0) {
						cudaError_t e = k == 0	 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[k], osc_blend_classify_kernel<N, JT>, 64, 0)
										: k == 1 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[k], osc_blend_variants_kernel<N, JT, false>, kBlendBlock, vsmem)
												 : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[k], osc_blend_variants_kernel<N, JT, true>, kBlendBlock, vsmem);
						if (e != cudaSuccess) return e;
						if (occ[k] < 1) occ[k] = 1;
						if (dev >= 0 && dev < 64) per_sm[dev][k].store(occ[k], std::memory_order_release);
					}
				}
				const unsigned fallback_grid = cfg.gridDim.x;
				long long g = (long long)sm_count() * occ[0];
				cfg.gridDim = dim3((unsigned)(want < g ? want : g));
				cudaError_t e = cudaLaunchKernelEx(&cfg, osc_blend_classify_kernel<N, JT>, P);
				if (e != cudaSuccess) return e;
				g = (long long)sm_count() * occ[motion ? 2 : 1];
				cfg.gridDim = dim3((unsigned)(want < g ? want : g));
				cfg.dynamicSmemBytes = vsmem;
				e = motion ? cudaLaunchKernelEx(&cfg, osc_blend_variants_kernel<N, JT, true>, P) : cudaLaunchKernelEx(&cfg, osc_blend_variants_kernel<N, JT, false>, P);
				if (e != cudaSuccess) return e;
				cfg.gridDim = dim3(fallback_grid);
				cfg.dynamicSmemBytes = 0;
				return cudaLaunchKernelEx(&cfg, osc_blend_fallback_kernel<N>, P);
			}
			if (P.mft[0].full) return cudaLaunchKernelEx(&cfg, osc_blend_kernel<N, JT>, P);
		}
		return cudaLaunchKernelEx(&cfg, osc_singular_kernel<N>, P);
	}
	return cudaGetLastError();
}

// motion-force task of rank R (1..min(6,N)), with or without a closing full joint task
template <int N, int R>
static cudaError_t launch_rank(bool has_jt, const OscProgram& P, cudaStream_t stream) {
	if constexpr (R >= 1 && R <= N && R <= 6 && OSC_ONLY_R != 0) {
		if constexpr (R == OSC_ONLY_R) return has_jt ? launch_one<N, R, true>(P, stream) : cudaErrorNotSupported;
		return cudaErrorNotSupported;
	} else if constexpr (R >= 1 && R <= N && R <= 6) {
		return has_jt ? launch_one<N, R, true>(P, stream) : launch_one<N, R, false>(P, stream);
	} else {
		return cudaErrorNotSupported;
	}
}

template <int N>
static cudaError_t launch_generic(const OscProgram& P, cudaStream_t stream) {
	const unsigned grid = (unsigned)((P.n_robots + 63) / 64);
	osc_generic_kernel<N><<<grid, 64, 0, stream>>>(P);
	return cudaGetLastError();
}

#define CONCAT_(a, b) a##b
#define CONCAT(a, b) CONCAT_(a, b)

cudaError_t CONCAT(launch_cycle_n, OSC_INST_N)(int R, bool has_jt, const OscProgram& P, cudaStream_t stream) {
	constexpr int N = OSC_INST_N;
	if (R < 0) return launch_generic<N>(P, stream);	 // general hierarchy: every robot on the general path
	switch (R) {
		case 0:
			if constexpr (OSC_ONLY_R != 0) return cudaErrorNotSupported;
			else return has_jt ? launch_one<N, 0, true>(P, stream) : cudaErrorNotSupported;
		case 1: return launch_rank<N, 1>(has_jt, P, stream);
		case 2: return launch_rank<N, 2>(has_jt, P, stream);
		case 3: return launch_rank<N, 3>(has_jt, P, stream);
		case 4: return launch_rank<N, 4>(has_jt, P, stream);
		case 5: return launch_rank<N, 5>(has_jt, P, stream);
		case 6: return launch_rank<N, 6>(has_jt, P, stream);
	}
	return cudaErrorNotSupported;
}

}  // namespace osc
