// Instantiations of the fused cycle kernel, one translation unit per robot dof (OSC_INST_N)
// so that nvcc compiles them in parallel.
#include "osc_cycle.cuh"
#include "osc_singular.cuh"
#include "osc_blend.cuh"
#include "osc_launch.h"
#include <algorithm>
#include <atomic>
#include <cmath>
#include <utility>
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

template <int N, int R, bool JT, unsigned V>
static cudaError_t launch_fused(const OscProgram& P, cudaStream_t stream) {
	constexpr int smem = cycle_smem_doubles<N, R, V>() * kCycleBlock * (int)sizeof(double);
#if defined(OSC_TRACE)
	const unsigned grid = (unsigned)((P.n_robots + kCycleBlock - 1) / kCycleBlock);
	static unsigned long long* d_trace = nullptr;
	const size_t tbytes = (size_t)grid * 32 * 2 * sizeof(unsigned long long);
	if (!d_trace) {
		cudaMalloc(&d_trace, (size_t)1 << 26);
		cudaMemcpyToSymbol(g_trace, &d_trace, sizeof(d_trace));
	}
	cudaMemsetAsync(d_trace, 0, tbytes, stream);
#endif
	cudaError_t e = launch_fused_kernel<osc_cycle_kernel<N, R, JT, V>>(P, smem, stream);
	if (e != cudaSuccess) return e;
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

// the fused kernel of the planned word: one instantiation per word of the signature's list (cycle_words, osc_launch.h)
template <int N, int R, bool JT, size_t... I>
static cudaError_t launch_listed(unsigned v, const OscProgram& P, cudaStream_t stream, std::index_sequence<I...>) {
	constexpr CycleWordList L = cycle_words(R);
	cudaError_t e = cudaErrorNotSupported;
	(void)((v == L.word[I] && ((e = launch_fused<N, R, JT, L.word[I]>(P, stream)), true)) || ...);
	return e;
}

template <int N, int R, bool JT>
static cudaError_t launch_one(const CyclePlan& plan, const OscProgram& P, cudaStream_t stream) {
	const cudaError_t e0 = (plan.fused & CV_F32) ? launch_cycle_fused_f32(N, JT, plan.fused, P, stream)
												: launch_listed<N, R, JT>(plan.fused, P, stream, std::make_index_sequence<cycle_words(R).count>{});
	if (e0 != cudaSuccess) return e0;
	if (plan.general != GeneralPath::None) {
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
			if (plan.general == GeneralPath::BlendSplit) {
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
			if (plan.general == GeneralPath::Blend) return cudaLaunchKernelEx(&cfg, osc_blend_kernel<N, JT>, P);
		}
		return cudaLaunchKernelEx(&cfg, osc_singular_kernel<N>, P);
	}
	return cudaGetLastError();
}

// motion-force task of rank R (1..min(6,N)), with or without a closing full joint task
template <int N, int R>
static cudaError_t launch_rank(bool has_jt, const CyclePlan& plan, const OscProgram& P, cudaStream_t stream) {
	if constexpr (R >= 1 && R <= N && R <= 6 && OSC_ONLY_R != 0) {
		if constexpr (R == OSC_ONLY_R) return has_jt ? launch_one<N, R, true>(plan, P, stream) : cudaErrorNotSupported;
		return cudaErrorNotSupported;
	} else if constexpr (R >= 1 && R <= N && R <= 6) {
		return has_jt ? launch_one<N, R, true>(plan, P, stream) : launch_one<N, R, false>(plan, P, stream);
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

cudaError_t CONCAT(launch_cycle_n, OSC_INST_N)(int R, bool has_jt, const CyclePlan& plan, const OscProgram& P, cudaStream_t stream) {
	constexpr int N = OSC_INST_N;
	if (R < 0) return launch_generic<N>(P, stream);	 // general hierarchy: every robot on the general path
	switch (R) {
		case 0:
			if constexpr (OSC_ONLY_R != 0) return cudaErrorNotSupported;
			else return has_jt ? launch_one<N, 0, true>(plan, P, stream) : cudaErrorNotSupported;
		case 1: return launch_rank<N, 1>(has_jt, plan, P, stream);
		case 2: return launch_rank<N, 2>(has_jt, plan, P, stream);
		case 3: return launch_rank<N, 3>(has_jt, plan, P, stream);
		case 4: return launch_rank<N, 4>(has_jt, plan, P, stream);
		case 5: return launch_rank<N, 5>(has_jt, plan, P, stream);
		case 6: return launch_rank<N, 6>(has_jt, plan, P, stream);
	}
	return cudaErrorNotSupported;
}

}  // namespace osc
