// The optional FP32 mode of the north star: the fused control-cycle kernel of the flagship hierarchy instantiated in single
// precision.  The kernel source is the FP64 one (osc_cycle.cuh and the headers under it) passed through gen_fp32.py; the data
// in global memory (inputs, task state, torques) stay FP64, so robots the kernel hands over continue on the FP64 general path.
#include "osc_dev_types.h"
#include "osc_launch.h"
#include <utility>
#define OSC_FP32_BUILD 1
#define OSC_MIN_BLOCKS 3  // 168 registers, 54 KB of shared memory per block: three blocks (12 warps) per SM; four (128 registers) measured 4-8 % slower
#include "fp32/osc_types32.h"
#include "fp32/osc_cycle.cuh"

namespace osc {

// the single-precision kernel of word v: one instantiation per word of its list (cycle_words, osc_launch.h)
template <int N, bool JT, size_t... I>
static cudaError_t launch_f32(unsigned v, const osc32::OscProgram& P32, cudaStream_t stream, std::index_sequence<I...>) {
	constexpr CycleWordList L = cycle_words(6, true);
	cudaError_t e = cudaErrorNotSupported;
	(void)((v == L.word[I] && ((e = launch_fused_kernel<osc32::osc_cycle_kernel<N, 6, JT, L.word[I]>>(
										P32, osc32::cycle_smem_doubles<N, 6, L.word[I]>() * kCycleBlock * (int)sizeof(float), stream)),
								true)) ||
		   ...);
	return e;
}

cudaError_t launch_cycle_fused_f32(int n, bool has_jt, unsigned word, const OscProgram& P, cudaStream_t stream) {
	osc32::OscProgram P32;
	osc32::to_f32(P, P32);
	constexpr auto seq = std::make_index_sequence<cycle_words(6, true).count>{};
#define OSC_F32_CASE(NN) \
	if (n == NN) return has_jt ? launch_f32<NN, true>(word & ~CV_F32, P32, stream, seq) : launch_f32<NN, false>(word & ~CV_F32, P32, stream, seq);
	OSC_F32_DOFS(OSC_F32_CASE)
#undef OSC_F32_CASE
	return cudaErrorNotSupported;
}

}  // namespace osc
