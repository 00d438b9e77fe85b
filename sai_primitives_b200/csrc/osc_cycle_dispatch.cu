#include "osc_launch.h"

namespace osc {
#define DECL(n) cudaError_t launch_cycle_n##n(int R, bool has_jt, const CyclePlan& plan, const OscProgram& P, cudaStream_t stream);
OSC_CYCLE_DOFS(DECL)
#undef DECL

bool cycle_signature_available(int n, int R, bool has_jt) {
	if (R > 6 || R > n) return false;
	if (R < 0) R = 1;  // general-hierarchy kernel: only the dof has to be compiled in
	if (R == 0 && !has_jt) return false;
#define CHECK(m) \
	if (n == m) return true;
	OSC_CYCLE_DOFS(CHECK)
#undef CHECK
	return false;
}

cudaError_t launch_cycle(int n, int R, bool has_jt, const CyclePlan& plan, const OscProgram& P, cudaStream_t stream) {
	if (!cycle_signature_available(n, R, has_jt) || plan.error != OSC_OK) return cudaErrorNotSupported;
#define CALL(m) \
	if (n == m) return launch_cycle_n##m(R, has_jt, plan, P, stream);
	OSC_CYCLE_DOFS(CALL)
#undef CALL
	return cudaErrorNotSupported;
}
}  // namespace osc
