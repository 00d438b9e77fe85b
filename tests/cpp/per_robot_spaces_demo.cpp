// Per-robot force / moment spaces through the batched C++ mirror: the example-05 hierarchy (MotionForceTask at end-effector
// (0,0,0.07) + JointTask in its null space) for N robots, each with its own force space (dimension and axis) and closed-loop
// force flag set through the pointer overloads, a sensed force per robot, three control cycles.  Also reads the spaces back and
// checks that an invalid dimension throws and changes nothing.
// Usage: per_robot_spaces_demo <state.bin> <spaces.bin> <N> <tau_out.bin>
//   state.bin: q then dq (7 x N each, SoA), float64
//   spaces.bin: force space dimension (N), closed-loop flag (N), as float64; axes (3 x N, SoA); sensed force (3 x N, SoA)
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "sai_b200/sai_primitives_batched.hpp"

using namespace SaiPrimitivesB200;

int main(int argc, char** argv) {
	if (argc < 5) return 2;
	const int64_t N = std::atoll(argv[3]);
	const int dof = 7;
	std::vector<double> q((size_t)dof * N), dq((size_t)dof * N), sp((size_t)8 * N);
	FILE* f = std::fopen(argv[1], "rb");
	if (!f || std::fread(q.data(), 8, q.size(), f) != q.size() || std::fread(dq.data(), 8, dq.size(), f) != dq.size()) return 3;
	std::fclose(f);
	f = std::fopen(argv[2], "rb");
	if (!f || std::fread(sp.data(), 8, sp.size(), f) != sp.size()) return 3;
	std::fclose(f);
	std::vector<int32_t> dims(N), flags(N), reset(N, -1);
	for (int64_t i = 0; i < N; i++) {
		dims[i] = (int32_t)sp[i];
		flags[i] = (int32_t)sp[N + i];
	}
	const double* axes = sp.data() + 2 * N;
	const double* force = axes + 3 * N;
	try {
		auto robot = std::make_shared<BatchedRobot>("panda", N);
		robot->setState(q.data(), dq.data());
		auto motion_force_task = std::make_shared<MotionForceTask>(robot, "end-effector", Affine::Translation(0.0, 0.0, 0.07));
		motion_force_task->disableInternalOtg();
		auto joint_task = std::make_shared<JointTask>(robot);
		joint_task->disableInternalOtg();
		std::vector<std::shared_ptr<TemplateTask>> task_list = {motion_force_task, joint_task};
		auto robot_controller = std::make_unique<RobotController>(robot, task_list);
		motion_force_task->setForceControlGains(0.8, 12.0, 1.5);
		motion_force_task->setGoalForce(Vec3{0.0, 0.0, -5.0});
		motion_force_task->parametrizeForceMotionSpaces(dims.data(), axes, reset.data(), OSC_MEM_HOST);
		motion_force_task->setClosedLoopForceControl(flags.data(), OSC_MEM_HOST);
		for (int64_t i = 0; i < N; i++)
			if (reset[i] != (dims[i] != 0 ? 1 : 0)) return 4;	// every robot starts at dimension 0
		std::vector<int32_t> got_dims(N), got_cl(N);
		std::vector<double> got_axes((size_t)3 * N);
		motion_force_task->getForceMotionSpaces(got_dims.data(), got_axes.data(), got_cl.data());
		for (int64_t i = 0; i < N; i++)
			if (got_dims[i] != dims[i] || got_cl[i] != flags[i]) return 5;
		std::vector<int32_t> bad(dims);
		bad[N / 2] = 4;
		bool threw = false;
		try {
			motion_force_task->parametrizeForceMotionSpaces(bad.data(), axes, nullptr, OSC_MEM_HOST);
		} catch (const std::invalid_argument&) {
			threw = true;
		}
		if (!threw) return 6;
		motion_force_task->getForceMotionSpaces(got_dims.data(), nullptr, nullptr);
		for (int64_t i = 0; i < N; i++)
			if (got_dims[i] != dims[i]) return 7;
		const std::vector<double> zero((size_t)3 * N, 0.0);
		motion_force_task->updateSensedForceAndMoment(force, zero.data());
		std::vector<double> tau;
		for (int k = 0; k < 3; k++) {
			robot_controller->updateControllerTaskModels();
			tau = robot_controller->computeControlTorques();
		}
		FILE* o = std::fopen(argv[4], "wb");
		std::fwrite(tau.data(), 8, tau.size(), o);
		std::fclose(o);
		size_t unhandled = 0;
		for (uint32_t s : robot->status()) unhandled += (s & OSC_STATUS_UNHANDLED) ? 1 : 0;
		std::printf("ok %lld robots, %zu unhandled\n", (long long)N, unhandled);
	} catch (const std::exception& e) {
		std::fprintf(stderr, "error: %s\n", e.what());
		return 1;
	}
	return 0;
}
