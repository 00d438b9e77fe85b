// Per-robot resets through the batched C++ mirror: the example-05 hierarchy (MotionForceTask at end-effector (0,0,0.07) +
// JointTask in its null space) for N robots, three cycles at state 1, then every robot moves to state 2 and the robots a mask
// selects get reinitializeTasks(mask); three more cycles.  An all-zero mask through resetRobots and a task's reInitializeTask
// must change nothing in between.
// Usage: robot_reset_demo <state1.bin> <state2.bin> <mask.bin> <N> <tau_out.bin>
//   state*.bin: q then dq (7 x N each, SoA), float64;  mask.bin: int32 x N
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "sai_b200/sai_primitives_batched.hpp"

using namespace SaiPrimitivesB200;

static bool read(const char* path, void* dst, size_t bytes) {
	FILE* f = std::fopen(path, "rb");
	if (!f) return false;
	const bool ok = std::fread(dst, 1, bytes, f) == bytes;
	std::fclose(f);
	return ok;
}

int main(int argc, char** argv) {
	if (argc < 6) return 2;
	const int64_t N = std::atoll(argv[4]);
	const int dof = 7;
	std::vector<double> s1((size_t)2 * dof * N), s2((size_t)2 * dof * N);
	std::vector<int32_t> mask(N), none(N, 0);
	if (!read(argv[1], s1.data(), s1.size() * 8) || !read(argv[2], s2.data(), s2.size() * 8) || !read(argv[3], mask.data(), mask.size() * 4)) return 3;
	try {
		auto robot = std::make_shared<BatchedRobot>("panda", N);
		robot->setState(s1.data(), s1.data() + dof * N);
		auto motion_force_task = std::make_shared<MotionForceTask>(robot, "end-effector", Affine::Translation(0.0, 0.0, 0.07));
		motion_force_task->disableInternalOtg();
		auto joint_task = std::make_shared<JointTask>(robot);
		joint_task->disableInternalOtg();
		std::vector<std::shared_ptr<TemplateTask>> task_list = {motion_force_task, joint_task};
		auto robot_controller = std::make_unique<RobotController>(robot, task_list);
		motion_force_task->setGoalLinearVelocity(Vec3{0.01, -0.02, 0.03});
		joint_task->setGoalVelocity(std::vector<double>(dof, 0.1));
		std::vector<double> tau, before;
		for (int k = 0; k < 3; k++) {
			robot_controller->updateControllerTaskModels();
			tau = robot_controller->computeControlTorques();
		}
		robot->setState(s2.data(), s2.data() + dof * N);
		robot_controller->resetRobots(none.data(), OSC_MEM_HOST);
		motion_force_task->reInitializeTask(none.data(), OSC_MEM_HOST);
		robot_controller->reinitializeTasks(mask.data(), OSC_MEM_HOST);
		for (int k = 0; k < 3; k++) {
			robot_controller->updateControllerTaskModels();
			tau = robot_controller->computeControlTorques();
		}
		FILE* o = std::fopen(argv[5], "wb");
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
