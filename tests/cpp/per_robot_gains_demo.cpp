// Per-robot gains through the batched C++ mirror: the example-05 hierarchy (MotionForceTask at end-effector (0,0,0.07) +
// JointTask in its null space) for N robots, each with its own position, orientation and joint gains set through the SoA
// overloads, three control cycles.  Also drives the broadcast gain setters of a one-row partial JointTask (task dof 1).
// Usage: per_robot_gains_demo <state.bin> <gains.bin> <N> <tau_out.bin>
//   state.bin: q then dq (7 x N each, SoA), float64
//   gains.bin: kp, kv, ki of position (3 x N each), of orientation (3 x N each), of the joint task (7 x N each), SoA, float64
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "sai_b200/sai_primitives_batched.hpp"

using namespace SaiPrimitivesB200;

static bool same(const std::vector<double>& a, const double* b) {
	for (size_t k = 0; k < a.size(); k++)
		if (a[k] != b[k]) return false;
	return true;
}

int main(int argc, char** argv) {
	if (argc < 5) return 2;
	const int64_t N = std::atoll(argv[3]);
	const int dof = 7;
	std::vector<double> q((size_t)dof * N), dq((size_t)dof * N), g((size_t)(6 * 3 + 3 * dof) * N);
	FILE* f = std::fopen(argv[1], "rb");
	if (!f || std::fread(q.data(), 8, q.size(), f) != q.size() || std::fread(dq.data(), 8, dq.size(), f) != dq.size()) return 3;
	std::fclose(f);
	f = std::fopen(argv[2], "rb");
	if (!f || std::fread(g.data(), 8, g.size(), f) != g.size()) return 3;
	std::fclose(f);
	const double* kp_pos = g.data();
	const double* kv_pos = kp_pos + 3 * N;
	const double* ki_pos = kv_pos + 3 * N;
	const double* kp_ori = ki_pos + 3 * N;
	const double* kv_ori = kp_ori + 3 * N;
	const double* ki_ori = kv_ori + 3 * N;
	const double* kp_j = ki_ori + 3 * N;
	const double* kv_j = kp_j + dof * N;
	const double* ki_j = kv_j + dof * N;
	try {
		// ---- a one-row partial JointTask: broadcast setters with task dof 1, then per robot, read back
		{
			auto robot = std::make_shared<BatchedRobot>("panda", N);
			robot->setState(q.data(), dq.data());
			std::vector<double> S(dof, 0.0);
			S[3] = 1.0;
			JointTask one(robot, S, 1);
			one.setGains(40.0, 11.0, 0.5);
			std::vector<double> kp(N), kv(N), ki(N);
			one.getGains(kp.data(), kv.data(), ki.data());
			if (kp[0] != 40.0 || kv[N - 1] != 11.0 || ki[0] != 0.5) return 5;
			one.setGains(std::vector<double>{41.0}, std::vector<double>{12.0}, std::vector<double>{0.25});
			one.getGains(kp.data(), kv.data(), ki.data());
			if (kp[N - 1] != 41.0 || kv[0] != 12.0 || ki[N - 1] != 0.25) return 5;
			std::vector<double> rp(N), rv(N, 3.0), ri(N, 0.0);
			for (int64_t i = 0; i < N; i++) rp[i] = 10.0 + (double)i;
			one.setGains(rp.data(), rv.data(), ri.data(), OSC_MEM_HOST);
			one.setGains(7.0, 2.0, 1.0);	// broadcast in per-robot mode: every robot
			one.getGains(kp.data(), kv.data(), ki.data());
			for (int64_t i = 0; i < N; i++)
				if (kp[i] != 7.0 || kv[i] != 2.0 || ki[i] != 1.0) return 5;
			bool threw = false;
			try {
				one.setGains(rp.data(), std::vector<double>(N, -1.0).data(), ri.data(), OSC_MEM_HOST);
			} catch (const std::invalid_argument&) {
				threw = true;
			}
			if (!threw) return 6;
		}
		// ---- the example-05 hierarchy with per-robot gains
		auto robot = std::make_shared<BatchedRobot>("panda", N);
		robot->setState(q.data(), dq.data());
		auto motion_force_task = std::make_shared<MotionForceTask>(robot, "end-effector", Affine::Translation(0.0, 0.0, 0.07));
		motion_force_task->disableInternalOtg();
		auto joint_task = std::make_shared<JointTask>(robot);
		joint_task->disableInternalOtg();
		std::vector<std::shared_ptr<TemplateTask>> task_list = {motion_force_task, joint_task};
		auto robot_controller = std::make_unique<RobotController>(robot, task_list);
		motion_force_task->setPosControlGains(kp_pos, kv_pos, ki_pos, OSC_MEM_HOST);
		motion_force_task->setOriControlGains(kp_ori, kv_ori, ki_ori, OSC_MEM_HOST);
		joint_task->setGains(kp_j, kv_j, ki_j, OSC_MEM_HOST);
		std::vector<double> a((size_t)3 * N), b((size_t)3 * N), c((size_t)3 * N);
		motion_force_task->getOriControlGains(a.data(), b.data(), c.data());
		if (!same(a, kp_ori) || !same(b, kv_ori) || !same(c, ki_ori)) return 7;
		std::vector<double> ja((size_t)dof * N), jb((size_t)dof * N), jc((size_t)dof * N);
		joint_task->getGains(ja.data(), jb.data(), jc.data());
		if (!same(ja, kp_j) || !same(jb, kv_j) || !same(jc, ki_j)) return 7;
		motion_force_task->setGoalLinearVelocity(Vec3{0.01, -0.02, 0.03});
		joint_task->setGoalVelocity(std::vector<double>(dof, 0.1));
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
