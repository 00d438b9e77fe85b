// Header-only C++17 mirror of the sai-primitives interface for the batched path, on top of the C ABI
// (sai_b200_osc.h).  Class and method names are the reference's (src/tasks/JointTask.h,
// src/tasks/MotionForceTask.h, src/RobotController.h); every per-robot quantity exists in two forms:
//   - broadcast: one value for all robots (same signature shape as the reference, plain arrays instead of Eigen);
//   - batched:   a pointer to SoA data (component-major, data[c * n_robots + i]) in host or device memory.
// Errors the reference reports with std::invalid_argument are re-thrown as std::invalid_argument.
// Internal OTG: the acceleration-limited, phase-synchronised generator (the reference's default, JointTask.h:38-42,
// MotionForceTask.h:67-74) runs batched on the device and is ON after construction like in the reference; the jerk-limited
// variant is not built (enableInternalOtgJerkLimited throws).
#pragma once

#include <array>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../sai_b200_osc.h"

namespace SaiPrimitivesB200 {

using Vec3 = std::array<double, 3>;
using Mat3 = std::array<double, 9>;	 // row-major

enum DynamicDecouplingType {  // src/helper_modules/SaiPrimitivesCommonDefinitions.h:14-20
	FULL_DYNAMIC_DECOUPLING = OSC_FULL_DYNAMIC_DECOUPLING,
	BOUNDED_INERTIA_ESTIMATES = OSC_BOUNDED_INERTIA_ESTIMATES,
	IMPEDANCE = OSC_IMPEDANCE,
};
enum TaskType { JOINT_TASK = OSC_TASK_JOINT, MOTION_FORCE_TASK = OSC_TASK_MOTION_FORCE };  // TemplateTask.h:19-24

struct Affine {	 // Eigen::Affine3d stand-in
	Mat3 R{1, 0, 0, 0, 1, 0, 0, 0, 1};
	Vec3 t{0, 0, 0};
	static Affine Translation(double x, double y, double z) {
		Affine a;
		a.t = {x, y, z};
		return a;
	}
};

inline void check(osc_handle* h, int rc) {
	if (rc == OSC_OK) return;
	const char* m = osc_last_error(h);
	const std::string msg = m ? m : "";
	if (rc == OSC_ERR_INVALID_ARGUMENT) throw std::invalid_argument(msg);
	if (rc == OSC_ERR_UNSUPPORTED) throw std::logic_error("unsupported on the batched path: " + msg);
	throw std::runtime_error("sai_b200_osc error " + std::to_string(rc) + ": " + msg);
}

// The SaiModel of the batch: N copies of one robot on one CUDA device.
// SURVEY.md row f-3: the counterpart of `std::make_shared<SaiModel::SaiModel>(robot_file)`
// (examples/05-using_robot_controller/05-using_robot_controller.cpp:64): registers a URDF serial chain under a name that
// BatchedRobot(name, n) and the link-name arguments of the tasks then accept.
inline void registerUrdfFile(const std::string& model_name, const std::string& urdf_file) {
	if (osc_urdf_register_file(model_name.c_str(), urdf_file.c_str()) != OSC_OK)
		throw std::invalid_argument("URDF [" + urdf_file + "]: " + osc_urdf_last_error());
}

class BatchedRobot {
public:
	BatchedRobot(const std::string& builtin_robot, int64_t n_robots, int device = 0) : _name(builtin_robot) {
		if (osc_builtin_model(builtin_robot.c_str(), &_desc) != OSC_OK)
			throw std::invalid_argument("unknown built-in robot model [" + builtin_robot + "]");
		create(n_robots, device);
	}
	BatchedRobot(const osc_model_desc& desc, int64_t n_robots, int device = 0) : _desc(desc) { create(n_robots, device); }
	~BatchedRobot() { osc_destroy(_h); }
	BatchedRobot(const BatchedRobot&) = delete;
	BatchedRobot& operator=(const BatchedRobot&) = delete;

	int dof() const { return _desc.n; }
	int64_t numRobots() const { return osc_num_robots(_h); }
	osc_handle* handle() const { return _h; }
	// setQ + setDq + updateModel of the reference's user loop (examples/05-...cpp:143-145), SoA n x N
	void setState(const double* q, const double* dq, osc_mem_kind where = OSC_MEM_HOST) { check(_h, osc_set_state(_h, q, dq, where)); }
	osc_link_frame linkFrame(const std::string& link_name) const {
		osc_link_frame f;
		if (_name.empty() || osc_builtin_link(_name.c_str(), link_name.c_str(), &f) != OSC_OK)
			throw std::invalid_argument("link [" + link_name + "] does not exist");
		return f;
	}
	std::vector<uint32_t> status() const {
		std::vector<uint32_t> s((size_t)numRobots());
		check(_h, osc_get_status(_h, s.data(), OSC_MEM_HOST));
		return s;
	}
	void sync() { check(_h, osc_sync(_h)); }

private:
	void create(int64_t n, int device) {
		int rc = osc_create(&_desc, n, device, &_h);
		if (rc != OSC_OK) {
			const char* m = osc_last_error(nullptr);
			throw std::runtime_error(std::string("osc_create failed: ") + (m ? m : ""));
		}
	}
	std::string _name;
	osc_model_desc _desc{};
	osc_handle* _h = nullptr;
};

// src/tasks/TemplateTask.h:26-124
class TemplateTask {
public:
	TemplateTask(std::shared_ptr<BatchedRobot>& robot, const std::string& task_name, TaskType type, double loop_timestep)
		: _robot(robot), _task_name(task_name), _task_type(type), _loop_timestep(loop_timestep) {}
	virtual ~TemplateTask() = default;
	virtual void reInitializeTask() { check(h(), osc_reinitialize_task(h(), _id)); }
	// the robots a non-zero entry of mask (int32 x n_robots in `where` memory) selects (osc_reset_robots, OSC_RESET_REINITIALIZE)
	void reInitializeTask(const int32_t* mask, osc_mem_kind where) { check(h(), osc_reset_robots(h(), _id, mask, where, OSC_RESET_REINITIALIZE)); }
	const std::shared_ptr<BatchedRobot>& getConstRobotModel() const { return _robot; }
	const double& getLoopTimestep() const { return _loop_timestep; }
	const TaskType& getTaskType() const { return _task_type; }
	const std::string& getTaskName() const { return _task_name; }
	int id() const { return _id; }
	// TemplateTask.h:74,82,89: n x n row-major per robot, SoA out (component r * n + c of robot i at soa[(r * n + c) * N + i]);
	// evaluated from the robot's current state (what updateControllerTaskModels() yields there)
	void getTaskNullspace(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_TASK_NULLSPACE, soa, w); }
	void getPreviousTasksNullspace(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_TASK_PREVIOUS_NULLSPACE, soa, w); }
	void getTaskAndPreviousNullspace(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_TASK_AND_PREVIOUS_NULLSPACE, soa, w); }

protected:
	osc_handle* h() const { return _robot->handle(); }
	void setBroadcast(int field, const double* v) { check(h(), osc_set_field(h(), _id, field, v, OSC_MEM_HOST, 1)); }
	void setBatched(int field, const double* soa, osc_mem_kind where) { check(h(), osc_set_field(h(), _id, field, soa, where, 0)); }
	void get(int field, double* soa, osc_mem_kind where) const { check(h(), osc_get_field(h(), _id, field, soa, where)); }
	// osc_set_gains / osc_get_gains: broadcast (ncomp values each) or per robot (SoA ncomp x N each, host or device memory)
	void setGainsBroadcast(int group, const double* kp, const double* kv, const double* ki) {
		check(h(), osc_set_gains(h(), _id, group, kp, kv, ki, OSC_MEM_HOST, 0));
	}
	void setGainsBatched(int group, const double* kp, const double* kv, const double* ki, osc_mem_kind where) {
		check(h(), osc_set_gains(h(), _id, group, kp, kv, ki, where, 1));
	}
	void getGainsBatched(int group, double* kp, double* kv, double* ki, osc_mem_kind where) const {
		check(h(), osc_get_gains(h(), _id, group, kp, kv, ki, where));
	}
	std::shared_ptr<BatchedRobot> _robot;
	std::string _task_name;
	TaskType _task_type;
	double _loop_timestep;
	int _id = -1;
};

// src/tasks/JointTask.h
class JointTask : public TemplateTask {
public:
	struct DefaultParameters {	// JointTask.h:31-45 (the entries this mirror consults)
		static constexpr bool use_internal_otg = true;
		static constexpr double otg_max_velocity = 3.14159265358979323846 / 3.0;
		static constexpr double otg_max_acceleration = 2.0 * 3.14159265358979323846;
	};
	JointTask(std::shared_ptr<BatchedRobot>& robot, const std::string& task_name = "joint_task", double loop_timestep = 0.001)
		: TemplateTask(robot, task_name, JOINT_TASK, loop_timestep) {
		check(h(), osc_add_joint_task(h(), nullptr, 0, loop_timestep, &_id));
		_task_dof = osc_get_task_dof(h(), _id);
		if (DefaultParameters::use_internal_otg) enableInternalOtgAccelerationLimited(DefaultParameters::otg_max_velocity, DefaultParameters::otg_max_acceleration);
	}
	// joint_selection_matrix: row-major k x dof
	JointTask(std::shared_ptr<BatchedRobot>& robot, const std::vector<double>& joint_selection_matrix, int rows,
			  const std::string& task_name = "partial_joint_task", double loop_timestep = 0.001)
		: TemplateTask(robot, task_name, JOINT_TASK, loop_timestep) {
		if ((int)joint_selection_matrix.size() != rows * robot->dof())
			throw std::invalid_argument("joint selection matrix size not consistent with robot dof in JointTask constructor\n");
		check(h(), osc_add_joint_task(h(), joint_selection_matrix.data(), rows, loop_timestep, &_id));
		_task_dof = osc_get_task_dof(h(), _id);
		if (DefaultParameters::use_internal_otg) enableInternalOtgAccelerationLimited(DefaultParameters::otg_max_velocity, DefaultParameters::otg_max_acceleration);
	}
	int getTaskDof() const { return _task_dof; }
	bool isFullJointTask() const { return _task_dof == _robot->dof(); }

	void setGoalPosition(const std::vector<double>& goal) { sized(goal, "goal position"); setBroadcast(OSC_JT_GOAL_POSITION, goal.data()); }
	void setGoalVelocity(const std::vector<double>& goal) { sized(goal, "goal velocity"); setBroadcast(OSC_JT_GOAL_VELOCITY, goal.data()); }
	void setGoalAcceleration(const std::vector<double>& goal) { sized(goal, "goal acceleration"); setBroadcast(OSC_JT_GOAL_ACCELERATION, goal.data()); }
	void setGoalPosition(const double* soa, osc_mem_kind where) { setBatched(OSC_JT_GOAL_POSITION, soa, where); }
	void setGoalVelocity(const double* soa, osc_mem_kind where) { setBatched(OSC_JT_GOAL_VELOCITY, soa, where); }
	void setGoalAcceleration(const double* soa, osc_mem_kind where) { setBatched(OSC_JT_GOAL_ACCELERATION, soa, where); }
	void getGoalPosition(double* soa, osc_mem_kind where = OSC_MEM_HOST) const { get(OSC_JT_GOAL_POSITION, soa, where); }

	void setGains(double kp, double kv, double ki = 0) {
		const std::vector<double> p(_task_dof, kp), v(_task_dof, kv), i(_task_dof, ki);
		setGainsBroadcast(OSC_GAINS_JOINT, p.data(), v.data(), i.data());
	}
	void setGains(const std::vector<double>& kp, const std::vector<double>& kv, const std::vector<double>& ki) {
		if (kp.size() == 1 && kv.size() == 1 && ki.size() == 1) return setGains(kp[0], kv[0], ki[0]);
		if ((int)kp.size() != _task_dof || (int)kv.size() != _task_dof || (int)ki.size() != _task_dof)
			throw std::invalid_argument("size of gain vectors inconsistent with number of task dofs in JointTask::setGains\n");
		setGainsBroadcast(OSC_GAINS_JOINT, kp.data(), kv.data(), ki.data());
	}
	// per robot: SoA k x N each (gain a of robot i at soa[a * N + i]), host or device memory
	void setGains(const double* kp, const double* kv, const double* ki, osc_mem_kind where) { setGainsBatched(OSC_GAINS_JOINT, kp, kv, ki, where); }
	void getGains(double* kp, double* kv, double* ki, osc_mem_kind where = OSC_MEM_HOST) const { getGainsBatched(OSC_GAINS_JOINT, kp, kv, ki, where); }
	void setDynamicDecouplingType(DynamicDecouplingType type) {
		osc_joint_params p = params();
		p.dynamic_decoupling_type = type;
		apply(p);
	}
	void setBoundedInertiaEstimateThreshold(double threshold) {
		osc_joint_params p = params();
		p.bie_threshold = threshold;
		apply(p);
	}
	void enableVelocitySaturation(double saturation_velocity) {
		osc_joint_params p = params();
		p.use_velocity_saturation = 1;
		for (int a = 0; a < _task_dof; a++) p.saturation_velocity[a] = saturation_velocity;
		apply(p);
	}
	void disableVelocitySaturation() {
		osc_joint_params p = params();
		p.use_velocity_saturation = 0;
		apply(p);
	}
	// JointTask.cpp:358-380
	void enableInternalOtgAccelerationLimited(double max_velocity, double max_acceleration) {
		enableInternalOtgAccelerationLimited(std::vector<double>(_task_dof, max_velocity), std::vector<double>(_task_dof, max_acceleration));
	}
	void enableInternalOtgAccelerationLimited(const std::vector<double>& max_velocity, const std::vector<double>& max_acceleration) {
		sized(max_velocity, "max velocity");
		sized(max_acceleration, "max acceleration");
		check(h(), osc_joint_enable_internal_otg(h(), _id, max_velocity.data(), max_acceleration.data()));
	}
	void enableInternalOtgJerkLimited(double, double, double) { throw std::logic_error("the jerk-limited internal OTG is not built"); }
	void disableInternalOtg() { check(h(), osc_disable_internal_otg(h(), _id)); }
	bool getInternalOtgEnabled() const { return osc_internal_otg_enabled(h(), _id) == 1; }
	// JointTask.h:162-176 (SoA k x N out)
	void getDesiredPosition(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_JT_DESIRED_POSITION, soa, w); }
	void getDesiredVelocity(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_JT_DESIRED_VELOCITY, soa, w); }
	void getDesiredAcceleration(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_JT_DESIRED_ACCELERATION, soa, w); }

private:
	void sized(const std::vector<double>& v, const char* what) const {
		if ((int)v.size() != _task_dof) throw std::invalid_argument(std::string(what) + " vector size not consistent with task dof in JointTask\n");
	}
	osc_joint_params params() const {
		osc_joint_params p;
		check(h(), osc_joint_get_params(h(), _id, &p));
		return p;
	}
	void apply(const osc_joint_params& p) { check(h(), osc_joint_set_params(h(), _id, &p)); }
	int _task_dof = 0;
};

// src/tasks/MotionForceTask.h
class MotionForceTask : public TemplateTask {
public:
	MotionForceTask(std::shared_ptr<BatchedRobot>& robot, const std::string& link_name, const Affine& compliant_frame = Affine(),
					const std::string& task_name = "motion_force_task", bool is_force_motion_parametrization_in_compliant_frame = false,
					double loop_timestep = 0.001)
		: TemplateTask(robot, task_name, MOTION_FORCE_TASK, loop_timestep), _link_name(link_name) {
		osc_mft_desc d = base_desc(link_name, compliant_frame, is_force_motion_parametrization_in_compliant_frame, loop_timestep);
		d.partial = 0;
		check(h(), osc_add_motion_force_task(h(), &d, &_id));
		defaultOtg();
	}
	MotionForceTask(std::shared_ptr<BatchedRobot>& robot, const std::string& link_name, const std::vector<Vec3>& controlled_directions_translation,
					const std::vector<Vec3>& controlled_directions_rotation, const Affine& compliant_frame = Affine(),
					const std::string& task_name = "partial_motion_force_task",
					bool is_force_motion_parametrization_in_compliant_frame = false, double loop_timestep = 0.001)
		: TemplateTask(robot, task_name, MOTION_FORCE_TASK, loop_timestep), _link_name(link_name) {
		if (controlled_directions_translation.size() > 3 || controlled_directions_rotation.size() > 3)
			throw std::invalid_argument("at most 3 controlled directions per block");
		osc_mft_desc d = base_desc(link_name, compliant_frame, is_force_motion_parametrization_in_compliant_frame, loop_timestep);
		d.partial = 1;
		d.n_dirs_translation = (int)controlled_directions_translation.size();
		d.n_dirs_rotation = (int)controlled_directions_rotation.size();
		for (int i = 0; i < d.n_dirs_translation; i++)
			for (int k = 0; k < 3; k++) d.dirs_translation[i][k] = controlled_directions_translation[i][k];
		for (int i = 0; i < d.n_dirs_rotation; i++)
			for (int k = 0; k < 3; k++) d.dirs_rotation[i][k] = controlled_directions_rotation[i][k];
		check(h(), osc_add_motion_force_task(h(), &d, &_id));
		defaultOtg();
	}

	// ---- goals: broadcast (reference signatures) and batched SoA
	void setGoalPosition(const Vec3& v) { setBroadcast(OSC_MFT_GOAL_POSITION, v.data()); }
	void setGoalOrientation(const Mat3& R) { setBroadcast(OSC_MFT_GOAL_ORIENTATION, R.data()); }
	void setGoalLinearVelocity(const Vec3& v) { setBroadcast(OSC_MFT_GOAL_LINEAR_VELOCITY, v.data()); }
	void setGoalAngularVelocity(const Vec3& v) { setBroadcast(OSC_MFT_GOAL_ANGULAR_VELOCITY, v.data()); }
	void setGoalLinearAcceleration(const Vec3& v) { setBroadcast(OSC_MFT_GOAL_LINEAR_ACCELERATION, v.data()); }
	void setGoalAngularAcceleration(const Vec3& v) { setBroadcast(OSC_MFT_GOAL_ANGULAR_ACCELERATION, v.data()); }
	void setGoalForce(const Vec3& v) { setBroadcast(OSC_MFT_GOAL_FORCE, v.data()); }
	void setGoalMoment(const Vec3& v) { setBroadcast(OSC_MFT_GOAL_MOMENT, v.data()); }
	void setGoalPosition(const double* soa, osc_mem_kind w) { setBatched(OSC_MFT_GOAL_POSITION, soa, w); }
	void setGoalOrientation(const double* soa, osc_mem_kind w) { setBatched(OSC_MFT_GOAL_ORIENTATION, soa, w); }
	void setGoalLinearVelocity(const double* soa, osc_mem_kind w) { setBatched(OSC_MFT_GOAL_LINEAR_VELOCITY, soa, w); }
	void setGoalAngularVelocity(const double* soa, osc_mem_kind w) { setBatched(OSC_MFT_GOAL_ANGULAR_VELOCITY, soa, w); }
	void setGoalLinearAcceleration(const double* soa, osc_mem_kind w) { setBatched(OSC_MFT_GOAL_LINEAR_ACCELERATION, soa, w); }
	void setGoalAngularAcceleration(const double* soa, osc_mem_kind w) { setBatched(OSC_MFT_GOAL_ANGULAR_ACCELERATION, soa, w); }
	void setGoalForce(const double* soa, osc_mem_kind w) { setBatched(OSC_MFT_GOAL_FORCE, soa, w); }
	void setGoalMoment(const double* soa, osc_mem_kind w) { setBatched(OSC_MFT_GOAL_MOMENT, soa, w); }
	// ---- observers (SoA out)
	void getCurrentPosition(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_CURRENT_POSITION, soa, w); }
	void getCurrentOrientation(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_CURRENT_ORIENTATION, soa, w); }
	void getCurrentLinearVelocity(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_CURRENT_LINEAR_VELOCITY, soa, w); }
	void getCurrentAngularVelocity(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_CURRENT_ANGULAR_VELOCITY, soa, w); }
	void getGoalPosition(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_GOAL_POSITION, soa, w); }
	void getSensedForceControlWorldFrame(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_SENSED_FORCE_CONTROL_WORLD, soa, w); }
	void getSensedMomentControlWorldFrame(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_SENSED_MOMENT_CONTROL_WORLD, soa, w); }
	void getUnitMassForce(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_UNIT_MASS_FORCE, soa, w); }
	// MotionForceTask.h:268-269, :613-616
	void getPositionError(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_POSITION_ERROR, soa, w); }
	void getOrientationError(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_ORIENTATION_ERROR, soa, w); }
	void sigmaForce(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_SIGMA_FORCE, soa, w); }
	void sigmaPosition(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_SIGMA_POSITION, soa, w); }
	void sigmaMoment(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_SIGMA_MOMENT, soa, w); }
	void sigmaOrientation(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_SIGMA_ORIENTATION, soa, w); }

	// ---- gains and options
	void setPosControlGains(double kp, double kv, double ki = 0) { setPosControlGains(Vec3{kp, kp, kp}, Vec3{kv, kv, kv}, Vec3{ki, ki, ki}); }
	void setPosControlGains(const Vec3& kp, const Vec3& kv, const Vec3& ki = Vec3{0, 0, 0}) {
		setGainsBroadcast(OSC_GAINS_POSITION, kp.data(), kv.data(), ki.data());
	}
	void setOriControlGains(double kp, double kv, double ki = 0) { setOriControlGains(Vec3{kp, kp, kp}, Vec3{kv, kv, kv}, Vec3{ki, ki, ki}); }
	void setOriControlGains(const Vec3& kp, const Vec3& kv, const Vec3& ki = Vec3{0, 0, 0}) {
		setGainsBroadcast(OSC_GAINS_ORIENTATION, kp.data(), kv.data(), ki.data());
	}
	void setForceControlGains(double kp, double kv, double ki) { setGainsBroadcast(OSC_GAINS_FORCE, &kp, &kv, &ki); }
	void setMomentControlGains(double kp, double kv, double ki) { setGainsBroadcast(OSC_GAINS_MOMENT, &kp, &kv, &ki); }
	// per robot: SoA 3 x N (position, orientation) or 1 x N (force, moment) each, host or device memory; getters likewise
	void setPosControlGains(const double* kp, const double* kv, const double* ki, osc_mem_kind w) { setGainsBatched(OSC_GAINS_POSITION, kp, kv, ki, w); }
	void setOriControlGains(const double* kp, const double* kv, const double* ki, osc_mem_kind w) { setGainsBatched(OSC_GAINS_ORIENTATION, kp, kv, ki, w); }
	void setForceControlGains(const double* kp, const double* kv, const double* ki, osc_mem_kind w) { setGainsBatched(OSC_GAINS_FORCE, kp, kv, ki, w); }
	void setMomentControlGains(const double* kp, const double* kv, const double* ki, osc_mem_kind w) { setGainsBatched(OSC_GAINS_MOMENT, kp, kv, ki, w); }
	void getPosControlGains(double* kp, double* kv, double* ki, osc_mem_kind w = OSC_MEM_HOST) const { getGainsBatched(OSC_GAINS_POSITION, kp, kv, ki, w); }
	void getOriControlGains(double* kp, double* kv, double* ki, osc_mem_kind w = OSC_MEM_HOST) const { getGainsBatched(OSC_GAINS_ORIENTATION, kp, kv, ki, w); }
	void getForceControlGains(double* kp, double* kv, double* ki, osc_mem_kind w = OSC_MEM_HOST) const { getGainsBatched(OSC_GAINS_FORCE, kp, kv, ki, w); }
	void getMomentControlGains(double* kp, double* kv, double* ki, osc_mem_kind w = OSC_MEM_HOST) const { getGainsBatched(OSC_GAINS_MOMENT, kp, kv, ki, w); }
	void setFeedforwardForceGain(double k) { auto p = params(); p.kff_force = k; apply(p); }
	void setFeedforwardmomentGain(double k) { auto p = params(); p.kff_moment = k; apply(p); }
	void setMaxForceControlFeedbackOutput(double v) { auto p = params(); p.max_force_control_feedback_output = v; apply(p); }
	void setMaxMomentControlFeedbackOutput(double v) { auto p = params(); p.max_moment_control_feedback_output = v; apply(p); }
	void enableVelocitySaturation(double linear_vel_sat = 0.3, double angular_vel_sat = 3.14159265358979323846 / 3) {
		auto p = params();
		p.use_velocity_saturation = 1;
		p.linear_saturation_velocity = linear_vel_sat;
		p.angular_saturation_velocity = angular_vel_sat;
		apply(p);
	}
	void disableVelocitySaturation() { auto p = params(); p.use_velocity_saturation = 0; apply(p); }
	void setDynamicDecouplingType(DynamicDecouplingType type) { auto p = params(); p.dynamic_decoupling_type = type; apply(p); }
	void setBoundedInertiaEstimateThreshold(double thr) { auto p = params(); p.bie_threshold = thr; apply(p); }
	double getBoundedInertiaEstimateThreshold() const { return params().bie_threshold; }
	void handleAllSingularitiesAsType1(bool flag) { auto p = params(); p.enforce_type_1_strategy = flag; apply(p); }
	void enableSingularityHandling() { auto p = params(); p.singularity_handling_enabled = 1; apply(p); }
	void disableSingularityHandling() { auto p = params(); p.singularity_handling_enabled = 0; apply(p); }
	void setSingularityHandlingBounds(double s_min, double s_max) { auto p = params(); p.s_min = s_min; p.s_max = s_max; apply(p); }
	void setSingularityHandlingGains(double kp1, double kv1, double kv2) { auto p = params(); p.kp_type_1 = kp1; p.kv_type_1 = kv1; p.kv_type_2 = kv2; apply(p); }
	void setType1Posture(const std::vector<double>& q_des) { setBroadcast(OSC_MFT_TYPE1_POSTURE, q_des.data()); }

	bool parametrizeForceMotionSpaces(int force_space_dimension, const Vec3& axis = Vec3{0, 0, 0}) {
		int reset = 0;
		check(h(), osc_mft_parametrize_force_motion_spaces(h(), _id, force_space_dimension, axis.data(), &reset));
		return reset != 0;
	}
	bool parametrizeMomentRotMotionSpaces(int moment_space_dimension, const Vec3& axis = Vec3{0, 0, 0}) {
		int reset = 0;
		check(h(), osc_mft_parametrize_moment_rotmotion_spaces(h(), _id, moment_space_dimension, axis.data(), &reset));
		return reset != 0;
	}
	int getForceSpaceDimension() const { return params().force_space_dimension; }
	int getMomentSpaceDimension() const { return params().moment_space_dimension; }
	void setClosedLoopForceControl(bool on = true) { check(h(), osc_mft_set_closed_loop_force_control(h(), _id, on)); }
	void setClosedLoopMomentControl(bool on = true) { check(h(), osc_mft_set_closed_loop_moment_control(h(), _id, on)); }
	// per robot (osc_mft_parametrize_spaces_batched / osc_mft_set_closed_loop_batched), host or device memory: dims int32 x N, axes
	// SoA 3 x N (axis of robot i at axes[k * N + i]), was_reset int32 x N or null; flags int32 x N of 0 / 1
	void parametrizeForceMotionSpaces(const int32_t* dims, const double* axes, int32_t* was_reset, osc_mem_kind where) {
		check(h(), osc_mft_parametrize_spaces_batched(h(), _id, 0, dims, axes, was_reset, where));
	}
	void parametrizeMomentRotMotionSpaces(const int32_t* dims, const double* axes, int32_t* was_reset, osc_mem_kind where) {
		check(h(), osc_mft_parametrize_spaces_batched(h(), _id, 1, dims, axes, was_reset, where));
	}
	void setClosedLoopForceControl(const int32_t* flags, osc_mem_kind where) { check(h(), osc_mft_set_closed_loop_batched(h(), _id, 0, flags, where)); }
	void setClosedLoopMomentControl(const int32_t* flags, osc_mem_kind where) { check(h(), osc_mft_set_closed_loop_batched(h(), _id, 1, flags, where)); }
	// what the kernels use: dims int32 x N, axes SoA 3 x N, closed_loop int32 x N (any may be null)
	void getForceMotionSpaces(int32_t* dims, double* axes, int32_t* closed_loop, osc_mem_kind where = OSC_MEM_HOST) const {
		check(h(), osc_mft_get_spaces(h(), _id, 0, dims, axes, closed_loop, where));
	}
	void getMomentRotMotionSpaces(int32_t* dims, double* axes, int32_t* closed_loop, osc_mem_kind where = OSC_MEM_HOST) const {
		check(h(), osc_mft_get_spaces(h(), _id, 1, dims, axes, closed_loop, where));
	}
	void enablePassivity(int ring_capacity = 0) { check(h(), osc_mft_enable_passivity(h(), _id, 1, ring_capacity)); }
	void disablePassivity() { check(h(), osc_mft_enable_passivity(h(), _id, 0, 0)); }
	void setForceSensorFrame(const std::string& link_name, const Affine& transformation_in_link) {
		if (link_name != _link_name)
			throw std::invalid_argument("The link to which is attached the sensor should be the same as the link to which is attached the "
										"control frame in MotionForceTask::setForceSensorFrame\n");
		check(h(), osc_mft_set_force_sensor_frame(h(), _id, transformation_in_link.R.data(), transformation_in_link.t.data()));
	}
	// per-robot sensed wrench in the sensor frame, SoA 3 x N each
	void updateSensedForceAndMoment(const double* force_soa, const double* moment_soa, osc_mem_kind w = OSC_MEM_HOST) {
		check(h(), osc_mft_update_sensed_force_and_moment(h(), _id, force_soa, moment_soa, w));
	}
	void resetIntegrators() { check(h(), osc_mft_reset_integrators(h(), _id, 0)); }
	void resetIntegratorsLinear() { check(h(), osc_mft_reset_integrators(h(), _id, 1)); }
	void resetIntegratorsAngular() { check(h(), osc_mft_reset_integrators(h(), _id, 2)); }
	// MotionForceTask.cpp:511-523
	void enableInternalOtgAccelerationLimited(double max_linear_velelocity, double max_linear_acceleration, double max_angular_velocity,
											  double max_angular_acceleration) {
		check(h(), osc_mft_enable_internal_otg(h(), _id, max_linear_velelocity, max_linear_acceleration, max_angular_velocity, max_angular_acceleration));
	}
	void enableInternalOtgJerkLimited(double, double, double, double, double, double) { throw std::logic_error("the jerk-limited internal OTG is not built"); }
	void disableInternalOtg() { check(h(), osc_disable_internal_otg(h(), _id)); }
	bool getInternalOtgEnabled() const { return osc_internal_otg_enabled(h(), _id) == 1; }
	// MotionForceTask.h:249-266 (SoA out)
	void getDesiredPosition(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_DESIRED_POSITION, soa, w); }
	void getDesiredOrientation(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_DESIRED_ORIENTATION, soa, w); }
	void getDesiredLinearVelocity(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_DESIRED_LINEAR_VELOCITY, soa, w); }
	void getDesiredAngularVelocity(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_DESIRED_ANGULAR_VELOCITY, soa, w); }
	void getDesiredLinearAcceleration(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_DESIRED_LINEAR_ACCELERATION, soa, w); }
	void getDesiredAngularAcceleration(double* soa, osc_mem_kind w = OSC_MEM_HOST) const { get(OSC_MFT_DESIRED_ANGULAR_ACCELERATION, soa, w); }

private:
	void defaultOtg() {	 // MotionForceTask.h:67-74, MotionForceTask.cpp:170-191
		enableInternalOtgAccelerationLimited(0.3, 2.0, 3.14159265358979323846 / 3.0, 2.0 * 3.14159265358979323846);
	}
	osc_mft_desc base_desc(const std::string& link_name, const Affine& c, bool in_compliant, double dt) {
		osc_mft_desc d{};
		d.link = _robot->linkFrame(link_name);
		for (int k = 0; k < 9; k++) d.compliant_R[k] = c.R[k];
		for (int k = 0; k < 3; k++) d.compliant_t[k] = c.t[k];
		d.force_motion_in_compliant_frame = in_compliant ? 1 : 0;
		d.loop_timestep = dt;
		return d;
	}
	osc_mft_params params() const {
		osc_mft_params p;
		check(h(), osc_mft_get_params(h(), _id, &p));
		return p;
	}
	void apply(const osc_mft_params& p) { check(h(), osc_mft_set_params(h(), _id, &p)); }
	std::string _link_name;
};

// src/RobotController.h:30-112
class RobotController {
public:
	struct DefaultParameters {
		static constexpr bool enable_gravity_compensation = false;
		static constexpr bool enable_joint_limit_avoidance = false;
		static constexpr bool enable_torque_saturation = false;
	};
	// use_previous_torques = false reproduces the manual sum of examples/04-task_and_redundancy (computeTorques() without argument)
	RobotController(std::shared_ptr<BatchedRobot>& robot, std::vector<std::shared_ptr<TemplateTask>>& tasks, bool use_previous_torques = true)
		: _robot(robot) {
		if (tasks.empty()) throw std::invalid_argument("RobotController must have at least one task");
		for (size_t i = 0; i < tasks.size(); i++) {
			auto& task = tasks[i];
			if (task->getConstRobotModel() != _robot) throw std::invalid_argument("All tasks must have the same robot model in RobotController");
			for (auto& n : _task_names)
				if (n == task->getTaskName()) throw std::invalid_argument("Tasks in RobotController must have unique names");
			if (task->id() != (int)i) throw std::invalid_argument("tasks must be listed in the order they were constructed on this robot");
			_task_names.push_back(task->getTaskName());
			_tasks.push_back(task);
		}
		check(_robot->handle(), osc_finalize_controller(_robot->handle(), use_previous_torques ? 1 : 0));
	}
	void updateControllerTaskModels() { check(_robot->handle(), osc_update_task_models(_robot->handle())); }
	// control torques of every robot, SoA dof x N
	void computeControlTorques(double* tau_soa, osc_mem_kind where = OSC_MEM_HOST) {
		check(_robot->handle(), osc_compute_control_torques(_robot->handle(), tau_soa, where));
	}
	std::vector<double> computeControlTorques() {
		std::vector<double> tau((size_t)_robot->dof() * _robot->numRobots());
		computeControlTorques(tau.data(), OSC_MEM_HOST);
		return tau;
	}
	// setQ/setDq/updateModel + updateControllerTaskModels + computeControlTorques in one launch
	void step(const double* q, const double* dq, double* tau, osc_mem_kind where) { check(_robot->handle(), osc_step(_robot->handle(), q, dq, tau, where)); }
	// optional single-precision mode of the fused kernel (no reference counterpart; sai_b200_osc.h, osc_set_precision)
	void setPrecision(osc_precision precision) { check(_robot->handle(), osc_set_precision(_robot->handle(), precision)); }
	osc_precision getPrecision() const { return (osc_precision)osc_get_precision(_robot->handle()); }
	void enableGravityCompensation(bool on) { check(_robot->handle(), osc_enable_gravity_compensation(_robot->handle(), on)); }
	void enableJointLimitAvoidance(bool on) { check(_robot->handle(), osc_enable_joint_limit_avoidance(_robot->handle(), on)); }
	void enableTorqueSaturation(bool on) { check(_robot->handle(), osc_enable_torque_saturation(_robot->handle(), on)); }
	void reinitializeTasks() { check(_robot->handle(), osc_reinitialize_task(_robot->handle(), -1)); }
	void reinitializeTasks(const int32_t* mask, osc_mem_kind where) {
		check(_robot->handle(), osc_reset_robots(_robot->handle(), -1, mask, where, OSC_RESET_REINITIALIZE));
	}
	// episode reset (no reference counterpart): every task of the selected robots as right after construction at the current state
	// (osc_reset_robots, OSC_RESET_CONSTRUCT); mask == nullptr: every robot
	void resetRobots(const int32_t* mask = nullptr, osc_mem_kind where = OSC_MEM_HOST) {
		check(_robot->handle(), osc_reset_robots(_robot->handle(), -1, mask, where, OSC_RESET_CONSTRUCT));
	}
	std::shared_ptr<JointTask> getJointTaskByName(const std::string& task_name) {
		for (auto& t : _tasks)
			if (t->getTaskName() == task_name) {
				if (t->getTaskType() != JOINT_TASK)
					throw std::invalid_argument("Task " + task_name + " is not a JointTask, and cannot be casted as such in RobotController::GetTaskByName");
				return std::dynamic_pointer_cast<JointTask>(t);
			}
		throw std::invalid_argument("Task " + task_name + " not found in RobotController::GetTaskByName");
	}
	std::shared_ptr<MotionForceTask> getMotionForceTaskByName(const std::string& task_name) {
		for (auto& t : _tasks)
			if (t->getTaskName() == task_name) {
				if (t->getTaskType() != MOTION_FORCE_TASK)
					throw std::invalid_argument("Task " + task_name + " is not a MotionForceTask, and cannot be casted as such in RobotController::GetTaskByName");
				return std::dynamic_pointer_cast<MotionForceTask>(t);
			}
		throw std::invalid_argument("Task " + task_name + " not found in RobotController::GetTaskByName");
	}

private:
	std::shared_ptr<BatchedRobot> _robot;
	std::vector<std::shared_ptr<TemplateTask>> _tasks;
	std::vector<std::string> _task_names;
};

// Simulation side of the loop for N robots (SURVEY.md row f-1) with the method names the reference examples use on
// sai-simulation (examples/05-using_robot_controller/05-using_robot_controller.cpp:223-231).  q, dq and tau are
// caller-owned SoA arrays (dof x N), host or device; integrate() advances q and dq in place.
class BatchedSimulation {
public:
	BatchedSimulation(std::shared_ptr<BatchedRobot>& robot, double* q, double* dq, osc_mem_kind where = OSC_MEM_HOST)
		: _robot(robot), _q(q), _dq(dq), _where(where) {}
	void setTimestep(double dt) { _dt = dt; }
	void setJointTorques(const double* tau) { _tau = tau; }
	void integrate(int substeps = 1) {
		if (!_tau) throw std::invalid_argument("BatchedSimulation::integrate: no joint torques set");
		check(_robot->handle(), osc_sim_integrate(_robot->handle(), _q, _dq, _tau, _dt, substeps, _where));
	}
	const double* getJointPositions() const { return _q; }
	const double* getJointVelocities() const { return _dq; }

private:
	std::shared_ptr<BatchedRobot> _robot;
	double* _q;
	double* _dq;
	const double* _tau = nullptr;
	double _dt = 0.001;
	osc_mem_kind _where;
};

}  // namespace SaiPrimitivesB200
