/*
 * sai_b200_osc.h -- C ABI of the B200-native batched operational-space controller.
 *
 * The reference (manips-sai-org/sai-primitives) has no FFI: its boundary for this
 * path is the C++ virtual interface TemplateTask (src/tasks/TemplateTask.h:26-124)
 * consumed by RobotController (src/RobotController.cpp:68-118), plus the concrete
 * setters of JointTask / MotionForceTask.  Every entry point below names the
 * reference interface it replaces.  One handle evaluates the control law for
 * n_robots independent robots that share one model and one task hierarchy, on one
 * CUDA device; robots are sharded across devices by creating one handle per device.
 *
 * Conventions
 *   - all floating point data is IEEE FP64;
 *   - per-robot arrays are structure-of-arrays, component-major: element
 *     (component c, robot i) lives at  data[c * n_robots + i];
 *     3x3 matrices are 9 components, row-major;
 *   - mem_kind says where a caller buffer lives (OSC_MEM_HOST / OSC_MEM_DEVICE);
 *     host buffers are copied inside the call, device buffers are used in stream order;
 *   - every function returns OSC_OK (0) or a negative osc_status; osc_last_error()
 *     gives the message.  The C++ wrappers in include/sai_b200/ re-throw
 *     std::invalid_argument where the reference throws it;
 *   - a handle is single-caller (like the reference's tasks); calls are asynchronous
 *     on the handle's stream unless they return data to a host buffer.
 *   - there is NO CPU fallback: without a CUDA device osc_create fails.
 */
#ifndef SAI_B200_OSC_H_
#define SAI_B200_OSC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OSC_MAX_DOF 8
#define OSC_MAX_TASKS 4
#define OSC_ABI_VERSION 2

typedef enum {
	OSC_OK = 0,
	OSC_ERR_INVALID_ARGUMENT = -1, /* what the reference reports with std::invalid_argument */
	OSC_ERR_UNSUPPORTED = -2,	   /* feature excluded from the path (internal OTG, JLA) or signature not compiled */
	OSC_ERR_CUDA = -3,			   /* sticky CUDA error, see osc_last_error */
	OSC_ERR_NO_DEVICE = -4,
	OSC_ERR_STATE = -5			   /* call order violated (e.g. tasks added after finalize) */
} osc_status;

typedef enum { OSC_MEM_HOST = 0, OSC_MEM_DEVICE = 1 } osc_mem_kind;

/* reference src/helper_modules/SaiPrimitivesCommonDefinitions.h:14-20 */
typedef enum {
	OSC_FULL_DYNAMIC_DECOUPLING = 0,
	OSC_BOUNDED_INERTIA_ESTIMATES = 1,
	OSC_IMPEDANCE = 2
} osc_decoupling_type;

/* reference src/tasks/TemplateTask.h:19-24 */
typedef enum { OSC_TASK_JOINT = 2, OSC_TASK_MOTION_FORCE = 3 } osc_task_type;

/* per-robot status bits, osc_get_status() */
#define OSC_STATUS_SINGULAR_PATH 0x1u	 /* robot went through the singular (SVD) path this cycle */
#define OSC_STATUS_NAN_SCRUBBED 0x2u	 /* SingularityHandler.cpp:357-359 replaced a NaN torque by 0 */
#define OSC_STATUS_ZERO_RANGE 0x4u		 /* a joint task had no controllable dof left (JointTask.cpp:234-239) */
#define OSC_STATUS_POPC_OVERFLOW 0x8u	 /* POPC window ring buffer overflowed (oldest sample dropped) */
#define OSC_STATUS_UNHANDLED 0x10u		 /* robot needs a path this build does not have; torque is NaN */
#define OSC_STATUS_TYPE1 0x20u			 /* singular path: type-1 joint strategy active */
#define OSC_STATUS_TYPE2 0x40u			 /* singular path: type-2 joint strategy active */

/* Serial-chain robot model after fixed-joint bodies have been merged into their
 * parent (what sai-model/RBDL hands the reference).  Body i is moved by joint i,
 * its parent is body i-1 (body -1 = world).  Replaces the SaiModel object the
 * reference tasks hold (TemplateTask.h:119). */
typedef struct {
	int32_t n;						   /* degrees of freedom, 1..OSC_MAX_DOF */
	int32_t jtype[OSC_MAX_DOF];		   /* 0 revolute, 1 prismatic */
	double axis[OSC_MAX_DOF][3];	   /* unit joint axis in the joint frame */
	double R_fix[OSC_MAX_DOF][9];	   /* parent body frame -> joint frame at q=0, row-major */
	double t_fix[OSC_MAX_DOF][3];
	double mass[OSC_MAX_DOF];
	double com[OSC_MAX_DOF][3];		   /* centre of mass in the body frame */
	double inertia[OSC_MAX_DOF][9];	   /* about the com, body axes, row-major symmetric */
	double q_lower[OSC_MAX_DOF], q_upper[OSC_MAX_DOF], dq_max[OSC_MAX_DOF], effort[OSC_MAX_DOF];
	double R_world_base[9], t_world_base[3]; /* SaiModel::TRobotBase */
	double gravity_world[3];
} osc_model_desc;

/* A frame rigidly attached to a body (a URDF link that hangs off body `body` through fixed joints). */
typedef struct {
	int32_t body;
	double R[9];
	double t[3];
} osc_link_frame;

/* MotionForceTask constructor arguments (MotionForceTask.h:96-110). */
typedef struct {
	osc_link_frame link;		 /* resolved link frame */
	double compliant_R[9];		 /* compliant frame w.r.t. the link frame */
	double compliant_t[3];
	int32_t partial;			 /* 0: full 6-dof constructor; 1: direction-list constructor */
	int32_t n_dirs_translation;	 /* 0..3 */
	double dirs_translation[3][3];
	int32_t n_dirs_rotation;	 /* 0..3 */
	double dirs_rotation[3][3];
	int32_t force_motion_in_compliant_frame;
	double loop_timestep;
} osc_mft_desc;

/* Broadcast parameters of one MotionForceTask; defaults = MotionForceTask.h:40-75
 * and SingularityHandler.cpp:10-20, except internal OTG which is excluded. */
typedef struct {
	double kp_pos[3], kv_pos[3], ki_pos[3]; /* diagonal, world axes (MotionForceTask.cpp:581-628) */
	double kp_ori[3], kv_ori[3], ki_ori[3];
	double kp_force, kv_force, ki_force;
	double kp_moment, kv_moment, ki_moment;
	double kff_force, kff_moment;
	double max_force_control_feedback_output, max_moment_control_feedback_output;
	double linear_saturation_velocity, angular_saturation_velocity;
	double bie_threshold;
	double s_min, s_max;				  /* singularity blending bounds (MotionForceTask.cpp:197) */
	double kp_type_1, kv_type_1, kv_type_2;
	double s_abs_tol, type_1_tol, type_2_torque_ratio, type_2_angle_threshold, perturb_step_size;
	double force_or_motion_axis[3], moment_or_rotmotion_axis[3];
	int32_t force_space_dimension, moment_space_dimension;
	int32_t closed_loop_force_control, closed_loop_moment_control;
	int32_t passivity_enabled;
	int32_t use_velocity_saturation;
	int32_t dynamic_decoupling_type;
	int32_t singularity_handling_enabled;
	int32_t enforce_type_1_strategy;
	int32_t buffer_size;
} osc_mft_params;

/* Broadcast parameters of one JointTask; defaults = JointTask.h:31-45 (OTG excluded). */
typedef struct {
	double kp[OSC_MAX_DOF], kv[OSC_MAX_DOF], ki[OSC_MAX_DOF];
	double saturation_velocity[OSC_MAX_DOF];
	double bie_threshold;
	int32_t use_velocity_saturation;
	int32_t dynamic_decoupling_type;
} osc_joint_params;

/* Per-robot fields (osc_set_field / osc_get_field).  ncomp in parentheses; k = joint task dof. */
typedef enum {
	/* MotionForceTask goals: MotionForceTask.h:211-247, :362-385 */
	OSC_MFT_GOAL_POSITION = 0,			   /* (3) */
	OSC_MFT_GOAL_ORIENTATION = 1,		   /* (9) */
	OSC_MFT_GOAL_LINEAR_VELOCITY = 2,	   /* (3) */
	OSC_MFT_GOAL_ANGULAR_VELOCITY = 3,	   /* (3) */
	OSC_MFT_GOAL_LINEAR_ACCELERATION = 4,  /* (3) */
	OSC_MFT_GOAL_ANGULAR_ACCELERATION = 5, /* (3) */
	OSC_MFT_GOAL_FORCE = 6,				   /* (3) as set by setGoalForce (parametrisation frame) */
	OSC_MFT_GOAL_MOMENT = 7,			   /* (3) */
	/* MotionForceTask observers (read only): MotionForceTask.h:121-190, :266 */
	OSC_MFT_CURRENT_POSITION = 8,			  /* (3) */
	OSC_MFT_CURRENT_ORIENTATION = 9,		  /* (9) */
	OSC_MFT_CURRENT_LINEAR_VELOCITY = 10,	  /* (3) */
	OSC_MFT_CURRENT_ANGULAR_VELOCITY = 11,	  /* (3) */
	OSC_MFT_SENSED_FORCE_CONTROL_WORLD = 12,  /* (3) */
	OSC_MFT_SENSED_MOMENT_CONTROL_WORLD = 13, /* (3) */
	OSC_MFT_UNIT_MASS_FORCE = 14,			  /* (6) */
	OSC_MFT_INTEGRATED_POSITION_ERROR = 15,	  /* (3) */
	OSC_MFT_INTEGRATED_ORIENTATION_ERROR = 16, /* (3) */
	OSC_MFT_INTEGRATED_FORCE_ERROR = 17,	  /* (3) */
	OSC_MFT_INTEGRATED_MOMENT_ERROR = 18,	  /* (3) */
	OSC_MFT_POPC_STATE = 19,				  /* (4) passivity observer, E_correction, Rc, sum vcl^2 */
	OSC_MFT_TYPE1_POSTURE = 20,				  /* (n) SingularityHandler::setType1Posture / _q_prior */
	/* computed on request from the state the last osc_compute_control_torques left (read only):
	 * MotionForceTask::getPositionError / getOrientationError (MotionForceTask.cpp:540-546, MotionForceTask.h:268-269),
	 * sigmaForce / sigmaPosition / sigmaMoment / sigmaOrientation (MotionForceTask.cpp:892-971, MotionForceTask.h:613-616) */
	OSC_MFT_POSITION_ERROR = 21,	 /* (3) */
	OSC_MFT_ORIENTATION_ERROR = 22,	 /* (3) */
	OSC_MFT_SIGMA_FORCE = 23,		 /* (9) row-major */
	OSC_MFT_SIGMA_POSITION = 24,	 /* (9) */
	OSC_MFT_SIGMA_MOMENT = 25,		 /* (9) */
	OSC_MFT_SIGMA_ORIENTATION = 26,	 /* (9) */
	/* JointTask: JointTask.h:140-182 */
	OSC_JT_GOAL_POSITION = 32,		 /* (k) */
	OSC_JT_GOAL_VELOCITY = 33,		 /* (k) */
	OSC_JT_GOAL_ACCELERATION = 34,	 /* (k) */
	OSC_JT_INTEGRATED_POSITION_ERROR = 35, /* (k) */
	/* JointTask::getDesiredPosition / Velocity / Acceleration (JointTask.h:162-176): the state the control law tracks -- the
	 * internal OTG's output when it is enabled, the goal otherwise (JointTask.cpp:308-319).  Read only. */
	OSC_JT_DESIRED_POSITION = 36,	  /* (k) */
	OSC_JT_DESIRED_VELOCITY = 37,	  /* (k) */
	OSC_JT_DESIRED_ACCELERATION = 38, /* (k) */
	/* MotionForceTask::getDesired* (MotionForceTask.h:249-266; MotionForceTask.cpp:387-407).  Read only. */
	OSC_MFT_DESIRED_POSITION = 40,			   /* (3) */
	OSC_MFT_DESIRED_ORIENTATION = 41,		   /* (9) */
	OSC_MFT_DESIRED_LINEAR_VELOCITY = 42,	   /* (3) */
	OSC_MFT_DESIRED_ANGULAR_VELOCITY = 43,	   /* (3) */
	OSC_MFT_DESIRED_LINEAR_ACCELERATION = 44,  /* (3) */
	OSC_MFT_DESIRED_ANGULAR_ACCELERATION = 45, /* (3) */
	/* any task: TemplateTask::getTaskNullspace / getPreviousTasksNullspace / getTaskAndPreviousNullspace
	 * (TemplateTask.h:74,82,89; JointTask.h:222-226, MotionForceTask.h:205-209), n x n row-major per robot, read only.
	 * Evaluated on request from the handle's current state: what updateControllerTaskModels() yields at that state. */
	OSC_TASK_NULLSPACE = 48,				/* (n*n) */
	OSC_TASK_PREVIOUS_NULLSPACE = 49,		/* (n*n) */
	OSC_TASK_AND_PREVIOUS_NULLSPACE = 50	/* (n*n) */
} osc_field;

typedef struct osc_handle osc_handle;

/* ---- library ---- */
int osc_abi_version(void);
/* message of the last failing call on this handle (or of osc_create when h == NULL) */
const char* osc_last_error(const osc_handle* h);

/* ---- built-in robot models (data from the reference's URDF files, see DESIGN.md) ---- */
/* names: "panda", "panda_sliding_base", "rrrr", "puma_like" */
int osc_builtin_model(const char* robot_name, osc_model_desc* out);
int osc_builtin_link(const char* robot_name, const char* link_name, osc_link_frame* out);

/* ---- URDF models (SURVEY.md row f-3).  Replaces std::make_shared<SaiModel::SaiModel>(robot_file)
 * (examples/05-using_robot_controller/05-using_robot_controller.cpp:64) for serial chains: links attached through
 * fixed joints are merged into their parent body, the root link is welded to the world.  The model is registered
 * under `model_name` and then served by osc_builtin_model / osc_builtin_link like the built-in ones (set
 * R_world_base / t_world_base of the description for SaiModel::setTRobotBase). ---- */
int osc_urdf_register(const char* model_name, const char* urdf_xml);
int osc_urdf_register_file(const char* model_name, const char* path);
const char* osc_urdf_last_error(void);
/* SaiModel::URDF_FOLDERS[prefix_name] = folder and SaiModel::ReplaceUrdfPathPrefix (examples/01-joint_control/01-joint_control.cpp:40-71):
 * "${PREFIX}/file" in any path handed to this library is replaced by the registered folder. */
int osc_urdf_set_folder(const char* prefix_name, const char* folder);
int osc_urdf_replace_path_prefix(const char* path, char* out, int out_capacity);
/* World file (examples/15-haptic_control_impedance_type/world.urdf): <world gravity="..."><robot name="R"><model dir="${...}" path="x.urdf"/>
 * <origin xyz rpy/></robot>...  Loads the URDF of robot `robot_name_in_world`, registers it under `model_name` and sets the
 * description's R_world_base / t_world_base to the robot's <origin>: sim->getRobotBaseTransform(name) + robot->setTRobotBase(T)
 * (examples/15-...cpp:124-126).  gravity_out (may be NULL) receives the world's gravity attribute. */
int osc_world_register_robot(const char* world_file, const char* robot_name_in_world, const char* model_name, double gravity_out[3]);

/* ---- lifetime.  Replaces make_shared<SaiModel>(urdf) + task/controller construction ---- */
int osc_create(const osc_model_desc* model, int64_t n_robots, int device, osc_handle** out);
int osc_destroy(osc_handle* h);
/* run on a caller-owned CUDA stream (cudaStream_t passed as void*); NULL restores the handle's own stream */
int osc_set_stream(osc_handle* h, void* cuda_stream);
int osc_sync(osc_handle* h);
int64_t osc_num_robots(const osc_handle* h);
int osc_dof(const osc_handle* h);

/* ---- robot state.  Replaces SaiModel::setQ / setDq / updateModel (examples/05-...cpp:143-145) ---- */
int osc_set_state(osc_handle* h, const double* q, const double* dq, int mem_kind);

/* ---- task construction, in hierarchy order.  The new task is initialised from the current
 *      state exactly like the reference constructors (JointTask.cpp:45-107, MotionForceTask.cpp:92-245). */
/* JointTask(robot, name, dt) / JointTask(robot, S, name, dt): selection == NULL -> full joint task;
 * otherwise row-major k x n (JointTask.h:56-75) */
int osc_add_joint_task(osc_handle* h, const double* selection, int k, double loop_timestep, int* task_id);
/* MotionForceTask(robot, link, compliant_frame, ...) both constructors (MotionForceTask.h:96-110) */
int osc_add_motion_force_task(osc_handle* h, const osc_mft_desc* desc, int* task_id);
/* RobotController(robot, tasks): validates the hierarchy (RobotController.cpp:27-59) and selects the kernel.
 * use_previous_torques = 1 reproduces RobotController::computeControlTorques (each task is given the sum of the
 * previous torques); 0 reproduces the manual sum of examples/04-...cpp:188-206 (computeTorques() without argument). */
int osc_finalize_controller(osc_handle* h, int use_previous_torques);
int osc_num_tasks(const osc_handle* h);
int osc_get_task_type(const osc_handle* h, int task_id);
int osc_get_task_dof(const osc_handle* h, int task_id); /* joint task: k; motion-force task: pos_range + ori_range */

/* ---- broadcast parameters ---- */
int osc_mft_default_params(osc_mft_params* p);
int osc_mft_get_params(const osc_handle* h, int task_id, osc_mft_params* p);
/* plain parameter update: gains, saturation, decoupling, singularity knobs.  Fields with side effects
 * (force/moment space, closed loop flags, passivity) must go through the dedicated calls below and are
 * rejected here when they differ from the current value. */
int osc_mft_set_params(osc_handle* h, int task_id, const osc_mft_params* p);
/* MotionForceTask::parametrizeForceMotionSpaces (MotionForceTask.cpp:830-858); *was_reset mirrors its return value */
int osc_mft_parametrize_force_motion_spaces(osc_handle* h, int task_id, int dim, const double axis[3], int* was_reset);
/* MotionForceTask::parametrizeMomentRotMotionSpaces (MotionForceTask.cpp:860-890) */
int osc_mft_parametrize_moment_rotmotion_spaces(osc_handle* h, int task_id, int dim, const double axis[3], int* was_reset);
/* MotionForceTask::setClosedLoopForceControl / setClosedLoopMomentControl (MotionForceTask.cpp:973-986) */
int osc_mft_set_closed_loop_force_control(osc_handle* h, int task_id, int enabled);
int osc_mft_set_closed_loop_moment_control(osc_handle* h, int task_id, int enabled);
/* MotionForceTask::enablePassivity / disablePassivity (MotionForceTask.h:630-631).
 * ring_capacity: samples of the POPC window kept per robot (the reference queue is unbounded,
 * POPCExplicitForceControl.cpp:47-61); <= 0 selects the default 1024. */
int osc_mft_enable_passivity(osc_handle* h, int task_id, int enabled, int ring_capacity);
/* MotionForceTask::setForceSensorFrame (MotionForceTask.cpp:794-803): sensor frame w.r.t. the task's link frame */
int osc_mft_set_force_sensor_frame(osc_handle* h, int task_id, const double R_in_link[9], const double t_in_link[3]);
/* MotionForceTask::updateSensedForceAndMoment (MotionForceTask.cpp:805-828), per robot, (3)+(3) SoA;
 * evaluated with the state of the latest osc_set_state */
int osc_mft_update_sensed_force_and_moment(osc_handle* h, int task_id, const double* force_sensor_frame,
										   const double* moment_sensor_frame, int mem_kind);
/* MotionForceTask::resetIntegrators{,Linear,Angular} (MotionForceTask.cpp:988-1001): which = 0 both, 1 linear, 2 angular */
int osc_mft_reset_integrators(osc_handle* h, int task_id, int which);

int osc_joint_default_params(osc_joint_params* p);
int osc_joint_get_params(const osc_handle* h, int task_id, osc_joint_params* p);
int osc_joint_set_params(osc_handle* h, int task_id, const osc_joint_params* p);

/* ---- per-robot control gains.  JointTask::setGains (JointTask.cpp), MotionForceTask::setPosControlGains /
 * setOriControlGains / setForceControlGains / setMomentControlGains (MotionForceTask.cpp:581-628), each robot of the batch
 * with its own values (gain sweeps, randomised gains, variable-impedance policies).  Components per robot (ncomp): joint k,
 * position and orientation 3 (diagonal, world axes), force and moment 1.  Only these PID gains can be per robot; the
 * feed-forward gains, the maximum feedback outputs, the saturation velocities, the bounded-inertia thresholds, the
 * singularity handler's gains and bounds and the OTG limits stay broadcast parameters.
 *   per_robot = 0: kp, kv, ki hold ncomp host values each, applied to every robot.
 *   per_robot = 1: kp, kv, ki are SoA ncomp x n_robots each, host or device memory (mem_kind).  Device input is checked by a
 *                  reduction kernel and the call synchronises the handle's stream.
 * Every value of the three arrays is checked before anything is written: joint, position and orientation gains must be finite
 * and >= 0, force and moment gains finite (the reference accepts any value there).  A violation returns
 * OSC_ERR_INVALID_ARGUMENT and leaves the gains as they were.  (The finiteness check is the one difference from the gain update of
 * osc_mft_set_params / osc_joint_set_params, which checks the sign only.)
 * The first per_robot = 1 call on a task allocates its gain block (24 doubles per robot), fills it with the current broadcast
 * gains of every group and then writes the given group; from then on the kernels read that task's gains from the block (there
 * is no way back), a per_robot = 0 call writes the group for every robot, and osc_mft_set_params / osc_joint_set_params
 * return OSC_ERR_STATE when a gain member differs from its current broadcast value (other members stay settable).  Before
 * the first per_robot = 1 call, per_robot = 0 is the gain update osc_*_set_params makes; after it, osc_*_get_params keeps
 * returning the broadcast gains the task had when it entered per-robot mode, and osc_get_gains is what the kernels use.
 * osc_reinitialize_task leaves the gains alone.  While a task of the handle has per-robot gains, osc_compute_control_torques / osc_step return
 * OSC_ERR_UNSUPPORTED in the FP32 mode.  Writes are ordered with the control cycles in the handle's stream like goal writes.
 * osc_get_gains returns ncomp x n_robots per array in either mode. ---- */
typedef enum {
	OSC_GAINS_JOINT = 0,
	OSC_GAINS_POSITION = 1,
	OSC_GAINS_ORIENTATION = 2,
	OSC_GAINS_FORCE = 3,
	OSC_GAINS_MOMENT = 4
} osc_gain_group;
int osc_set_gains(osc_handle* h, int task_id, int group, const double* kp, const double* kv, const double* ki, int mem_kind,
				  int per_robot);
int osc_get_gains(osc_handle* h, int task_id, int group, double* kp, double* kv, double* ki, int mem_kind);

/* ---- per-robot force / moment spaces and closed-loop flags.  MotionForceTask::parametrizeForceMotionSpaces /
 * parametrizeMomentRotMotionSpaces (MotionForceTask.cpp:830-890) and setClosedLoopForceControl / setClosedLoopMomentControl
 * (:973-986), each robot of the batch with its own values (robots that touch their surfaces on different cycles and along
 * different normals).  which = 0: force / motion space and closed-loop force control; which = 1: moment / rot-motion space and
 * closed-loop moment control.  Passivity, in_compliant, the selection, the force sensor frame and the feed-forward and
 * saturation parameters stay task-wide.
 *   osc_mft_parametrize_spaces_batched: dims int32 x n_robots (0..3), axes SoA 3 x n_robots (read for robots of dimension 1 or
 *     2 only), was_reset int32 x n_robots or NULL, all in mem_kind memory.  Robot i gets exactly what parametrize*(dims[i],
 *     axis_i) does to a task object of the reference: the axis is normalised (dimension 0 or 3: the stored axis stays), and
 *     the robot is reset when its dimension changes or its normalised axis is not Eigen's isApprox to the stored one -- goal
 *     position (orientation) := current, linear (angular) velocity and acceleration goals := 0, position and force
 *     (orientation and moment) integrators := 0; with the internal OTG on, its generator is re-initialised linearly (angularly)
 *     instead of the goal copy.  was_reset[i] = 1 for a robot that was reset.  Robots that are not reset are left untouched.
 *   osc_mft_set_closed_loop_batched: enabled int32 x n_robots (0 or 1).  A robot whose flag changes gets its linear (force) or
 *     angular (moment) integrators zeroed.  POPC state advances only for robots with closed-loop force control on.
 *   osc_mft_get_spaces: what the kernels use, in either mode: dims int32 x n_robots, axes SoA 3 x n_robots (normalised),
 *     closed_loop int32 x n_robots; any pointer may be NULL.
 * Every value is checked before anything is written: a dimension outside 0..3, an axis of a dimension-1/2 robot that is not
 * finite or shorter than 1e-2, or a flag other than 0/1 returns OSC_ERR_INVALID_ARGUMENT with the reference's message and
 * leaves every robot as it was.  Device input is checked by a reduction kernel and the call synchronises the handle's stream;
 * host input and output synchronise too.  Writes are ordered with the control cycles in the handle's stream like goal writes.
 * The first batched call on a task allocates its space block (one int32 and 6 doubles per robot), fills it from the task's
 * broadcast parameters and then applies the call; there is no way back.  From then on osc_mft_parametrize_* and
 * osc_mft_set_closed_loop_* apply the same values to every robot through the per-robot path, each robot deciding its own
 * reset (*was_reset = 1 if any robot was reset), osc_mft_set_params keeps rejecting changes to these fields, and
 * osc_mft_get_params reports the values of the last broadcast call.
 * While every robot of the task is in free motion (dimension 0 in both spaces, both loops open) the launch selects the same
 * pure-motion kernels as for a broadcast task, which never read the block; once one robot is not, the force-capable kernels.
 * The FP32 mode follows the same rule: it runs while every robot is in free motion and returns OSC_ERR_UNSUPPORTED otherwise.
 * ---- */
int osc_mft_parametrize_spaces_batched(osc_handle* h, int task_id, int which, const int32_t* dims, const double* axes, int32_t* was_reset,
									   int mem_kind);
int osc_mft_set_closed_loop_batched(osc_handle* h, int task_id, int which, const int32_t* enabled, int mem_kind);
int osc_mft_get_spaces(osc_handle* h, int task_id, int which, int32_t* dims, double* axes, int32_t* closed_loop, int mem_kind);

/* ---- internal online trajectory generation (SURVEY.md row f-4).  The reference interpolates every task's goal with its
 * vendored Ruckig by default (JointTask.h:38-42, MotionForceTask.h:67-74): acceleration-limited, phase-synchronised.  Tasks are
 * created here with the generator OFF (BASELINE.json runs with it off, and so do the reference's examples that call
 * disableInternalOtg()); the host mirrors switch it on in their constructors to keep the reference's default.
 *   JointTask::enableInternalOtgAccelerationLimited (JointTask.cpp:358-380): k max velocities and k max accelerations (> 0);
 *   MotionForceTask::enableInternalOtgAccelerationLimited (MotionForceTask.cpp:511-523);
 *   disableInternalOtg (JointTask.h:310, MotionForceTask.h:425); getInternalOtgEnabled.
 * The jerk-limited variants (enableInternalOtgJerkLimited) are not built: OSC_ERR_UNSUPPORTED through the mirrors.
 * While the generator is on, the goal fields hold the user's goals and the OSC_*_DESIRED_* fields its output. ---- */
int osc_joint_enable_internal_otg(osc_handle* h, int task_id, const double* max_velocity, const double* max_acceleration);
int osc_mft_enable_internal_otg(osc_handle* h, int task_id, double max_linear_velocity, double max_linear_acceleration,
								double max_angular_velocity, double max_angular_acceleration);
int osc_disable_internal_otg(osc_handle* h, int task_id);
int osc_internal_otg_enabled(const osc_handle* h, int task_id);
/* per-robot generator flags of a task (int32 x N): 1 goal reached, 2 recalculation pending, 4 the last update failed (Ruckig
 * error branch, OTG_joints.cpp:141-149: output held, velocity reset), 8 finished with a residual velocity */
int osc_get_internal_otg_flags(osc_handle* h, int task_id, int32_t* flags_out, int mem_kind);

/* ---- per-robot fields.  broadcast != 0: data holds ncomp values applied to every robot (host memory only) ---- */
int osc_field_ncomp(const osc_handle* h, int task_id, int field);
int osc_set_field(osc_handle* h, int task_id, int field, const double* data, int mem_kind, int broadcast);
int osc_get_field(osc_handle* h, int task_id, int field, double* out, int mem_kind);

/* ---- re-initialisation.  TemplateTask::reInitializeTask (JointTask.cpp:91-107, MotionForceTask.cpp:204-245);
 *      task_id < 0: RobotController::reinitializeTasks (RobotController.cpp:120-125).  Every robot; the same as
 *      osc_reset_robots(h, task_id, NULL, OSC_MEM_DEVICE, OSC_RESET_REINITIALIZE) ---- */
int osc_reinitialize_task(osc_handle* h, int task_id);

/* ---- per-robot resets (episode ends of batched rollouts: a robot moved to a new state starts its controller over there).
 *   robot_mask: int32 x n_robots in mem_kind memory, a non-zero entry selects the robot; NULL selects every robot.  Any int32 is
 *     a valid entry, so a device mask is never read by the host: the call is asynchronous and ordered with the control cycles
 *     in the handle's stream like a goal write.  A host mask is copied into a handle-owned device buffer with cudaMemcpyAsync;
 *     a pageable one may be reused when the call returns, a page-locked one must stay unchanged until the stream has reached
 *     the call.
 *   task_id < 0: every task of the handle, in hierarchy order (RobotController::reinitializeTasks); otherwise that task.
 *   The reset is evaluated at the state of the latest osc_set_state / osc_step (device state buffers are borrowed, so values
 *   written into them earlier in the handle's stream are the ones seen).
 *   OSC_RESET_REINITIALIZE: TemplateTask::reInitializeTask for each selected robot, i.e. what osc_reinitialize_task does,
 *     restricted to those robots: goals := current pose / position with zero velocity, acceleration, force and moment goals,
 *     integrators and sensed wrench zeroed; a task with the internal OTG on has its generator re-initialised at the current
 *     pose.  The singularity handler's memory and the POPC state stay, as in the reference.
 *   OSC_RESET_CONSTRUCT: the state the tasks had right after construction at the current state (what osc_add_*_task leaves),
 *     with the generator of a task that has the internal OTG on constructed anew as enabling it does.  On top of the above,
 *     the singularity handler's memory is reset (type-1 posture _q_prior to mid-range -- so a posture set with
 *     OSC_MFT_TYPE1_POSTURE is reset too --, type-2 directions, counters and history) and so are the POPC observer and window.
 *   Configuration is never touched by either mode: broadcast parameters, per-robot gains, per-robot spaces and closed-loop
 *   flags, passivity on/off and ring capacity, the force sensor frame, the OTG's enabled flag and limits.  Robots that are not
 *   selected are not written.  A bad task_id, mode or mem_kind returns OSC_ERR_INVALID_ARGUMENT and changes nothing.  One
 *   kernel launch per call, whatever the number of tasks. ---- */
typedef enum { OSC_RESET_REINITIALIZE = 0, OSC_RESET_CONSTRUCT = 1 } osc_reset_mode;
int osc_reset_robots(osc_handle* h, int task_id, const int32_t* robot_mask, int mem_kind, int mode);

/* ---- controller options (RobotController.h:66-76) ---- */
int osc_enable_gravity_compensation(osc_handle* h, int enabled);
int osc_enable_torque_saturation(osc_handle* h, int enabled);
/* RobotController::enableJointLimitAvoidance (RobotController.h:70-72): JointLimitAvoidanceTask with its default zones
 * and gains (JointLimitAvoidanceTask.h:26-35) blended into the torques as in RobotController.cpp:96-112. */
int osc_enable_joint_limit_avoidance(osc_handle* h, int enabled);

/* ---- the control cycle ---- */
/* RobotController::updateControllerTaskModels (RobotController.cpp:68-77).  The task models are a pure function
 * of the state; the call arms the (stateful) singularity classification for the next torque computation. */
int osc_update_task_models(osc_handle* h);
/* RobotController::computeControlTorques (RobotController.cpp:79-118): tau_out is (n) SoA */
int osc_compute_control_torques(osc_handle* h, double* tau_out, int mem_kind);
/* fused cycle: set_state + update_task_models + compute_control_torques in one launch */
int osc_step(osc_handle* h, const double* q, const double* dq, double* tau_out, int mem_kind);
/* osc_step without the final synchronisation: with OSC_MEM_HOST the buffers must be page-locked and stay valid (and
 * tau_out unread) until osc_sync(h) returns; lets a caller pipeline the host<->device copies of several handles */
int osc_step_async(osc_handle* h, const double* q, const double* dq, double* tau_out, int mem_kind);
int osc_get_status(osc_handle* h, uint32_t* flags_out, int mem_kind);
/* Per-cycle observers of MotionForceTask that the torques do not need: getCurrentLinearVelocity / getCurrentAngularVelocity /
 * getUnitMassForce (MotionForceTask.h:121-129, :266) and the orientation error behind getOrientationError.  The reference
 * refreshes them in every computeTorques (MotionForceTask.cpp:291-298, :478); so does this library by default (enabled = 1).
 * With enabled = 0 the cycle kernels skip the 15 stores per robot and reading those fields returns OSC_ERR_STATE. */
int osc_enable_observers(osc_handle* h, int enabled);
/* Contiguous shard of a batch (SURVEY.md 8e): robots [*first, *first + *count) of n_robots belong to shard `rank` of
 * `world` (robot i -> shard floor(i * world / n_robots)).  One handle per device is created with *count robots; no call of
 * this library ever exchanges data between handles. */
int osc_shard_range(int64_t n_robots, int rank, int world, int64_t* first, int64_t* count);
/* number of kernels this handle has launched since creation (bench.py's gpu_launches) */
int64_t osc_launch_count(const osc_handle* h);

/* ---- kinematics/dynamics stage on its own (parity checks against the sai-model restatement) ----
 * For the link frame + point of motion-force task `task_id` (or, when task_id < 0, of `frame` and `point`):
 *   M (n*n, row-major), J (6*n row-major, linear rows first: SaiModel::JWorldFrame), x (3), R (9), g (n).
 * Any output pointer may be NULL. */
/* ---- test probe: n_steps consecutive POPCExplicitForceControl::computePassivitySaturatedForce calls
 * (POPCExplicitForceControl.cpp:30-96, kv_force = kv * I as MotionForceTask.h:308 builds it) on the POPC state of every
 * robot of the task, host inputs n_steps x 3 row major shared by all robots, out = the results of robot 0.  Passivity
 * must be enabled on the task.  Lets the device code be checked against vectors produced by the reference's own source
 * (tests/golden/popc_reference.npz). ---- */
int osc_debug_popc_sequence(osc_handle* h, int task_id, int n_steps, const double* fd, const double* fs, const double* vcl,
							const double* vr, double kv_force, double kff_force, double* out);

/* ---- optional single-precision mode (BASELINE.json north_star: "an optional FP32 mode is held to 1e-4 relative and reported
 * separately"; the reference itself is double precision throughout, e.g. RobotController.cpp:75-120).  OSC_PRECISION_FP32 runs
 * the fused kernel of the flagship hierarchy -- a full six-dof MotionForceTask under pure motion control, alone or with a full
 * JointTask in its null space, on a robot whose joints are all revolute about their local z axis (seven joints compiled in) --
 * in FP32 arithmetic.  All data in device memory (state, goals, integrators, torques) stay FP64, and robots inside the
 * singularity band continue on the FP64 general path.  A hierarchy outside that description makes
 * osc_compute_control_torques / osc_step return OSC_ERR_UNSUPPORTED while the mode is on; there is no silent fallback. ---- */
typedef enum { OSC_PRECISION_FP64 = 0, OSC_PRECISION_FP32 = 1 } osc_precision;
int osc_set_precision(osc_handle* h, int precision);
int osc_get_precision(osc_handle* h);

/* ---- measurement aid (no reference counterpart): %globaltimer stamps of every block of the fused kernel over the last 8 cycles,
 * so that the overlap of consecutive cycles can be looked at (tools/pipeline_trace.py).  out == NULL: switch the stamps on / off;
 * out != NULL: read back [cycle & 7][block][start, end] (nanoseconds).  Returns the number of blocks per cycle. ---- */
int osc_debug_block_times(osc_handle* h, int enabled, unsigned long long* out, int64_t out_capacity);

/* ---- measurement aid (no reference counterpart): how the last cycle that took the split blending path (many robots inside the
 * reference's singularity band, SingularityHandler.cpp:75-368) distributed them: out4 = robots with 0, 1 and 2 singular
 * directions handled by the blending kernels, and robots sent on to the rolled general path.  -1 four times when the handle
 * has not used that path. ---- */
int osc_debug_general_path_counts(osc_handle* h, int32_t* out4);

/* ---- measurement aid (no reference counterpart): sustained FP64 FMA rate of the device in TFLOP/s, from a DFMA-only
 * kernel run for about `seconds` (bench.py reports the roofline against it next to the datasheet figure) ---- */
int osc_measure_fp64_peak(osc_handle* h, double seconds, double* tflops_out);

/* ---- simulation side of the loop (SURVEY.md row f-1).  Replaces what the reference examples obtain from
 * sai-simulation: sim->setJointTorques(name, tau); sim->integrate()
 * (examples/05-using_robot_controller/05-using_robot_controller.cpp:223-231).  Forward dynamics
 * ddq = M^-1 (tau - b(q, dq) - g(q)) of the handle's model for every robot, `substeps` semi-implicit Euler steps of
 * `dt` with the torque held; q and dq (n x N, SoA) are updated in place, host or device memory. ---- */
int osc_sim_integrate(osc_handle* h, double* q, double* dq, const double* tau, double dt, int substeps, int mem_kind);

int osc_eval_model(osc_handle* h, int task_id, const osc_link_frame* frame, const double point[3], double* M,
				   double* J, double* x, double* R, double* g, int mem_kind);

#ifdef __cplusplus
}
#endif
#endif /* SAI_B200_OSC_H_ */
