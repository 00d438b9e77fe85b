"""ctypes binding of the C ABI in include/sai_b200_osc.h (libsai_b200_osc.so, built in-tree).

This is the reference-side binding a maintainer would write for a Python caller; the
C++ wrappers live in include/sai_b200/.  There is no fallback: if the shared library is
missing, import fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# SAI_B200_OSC_LIB selects another build of the SAME library (kernel tuning experiments); never a fallback
LIB_PATH = os.environ.get("SAI_B200_OSC_LIB", os.path.join(_HERE, "libsai_b200_osc.so"))

OSC_MAX_DOF = 8
OSC_MAX_TASKS = 4
OSC_ABI_VERSION = 2

OSC_OK = 0
OSC_ERR_INVALID_ARGUMENT = -1
OSC_ERR_UNSUPPORTED = -2
OSC_ERR_CUDA = -3
OSC_ERR_NO_DEVICE = -4
OSC_ERR_STATE = -5

OSC_MEM_HOST = 0
OSC_MEM_DEVICE = 1
OSC_PRECISION_FP64, OSC_PRECISION_FP32 = 0, 1
OSC_RESET_REINITIALIZE, OSC_RESET_CONSTRUCT = 0, 1

FULL_DYNAMIC_DECOUPLING = 0
BOUNDED_INERTIA_ESTIMATES = 1
IMPEDANCE = 2

OSC_TASK_JOINT = 2
OSC_TASK_MOTION_FORCE = 3

STATUS_SINGULAR_PATH = 0x1
STATUS_NAN_SCRUBBED = 0x2
STATUS_ZERO_RANGE = 0x4
STATUS_POPC_OVERFLOW = 0x8
STATUS_UNHANDLED = 0x10
STATUS_TYPE1 = 0x20
STATUS_TYPE2 = 0x40

# osc_field
MFT_GOAL_POSITION = 0
MFT_GOAL_ORIENTATION = 1
MFT_GOAL_LINEAR_VELOCITY = 2
MFT_GOAL_ANGULAR_VELOCITY = 3
MFT_GOAL_LINEAR_ACCELERATION = 4
MFT_GOAL_ANGULAR_ACCELERATION = 5
MFT_GOAL_FORCE = 6
MFT_GOAL_MOMENT = 7
MFT_CURRENT_POSITION = 8
MFT_CURRENT_ORIENTATION = 9
MFT_CURRENT_LINEAR_VELOCITY = 10
MFT_CURRENT_ANGULAR_VELOCITY = 11
MFT_SENSED_FORCE_CONTROL_WORLD = 12
MFT_SENSED_MOMENT_CONTROL_WORLD = 13
MFT_UNIT_MASS_FORCE = 14
MFT_INTEGRATED_POSITION_ERROR = 15
MFT_INTEGRATED_ORIENTATION_ERROR = 16
MFT_INTEGRATED_FORCE_ERROR = 17
MFT_INTEGRATED_MOMENT_ERROR = 18
MFT_POPC_STATE = 19
MFT_TYPE1_POSTURE = 20
MFT_POSITION_ERROR = 21
MFT_ORIENTATION_ERROR = 22
MFT_SIGMA_FORCE = 23
MFT_SIGMA_POSITION = 24
MFT_SIGMA_MOMENT = 25
MFT_SIGMA_ORIENTATION = 26
JT_GOAL_POSITION = 32
JT_GOAL_VELOCITY = 33
JT_GOAL_ACCELERATION = 34
JT_INTEGRATED_POSITION_ERROR = 35
JT_DESIRED_POSITION = 36
JT_DESIRED_VELOCITY = 37
JT_DESIRED_ACCELERATION = 38
MFT_DESIRED_POSITION = 40
MFT_DESIRED_ORIENTATION = 41
MFT_DESIRED_LINEAR_VELOCITY = 42
MFT_DESIRED_ANGULAR_VELOCITY = 43
MFT_DESIRED_LINEAR_ACCELERATION = 44
MFT_DESIRED_ANGULAR_ACCELERATION = 45
OTG_GOAL_REACHED = 1
OTG_DIRTY = 2
OTG_ERROR = 4
OTG_BAD_FINISH = 8
TASK_NULLSPACE = 48
TASK_PREVIOUS_NULLSPACE = 49
TASK_AND_PREVIOUS_NULLSPACE = 50
# osc_gain_group
GAINS_JOINT = 0
GAINS_POSITION = 1
GAINS_ORIENTATION = 2
GAINS_FORCE = 3
GAINS_MOMENT = 4

D = C.c_double
I32 = C.c_int32


class ModelDesc(C.Structure):
    _fields_ = [
        ("n", I32), ("jtype", I32 * OSC_MAX_DOF),
        ("axis", (D * 3) * OSC_MAX_DOF), ("R_fix", (D * 9) * OSC_MAX_DOF), ("t_fix", (D * 3) * OSC_MAX_DOF),
        ("mass", D * OSC_MAX_DOF), ("com", (D * 3) * OSC_MAX_DOF), ("inertia", (D * 9) * OSC_MAX_DOF),
        ("q_lower", D * OSC_MAX_DOF), ("q_upper", D * OSC_MAX_DOF), ("dq_max", D * OSC_MAX_DOF), ("effort", D * OSC_MAX_DOF),
        ("R_world_base", D * 9), ("t_world_base", D * 3), ("gravity_world", D * 3),
    ]


class LinkFrame(C.Structure):
    _fields_ = [("body", I32), ("R", D * 9), ("t", D * 3)]


class MftDesc(C.Structure):
    _fields_ = [
        ("link", LinkFrame), ("compliant_R", D * 9), ("compliant_t", D * 3),
        ("partial", I32), ("n_dirs_translation", I32), ("dirs_translation", (D * 3) * 3),
        ("n_dirs_rotation", I32), ("dirs_rotation", (D * 3) * 3),
        ("force_motion_in_compliant_frame", I32), ("loop_timestep", D),
    ]


class MftParams(C.Structure):
    _fields_ = [
        ("kp_pos", D * 3), ("kv_pos", D * 3), ("ki_pos", D * 3),
        ("kp_ori", D * 3), ("kv_ori", D * 3), ("ki_ori", D * 3),
        ("kp_force", D), ("kv_force", D), ("ki_force", D),
        ("kp_moment", D), ("kv_moment", D), ("ki_moment", D),
        ("kff_force", D), ("kff_moment", D),
        ("max_force_control_feedback_output", D), ("max_moment_control_feedback_output", D),
        ("linear_saturation_velocity", D), ("angular_saturation_velocity", D),
        ("bie_threshold", D), ("s_min", D), ("s_max", D),
        ("kp_type_1", D), ("kv_type_1", D), ("kv_type_2", D),
        ("s_abs_tol", D), ("type_1_tol", D), ("type_2_torque_ratio", D), ("type_2_angle_threshold", D),
        ("perturb_step_size", D),
        ("force_or_motion_axis", D * 3), ("moment_or_rotmotion_axis", D * 3),
        ("force_space_dimension", I32), ("moment_space_dimension", I32),
        ("closed_loop_force_control", I32), ("closed_loop_moment_control", I32),
        ("passivity_enabled", I32), ("use_velocity_saturation", I32), ("dynamic_decoupling_type", I32),
        ("singularity_handling_enabled", I32), ("enforce_type_1_strategy", I32), ("buffer_size", I32),
    ]


class JointParams(C.Structure):
    _fields_ = [
        ("kp", D * OSC_MAX_DOF), ("kv", D * OSC_MAX_DOF), ("ki", D * OSC_MAX_DOF),
        ("saturation_velocity", D * OSC_MAX_DOF), ("bie_threshold", D),
        ("use_velocity_saturation", I32), ("dynamic_decoupling_type", I32),
    ]


# every symbol include/sai_b200_osc.h declares: name -> (restype, argtypes)
_H = C.c_void_p
_PD = C.c_void_p  # double* that may be a host numpy buffer or a raw device pointer
SYMBOLS = {
    "osc_abi_version": (C.c_int, []),
    "osc_last_error": (C.c_char_p, [_H]),
    "osc_builtin_model": (C.c_int, [C.c_char_p, C.POINTER(ModelDesc)]),
    "osc_builtin_link": (C.c_int, [C.c_char_p, C.c_char_p, C.POINTER(LinkFrame)]),
    "osc_create": (C.c_int, [C.POINTER(ModelDesc), C.c_int64, C.c_int, C.POINTER(_H)]),
    "osc_destroy": (C.c_int, [_H]),
    "osc_set_stream": (C.c_int, [_H, C.c_void_p]),
    "osc_sync": (C.c_int, [_H]),
    "osc_num_robots": (C.c_int64, [_H]),
    "osc_dof": (C.c_int, [_H]),
    "osc_set_state": (C.c_int, [_H, _PD, _PD, C.c_int]),
    "osc_add_joint_task": (C.c_int, [_H, _PD, C.c_int, D, C.POINTER(C.c_int)]),
    "osc_add_motion_force_task": (C.c_int, [_H, C.POINTER(MftDesc), C.POINTER(C.c_int)]),
    "osc_finalize_controller": (C.c_int, [_H, C.c_int]),
    "osc_num_tasks": (C.c_int, [_H]),
    "osc_get_task_type": (C.c_int, [_H, C.c_int]),
    "osc_get_task_dof": (C.c_int, [_H, C.c_int]),
    "osc_mft_default_params": (C.c_int, [C.POINTER(MftParams)]),
    "osc_mft_get_params": (C.c_int, [_H, C.c_int, C.POINTER(MftParams)]),
    "osc_mft_set_params": (C.c_int, [_H, C.c_int, C.POINTER(MftParams)]),
    "osc_mft_parametrize_force_motion_spaces": (C.c_int, [_H, C.c_int, C.c_int, C.POINTER(D), C.POINTER(C.c_int)]),
    "osc_mft_parametrize_moment_rotmotion_spaces": (C.c_int, [_H, C.c_int, C.c_int, C.POINTER(D), C.POINTER(C.c_int)]),
    "osc_mft_set_closed_loop_force_control": (C.c_int, [_H, C.c_int, C.c_int]),
    "osc_mft_set_closed_loop_moment_control": (C.c_int, [_H, C.c_int, C.c_int]),
    "osc_mft_enable_passivity": (C.c_int, [_H, C.c_int, C.c_int, C.c_int]),
    "osc_mft_set_force_sensor_frame": (C.c_int, [_H, C.c_int, C.POINTER(D), C.POINTER(D)]),
    "osc_mft_update_sensed_force_and_moment": (C.c_int, [_H, C.c_int, _PD, _PD, C.c_int]),
    "osc_mft_reset_integrators": (C.c_int, [_H, C.c_int, C.c_int]),
    "osc_joint_default_params": (C.c_int, [C.POINTER(JointParams)]),
    "osc_joint_get_params": (C.c_int, [_H, C.c_int, C.POINTER(JointParams)]),
    "osc_joint_set_params": (C.c_int, [_H, C.c_int, C.POINTER(JointParams)]),
    "osc_field_ncomp": (C.c_int, [_H, C.c_int, C.c_int]),
    "osc_set_field": (C.c_int, [_H, C.c_int, C.c_int, _PD, C.c_int, C.c_int]),
    "osc_get_field": (C.c_int, [_H, C.c_int, C.c_int, _PD, C.c_int]),
    "osc_reinitialize_task": (C.c_int, [_H, C.c_int]),
    "osc_reset_robots": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_int, C.c_int]),
    "osc_enable_gravity_compensation": (C.c_int, [_H, C.c_int]),
    "osc_enable_torque_saturation": (C.c_int, [_H, C.c_int]),
    "osc_enable_joint_limit_avoidance": (C.c_int, [_H, C.c_int]),
    "osc_update_task_models": (C.c_int, [_H]),
    "osc_compute_control_torques": (C.c_int, [_H, _PD, C.c_int]),
    "osc_step": (C.c_int, [_H, _PD, _PD, _PD, C.c_int]),
    "osc_step_async": (C.c_int, [_H, _PD, _PD, _PD, C.c_int]),
    "osc_get_status": (C.c_int, [_H, C.c_void_p, C.c_int]),
    "osc_launch_count": (C.c_int64, [_H]),
    "osc_enable_observers": (C.c_int, [_H, C.c_int]),
    "osc_joint_enable_internal_otg": (C.c_int, [_H, C.c_int, C.POINTER(D), C.POINTER(D)]),
    "osc_mft_enable_internal_otg": (C.c_int, [_H, C.c_int, D, D, D, D]),
    "osc_disable_internal_otg": (C.c_int, [_H, C.c_int]),
    "osc_internal_otg_enabled": (C.c_int, [_H, C.c_int]),
    "osc_get_internal_otg_flags": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_int]),
    "osc_shard_range": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "osc_urdf_register": (C.c_int, [C.c_char_p, C.c_char_p]),
    "osc_urdf_register_file": (C.c_int, [C.c_char_p, C.c_char_p]),
    "osc_urdf_last_error": (C.c_char_p, []),
    "osc_urdf_set_folder": (C.c_int, [C.c_char_p, C.c_char_p]),
    "osc_urdf_replace_path_prefix": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int]),
    "osc_world_register_robot": (C.c_int, [C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(D)]),
    "osc_debug_popc_sequence": (C.c_int, [_H, C.c_int, C.c_int, _PD, _PD, _PD, _PD, C.c_double, C.c_double, _PD]),
    "osc_measure_fp64_peak": (C.c_int, [_H, C.c_double, _PD]),
    "osc_debug_block_times": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_int64]),
    "osc_debug_general_path_counts": (C.c_int, [_H, C.POINTER(C.c_int32)]),
    "osc_set_precision": (C.c_int, [_H, C.c_int]),
    "osc_get_precision": (C.c_int, [_H]),
    "osc_sim_integrate": (C.c_int, [_H, _PD, _PD, _PD, C.c_double, C.c_int, C.c_int]),
    "osc_set_gains": (C.c_int, [_H, C.c_int, C.c_int, _PD, _PD, _PD, C.c_int, C.c_int]),
    "osc_get_gains": (C.c_int, [_H, C.c_int, C.c_int, _PD, _PD, _PD, C.c_int]),
    "osc_mft_parametrize_spaces_batched": (C.c_int, [_H, C.c_int, C.c_int, _PD, _PD, _PD, C.c_int]),
    "osc_mft_set_closed_loop_batched": (C.c_int, [_H, C.c_int, C.c_int, _PD, C.c_int]),
    "osc_mft_get_spaces": (C.c_int, [_H, C.c_int, C.c_int, _PD, _PD, _PD, C.c_int]),
    "osc_eval_model": (C.c_int, [_H, C.c_int, C.POINTER(LinkFrame), C.POINTER(D), _PD, _PD, _PD, _PD, _PD, C.c_int]),
}

_lib = None


def load_library():
    """Load libsai_b200_osc.so and bind every declared symbol.  Raises if the library or a
    symbol is missing -- the product has no other execution path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or make -C sai_primitives_b200/csrc).  There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the export is missing
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.osc_abi_version() != OSC_ABI_VERSION:
        raise ImportError("ABI version mismatch between capi.py and libsai_b200_osc.so")
    _lib = lib
    return lib


class OscError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("osc error %d: %s" % (code, message))
        self.code = code
        self.message = message


def host_ptr(a: np.ndarray):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)
