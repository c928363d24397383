"""ctypes mirror of ``include/r2ik.h`` (structs, constants) and the builders that turn the
reference's constructor / call arguments into them.  No computation happens here."""
from __future__ import annotations

import ctypes as C

import numpy as np

ABI_VERSION = 5

POSE_EULER6 = 0
POSE_MAT4 = 1
POSE_MAT34 = 2

EMG_SHOULDER_PITCH = 1
EMG_ELBOW_YAW = 2
EMG_WRIST_YAW = 4
EMG_DISCONTINUITY = 8


class ArmConfig(C.Structure):
    """R2ikArmConfig: raw SymbolicIK constructor arguments for one arm (symbolic_ik.py:26-63)."""

    _fields_ = [
        ("shoulder_position", C.c_double * 3),
        ("shoulder_orientation_deg", C.c_double * 3),
        ("upper_arm_size", C.c_double),
        ("forearm_size", C.c_double),
        ("tip_position", C.c_double * 3),
        ("elbow_limit_deg", C.c_double),
        ("wrist_limit_deg", C.c_double),
        ("projection_margin", C.c_double),
        ("backward_limit", C.c_double),
        ("normal_vector_margin", C.c_double),
        ("singularity_offset", C.c_double),
        ("singularity_limit_coeff", C.c_double),
        ("side", C.c_int32),
        ("reserved", C.c_int32),
    ]


class ArmConstants(C.Structure):
    _fields_ = [
        ("gripper_size", C.c_double),
        ("max_arm_length", C.c_double),
        ("shoulder_wrist_min_distance", C.c_double),
        ("elbow_singularity_position", C.c_double * 3),
        ("wrist_singularity_position", C.c_double * 3),
    ]


class CtlParams(C.Structure):
    _fields_ = [
        ("preferred_theta", C.c_double),
        ("preferred_theta_ctor", C.c_double),
        ("interval_limit", C.c_double * 2),
        ("d_theta_max", C.c_double),
        ("orbita3d_max_angle", C.c_double),
        ("nb_search_points", C.c_int32),
        ("nb_search_points_continuous", C.c_int32),
    ]


class TrajState(C.Structure):
    _fields_ = [
        ("previous_theta", C.c_double),
        ("previous_sol", C.c_double * 7),
        ("has_previous_sol", C.c_int32),
        ("init", C.c_int32),
        ("emergency_stop", C.c_int32),
        ("emergency_bits", C.c_int32),
    ]


class ScalarQuery(C.Structure):
    """R2ikScalarQuery: one scalar call sequence of SymbolicIK."""

    _fields_ = [("goal_pose", C.c_double * 6), ("theta", C.c_double), ("previous_joints", C.c_double * 7),
                ("no_limits", C.c_int32), ("has_theta", C.c_int32)]


class ScalarResult(C.Structure):
    """R2ikScalarResult."""

    _fields_ = [("interval", C.c_double * 2), ("joints", C.c_double * 7), ("elbow", C.c_double * 3),
                ("elbow_on_circle", C.c_double * 3), ("goal_position_solved", C.c_double * 3),
                ("wrist_position_solved", C.c_double * 3), ("goal_position", C.c_double * 3),
                ("wrist_position", C.c_double * 3), ("reachable", C.c_int32), ("state", C.c_int32),
                ("projected", C.c_int32), ("reserved", C.c_int32)]


SCALAR_RESULT_DTYPE = np.dtype([
    ("interval", "f8", (2,)), ("joints", "f8", (7,)), ("elbow", "f8", (3,)), ("elbow_on_circle", "f8", (3,)),
    ("goal_position_solved", "f8", (3,)), ("wrist_position_solved", "f8", (3,)), ("goal_position", "f8", (3,)),
    ("wrist_position", "f8", (3,)), ("reachable", "i4"), ("state", "i4"), ("projected", "i4"), ("reserved", "i4")])
assert SCALAR_RESULT_DTYPE.itemsize == C.sizeof(ScalarResult) == 232


class FkChain(C.Structure):
    """R2ikFkChain: fixed 3x4 transforms between the 7 revolute joints (+ tip) and the joint axes."""

    _fields_ = [("fixed", (C.c_double * 12) * 8), ("axis", (C.c_double * 3) * 7)]


TRAJ_STATE_DTYPE = np.dtype(
    [
        ("previous_theta", "f8"),
        ("previous_sol", "f8", (7,)),
        ("has_previous_sol", "i4"),
        ("init", "i4"),
        ("emergency_stop", "i4"),
        ("emergency_bits", "i4"),
    ]
)
assert TRAJ_STATE_DTYPE.itemsize == C.sizeof(TrajState) == 80

# SymbolicIK default parameters (symbolic_ik.py:38-51)
DEFAULT_IK_PARAMETERS = {
    "r_shoulder_position": np.array([0.0, -0.2, 0.0]),
    "r_shoulder_orientation": [-15, 0, 10],
    "r_upper_arm_size": np.float64(0.28),
    "r_forearm_size": np.float64(0.28),
    "r_tip_position": np.array([-0.0, 0.0, 0.10]),
    "l_shoulder_position": np.array([0.0, 0.2, 0.0]),
    "l_shoulder_orientation": [15, 0, -10],
    "l_upper_arm_size": np.float64(0.28),
    "l_forearm_size": np.float64(0.28),
    "l_tip_position": np.array([-0.0, 0.0, 0.10]),
}


def make_arm_config(arm, ik_parameters, elbow_limit, wrist_limit, projection_margin, backward_limit,
                    normal_vector_margin, singularity_offset, singularity_limit_coeff) -> ArmConfig:
    n = arm[0]
    c = ArmConfig()
    c.shoulder_position[:] = [float(x) for x in ik_parameters[f"{n}_shoulder_position"]]
    c.shoulder_orientation_deg[:] = [float(x) for x in ik_parameters[f"{n}_shoulder_orientation"]]
    c.upper_arm_size = float(ik_parameters[f"{n}_upper_arm_size"])
    c.forearm_size = float(ik_parameters[f"{n}_forearm_size"])
    c.tip_position[:] = [float(x) for x in ik_parameters[f"{n}_tip_position"]]
    c.elbow_limit_deg = float(elbow_limit)
    c.wrist_limit_deg = float(wrist_limit)
    c.projection_margin = float(projection_margin)
    c.backward_limit = float(backward_limit)
    c.normal_vector_margin = float(normal_vector_margin)
    c.singularity_offset = float(singularity_offset)
    c.singularity_limit_coeff = float(singularity_limit_coeff)
    c.side = 1 if arm == "r_arm" else -1
    return c
