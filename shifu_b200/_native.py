"""ctypes binding of ``libshifu_b200.so`` — the only way the host layer reaches the kernels.

There is deliberately no fallback: if the library is missing or a call fails, a
:class:`ShifuNativeError` is raised (the product path must fail loudly, never route through torch
or the oracle).  Structures mirror ``include/shifu_b200.h`` field for field
(``tests/test_abi.py`` checks sizes/offsets against the header with the C compiler).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

MAX_DOF, MAX_LEG, MAX_PX, MAX_PY, MAX_TERMS, NUM_STATS = 12, 8, 17, 11, 8, 16
ABI_VERSION = 5
OBS_HEAD = 72
OBS_HEAD_ACT = 48          # the action head (num_obs = 235 or 48): SHIFU_OBS_HEAD_ACT

# enum ShifuRewardTerm
REW_TRACKING_LIN_VEL, REW_TRACKING_ANG_VEL, REW_STABILIZING_BASE, REW_SMOOTHING_ACTION = 0, 1, 2, 3
REW_LEG_COLLISION, REW_TORQUES, REW_ABB_REACHING, REW_ABB_SUCCESS = 4, 5, 6, 7
REW_LIN_VEL_Z, REW_ANG_VEL_XY, REW_ORIENTATION, REW_DOF_VEL, REW_ACTION_RATE, REW_BASE_HEIGHT = 8, 9, 10, 11, 12, 13
REW_DOF_POS_LIMITS, REW_FEET_AIR_TIME = 14, 15
# enum ShifuObsVec
OBS_COMMAND, OBS_BASE_LIN_VEL, OBS_BASE_ANG_VEL, OBS_GRAVITY_VEC, OBS_PROJECTED_GRAVITY, OBS_VEC_COUNT = range(6)
STAT_TERM0, STAT_NRESET, STAT_LEVEL_SUM, STAT_SUCCESS, STAT_NENVS = 0, 8, 9, 10, 11

E_NULL, E_RANGE, E_STATE, E_NODEVICE, E_ALIGN = -1, -2, -3, -4, -5


class ShifuNativeError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libshifu_b200 error {code}: {msg}")
        self.code = code


class A1Desc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("num_envs", C.c_int32), ("env_offset", C.c_int64),
        ("rng_seed", C.c_uint64),
        ("num_dof", C.c_int32), ("num_bodies", C.c_int32), ("num_hist", C.c_int32), ("num_obs", C.c_int32),
        ("base_body", C.c_int32), ("num_leg_bodies", C.c_int32), ("leg_bodies", C.c_int32 * MAX_LEG),
        ("force_body", C.c_int32), ("root_stride", C.c_int32), ("root_offset", C.c_int32),
        ("q0", C.c_float * MAX_DOF), ("kp", C.c_float * MAX_DOF), ("kd", C.c_float * MAX_DOF),
        ("torque_limit", C.c_float * MAX_DOF),
        ("action_scale", C.c_float), ("clip_actions", C.c_float), ("clip_obs", C.c_float),
        ("num_points_x", C.c_int32), ("num_points_y", C.c_int32),
        ("points_x", C.c_float * MAX_PX), ("points_y", C.c_float * MAX_PY),
        ("border_size", C.c_float), ("horizontal_scale", C.c_float), ("vertical_scale", C.c_float),
        ("height_offset", C.c_float), ("height_clip", C.c_float),
        ("max_episode_length", C.c_int64), ("max_episode_length_s", C.c_float),
        ("contact_term_force", C.c_float), ("default_root", C.c_float * 7),
        ("reset_xy_range", C.c_float), ("push_force_max", C.c_float),
        ("cmd_low", C.c_float * 3), ("cmd_high", C.c_float * 3),
        ("curriculum", C.c_int32), ("max_terrain_level", C.c_int32), ("num_terrain_types", C.c_int32),
        ("level_up_distance", C.c_float), ("level_down_factor", C.c_float),
        ("num_reward_terms", C.c_int32), ("reward_terms", C.c_int32 * MAX_TERMS),
        ("reward_params", (C.c_float * 2) * MAX_TERMS),
        ("dof_pos_limit_low", C.c_float * MAX_DOF), ("dof_pos_limit_high", C.c_float * MAX_DOF),
        ("num_feet", C.c_int32), ("feet_bodies", C.c_int32 * 4), ("feet_contact_force", C.c_float),
        ("air_time_cmd_min", C.c_float), ("air_time_dt", C.c_float), ("air_time_reset", C.c_int32),
        ("obs_layout", C.c_int32), ("obs_vec_src", C.c_int32 * 4), ("obs_scale", C.c_float * OBS_HEAD),
        ("obs_height_scale", C.c_float), ("obs_noise", C.c_float * OBS_HEAD), ("obs_height_noise", C.c_float),
    ]


class A1StepIO(C.Structure):
    _fields_ = [
        ("root_state", C.c_void_p), ("dof_state", C.c_void_p), ("contact_state", C.c_void_p),
        ("actions", C.c_void_p), ("torques", C.c_void_p), ("history", C.c_void_p), ("command", C.c_void_p),
        ("ep_len", C.c_void_p), ("ep_sums", C.c_void_p * MAX_TERMS),
        ("base_lin_vel", C.c_void_p), ("base_ang_vel", C.c_void_p), ("projected_gravity", C.c_void_p),
        ("env_origins", C.c_void_p), ("terrain_levels", C.c_void_p), ("terrain_types", C.c_void_p),
        ("terrain_origins", C.c_void_p), ("dof_targets", C.c_void_p), ("rand_force", C.c_void_p),
        ("obs_buf", C.c_void_p), ("rew_buf", C.c_void_p), ("reset_buf", C.c_void_p),
        ("time_out_buf", C.c_void_p), ("contact_term_buf", C.c_void_p), ("measured_heights", C.c_void_p),
        ("step", C.c_int64), ("step_dev", C.c_void_p), ("swing_time", C.c_void_p), ("last_contacts", C.c_void_p),
        ("carry_body_frame", C.c_int32),
    ]


class AbbDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("num_envs", C.c_int32), ("env_offset", C.c_int64),
        ("rng_seed", C.c_uint64),
        ("num_actors", C.c_int32), ("num_bodies", C.c_int32), ("num_dof", C.c_int32), ("ee_body", C.c_int32),
        ("robot_actor", C.c_int32), ("table_actor", C.c_int32), ("cube_actor", C.c_int32),
        ("goal_actor", C.c_int32),
        ("min_ee_pos", C.c_float * 3), ("max_ee_pos", C.c_float * 3), ("q0", C.c_float * MAX_DOF),
        ("robot_root", C.c_float * 7), ("table_root", C.c_float * 7),
        ("box_pos_low", C.c_double * 3), ("box_pos_high", C.c_double * 3), ("goal_z", C.c_double),
        ("success_distance", C.c_float),
        ("max_episode_length", C.c_int64), ("max_episode_length_s", C.c_float), ("clip_obs", C.c_float),
        ("num_reward_terms", C.c_int32), ("reward_terms", C.c_int32 * MAX_TERMS),
        ("reward_params", (C.c_float * 2) * MAX_TERMS),
    ]


class AbbStepIO(C.Structure):
    _fields_ = [
        ("root_state", C.c_void_p), ("body_state", C.c_void_p), ("dof_state", C.c_void_p),
        ("dof_targets", C.c_void_p), ("ep_len", C.c_void_p), ("ep_sums", C.c_void_p * MAX_TERMS),
        ("obs_buf", C.c_void_p), ("rew_buf", C.c_void_p), ("reset_buf", C.c_void_p),
        ("time_out_buf", C.c_void_p), ("success_buf", C.c_void_p), ("step", C.c_int64),
        ("step_dev", C.c_void_p),
    ]


class ArmIkIO(C.Structure):
    _fields_ = [
        ("body_state", C.c_void_p), ("jacobian", C.c_void_p), ("dof_state", C.c_void_p),
        ("goal_pose", C.c_void_p), ("actions", C.c_void_p), ("dof_targets", C.c_void_p),
        ("num_bodies", C.c_int32), ("ee_body", C.c_int32), ("num_links", C.c_int32), ("ee_link", C.c_int32),
        ("num_dof", C.c_int32), ("ee_velocity", C.c_float), ("dt", C.c_float),
        ("min_ee_pos", C.c_float * 3), ("max_ee_pos", C.c_float * 3), ("tar_quat", C.c_float * 4),
        ("damping", C.c_float),
    ]


class CameraGatherIO(C.Structure):
    _fields_ = [
        ("color_src", C.c_void_p), ("depth_src", C.c_void_p), ("seg_src", C.c_void_p), ("flow_src", C.c_void_p),
        ("color_out", C.c_void_p), ("depth_out", C.c_void_p), ("seg_out", C.c_void_p), ("flow_out", C.c_void_p),
        ("height", C.c_int32), ("width", C.c_int32), ("normalize_color", C.c_int32),
    ]


class TerrainTile(C.Structure):
    _fields_ = [("kind", C.c_int32), ("i", C.c_int32), ("j", C.c_int32), ("p", C.c_int32 * 4), ("table_off", C.c_int32)]


class TerrainDesc(C.Structure):
    _fields_ = [("num_rows", C.c_int32), ("num_cols", C.c_int32), ("width_px", C.c_int32), ("length_px", C.c_int32),
                ("border_px", C.c_int32), ("env_length", C.c_double), ("env_width", C.c_double),
                ("horizontal_scale", C.c_double), ("vertical_scale", C.c_double)]


TERRAIN_PYRAMID, TERRAIN_PYRAMID_NOISE, TERRAIN_STAIRS, TERRAIN_OBSTACLES, TERRAIN_STONES, TERRAIN_GAP, TERRAIN_PIT = range(7)

_VP, _I32, _I64, _F = C.c_void_p, C.c_int32, C.c_int64, C.c_float

# name -> argtypes (restype is int unless listed in _RESTYPES)
SIGNATURES = {
    "shifu_ctx_create": [C.c_int, C.POINTER(A1Desc), C.POINTER(AbbDesc), C.POINTER(_VP)],
    "shifu_ctx_create_util": [C.c_int, _I32, C.POINTER(_VP)],
    "shifu_ctx_destroy": [_VP],
    "shifu_last_error": [],
    "shifu_abi_version": [],
    "shifu_set_height_map": [_VP, _VP, _I32, _I32, _VP],
    "shifu_set_level_sum": [_VP, _VP, _VP],
    "shifu_pd_torque": [_VP, _VP, _VP, _VP, _VP, _I32, _VP],
    "shifu_body_frame": [_VP, _VP, _I32, _I32, _I32, _VP, _VP, _VP, _VP, _VP],
    "shifu_get_heights": [_VP, _VP, _VP, _VP, _VP],
    "shifu_a1_post_physics": [_VP, C.POINTER(A1StepIO), _VP],
    "shifu_a1_eval_terms": [_VP, C.POINTER(A1StepIO), _VP, _VP],
    "shifu_abb_post_physics": [_VP, C.POINTER(AbbStepIO), _VP],
    "shifu_compact_reset_ids": [_VP, _VP, _I32, _VP, _VP, _VP],
    "shifu_history_add": [_VP, _VP, _VP, _I32, _I32, _I32, _VP],
    "shifu_clip": [_VP, _VP, _VP, _I64, _F, _VP],
    "shifu_arm_ik": [_VP, C.POINTER(ArmIkIO), _I32, _VP],
    "shifu_camera_gather": [_VP, C.POINTER(CameraGatherIO), _I32, _VP],
    "shifu_a1_reset_idx": [_VP, C.POINTER(A1StepIO), _VP, _I32, _VP],
    "shifu_abb_reset_idx": [_VP, C.POINTER(AbbStepIO), _VP, _I32, _VP],
    "shifu_collect_stats": [_VP, _VP, _VP, _VP],
    "shifu_collect_stats_ring": [_VP, _VP, _I32, _I32, _VP, _VP],
    "shifu_publish_extras": [_VP, _VP, _VP, _VP],
    "shifu_publish_extras_ring": [_VP, _VP, _VP, _I32, _I32, _VP, _VP],
    "shifu_read_stats_host": [_VP, _VP, _VP],
    "shifu_terrain_generate": [_VP, C.POINTER(TerrainDesc), C.POINTER(TerrainTile), _I32, C.POINTER(C.c_double), _I32,
                               _VP, _VP, _VP],
}
_RESTYPES = {"shifu_last_error": C.c_char_p}

_LIB: Optional[C.CDLL] = None


def lib_path() -> str:
    return os.environ.get("SHIFU_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)),
                                                            "libshifu_b200.so")


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (building first when the sources are newer) and type the library."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if build_if_missing and "SHIFU_B200_LIB" not in os.environ:
        from . import build as _build
        try:
            _build.build()
        except Exception as exc:      # pragma: no cover - surfaced with context
            # never run stale kernels against new headers / bindings: a failed rebuild is fatal unless
            # the existing library was built from exactly these sources
            if not os.path.exists(path) or _build.needs_build():
                raise ShifuNativeError(E_STATE, f"cannot build {path}: {exc}") from exc
    if not os.path.exists(path):
        raise ShifuNativeError(E_STATE, f"{path} not found; run `python -m shifu_b200.build` "
                                        "(there is no CPU / torch fallback)")
    lib = C.CDLL(path)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, C.c_int)
    if lib.shifu_abi_version() != ABI_VERSION:
        raise ShifuNativeError(E_STATE, f"ABI version mismatch: library {lib.shifu_abi_version()}, "
                                        f"binding {ABI_VERSION}")
    _LIB = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load(False).shifu_last_error()
        raise ShifuNativeError(rc, msg.decode() if msg else "")


def ptr(t) -> Optional[int]:
    """data_ptr of a torch tensor (None -> NULL).  The tensor must be contiguous and on CUDA."""
    if t is None:
        return None
    if not t.is_cuda:
        raise ShifuNativeError(E_NODEVICE, "tensor is not on a CUDA device: the shifu_b200 hot path has "
                                           "no CPU fallback")
    if not t.is_contiguous():
        raise ShifuNativeError(E_ALIGN, "tensor must be contiguous")
    return t.data_ptr()


def current_stream() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream
