"""Host-side drivers of the fused CUDA hot path (thin; all arithmetic lives in ``csrc/``).

``A1HotPath`` / ``AbbHotPath`` own a native context, hold the env-side tensors the reference
keeps on ``ShifuVecEnv`` / ``Robot`` objects (``shifu/gym/env.py:44-63``,
``examples/a1_conditional/a1_conditional.py:52-62,100-114``) and enqueue the C-ABI calls in the
reference's order (SURVEY.md §3.2).  The flat simulator tensors (root / dof / contact / body
state) are *borrowed* from the gym, exactly like the reference borrows them from PhysX.

The ``shifu_b200.gym`` / ``shifu_b200.tasks`` classes wrap these objects behind the reference's
class API; tests and ``bench.py`` may also drive them directly.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as nv

A1_TERM_CODES = {
    "tracking_lin_vel": nv.REW_TRACKING_LIN_VEL, "tracking_ang_vel": nv.REW_TRACKING_ANG_VEL,
    "stabilizing_base": nv.REW_STABILIZING_BASE, "smoothing_action": nv.REW_SMOOTHING_ACTION,
    "leg_collision": nv.REW_LEG_COLLISION, "torques_penalize": nv.REW_TORQUES,
    # legged_gym-style additions (SURVEY.md 8f row N1); constants come from shifu_b200.terms (fitted from the hook)
    "lin_vel_z": nv.REW_LIN_VEL_Z, "ang_vel_xy": nv.REW_ANG_VEL_XY, "orientation": nv.REW_ORIENTATION,
    "dof_vel": nv.REW_DOF_VEL, "action_rate": nv.REW_ACTION_RATE, "base_height": nv.REW_BASE_HEIGHT,
    "dof_pos_limits": nv.REW_DOF_POS_LIMITS, "feet_air_time": nv.REW_FEET_AIR_TIME,
}
A1_DEFAULT_TERMS = ("tracking_lin_vel", "tracking_ang_vel", "stabilizing_base", "smoothing_action", "leg_collision",
                    "torques_penalize")              # build_reward_functions() of a1_conditional.py:152-160
# literal constants of the reward methods, examples/a1_conditional/a1_conditional.py:162-192
A1_TERM_PARAMS = {
    "tracking_lin_vel": (1.0, 0.25), "tracking_ang_vel": (0.5, 0.25), "stabilizing_base": (-2.0, -0.005),
    "smoothing_action": (-0.005, 0.0), "leg_collision": (-1.0, 0.1), "torques_penalize": (-2e-5, 0.0),
}
ABB_TERM_CODES = {"reward_reaching": nv.REW_ABB_REACHING, "reward_success": nv.REW_ABB_SUCCESS}
# examples/abb_pushbox_vision/a_prior_stage.py:118-131
ABB_TERM_PARAMS = {"reward_reaching": (0.1, 0.05), "reward_success": (200.0, 0.02)}


# enum ShifuObsVec: the sources a 3-column vector slot of the observation head can take
OBS_SOURCES = {"COMMAND": nv.OBS_COMMAND, "BASE_LIN_VEL": nv.OBS_BASE_LIN_VEL, "BASE_ANG_VEL": nv.OBS_BASE_ANG_VEL,
               "GRAVITY_VEC": nv.OBS_GRAVITY_VEC, "PROJECTED_GRAVITY": nv.OBS_PROJECTED_GRAVITY}
A1_OBS_SLOTS = ("COMMAND", "BASE_LIN_VEL", "BASE_ANG_VEL", "GRAVITY_VEC")      # a1_conditional.py:137-140


@dataclass(frozen=True)
class ObsLayout:
    """Layout of the 259-column A1 observation the fused kernel builds, or of the 235-column action head.

    Columns 0-11 are four 3-column slots, ``slots[i]`` naming the source of columns 3i..3i+2 (a key of
    ``OBS_SOURCES``); every head column j < 72 is ``clip(x_j * scales[j], +-clip_obs)`` (the dof-position
    columns' x_j is ``dof_pos - default_dof_pos``); the 187 heights are
    ``clip(clip(z - 0.5 - h, +-1) * height_scale, +-clip_obs)``, legged_gym's clip-then-scale order.
    PROJECTED_GRAVITY is the value the tensor holds when the step starts (``LeggedRobot.post_step`` on
    the previous state, like the body-frame velocities).  Scales are kept as fp32 values.

    ``noise`` / ``height_noise``: legged_gym's uniform observation noise (``noise_scale_vec``), one scale per
    head column and one for all 187 heights.  Column j gets ``+ (2u - 1) * noise[j]`` before the clip to
    +-clip_obs, u drawn per env, step and column from the kernels' Philox stream
    (``shifu_b200.utils.philox.obs_noise_u01``).  All zero: no noise.

    The head width is ``len(scales)``: 72, or 48 for the action head (legged_gym's own observation), whose
    columns 0-35 are the 72-column head's and whose column 36 + d is the step's ``actions[:, d]`` times
    ``scales[36 + d]``; its heights follow at column 48.  ``noise`` has one scale per head column (default:
    zeros of the head width)."""
    slots: Tuple[str, str, str, str] = A1_OBS_SLOTS
    scales: Tuple[float, ...] = (1.0,) * nv.OBS_HEAD
    height_scale: float = 1.0
    noise: Optional[Tuple[float, ...]] = None
    height_noise: float = 0.0

    def __post_init__(self):
        slots = tuple(self.slots)
        if len(slots) != 4 or any(s not in OBS_SOURCES for s in slots):
            raise ValueError(f"slots must be 4 names out of {sorted(OBS_SOURCES)}, got {slots}")
        scales = tuple(float(np.float32(v)) for v in self.scales)
        if len(scales) not in (nv.OBS_HEAD, nv.OBS_HEAD_ACT):
            raise ValueError(f"{len(scales)} column scales: the observation head has {nv.OBS_HEAD} columns, or "
                             f"{nv.OBS_HEAD_ACT} with the step's actions")
        hs = float(np.float32(self.height_scale))
        if not all(math.isfinite(v) for v in (*scales, hs)):
            raise ValueError("observation scales must be finite")
        noise = tuple(float(np.float32(v)) for v in (self.noise if self.noise is not None else (0.0,) * len(scales)))
        if len(noise) != len(scales):
            raise ValueError(f"{len(noise)} column noise scales: the observation head has {len(scales)} columns")
        hn = float(np.float32(self.height_noise))
        if not all(math.isfinite(v) for v in (*noise, hn)):
            raise ValueError("observation noise scales must be finite")
        object.__setattr__(self, "slots", slots)
        object.__setattr__(self, "scales", scales)
        object.__setattr__(self, "height_scale", hs)
        object.__setattr__(self, "noise", noise)
        object.__setattr__(self, "height_noise", hn)

    @property
    def head(self) -> int:
        """The head width: 72, or 48 for the action head."""
        return len(self.scales)

    def has_noise(self) -> bool:
        return any(v != 0.0 for v in self.noise) or self.height_noise != 0.0

    def is_reference(self) -> bool:
        """The reference observation (a1_conditional.py:131-144): identity scales, reference slots, no noise.
        The action head never is."""
        return (self.head == nv.OBS_HEAD and self.slots == A1_OBS_SLOTS and all(v == 1.0 for v in self.scales)
                and self.height_scale == 1.0 and not self.has_noise())


def compile_reward_terms(names: Sequence[str], codes: Dict[str, int], params: Dict[str, tuple]):
    """The reward-term registry: ``build_reward_functions()`` names -> (enum, p0, p1) in list order
    (``shifu/gym/env.py:160-166`` keys ``episode_rewards`` by ``fn.__name__``)."""
    if len(names) == 0:
        raise ValueError("at least one reward term is required (env.py:161)")
    if len(names) > nv.MAX_TERMS:
        raise ValueError(f"at most {nv.MAX_TERMS} fused reward terms are supported")
    out = []
    for n in names:
        if isinstance(n, (tuple, list)):          # already compiled: (name, code, p0, p1) from shifu_b200.terms
            out.append((int(n[1]), float(n[2]), float(n[3])))
            continue
        if n not in codes:
            raise KeyError(f"reward term {n!r} has no fused implementation; known: {sorted(codes)}")
        if n not in params:
            raise KeyError(f"reward term {n!r} needs its constants: pass term_params or compile the list with "
                           "shifu_b200.terms.compile_a1_terms")
        out.append((codes[n], float(params[n][0]), float(params[n][1])))
    return out


def a1_desc(num_envs: int, *, env_offset: int = 0, rng_seed: int = 0x5EED,
            terms: Sequence[str] = A1_DEFAULT_TERMS, term_params: Optional[Dict[str, tuple]] = None,
            q0=(0.1, 0.8, -1.5, 0.1, 0.8, -1.5, -0.1, 0.8, -1.5, -0.1, 0.8, -1.5),
            kp=(20.,) * 12, kd=(.5,) * 12, torque_limit=(20., 55., 55.) * 4,
            points_x=(-0.8, -0.7, -0.6, -0.5, -0.4, -0.3, -0.2, -0.1, 0., 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8),
            points_y=(-0.5, -0.4, -0.3, -0.2, -0.1, 0., 0.1, 0.2, 0.3, 0.4, 0.5),
            border_size=25., horizontal_scale=0.1, vertical_scale=0.005, max_episode_length=500,
            max_episode_length_s=10., default_root=(0, 0, 0.42, 0, 0, 0, 1.), curriculum=True,
            max_terrain_level=10, num_terrain_types=20, env_length=8., base_body=0,
            leg_bodies=(2, 3, 6, 7, 10, 11, 14, 15), force_body=0, root_stride=1, root_offset=0,
            action_scale=0.5, clip_actions=1., clip_obs=100.,
            dof_pos_limits=None, feet_bodies=(4, 8, 12, 16), feet_contact_force=1.0, air_time_cmd_min=0.1,
            air_time_dt=0.02, air_time_reset=True, obs: Optional[ObsLayout] = None,
            num_obs: int = nv.OBS_HEAD + 187) -> nv.A1Desc:
    """Defaults = the constants of ``examples/a1_conditional`` (SURVEY.md Appendix A).  ``obs``: the
    observation layout; ``None`` or the reference layout writes ``obs_layout = 0``.  ``num_obs``: 259, or
    72 for a blind task (the observation without its 187 height columns; ``obs.height_noise`` must be 0);
    235 or 48 (blind) for the action head, which needs an ``obs`` of head width 48 and always writes
    ``obs_layout = 1``."""
    head = nv.OBS_HEAD_ACT if num_obs in (nv.OBS_HEAD_ACT, nv.OBS_HEAD_ACT + 187) else nv.OBS_HEAD
    if num_obs not in (head, head + 187):
        raise ValueError(f"num_obs={num_obs}: the fused A1 observation has {nv.OBS_HEAD + 187} columns, or "
                         f"{nv.OBS_HEAD} without the height scan ({nv.OBS_HEAD_ACT + 187} or {nv.OBS_HEAD_ACT} "
                         "with the step's actions in place of the action history)")
    if head == nv.OBS_HEAD_ACT and obs is None:
        raise ValueError(f"num_obs={num_obs} (the action head) needs an ObsLayout: it is never the reference "
                         "observation")
    if obs is not None and obs.head != head:
        raise ValueError(f"num_obs={num_obs} has a {head}-column head; the layout has {obs.head} columns")
    if num_obs == head and obs is not None and obs.height_noise != 0.0:
        raise ValueError(f"a blind observation (num_obs = {num_obs}) has no height columns to add height noise to")
    d = nv.A1Desc()
    d.abi_version = nv.ABI_VERSION
    d.num_envs, d.env_offset, d.rng_seed = num_envs, env_offset, rng_seed
    d.num_dof, d.num_bodies, d.num_hist, d.num_obs = 12, 17, 3, num_obs
    d.base_body, d.force_body = base_body, force_body
    d.num_leg_bodies = len(leg_bodies)
    for i, b in enumerate(leg_bodies):
        d.leg_bodies[i] = b
    d.root_stride, d.root_offset = root_stride, root_offset
    for i in range(12):
        d.q0[i], d.kp[i], d.kd[i], d.torque_limit[i] = q0[i], kp[i], kd[i], torque_limit[i]
    d.action_scale, d.clip_actions, d.clip_obs = action_scale, clip_actions, clip_obs
    d.num_points_x, d.num_points_y = len(points_x), len(points_y)
    if len(points_x) > nv.MAX_PX or len(points_y) > nv.MAX_PY:
        raise ValueError("measured-point grid larger than the compiled 17x11")
    for i, v in enumerate(points_x):
        d.points_x[i] = v
    for i, v in enumerate(points_y):
        d.points_y[i] = v
    d.border_size, d.horizontal_scale, d.vertical_scale = border_size, horizontal_scale, vertical_scale
    d.height_offset, d.height_clip = 0.5, 1.0
    d.max_episode_length, d.max_episode_length_s = int(max_episode_length), max_episode_length_s
    d.contact_term_force = 1.0
    for i in range(7):
        d.default_root[i] = default_root[i]
    d.reset_xy_range, d.push_force_max = 1.0, 5.0
    for i in range(3):
        d.cmd_low[i], d.cmd_high[i] = -1.0, 1.0
    d.curriculum = int(bool(curriculum))
    d.max_terrain_level, d.num_terrain_types = max_terrain_level, num_terrain_types
    d.level_up_distance, d.level_down_factor = env_length / 2, 0.5
    # constants of the row-N1 terms: dof_pos_limits (per-dof soft limits) and feet_air_time
    for i in range(12):
        lo, hi = dof_pos_limits[i] if dof_pos_limits is not None else (-3.0e38, 3.0e38)
        d.dof_pos_limit_low[i], d.dof_pos_limit_high[i] = lo, hi
    if len(feet_bodies) > 4:
        raise ValueError("at most 4 feet")
    d.num_feet = len(feet_bodies)
    for i, b in enumerate(feet_bodies):
        d.feet_bodies[i] = int(b)
    d.feet_contact_force, d.air_time_cmd_min, d.air_time_dt = feet_contact_force, air_time_cmd_min, air_time_dt
    d.air_time_reset = int(bool(air_time_reset))
    comp = compile_reward_terms(list(terms), A1_TERM_CODES, {**A1_TERM_PARAMS, **(term_params or {})})
    d.num_reward_terms = len(comp)
    for i, (code, p0, p1) in enumerate(comp):
        d.reward_terms[i] = code
        d.reward_params[i][0], d.reward_params[i][1] = p0, p1
    if obs is not None and not obs.is_reference():           # (the action head never collapses to layout 0)
        d.obs_layout = 1
        for i, name in enumerate(obs.slots):
            d.obs_vec_src[i] = OBS_SOURCES[name]
        for j, v in enumerate(obs.scales):
            d.obs_scale[j] = v
        d.obs_height_scale = obs.height_scale
        for j, v in enumerate(obs.noise):
            d.obs_noise[j] = v
        d.obs_height_noise = obs.height_noise
    return d


class _Ctx:
    """RAII holder of a native ShifuCtx."""

    def __init__(self, device: torch.device, a1: Optional[nv.A1Desc] = None, abb: Optional[nv.AbbDesc] = None):
        self.lib = nv.load()
        if device.type != "cuda":
            raise nv.ShifuNativeError(nv.E_NODEVICE, f"device {device} is not CUDA: the shifu_b200 hot "
                                                     "path has no CPU fallback")
        self.handle = C.c_void_p()
        idx = device.index if device.index is not None else torch.cuda.current_device()
        nv.check(self.lib.shifu_ctx_create(idx, C.byref(a1) if a1 is not None else None,
                                           C.byref(abb) if abb is not None else None, C.byref(self.handle)))

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            self.lib.shifu_ctx_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class EnvKernels:
    """Task-independent rows for envs whose hooks stay user-written torch code: reset-id
    compaction (a8), history push (a13), clip (a14), body-frame velocities (a3)."""

    def __init__(self, device, num_envs: int):
        self.lib = nv.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise nv.ShifuNativeError(nv.E_NODEVICE, f"device {device} is not CUDA: the shifu_b200 kernels "
                                                     "have no CPU fallback")
        self.n = num_envs
        self.handle = C.c_void_p()
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        nv.check(self.lib.shifu_ctx_create_util(idx, num_envs, C.byref(self.handle)))
        self._ids = torch.zeros(num_envs, device=self.device, dtype=torch.long)
        self._cnt = torch.zeros(1, device=self.device, dtype=torch.int32)

    def __del__(self):
        try:
            if self.handle.value:
                self.lib.shifu_ctx_destroy(self.handle)
        except Exception:
            pass

    def nonzero(self, flags: torch.Tensor) -> torch.Tensor:
        """``flags.nonzero().flatten()`` (env.py:101): ascending int64 ids.  Synchronises to learn
        the length, like the reference's ``nonzero`` does."""
        f = flags if flags.dtype in (torch.bool, torch.uint8) else (flags != 0)
        f = f.contiguous()
        nv.check(self.lib.shifu_compact_reset_ids(self.handle, nv.ptr(f), f.numel(), nv.ptr(self._ids),
                                                  nv.ptr(self._cnt), nv.current_stream()))
        return self._ids[: int(self._cnt.item())].clone()

    def history_add(self, history_buf: torch.Tensor, x: torch.Tensor):
        n, a, h = history_buf.shape
        nv.check(self.lib.shifu_history_add(self.handle, nv.ptr(history_buf), nv.ptr(x.contiguous()), n, a, h,
                                            nv.current_stream()))

    def clip(self, x: torch.Tensor, c: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        x = x.contiguous()
        out = torch.empty_like(x) if out is None else out
        nv.check(self.lib.shifu_clip(self.handle, nv.ptr(x), nv.ptr(out), x.numel(), float(c), nv.current_stream()))
        return out

    def arm_ik(self, *, body_state, num_bodies: int, ee_body: int, jacobian, ee_link: int, dof_state, num_dof: int,
               dof_targets, goal_pose=None, actions=None, ee_velocity: float = 0.0, dt: float = 0.0,
               min_ee_pos=(0., 0., 0.), max_ee_pos=(0., 0., 0.), tar_quat=(0., 0., 0., 1.), damping: float = 0.05):
        """Row N2: ``ArmRobot.inverse_kinematics`` (robot.py:156-182), optionally preceded by the
        action -> end-effector goal of ``AbbRobot.step`` (a_prior_stage.py:67-71)."""
        io = nv.ArmIkIO()
        if not (jacobian.is_contiguous() and jacobian.dim() == 4 and jacobian.shape[2] == 6):
            raise ValueError("jacobian must be the contiguous (N, links, 6, dofs) gym tensor")
        io.body_state, io.jacobian, io.dof_state = nv.ptr(body_state), nv.ptr(jacobian), nv.ptr(dof_state)
        io.goal_pose = nv.ptr(goal_pose.contiguous()) if goal_pose is not None else None
        io.actions = nv.ptr(actions.contiguous()) if actions is not None else None
        io.dof_targets = nv.ptr(dof_targets)
        io.num_bodies, io.ee_body, io.num_links, io.ee_link = num_bodies, ee_body, jacobian.shape[1], ee_link
        io.num_dof, io.ee_velocity, io.dt, io.damping = num_dof, ee_velocity, dt, damping
        for i in range(3):
            io.min_ee_pos[i], io.max_ee_pos[i] = float(min_ee_pos[i]), float(max_ee_pos[i])
        for i in range(4):
            io.tar_quat[i] = float(tar_quat[i])
        nv.check(self.lib.shifu_arm_ik(self.handle, C.byref(io), jacobian.shape[0], nv.current_stream()))
        return dof_targets

    def camera_gather(self, *, height: int, width: int, normalize_color: bool, color=None, depth=None, seg=None,
                      flow=None):
        """Row N4: ``CameraSensor.refresh_image_tensors`` (sensors.py:165-188) in one launch.  Each of
        color / depth / seg / flow is ``(pointer_table, out)``: an int64 device tensor holding the N
        per-env image addresses and the batched output buffer."""
        io = nv.CameraGatherIO()
        io.height, io.width, io.normalize_color = height, width, int(bool(normalize_color))
        n = None
        for name, pair in (("color", color), ("depth", depth), ("seg", seg), ("flow", flow)):
            if pair is None:
                continue
            table, out = pair
            if table.dtype != torch.int64 or not table.is_contiguous():
                raise ValueError(f"{name}: the pointer table must be a contiguous int64 tensor")
            n = table.numel() if n is None else n
            if table.numel() != n or out.shape[0] != n or not out.is_contiguous():
                raise ValueError(f"{name}: table / output size mismatch")
            setattr(io, name + "_src", nv.ptr(table))
            setattr(io, name + "_out", nv.ptr(out))
        if n is not None:
            nv.check(self.lib.shifu_camera_gather(self.handle, C.byref(io), n, nv.current_stream()))

    def body_frame(self, root_state, n, stride, offset, lin, ang, pg, gvec=None):
        nv.check(self.lib.shifu_body_frame(self.handle, nv.ptr(root_state), n, stride, offset, nv.ptr(lin),
                                           nv.ptr(ang), nv.ptr(pg), nv.ptr(gvec), nv.current_stream()))


EXTRAS_SLOTS = 64      # ring of per-step extras arrays (rsl_rl holds the dicts of one 24-step rollout)


class _StepStats:
    """Per-step statistics -> ``extras`` plumbing shared by the two hot paths.

    Every step publishes into its own slot of ``extras_ring`` so the dict returned for step t is
    not overwritten by step t+1 (the reference allocates fresh tensors whenever somebody resets,
    env.py:124-130).  In sharded runs the 16-double all-reduce and the publish run on a side
    stream: the next step's kernels never wait for the collective (SURVEY.md §5); the main stream
    re-joins at the start of the next step (``wait_stats``), by which time it has long finished."""

    def _init_stats(self, dev):
        self.stats_ring = torch.zeros(EXTRAS_SLOTS, nv.NUM_STATS, device=dev, dtype=torch.double)
        self.extras_ring = torch.zeros(EXTRAS_SLOTS, nv.NUM_STATS, device=dev, dtype=torch.float)
        self._stats_slot = 0
        self._side = None
        self._pending = None
        self._slot_events = {}

    @property
    def slot(self) -> int:
        return self.step_counter % EXTRAS_SLOTS

    @property
    def stats(self) -> torch.Tensor:
        return self.stats_ring[self._stats_slot]

    @property
    def extras_arr(self) -> torch.Tensor:
        return self.extras_ring[self.slot]

    def wait_stats(self):
        """Main stream waits for the side-stream all-reduce + publish still in flight (call before reading
        ``extras`` values of a sharded run on the main stream; single-GPU runs publish in-stream)."""
        if self._pending is not None:
            torch.cuda.current_stream().wait_event(self._pending)
            self._pending = None

    def _slot_guard(self):
        """Before a slot of the rings is reused: its side-stream user of EXTRAS_SLOTS steps ago is done."""
        done = self._slot_events.pop(self.slot, None)
        if done is not None:
            torch.cuda.current_stream().wait_event(done)

    def _collect(self, advance_step_dev: bool):
        """Step statistics -> this step's slot of the ring (capturable: the slot can come from the device
        step counter)."""
        self._stats_slot = self.slot
        if not torch.cuda.is_current_stream_capturing():
            self._slot_guard()
        nv.check(self.lib.shifu_collect_stats_ring(self.ctx.handle, nv.ptr(self.stats_ring), EXTRAS_SLOTS,
                                                   -1 if advance_step_dev else self.slot,
                                                   nv.ptr(self.step_dev) if advance_step_dev else None,
                                                   nv.current_stream()))

    def _publish(self, allreduce, from_step_dev: bool = False):
        """(all-reduce over ranks ->) extras of this step's slot.  With a collective both run on a side
        stream: nothing on the main stream waits for them, the next step starts right away; the slot's
        previous user (EXTRAS_SLOTS steps ago) has long finished."""
        lib, h, slot = self.lib, self.ctx.handle, self.slot
        st = self.stats_ring[slot]
        if allreduce is None:
            nv.check(lib.shifu_publish_extras_ring(h, nv.ptr(self.stats_ring) if from_step_dev else nv.ptr(st),
                                                   nv.ptr(self.extras_ring), EXTRAS_SLOTS, -1 if from_step_dev else slot,
                                                   nv.ptr(self.step_dev), nv.current_stream()))
            return
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.device)
        self._side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self._side):
            allreduce(st)
            nv.check(lib.shifu_publish_extras_ring(h, nv.ptr(st), nv.ptr(self.extras_ring), EXTRAS_SLOTS, slot, None,
                                                   nv.current_stream()))
            self._pending = torch.cuda.Event()
            self._pending.record(self._side)
            self._slot_events[slot] = self._pending

    def _finalize_stats(self, allreduce, advance_step_dev: bool):
        self._collect(advance_step_dev)
        self._publish(allreduce, from_step_dev=advance_step_dev)


class HeightScan:
    """Stand-alone row a5 (``TerrainGymEnv.get_heights``) for user-hook tasks."""

    def __init__(self, desc: nv.A1Desc, height_samples: torch.Tensor, root_state: torch.Tensor):
        self.ctx = _Ctx(root_state.device, a1=desc)
        self.lib = self.ctx.lib
        self.root_state = root_state
        self.height_samples = height_samples.contiguous()
        self.out = torch.zeros(desc.num_envs, desc.num_points_x * desc.num_points_y, device=root_state.device)
        nv.check(self.lib.shifu_set_height_map(self.ctx.handle, nv.ptr(self.height_samples),
                                               self.height_samples.shape[0], self.height_samples.shape[1],
                                               nv.current_stream()))

    def run(self, cell_idx: Optional[torch.Tensor] = None) -> torch.Tensor:
        nv.check(self.lib.shifu_get_heights(self.ctx.handle, nv.ptr(self.root_state), nv.ptr(self.out),
                                            nv.ptr(cell_idx), nv.current_stream()))
        return self.out


class A1HotPath(_StepStats):
    """Fused A1 step. ``root_state`` / ``dof_state`` / ``contact_state`` are the gym's flat tensors.

    A blind descriptor (``num_obs = 72``, or 48 with the action head) builds the (N, 72) or (N, 48)
    observation without the height scan: it takes ``height_samples=None`` and keeps no ``measured_heights``.  A height map, when given, is uploaded for
    ``get_heights(out=...)``, which then needs its own output tensor."""

    def __init__(self, desc: nv.A1Desc, *, root_state, dof_state, contact_state, height_samples,
                 terrain_origins, terrain_types, env_origins, terms: Sequence[str] = A1_DEFAULT_TERMS,
                 carry_body_frame: bool = False, want_measured_heights: bool = True):
        dev = root_state.device
        self.device = dev
        self.desc = desc
        self.n = n = desc.num_envs
        self.terms = list(terms)
        self.blind = desc.num_obs in (nv.OBS_HEAD, nv.OBS_HEAD_ACT)
        if self.blind and want_measured_heights:
            raise ValueError(f"a blind A1 step (num_obs = {desc.num_obs}) does not scan: it cannot store "
                             "measured_heights")
        if height_samples is None and not self.blind:
            raise ValueError(f"the {desc.num_obs}-column A1 step scans the height map: height_samples is required")
        self.ctx = _Ctx(dev, a1=desc)
        self.lib = self.ctx.lib
        f = dict(device=dev, dtype=torch.float)
        # borrowed simulator tensors
        self.root_state, self.dof_state, self.contact_state = root_state, dof_state, contact_state
        # terrain (isaac_gym.py:336-347)
        self.height_samples = height_samples.to(dev).contiguous() if height_samples is not None else None
        assert self.height_samples is None or self.height_samples.dtype == torch.int16
        self.terrain_origins = terrain_origins.to(**f).contiguous()
        self.terrain_types = terrain_types.to(dev, torch.long).contiguous()
        self.env_origins = env_origins            # (N,3) fp32, shared with the gym façade
        # env-side buffers (env.py:44-63, a1_conditional.py:52-62,100-114)
        self.actions = torch.zeros(n, 12, **f)
        self.torques = torch.zeros(n, 12, **f)
        self.history = torch.zeros(n, 12, 3, **f)
        self.command = torch.zeros(n, 3, **f)
        self.ep_len = torch.zeros(n, device=dev, dtype=torch.long)
        self.ep_sums = {k: torch.zeros(n, **f) for k in self.terms}
        self.base_lin_vel = torch.zeros(n, 3, **f)
        self.base_ang_vel = torch.zeros(n, 3, **f)
        self.projected_gravity = torch.zeros(n, 3, **f)
        self.gravity_vec = torch.tensor([0., 0., -1.], **f).repeat(n, 1)
        self.terrain_levels = torch.zeros(n, device=dev, dtype=torch.long)
        self.dof_targets = torch.zeros(n, 12, **f)
        self.rand_force = torch.zeros(n, 17, 3, **f)
        self.obs_buf = torch.zeros(n, desc.num_obs, **f)
        self.rew_buf = torch.zeros(n, **f)
        self.reset_buf = torch.ones(n, device=dev, dtype=torch.bool)
        self.time_out_buf = torch.zeros(n, device=dev, dtype=torch.bool)
        self.contact_terminate_buf = torch.zeros(n, device=dev, dtype=torch.bool)
        self.measured_heights = torch.zeros(n, 187, **f) if want_measured_heights else None
        self.reset_ids = torch.zeros(n, device=dev, dtype=torch.long)
        self.n_reset = torch.zeros(1, device=dev, dtype=torch.int32)
        self.step_dev = torch.zeros(1, device=dev, dtype=torch.long)
        # feet-air-time state (legged_gym feet_air_time / last_contacts), used by the term of that name only
        self.swing_time = torch.zeros(n, max(desc.num_feet, 1), **f)
        self.last_contacts = torch.zeros(n, max(desc.num_feet, 1), device=dev, dtype=torch.bool)
        self.step_counter = 0
        self._pd_substep = -1            # decimation substep of the last pd_torque call
        self._init_stats(dev)
        self._graph, self._graph_warm, self._dev_step, self._graph_actions = None, 0, -1, None
        self._fork = None
        self.carry_body_frame = carry_body_frame
        self._io = None
        if self.height_samples is not None:
            nv.check(self.lib.shifu_set_height_map(self.ctx.handle, nv.ptr(self.height_samples),
                                                   self.height_samples.shape[0], self.height_samples.shape[1],
                                                   nv.current_stream()))
        self.sync_level_sum()

    # ------------------------------------------------------------------
    def _build_io(self, use_step_dev: bool) -> nv.A1StepIO:
        io = nv.A1StepIO()
        p = nv.ptr
        io.root_state, io.dof_state, io.contact_state = p(self.root_state), p(self.dof_state), p(self.contact_state)
        io.actions, io.torques, io.history, io.command = p(self.actions), p(self.torques), p(self.history), p(self.command)
        io.ep_len = p(self.ep_len)
        for i, k in enumerate(self.terms):
            io.ep_sums[i] = p(self.ep_sums[k])
        io.base_lin_vel, io.base_ang_vel = p(self.base_lin_vel), p(self.base_ang_vel)
        io.projected_gravity = p(self.projected_gravity)
        io.env_origins, io.terrain_levels = p(self.env_origins), p(self.terrain_levels)
        io.terrain_types, io.terrain_origins = p(self.terrain_types), p(self.terrain_origins)
        io.dof_targets, io.rand_force = p(self.dof_targets), p(self.rand_force)
        io.obs_buf, io.rew_buf, io.reset_buf = p(self.obs_buf), p(self.rew_buf), p(self.reset_buf)
        io.time_out_buf, io.contact_term_buf = p(self.time_out_buf), p(self.contact_terminate_buf)
        io.measured_heights = p(self.measured_heights)
        io.step = self.step_counter
        io.step_dev = p(self.step_dev) if use_step_dev else None
        io.swing_time, io.last_contacts = p(self.swing_time), p(self.last_contacts)
        io.carry_body_frame = int(self.carry_body_frame)
        return io

    def io(self, use_step_dev: bool = False) -> nv.A1StepIO:
        if self._io is None or bool(self._io.step_dev) != use_step_dev:
            self._io = self._build_io(use_step_dev)
        self._io.step = self.step_counter
        self._io.carry_body_frame = int(self.carry_body_frame)
        return self._io

    def invalidate_io(self):
        """Call after re-binding any tensor attribute (pointers are cached)."""
        self._io = None

    _ADOPTABLE = ("actions", "torques", "history", "command", "ep_len", "base_lin_vel", "base_ang_vel",
                  "projected_gravity", "terrain_levels", "dof_targets", "rand_force", "swing_time", "last_contacts")

    def adopt(self, **tensors):
        """Use the caller's existing tensors instead of the ones allocated here (an env built by user
        code already owns them; its hooks close over them).  Shapes / dtypes must match."""
        for name, t in tensors.items():
            if name not in self._ADOPTABLE:
                raise KeyError(f"{name} cannot be adopted")
            mine = getattr(self, name)
            if t.shape != mine.shape or t.dtype != mine.dtype or t.device != mine.device or not t.is_contiguous():
                raise ValueError(f"{name}: expected contiguous {tuple(mine.shape)} {mine.dtype} on {mine.device}, got "
                                 f"{tuple(t.shape)} {t.dtype} on {t.device}")
            setattr(self, name, t)
        self.invalidate_io()
        if "terrain_levels" in tensors:
            self.sync_level_sum()

    def eval_terms(self) -> torch.Tensor:
        """(num_terms, N): every listed reward term on the current tensors (``shifu_a1_eval_terms``)."""
        out = torch.empty(len(self.terms), self.n, device=self.device, dtype=torch.float)
        nv.check(self.lib.shifu_a1_eval_terms(self.ctx.handle, C.byref(self.io(False)), nv.ptr(out), nv.current_stream()))
        return out

    def sync_level_sum(self):
        nv.check(self.lib.shifu_set_level_sum(self.ctx.handle, nv.ptr(self.terrain_levels), nv.current_stream()))

    # -- individual rows -------------------------------------------------
    def pd_torque(self, raw_actions: Optional[torch.Tensor] = None):
        """Row a2 (+a1 when ``raw_actions`` is given: env.actions = clip(0.5*a, +-1) is produced too).
        A call with ``raw_actions`` is decimation substep 0, one without is the previous substep + 1;
        the library picks each substep's sweep order from that number (the results do not depend on it)."""
        s = nv.current_stream()
        self._pd_substep = 0 if raw_actions is not None else self._pd_substep + 1
        if raw_actions is not None:
            nv.check(self.lib.shifu_pd_torque(self.ctx.handle, nv.ptr(raw_actions), nv.ptr(self.actions),
                                              nv.ptr(self.dof_state), nv.ptr(self.torques), self._pd_substep, s))
        else:
            nv.check(self.lib.shifu_pd_torque(self.ctx.handle, nv.ptr(self.actions), None,
                                              nv.ptr(self.dof_state), nv.ptr(self.torques), self._pd_substep, s))

    def body_frame(self):
        """Row a3: LeggedRobot.post_step on the CURRENT content of root_state (S_prev, D7)."""
        nv.check(self.lib.shifu_body_frame(self.ctx.handle, nv.ptr(self.root_state), self.n,
                                           self.desc.root_stride, self.desc.root_offset,
                                           nv.ptr(self.base_lin_vel), nv.ptr(self.base_ang_vel),
                                           nv.ptr(self.projected_gravity), nv.ptr(self.gravity_vec),
                                           nv.current_stream()))

    def get_heights(self, out: Optional[torch.Tensor] = None, cell_idx: Optional[torch.Tensor] = None):
        """Row a5 stand-alone."""
        out = self.measured_heights if out is None else out
        nv.check(self.lib.shifu_get_heights(self.ctx.handle, nv.ptr(self.root_state), nv.ptr(out),
                                            nv.ptr(cell_idx), nv.current_stream()))
        return out

    def post_physics(self, use_step_dev: bool = False):
        """Rows a5-a7, a9-a14 in one kernel.  Advances the host step counter (env.py:96)."""
        self.step_counter += 1
        nv.check(self.lib.shifu_a1_post_physics(self.ctx.handle, C.byref(self.io(use_step_dev)), nv.current_stream()))

    def compact(self):
        """Row a8: ascending reset ids + count (device)."""
        nv.check(self.lib.shifu_compact_reset_ids(self.ctx.handle, nv.ptr(self.reset_buf), self.n,
                                                  nv.ptr(self.reset_ids), nv.ptr(self.n_reset), nv.current_stream()))

    def reset_idx(self, env_ids: Optional[torch.Tensor], allreduce=None):
        """Rows a9-a11 stand-alone (``A1Conditional.reset_idx``); ``None`` = all envs.  In a sharded
        run every rank must call it (possibly with no ids): the statistics all-reduce is collective."""
        n_ids = self.n if env_ids is None else int(env_ids.numel())
        if env_ids is not None:
            env_ids = env_ids.to(self.device, torch.long).contiguous()
        self.wait_stats()
        nv.check(self.lib.shifu_a1_reset_idx(self.ctx.handle, C.byref(self.io(False)), nv.ptr(env_ids), n_ids,
                                             nv.current_stream()))
        if n_ids > 0 and self.carry_body_frame:
            self.body_frame()               # the carried velocities follow the rewritten root rows (robot.py:222-229)
        if n_ids > 0 or allreduce is not None:      # log_info runs inside reset_idx (env.py:124-130)
            self._finalize_stats(allreduce, False)

    def finalize(self, allreduce=None, advance_step_dev: bool = False):
        """compaction + stats -> (optional all-reduce over ranks, on a side stream) -> extras."""
        self.compact()
        self._finalize_stats(allreduce, advance_step_dev)

    # -- the whole control step without a simulator in between (bench / graph capture) ------
    def step_resident(self, raw_actions: torch.Tensor, decimation: int = 4, use_step_dev: bool = False,
                      allreduce=None, publish: bool = True):
        """PD x decimation, (body-frame unless carried), fused post-physics, compaction, stats —
        on whatever the flat state tensors currently hold."""
        self.pd_torque(raw_actions)
        for _ in range(decimation - 1):
            self.pd_torque()
        if not self.carry_body_frame:
            self.body_frame()
        self.post_physics(use_step_dev)
        main = torch.cuda.current_stream()
        if torch.cuda.is_current_stream_capturing():
            # inside the step graph the id compaction and the statistics collect / publish are independent
            # branches after the fused kernel: two latency-bound tails run side by side
            if self._fork is None:
                self._fork = torch.cuda.Stream(device=self.device)
            self._fork.wait_stream(main)
            with torch.cuda.stream(self._fork):
                self.compact()
        else:
            self.compact()
        self._collect(use_step_dev)
        if publish:
            self._publish(allreduce, from_step_dev=use_step_dev)
        if torch.cuda.is_current_stream_capturing():
            main.wait_stream(self._fork)

    # -- the same step as ONE CUDA-graph replay (launch-bound small-N configurations) -----------
    def graph_step(self, raw_actions: torch.Tensor, decimation: int = 4, allreduce=None):
        """``step_resident`` captured once and replayed: PD x decimation, (body frame), fused post-physics,
        compaction, statistics and extras publish cost one graph launch instead of 8-9 kernel launches
        (52 -> ~20 us per step at 4 096 envs).  Only valid when nothing has to run between the launches
        (resident state: no simulator crossing).  The Philox step counter lives on the device
        (``step_dev``) and is advanced inside the graph.  In a sharded run the graph ends with the
        statistics collect; the all-reduce and the publish follow on the side stream."""
        if self._graph is None:
            if self._graph_warm < 2:                     # first launches outside capture (module loading)
                self._graph_warm += 1
                return self.step_resident(raw_actions, decimation, allreduce=allreduce)
            if self._graph_actions is None:
                self._graph_actions = torch.empty_like(raw_actions)
            if raw_actions.data_ptr() != self._graph_actions.data_ptr():
                self._graph_actions.copy_(raw_actions)
            self.step_dev.fill_(self.step_counter + 1)
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            before = self.step_counter
            with torch.cuda.graph(graph):
                self.step_resident(self._graph_actions, decimation, use_step_dev=True, publish=allreduce is None)
            self.step_counter = before                   # capture recorded the launches without running them
            self._graph, self._graph_decimation, self._dev_step = graph, decimation, before + 1
            self._graph_publishes = allreduce is None
        if decimation != self._graph_decimation or raw_actions.shape != self._graph_actions.shape or \
                self._graph_publishes != (allreduce is None):
            raise ValueError("graph_step was captured for another decimation / action shape / collective mode")
        if self._dev_step != self.step_counter + 1:      # eager steps or resets ran in between
            self.step_dev.fill_(self.step_counter + 1)
        if raw_actions.data_ptr() != self._graph_actions.data_ptr():   # callers that write into
            self._graph_actions.copy_(raw_actions)                       # action_input() skip this copy
        self.step_counter += 1
        self._stats_slot = self.slot
        self._slot_guard()
        self._graph.replay()
        self._dev_step = self.step_counter + 1
        if allreduce is not None:
            self._publish(allreduce)

    def action_input(self) -> torch.Tensor:
        """The (N, 12) buffer the captured step reads its raw actions from: a policy that writes its
        output here (``out=``) and passes this tensor to ``step`` saves the per-step action copy."""
        if self._graph_actions is None:
            self._graph_actions = torch.zeros(self.n, 12, device=self.device)
        return self._graph_actions

    def extras(self) -> Dict:
        """``extras`` of the last finalised step: a fresh dict of 0-dim views into that step's own slot
        of the ring (env.py:124-130, a1_conditional.py:126-129)."""
        arr = self.extras_arr
        ep = {k: arr[i] for i, k in enumerate(self.terms)}
        ep["terrain_levels"] = arr[nv.STAT_LEVEL_SUM]
        return {"episode": ep, "time_outs": self.time_out_buf}

    def reset_id_list(self) -> torch.Tensor:
        """Host-synchronising view of the compacted ids (like ``nonzero`` in the reference)."""
        return self.reset_ids[: int(self.n_reset.item())]


def abb_desc(num_envs: int, *, env_offset: int = 0, rng_seed: int = 0x5EED,
             terms: Sequence[str] = tuple(ABB_TERM_CODES), term_params: Optional[Dict[str, tuple]] = None) -> nv.AbbDesc:
    """Constants of ``examples/abb_pushbox_vision`` prior stage (task_config.py:49-91)."""
    d = nv.AbbDesc()
    d.abi_version = nv.ABI_VERSION
    d.num_envs, d.env_offset, d.rng_seed = num_envs, env_offset, rng_seed
    d.num_actors, d.num_bodies, d.num_dof, d.ee_body = 4, 10, 6, 6
    d.robot_actor, d.table_actor, d.cube_actor, d.goal_actor = 0, 1, 2, 3
    for i, v in enumerate((-0.2, -0.2, 0.11)):
        d.min_ee_pos[i] = v
    for i, v in enumerate((0.2, 0.2, 0.14)):
        d.max_ee_pos[i] = v
    for i, v in enumerate((0., 0.6437, 0.1748, 0., 0.7541, 0.)):
        d.q0[i] = v
    for i, v in enumerate((-0.48, 0, 0, 0, 0, 0, 1)):
        d.robot_root[i] = v
    for i, v in enumerate((0, 0, 0.05, 0, 0, 0, 1)):
        d.table_root[i] = v
    for i, (lo, hi) in enumerate(((-0.1, 0.1), (-0.1, 0.1), (0.125, 0.125))):
        d.box_pos_low[i], d.box_pos_high[i] = lo, hi
    d.goal_z = 0.1
    d.success_distance = 0.02
    d.max_episode_length, d.max_episode_length_s, d.clip_obs = 200, 20., 10.
    comp = compile_reward_terms(list(terms), ABB_TERM_CODES, {**ABB_TERM_PARAMS, **(term_params or {})})
    d.num_reward_terms = len(comp)
    for i, (code, p0, p1) in enumerate(comp):
        d.reward_terms[i] = code
        d.reward_params[i][0], d.reward_params[i][1] = p0, p1
    return d


class AbbHotPath(_StepStats):
    def __init__(self, desc: nv.AbbDesc, *, root_state, body_state, dof_state,
                 terms: Sequence[str] = tuple(ABB_TERM_CODES)):
        dev = root_state.device
        self.device, self.desc, self.n = dev, desc, desc.num_envs
        n = self.n
        self.terms = list(terms)
        self.ctx = _Ctx(dev, abb=desc)
        self.lib = self.ctx.lib
        f = dict(device=dev, dtype=torch.float)
        self.root_state, self.body_state, self.dof_state = root_state, body_state, dof_state
        self.dof_targets = torch.zeros(n, 6, **f)
        self.ep_len = torch.zeros(n, device=dev, dtype=torch.long)
        self.ep_sums = {k: torch.zeros(n, **f) for k in self.terms}
        self.obs_buf = torch.zeros(n, 6, **f)
        self.rew_buf = torch.zeros(n, **f)
        self.reset_buf = torch.ones(n, device=dev, dtype=torch.bool)
        self.time_out_buf = torch.zeros(n, device=dev, dtype=torch.bool)
        self.success_buf = torch.zeros(n, device=dev, dtype=torch.bool)
        self.reset_ids = torch.zeros(n, device=dev, dtype=torch.long)
        self.n_reset = torch.zeros(1, device=dev, dtype=torch.int32)
        self.step_dev = torch.zeros(1, device=dev, dtype=torch.long)
        self.step_counter = 0
        self._init_stats(dev)
        self._io = None

    def io(self, use_step_dev: bool = False) -> nv.AbbStepIO:
        if self._io is None or bool(self._io.step_dev) != use_step_dev:
            io = nv.AbbStepIO()
            p = nv.ptr
            io.root_state, io.body_state, io.dof_state = p(self.root_state), p(self.body_state), p(self.dof_state)
            io.dof_targets, io.ep_len = p(self.dof_targets), p(self.ep_len)
            for i, k in enumerate(self.terms):
                io.ep_sums[i] = p(self.ep_sums[k])
            io.obs_buf, io.rew_buf, io.reset_buf = p(self.obs_buf), p(self.rew_buf), p(self.reset_buf)
            io.time_out_buf, io.success_buf = p(self.time_out_buf), p(self.success_buf)
            io.step_dev = p(self.step_dev) if use_step_dev else None
            self._io = io
        self._io.step = self.step_counter
        return self._io

    def post_physics(self, use_step_dev: bool = False):
        self.step_counter += 1
        nv.check(self.lib.shifu_abb_post_physics(self.ctx.handle, C.byref(self.io(use_step_dev)), nv.current_stream()))

    def finalize(self, allreduce=None, advance_step_dev: bool = False):
        nv.check(self.lib.shifu_compact_reset_ids(self.ctx.handle, nv.ptr(self.reset_buf), self.n,
                                                  nv.ptr(self.reset_ids), nv.ptr(self.n_reset), nv.current_stream()))
        self._finalize_stats(allreduce, advance_step_dev)

    def reset_idx(self, env_ids: Optional[torch.Tensor], allreduce=None):
        """``ShifuVecEnv.reset_idx(env_ids)`` of the push-box scene stand-alone (env.py:114-130 with the
        random cube / goal poses of a_prior_stage.py:39-51); ``None`` = all envs."""
        n_ids = self.n if env_ids is None else int(env_ids.numel())
        if env_ids is not None:
            env_ids = env_ids.to(self.device, torch.long).contiguous()
        self.wait_stats()
        nv.check(self.lib.shifu_abb_reset_idx(self.ctx.handle, C.byref(self.io(False)), nv.ptr(env_ids), n_ids,
                                              nv.current_stream()))
        if n_ids > 0 or allreduce is not None:
            self._finalize_stats(allreduce, False)

    def step_resident(self, use_step_dev: bool = False, allreduce=None):
        self.post_physics(use_step_dev)
        self.finalize(allreduce, advance_step_dev=use_step_dev)

    def extras(self) -> Dict:
        arr = self.extras_arr
        ep = {k: arr[i] for i, k in enumerate(self.terms)}
        ep["success_rate"] = arr[nv.STAT_SUCCESS]
        return {"episode": ep, "time_outs": self.time_out_buf}

    def reset_id_list(self) -> torch.Tensor:
        return self.reset_ids[: int(self.n_reset.item())]
