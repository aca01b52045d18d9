"""ORACLE — test infrastructure, NOT product code.

A CPU restatement (torch, fp32, eager) of the reference's per-step post-physics
hot path, written as plain functions over plain tensors: no Isaac Gym, no class
tree.  Every function cites the reference lines it follows
(paths relative to ``/root/reference``).  torch CPU is used on purpose: the
parity target named by BASELINE.json is "the reference's own torch
implementation ... on torch CPU", and using the same aten ops in the same order
makes this restatement bit-identical to the unmodified reference
(checked by ``tests/test_oracle_cpu.py`` in the build container and
through the committed fixtures under ``tests/golden/`` everywhere else).

PARITY PINNING: the reference ships **no** tests, golden vectors or fixtures for
this path (SURVEY.md §4, §8c).  The pin is therefore "outputs of the reference
itself run here": ``oracle/make_golden.py`` drives the unmodified reference
through ``oracle/ref_harness.py`` and commits the vectors; this file must
reproduce them exactly.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline``
/ ``--impl reference`` legs may import this module.

Third-party arithmetic (un-vendored): ``isaacgym.torch_utils`` of Isaac Gym
Preview 3 (``README.md:30``); restated from the public BSD-3 definitions in
``isaacgymenvs/utils/torch_jit_utils.py``: ``quat_rotate_inverse``,
``quat_apply``, ``normalize``, ``quat_from_euler_xyz``, ``torch_rand_float``.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from . import philox_np as px

# ---------------------------------------------------------------------------
# isaacgym.torch_utils restatements
# ---------------------------------------------------------------------------


def normalize(x, eps: float = 1e-9):
    return x / x.norm(p=2, dim=-1).clamp(min=eps, max=None).unsqueeze(-1)


def quat_apply(a, b):
    shape = b.shape
    a = a.reshape(-1, 4)
    b = b.reshape(-1, 3)
    xyz = a[:, :3]
    t = xyz.cross(b, dim=-1) * 2
    return (b + a[:, 3:] * t + xyz.cross(t, dim=-1)).view(shape)


def quat_rotate_inverse(q, v):
    shape = q.shape
    q_w = q[:, -1]
    q_vec = q[:, :3]
    a = v * (2.0 * q_w ** 2 - 1.0).unsqueeze(-1)
    b = torch.cross(q_vec, v, dim=-1) * q_w.unsqueeze(-1) * 2.0
    c = q_vec * torch.bmm(q_vec.view(shape[0], 1, 3), v.view(shape[0], 3, 1)).squeeze(-1) * 2.0
    return a - b + c


def quat_from_euler_xyz(roll, pitch, yaw):
    cy, sy = torch.cos(yaw * 0.5), torch.sin(yaw * 0.5)
    cr, sr = torch.cos(roll * 0.5), torch.sin(roll * 0.5)
    cp, sp = torch.cos(pitch * 0.5), torch.sin(pitch * 0.5)
    qw = cy * cr * cp + sy * sr * sp
    qx = cy * sr * cp - sy * cr * sp
    qy = cy * cr * sp + sy * sr * cp
    qz = sy * cr * cp - cy * sr * sp
    return torch.stack([qx, qy, qz, qw], dim=-1)


def quat_apply_yaw(quat, vec):
    """shifu/utils/terrain.py:202-206"""
    quat_yaw = quat.clone().view(-1, 4)
    quat_yaw[:, :2] = 0.
    quat_yaw = normalize(quat_yaw)
    return quat_apply(quat_yaw, vec)


# ---------------------------------------------------------------------------
# A1 conditional walking
# ---------------------------------------------------------------------------

A1_REWARD_TERMS = ["tracking_lin_vel", "tracking_ang_vel", "stabilizing_base", "smoothing_action",
                   "leg_collision", "torques_penalize"]   # a1_conditional.py:152-160
# (p0, p1) of each term: the literals of a1_conditional.py:162-192 for the reference's six terms
A1_TERM_PARAMS = {"tracking_lin_vel": (1.0, 0.25), "tracking_ang_vel": (0.5, 0.25), "stabilizing_base": (-2.0, -0.005),
                  "smoothing_action": (-0.005, 0.0), "leg_collision": (-1., 0.1), "torques_penalize": (-2e-5, 0.0)}
# legged_gym-style terms a user task may list (enum ShifuRewardTerm 8-15); their constants come with the list
A1_EXTRA_TERMS = ("lin_vel_z", "ang_vel_xy", "orientation", "dof_vel", "action_rate", "base_height", "dof_pos_limits",
                  "feet_air_time")
A1_DOF_UNBOUNDED = 3.0e38                 # default dof_pos_limits: (-3e38, 3e38), never reached


@dataclass
class A1Params:
    """Constants the reference reads from its config tree / URDF (SURVEY.md Appendix A)."""
    n: int
    q0: torch.Tensor = None                  # task_config.py:17-20
    kp: torch.Tensor = None                  # task_config.py:22
    kd: torch.Tensor = None                  # task_config.py:23
    torque_limits: torch.Tensor = None       # a1.urdf:95,137,165 via shifu/units/robot.py:42
    points_x: List[float] = None             # shifu/configs/env_config.py:87-88
    points_y: List[float] = None             # env_config.py:89
    border_size: float = 25                  # env_config.py:80 (python int in the reference)
    horizontal_scale: float = 0.1            # env_config.py:78
    vertical_scale: float = 0.005            # env_config.py:79
    env_length: float = 8.                   # env_config.py:92 -> Terrain.env_length
    max_terrain_level: int = 10              # shifu/gym/isaac_gym.py:345
    num_cols: int = 20
    max_episode_length: float = 500.0        # shifu/gym/env.py:42  ceil(10 / 0.02)
    max_episode_length_s: float = 10.        # task_config.py:36
    clip_obs: float = 100.                   # task_config.py:48-50
    clip_actions: float = 1.
    action_scale: float = 0.5                # a1_conditional.py:123
    decimation: int = 4                      # task_config.py:41-42
    base_index: int = 0                      # a1_conditional.py:98-99
    leg_indices: List[int] = None            # a1_conditional.py:59-61
    default_base_pose: torch.Tensor = None   # task_config.py:15-16
    n_bodies: int = 17
    n_dof: int = 12
    n_hist: int = 3
    curriculum: bool = True
    rng_seed: int = 0x5EED
    env_offset: int = 0                      # global id of local env 0 (sharded runs)
    # reward-term list in accumulation order: (name, p0, p1); default = the reference's six terms
    terms: List[Tuple[str, float, float]] = None
    # constants of the legged_gym-style terms beyond (p0, p1)
    dof_pos_limits: torch.Tensor = None      # (12, 2) lower / upper soft limits; default unbounded
    feet_bodies: Tuple[int, ...] = (4, 8, 12, 16)
    feet_contact_force: float = 1.0          # a foot touches when F_z > this
    air_time_cmd_min: float = 0.1            # feet_air_time is 0 unless |cmd_xy| > this
    air_time_dt: float = 0.02                # control dt added to swing_time every step
    air_time_reset: bool = True              # reset_idx zeroes swing_time / last_contacts of the env

    def __post_init__(self):
        f = lambda x: torch.tensor(x, dtype=torch.float)
        if self.terms is None:
            self.terms = [(k, *A1_TERM_PARAMS[k]) for k in A1_REWARD_TERMS]
        if self.dof_pos_limits is None:
            self.dof_pos_limits = f([[-A1_DOF_UNBOUNDED, A1_DOF_UNBOUNDED]] * 12)
        if self.q0 is None:
            self.q0 = f([0.1, 0.8, -1.5, 0.1, 0.8, -1.5, -0.1, 0.8, -1.5, -0.1, 0.8, -1.5])
        if self.kp is None:
            self.kp = f([20] * 12)
        if self.kd is None:
            self.kd = f([.5] * 12)
        if self.torque_limits is None:
            self.torque_limits = f([20., 55., 55.] * 4)
        if self.points_x is None:
            self.points_x = [-0.8, -0.7, -0.6, -0.5, -0.4, -0.3, -0.2, -0.1, 0., 0.1, 0.2, 0.3, 0.4, 0.5, 0.6,
                             0.7, 0.8]
        if self.points_y is None:
            self.points_y = [-0.5, -0.4, -0.3, -0.2, -0.1, 0., 0.1, 0.2, 0.3, 0.4, 0.5]
        if self.leg_indices is None:
            self.leg_indices = [2, 3, 6, 7, 10, 11, 14, 15]
        if self.default_base_pose is None:
            self.default_base_pose = f([0, 0, 0.42] + [0, 0, 0, 1.])

    def height_points(self):
        """shifu/gym/isaac_gym.py:304-318"""
        y = torch.tensor(self.points_y)
        x = torch.tensor(self.points_x)
        grid_x, grid_y = torch.meshgrid(x, y, indexing='xy')
        pts = torch.zeros(self.n, grid_x.numel(), 3)
        pts[:, :, 0] = grid_x.flatten()
        pts[:, :, 1] = grid_y.flatten()
        return pts


@dataclass
class A1State:
    """The mutable tensors of one A1 env set (flat gym layouts, SURVEY.md §8b.3)."""
    root_state: torch.Tensor         # (N,13)  one actor per env
    dof_state: torch.Tensor          # (N*12,2)
    contact_state: torch.Tensor      # (N*17,3)
    height_samples: torch.Tensor     # (rows, cols) int16
    terrain_origins: torch.Tensor    # (levels, types, 3)
    terrain_types: torch.Tensor      # (N,) int64
    env_origins: torch.Tensor        # (N,3)
    terrain_levels: torch.Tensor     # (N,) int64   (A1Conditional.terrain_levels)
    command: torch.Tensor            # (N,3)
    history: torch.Tensor            # (N,12,3)
    ep_len: torch.Tensor             # (N,) int64
    ep_sums: Dict[str, torch.Tensor]
    dof_targets: torch.Tensor        # (N,12)
    rand_force: torch.Tensor         # (N,17,3)
    torques: torch.Tensor            # (N,12)
    base_lin_vel: torch.Tensor       # (N,3)
    base_ang_vel: torch.Tensor
    projected_gravity: torch.Tensor
    gravity_vec: torch.Tensor
    step_counter: int = 0
    extras: Dict = field(default_factory=dict)
    # outputs of the last step
    actions: torch.Tensor = None
    obs: torch.Tensor = None
    rew: torch.Tensor = None
    reset: torch.Tensor = None
    time_out: torch.Tensor = None
    contact_term: torch.Tensor = None
    measured_heights: torch.Tensor = None
    reset_ids: torch.Tensor = None
    height_idx: Optional[torch.Tensor] = None   # (2, N*187) int64 px, py of the last scan
    swing_time: torch.Tensor = None             # (N, feet) legged_gym feet_air_time
    last_contacts: torch.Tensor = None          # (N, feet) bool


def a1_new_state(p: A1Params, height_samples, terrain_origins, terrain_types, env_origins) -> A1State:
    n = p.n
    z = torch.zeros
    root = z(n, 13)
    root[:, 6] = 1.0
    g = torch.tensor([0., 0., -1.]).repeat((n, 1))
    return A1State(
        root_state=root, dof_state=z(n * p.n_dof, 2), contact_state=z(n * p.n_bodies, 3),
        height_samples=height_samples, terrain_origins=terrain_origins, terrain_types=terrain_types,
        env_origins=env_origins.clone(), terrain_levels=z(n, dtype=torch.long), command=z(n, 3),
        history=z(n, p.n_dof, p.n_hist), ep_len=z(n, dtype=torch.long),
        ep_sums={t[0]: z(n) for t in p.terms}, dof_targets=z(n, p.n_dof),
        rand_force=z(n, p.n_bodies, 3), torques=z(n, p.n_dof),
        base_lin_vel=z(n, 3), base_ang_vel=z(n, 3), projected_gravity=g.clone(), gravity_vec=g,
        reset=torch.ones(n, dtype=torch.long), time_out=z(n, dtype=torch.bool),
        obs=z(n, 259), rew=z(n), swing_time=z(n, len(p.feet_bodies)),
        last_contacts=z(n, len(p.feet_bodies), dtype=torch.bool),
    )


def a1_pd_torque(p: A1Params, actions, dof_state):
    """One PD substep — examples/a1_conditional/a1_conditional.py:66-67 (row a2)."""
    dof = dof_state.view(p.n, p.n_dof, 2)
    dof_pos, dof_vel = dof[..., 0], dof[..., 1]          # shifu/units/robot.py:51-52
    torques = p.kp * (actions + p.q0 - dof_pos) - p.kd * dof_vel
    return torch.clip(torques, -p.torque_limits, p.torque_limits)


def body_frame(root_rows):
    """LeggedRobot.post_step — shifu/units/robot.py:222-229 (row a3).  ``root_rows`` (N,13)."""
    n = root_rows.shape[0]
    q = root_rows[:, 3:7]
    g = torch.tensor([0., 0., -1.]).repeat((n, 1))
    return (quat_rotate_inverse(q, root_rows[:, 7:10]), quat_rotate_inverse(q, root_rows[:, 10:13]),
            quat_rotate_inverse(q, g), g)


def get_heights(p: A1Params, base_pose, height_samples, height_points, return_idx=False):
    """TerrainGymEnv.get_heights — shifu/gym/isaac_gym.py:393-433 (row a5)."""
    n, k = height_points.shape[0], height_points.shape[1]
    points = quat_apply_yaw(base_pose[:, 3:7].repeat(1, k), height_points) + (base_pose[:, :3]).unsqueeze(1)
    points += p.border_size
    points = (points / p.horizontal_scale).long()
    px_ = points[:, :, 0].view(-1)
    py_ = points[:, :, 1].view(-1)
    px_ = torch.clip(px_, 0, height_samples.shape[0] - 2)
    py_ = torch.clip(py_, 0, height_samples.shape[1] - 2)
    heights1 = height_samples[px_, py_]
    heights2 = height_samples[px_ + 1, py_]
    heights3 = height_samples[px_, py_ + 1]
    heights = torch.min(heights1, heights2)
    heights = torch.min(heights, heights3)
    out = heights.view(n, -1) * p.vertical_scale
    if return_idx:
        return out, torch.stack([px_, py_])
    return out


def a1_compute_termination(p: A1Params, st: A1State):
    """a1_conditional.py:146-150 (row a6)."""
    contact_forces = st.contact_state.view(p.n, -1, 3)              # robot.py:201
    st.contact_term = torch.norm(contact_forces[:, p.base_index, :], dim=-1) > 1.
    st.time_out = st.ep_len > p.max_episode_length
    st.reset = st.time_out | st.contact_term


def a1_reward_terms(p: A1Params, st: A1State) -> Dict[str, torch.Tensor]:
    """The listed terms in list order, keyed by name (env.py:160-166).  The reference's six terms
    follow a1_conditional.py:162-192 with their literals replaced by (p0, p1); the legged_gym-style
    terms are written in legged_gym's torch form.  feet_air_time updates st.swing_time /
    st.last_contacts (row a7)."""
    out = {}
    for name, p0, p1 in p.terms:
        out[name] = _A1_TERMS[name](p, st, p0, p1)
    return out


def _tracking_lin_vel(p, st, p0, p1):
    lin_vel_error = torch.sum(torch.square(st.command[:, :2] - st.base_lin_vel[:, :2]), dim=1)
    return p0 * torch.exp(-lin_vel_error / p1)


def _tracking_ang_vel(p, st, p0, p1):
    ang_vel_error = torch.square(st.command[:, 2] - st.base_ang_vel[:, 2])
    return p0 * torch.exp(-ang_vel_error / p1)


def _stabilizing_base(p, st, p0, p1):
    z_vel = p0 * torch.square(st.base_lin_vel[:, 2])
    ang_vel = p1 * torch.sum(torch.square(st.base_ang_vel[:, :2]), dim=1)
    return z_vel + ang_vel


def _smoothing_action(p, st, p0, p1):
    a0, a1, a2 = st.history[..., 0], st.history[..., 1], st.history[..., 2]
    first = torch.sum(torch.square(a1 - a0), dim=1)
    second = torch.sum(torch.square(a2 - 2 * a1 + a0), dim=1)
    return p0 * (first + second)


def _leg_collision(p, st, p0, p1):
    cf = st.contact_state.view(p.n, -1, 3)
    leg_idx = torch.tensor(p.leg_indices, dtype=torch.long)
    leg_touch = (torch.norm(cf[:, leg_idx, :], dim=-1) > p1)
    return p0 * torch.sum(leg_touch.to(torch.float), dim=1)


def _torques_penalize(p, st, p0, p1):
    return p0 * torch.sum(torch.square(st.torques), dim=1)


def _lin_vel_z(p, st, p0, p1):
    return p0 * torch.square(st.base_lin_vel[:, 2])


def _ang_vel_xy(p, st, p0, p1):
    return p0 * torch.sum(torch.square(st.base_ang_vel[:, :2]), dim=1)


def _orientation(p, st, p0, p1):
    return p0 * torch.sum(torch.square(st.projected_gravity[:, :2]), dim=1)


def _dof_vel(p, st, p0, p1):
    return p0 * torch.sum(torch.square(st.dof_state.view(p.n, p.n_dof, 2)[..., 1]), dim=1)


def _action_rate(p, st, p0, p1):
    # actions_recorder.get_last(0): the history is pushed after the reward, so slot 0 is a_{t-1}
    return p0 * torch.sum(torch.square(st.history[..., 0] - st.actions), dim=1)


def _base_height(p, st, p0, p1):
    return p0 * torch.square(st.root_state[:, 2] - p1)


def _dof_pos_limits(p, st, p0, p1):
    dof_pos = st.dof_state.view(p.n, p.n_dof, 2)[..., 0]
    out_of_limits = -(dof_pos - p.dof_pos_limits[:, 0]).clip(max=0.)
    out_of_limits += (dof_pos - p.dof_pos_limits[:, 1]).clip(min=0.)
    return p0 * torch.sum(out_of_limits, dim=1)


def _feet_air_time(p, st, p0, p1):
    """legged_gym _reward_feet_air_time on st.swing_time / st.last_contacts."""
    cf = st.contact_state.view(p.n, -1, 3)
    contact = cf[:, list(p.feet_bodies), 2] > p.feet_contact_force
    contact_filt = torch.logical_or(contact, st.last_contacts)
    st.last_contacts[:] = contact
    first_contact = (st.swing_time > 0.) * contact_filt
    st.swing_time += p.air_time_dt
    rew = torch.sum((st.swing_time - p1) * first_contact, dim=1)
    rew *= torch.norm(st.command[:, :2], dim=1) > p.air_time_cmd_min
    st.swing_time *= ~contact_filt
    return p0 * rew


_A1_TERMS = {"tracking_lin_vel": _tracking_lin_vel, "tracking_ang_vel": _tracking_ang_vel,
             "stabilizing_base": _stabilizing_base, "smoothing_action": _smoothing_action,
             "leg_collision": _leg_collision, "torques_penalize": _torques_penalize, "lin_vel_z": _lin_vel_z,
             "ang_vel_xy": _ang_vel_xy, "orientation": _orientation, "dof_vel": _dof_vel,
             "action_rate": _action_rate, "base_height": _base_height, "dof_pos_limits": _dof_pos_limits,
             "feet_air_time": _feet_air_time}


def a1_compute_reward(p: A1Params, st: A1State):
    """ShifuVecEnv.compute_reward — shifu/gym/env.py:180-185."""
    st.rew[:] = 0.
    for name, rew in a1_reward_terms(p, st).items():
        st.ep_sums[name] += rew
        st.rew[:] += rew


def _u(p: A1Params, env_ids, step, stream, lanes):
    gids = env_ids.numpy().astype(np.int64) + p.env_offset
    u = px.u01_f32(px.draw_u32(p.rng_seed, gids, step, stream)[lanes]).T
    return torch.from_numpy(np.ascontiguousarray(u))


def a1_update_terrain_curriculum(p: A1Params, st: A1State, env_ids, step):
    """a1_conditional.py:204-221 + TerrainGymEnv.update_terrain_level isaac_gym.py:387-391 (row a9)."""
    base_pose = st.root_state[:, :7]
    distance = torch.norm(base_pose[env_ids, :2] - st.env_origins[env_ids, :2], dim=1)
    move_up = distance > p.env_length / 2
    move_down = (distance < torch.norm(st.command[env_ids, :2], dim=1) * p.max_episode_length_s * 0.5) * ~move_up
    st.terrain_levels[env_ids] += 1 * move_up - 1 * move_down
    gids = env_ids.numpy().astype(np.int64) + p.env_offset
    rnd = torch.from_numpy(px.randint10(px.draw_u32(p.rng_seed, gids, step, px.STREAM_LEVEL)[0],
                                        p.max_terrain_level))
    st.terrain_levels[env_ids] = torch.where(st.terrain_levels[env_ids] >= p.max_terrain_level, rnd,
                                             torch.clip(st.terrain_levels[env_ids], 0))
    st.env_origins[env_ids] = st.terrain_origins[st.terrain_levels[env_ids], st.terrain_types[env_ids]]


def a1_reset_idx(p: A1Params, st: A1State, env_ids):
    """A1Conditional.reset_idx — a1_conditional.py:116-120 and everything below it (rows a9-a11)."""
    step = st.step_counter
    if p.curriculum:
        a1_update_terrain_curriculum(p, st, env_ids, step)
    if len(env_ids) == 0:                                   # shifu/gym/env.py:115-116
        return
    # --- IsaacGymEnv.reset_idx -> A1Robot.reset_idx (isaac_gym.py:54-73, robot.py:25-27) ---
    dof = st.dof_state.view(p.n, p.n_dof, 2)
    st.dof_targets[env_ids] = p.q0.clone()                  # robot.py:75-77
    dof[..., 0][env_ids] = p.q0.clone()
    dof[..., 1][env_ids] = 0.
    st.root_state[env_ids, :3] = p.default_base_pose[:3] + st.env_origins[env_ids]   # a1_conditional.py:45
    rand_xy = (1 - -1) * _u(p, env_ids, step, px.STREAM_XY, slice(0, 2)) + -1          # :47
    st.root_state[env_ids, :2] += rand_xy
    st.root_state[env_ids, 3:7] = p.default_base_pose[3:7]
    st.root_state[env_ids, 7:] = 0.
    max_force = 5.
    st.rand_force[env_ids, p.base_index] = (max_force - -max_force) * _u(p, env_ids, step, px.STREAM_FORCE,
                                                                           slice(0, 3)) + -max_force  # :82-87
    # --- ShifuVecEnv.reset_idx (env.py:119-130) ---
    st.ep_len[env_ids] = 0
    st.reset[env_ids] = 1
    st.history.index_fill_(0, env_ids, 0.)                  # shifu/utils/train.py:16-17
    if p.air_time_reset:                                    # legged_gym reset_idx: feet_air_time[env_ids] = 0
        st.swing_time[env_ids] = 0.
        st.last_contacts[env_ids] = False
    st.extras["episode"] = {}
    # un-normalised sums of this reset (what a sharded run all-reduces, SURVEY.md §8e)
    st.extras["_stats"] = {"sums": [float(st.ep_sums[k][env_ids].double().sum()) for k in st.ep_sums],
                           "n_reset": int(len(env_ids)), "level_sum": int(st.terrain_levels.sum()), "n_envs": p.n}
    for key in st.ep_sums.keys():                           # log_info env.py:149-153
        st.extras["episode"][key] = torch.mean(st.ep_sums[key][env_ids]) / p.max_episode_length_s
        st.ep_sums[key][env_ids] = 0.
    st.extras["episode"]["terrain_levels"] = torch.mean(st.terrain_levels.to(torch.float))  # :126-129
    st.extras["time_outs"] = st.time_out
    # --- sample_command (a1_conditional.py:194-200) ---
    for j in range(3):
        st.command[env_ids, j] = ((1. - -1.) * _u(p, env_ids, step, px.STREAM_CMD, slice(j, j + 1)) + -1.).squeeze(1)


def a1_compute_observations(p: A1Params, st: A1State):
    """a1_conditional.py:131-144 (row a12) + HistoryRecorder.flatten train.py:33-35."""
    dof = st.dof_state.view(p.n, p.n_dof, 2)
    heights = torch.clip(st.root_state[:, 2].unsqueeze(1) - 0.5 - st.measured_heights, -1, 1.)
    hist_flat = st.history.permute(0, 2, 1).reshape(p.n, p.n_dof * p.n_hist)
    st.obs = torch.cat([st.command, st.base_lin_vel, st.base_ang_vel, st.gravity_vec,
                        dof[..., 0] - p.q0, dof[..., 1], hist_flat, heights], dim=1)


def a1_history_add(st: A1State, x):
    """HistoryRecorder.add — shifu/utils/train.py:12-14 (row a13)."""
    st.history[..., 1:] = st.history[..., :-1].clone()
    st.history[..., 0] = x


def a1_step(p: A1Params, st: A1State, raw_actions, snap, height_points=None):
    """One control step, in the reference's exact order (SURVEY.md §3.2).

    ``snap`` provides what the simulator would write: ``snap.dof (5,N,12,2)``,
    ``snap.root_offset (N,13)`` (xyz relative to ``env_origins``), ``snap.contact (N,17,3)``.
    """
    if height_points is None:
        height_points = p.height_points()
    scaled = raw_actions * p.action_scale                               # a1_conditional.py:123
    st.actions = torch.clip(scaled, -p.clip_actions, p.clip_actions)    # env.py:87
    dofv = st.dof_state.view(p.n, p.n_dof, 2)
    for i in range(p.decimation):                                       # a1_conditional.py:65-72
        st.torques = a1_pd_torque(p, st.actions, st.dof_state)
        dofv.copy_(snap.dof[i])                                         # gym.simulate + refresh_dof_state
    lin, ang, pg, g = body_frame(st.root_state)                         # :73  (S_prev root, D7)
    st.gravity_vec[:] = g
    st.base_lin_vel[:] = lin
    st.base_ang_vel[:] = ang
    st.projected_gravity[:] = pg
    # refresh_state (isaac_gym.py:139-154): S_new
    root = snap.root_offset.clone()
    root[:, 0:3] += st.env_origins
    st.root_state.copy_(root)
    dofv.copy_(snap.dof[4])
    st.contact_state.view(p.n, -1, 3).copy_(snap.contact)
    st.measured_heights, st.height_idx = get_heights(p, st.root_state[:, :7], st.height_samples,
                                                     height_points, return_idx=True)   # isaac_gym.py:320-322
    # post_step (env.py:93-106)
    st.ep_len += 1
    st.step_counter += 1
    a1_compute_termination(p, st)
    a1_compute_reward(p, st)
    st.reset_ids = st.reset.nonzero(as_tuple=False).flatten()           # env.py:101 (row a8)
    a1_reset_idx(p, st, st.reset_ids)
    a1_compute_observations(p, st)
    a1_history_add(st, st.actions)
    st.obs = torch.clip(st.obs, -p.clip_obs, p.clip_obs)                # env.py:90 (row a14)
    return st.obs, st.rew, st.reset, st.extras


def a1_reset(p: A1Params, st: A1State, snap, height_points=None):
    """ShifuVecEnv.reset — env.py:108-112."""
    a1_reset_idx(p, st, torch.arange(p.n))
    return a1_step(p, st, torch.zeros(p.n, p.n_dof), snap, height_points)


# ---------------------------------------------------------------------------
# ABB push-box prior stage (row a16)
# ---------------------------------------------------------------------------

ABB_REWARD_TERMS = ["reward_reaching", "reward_success"]     # a_prior_stage.py:112-116


@dataclass
class AbbParams:
    n: int
    min_ee_pos: torch.Tensor = None          # abb task_config.py:63
    max_ee_pos: torch.Tensor = None          # abb task_config.py:64
    max_episode_length: float = 200.0        # ceil(20 / (0.02*5))
    max_episode_length_s: float = 20.
    clip_obs: float = 10.
    clip_actions: float = 1.
    q0: torch.Tensor = None                  # task_config.py:56
    ee_index: int = 6
    n_actors: int = 4
    n_bodies: int = 10
    n_dof: int = 6
    robot_pose: torch.Tensor = None
    table_pose: torch.Tensor = None
    cube_z: float = 0.125                    # a_prior_stage.py:31-32
    goal_z: float = 0.1                      # task_config.py:38 via GoalBox a_prior_stage.py:57-58
    rng_seed: int = 0x5EED
    env_offset: int = 0

    def __post_init__(self):
        f = lambda x: torch.tensor(x, dtype=torch.float)
        if self.min_ee_pos is None:
            self.min_ee_pos = f([-0.2, -0.2, 0.11])
        if self.max_ee_pos is None:
            self.max_ee_pos = f([0.2, 0.2, 0.14])
        if self.q0 is None:
            self.q0 = f([0., 0.6437, 0.1748, 0., 0.7541, 0.])
        if self.robot_pose is None:
            self.robot_pose = f([-0.48, 0, 0, 0, 0, 0, 1])
        if self.table_pose is None:
            self.table_pose = f([0, 0, 0.05, 0, 0, 0, 1])


@dataclass
class AbbState:
    root_state: torch.Tensor     # (4N,13): robot, table, cube, goal per env
    body_state: torch.Tensor     # (10N,13)
    dof_state: torch.Tensor      # (6N,2)
    ep_len: torch.Tensor
    ep_sums: Dict[str, torch.Tensor]
    dof_targets: torch.Tensor
    step_counter: int = 0
    extras: Dict = field(default_factory=dict)
    obs: torch.Tensor = None
    rew: torch.Tensor = None
    reset: torch.Tensor = None
    time_out: torch.Tensor = None
    success: torch.Tensor = None
    reset_ids: torch.Tensor = None


def abb_new_state(p: AbbParams) -> AbbState:
    n = p.n
    root = torch.zeros(n * p.n_actors, 13)
    root[:, 6] = 1
    body = torch.zeros(n * p.n_bodies, 13)
    body[:, 6] = 1
    return AbbState(root_state=root, body_state=body, dof_state=torch.zeros(n * p.n_dof, 2),
                    ep_len=torch.zeros(n, dtype=torch.long),
                    ep_sums={k: torch.zeros(n) for k in ABB_REWARD_TERMS},
                    dof_targets=torch.zeros(n, p.n_dof), rew=torch.zeros(n), obs=torch.zeros(n, 6),
                    reset=torch.ones(n, dtype=torch.long), time_out=torch.zeros(n, dtype=torch.bool))


def _abb_views(p: AbbParams, st: AbbState):
    root = st.root_state.view(p.n, p.n_actors, 13)
    cube_idx = torch.arange(p.n) * p.n_actors + 2
    goal_idx = torch.arange(p.n) * p.n_actors + 3
    cube_pose = st.root_state[cube_idx, :7]                       # Actor.base_pose units.py:136-138
    goal_pose = st.root_state[goal_idx, :7]
    ee_pose = st.body_state.view(p.n, -1, 13)[:, :7].view(p.n, 7, -1)[:, [p.ee_index], :7]  # robot.py:138-146
    return root, cube_pose, goal_pose, ee_pose


def abb_is_success(p, st):
    """a_prior_stage.py:129-131"""
    _, cube, goal, _ = _abb_views(p, st)
    d = torch.linalg.norm(goal[:, :2] - cube[:, :2], axis=1)
    return (d < 0.02).to(torch.long)


def abb_compute_termination(p: AbbParams, st: AbbState):
    """a_prior_stage.py:102-110"""
    _, cube, goal, ee = _abb_views(p, st)
    st.time_out = st.ep_len > p.max_episode_length
    st.success = abb_is_success(p, st).to(torch.bool)
    obj_outbound = (torch.any(cube[:, :2] < p.min_ee_pos[:2], dim=1) |
                    torch.any(cube[:, :2] > p.max_ee_pos[:2], dim=1))
    ee_outbound = (torch.any(ee[:, 0, :2] < p.min_ee_pos[:2], dim=1) |
                   torch.any(ee[:, 0, :2] > p.max_ee_pos[:2], dim=1))
    st.reset = st.time_out | (obj_outbound | ee_outbound) | st.success


def abb_reward_terms(p: AbbParams, st: AbbState):
    """a_prior_stage.py:118-127"""
    _, cube, goal, ee = _abb_views(p, st)
    curr_dist = torch.linalg.norm(goal[:, :2] - cube[:, :2], axis=1)
    ee_obj_dist = torch.linalg.norm(ee[:, 0, :2] - cube[:, :2], axis=1)
    in_ws = (ee_obj_dist < 0.1).to(torch.long)
    reach = in_ws * torch.exp(-torch.square(curr_dist) / 0.05)
    succ = abb_is_success(p, st).to(torch.float) * 200
    return {"reward_reaching": reach, "reward_success": succ}


def _abb_box_reset(p: AbbParams, st: AbbState, env_ids, actor, z, step, s_pos, s_eul):
    """RandPosBox._reset_root_state — a_prior_stage.py:39-51 (numpy float64 draws, then fp32)."""
    gids = env_ids.numpy().astype(np.int64) + p.env_offset
    low = np.array([-0.1, -0.1, z])
    high = np.array([0.1, 0.1, z])
    u = px.u01_f64(px.draw_u32(p.rng_seed, gids, step, s_pos)[:3]).T
    rand_pos = torch.tensor(low + (high - low) * u, dtype=torch.float)
    elow = np.array([0, 0, -np.pi])
    ehigh = np.array([0, 0, np.pi])
    ue = px.u01_f64(px.draw_u32(p.rng_seed, gids, step, s_eul)[:3]).T
    rand_euler = torch.tensor(elow + (ehigh - elow) * ue, dtype=torch.float)
    rand_quat = quat_from_euler_xyz(rand_euler[:, 0], rand_euler[:, 1], rand_euler[:, 2])
    idx = env_ids * p.n_actors + actor
    st.root_state[idx, :3] = rand_pos
    st.root_state[idx, 3:7] = rand_quat
    st.root_state[idx, 7:13] = 0.


def abb_reset_idx(p: AbbParams, st: AbbState, env_ids):
    """ShifuVecEnv.reset_idx (env.py:114-130) for the 4-actor ABB scene."""
    if len(env_ids) == 0:
        return
    step = st.step_counter
    dof = st.dof_state.view(p.n, p.n_dof, 2)
    st.dof_targets[env_ids] = p.q0.clone()
    dof[..., 0][env_ids] = p.q0.clone()
    dof[..., 1][env_ids] = 0.
    for actor, pose in ((0, p.robot_pose), (1, p.table_pose)):     # Actor._reset_root_state units.py:130-134
        idx = env_ids * p.n_actors + actor
        st.root_state[idx, :3] = pose[:3]                          # env_origins are zero on the plane
        st.root_state[idx, 3:7] = pose[3:7]
        st.root_state[idx, 7:] = 0.
    _abb_box_reset(p, st, env_ids, 2, p.cube_z, step, px.STREAM_CUBE_POS, px.STREAM_CUBE_EUL)
    _abb_box_reset(p, st, env_ids, 3, p.goal_z, step, px.STREAM_GOAL_POS, px.STREAM_GOAL_EUL)
    st.ep_len[env_ids] = 0
    st.reset[env_ids] = 1
    st.extras["episode"] = {}
    for key in st.ep_sums:
        st.extras["episode"][key] = torch.mean(st.ep_sums[key][env_ids]) / p.max_episode_length_s
        st.ep_sums[key][env_ids] = 0.
    st.extras["episode"]["success_rate"] = torch.mean(st.success.to(torch.float)[env_ids])  # :92-93
    st.extras["time_outs"] = st.time_out


def abb_post_physics(p: AbbParams, st: AbbState):
    """post_step (env.py:93-106) + obs clip (env.py:90) for AbbPushBox."""
    st.ep_len += 1
    st.step_counter += 1
    abb_compute_termination(p, st)
    st.rew[:] = 0.
    for name, rew in abb_reward_terms(p, st).items():
        st.ep_sums[name] += rew
        st.rew[:] += rew
    st.reset_ids = st.reset.nonzero(as_tuple=False).flatten()
    abb_reset_idx(p, st, st.reset_ids)
    _, cube, goal, ee = _abb_views(p, st)
    st.obs = torch.cat([cube[:, :2], goal[:, :2], ee[:, 0, :2]], dim=1)     # a_prior_stage.py:95-100
    st.obs = torch.clip(st.obs, -p.clip_obs, p.clip_obs)
    return st.obs, st.rew, st.reset, st.extras


def abb_step(p: AbbParams, st: AbbState, snap):
    """Simulator refresh (S_new) then the post-physics path.  The pre-physics IK/action path
    (AbbRobot.step, a_prior_stage.py:67-73) is row N2 — not part of this oracle."""
    st.root_state.view(p.n, p.n_actors, 13).copy_(snap.root)
    st.body_state.view(p.n, p.n_bodies, 13).copy_(snap.body)
    st.dof_state.view(p.n, p.n_dof, 2).copy_(snap.dof)
    return abb_post_physics(p, st)


# ==============================================================================================
# Row N2 (SURVEY.md 8f): the arm's pre-physics action path
# ==============================================================================================
def quat_mul(a, b):
    """shifu/utils/torch_utils.py:12-31 (== isaacgym.torch_utils.quat_mul), xyzw."""
    x1, y1, z1, w1 = a[:, 0], a[:, 1], a[:, 2], a[:, 3]
    x2, y2, z2, w2 = b[:, 0], b[:, 1], b[:, 2], b[:, 3]
    ww = (z1 + x1) * (x2 + y2)
    yy = (w1 - y1) * (w2 + z2)
    zz = (w1 + y1) * (w2 - z2)
    xx = ww + yy + zz
    qq = 0.5 * (xx + (z1 - x1) * (x2 - y2))
    w = qq - ww + (z1 - y1) * (y2 - z2)
    x = qq - xx + (x1 + w1) * (x2 + w2)
    y = qq - yy + (w1 - x1) * (y2 + z2)
    z = qq - zz + (z1 + y1) * (w2 - x2)
    return torch.stack([x, y, z, w], dim=-1)


def quat_conjugate(a):
    """shifu/utils/torch_utils.py:34-38."""
    return torch.cat((-a[:, :3], a[:, -1:]), dim=-1)


def arm_goal_from_actions(ee_pos, actions, ee_velocity, dt, min_ee_pos, max_ee_pos, tar_quat):
    """AbbRobot.step, examples/abb_pushbox_vision/a_prior_stage.py:67-71."""
    tar_pos = ee_pos + actions * ee_velocity * dt
    tar_pos = torch.clip(tar_pos, torch.as_tensor(min_ee_pos, dtype=ee_pos.dtype),
                         torch.as_tensor(max_ee_pos, dtype=ee_pos.dtype))
    quat = torch.as_tensor(tar_quat, dtype=ee_pos.dtype).repeat((ee_pos.shape[0], 1))
    return torch.cat([tar_pos, quat], dim=1)


def arm_ik(dof_pos, ee_pose, j_ee, goal_pose, damping=0.05):
    """ArmRobot.inverse_kinematics, shifu/units/robot.py:156-182 (the stand-alone
    shifu/utils/torch_utils.py:41-58 is the same math).  Works in the dtype of its inputs: float32
    reproduces the reference, float64 is the yardstick the CUDA test measures both against."""
    pos_err = goal_pose[:, :3] - ee_pose[:, :3]
    q_r = quat_mul(goal_pose[:, 3:7], quat_conjugate(ee_pose[:, 3:7]))
    orn_err = q_r[:, 0:3] * torch.sign(q_r[:, 3]).unsqueeze(-1)
    dpose = torch.cat([pos_err, orn_err], -1).unsqueeze(-1)
    j_t = torch.transpose(j_ee, 1, 2)
    lmbda = torch.eye(6, dtype=j_ee.dtype) * (damping ** 2)
    u = (j_t @ torch.inverse(j_ee @ j_t + lmbda) @ dpose).view(dof_pos.shape[0], dof_pos.shape[1])
    return dof_pos + u


# ==============================================================================================
# Row N4 (SURVEY.md 8f): CameraSensor.refresh_image_tensors
# ==============================================================================================
def camera_refresh(color=None, depth=None, seg=None, flow=None, image_normalization=False):
    """shifu/units/sensors.py:165-188 with normalize_color of shifu/utils/image.py:12-15.  Each
    argument is the list of per-env image tensors Isaac Gym hands out; returns the batched buffers."""
    out = {}
    if color is not None:
        rows = [(c[..., :3].to(torch.float32) / 255) if image_normalization else c for c in color]
        out["color"] = torch.stack(rows)
    if depth is not None:
        out["depth"] = torch.stack([-d for d in depth])            # "Isaac gives negative depth map !"
    if seg is not None:
        out["seg"] = torch.stack(list(seg))
    if flow is not None:
        out["flow"] = torch.stack(list(flow))
    return out
