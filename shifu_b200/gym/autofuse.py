"""Automatic fusion of UNMODIFIED reference task classes (``examples/a1_conditional``,
``examples/abb_pushbox_vision/a_prior_stage``) and of user tasks shaped like them.

``ShifuVecEnv`` subclasses describe their task with Python hooks (README.md:95-128).  On the first
``reset()`` / ``step()`` the base class asks this module whether the hooks are — provably — what one
of the fused kernels computes.  The proof has three parts, none of which reads source text:

* **structure**: config shapes (obs width, measured-point grid, history depth, dof / body counts),
  affine actor layout, and for the hooks the kernel replaces without a numerical check (reset
  sampling, curriculum, the PD loop — they are stochastic or call the simulator) the set of
  attribute names and literals their code objects reference (``co_names`` / ``co_consts``;
  stable across Python versions, unlike bytecode);
* **term compilation** (``shifu_b200.terms``): reward hooks -> (opcode, constants) and the observation
  hook -> its layout (slot sources, column scales, height scale), by probing;
* **numerical check**: reward hooks against ``shifu_a1_eval_terms``; observation and termination
  hooks against the layout / predicates the kernel implements, on a seeded random state.

Anything that fails leaves the env in user-hook mode (eager torch hooks on CUDA tensors, with the
base-class rows still done by kernels) and records the reason in ``env.fusion_report``.

The task classes of ``shifu_b200.tasks`` fuse explicitly, without the proof, through the same
pieces: the descriptor builders (``a1_env_desc``, ``abb_hot_path``), the bindings (``bind_a1``,
``bind_abb``) and ``install``, which routes ``step`` / ``reset_idx`` to the fused kernels.
"""
from __future__ import annotations

from typing import Callable, Dict, Iterable, Optional

import torch

from shifu_b200 import hotpath, terms
from shifu_b200 import _native as nv


NotFusable = terms.NotFusable


def _code(fn):
    fn = getattr(fn, "__func__", fn)
    code = getattr(fn, "__code__", None)
    if code is None:
        raise NotFusable(f"{fn!r} is not a Python function")
    return code


def _names(fn) -> set:
    code = _code(fn)
    out = set(code.co_names)
    for c in code.co_consts:                      # nested lambdas / comprehensions
        if hasattr(c, "co_names"):
            out |= set(c.co_names)
    return out


def _numbers(fn) -> set:
    return {float(c) for c in _code(fn).co_consts if isinstance(c, (int, float)) and not isinstance(c, bool)}


def _require(fn, what: str, names: Iterable[str] = (), numbers: Iterable[float] = ()):
    missing = set(names) - _names(fn)
    if missing:
        raise NotFusable(f"{what}: does not reference {sorted(missing)} — not the hook the fused kernel replaces")
    nums = _numbers(fn)
    for v in numbers:
        if not any(abs(v - c) <= 1e-12 * max(1.0, abs(v)) for c in nums):
            raise NotFusable(f"{what}: literal {v} not found (found {sorted(nums)})")


_AIR_STATE = {"swing_time", "feet_air_time", "last_contacts"}


def _require_reset_idx(cls) -> bool:
    """The class's reset_idx must be the reference's (a1_conditional.py:89-98), possibly under overrides
    that only call ``super().reset_idx`` and clear the feet-air-time state (legged_gym's reset_idx does;
    the kernel's reset then clears it too).  Returns whether the state is cleared on reset."""
    clears = False
    for klass in cls.__mro__:
        fn = klass.__dict__.get("reset_idx")
        if fn is None:
            continue
        names = _names(fn)
        if {"update_terrain_curriculum", "sample_command"} <= names:
            return clears or bool(names & _AIR_STATE)
        other = names - _AIR_STATE - {"super", "reset_idx"}
        if other or not (names & _AIR_STATE):
            raise NotFusable(f"reset_idx: {klass.__name__}.reset_idx also touches {sorted(other)} — not a hook the "
                             "fused kernel replaces")
        clears = True
    raise NotFusable("reset_idx: does not reference ['sample_command', 'update_terrain_curriculum'] — not the hook "
                     "the fused kernel replaces")


def _overridden(obj, name: str, base) -> bool:
    return getattr(type(obj), name, None) is not getattr(base, name, None)


_close = terms.check_close


# =============================================================================================
# A1 conditional walking (examples/a1_conditional/a1_conditional.py)
# =============================================================================================

def fuse_a1(env, carry_body_frame: bool = True, rng_seed: int = 0x5EED):
    """Returns an ``A1HotPath`` bound to the env's tensors, or raises NotFusable / TermMismatch."""
    from shifu_b200.gym.sim_facade import TerrainGymEnv
    from shifu_b200.gym.vec_env import ShifuVecEnv
    from shifu_b200.units import LeggedRobot
    isg, cfg = env.isg_env, env.cfg
    rb = getattr(env, "robot", None)
    # ---- structure ---------------------------------------------------------------------------
    if not isinstance(isg, TerrainGymEnv) or not isinstance(rb, LeggedRobot):
        raise NotFusable("needs a TerrainGymEnv with a LeggedRobot")
    tc = cfg.terrain
    # the observation width picks the step: 72 + 187 scans the terrain, 72 is blind (no height columns)
    num_obs = cfg.num_obs
    if num_obs not in (nv.OBS_HEAD, nv.OBS_HEAD + nv.MAX_PX * nv.MAX_PY) or cfg.num_privileged_obs is not None:
        raise NotFusable("observation width is not 72 + 187 or 72")
    blind = num_obs == nv.OBS_HEAD
    if not blind and ((len(tc.measured_points_x), len(tc.measured_points_y)) != (nv.MAX_PX, nv.MAX_PY)
                      or not tc.measure_heights):
        raise NotFusable("the fused kernel is compiled for the 17x11 measured-point grid")
    store_heights = bool(getattr(cfg, "store_measured_heights", False))
    if blind and store_heights:
        raise NotFusable("store_measured_heights with a 72-column observation: the fused blind step does not scan "
                         "the terrain")
    if (rb.num_dof, rb.num_bodies, cfg.num_actions, cfg.num_actions_history) != (12, 17, 12, 3):
        raise NotFusable("the fused kernel is compiled for 12 dofs / 17 bodies / 3 past actions")
    layout = rb.affine_root_layout()
    if layout is None:
        raise NotFusable("non-affine root_indices")
    for attr in ("command_buf", "terrain_levels", "contact_terminate_indices", "cmd_lin_vel_x", "cmd_lin_vel_y",
                 "cmd_ang_vel_yaw"):
        if not hasattr(env, attr):
            raise NotFusable(f"env.{attr} is missing")
    for attr in ("torques", "rand_force_buf", "leg_indices", "p_gains", "d_gains"):
        if not hasattr(rb, attr):
            raise NotFusable(f"robot.{attr} is missing")
    # ---- hooks replaced without a numerical check: reference structure by names / literals -----
    air_time_reset = _require_reset_idx(type(env))
    _require(type(env).sample_command, "sample_command",
             ("torch_rand_float", "cmd_lin_vel_x", "cmd_lin_vel_y", "cmd_ang_vel_yaw", "command_buf"))
    _require(type(env).update_terrain_curriculum, "update_terrain_curriculum",
             ("init_done", "norm", "base_pose", "env_origins", "env_length", "command_buf", "max_episode_length_s",
              "terrain_levels", "randint_like", "max_terrain_level", "where", "clip", "update_terrain_level"),
             (2, 0.5, 1, 0))
    if _overridden(env, "step", ShifuVecEnv):
        _require(type(env).step, "step", ("step",))
        scales = [c for c in _numbers(type(env).step) if c not in (0.0,)]
        if len(scales) != 1:
            raise NotFusable(f"step: expected exactly one action-scale literal, found {scales}")
    if _overridden(env, "episode_log", ShifuVecEnv):
        _require(type(env).episode_log, "episode_log", ("terrain_levels", "mean"))
    _require(type(rb).step, "robot.step",
             ("decimation", "p_gains", "default_dof_pos", "dof_pos", "d_gains", "dof_vel", "clip", "torque_limits",
              "_internal_motor_step", "simulate", "refresh_dof_state_tensor", "post_step", "apply_force_on_base",
              "rand_force_buf"))
    _require(type(rb)._reset_root_state, "robot._reset_root_state",
             ("root_indices", "root_state", "default_base_pose", "env_origins", "torch_rand_float"), (-1, 1, 2, 3, 7))
    force_fn = getattr(type(rb), "update_rand_force_buf", None) or type(rb).reset_idx
    _require(force_fn, "robot.update_rand_force_buf", ("rigid_body_dict", "rand_force_buf", "torch_rand_float"))
    forces = [c for c in _numbers(force_fn) if c > 0 and c != 3.0]
    if len(forces) != 1:
        raise NotFusable(f"robot.update_rand_force_buf: expected one force literal, found {forces}")
    base_name = [c for c in _code(force_fn).co_consts if isinstance(c, str)]
    force_body = rb.rigid_body_dict[base_name[0]] if base_name and base_name[0] in rb.rigid_body_dict else 0
    # ---- reward terms: match + fit ------------------------------------------------------------
    compiled = terms.compile_a1_terms(env, env.reward_functions)
    names = [t.name for t in compiled]
    # ---- observation: slot sources, scales and noise scales ------------------------------------
    # (read once, here, like every fitted constant: a noise curriculum that changes noise_scale_vec
    # later does not reach the kernel)
    obs = terms.compile_a1_obs(env, num_obs)
    # ---- the hot path over the env's own tensors -----------------------------------------------
    desc = a1_env_desc(env, [(t.name, t.code, t.p0, t.p1) for t in compiled], rng_seed=rng_seed, obs=obs,
                       action_scale=1.0,         # a subclass step() has already scaled (a1_conditional.py:122-124)
                       force_body=force_body, push_force_max=float(forces[0]), air_time_reset=air_time_reset,
                       num_obs=num_obs, **terms.desc_extras(compiled))
    hp = a1_hot_path(env, desc, names, carry_body_frame, store_heights)
    # the probes below run the user's hooks on the env's CURRENT tensors: point the hot path at them
    hp.adopt(actions=env.actions, history=env.actions_recorder.history_buf, command=env.command_buf,
             torques=rb.torques, base_lin_vel=rb.base_lin_vel, base_ang_vel=rb.base_ang_vel,
             projected_gravity=rb.projected_gravity, ep_len=env.episode_length_buf, rand_force=rb.rand_force_buf,
             dof_targets=rb.dof_targets, terrain_levels=env.terrain_levels)
    air = terms.air_time_state(env)
    if air is not None and any(t.code == nv.REW_FEET_AIR_TIME for t in compiled):
        hp.adopt(swing_time=air[0], last_contacts=air[1])
    # ---- numerical checks ----------------------------------------------------------------------
    terms.verify_a1_terms(env, hp, env.reward_functions, compiled)
    terms.verify_a1_obs(env, obs, num_obs=num_obs)
    _check_a1_termination(env)
    return hp


def _check_a1_termination(env):
    """compute_termination against the kernel's definition (a1_conditional.py:146-150) on a random state."""
    rb, isg = env.robot, env.isg_env
    with terms.A1Probe(env) as pr:
        pr.randomize(4321)
        had = isg.__dict__.get("_measured_heights")
        isg.measured_heights = torch.randn(env.num_envs, isg.num_height_points, device=env.device)
        try:
            env.compute_termination()
            force = rb.contact_forces[:, int(env.contact_terminate_indices), :]
            contact = torch.norm(force, dim=-1) > 1.
            time_out = env.episode_length_buf > env.max_episode_length
            _close(env.time_out_buf, time_out, "compute_termination (time_out_buf)")
            _close(env.reset_buf, time_out | contact, "compute_termination (reset_buf)")
        finally:
            if had is None:
                del isg.measured_heights
            else:
                isg.measured_heights = had


def a1_env_desc(env, terms, *, rng_seed: int, force_body: int, push_force_max: float, **kw) -> nv.A1Desc:
    """``hotpath.a1_desc`` of an A1-shaped env: dof gains and limits from its robot, the point grid and
    terrain scales from its config, curriculum, levels and env length from its gym env, and its episode
    lengths, clips and command ranges.  ``terms`` and ``kw`` (``obs``, ``action_scale``, ``air_time_reset``,
    the compiled terms' extras) go to ``a1_desc`` as they are; ``num_obs`` defaults to the config's.  A blind
    descriptor (``num_obs = 72``) keeps the compiled 17x11 grid whatever the config's: the blind step does not
    scan, and the on-demand heights come from the gym env's own scan."""
    rb, isg, tc = env.robot, env.isg_env, env.cfg.terrain
    stride, offset = rb.affine_root_layout()
    kw.setdefault("num_obs", env.cfg.num_obs)
    grid = {} if kw["num_obs"] == nv.OBS_HEAD else dict(points_x=tuple(tc.measured_points_x),
                                                         points_y=tuple(tc.measured_points_y))
    desc = hotpath.a1_desc(
        env.num_envs, env_offset=env.env_offset, rng_seed=rng_seed, terms=terms,
        q0=tuple(rb.cfg.default_dof_pos), kp=tuple(float(v) for v in rb.p_gains.tolist()),
        kd=tuple(float(v) for v in rb.d_gains.tolist()), torque_limit=tuple(rb.torque_limits.tolist()),
        **grid, border_size=float(tc.border_size), horizontal_scale=tc.horizontal_scale, vertical_scale=tc.vertical_scale,
        max_episode_length=int(env.max_episode_length), max_episode_length_s=float(env.max_episode_length_s),
        default_root=tuple(rb.cfg.default_pos) + tuple(rb.cfg.default_quat), curriculum=tc.curriculum,
        max_terrain_level=isg.max_terrain_level, num_terrain_types=tc.num_cols, env_length=isg.terrain.env_length,
        base_body=int(env.contact_terminate_indices), leg_bodies=tuple(rb.leg_indices.tolist()),
        force_body=force_body, root_stride=stride, root_offset=offset,
        clip_actions=float(env.clip_actions), clip_obs=float(env.clip_obs), **kw)
    desc.push_force_max = push_force_max
    desc.cmd_low[0], desc.cmd_high[0] = env.cmd_lin_vel_x
    desc.cmd_low[1], desc.cmd_high[1] = env.cmd_lin_vel_y
    desc.cmd_low[2], desc.cmd_high[2] = env.cmd_ang_vel_yaw
    return desc


def a1_hot_path(env, desc: nv.A1Desc, names, carry_body_frame: bool, want_measured_heights: bool) -> hotpath.A1HotPath:
    """An ``A1HotPath`` for ``desc`` over the env's gym tensors (a blind descriptor takes no height map)."""
    isg = env.isg_env
    blind = desc.num_obs == nv.OBS_HEAD
    return hotpath.A1HotPath(desc, root_state=isg.root_state, dof_state=isg.dof_state, contact_state=isg.contact_state,
                             height_samples=None if blind else isg.height_samples, terrain_origins=isg.terrain_origins,
                             terrain_types=isg.terrain_types, env_origins=isg.env_origins, terms=names,
                             carry_body_frame=carry_body_frame, want_measured_heights=want_measured_heights)


def bind_a1(env, hp):
    """Make the env / robot attributes BE the tensors the kernel reads and writes, and derive the
    body-frame velocities the first step reads from the current root rows."""
    rb, isg = env.robot, env.isg_env
    env.actions, env.obs_buf, env.rew_buf, env.reset_buf = hp.actions, hp.obs_buf, hp.rew_buf, hp.reset_buf
    env._episode_length_buf = hp.ep_len
    env.time_out_buf, env.contact_terminate_buf = hp.time_out_buf, hp.contact_terminate_buf
    env.episode_rewards = hp.ep_sums
    env.command_buf, env.terrain_levels = hp.command, hp.terrain_levels
    env.actions_recorder.history_buf = hp.history
    rb.torques, rb.dof_targets, rb.rand_force_buf = hp.torques, hp.dof_targets, hp.rand_force
    rb.base_lin_vel, rb.base_ang_vel = hp.base_lin_vel, hp.base_ang_vel
    rb.projected_gravity, rb.gravity_vec = hp.projected_gravity, hp.gravity_vec
    isg.measured_heights = hp.measured_heights          # None unless cfg.store_measured_heights: filled on demand
    # (a blind task fills it on demand only when it measures heights, like user-hook mode does)
    isg.__dict__["_heights_on_demand"] = hp.measured_heights is None and (not hp.blind or
                                                                          bool(env.cfg.terrain.measure_heights))
    env.extras.update(hp.extras())
    hp.body_frame()


def _resident_state(env) -> bool:
    """True when nothing runs between the kernel launches of a step: the stand-in simulator with no
    snapshot provider (state resident in HBM, refresh calls are no-ops).  A cross-rank collective is
    fine: it runs after the replay, on the side stream."""
    sim = env.isg_env.sim
    return (getattr(sim, "provider", 0) is None and not getattr(env.isg_env.gym, "needs_indexed_resets", True)
            and getattr(env, "use_cuda_graph", True))


def a1_fused_step(env, hp, actions: torch.Tensor):
    """ShifuVecEnv.step (env.py:85-106) with the A1 hooks, as kernel launches around the simulator
    crossings of A1Robot.step / IsaacGymEnv.refresh_state (a1_conditional.py:64-75, isaac_gym.py:139-154).
    On resident state (no simulator between the launches) the whole step is one CUDA-graph replay."""
    gym, sim, rb, isg = env.isg_env.gym, env.isg_env.sim, env.robot, env.isg_env
    actions = actions.contiguous()
    env.common_step_counter += 1
    hp.step_counter = env.common_step_counter - 1
    if _resident_state(env):
        hp.graph_step(actions, isg.decimation, allreduce=env.stats_allreduce)
        env.extras.update(hp.extras())
        return env.obs_buf, env.privileged_obs_buf, env.rew_buf, env.reset_buf, env.extras
    for i in range(isg.decimation):
        hp.pd_torque(actions if i == 0 else None)
        rb._internal_motor_step(rb.torques)
        gym.simulate(sim)
        gym.refresh_dof_state_tensor(sim)
    if not hp.carry_body_frame:
        hp.body_frame()                                                 # S_prev root (SURVEY.md D7)
    rb.apply_force_on_base(rb.rand_force_buf.view(-1, 3))
    isg.refresh_state()
    hp.post_physics()
    hp.finalize(env.stats_allreduce)
    push_resets(env, hp)
    env.extras.update(hp.extras())
    return env.obs_buf, env.privileged_obs_buf, env.rew_buf, env.reset_buf, env.extras


# =============================================================================================
# ABB push-box prior stage (examples/abb_pushbox_vision/a_prior_stage.py)
# =============================================================================================

def fuse_abb(env, rng_seed: int = 0x5EED):
    from shifu_b200.units import ArmRobot, Box
    cfg = env.cfg
    rb = getattr(env, "robot", None)
    if not isinstance(rb, ArmRobot) or not all(isinstance(getattr(env, a, None), Box) for a in ("table", "cube", "goal")):
        raise NotFusable("needs an ArmRobot with table / cube / goal boxes")
    if cfg.num_obs != 6 or cfg.num_actions_history or cfg.num_privileged_obs is not None:
        raise NotFusable("observation is not the 6-column push-box observation")
    actors = [rb, env.table, env.cube, env.goal]
    layouts = [a.affine_root_layout() for a in actors]
    if any(l is None or l[0] != len(actors) for l in layouts):
        raise NotFusable("needs the 4-actor interleaved root layout")
    for box in (env.cube, env.goal):
        _require(type(box)._reset_root_state, f"{type(box).__name__}._reset_root_state",
                 ("root_indices", "uniform", "pos_range", "euler_range", "quat_from_euler_xyz", "root_state"), (3, 7, 13))
        if not (hasattr(box, "pos_range") and hasattr(box, "euler_range")):
            raise NotFusable("boxes without pos_range / euler_range")
    names = [fn.__name__ for fn in env.reward_functions]
    if names != ["reward_reaching", "reward_success"]:
        raise NotFusable(f"reward list {names} is not [reward_reaching, reward_success]")
    return abb_hot_path(env, rng_seed, _fit_abb_terms(env))


def abb_hot_path(env, rng_seed: int, term_params: Dict[str, tuple]) -> hotpath.AbbHotPath:
    """An ``AbbHotPath`` over the env's gym tensors, its descriptor read off the 4-actor scene (layout,
    robot and table poses, end-effector box, cube and goal ranges) with the given reward constants."""
    isg, rb = env.isg_env, env.robot
    actors = [rb, env.table, env.cube, env.goal]
    names = [fn.__name__ for fn in env.reward_functions]
    desc = hotpath.abb_desc(env.num_envs, env_offset=env.env_offset, rng_seed=rng_seed, terms=names,
                            term_params=term_params)
    desc.num_actors = len(actors)
    desc.robot_actor, desc.table_actor, desc.cube_actor, desc.goal_actor = (a.affine_root_layout()[1] for a in actors)
    desc.num_bodies = sum(a.num_bodies for a in actors)
    desc.num_dof, desc.ee_body = rb.num_dof, int(rb.ee_indices[0])
    for i in range(3):
        desc.min_ee_pos[i], desc.max_ee_pos[i] = float(rb.cfg.min_ee_pos[i]), float(rb.cfg.max_ee_pos[i])
        desc.box_pos_low[i], desc.box_pos_high[i] = env.cube.pos_range["low"][i], env.cube.pos_range["high"][i]
    for i, v in enumerate(rb.cfg.default_dof_pos):
        desc.q0[i] = v
    for i, v in enumerate([*rb.cfg.default_pos, *rb.cfg.default_quat]):
        desc.robot_root[i] = v
    for i, v in enumerate([*env.table.cfg.default_pos, *env.table.cfg.default_quat]):
        desc.table_root[i] = v
    desc.goal_z = env.goal.pos_range["low"][2]
    desc.success_distance = term_params["reward_success"][1]
    desc.max_episode_length, desc.max_episode_length_s = int(env.max_episode_length), float(env.max_episode_length_s)
    desc.clip_obs = float(env.clip_obs)
    return hotpath.AbbHotPath(desc, root_state=isg.root_state, body_state=isg.body_state, dof_state=isg.dof_state,
                              terms=names)


def _fit_abb_terms(env) -> Dict[str, tuple]:
    """Constants of reward_reaching / reward_success / is_success by probing the hooks, then a check
    of hooks, observation and termination against the kernel's definition on a random scene."""
    import math
    isg, rb = env.isg_env, env.robot
    n = env.num_envs
    root = isg.root_state.view(n, -1, 13)
    body = isg.body_state.view(n, -1, 13)
    ee = int(rb.ee_indices[0])
    saved = (isg.root_state.clone(), isg.body_state.clone(), env.episode_length_buf.clone())
    attrs = {a: getattr(env, a, None) for a in ("obs_buf", "reset_buf", "time_out_buf", "success_buf")}

    def scene(cube_xy, goal_xy, ee_xy):
        root.zero_(); body.zero_()
        root[0, 2, :2] = torch.tensor(cube_xy, device=env.device)
        root[0, 3, :2] = torch.tensor(goal_xy, device=env.device)
        body[0, ee, :2] = torch.tensor(ee_xy, device=env.device)

    def bisect(f, lo, hi):
        for _ in range(50):
            mid = 0.5 * (lo + hi)
            lo, hi = (mid, hi) if f(mid) else (lo, mid)
        return 0.5 * (lo + hi)

    try:
        scene((0, 0), (0, 0), (0, 0))
        success_rew = float(env.reward_success()[0])                              # distance 0 -> success
        thr = bisect(lambda d: (scene((0, 0), (d, 0), (0, 0)), float(env.reward_success()[0]) != 0.0)[1], 0.0, 1.0)
        thr = terms._snap(thr, type(env).is_success if hasattr(type(env), "is_success") else env.reward_success)
        ws = bisect(lambda d: (scene((0, 0), (0, 0), (d, 0)), float(env.reward_reaching()[0]) != 0.0)[1], 0.0, 1.0)
        ws = terms._snap(ws, env.reward_reaching)
        scene((0, 0), (0.1, 0), (0, 0))
        r = float(env.reward_reaching()[0])                                       # exp(-0.01 / p1)
        if not 0.0 < r < 1.0:
            raise NotFusable("reward_reaching is not [ee near cube] * exp(-d^2 / c)")
        width = terms._snap(-0.01 / math.log(r), env.reward_reaching)
        params = {"reward_reaching": (ws, width), "reward_success": (success_rew, thr)}
        # check on a random scene
        g = torch.Generator(device=env.device).manual_seed(7)
        root.copy_(torch.randn(root.shape, generator=g, device=env.device) * 0.08)
        body.copy_(torch.randn(body.shape, generator=g, device=env.device) * 0.08)
        env.episode_length_buf.copy_(torch.randint(0, int(env.max_episode_length) + 20, (n,), generator=g,
                                                   device=env.device))
        cube, goal, eep = root[:, 2, :2], root[:, 3, :2], body[:, ee, :2]
        dist = torch.linalg.norm(goal - cube, dim=1)
        ee_dist = torch.linalg.norm(eep - cube, dim=1)
        _close(env.reward_reaching(), (ee_dist < ws).float() * torch.exp(-torch.square(dist) / width), "reward_reaching")
        _close(env.reward_success(), (dist < thr).float() * success_rew, "reward_success")
        env.compute_observations()
        _close(env.obs_buf, torch.cat([cube, goal, eep], dim=1), "compute_observations")
        env.compute_termination()
        lo = torch.tensor(rb.cfg.min_ee_pos[:2], device=env.device)
        hi = torch.tensor(rb.cfg.max_ee_pos[:2], device=env.device)
        out = ((cube < lo).any(1) | (cube > hi).any(1) | (eep < lo).any(1) | (eep > hi).any(1))
        time_out = env.episode_length_buf > env.max_episode_length
        _close(env.reset_buf, time_out | out | (dist < thr), "compute_termination")
        return params
    finally:
        isg.root_state.copy_(saved[0]); isg.body_state.copy_(saved[1]); env.episode_length_buf.copy_(saved[2])
        for a, v in attrs.items():
            if v is not None:
                setattr(env, a, v)


def bind_abb(env, hp):
    env.obs_buf, env.rew_buf, env.reset_buf = hp.obs_buf, hp.rew_buf, hp.reset_buf
    env._episode_length_buf, env.time_out_buf, env.success_buf = hp.ep_len, hp.time_out_buf, hp.success_buf
    env.episode_rewards = hp.ep_sums
    hp.dof_targets = env.robot.dof_targets          # written by the robot's own step() (IK kernel)
    hp._io = None
    env.extras.update(hp.extras())


def abb_fused_step(env, hp, actions: torch.Tensor):
    k = env.isg_env.kernels()
    k.clip(actions, env.clip_actions, out=env.actions)                         # env.py:87
    env.isg_env.step(env.actions)                                              # user's robot.step + refresh_state
    env.common_step_counter += 1
    hp.step_counter = env.common_step_counter - 1
    hp.post_physics()
    hp.finalize(env.stats_allreduce)
    push_resets(env, hp)
    env.extras.update(hp.extras())
    return env.obs_buf, env.privileged_obs_buf, env.rew_buf, env.reset_buf, env.extras


# =============================================================================================
# both recipes
# =============================================================================================

def push_resets(env, hp, env_ids: Optional[torch.Tensor] = None):
    """Indexed setters of the simulator for the rows the kernel rewrote (isaac_gym.py:70-73,
    robot.py:78-86): ``env_ids``, or the step's compacted reset ids when None.  They need the id count
    on the host (one sync, like the reference's ``nonzero``); the stand-in simulator has no hidden
    state and skips this."""
    if not getattr(env.isg_env.gym, "needs_indexed_resets", True):
        return
    ids = hp.reset_id_list() if env_ids is None else env_ids
    if len(ids):
        env.robot.push_dof_reset(ids)
        env.isg_env.push_root_reset(ids)


def fused_reset_idx(env, hp, env_ids: Optional[torch.Tensor]):
    """``reset_idx`` of a fused env in one launch (env.py:114-130 with the task's reset hooks);
    ``None`` = all envs.  ``extras`` keeps pointing at the hot path's ring, never a detached dict."""
    hp.step_counter = env.common_step_counter
    hp.reset_idx(env_ids, env.stats_allreduce)
    push_resets(env, hp, torch.arange(env.num_envs, device=env.device) if env_ids is None else env_ids)
    env.extras.update(hp.extras())


RECIPES = {"a1": (fuse_a1, bind_a1, a1_fused_step), "abb": (fuse_abb, bind_abb, abb_fused_step)}


def install(env, recipe: str, hp):
    """Run the env on ``hp``: bind its attributes to the hot path's tensors, and route ``step`` (through
    ``ShifuVecEnv.step``) and ``reset_idx`` (which a subclass may override: it is part of what got
    fused) to the fused kernels."""
    _, bind, step = RECIPES[recipe]
    bind(env, hp)
    env.hot, env._fusion, env._fusion_tried = hp, (recipe, hp, step), True
    env.reset_idx = lambda env_ids: fused_reset_idx(env, hp, env_ids)


def try_fuse(env, **kw):
    """Installs the first recipe whose proof holds; the reasons go to env.fusion_report."""
    report = []
    for name, (fuse, _, _) in RECIPES.items():
        try:
            hp = fuse(env, **{k: v for k, v in kw.items() if k in fuse.__code__.co_varnames})
        except (NotFusable, terms.TermMismatch, KeyError, AttributeError) as exc:
            report.append(f"{name}: {exc}")
            continue
        install(env, name, hp)
        env.fusion_report = f"fused: {name}"
        return
    env.fusion_report = "user-hook mode — " + "; ".join(report)
