"""A1 conditional walking on the shifu_b200 API (the workload of BASELINE configs 1, 2, 3, 5).

Counterpart of ``examples/a1_conditional`` of the reference: same classes (``A1Robot``,
``A1Conditional``), same hooks, same constants (cited).  Two ways to run it:

* ``fused=True`` (default): the reward list is handed to the reward-term registry and
  ``post_step`` is ONE CUDA kernel (``shifu_a1_post_physics``) — PD torques, body-frame
  velocities, height scan, termination, rewards + episode sums, reset with Philox draws,
  observation, history push and clips never go through torch.  The descriptor builder, the
  binding of the env's tensors, the fused step and the ``reset_idx`` dispatch are automatic
  fusion's (``shifu_b200.gym.autofuse``), without its proof: the named terms run the reference
  constants;
* ``fused=False``: the hooks below run as ordinary torch code on the same CUDA tensors through
  ``ShifuVecEnv``'s user-hook orchestration (what an unmodified user subclass gets).  Random
  draws come from the same counter-based Philox streams so the two modes can be compared.
"""
from __future__ import annotations

import typing

import numpy as np
import torch
from isaacgym import gymapi

from shifu_b200.configs import LeggedRobotActorConfig, PPOConfig, TerrainEnvConfig
from shifu_b200.gym import ShifuVecEnv
from shifu_b200.units import LeggedRobot

ASSET_ROOT = "./asset"


class A1ActorConfig(LeggedRobotActorConfig):       # examples/a1_conditional/task_config.py:11-26
    name = "a1_robot"
    root_dir = ASSET_ROOT
    urdf_filename = "urdf/a1/urdf/a1.urdf"
    default_pos = [0, 0, 0.42]
    default_quat = [0, 0, 0, 1.]
    default_dof_pos = [0.1, 0.8, -1.5, 0.1, 0.8, -1.5, -0.1, 0.8, -1.5, -0.1, 0.8, -1.5]
    end_effector_names = ['FR_foot', 'FL_foot', 'RR_foot', 'RL_foot']
    dof_stiffness = [20] * 12
    dof_damping = [.5] * 12

    class asset_options(LeggedRobotActorConfig.asset_options):
        default_dof_drive_mode = gymapi.DOF_MODE_EFFORT


class A1EnvConfig(TerrainEnvConfig):               # task_config.py:29-56
    num_envs = 4000
    num_obs = 259
    num_privileged_obs = None
    num_actions = 12
    num_actions_history = 3
    send_timeouts = True
    episode_length_s = 10.

    class sim(TerrainEnvConfig.sim):
        dt = 0.005

    class control(TerrainEnvConfig.control):
        decimation = 4

    class debug(TerrainEnvConfig.debug):
        headless = True
        camera_pos = [1., -1., 1.]

    class normalization(TerrainEnvConfig.normalization):
        clip_observations = 100.
        clip_actions = 1.
    # NB: the reference spells its terrain override ``terrian`` (task_config.py:52), so the base
    # TerrainEnvConfig.terrain (10x20 tiles, 1300x2100 map) is what actually runs (SURVEY.md D6).


class A1PPOConfig(PPOConfig):
    seed = 42
    runner_class_name = "A1Conditional"

    class runner(PPOConfig.runner):
        num_steps_per_env = 24
        max_iterations = 3000
        save_interval = 100
        experiment_name = 'commands_and_terrain'
        run_name = 'ppo_A1Conditional'


class A1Robot(LeggedRobot):
    def __init__(self, cfg):
        super().__init__(cfg)
        self.p_gains = torch.tensor(self.cfg.dof_stiffness, dtype=torch.float)
        self.d_gains = torch.tensor(self.cfg.dof_damping, dtype=torch.float)

    def random_rigid_shape_props(self, env_ids, rigid_shape_props):
        for prop in rigid_shape_props:
            prop.friction = np.random.uniform(0.5, 1.25)
        return rigid_shape_props

    def init_buffers(self):
        super().init_buffers()
        n, dev = self.env.num_envs, self.device
        self.p_gains, self.d_gains = self.p_gains.to(dev), self.d_gains.to(dev)
        self.torques = torch.zeros(n, self.num_dof, dtype=torch.float, device=dev)
        legs = [i for name, i in self.rigid_body_dict.items() if "thigh" in name or "calf" in name]
        self.leg_indices = torch.tensor(legs, dtype=torch.long, device=dev)
        self.rand_force_buf = torch.zeros(n, self.num_bodies, 3, device=dev)

    # user-hook mode reset (a1_conditional.py:43-50, 77-87) with Philox streams 1 (xy) and 2 (force)
    def _reset_root_state(self, env_ids):
        rows = self.root_indices[env_ids]
        task = self.task
        self.env.root_state[rows, :3] = self.default_base_pose[:3] + self.env.env_origins[env_ids]
        self.env.root_state[rows, :2] += 2.0 * task._draw(env_ids, 1, 2) + -1.0
        self.env.root_state[rows, 3:7] = self.default_base_pose[3:7]
        self.env.root_state[rows, 7:] = 0.

    def reset_idx(self, env_ids):
        super().reset_idx(env_ids)
        self.rand_force_buf[env_ids, self.rigid_body_dict['base']] = 10.0 * self.task._draw(env_ids, 2, 3) + -5.0

    # user-hook mode: torch PD loop, a1_conditional.py:64-75
    def step(self, actions):
        for _ in range(self.env.decimation):
            self.torques = self.p_gains * (actions + self.default_dof_pos - self.dof_pos) - self.d_gains * self.dof_vel
            self.torques = torch.clip(self.torques, -self.torque_limits, self.torque_limits)
            self._internal_motor_step(self.torques)
            self.gym.simulate(self.sim)
            self.gym.refresh_dof_state_tensor(self.sim)
        self.post_step()
        self.apply_force_on_base(self.rand_force_buf.view(-1, 3))


class A1Conditional(ShifuVecEnv):
    TERMS = ("tracking_lin_vel", "tracking_ang_vel", "stabilizing_base", "smoothing_action", "leg_collision",
             "torques_penalize")

    def __init__(self, cfg, fused: bool = True, carry_body_frame: bool = True, rng_seed: int = 0x5EED,
                 env_offset: int = 0, num_envs_global: int = None, store_measured_heights: bool = False,
                 use_cuda_graph: bool = True):
        super().__init__(cfg, env_offset=env_offset, num_envs_global=num_envs_global)
        self.auto_fuse = False          # this class fuses explicitly (fused= switch)
        self.fused = fused
        self.rng_seed = rng_seed
        self.use_cuda_graph = use_cuda_graph
        self._store_heights = store_measured_heights
        self.robot = A1Robot(A1ActorConfig())
        self.robot.task = self
        self.isg_env.create_envs(robot=self.robot)
        n, dev = self.num_envs, self.device
        self.num_commands = 3
        self.cmd_lin_vel_x, self.cmd_lin_vel_y, self.cmd_ang_vel_yaw = [-1., 1.], [-1., 1.], [-1., 1.]
        self.command_buf = torch.zeros(n, self.num_commands, dtype=torch.float32, device=dev)
        self.contact_terminate_indices = self.isg_env.gym.find_actor_rigid_body_handle(
            self.isg_env.env_handles[0], self.robot.actor_handle, 'base')
        # a1_conditional.py:99-102 (read by a feet_air_time term, if a subclass lists one)
        self.swing_time = torch.zeros(n, self.robot.ee_indices.shape[0], dtype=torch.float, device=dev)
        self.last_contacts = torch.zeros(n, len(self.robot.ee_indices), dtype=torch.bool, device=dev)
        self.contact_terminate_buf = torch.zeros(n, dtype=torch.bool, device=dev)
        self.terrain_levels = torch.zeros(n, dtype=torch.long, device=dev)
        self.hot = None
        if fused:
            self._fuse(carry_body_frame)

    # ------------------------------------------------------------------------------------------
    # fused mode
    # ------------------------------------------------------------------------------------------
    def _fuse(self, carry_body_frame):
        from shifu_b200 import terms
        from shifu_b200.gym import autofuse
        if self.robot.affine_root_layout() is None:
            raise NotImplementedError("the fused A1 kernel needs affine root_indices")
        names = [fn.__name__ for fn in self.reward_functions]
        obs = None
        num_obs = self.cfg.num_obs                  # 72 + 187, or 72 for a blind subclass
        if num_obs == 72 and self._store_heights:
            raise NotImplementedError("store_measured_heights with a 72-column observation: the fused blind step "
                                      "does not scan the terrain (fused=False measures and keeps the heights)")
        if type(self).compute_observations is not A1Conditional.compute_observations or num_obs != 259:
            # an edited observation hook: fused only when the kernel's observation layout expresses it,
            # never silently replaced by the reference observation
            try:
                obs = terms.compile_a1_obs(self, num_obs)
                terms.verify_a1_obs(self, obs, num_obs=num_obs)
            except terms.NotFusable as exc:
                raise NotImplementedError(f"{exc} (fused=False runs any observation hook)") from exc
        # reference constants: the named terms' (hotpath.A1_TERM_PARAMS) and the push force
        # (a1_conditional.py:82-87); step() hands the kernel raw actions, which a1_desc's default
        # action_scale scales (a1_conditional.py:122-124)
        desc = autofuse.a1_env_desc(self, names, rng_seed=self.rng_seed, obs=obs,
                                    force_body=self.robot.rigid_body_dict['base'], push_force_max=5.0)
        autofuse.install(self, "a1", autofuse.a1_hot_path(self, desc, names, carry_body_frame, self._store_heights))

    def step(self, actions: torch.Tensor):
        if not self.fused:
            return super().step(actions * 0.5)                              # a1_conditional.py:122-124
        from shifu_b200.gym import autofuse
        return autofuse.a1_fused_step(self, self.hot, actions)       # kernel launches, or one graph replay

    def reset_idx(self, env_ids):                   # user-hook mode; fused mode installs the kernel's
        if self.cfg.terrain.curriculum:
            self.update_terrain_curriculum(env_ids)
        super().reset_idx(env_ids)
        self.sample_command(env_ids)

    # ------------------------------------------------------------------------------------------
    # hooks (names feed the reward-term registry; bodies are the user-hook-mode torch code)
    # ------------------------------------------------------------------------------------------
    def build_reward_functions(self) -> typing.List:
        return [getattr(self, name) for name in self.TERMS]

    def episode_log(self, env_ids) -> typing.Dict:
        return {"terrain_levels": torch.mean(self.terrain_levels.to(torch.float))}

    def compute_observations(self):
        rb = self.robot
        heights = torch.clip(rb.base_pose[:, 2].unsqueeze(1) - 0.5 - self.isg_env.measured_heights, -1, 1.)
        self.obs_buf = torch.cat([self.command_buf, rb.base_lin_vel, rb.base_ang_vel, rb.gravity_vec,
                                  rb.dof_pos - rb.default_dof_pos, rb.dof_vel, self.actions_recorder.flatten(),
                                  heights], dim=1)

    def compute_termination(self):
        force = self.robot.contact_forces[:, self.contact_terminate_indices, :]
        self.contact_terminate_buf = torch.norm(force, dim=-1) > 1.
        self.time_out_buf = self.episode_length_buf > self.max_episode_length
        self.reset_buf = self.time_out_buf | self.contact_terminate_buf

    def tracking_lin_vel(self):
        err = torch.sum(torch.square(self.command_buf[:, :2] - self.robot.base_lin_vel[:, :2]), dim=1)
        return 1.0 * torch.exp(-err / 0.25)

    def tracking_ang_vel(self):
        err = torch.square(self.command_buf[:, 2] - self.robot.base_ang_vel[:, 2])
        return 0.5 * torch.exp(-err / 0.25)

    def stabilizing_base(self):
        return -2.0 * torch.square(self.robot.base_lin_vel[:, 2]) \
            + -0.005 * torch.sum(torch.square(self.robot.base_ang_vel[:, :2]), dim=1)

    def smoothing_action(self):
        a0, a1, a2 = (self.actions_recorder.get_last(i) for i in range(3))
        return -0.005 * (torch.sum(torch.square(a1 - a0), dim=1) + torch.sum(torch.square(a2 - 2 * a1 + a0), dim=1))

    def leg_collision(self):
        touch = torch.norm(self.robot.contact_forces[:, self.robot.leg_indices, :], dim=-1) > 0.1
        return -1. * torch.sum(touch.to(torch.float), dim=1)

    def torques_penalize(self):
        return -2e-5 * torch.sum(torch.square(self.robot.torques), dim=1)

    # -- user-hook-mode reset pieces (Philox-driven so both modes draw identical samples) --------
    def _draw(self, env_ids, stream, lanes):
        from shifu_b200.utils.philox import draw_u01
        return draw_u01(self.rng_seed, env_ids + self.env_offset, self.common_step_counter, stream, lanes)

    def sample_command(self, env_ids):
        if len(env_ids):
            self.command_buf[env_ids] = 2.0 * self._draw(env_ids, 3, 3) + -1.0

    def update_terrain_curriculum(self, env_ids):
        if not self.isg_env.init_done or len(env_ids) == 0:
            return
        from shifu_b200.utils.philox import draw_randint
        dist = torch.norm(self.robot.base_pose[env_ids, :2] - self.isg_env.env_origins[env_ids, :2], dim=1)
        up = dist > self.isg_env.terrain.env_length / 2
        down = (dist < torch.norm(self.command_buf[env_ids, :2], dim=1) * self.max_episode_length_s * 0.5) * ~up
        lv = self.terrain_levels[env_ids] + 1 * up - 1 * down
        rnd = draw_randint(self.rng_seed, env_ids + self.env_offset, self.common_step_counter, 0,
                           self.isg_env.max_terrain_level)
        self.terrain_levels[env_ids] = torch.where(lv >= self.isg_env.max_terrain_level, rnd, torch.clip(lv, 0))
        self.isg_env.update_terrain_level(env_ids, self.terrain_levels)
