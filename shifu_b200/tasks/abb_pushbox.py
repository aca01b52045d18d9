"""ABB push-box, prior (state-input) stage on the shifu_b200 API (BASELINE config 4).

Counterpart of ``examples/abb_pushbox_vision/a_prior_stage.py`` + ``task_config.py:49-91``.
The post-physics path (termination, 2 reward terms, reset incl. the random cube / goal poses,
6-column observation) is one CUDA kernel; the box poses come from device-side Philox draws
instead of the reference's per-env Python ``np.random.uniform`` loop (96 % of its step).  The
pre-physics action path (end-effector target -> damped-least-squares IK, a_prior_stage.py:67-73)
is row N2 of SURVEY.md §8f and stays torch code in this round.
"""
from __future__ import annotations

import numpy as np
import torch

from shifu_b200 import hotpath
from isaacgym import gymapi

from shifu_b200.configs import ArmRobotActorConfig, BaseEnvConfig, BoxActorConfig, CameraSensorConfig, PPOConfig
from shifu_b200.gym import ShifuVecEnv
from shifu_b200.units import ArmRobot, Box

ASSET_ROOT = "./asset"


class TableConfig(BoxActorConfig):                 # task_config.py:13-24
    root_dir = ASSET_ROOT
    name = "table"
    default_pos = [0, 0, 0.05]
    default_quat = [0, 0, 0, 1]
    box_dim = [0.6, 0.6, 0.1]
    mass = 0.
    color = [0.8, 0.8, 0.8]

    class asset_options(BoxActorConfig.asset_options):
        fix_base_link = True


class PushBoxConfig(BoxActorConfig):               # task_config.py:27-34
    root_dir = ASSET_ROOT
    name = "box"
    default_pos = [0, 0, 0.125]
    default_quat = [0, 0, 0, 1]
    box_dim = [0.05, 0.05, 0.05]
    mass = 0.1
    color = [.25, .65, .3]


class GoalBoxConfig(BoxActorConfig):               # task_config.py:37-47
    root_dir = ASSET_ROOT
    name = "goal"
    default_pos = [0, 0, 0.1]
    default_quat = [0, 0, 0, 1]
    box_dim = [0.08, 0.08, 0.002]
    mass = 0.
    color = [0.8, 0., 0.]

    class asset_options(BoxActorConfig.asset_options):
        fix_base_link = True


class AbbRobotConfig(ArmRobotActorConfig):         # task_config.py:49-64
    root_dir = ASSET_ROOT
    name = "AbbRobot-VacuumRod"
    urdf_filename = "urdf/abb_rod_description/urdf/abb_rod_isaac.urdf"
    end_effector_names = ['tip0']
    default_pos = [-0.48, 0, 0]
    default_quat = [0, 0, 0, 1]
    default_dof_pos = [0., 0.6437, 0.1748, 0., 0.7541, 0.]
    dof_stiffness = [800] * 6
    dof_damping = [40] * 6
    end_effector_velocity = 0.2
    default_ee_quat = [0., 1., 0., 0]
    min_ee_pos = [-0.2, -0.2, 0.11]
    max_ee_pos = [0.2, 0.2, 0.14]


class PushBoxCameraConfig(CameraSensorConfig):     # task_config.py:124-145 (RealSense D415-like)
    name = 'rgbd_camera'
    local_lookat_positions = [[0.7, 0., 0.7], [0., 0., 0.1]]
    image_types = [gymapi.IMAGE_COLOR, gymapi.IMAGE_DEPTH, gymapi.IMAGE_SEGMENTATION]
    image_normalization = True

    class camera_props(CameraSensorConfig.camera_props):
        enable_tensors = True
        use_collision_geometry = False
        width = 128
        height = 128
        horizontal_fov = 42
        near_plane = 0.1
        far_plane = 3


class PriorStageEnvConfig(BaseEnvConfig):          # task_config.py:72-91
    num_envs = 3000
    num_obs = 6
    num_privileged_obs = None
    num_actions = 3
    send_timeouts = True
    episode_length_s = 20.

    class sim(BaseEnvConfig.sim):
        dt = 0.02

    class control(BaseEnvConfig.control):
        decimation = int(0.1 / 0.02)

    class debug(BaseEnvConfig.debug):
        headless = True

    class normalization(BaseEnvConfig.normalization):
        clip_observations = 10.
        clip_actions = 1.


class PriorStagePPOConfig(PPOConfig):
    seed = 42
    runner_class_name = "AbbPushBoxTask"


class RandPosBox(Box):
    """Box whose reset pose is random (a_prior_stage.py:24-51); in the fused task the draw happens
    inside the kernel, these ranges only parameterise it."""

    def __init__(self, cfg):
        super().__init__(cfg)
        self.pos_range = {"low": [-0.1, -0.1, 0.125], "high": [0.1, 0.1, 0.125]}
        self.euler_range = {"low": [0, 0, -np.pi], "high": [0, 0, np.pi]}


class GoalBox(RandPosBox):
    def __init__(self, cfg):
        super().__init__(cfg)
        self.pos_range['low'][2] = self.pos_range['high'][2] = self.cfg.default_pos[2]


class AbbRobot(ArmRobot):
    def init_buffers(self):
        super().init_buffers()
        self.min_ee_pos = torch.tensor(self.cfg.min_ee_pos, dtype=torch.float, device=self.device)
        self.max_ee_pos = torch.tensor(self.cfg.max_ee_pos, dtype=torch.float, device=self.device)

    def step(self, actions):
        # a_prior_stage.py:67-73 — goal construction, clamp and IK in one shifu_arm_ik launch (row N2)
        self.env.kernels().arm_ik(actions=actions, ee_velocity=self.end_effector_velocity, dt=self.env.dt,
                                  min_ee_pos=self.cfg.min_ee_pos, max_ee_pos=self.cfg.max_ee_pos,
                                  tar_quat=self.cfg.default_ee_quat, dof_targets=self.dof_targets,
                                  **self._ik_layout())
        self.apply_dof_targets(self.dof_targets)


class AbbPushBox(ShifuVecEnv):
    TERMS = ("reward_reaching", "reward_success")

    def __init__(self, cfg, rng_seed: int = 0x5EED, env_offset: int = 0):
        super().__init__(cfg, env_offset=env_offset)
        self.rng_seed = rng_seed
        self.robot = AbbRobot(AbbRobotConfig())
        self.table = Box(TableConfig())
        self.cube = RandPosBox(PushBoxConfig())
        self.goal = GoalBox(GoalBoxConfig())
        self.isg_env.create_envs(robot=self.robot, objects=[self.table, self.cube, self.goal],
                                 sensors=self._sensors())
        self.success_buf = torch.zeros(self.num_envs, device=self.device, dtype=torch.bool)
        self._fuse()

    def _sensors(self):
        """Extra units of the perceptual stages (b_regression_stage.py:42-48); none in the prior stage."""
        return []

    def _fuse(self):
        """Step and reset_idx (env.py:85-130) of the 4-actor scene run ``shifu_abb_post_physics`` /
        ``shifu_abb_reset_idx``: default robot / table poses and Philox-drawn cube and goal poses
        (a_prior_stage.py:39-51) with the reference's reward constants."""
        from shifu_b200.gym import autofuse
        actors = [self.robot, self.table, self.cube, self.goal]
        layouts = [a.affine_root_layout() for a in actors]
        if any(l is None or l[0] != len(actors) for l in layouts):
            raise NotImplementedError("the fused ABB kernel needs the 4-actor interleaved root layout")
        autofuse.install(self, "abb", autofuse.abb_hot_path(self, self.rng_seed, hotpath.ABB_TERM_PARAMS))

    # hooks: the names feed the reward-term registry (a_prior_stage.py:112-127)
    def build_reward_functions(self):
        return [self.reward_reaching, self.reward_success]

    def reward_reaching(self):
        raise NotImplementedError("evaluated inside shifu_abb_post_physics")

    def reward_success(self):
        raise NotImplementedError("evaluated inside shifu_abb_post_physics")

    def episode_log(self, env_ids):
        return {'success_rate': self.extras["episode"]["success_rate"]}


class VisionAbbPushBox(AbbPushBox):
    """The perceptual stages' env (b_regression_stage.py:34-50, c_vision_stage.py:31-47): the prior
    stage plus an RGB-D camera per env, refreshed by ``isg_env.refresh_sensors()`` — one
    ``shifu_camera_gather`` launch instead of a Python loop over the envs (row N4)."""

    def __init__(self, cfg, camera_cfg=None, **kw):
        from shifu_b200.units.sensors import CameraSensor
        self.camera = CameraSensor(camera_cfg if camera_cfg is not None else PushBoxCameraConfig())
        super().__init__(cfg, **kw)

    def _sensors(self):
        return [self.camera]
