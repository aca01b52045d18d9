"""ShifuVecEnv — the rsl_rl-compatible vectorised env (interface mirror of ``shifu/gym/env.py``).

Upward contract (``rsl_rl.env.VecEnv``): ``num_envs, num_obs, num_privileged_obs, num_actions,
max_episode_length, episode_length_buf, obs_buf, rew_buf, reset_buf, extras, device``;
``step(actions) -> (obs, privileged_obs, rew, dones, extras)``, ``reset()``,
``get_observations()``, ``get_privileged_observations()``.

User hooks (README.md:95-128): ``build_reward_functions``, ``compute_observations``,
``compute_termination``, optional ``reset_idx`` / ``episode_log`` / ``step``.

Two execution modes, both CUDA-only (no CPU fallback):

* **user-hook mode** (default): the hooks are arbitrary torch code on CUDA tensors and this class
  runs the reference's orchestration (env.py:85-130) around them, with the rows it owns itself —
  action / obs clip, reset-id compaction, history push — done by the ``libshifu_b200`` kernels;
* **fused mode**: ``post_step`` becomes one fused kernel.  A subclass whose hooks provably are what
  the kernel computes is fused on its first ``reset()`` / ``step()`` (``autofuse.py``); the task
  classes of ``shifu_b200/tasks`` fuse explicitly at construction.  Both ways build the descriptor,
  bind the env's tensors and dispatch ``step`` / ``reset_idx`` with the same code
  (``autofuse.install``).
"""
from __future__ import annotations

import math
from typing import Callable, Dict, List, Optional

import torch
from rsl_rl.env import VecEnv

from shifu_b200.configs import BaseEnvConfig, TerrainEnvConfig
from shifu_b200.gym.sim_facade import IsaacGymEnv, TerrainGymEnv
from shifu_b200.utils.history import HistoryRecorder


class ShifuVecEnv(VecEnv):
    #: try to replace the Python hooks by a fused kernel on the first reset()/step() (see autofuse.py);
    #: set to False (class or instance) to keep the hooks as eager torch code
    auto_fuse = True

    # ------------------------------------------------------------------ construction (env.py:19-63)
    def __init__(self, cfg: BaseEnvConfig, env_offset: int = 0, num_envs_global: Optional[int] = None):
        self.cfg = cfg
        self.env_offset = int(env_offset)
        self.num_envs_global = int(num_envs_global or cfg.num_envs)
        terrain = isinstance(cfg, TerrainEnvConfig)
        self.isg_env = (TerrainGymEnv(cfg, env_offset=env_offset, num_envs_global=num_envs_global) if terrain
                        else IsaacGymEnv(cfg))
        sim = self.isg_env
        self.num_envs, self.device = sim.num_envs, sim.device
        self.num_obs, self.num_privileged_obs, self.num_actions = cfg.num_obs, cfg.num_privileged_obs, cfg.num_actions
        norm = cfg.normalization
        self.clip_obs, self.clip_actions = norm.clip_observations, norm.clip_actions
        self.max_episode_length_s = cfg.episode_length_s
        self.max_episode_length = float(math.ceil(self.max_episode_length_s / sim.dt))
        self.common_step_counter = 0
        self.stats_allreduce: Optional[Callable] = None    # sums a tensor over ranks (sharded runs)
        self.extras: Dict = {}
        self.fusion_report = "not attempted"
        self._fusion = None            # (recipe, hot path, step fn) once fused (autofuse.install)
        self._fusion_tried = False
        self._allocate()
        self.reward_functions: List[Callable] = self.build_reward_functions()
        self._prepare_reward_functions()

    def _allocate(self):
        """The VecEnv buffers.  Their addresses are handed to the kernels, so they are created once
        and only ever written in place."""
        def new(*shape, dtype=torch.float, fill=0):
            return torch.full(shape, fill, device=self.device, dtype=dtype, requires_grad=False)

        n = self.num_envs
        self.actions = new(n, self.num_actions)
        self.obs_buf = new(n, self.num_obs)
        self.privileged_obs_buf = new(n, self.num_privileged_obs) if self.num_privileged_obs is not None else None
        self.rew_buf = new(n)
        self.reset_buf = new(n, dtype=torch.long, fill=1)
        self.time_out_buf = new(n, dtype=torch.bool)
        self._episode_length_buf = new(n, dtype=torch.long)
        if self.cfg.num_actions_history:
            self.actions_recorder = HistoryRecorder(self.actions.shape, self.cfg.num_actions_history,
                                                    device=self.device, kernels=self.isg_env.kernels)

    def _prepare_reward_functions(self):
        if not self.reward_functions:
            raise AssertionError("build_reward_functions() returned no reward term")
        self.episode_rewards = {}
        for term in self.reward_functions:
            self.episode_rewards[term.__name__] = torch.zeros(self.num_envs, device=self.device, dtype=torch.float)

    # rsl_rl re-binds ``env.episode_length_buf = randint_like(...)`` (init_at_random_ep_len,
    # policy_runner.py:22); the kernels hold the buffer's address, so assignment copies in place.
    @property
    def episode_length_buf(self):
        return self._episode_length_buf

    @episode_length_buf.setter
    def episode_length_buf(self, value):
        if value is not self._episode_length_buf:
            self._episode_length_buf.copy_(torch.as_tensor(value, device=self.device))

    def destroy(self):
        self.isg_env.destroy()

    # ------------------------------------------------------------------ user hooks
    def build_reward_functions(self) -> List[Callable]:
        raise NotImplementedError

    def compute_observations(self):
        raise NotImplementedError

    def compute_termination(self):
        raise NotImplementedError

    def episode_log(self, env_ids) -> Optional[Dict]:
        return None

    # ------------------------------------------------------------------ automatic fusion
    def _maybe_fuse(self):
        """First reset()/step(): replace the hooks by a fused kernel when they provably are what the kernel
        computes (autofuse.py).  Tasks that fuse explicitly (shifu_b200.tasks) have installed theirs."""
        if not self._fusion_tried:
            self._fusion_tried = True
            if self.auto_fuse and hasattr(self, "robot"):
                from shifu_b200.gym import autofuse
                autofuse.try_fuse(self, rng_seed=getattr(self.cfg, "rng_seed", 0x5EED),
                                  carry_body_frame=getattr(self.cfg, "carry_body_frame", True))
        return self._fusion

    # ------------------------------------------------------------------ orchestration, user-hook mode
    def step(self, actions: torch.Tensor):
        assert self.isg_env.robot, "add robot before step"
        fusion = self._maybe_fuse()
        if fusion is not None:
            return fusion[2](self, fusion[1], actions)
        kernels = self.isg_env.kernels()
        kernels.clip(actions, self.clip_actions, out=self.actions)               # env.py:87
        self.isg_env.step(self.actions)
        self.post_step()
        self.obs_buf = kernels.clip(self.obs_buf, self.clip_obs)                 # env.py:90
        return self.obs_buf, self.privileged_obs_buf, self.rew_buf, self.reset_buf, self.extras

    def post_step(self):                                                         # env.py:93-106
        self._episode_length_buf += 1
        self.common_step_counter += 1
        self.compute_termination()
        self.compute_reward()
        self.reset_idx(self.isg_env.kernels().nonzero(self.reset_buf))           # env.py:101, compaction kernel
        self.compute_observations()
        self.isg_env.refresh_sensors()
        if self.cfg.num_actions_history:
            self.actions_recorder.add(self.actions)

    def compute_reward(self):                                                    # env.py:180-185
        self.rew_buf.zero_()
        for term in self.reward_functions:
            value = term()
            self.episode_rewards[term.__name__] += value
            self.rew_buf += value

    def reset(self):
        self._maybe_fuse()
        everyone = torch.arange(self.num_envs, device=self.device)
        self.reset_idx(everyone)
        idle = torch.zeros(self.num_envs, self.num_actions, device=self.device, requires_grad=False)
        obs, privileged, *_ = self.step(idle)
        return obs, privileged

    def reset_idx(self, env_ids):                                                # env.py:114-130
        if len(env_ids) == 0:
            return
        self.isg_env.reset_idx(env_ids)
        self._episode_length_buf[env_ids] = 0
        self.reset_buf[env_ids] = 1
        if self.cfg.num_actions_history:
            self.actions_recorder.reset_idx(env_ids)
        self.extras["episode"] = {}
        self.log_info(env_ids)
        if self.cfg.send_timeouts:
            self.extras["time_outs"] = self.time_out_buf

    def log_info(self, env_ids):                                                 # env.py:149-158
        log = self.extras["episode"]
        for name, sums in self.episode_rewards.items():
            log[name] = torch.mean(sums[env_ids]) / self.max_episode_length_s
            sums[env_ids] = 0.
        log.update(self.episode_log(env_ids) or {})

    def get_observations(self):
        return self.obs_buf

    def get_privileged_observations(self):
        return self.privileged_obs_buf
