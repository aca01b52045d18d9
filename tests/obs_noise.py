"""Noisy observation layouts of the observation-noise tests and ``oracle_obs_noisy``, the test oracle's
observation with legged_gym's uniform noise added before the clip to +-clip_obs."""
from __future__ import annotations

import copy
import math

import numpy as np
import torch

from tests import obs_layouts

# legged_gym's noise_scale_vec on its observation (noise_level 1, scaled by obs_scales): lin_vel 0.1 * 2,
# ang_vel 0.2 * 0.25, gravity 0.05, commands 0, dof_pos 0.01 * 1, dof_vel 1.5 * 0.05, actions 0,
# heights 0.1 * 5
LG_NOISE = [0.2] * 3 + [0.05] * 3 + [0.05] * 3 + [0.0] * 3 + [0.01] * 12 + [0.075] * 12 + [0.0] * 36
LG_HEIGHT_NOISE = 0.5


def legged_gym_noisy():
    """legged_gym's layout with legged_gym's noise."""
    return _with_noise(obs_layouts.legged_gym(), LG_NOISE, LG_HEIGHT_NOISE)


def loud():
    """Noise scales that push columns past clip_obs = 100 in both directions (and a negative scale)."""
    noise = [150.0, -80.0, 300.0] * 4 + [0.0, 1e3] * 6 + [0.5] * 12 + [120.0, 0.0, -250.0] * 12
    return _with_noise(obs_layouts.d1_fix(), noise, 180.0)


def _with_noise(layout, noise, height_noise):
    from shifu_b200.hotpath import ObsLayout
    return ObsLayout(layout.slots, layout.scales, layout.height_scale, tuple(noise), height_noise)


NOISY = {"legged_gym": legged_gym_noisy, "loud": loud}


def noise_values(layout, seed, env_ids, step):
    """(R, 259) fp32 noise fl((2u - 1) * scale) of envs ``env_ids`` (global ids) at ``step``."""
    from oracle import obs_noise_np as onp
    u = torch.from_numpy(onp.obs_noise_u01(seed, np.asarray(env_ids), step))
    scale = torch.tensor(layout.noise + (layout.height_noise,) * onp.OBS_POINTS, dtype=torch.float)
    return (2 * u - 1) * scale


def oracle_obs_noisy(p, st, layout, seed, step):
    """``obs_layouts.oracle_obs`` with the noise of ``layout`` drawn at (seed, step) for the oracle's envs
    (global ids p.env_offset + i): every column fl(fl(x_j * scale_j) + n_j), the heights fl(fl(clip(z - 0.5
    - h, +-1) * height_scale) + n_j), then the clip to +-clip_obs."""
    if not layout.has_noise():
        return obs_layouts.oracle_obs(p, st, layout)
    unclipped = copy.copy(p)
    unclipped.clip_obs = math.inf
    clean = obs_layouts.oracle_obs(unclipped, st, layout)
    n = noise_values(layout, seed, np.arange(p.n) + p.env_offset, step)
    return torch.clip(clean + n, -p.clip_obs, p.clip_obs)
