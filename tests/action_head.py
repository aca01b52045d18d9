"""The action head of the fused-observation tests: legged_gym's own observation, whose 48-column head ends
with the step's actions (``obs_buf`` = 235 columns with the heights, 48 blind), and its oracle.

The noise map of the 235-column observation is derived here from the oracle's 259-column map
(``oracle.obs_noise_np``): column j < 48 keeps the word and lane of column j, and height column 48 + k
those of column 72 + k.  So the draws of the 235-column observation are columns 0-47 and 72-258 of the
259-column draws, independently of the kernels' and ``shifu_b200.utils.philox``'s width-aware formula."""
from __future__ import annotations

import copy
import math

import numpy as np
import torch

from tests import obs_layouts, obs_noise

HEAD_ACT, POINTS = 48, 187
# the columns of the 259-column observation that the 235-column one keeps, in order
KEPT = np.concatenate([np.arange(HEAD_ACT), np.arange(72, 72 + POINTS)])


def _act(layout, action_scales, action_noise, height_noise):
    from shifu_b200.hotpath import ObsLayout
    return ObsLayout(layout.slots, layout.scales[:36] + tuple(action_scales), layout.height_scale,
                     layout.noise[:36] + tuple(action_noise), height_noise)


def legged_gym():
    """legged_gym's observation: its order and obs_scales, the step's actions unscaled."""
    return _act(obs_layouts.legged_gym(), (1.0,) * 12, (0.0,) * 12, 0.0)


def legged_gym_noisy():
    """legged_gym's observation with its noise_scale_vec (the actions get no noise in legged_gym)."""
    lay = obs_noise.legged_gym_noisy()
    return _act(lay, (1.0,) * 12, (0.0,) * 12, lay.height_noise)


def loud():
    """Scales and noise on the action columns that push them past clip_obs = 100 in both directions."""
    lay = obs_noise.loud()
    return _act(lay, [-150.0, 0.5, 300.0] * 4, [0.0, 90.0, -200.0] * 4, lay.height_noise)


LAYOUTS = {"legged_gym": legged_gym, "legged_gym_noisy": legged_gym_noisy, "loud": loud}


def blind(layout):
    """The layout for a 48-column (blind) observation: no height noise."""
    from shifu_b200.hotpath import ObsLayout
    return ObsLayout(layout.slots, layout.scales, layout.height_scale, layout.noise, 0.0)


def with_history(layout):
    """The 72-column layout with the same columns 0-35, scales and noise (history columns scale 1, no noise)."""
    from shifu_b200.hotpath import ObsLayout
    return ObsLayout(layout.slots, layout.scales[:36] + (1.0,) * 36, layout.height_scale,
                     layout.noise[:36] + (0.0,) * 36, layout.height_noise)


def noise_map():
    """(word, lane) of the 235 columns, from the oracle's 259-column map."""
    from oracle import obs_noise_np as onp
    word, lane = onp.obs_noise_map()
    return word[KEPT], lane[KEPT]


def noise_u01(seed, env_ids, step):
    """(R, 235) float32 u of the 235-column observation noise (the oracle's draws, columns KEPT)."""
    from oracle import obs_noise_np as onp
    return onp.obs_noise_u01(seed, np.asarray(env_ids), step)[:, KEPT]


def oracle_obs(p, st, layout, seed=None, step=None):
    """The (n, 235) action-head observation of the oracle's last step under ``layout`` (columns [:48] are
    the blind one): the slots, dof_pos - q0 and dof_vel as ``obs_layouts.oracle_obs`` builds them, then the
    step's actions ``st.actions`` (env.actions after the action clip), every column times its fp32 scale,
    the heights of the oracle's reference observation times the height scale; with noise (drawn at
    ``seed``, ``step`` for global env ids p.env_offset + i) fl(fl(x * scale) + n), then the clip to
    +-clip_obs."""
    unclipped = copy.copy(p)
    unclipped.clip_obs = math.inf
    ref = obs_layouts.oracle_obs(unclipped, st, obs_noise._with_noise(with_history(layout), (0.0,) * 72, 0.0))
    act = st.actions * torch.tensor(layout.scales[36:], dtype=torch.float)
    obs = torch.cat([ref[:, :36], act, ref[:, 72:]], dim=1)
    if layout.has_noise():
        u = torch.from_numpy(noise_u01(seed, np.arange(p.n) + p.env_offset, step))
        scale = torch.tensor(layout.noise + (layout.height_noise,) * POINTS, dtype=torch.float)
        obs = obs + (2 * u - 1) * scale
    return torch.clip(obs, -p.clip_obs, p.clip_obs)
