"""Observation layouts of the fused-observation tests (shifu_b200.hotpath.ObsLayout values)."""
from __future__ import annotations

# legged_gym's obs_scales / commands_scale (legged_robot_config.py): lin_vel 2, ang_vel 0.25, dof_pos 1,
# dof_vel 0.05, height_measurements 5, commands_scale = [lin_vel, lin_vel, ang_vel]
LG = dict(lin_vel=2.0, ang_vel=0.25, dof_pos=1.0, dof_vel=0.05, heights=5.0)


def d1_fix():
    """The reference observation with projected_gravity in place of gravity_vec (SURVEY D1)."""
    from shifu_b200.hotpath import ObsLayout
    return ObsLayout(slots=("COMMAND", "BASE_LIN_VEL", "BASE_ANG_VEL", "PROJECTED_GRAVITY"))


def legged_gym():
    """legged_gym's order (lin_vel, ang_vel, projected_gravity, commands) and scales."""
    from shifu_b200.hotpath import ObsLayout
    head = ([LG["lin_vel"]] * 3 + [LG["ang_vel"]] * 3 + [1.0] * 3 + [LG["lin_vel"], LG["lin_vel"], LG["ang_vel"]]
            + [LG["dof_pos"]] * 12 + [LG["dof_vel"]] * 12 + [1.0] * 36)
    return ObsLayout(slots=("BASE_LIN_VEL", "BASE_ANG_VEL", "PROJECTED_GRAVITY", "COMMAND"), scales=tuple(head),
                     height_scale=LG["heights"])


def extreme():
    """Negative and large scales that push columns past clip_obs = 100, and a scaled gravity_vec."""
    from shifu_b200.hotpath import ObsLayout
    head = ([-150.0, 7.0, 180.0] + [3.0, -3.0, 0.75] + [-250.0, 250.0, 1e3] + [40.0, -40.0, 0.1]
            + [-300.0 + 25.0 * d for d in range(12)] + [75.0, -75.0] * 6 + [-1000.0, 0.5, 130.0] * 12)
    return ObsLayout(slots=("GRAVITY_VEC", "PROJECTED_GRAVITY", "COMMAND", "BASE_ANG_VEL"), scales=tuple(head),
                     height_scale=-500.0)


LAYOUTS = {"d1": d1_fix, "legged_gym": legged_gym, "extreme": extreme}


def oracle_obs(p, st, layout):
    """The observation of the oracle's last step (oracle.shifu_oracle.a1_step) under ``layout``: every head
    column times its fp32 scale (one rounding per multiply), the clipped heights times the height scale,
    then the clip to +-clip_obs of env.py:90.

    Computed from the state a1_step leaves: command, body-frame velocities and projected gravity (the
    S_prev values body_frame wrote, D7), dof rows are what its observation read.  The history columns and
    the heights come from its reference observation: the history push follows the observation, and both
    are inside +-clip_obs (|actions| <= clip_actions = 1, heights clipped to +-1), so that clip left them
    exact."""
    import torch
    dof = st.dof_state.view(p.n, p.n_dof, 2)
    src = {"COMMAND": st.command, "BASE_LIN_VEL": st.base_lin_vel, "BASE_ANG_VEL": st.base_ang_vel,
           "GRAVITY_VEC": st.gravity_vec, "PROJECTED_GRAVITY": st.projected_gravity}
    head = torch.cat([src[s] for s in layout.slots] + [dof[..., 0] - p.q0, dof[..., 1], st.obs[:, 36:72]], dim=1)
    head = head * torch.tensor(layout.scales, dtype=torch.float)
    heights = st.obs[:, 72:] * torch.tensor(layout.height_scale, dtype=torch.float)
    return torch.clip(torch.cat([head, heights], dim=1), -p.clip_obs, p.clip_obs)
