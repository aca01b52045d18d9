"""Fused post-physics kernel time with the reference observation, legged_gym's observation layout, and that
layout with legged_gym's observation noise.

    python tools/obs_layout_cost.py [--envs 1048576] [--launches 200] [--rounds 6] [--out profiles/r5_obs_noise.json]

Three A1 tasks on the stand-in simulator with resident synthetic state (as bench.py builds them): the
unmodified ``A1Conditional`` (obs_layout 0, the default instantiations), a subclass whose
``compute_observations`` is legged_gym's (order lin_vel, ang_vel, projected_gravity, commands; obs_scales
and commands_scale), which the observation compiler turns into obs_layout 1 (the OBS instantiations), and
one whose hook also adds legged_gym's uniform noise (``cfg.noise.add_noise``; the NOISE instantiations).
Each round times ``--launches`` back-to-back launches of the fused kernel (``shifu_a1_post_physics``) of
one task with CUDA events, the tasks alternating round by round in one process; the card's name and
power limit are recorded with the numbers.  The noise's added time is set against the least time a
separate noise pass over the observation would take: it reads and writes the 1 036-byte row again."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def legged_gym_obs(self):
    import torch
    rb = self.robot
    cs = torch.tensor([2.0, 2.0, 0.25], device=self.device)
    heights = torch.clip(rb.base_pose[:, 2].unsqueeze(1) - 0.5 - self.isg_env.measured_heights, -1, 1.) * 5.0
    self.obs_buf = torch.cat([rb.base_lin_vel * 2.0, rb.base_ang_vel * 0.25, rb.projected_gravity,
                              self.command_buf * cs, (rb.dof_pos - rb.default_dof_pos) * 1.0, rb.dof_vel * 0.05,
                              self.actions_recorder.flatten(), heights], dim=1)


def legged_gym_noisy_obs(self):
    """legged_gym_obs + legged_gym's noise_scale_vec (noise_level 1, scaled by the obs_scales above)."""
    import torch
    legged_gym_obs(self)
    vec = torch.zeros(259, device=self.device)
    vec[:3], vec[3:6], vec[6:9] = 0.1 * 2.0, 0.2 * 0.25, 0.05
    vec[12:24], vec[24:36], vec[72:] = 0.01 * 1.0, 1.5 * 0.05, 0.1 * 5.0
    self.obs_buf += (2 * torch.rand_like(self.obs_buf) - 1) * vec


OBS_ROW_BYTES = 259 * 4
HBM_PEAK_GBS = 6540.5           # measured HBM peak of the B200 (DESIGN.md section 4)


def build(cls, n, device, seed=1234):
    import numpy as np
    import torch
    from shifu_b200.sim import fake_isaacgym
    fake_isaacgym.install(device)
    fake_isaacgym.reset_gym()
    fake_isaacgym.set_default_device(device)
    from shifu_b200.sim.synthetic import a1_snapshot
    from shifu_b200.tasks.a1_walking import A1EnvConfig
    cfg = A1EnvConfig()
    cfg.num_envs, cfg.device = n, device
    np.random.seed(0)
    torch.manual_seed(seed)
    env = cls(cfg, fused=True, carry_body_frame=True, rng_seed=seed)
    isg, hp = env.isg_env, env.hot
    snap = a1_snapshot(seed, 1, n, gen_device=device, p_base=0.01, p_leg=0.1, xy_range=3.0, offmap=False)
    root = snap.root_offset.clone()
    root[:, :3] += isg.env_origins
    isg.root_state.copy_(root)
    isg.dof_state.copy_(snap.dof[4].reshape(n * 12, 2))
    isg.contact_state.copy_(snap.contact.reshape(n * 17, 3))
    g = torch.Generator().manual_seed(seed)
    env.episode_length_buf = torch.randint(0, 500, (n,), generator=g).to(device)
    env.command_buf.copy_((torch.rand(n, 3, generator=g) * 2 - 1).to(device))
    hp.sync_level_sum()
    hp.body_frame()
    return env


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = [c.strip() for c in q.split(",")]
    except (OSError, ValueError, subprocess.SubprocessError) as exc:
        out["power_limit"] = f"unavailable ({exc})"
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_obs_noise.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures the fused kernel on the GPU")
    from shifu_b200.sim import fake_isaacgym
    fake_isaacgym.install("cuda:0")
    from shifu_b200.tasks.a1_walking import A1Conditional
    lg_cls = type("LeggedGymObsA1", (A1Conditional,), {"compute_observations": legged_gym_obs})
    noisy_cls = type("LeggedGymNoisyObsA1", (A1Conditional,), {"compute_observations": legged_gym_noisy_obs})
    envs = {"reference": build(A1Conditional, args.envs, "cuda:0"), "legged_gym": build(lg_cls, args.envs, "cuda:0"),
            "legged_gym_noise": build(noisy_cls, args.envs, "cuda:0")}
    layouts = {k: int(e.hot.desc.obs_layout) for k, e in envs.items()}
    assert layouts == {"reference": 0, "legged_gym": 1, "legged_gym_noise": 1}, layouts
    assert envs["legged_gym_noise"].hot.desc.obs_height_noise == 0.5
    for e in envs.values():
        for _ in range(args.warmup):
            e.hot.post_physics()
    torch.cuda.synchronize()
    ms = {k: [] for k in envs}
    for _ in range(args.rounds):
        for k, e in envs.items():
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(args.launches):
                e.hot.post_physics()
            t1.record()
            torch.cuda.synchronize()
            ms[k].append(t0.elapsed_time(t1) / args.launches)
    res = {"what": "fused post-physics kernel (shifu_a1_post_physics), ms per launch, resident state, carried body "
                   "frame, no measured_heights; rounds alternate the three tasks in one process",
           "card": card(), "envs": args.envs, "launches_per_round": args.launches, "rounds": args.rounds,
           "obs_layout": layouts,
           "ms_per_launch": {k: {"median": statistics.median(v), "min": min(v), "max": max(v), "all": v}
                             for k, v in ms.items()}}
    ref, lg = res["ms_per_launch"]["reference"]["median"], res["ms_per_launch"]["legged_gym"]["median"]
    noisy = res["ms_per_launch"]["legged_gym_noise"]["median"]
    res["legged_gym_over_reference"] = lg / ref
    res["noise_added_ms"] = noisy - lg
    # computed from sizes, not measured: a pass after the kernel reads and writes every observation row
    res["separate_noise_pass_floor_ms"] = 2 * OBS_ROW_BYTES * args.envs / (HBM_PEAK_GBS * 1e9) * 1e3
    res["separate_noise_pass_floor_basis"] = f"2 x {OBS_ROW_BYTES} B x envs / {HBM_PEAK_GBS} GB/s (measured HBM peak)"
    res["noise_added_over_floor"] = res["noise_added_ms"] / res["separate_noise_pass_floor_ms"]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "envs", "legged_gym_over_reference", "noise_added_ms",
                                         "separate_noise_pass_floor_ms", "noise_added_over_floor")}
                     | {"median_ms": {k: v["median"] for k, v in res["ms_per_launch"].items()}}))


if __name__ == "__main__":
    main()
