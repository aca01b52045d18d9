"""Fused A1 step of legged_gym's own observation (the action head: 235 columns, 48 blind) against the
72-column head it replaces.

    python tools/action_head_cost.py [--envs 1048576] [--launches 200] [--rounds 6] [--steps 100]
                                     [--out profiles/r7_action_head.json]

Six A1 tasks on the stand-in simulator with resident synthetic state and the carried body frame (as
bench.py builds them): legged_gym's layout with the 36 history columns (259, "hybrid") and legged_gym's
own observation, whose head ends with the step's actions (235), each with and without legged_gym's noise;
and the blind pair, 72 and 48 columns, with noise.  Reported, the tasks alternating round by round in one
process, with the card's name and power limit:
- kernel ms per launch (``shifu_a1_post_physics``, ``--launches`` back-to-back launches timed with CUDA events);
- ms per step through ``A1Conditional.step`` (CUDA-graph replay) of the noisy 235 task and its 259 sibling;
- each action-head kernel's share of the measured HBM peak on the bytes it must move (computed from sizes),
  and whether it is slower than its 72-column sibling beyond that sibling's spread over the rounds."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from blind_cost import BLIND_BYTES, blind_class, blind_legged_gym_noisy_obs, timed  # noqa: E402
from obs_layout_cost import HBM_PEAK_GBS, build, card, legged_gym_noisy_obs, legged_gym_obs  # noqa: E402

# bytes per env (DESIGN.md section 3): the action head writes 24 observation columns (96 B) fewer than the
# 72-column head; everything else the step reads and writes is the same
SIGHTED_BYTES = 1723                          # 235 columns: the 259-column step's 1 819 B less 96
BLIND_ACT_BYTES = BLIND_BYTES - 96            # 48 columns: 975


def _noise_vec(self, width):
    """legged_gym's noise_scale_vec (noise_level 1, obs_scales of tools/obs_layout_cost.py); none on the actions."""
    import torch
    vec = torch.zeros(width, device=self.device)
    vec[:3], vec[3:6], vec[6:9] = 0.1 * 2.0, 0.2 * 0.25, 0.05
    vec[12:24], vec[24:36] = 0.01 * 1.0, 1.5 * 0.05
    vec[48:] = 0.1 * 5.0
    return vec


def action_head_obs(self, noise=False):
    """legged_gym's compute_observations: its order and obs_scales, the step's actions, the heights when the
    task measures them, and its uniform noise when ``noise``."""
    import torch
    rb = self.robot
    cs = torch.tensor([2.0, 2.0, 0.25], device=self.device)
    cols = [rb.base_lin_vel * 2.0, rb.base_ang_vel * 0.25, rb.projected_gravity, self.command_buf * cs,
            (rb.dof_pos - rb.default_dof_pos) * 1.0, rb.dof_vel * 0.05, self.actions]
    if self.num_obs == 235:
        cols.append(torch.clip(rb.base_pose[:, 2].unsqueeze(1) - 0.5 - self.isg_env.measured_heights, -1, 1.) * 5.0)
    self.obs_buf = torch.cat(cols, dim=-1)
    if noise:
        self.obs_buf += (2 * torch.rand_like(self.obs_buf) - 1) * _noise_vec(self, self.obs_buf.shape[1])


def action_head_noisy_obs(self):
    action_head_obs(self, noise=True)


def action_head_class(obs_fn, num_obs):
    """An A1Conditional subclass with ``cfg.num_obs = num_obs`` (235, or 48 without height measurement)."""
    from shifu_b200.tasks.a1_walking import A1Conditional

    def init(self, cfg, **kw):
        cfg.num_obs = num_obs
        cfg.terrain.measure_heights = num_obs == 235
        A1Conditional.__init__(self, cfg, **kw)

    return type(f"ActionHead{num_obs}" + obs_fn.__name__, (A1Conditional,),
                {"compute_observations": obs_fn, "__init__": init})


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_action_head.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures the fused kernels on the GPU")
    from shifu_b200.sim import fake_isaacgym
    fake_isaacgym.install("cuda:0")
    from shifu_b200.tasks.a1_walking import A1Conditional
    classes = {
        "hybrid_259": type("HybridObsA1", (A1Conditional,), {"compute_observations": legged_gym_obs}),
        "legged_gym_235": action_head_class(action_head_obs, 235),
        "hybrid_259_noise": type("HybridNoisyObsA1", (A1Conditional,), {"compute_observations": legged_gym_noisy_obs}),
        "legged_gym_235_noise": action_head_class(action_head_noisy_obs, 235),
        "blind_72_noise": blind_class(blind_legged_gym_noisy_obs),
        "blind_48_noise": action_head_class(action_head_noisy_obs, 48),
    }
    siblings = {"legged_gym_235": "hybrid_259", "legged_gym_235_noise": "hybrid_259_noise",
                "blind_48_noise": "blind_72_noise"}
    envs = {k: build(c, args.envs, "cuda:0") for k, c in classes.items()}
    widths = {k: int(e.hot.desc.num_obs) for k, e in envs.items()}
    assert widths == {"hybrid_259": 259, "legged_gym_235": 235, "hybrid_259_noise": 259, "legged_gym_235_noise": 235,
                      "blind_72_noise": 72, "blind_48_noise": 48}, widths
    for k in ("hybrid_259_noise", "legged_gym_235_noise", "blind_72_noise", "blind_48_noise"):
        assert envs[k].hot.desc.obs_noise[0] > 0, k
    for e in envs.values():
        for _ in range(args.warmup):
            e.hot.post_physics()
    torch.cuda.synchronize()
    # ---- kernel time, tasks alternating round by round
    ms = {k: [] for k in envs}
    for _ in range(args.rounds):
        for k, e in envs.items():
            ms[k].append(timed(e.hot.post_physics, args.launches))
    # ---- whole step through A1Conditional.step (graph replay on resident state)
    step_keys = ("hybrid_259_noise", "legged_gym_235_noise")
    act = {k: envs[k].hot.action_input() for k in step_keys}
    for k in step_keys:
        envs[k].reset()
        for _ in range(args.warmup):
            envs[k].step(act[k])
        assert envs[k].hot._graph is not None, f"{k}: the step did not replay a graph"
    torch.cuda.synchronize()
    step_ms = {k: [] for k in step_keys}
    for _ in range(args.rounds):
        for k in step_keys:
            step_ms[k].append(timed(lambda k=k: envs[k].step(act[k]), args.steps))
    stat = lambda v: {"median": statistics.median(v), "min": min(v), "max": max(v), "all": v}  # noqa: E731
    res = {"what": "fused A1 post-physics kernel (shifu_a1_post_physics) ms per launch, and A1Conditional.step "
                   "(CUDA-graph replay) ms per step; resident state, carried body frame, no measured_heights; "
                   "rounds alternate the tasks in one process",
           "card": card(), "envs": args.envs, "launches_per_round": args.launches, "steps_per_round": args.steps,
           "rounds": args.rounds, "num_obs": widths,
           "kernel_ms_per_launch": {k: stat(v) for k, v in ms.items()},
           "step_ms": {k: stat(v) for k, v in step_ms.items()}}
    kernel = res["kernel_ms_per_launch"]
    bytes_per_env = {"legged_gym_235": SIGHTED_BYTES, "legged_gym_235_noise": SIGHTED_BYTES,
                     "blind_48_noise": BLIND_ACT_BYTES}
    res["bytes_per_env"] = bytes_per_env
    res["floor_ms"] = {k: b * args.envs / (HBM_PEAK_GBS * 1e9) * 1e3 for k, b in bytes_per_env.items()}
    res["floor_basis"] = f"bytes per env x envs / {HBM_PEAK_GBS} GB/s (measured HBM peak); computed from sizes"
    res["share_of_peak"] = {k: res["floor_ms"][k] / kernel[k]["median"] for k in bytes_per_env}
    res["against_72_column_sibling"] = {
        k: {"sibling": s, "ratio": kernel[k]["median"] / kernel[s]["median"],
            "slower_beyond_spread": kernel[k]["median"] > kernel[s]["max"]}
        for k, s in siblings.items()}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "envs", "share_of_peak", "against_72_column_sibling")}
                     | {"kernel_median_ms": {k: v["median"] for k, v in kernel.items()},
                        "step_median_ms": {k: v["median"] for k, v in res["step_ms"].items()}}))


if __name__ == "__main__":
    main()
