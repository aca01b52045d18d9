"""Fused A1 step of blind tasks (72-column observation, no height scan) against the sighted ones.

    python tools/blind_cost.py [--envs 1048576] [--launches 200] [--rounds 6] [--steps 100] [--out profiles/r6_blind.json]

Four A1 tasks on the stand-in simulator with resident synthetic state and the carried body frame (as
bench.py builds them): sighted and blind, each with the reference head and with legged_gym's layout +
uniform noise.  A blind task is an ``A1Conditional`` subclass with ``cfg.num_obs = 72``,
``cfg.terrain.measure_heights = False`` and a ``compute_observations`` without the height columns.
Reported, the tasks alternating round by round in one process, with the card's name and power limit:
- kernel ms per launch (``shifu_a1_post_physics``, ``--launches`` back-to-back launches timed with CUDA events);
- ms per step through ``A1Conditional.step`` (CUDA-graph replay), sighted vs blind, reference head;
- the blind kernel's share of the measured HBM peak on the bytes it must move (computed from sizes)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from obs_layout_cost import HBM_PEAK_GBS, build, card, legged_gym_noisy_obs  # noqa: E402

# bytes per env of one blind step (DESIGN.md section 3): it reads what the sighted step reads, and writes obs
# 288, rew 4, flags 3, ep_len 8, ep_sums 24 (six terms), history 144 and the carried rows 36
BLIND_READ_BYTES = 564
BLIND_WRITE_BYTES = 288 + 4 + 3 + 8 + 24 + 144 + 36
BLIND_BYTES = BLIND_READ_BYTES + BLIND_WRITE_BYTES        # 1 071


def blind_obs(self):
    """The reference head without the height columns."""
    import torch
    rb = self.robot
    self.obs_buf = torch.cat([self.command_buf, rb.base_lin_vel, rb.base_ang_vel, rb.gravity_vec,
                              rb.dof_pos - rb.default_dof_pos, rb.dof_vel, self.actions_recorder.flatten()], dim=1)


def blind_legged_gym_noisy_obs(self):
    """legged_gym's blind observation (its flat configurations): layout, obs_scales and head noise."""
    import torch
    rb = self.robot
    cs = torch.tensor([2.0, 2.0, 0.25], device=self.device)
    self.obs_buf = torch.cat([rb.base_lin_vel * 2.0, rb.base_ang_vel * 0.25, rb.projected_gravity,
                              self.command_buf * cs, (rb.dof_pos - rb.default_dof_pos) * 1.0, rb.dof_vel * 0.05,
                              self.actions_recorder.flatten()], dim=1)
    vec = torch.zeros(72, device=self.device)
    vec[:3], vec[3:6], vec[6:9] = 0.1 * 2.0, 0.2 * 0.25, 0.05
    vec[12:24], vec[24:36] = 0.01 * 1.0, 1.5 * 0.05
    self.obs_buf += (2 * torch.rand_like(self.obs_buf) - 1) * vec


def blind_class(obs_fn):
    """An A1Conditional subclass with the blind config (num_obs = 72, no height measurement) and ``obs_fn``."""
    from shifu_b200.tasks.a1_walking import A1Conditional

    def init(self, cfg, **kw):
        cfg.num_obs, cfg.terrain.measure_heights = 72, False
        A1Conditional.__init__(self, cfg, **kw)

    return type("Blind" + obs_fn.__name__, (A1Conditional,), {"compute_observations": obs_fn, "__init__": init})


def timed(fn, reps):
    import torch
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_blind.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures the fused kernels on the GPU")
    from shifu_b200.sim import fake_isaacgym
    fake_isaacgym.install("cuda:0")
    from shifu_b200.tasks.a1_walking import A1Conditional
    noisy_cls = type("LeggedGymNoisyObsA1", (A1Conditional,), {"compute_observations": legged_gym_noisy_obs})
    classes = {"sighted_reference": A1Conditional, "sighted_legged_gym_noise": noisy_cls,
               "blind_reference": blind_class(blind_obs), "blind_legged_gym_noise": blind_class(blind_legged_gym_noisy_obs)}
    envs = {k: build(c, args.envs, "cuda:0") for k, c in classes.items()}
    widths = {k: int(e.hot.desc.num_obs) for k, e in envs.items()}
    assert widths == {"sighted_reference": 259, "sighted_legged_gym_noise": 259, "blind_reference": 72,
                      "blind_legged_gym_noise": 72}, widths
    assert envs["blind_legged_gym_noise"].hot.desc.obs_layout == 1 and envs["blind_legged_gym_noise"].hot.desc.obs_noise[0] > 0
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
    step_keys = ("sighted_reference", "blind_reference")
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
    floor = BLIND_BYTES * args.envs / (HBM_PEAK_GBS * 1e9) * 1e3
    res["blind_bytes_per_env"] = BLIND_BYTES
    res["blind_floor_ms"] = floor
    res["blind_floor_basis"] = f"{BLIND_BYTES} B x envs / {HBM_PEAK_GBS} GB/s (measured HBM peak); computed from sizes"
    res["blind_share_of_peak"] = {k: floor / res["kernel_ms_per_launch"][k]["median"]
                                  for k in ("blind_reference", "blind_legged_gym_noise")}
    res["blind_over_sighted_kernel"] = {
        "reference": res["kernel_ms_per_launch"]["blind_reference"]["median"]
        / res["kernel_ms_per_launch"]["sighted_reference"]["median"],
        "legged_gym_noise": res["kernel_ms_per_launch"]["blind_legged_gym_noise"]["median"]
        / res["kernel_ms_per_launch"]["sighted_legged_gym_noise"]["median"]}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "envs", "blind_floor_ms", "blind_share_of_peak",
                                         "blind_over_sighted_kernel")}
                     | {"kernel_median_ms": {k: v["median"] for k, v in res["kernel_ms_per_launch"].items()},
                        "step_median_ms": {k: v["median"] for k, v in res["step_ms"].items()}}))


if __name__ == "__main__":
    main()
