"""Where the flagship step's time goes, launch by launch.

    python tools/step_launches.py --out DIR [--label NAME] [--envs N] [--steps K] [--warmup W]

Builds the benchmark's A1 env (``bench.build_a1``, resident state, 1 Mi envs by default), runs W
warm-up steps through ``A1HotPath.step_resident`` and then times K steps eagerly with a CUDA event
between every launch: PD substeps 0-3, (body frame when it is not carried,) the fused post-physics
kernel and the finalize tail (id compaction, statistics collect and publish).  The host enqueues
faster than the device drains, so the device never waits for the host and each interval is one
launch plus its launch gap.  The graph step (``graph_step``, one replay per step, no events inside)
is timed in a separate loop.  Medians go to DIR/step_launches[_NAME].json with the card's name and
power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_info():
    """Name, power limit and max SM clock of cuda:0 (read-only query)."""
    q = "name,power.limit,clocks.max.sm,driver_version"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        vals = [v.strip() for v in r.stdout.strip().split(",")]
        return dict(zip(q.split(","), vals)) if r.returncode == 0 and len(vals) == 4 else {"error": r.stderr.strip()}
    except (OSError, subprocess.TimeoutExpired) as exc:
        return {"error": str(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--label", default="", help="suffix of the output file name")
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--decimation", type=int, default=4)
    args = ap.parse_args()

    import torch
    import bench
    if not torch.cuda.is_available():
        raise SystemExit("step_launches.py: no CUDA device")
    hp, raw = bench.build_a1(args.envs, 0, 1, "cuda:0")
    dec = args.decimation

    for _ in range(args.warmup):
        hp.step_resident(raw, dec)
    torch.cuda.synchronize()

    names = [f"pd_substep_{i}" for i in range(dec)]
    if not hp.carry_body_frame:
        names.append("body_frame")
    names += ["fused_post_physics", "finalize_tail"]
    per = {k: [] for k in names}
    steps = []
    ev = lambda: torch.cuda.Event(enable_timing=True)
    for _ in range(args.steps):
        marks = [ev()]
        marks[-1].record()
        hp.pd_torque(raw)
        marks.append(ev()); marks[-1].record()
        for _ in range(dec - 1):
            hp.pd_torque()
            marks.append(ev()); marks[-1].record()
        if not hp.carry_body_frame:
            hp.body_frame()
            marks.append(ev()); marks[-1].record()
        hp.post_physics()
        marks.append(ev()); marks[-1].record()
        hp.compact()
        hp._collect(False)
        hp._publish(None)
        marks.append(ev()); marks[-1].record()
        steps.append(marks)
    torch.cuda.synchronize()
    for marks in steps:
        for k, a, b in zip(names, marks[:-1], marks[1:]):
            per[k].append(a.elapsed_time(b) * 1e3)
    eager_step = [m[0].elapsed_time(m[-1]) * 1e3 for m in steps]

    for _ in range(args.warmup + 3):           # the first calls capture the graph
        hp.graph_step(raw, dec)
    torch.cuda.synchronize()
    t0, t1 = ev(), ev()
    t0.record()
    for _ in range(args.steps):
        hp.graph_step(raw, dec)
    t1.record()
    torch.cuda.synchronize()
    graph_us = t0.elapsed_time(t1) * 1e3 / args.steps

    med = {k: statistics.median(v) for k, v in per.items()}
    res = {
        "label": args.label, "gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0),
        "envs": args.envs, "steps": args.steps, "warmup": args.warmup, "decimation": dec,
        "unit": "us",
        "median_us": med,
        "min_us": {k: min(v) for k, v in per.items()},
        "eager_step_median_us": statistics.median(eager_step),
        "sum_of_launch_medians_us": sum(med.values()),
        "graph_step_us": graph_us,
        "note": "eager: CUDA events between the launches of each step; graph: one replay per step, no events inside",
    }
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, f"step_launches{'_' + args.label if args.label else ''}.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"label": args.label, "graph_step_us": round(graph_us, 2),
                      "median_us": {k: round(v, 2) for k, v in med.items()}}))


if __name__ == "__main__":
    main()
