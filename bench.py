#!/usr/bin/env python
"""Benchmark of the shifu post-physics hot path (BASELINE.json metric: env-steps/s + % HBM roofline).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, sm_100a)
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                   # + what the last timed step returned, as DIR/*.npy

A "step" = one control step of a1_conditional on resident simulator state:
PD torque x4 (+ action scale/clip), fused post-physics (body-frame carry, 187-point height scan,
termination, 6 reward terms + episode sums, reset with Philox draws, obs, history push, clips),
reset-id compaction, statistics collect (+ all-reduce over ranks when N>1) and extras publish.
Prints ONE JSON line on rank 0.  See DESIGN.md §Measurement for the definitions.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env-steps/sec (obs+reward+term+reset)"
UNIT = "env-steps/s"
B_ALG_POST = 1819          # algorithmic HBM bytes / env-step of the fused post-physics kernel (SURVEY §8d)
B_ALG_PD = 192             # per PD substep: 96 dof_state + 48 action read, 48 torque write
ENVS_PER_GPU = 1 << 20     # BASELINE configs[2]/[4]: 1M envs per B200 (weak scaling -> 8M on 8 GPUs)
SWEEP = (4096, 16384, 65536, 262144)


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i] == "Active"})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# workload construction
# ---------------------------------------------------------------------------------------------

def _terrain():
    import numpy as np
    from shifu_b200.sim import fake_isaacgym
    fake_isaacgym.install("cpu")
    from shifu_b200.configs import TerrainEnvConfig
    from shifu_b200.utils.heightmap import Terrain
    np.random.seed(0)
    cfg = TerrainEnvConfig()
    return Terrain(cfg.terrain, 1), cfg


def build_env(n_local, rank, world, device, seed=1234, store_heights=False, use_graph=True):
    """The product's class API (shifu_b200.tasks.a1_walking.A1Conditional — the counterpart of the
    reference's example class — over ShifuVecEnv / TerrainGymEnv / LeggedRobot) on the stand-in
    simulator with synthetic state RESIDENT in HBM (no snapshot provider: what the hot path sees between
    two PhysX steps).  Global env ids rank*n_local ... feed terrain types and Philox counters (§8e)."""
    import numpy as np
    import torch
    from shifu_b200.sim import fake_isaacgym
    fake_isaacgym.install(device)
    fake_isaacgym.reset_gym()
    fake_isaacgym.set_default_device(device)
    from shifu_b200.sim.synthetic import a1_snapshot
    from shifu_b200.tasks.a1_walking import A1Conditional, A1EnvConfig
    cfg = A1EnvConfig()
    cfg.num_envs, cfg.device = n_local, device
    np.random.seed(0)                       # terrain generator (host numpy, one-time init)
    torch.manual_seed(seed + rank)          # initial terrain levels
    env = A1Conditional(cfg, fused=True, carry_body_frame=True, rng_seed=seed, env_offset=rank * n_local,
                        num_envs_global=n_local * world, store_measured_heights=store_heights,
                        use_cuda_graph=use_graph)
    isg, hp = env.isg_env, env.hot
    snap = a1_snapshot(seed + rank, 1, n_local, gen_device=device, p_base=0.01, p_leg=0.1, xy_range=3.0,
                       offmap=False)
    root = snap.root_offset.clone()
    root[:, :3] += isg.env_origins
    isg.root_state.copy_(root)
    isg.dof_state.copy_(snap.dof[4].reshape(n_local * 12, 2))
    isg.contact_state.copy_(snap.contact.reshape(n_local * 17, 3))
    g = torch.Generator().manual_seed(seed + rank)
    env.episode_length_buf = torch.randint(0, 500, (n_local,), generator=g).to(device)
    env.command_buf.copy_((torch.rand(n_local, 3, generator=g) * 2 - 1).to(device))
    env.terrain_levels.copy_(isg.terrain_levels)
    hp.sync_level_sum()
    hp.body_frame()             # seed the carried body-frame velocities from the initial root rows
    raw = hp.action_input()     # the policy-output buffer of the captured step (no per-step action copy)
    raw.copy_(snap.actions)
    return env, raw


def build_a1(n_local, rank, world, device, terrain=None, seed=1234, carry=True, want_heights=False):
    """(hot path, raw actions) of build_env — for the dev tools that drive the kernels directly."""
    env, raw = build_env(n_local, rank, world, device, seed=seed, store_heights=want_heights)
    env.hot._env = env           # keep the env (and its simulator tensors) alive with the hot path
    return env.hot, raw


LAUNCHES_PER_STEP = 4 + 1 + 1 + 1 + 1      # pd x4, fused post-physics, compaction, collect, publish (libshifu_b200.so kernels;
                                           # the action copy into the graph input buffer is torch's)
DUMP_ROWS = 32768                          # envs written by --dump-outputs: 32768 x 262 floats = 34 MB


def dump_outputs(env, out_dir):
    """What ``A1Conditional.step`` returned in the last step (obs, rew, dones, extras) as float32 .npy
    files in ``out_dir``: per-env arrays for a fixed, seeded sample of DUMP_ROWS envs (all envs when
    there are fewer; ``env_ids.npy``, float64, lists them), the extras' episode statistics whole.  The inputs are
    seeded, so two builds run with the same arguments can be compared file by file."""
    import numpy as np
    import torch
    n = env.num_envs
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    idx = torch.from_numpy(rows).to(env.obs_buf.device)
    out = {"obs": env.obs_buf, "rew": env.rew_buf, "reset": env.reset_buf, "time_outs": env.extras["time_outs"]}
    out = {k: v.index_select(0, idx).float() for k, v in out.items()}
    out.update({"episode_" + k: v.float() for k, v in env.extras["episode"].items()})
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_ids.npy"), rows.astype(np.float64))
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.cpu().numpy())


def time_steps(env, raw_actions, steps, warmup, barrier=None, flush=None):
    """K control steps through ``A1Conditional.step`` (the user-facing call) on resident state.
    Returns the total device time in ms (CUDA events on the launching stream)."""
    import torch
    for _ in range(warmup):
        env.step(raw_actions)
    torch.cuda.synchronize()
    if barrier is not None:
        barrier()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if flush is None:
        t0.record()
        for _ in range(steps):
            env.step(raw_actions)
        t1.record()
        env.hot.wait_stats()                 # side-stream all-reduce of the last step (N>1)
        torch.cuda.synchronize()
        if barrier is not None:
            barrier()
        return t0.elapsed_time(t1)
    total = 0.0
    for _ in range(steps):
        flush.zero_()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        env.step(raw_actions)
        t1.record()
        t1.synchronize()
        total += t0.elapsed_time(t1)
    return total


def time_fused_kernel(hp, launches=20):
    """CUDA-event duration of the fused post-physics launch alone (the roofline's kernel), on the
    stream it is launched on; state + obs are larger than L2, so every launch streams from HBM."""
    import torch
    ms = []
    for i in range(launches + 3):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        hp.post_physics()
        b.record()
        b.synchronize()
        hp.finalize()
        if i >= 3:
            ms.append(a.elapsed_time(b))
    return ms


def measure_traffic_live(n):
    """dram__bytes_read + dram__bytes_write of one fused launch, from a one-kernel ncu capture of a
    child process (only when ncu is on PATH and profiling is permitted); None otherwise."""
    import shutil
    ncu = shutil.which("ncu")
    if ncu is None or os.environ.get("SHIFU_BENCH_NO_NCU"):
        return None, "ncu not on PATH"
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "-k",
           "regex:a1_post_physics_tma", "-s", "4", "-c", "1", "--csv", sys.executable, os.path.join(ROOT, "tools", "ncu_run.py")]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=dict(os.environ, N=str(n)))
    except (subprocess.TimeoutExpired, OSError) as exc:
        return None, f"ncu failed: {exc}"
    total = 0.0
    for line in r.stdout.splitlines():
        cells = [c.strip('"') for c in line.split('","')]
        if len(cells) > 3 and cells[-3].startswith("dram__bytes_"):
            unit, val = cells[-2], float(cells[-1].replace(",", ""))
            total += val * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(unit, 1)
    if total <= 0:
        return None, "ncu produced no dram metrics (profiling not permitted?)"
    return total, "measured live (ncu, one launch)"


def time_graph(hp, raw_actions, steps, warmup):
    """The step as CUDA-graph replays through the hot path's own graph_step (what the class API uses
    on resident state)."""
    import torch
    for _ in range(warmup + 3):
        hp.graph_step(raw_actions)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        hp.graph_step(raw_actions)
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1)


def time_abb(n, device, flush, steps=50, warmup=10):
    """BASELINE configs[3]: abb_pushbox_vision prior-stage obs/reward/reset, 65 536 envs.  ~90 B/env:
    launch-latency-bound, so env-steps/s is reported without a roofline fraction (SURVEY §8d)."""
    import torch
    from shifu_b200 import hotpath
    from shifu_b200.sim.synthetic import abb_snapshot
    snap = abb_snapshot(7, 1, n, gen_device=device)
    hp = hotpath.AbbHotPath(hotpath.abb_desc(n), root_state=snap.root.reshape(n * 4, 13).contiguous(),
                            body_state=snap.body.reshape(n * 10, 13).contiguous(),
                            dof_state=snap.dof.reshape(n * 6, 2).contiguous())
    hp.ep_len.copy_(torch.randint(0, 200, (n,), device=device))
    cube0 = hp.root_state.view(n, 4, 13)[:, 2].clone()
    for _ in range(warmup):
        hp.step_resident()
    torch.cuda.synchronize()
    total = 0.0
    for _ in range(steps):
        hp.root_state.view(n, 4, 13)[:, 2].copy_(cube0)      # undo the previous step's cube resets (untimed)
        flush.zero_()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        hp.step_resident()
        t1.record()
        t1.synchronize()
        total += t0.elapsed_time(t1)
    ms = total / steps
    # row N2 (pre-physics arm action path): action -> ee goal -> damped least-squares IK, one launch
    k = hotpath.EnvKernels(device, n)
    jac = (torch.rand(n, 9, 6, 6, device=device) * 2 - 1) * 0.6
    actions = torch.rand(n, 3, device=device) * 2 - 1
    ik = lambda: k.arm_ik(body_state=hp.body_state, num_bodies=10, ee_body=6, jacobian=jac, ee_link=5,
                          dof_state=hp.dof_state, num_dof=6, dof_targets=hp.dof_targets, actions=actions,
                          ee_velocity=0.2, dt=0.1, min_ee_pos=(-0.2, -0.2, 0.11), max_ee_pos=(0.2, 0.2, 0.14),
                          tar_quat=(0., 1., 0., 0.))
    for _ in range(warmup):
        ik()
    torch.cuda.synchronize()
    ik_total = 0.0
    for _ in range(steps):
        flush.zero_()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        ik()
        t1.record()
        t1.synchronize()
        ik_total += t0.elapsed_time(t1)
    ik_ms = ik_total / steps
    ik_bytes = 28 + 144 + 24 + 12 + 24             # ee pose, 6x6 jacobian, dof_pos, action, dof_targets
    return {"envs": n, "ms_per_step_l2_flushed": ms, "env_steps_per_s": n / (ms * 1e-3),
            "reset_fraction": float(hp.n_reset.item()) / n, "launches_per_step": 4,
            "note": "post-physics + compaction + stats; launch-latency-bound (about 90 B/env)",
            "arm_ik_ms_l2_flushed": ik_ms, "arm_ik_algorithmic_gbs": ik_bytes * n / (ik_ms * 1e-3) / 1e9,
            "arm_ik_note": "pre-physics action path (SURVEY 8f N2): goal + clamp + 6x6 damped least squares, "
                           "232 B/env algorithmic; launch-latency-bound at this size"}


def time_camera(n, device, flush, peak, steps=20, warmup=5, h=128, w=128):
    """SURVEY 8f row N4: CameraSensor.refresh_image_tensors for the reference's perceptual-stage
    camera (task_config.py:124-145: 128x128, colour normalised + depth + segmentation) as one launch."""
    import torch
    from shifu_b200 import hotpath
    k = hotpath.EnvKernels(device, n)
    color = torch.randint(0, 256, (n, h, w, 4), dtype=torch.uint8, device=device)
    depth = -torch.rand(n, h, w, device=device)
    seg = torch.randint(0, 5, (n, h, w), dtype=torch.int32, device=device)
    table = lambda t: (t.data_ptr() + torch.arange(n, dtype=torch.int64) * t[0].numel() * t.element_size()).to(device)
    args = dict(height=h, width=w, normalize_color=True,
                color=(table(color), torch.empty(n, h, w, 3, device=device)),
                depth=(table(depth), torch.empty(n, h, w, device=device)),
                seg=(table(seg), torch.empty(n, h, w, dtype=torch.int32, device=device)))
    for _ in range(warmup):
        k.camera_gather(**args)
    torch.cuda.synchronize()
    total = 0.0
    for _ in range(steps):
        flush.zero_()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        k.camera_gather(**args)
        t1.record()
        t1.synchronize()
        total += t0.elapsed_time(t1)
    ms = total / steps
    nbytes = n * h * w * (4 + 12 + 8 + 8)
    return {"envs": n, "image": f"{h}x{w} rgba+depth+seg, colour normalised", "ms_l2_flushed": ms,
            "algorithmic_gbs": nbytes / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": nbytes / (ms * 1e-3) / 1e9 / peak,
            "envs_per_s": n / (ms * 1e-3),
            "note": "one shifu_camera_gather launch replaces the reference's Python loop over the envs "
                    "(sensors.py:165-188); 32 B/pixel"}


def time_e2e(env, raw_actions, steps, warmup):
    """Same step through the public class API (``A1Conditional.step``) with HOST buffers: every step
    copies the simulator state + actions from pinned host memory and reads obs / reward / reset flags back."""
    import torch
    hp = env.hot
    n = hp.n
    pin = lambda t: torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t.cpu())
    h_root, h_dof, h_contact, h_act = pin(hp.root_state), pin(hp.dof_state), pin(hp.contact_state), pin(raw_actions)
    d_act = torch.empty_like(raw_actions)
    h_obs = torch.empty(hp.obs_buf.shape, dtype=torch.float, pin_memory=True)
    h_rew = torch.empty(n, dtype=torch.float, pin_memory=True)
    h_reset = torch.empty(n, dtype=torch.bool, pin_memory=True)
    h2d = sum(t.numel() * t.element_size() for t in (h_root, h_dof, h_contact, h_act))
    d2h = sum(t.numel() * t.element_size() for t in (h_obs, h_rew, h_reset))

    # Three streams so that the upload of step t+1 (host->device) overlaps the read-back of step t
    # (device->host) — PCIe is full duplex; events keep every buffer single-owner:
    #   in:      wait compute(t-1) done -> H2D state/actions of step t
    #   compute: wait in(t), wait out(t-1) done -> the step
    #   out:     wait compute(t) -> D2H obs / rew / reset
    s_in, s_cmp, s_out = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    ev_in, ev_cmp, ev_out = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()
    for s in (s_in, s_cmp, s_out):
        s.wait_stream(torch.cuda.current_stream())
    ev_cmp.record(s_cmp)
    ev_out.record(s_out)

    def one():
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_cmp)
            hp.root_state.copy_(h_root, non_blocking=True)
            hp.dof_state.copy_(h_dof, non_blocking=True)
            hp.contact_state.copy_(h_contact, non_blocking=True)
            d_act.copy_(h_act, non_blocking=True)
            ev_in.record(s_in)
        with torch.cuda.stream(s_cmp):
            s_cmp.wait_event(ev_in)
            s_cmp.wait_event(ev_out)
            env.step(d_act)
            ev_cmp.record(s_cmp)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_cmp)
            h_obs.copy_(hp.obs_buf, non_blocking=True)
            h_rew.copy_(hp.rew_buf, non_blocking=True)
            h_reset.copy_(hp.reset_buf, non_blocking=True)
            ev_out.record(s_out)

    for _ in range(warmup):
        one()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    torch.cuda.current_stream().wait_stream(s_cmp)
    return dt * 1e3, h2d, d2h, float(h_rew.mean())


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's torch-CPU path
# ---------------------------------------------------------------------------------------------

def cpu_oracle_rate(n, steps, warmup=1, seed=1234, shard=131072):
    """env-steps/s of oracle/shifu_oracle.py (torch CPU, all host threads) on the same synthetic
    workload, n envs per step, processed in contiguous shards of at most `shard` envs (bounded host
    memory; the envs are independent).  bench.py's only use of oracle/: the reported CPU baseline and
    the --impl reference arm."""
    import torch
    from oracle import shifu_oracle as so
    from shifu_b200.sim.synthetic import a1_snapshot
    torch.set_num_threads(os.cpu_count() or 1)
    ter, cfg = _terrain()
    origins = torch.from_numpy(ter.env_origins).float()
    hs = torch.from_numpy(ter.heightsamples)
    parts = []
    for off in range(0, n, shard):
        m = min(shard, n - off)
        gid = torch.arange(off, off + m)
        types = torch.div(gid, (n / cfg.terrain.num_cols), rounding_mode='floor').to(torch.long).clamp_(max=cfg.terrain.num_cols - 1)
        g = torch.Generator().manual_seed(seed + off)
        levels0 = torch.randint(0, cfg.terrain.max_init_terrain_level + 1, (m,), generator=g)
        p = so.A1Params(n=m, rng_seed=seed, env_offset=off)
        st = so.a1_new_state(p, hs, origins, types, origins[levels0, types])
        st.ep_len[:] = torch.randint(0, 500, (m,), generator=g)
        st.command[:] = torch.rand(m, 3, generator=g) * 2 - 1
        parts.append((p, st, p.height_points(), a1_snapshot(seed + off, 1, m, p_base=0.01, p_leg=0.1, xy_range=3.0,
                                                            offmap=False)))
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        for p, st, hpts, snap in parts:
            so.a1_step(p, st, snap.actions, snap, hpts)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return n / statistics.median(times), statistics.median(times) * 1e3, sum(times)


def run_reference(args):
    """The reference's torch-CPU path (oracle port; the reference itself is Python and does not travel to
    the GPU box) on the SAME workload as our arm: args.envs_per_gpu envs per step, all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.envs_per_gpu
    steps, warmup = max(args.steps, 1), min(args.warmup, 2)
    budget = float(os.environ.get("SHIFU_REF_BUDGET_S", "150"))
    probe_rate, probe_ms, _ = cpu_oracle_rate(65536, steps=2, warmup=1)
    est = (steps + warmup) * n / probe_rate
    sample = n
    while est > budget and sample > 65536:            # bounded run: shrink the sample, say so
        sample //= 2
        est = (steps + warmup) * sample / probe_rate
    rate, ms, spent = cpu_oracle_rate(sample, steps=steps, warmup=warmup)
    cores = os.cpu_count() or 1
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(n, 1),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample_envs": sample, "same_env_count_as_gpu_arm": sample == n,
                         "rate_65536_envs": probe_rate,
                         "sample": f"oracle/shifu_oracle.py a1_step (torch CPU restatement, bit-identical to the "
                                   f"reference), {sample} envs/step in shards of 131072, {steps} steps, median"},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)


def _config(n, world):
    return {"workload": "a1_conditional post-physics step incl. 187-pt heightfield scan + PD torques, "
                        f"{n} envs/GPU (BASELINE configs[2]; configs[4] when n_gpus=8)",
            "envs_per_gpu": n, "decimation": 4}


# ---------------------------------------------------------------------------------------------

def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the hot path has no CPU fallback; "
                         "use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    device = f"cuda:{local}"
    barrier = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(device))
        barrier = dist.barrier
    n = args.envs_per_gpu
    # the headline instantiation: class API, carried body-frame velocities, measured_heights not kept
    # (B_alg of SURVEY.md 8d excludes that optional tensor); the store-everything instantiation is
    # measured right after and reported beside it
    env, raw = build_env(n, rank, world, device, store_heights=False)
    if world > 1:
        env.stats_allreduce = lambda t: dist.all_reduce(t, op=dist.ReduceOp.SUM)
    hp = env.hot
    peak, peak_src = _peaks()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    total_ms = time_steps(env, raw, args.steps, args.warmup, barrier)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(env, args.dump_outputs)
    t = torch.tensor([total_ms], device=device, dtype=torch.double)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = n * world / (ms_per_step * 1e-3)
    kern_ms = time_fused_kernel(hp)
    kms = statistics.mean(kern_ms)
    achieved = B_ALG_POST * n / (kms * 1e-3) / 1e9
    reset_frac = float(hp.n_reset.item()) / n
    graphed = hp._graph is not None

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(_config(n, world), global_envs=n * world,
                           api="shifu_b200.tasks.a1_walking.A1Conditional.step on the stand-in simulator (resident state)",
                           instantiation="carry_body_frame=True, measured_heights not stored (HAS_MROW=0)",
                           l2="inputs larger than L2 (state + obs = %.0f MB per GPU vs 126 MB L2); no flush"
                              % ((B_ALG_POST + 4 * B_ALG_PD) * n / 1e6),
                           reset_fraction_per_step=reset_frac,
                           launch="one CUDA-graph replay per step (9 kernels)" if graphed else "direct (9 launches/step)",
                           collective="all_reduce(16 x f64) per step on a side stream" if world > 1 else "none"),
            "roofline": {"bound": "hbm", "kernel": "a1_post_physics_tma_kernel<0,0,0>", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "peak_source": peak_src, "algorithmic_bytes_per_env": B_ALG_POST,
                         "kernel_ms": kms, "kernel_share_of_step": kms / ms_per_step,
                         "step_frac": (B_ALG_POST + 4 * B_ALG_PD) * n / (ms_per_step * 1e-3) / 1e9 / peak},
            "clocks": clocks, "gpu_launches": LAUNCHES_PER_STEP * args.steps,
        }
    # ---- N=1 extras: e2e through host buffers, the other instantiation, the size sweep, the CPU baseline
    if world == 1 and args.quick:
        pass
    elif world == 1:
        e_steps = min(40, max(3, args.steps // 4))
        e_ms, h2d, d2h, _ = time_e2e(env, raw, e_steps, 2)
        line["e2e"] = {"value": n / (e_ms / e_steps * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": d2h, "ms_per_step": e_ms / e_steps,
                       "note": "A1Conditional.step with pinned host state+actions -> device, obs+rew+reset -> pinned host; "
                               "upload of step t+1 overlaps read-back of step t (3 streams); PCIe-bound"}
        if os.environ.get("SHIFU_BENCH_TRAFFIC", "1") != "0":
            tr, how = measure_traffic_live(n)
            if tr is None:
                tpath = os.path.join(ROOT, "profiles", "traffic.json")
                if os.path.exists(tpath):
                    with open(tpath) as f:
                        tr = json.load(f).get("a1_post_physics_kernel_bytes_per_launch")
                    how = f"from profiles/traffic.json ({how})"
            line["roofline"]["traffic"], line["roofline"]["traffic_source"] = tr, how
        del env, hp
        torch.cuda.empty_cache()
        # the store-everything instantiation of the class API (measured_heights kept: +748 B/env written)
        env2, raw2 = build_env(n, 0, 1, device, store_heights=True)
        tot2 = time_steps(env2, raw2, args.steps, args.warmup)
        k2 = statistics.mean(time_fused_kernel(env2.hot))
        line["with_measured_heights"] = {
            "value": n / (tot2 / args.steps * 1e-3), "ms_per_step": tot2 / args.steps, "kernel": "a1_post_physics_tma_kernel<0,1,0>",
            "kernel_ms": k2, "algorithmic_bytes_per_env": B_ALG_POST + 748,
            "frac": (B_ALG_POST + 748) * n / (k2 * 1e-3) / 1e9 / peak,
            "frac_on_1819_bytes": B_ALG_POST * n / (k2 * 1e-3) / 1e9 / peak}
        del env2
        torch.cuda.empty_cache()
        sweep = []
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
        for m in SWEEP:
            e_direct, r2 = build_env(m, 0, 1, device, use_graph=False)
            tot = time_steps(e_direct, r2, 20, 5, flush=flush)
            km = statistics.mean(time_fused_kernel(e_direct.hot, 10))
            del e_direct
            e_graph, r3 = build_env(m, 0, 1, device, use_graph=True)
            gms = time_steps(e_graph, r3, 200, 20) / 200
            sweep.append({"envs": m, "ms_per_step_l2_flushed": tot / 20, "env_steps_per_s_l2_flushed": m / (tot / 20 * 1e-3),
                          "ms_per_step_graph_l2_warm": gms, "env_steps_per_s_graph_l2_warm": m / (gms * 1e-3),
                          "fused_kernel_ms": km, "api": "A1Conditional.step"})
            del e_graph
        line["sweep"] = sweep
        line["abb_prior_stage"] = time_abb(65536, device, flush)
        line["camera_gather"] = time_camera(2048, device, flush, peak)
        if not args.no_cpu:
            rate, ms, _ = cpu_oracle_rate(262144, steps=8, warmup=1)
            rate4k, ms4k, _ = cpu_oracle_rate(4096, steps=20, warmup=3)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                                    "sample_envs": 262144, "rate_4096_envs": rate4k,
                                    "sample": "oracle a1_step (torch CPU, all cores), 262144 envs x 8 steps "
                                              f"(2 shards), median {ms:.0f} ms/step"}
    else:
        e_steps = min(40, max(3, args.steps // 4))
        e_ms, h2d, d2h, _ = time_e2e(env, raw, e_steps, 2)
        t = torch.tensor([e_ms], device=device, dtype=torch.double)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if rank == 0:
            line["e2e"] = {"value": n * world / (float(t.item()) / e_steps * 1e-3), "unit": UNIT,
                           "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
                           "ms_per_step": float(t.item()) / e_steps}
    if rank == 0:
        _emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_JSON_OUT = None


def _claim_stdout():
    """Keep stdout for the ONE JSON line: libraries that print there (e.g. NCCL's version banner)
    are sent to stderr instead."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def _emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def _count(low):
    def parse(s):
        v = int(s)
        if v < low:
            raise argparse.ArgumentTypeError(f"must be >= {low}")
        return v
    return parse


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_count(1), default=200, help="timed control steps")
    ap.add_argument("--warmup", type=_count(0), default=20, help="untimed control steps before them")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float32; "
                         "env ids float64; at most 35 MB)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--quick", action="store_true", help="timed region only (for runs under ncu)")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the CUDA path's outputs; it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
