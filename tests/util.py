"""Shared helpers of the parity tests: fixture loading and the two step drivers
(oracle on CPU, CUDA hot path through the C-ABI) that replay the same simulator snapshots in the
reference's refresh order (SURVEY.md §3.2)."""
from __future__ import annotations

import json
import os
import types
from typing import Dict, List

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

EXACT_KEYS = ("reset", "time_out", "contact_term", "ep_len", "terrain_levels", "measured_heights", "success",
              "swing_time", "last_contacts")
RTOL, ATOL = 1e-5, 1e-6      # BASELINE.json: obs/rew within 1e-5 relative (fp32); abs floor 1e-6 (SURVEY §8d)


def load_golden(name: str):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    meta = json.loads(bytes(z["meta"]).decode())
    return z, meta


def golden_snap(z, t: int, kind: str = "a1"):
    pre = f"s{t}/in/"
    keys = ("dof", "root_offset", "contact", "actions") if kind == "a1" else ("root", "body", "dof", "actions")
    return types.SimpleNamespace(**{k: torch.from_numpy(z[pre + k].copy()) for k in keys})


def golden_out(z, t: int) -> Dict[str, np.ndarray]:
    pre = f"s{t}/out/"
    return {k[len(pre):]: z[k] for k in z.files if k.startswith(pre)}


def assert_close(name: str, got, want, exact: bool):
    got = np.asarray(got)
    want = np.asarray(want)
    assert got.shape == want.shape, f"{name}: shape {got.shape} != {want.shape}"
    if exact or got.dtype.kind in "iub":
        bad = np.flatnonzero(got.reshape(-1) != want.reshape(-1))
        assert bad.size == 0, f"{name}: {bad.size} of {got.size} entries differ (first at {bad[:5]})"
    else:
        err = np.abs(got.astype(np.float64) - want.astype(np.float64))
        tol = ATOL + RTOL * np.abs(want.astype(np.float64))
        bad = np.flatnonzero((err > tol).reshape(-1))
        assert bad.size == 0, (f"{name}: {bad.size} of {got.size} entries outside rtol={RTOL} atol={ATOL}; "
                               f"max err {err.max():.3e} at {int(err.argmax())}")


# ---------------------------------------------------------------------------------------------
# A1: oracle driver
# ---------------------------------------------------------------------------------------------

def make_oracle_a1(n, height_samples, terrain_origins, terrain_types, env_origins, *, border_size=25,
                   max_terrain_level=10, num_cols=20, rng_seed=0x5EED, env_offset=0, horizontal_scale=0.1,
                   points_x=None, points_y=None, curriculum=True, terms=None, term_params=None, **term_consts):
    """``terms``: reward-term names in list order (default: the reference's six); ``term_params``:
    name -> (p0, p1) over the reference literals; ``term_consts``: the other A1Params term constants
    (dof_pos_limits, feet_bodies, feet_contact_force, air_time_cmd_min, air_time_dt, air_time_reset)."""
    from oracle import shifu_oracle as so
    grid = {k: list(v) for k, v in (("points_x", points_x), ("points_y", points_y)) if v is not None}
    if terms is not None:
        params = {**so.A1_TERM_PARAMS, **(term_params or {})}
        term_consts["terms"] = [(k, *params[k]) for k in terms]
    if term_consts.get("dof_pos_limits") is not None:
        term_consts["dof_pos_limits"] = torch.as_tensor(term_consts["dof_pos_limits"], dtype=torch.float)
    p = so.A1Params(n=n, border_size=border_size, max_terrain_level=max_terrain_level, num_cols=num_cols,
                    rng_seed=rng_seed, env_offset=env_offset, horizontal_scale=horizontal_scale, curriculum=curriculum,
                    **grid, **term_consts)
    st = so.a1_new_state(p, torch.as_tensor(height_samples), torch.as_tensor(terrain_origins).float(),
                         torch.as_tensor(terrain_types), torch.as_tensor(env_origins).float())
    return p, st


def oracle_a1_outputs(st) -> Dict[str, np.ndarray]:
    from oracle import shifu_oracle as so
    d = dict(obs=st.obs, rew=st.rew, reset=st.reset.to(torch.uint8), time_out=st.time_out.to(torch.uint8),
             contact_term=st.contact_term.to(torch.uint8), ep_len=st.ep_len, terrain_levels=st.terrain_levels,
             env_origins=st.env_origins, command=st.command, history=st.history, actions=st.actions,
             root_state=st.root_state, dof_state=st.dof_state, dof_targets=st.dof_targets,
             rand_force=st.rand_force, torques=st.torques, base_lin_vel=st.base_lin_vel,
             base_ang_vel=st.base_ang_vel, projected_gravity=st.projected_gravity,
             measured_heights=st.measured_heights, swing_time=st.swing_time,
             last_contacts=st.last_contacts.to(torch.uint8))
    for k in st.ep_sums:
        d["ep_sum/" + k] = st.ep_sums[k]
    for k, v in st.extras.get("episode", {}).items():
        d["extras/" + k] = torch.as_tensor(v)
    if "time_outs" in st.extras:
        d["extras_time_outs"] = st.extras["time_outs"].to(torch.uint8)
    return {k: v.detach().numpy().copy() for k, v in d.items()}


# ---------------------------------------------------------------------------------------------
# A1: CUDA driver (through the C-ABI via shifu_b200.hotpath)
# ---------------------------------------------------------------------------------------------

def make_cuda_a1(n, height_samples, terrain_origins, terrain_types, env_origins, *, border_size=25.,
                 max_terrain_level=10, num_cols=20, rng_seed=0x5EED, env_offset=0, carry=False, device="cuda:0",
                 horizontal_scale=0.1, want_measured_heights=True, points_x=None, points_y=None, curriculum=True,
                 terms=None, term_params=None, **term_consts):
    """``terms`` / ``term_params`` / ``term_consts``: as for :func:`make_oracle_a1`, passed to
    ``hotpath.a1_desc`` and ``A1HotPath``."""
    from shifu_b200 import hotpath
    grid = {k: tuple(v) for k, v in (("points_x", points_x), ("points_y", points_y)) if v is not None}
    dev = torch.device(device)
    root = torch.zeros(n, 13, device=dev)
    root[:, 6] = 1.0
    dof = torch.zeros(n * 12, 2, device=dev)
    contact = torch.zeros(n * 17, 3, device=dev)
    desc = hotpath.a1_desc(n, border_size=float(border_size), max_terrain_level=max_terrain_level,
                           num_terrain_types=num_cols, rng_seed=rng_seed, env_offset=env_offset,
                           horizontal_scale=horizontal_scale, curriculum=curriculum, **grid,
                           **({} if terms is None else dict(terms=tuple(terms))), term_params=term_params,
                           **term_consts)
    hp = hotpath.A1HotPath(desc, root_state=root, dof_state=dof, contact_state=contact,
                           height_samples=torch.as_tensor(height_samples),
                           terrain_origins=torch.as_tensor(terrain_origins),
                           terrain_types=torch.as_tensor(terrain_types),
                           env_origins=torch.as_tensor(env_origins).float().to(dev).contiguous(),
                           carry_body_frame=carry, want_measured_heights=want_measured_heights,
                           **({} if terms is None else dict(terms=tuple(terms))))
    return hp


def cuda_a1_step(hp, snap, raw_actions, before_post=None):
    """One control step with the simulator refreshes interleaved exactly like the reference
    (a1_conditional.py:64-75, isaac_gym.py:139-154).  ``before_post(hp)`` runs after the last
    refresh, right before the fused post-physics kernel."""
    dev = hp.device
    n = hp.n
    dofv = hp.dof_state.view(n, 12, 2)
    raw = raw_actions.to(dev).contiguous()
    hp.pd_torque(raw)
    dofv.copy_(snap.dof[0].to(dev))
    for i in range(1, 4):
        hp.pd_torque()
        dofv.copy_(snap.dof[i].to(dev))
    if not hp.carry_body_frame:
        hp.body_frame()                              # S_prev root (D7)
    root = snap.root_offset.to(dev).clone()
    root[:, 0:3] += hp.env_origins
    hp.root_state.copy_(root)
    dofv.copy_(snap.dof[4].to(dev))
    hp.contact_state.view(n, 17, 3).copy_(snap.contact.to(dev))
    if before_post is not None:
        before_post(hp)
    hp.post_physics()
    hp.finalize()


def cuda_a1_outputs(hp) -> Dict[str, np.ndarray]:
    d = dict(obs=hp.obs_buf, rew=hp.rew_buf, reset=hp.reset_buf.to(torch.uint8),
             time_out=hp.time_out_buf.to(torch.uint8), contact_term=hp.contact_terminate_buf.to(torch.uint8),
             ep_len=hp.ep_len, terrain_levels=hp.terrain_levels, env_origins=hp.env_origins,
             command=hp.command, history=hp.history, actions=hp.actions, root_state=hp.root_state,
             dof_state=hp.dof_state, dof_targets=hp.dof_targets, rand_force=hp.rand_force,
             torques=hp.torques, base_lin_vel=hp.base_lin_vel, base_ang_vel=hp.base_ang_vel,
             projected_gravity=hp.projected_gravity, swing_time=hp.swing_time[:, :hp.desc.num_feet],
             last_contacts=hp.last_contacts[:, :hp.desc.num_feet].to(torch.uint8))
    if hp.measured_heights is not None:
        d["measured_heights"] = hp.measured_heights
    for k in hp.terms:
        d["ep_sum/" + k] = hp.ep_sums[k]
    ex = hp.extras()
    for k, v in ex["episode"].items():
        d["extras/" + k] = v
    d["extras_time_outs"] = ex["time_outs"].to(torch.uint8)
    out = {k: v.detach().cpu().numpy().copy() for k, v in d.items()}
    out["reset_ids"] = hp.reset_id_list().cpu().numpy().copy()
    return out


def compare_a1(got: Dict, want: Dict, tag: str, skip=()):
    for k, w in want.items():
        if k in skip or k not in got:
            continue
        assert_close(f"{tag}:{k}", got[k], w, exact=(k in EXACT_KEYS))


# ---------------------------------------------------------------------------------------------
# A world of n_global envs cut into contiguous shards (SURVEY.md §8e): same global initial state and
# snapshots whatever the shard layout
# ---------------------------------------------------------------------------------------------

def slice_snap(snap, sl):
    return type(snap)(dof=snap.dof[:, sl], root_offset=snap.root_offset[sl], contact=snap.contact[sl],
                      actions=snap.actions[sl])


def world_state(n_global, seed, steps, height_origins):
    """Global initial state + per-step snapshots (CPU) of a seeded world."""
    from shifu_b200 import dist as sdist
    from shifu_b200.sim.synthetic import a1_snapshot
    origins = height_origins
    types = sdist.global_terrain_types(0, n_global, n_global, 20).clamp_(max=19)
    rs = np.random.RandomState(seed)
    levels0 = torch.from_numpy(rs.randint(0, 6, size=n_global))
    ep0 = torch.from_numpy(rs.randint(0, 500, size=n_global))
    cmd0 = torch.from_numpy(rs.uniform(-1, 1, size=(n_global, 3)).astype(np.float32))
    env_origins = origins[levels0, types]
    snaps = [a1_snapshot(seed, t, n_global, p_base=0.02, offmap=False) for t in range(steps + 1)]
    root0 = snaps[0].root_offset.clone()
    root0[:, :3] += env_origins
    return types, levels0, ep0, cmd0, env_origins, snaps, root0


def world_shard_cuda(world, sl, hs, origins, *, carry, want_heights, device="cuda:0"):
    """CUDA hot path over the envs `sl` of a world (env_offset = sl.start), seeded like the world."""
    types, levels0, ep0, cmd0, env_origins, snaps, root0 = world
    n = sl.stop - sl.start
    hp = make_cuda_a1(n, hs, origins, types[sl], env_origins[sl], carry=carry, want_measured_heights=want_heights,
                      env_offset=sl.start, device=device)
    hp.ep_len.copy_(ep0[sl])
    hp.command.copy_(cmd0[sl])
    hp.terrain_levels.copy_(levels0[sl])
    hp.sync_level_sum()
    hp.root_state.copy_(root0[sl].to(hp.device))     # S_prev of the first step's body-frame velocities (D7)
    hp.body_frame()
    return hp


# ---------------------------------------------------------------------------------------------
# A1 reward terms on their own: seeded inputs with crafted edge rows, shared by the CPU test of the
# oracle and the GPU test of the kernels against oracle/a1_terms_f64.py
# ---------------------------------------------------------------------------------------------

LEG_BODIES = (2, 3, 6, 7, 10, 11, 14, 15)
# constants of the legged_gym-style terms (legged_gym's reward scales; base_height target 0.35)
EXTRA_TERM_PARAMS = {"lin_vel_z": (-2.0, 0.0), "ang_vel_xy": (-0.05, 0.0), "orientation": (-0.2, 0.0),
                     "dof_vel": (-1e-4, 0.0), "action_rate": (-0.01, 0.0), "base_height": (-1.0, 0.35),
                     "dof_pos_limits": (-10.0, 0.0), "feet_air_time": (1.0, 0.5)}


def term_list(name):
    """Non-default term lists of the fused-step tests: keyword arguments of make_cuda_a1 / make_oracle_a1.
      L1  the 8-term legged_gym-style list (opcodes 0, 10, 8, 9, 11, 12, 13, 5)
      L2  the stateful list: feet_air_time + dof_pos_limits (limits the synthetic dofs cross)
      L3  the reference's six terms with edited constants: tracking p1 not a power of two, leg threshold 0.37"""
    if name == "L1":
        terms = ("tracking_lin_vel", "orientation", "lin_vel_z", "ang_vel_xy", "dof_vel", "action_rate", "base_height",
                 "torques_penalize")
        return dict(terms=terms, term_params={**EXTRA_TERM_PARAMS, "torques_penalize": (-1e-5, 0.0)})
    if name == "L2":
        terms = ("tracking_lin_vel", "tracking_ang_vel", "feet_air_time", "dof_pos_limits", "leg_collision",
                 "torques_penalize")
        return dict(terms=terms, term_params=EXTRA_TERM_PARAMS, dof_pos_limits=dof_limits())
    if name == "L3":
        return dict(terms=("tracking_lin_vel", "tracking_ang_vel", "stabilizing_base", "smoothing_action",
                           "leg_collision", "torques_penalize"),
                    term_params={"tracking_lin_vel": (1.0, 0.3), "tracking_ang_vel": (0.5, 0.15),
                                 "leg_collision": (-1.0, 0.37)})
    assert name is None
    return {}


def norm_edge_forces(thr: float, k: int, seed: int = 0):
    """fp32 force vectors whose aten fp32 norm is exactly ``thr``, one ulp above and one ulp below it:
    three (k, 3) arrays (each starts with an axis-aligned vector, then random directions)."""
    t = np.float32(thr)
    targets = (t, np.nextafter(t, np.float32(np.inf)), np.nextafter(t, np.float32(0)))
    rs = np.random.RandomState(seed)
    u = rs.normal(size=(4096, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    out = []
    for tg in targets:
        cand = (u * float(tg))[:, None, :] * (1 + np.arange(-6, 7)[None, :, None] * 2.0 ** -24)
        cand = cand.reshape(-1, 3).astype(np.float32)
        nrm = torch.norm(torch.from_numpy(cand), dim=-1).numpy()
        hit = cand[nrm == tg]
        # the smallest and largest fp32 sum of squares (fma-accumulated, like aten) of the hits come first:
        # a kernel that tests |F| > thr on the sum of squares meets its own threshold at one of them
        x, y, z = (hit[:, i].astype(np.float64) for i in range(3))
        ss = (z * z + (y * y + (x * x).astype(np.float32)).astype(np.float32)).astype(np.float32)
        order = np.argsort(ss, kind="stable")
        axis = np.array([[tg, 0, 0], [0, -tg, 0], [0, 0, tg]], np.float32)
        sel = np.concatenate([axis, hit[order[:1]], hit[order[-1:]], hit])[:k]
        assert len(sel) == k and np.all(torch.norm(torch.from_numpy(sel), dim=-1).numpy() == tg)
        out.append(sel)
    return out


def dof_limits():
    """(12, 2) soft dof limits around the default pose, tight enough that the synthetic dofs
    (q0 + 0.3 N(0,1)) cross them; fp32 values."""
    from oracle import shifu_oracle as so
    q0 = so.A1Params(n=1).q0.numpy()
    return np.stack([q0 - np.float32(0.35), q0 + np.float32(0.4)], axis=1).astype(np.float32)


def term_inputs(n, seed, *, leg_thr=0.1, limits=None, feet=(4, 8, 12, 16), feet_thr=1.0, cmd_min=0.1):
    """Seeded fp32 inputs of the A1 reward terms (the dict layout of oracle.a1_terms_f64) with crafted
    rows cycling over the envs:
      * one leg body per env with a force whose fp32 norm is exactly ``leg_thr`` or one ulp either side;
      * dof positions exactly at ``limits`` lo / hi, one ulp past them and one ulp inside;
      * feet_air_time: swing_time 0, |cmd_xy| exactly ``cmd_min`` and one ulp either side, foot F_z
        exactly ``feet_thr`` and one ulp either side, last_contacts set and clear."""
    rs = np.random.RandomState(seed)
    f = lambda *shape: rs.normal(size=shape).astype(np.float32)
    from oracle import shifu_oracle as so
    q0 = so.A1Params(n=1).q0.numpy()
    s = dict(command=rs.uniform(-1, 1, size=(n, 3)).astype(np.float32), lin=f(n, 3), ang=f(n, 3),
             pg=(0.3 * f(n, 3)).astype(np.float32), hist=rs.uniform(-1, 1, size=(n, 12, 3)).astype(np.float32),
             act=rs.uniform(-1, 1, size=(n, 12)).astype(np.float32), tau=(20 * f(n, 12)).astype(np.float32),
             base_z=rs.uniform(0.2, 0.6, size=n).astype(np.float32))
    s["pg"][:, 2] = -1
    dof = np.empty((n, 12, 2), np.float32)
    dof[..., 0] = q0 + 0.3 * f(n, 12)
    dof[..., 1] = 2 * f(n, 12)
    hit = (rs.uniform(size=(n, 17)) < 0.5) * rs.uniform(0, 3, size=(n, 17))
    contact = (f(n, 17, 3) * hit[..., None]).astype(np.float32)
    nf = len(feet)
    swing = (rs.randint(0, 30, size=(n, nf)) * np.float32(0.02)).astype(np.float32)
    last = rs.uniform(size=(n, nf)) < 0.5
    e = np.arange(n)
    # leg forces at the threshold
    edges = norm_edge_forces(leg_thr, max(4, n // 8 + 1), seed)
    kind, which = e % 3, (e // 3) % len(edges[0])
    for i in range(n):
        contact[i, LEG_BODIES[i % 8]] = edges[kind[i]][which[i]]
    # dof positions at the limits
    if limits is not None:
        lo, hi = np.asarray(limits, np.float32)[:, 0], np.asarray(limits, np.float32)[:, 1]
        up, dn = np.float32(np.inf), np.float32(-np.inf)
        cands = (lo, hi, np.nextafter(lo, dn), np.nextafter(hi, up), np.nextafter(lo, up), np.nextafter(hi, dn))
        for i in range(n):
            d = i % 12
            dof[i, d, 0] = cands[(i // 12) % 6][d]
            dof[i, (d + 5) % 12, 0] = cands[(i // 12 + 1) % 6][(d + 5) % 12]
    # feet-air-time edges
    t, c = np.float32(feet_thr), np.float32(cmd_min)
    fz = (t, np.nextafter(t, np.float32(np.inf)), np.nextafter(t, np.float32(0)))
    cm = (c, np.nextafter(c, np.float32(np.inf)), np.nextafter(c, np.float32(0)))
    for i in range(n):
        contact[i, feet[i % nf], 2] = fz[i % 3]
        if i % 4 == 1:
            swing[i, (i // 4) % nf] = 0
        if i % 5 == 2:
            s["command"][i, :2] = (cm[(i // 5) % 3], 0) if (i // 15) % 2 == 0 else (0, -cm[(i // 5) % 3])
    s.update(dof=dof, contact=contact, swing=swing, last=last)
    return s


def term_consts(limits=None, feet=(4, 8, 12, 16), feet_thr=1.0, cmd_min=0.1, air_dt=0.02):
    """The constants oracle.a1_terms_f64.eval_terms_f64 takes (defaults = hotpath.a1_desc's)."""
    from oracle import shifu_oracle as so
    big = np.float32(so.A1_DOF_UNBOUNDED)
    lim = np.asarray(limits, np.float32) if limits is not None else np.array([[-big, big]] * 12, np.float32)
    return dict(leg_bodies=LEG_BODIES, dof_lo=lim[:, 0], dof_hi=lim[:, 1], feet=tuple(feet), feet_thr=feet_thr,
                air_cmd_min=cmd_min, air_dt=air_dt)


def oracle_term_state(p, s):
    """An oracle A1State holding the term inputs ``s`` (fp32 copies)."""
    from oracle import shifu_oracle as so
    n = p.n
    st = so.a1_new_state(p, torch.zeros(2, 2, dtype=torch.int16), torch.zeros(1, 1, 3),
                         torch.zeros(n, dtype=torch.long), torch.zeros(n, 3))
    t = lambda k: torch.from_numpy(np.ascontiguousarray(s[k])).clone()
    st.command, st.base_lin_vel, st.base_ang_vel, st.projected_gravity = t("command"), t("lin"), t("ang"), t("pg")
    st.dof_state = t("dof").reshape(n * 12, 2)
    st.history, st.actions, st.torques = t("hist"), t("act"), t("tau")
    st.contact_state = t("contact").reshape(n * 17, 3)
    st.root_state[:, 2] = t("base_z")
    st.swing_time, st.last_contacts = t("swing"), t("last")
    return st
