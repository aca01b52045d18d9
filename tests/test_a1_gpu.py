"""GPU parity tests of the A1 hot path (run with -m gpu on a B200).  Everything goes through the
C-ABI (ctypes -> libshifu_b200.so); the oracle / fixtures are only the checker.

Tolerances (BASELINE.json north_star): bit-exact reset/time-out/contact flags, reset ids,
terrain levels, episode lengths and height-cell indices (hence measured_heights);
rtol 1e-5 (+ atol 1e-6) for obs, rewards, episode sums, torques, extras.
"""
import numpy as np
import pytest
import torch

from tests import util

pytestmark = pytest.mark.gpu


import functools


@functools.lru_cache(maxsize=4)
def _terrain(n):
    from shifu_b200.sim import fake_isaacgym
    fake_isaacgym.install("cpu")
    from shifu_b200.configs import TerrainEnvConfig
    from shifu_b200.utils.heightmap import Terrain
    np.random.seed(0)
    cfg = TerrainEnvConfig()
    ter = Terrain(cfg.terrain, n)
    types = torch.div(torch.arange(n), (n / cfg.terrain.num_cols), rounding_mode='floor').to(torch.long)
    origins = torch.from_numpy(ter.env_origins).float()
    levels0 = torch.from_numpy(np.random.RandomState(3).randint(0, 6, size=n))
    env_origins = origins[levels0, types]
    return ter.heightsamples, origins, types, env_origins


def _replay_golden(name, carry):
    z, meta = util.load_golden(name)
    n = meta["n"]
    if "height_samples" in z.files:
        hs = z["height_samples"]
    else:
        hs = _terrain(n)[0]
    hp = util.make_cuda_a1(n, hs, z["terrain_origins"], z["terrain_types"], z["env_origins_init"],
                           border_size=meta["border_size"], max_terrain_level=meta["max_terrain_level"],
                           num_cols=meta["num_cols"], rng_seed=meta["rng_seed"], carry=carry)
    # record 0 = env.reset(): reset_idx(all) at step counter 0, then a zero-action step
    hp.reset_idx(None)
    if carry:
        hp.body_frame()
    snap = util.golden_snap(z, 0)
    util.cuda_a1_step(hp, snap, torch.zeros(n, 12))
    skip = ("base_lin_vel", "base_ang_vel", "projected_gravity") if carry else ()
    util.compare_a1(util.cuda_a1_outputs(hp), util.golden_out(z, 0), f"{name}/reset", skip=skip)
    hp.ep_len.copy_(torch.from_numpy(z["ep_len_init"]))
    hp.terrain_levels.copy_(torch.from_numpy(z["levels_init"]))
    hp.sync_level_sum()
    for t in range(1, meta["steps"] + 1):
        snap = util.golden_snap(z, t)
        util.cuda_a1_step(hp, snap, snap.actions)
        got = util.cuda_a1_outputs(hp)
        util.compare_a1(got, util.golden_out(z, t), f"{name}/s{t}", skip=skip)
        assert np.array_equal(got["reset_ids"], z[f"s{t}/reset_ids"]), f"reset ids differ at step {t}"
    return z, meta, hp


@pytest.mark.parametrize("carry", [False, True])
def test_golden_a1_small(carry):
    z, meta, hp = _replay_golden("a1_small", carry)


@pytest.mark.parametrize("carry", [False, True])
def test_golden_a1_fullmap(carry):
    _replay_golden("a1_fullmap", carry)


@pytest.mark.parametrize("n", [1, 33, 1000, 4096, 32 * 1200 + 7])
def test_oracle_parity_random(n):
    """Fresh seeded inputs, default 1300x2100 map, ragged sizes; oracle (CPU) vs CUDA.
    The largest size gives every persistent CTA several tiles (shared-memory buffer reuse in the
    TMA pipeline) plus a ragged tail handled by the barrier-phased kernel."""
    from oracle import shifu_oracle as so
    from shifu_b200.sim.synthetic import a1_snapshot
    hs, origins, types, env_origins = _terrain(n)
    p, st = util.make_oracle_a1(n, hs, origins, types, env_origins)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins)
    ep = torch.from_numpy(np.random.RandomState(n).randint(0, 500, size=n))
    lv = torch.from_numpy(np.random.RandomState(n + 1).randint(0, 10, size=n))
    kw = dict(p_base=0.05)
    so.a1_reset(p, st, a1_snapshot(77, 0, n, **kw))
    hp.reset_idx(None)
    util.cuda_a1_step(hp, a1_snapshot(77, 0, n, **kw), torch.zeros(n, 12))
    util.compare_a1(util.cuda_a1_outputs(hp), util.oracle_a1_outputs(st), f"n{n}/reset")
    st.ep_len[:] = ep
    st.terrain_levels[:] = lv
    hp.ep_len.copy_(ep)
    hp.terrain_levels.copy_(lv)
    hp.sync_level_sum()
    for t in range(1, 4):
        snap = a1_snapshot(77, t, n, **kw)
        so.a1_step(p, st, snap.actions, snap)
        util.cuda_a1_step(hp, snap, snap.actions)
        got = util.cuda_a1_outputs(hp)
        util.compare_a1(got, util.oracle_a1_outputs(st), f"n{n}/s{t}")
        assert np.array_equal(got["reset_ids"], st.reset_ids.numpy())


def test_height_cell_indices_bit_exact():
    """Row a5 stand-alone: 65 536 envs x 187 points, clipped (px, py) and heights vs the oracle."""
    from oracle import shifu_oracle as so
    from shifu_b200.sim.synthetic import a1_snapshot
    n = 65536
    hs, origins, types, env_origins = _terrain(n)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins)
    snap = a1_snapshot(5, 1, n)
    root = snap.root_offset.clone()
    root[:, :3] += env_origins
    hp.root_state.copy_(root.cuda())
    idx = torch.zeros(n * 187, 2, dtype=torch.int32, device="cuda")
    mh = hp.get_heights(cell_idx=idx)
    p = so.A1Params(n=n)
    want, widx = so.get_heights(p, root[:, :7], torch.from_numpy(hs), p.height_points(), return_idx=True)
    assert torch.equal(idx[:, 0].cpu().long(), widx[0]) and torch.equal(idx[:, 1].cpu().long(), widx[1])
    assert torch.equal(mh.cpu(), want)


@pytest.mark.parametrize("n", [1, 31, 33, 4096 + 17, 65536])
def test_get_heights_fast_path_matches_oracle(n):
    """shifu_get_heights without the cell-index output takes the packed pair-rotation kernel
    (csrc/scan_pairs.cuh): heights bit-identical to the oracle and to the scalar kernel, ragged sizes and
    robots pushed off the map included."""
    from oracle import shifu_oracle as so
    from shifu_b200.sim.synthetic import a1_snapshot
    hs, origins, types, env_origins = _terrain(n)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins)
    root = a1_snapshot(7, 2, n).root_offset.clone()
    root[:, :3] += env_origins
    root[::7, 0] -= 300.0                                   # off the map: indices clip to 0 ...
    root[3::11, 1] += 500.0                                 # ... and to the last cell
    hp.root_state.copy_(root.cuda())
    fast = hp.get_heights(out=torch.full((n, 187), -7.0, device="cuda")).cpu()
    idx = torch.zeros(n * 187, 2, dtype=torch.int32, device="cuda")
    slow = hp.get_heights(out=torch.zeros(n, 187, device="cuda"), cell_idx=idx).cpu()
    p = so.A1Params(n=n)
    want = so.get_heights(p, root[:, :7], torch.from_numpy(hs), p.height_points())
    assert torch.equal(fast, want) and torch.equal(slow, want)


def test_pd_torque_and_body_frame():
    from oracle import shifu_oracle as so
    from shifu_b200.sim.synthetic import a1_snapshot
    n = 5000
    hs, origins, types, env_origins = _terrain(n)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins)
    snap = a1_snapshot(9, 2, n)
    p = so.A1Params(n=n)
    hp.dof_state.view(n, 12, 2).copy_(snap.dof[0].cuda())
    hp.pd_torque(snap.actions.cuda().contiguous())
    act = torch.clip(snap.actions * 0.5, -1, 1)
    want = so.a1_pd_torque(p, act, snap.dof[0].reshape(-1, 2).clone())
    util.assert_close("actions", hp.actions.cpu().numpy(), act.numpy(), exact=True)
    util.assert_close("torques", hp.torques.cpu().numpy(), want.numpy(), exact=False)
    hp.root_state.copy_(snap.root_offset.cuda())
    hp.body_frame()
    lin, ang, pg, g = so.body_frame(snap.root_offset)
    util.assert_close("lin", hp.base_lin_vel.cpu().numpy(), lin.numpy(), exact=False)
    util.assert_close("ang", hp.base_ang_vel.cpu().numpy(), ang.numpy(), exact=False)
    util.assert_close("pg", hp.projected_gravity.cpu().numpy(), pg.numpy(), exact=False)


@pytest.mark.parametrize("n,p", [(1, 1.0), (31, 0.5), (4096, 0.01), (4097, 0.3), (100003, 0.0), (100003, 1.0),
                                 (1 << 20, 0.012)])
def test_compaction_matches_nonzero(n, p):
    """Row a8: ascending int64 ids == reset_buf.nonzero().flatten() (env.py:101), any size/density."""
    hs, origins, types, env_origins = _terrain(64)
    from shifu_b200 import hotpath, _native as nv
    hp = util.make_cuda_a1(max(n, 64), np.zeros((4, 4), np.int16), origins, torch.zeros(max(n, 64), dtype=torch.long),
                           torch.zeros(max(n, 64), 3))
    g = torch.Generator().manual_seed(n)
    flags = (torch.rand(n, generator=g) < p)
    dflags = flags.cuda()
    ids = torch.full((n,), -1, dtype=torch.long, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    for _ in range(3):      # repeated launches re-arm the ticket / epoch correctly
        nv.check(hp.lib.shifu_compact_reset_ids(hp.ctx.handle, nv.ptr(dflags), n, nv.ptr(ids), nv.ptr(cnt),
                                                nv.current_stream()))
    want = flags.nonzero(as_tuple=False).flatten()
    assert int(cnt.item()) == want.numel()
    assert torch.equal(ids[: want.numel()].cpu(), want)


def test_history_add_and_clip():
    from shifu_b200 import _native as nv
    hp = util.make_cuda_a1(64, np.zeros((4, 4), np.int16), torch.zeros(1, 1, 3), torch.zeros(64, dtype=torch.long),
                           torch.zeros(64, 3))
    n, a, h = 1001, 12, 3
    hist = torch.randn(n, a, h)
    x = torch.randn(n, a)
    want = hist.clone()
    want[..., 1:] = want[..., :-1].clone()     # shifu/utils/train.py:12-14
    want[..., 0] = x
    dh, dx = hist.cuda(), x.cuda()
    nv.check(hp.lib.shifu_history_add(hp.ctx.handle, nv.ptr(dh), nv.ptr(dx), n, a, h, nv.current_stream()))
    assert torch.equal(dh.cpu(), want)
    v = torch.randn(100003) * 200
    dv = v.cuda()
    out = torch.empty_like(dv)
    nv.check(hp.lib.shifu_clip(hp.ctx.handle, nv.ptr(dv), nv.ptr(out), v.numel(), 100.0, nv.current_stream()))
    assert torch.equal(out.cpu(), torch.clip(v, -100, 100))


def test_exact_division_variant_matches_oracle():
    """horizontal_scale != 0.1 takes the IEEE-division instantiation of the kernels (EXACT_DIV)."""
    from oracle import shifu_oracle as so
    from shifu_b200.sim.synthetic import a1_snapshot
    n = 32 * 9 + 5
    hs, origins, types, env_origins = _terrain(n)
    p, st = util.make_oracle_a1(n, hs, origins, types, env_origins, horizontal_scale=0.13)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, horizontal_scale=0.13)
    so.a1_reset(p, st, a1_snapshot(5, 0, n, p_base=0.05))
    hp.reset_idx(None)
    util.cuda_a1_step(hp, a1_snapshot(5, 0, n, p_base=0.05), torch.zeros(n, 12))
    for t in range(1, 3):
        snap = a1_snapshot(5, t, n, p_base=0.05)
        so.a1_step(p, st, snap.actions, snap)
        util.cuda_a1_step(hp, snap, snap.actions)
        util.compare_a1(util.cuda_a1_outputs(hp), util.oracle_a1_outputs(st), f"hscale0.13/s{t}")


def test_without_terrain_curriculum_matches_oracle():
    """cfg.terrain.curriculum = False (a1_conditional.py:117-118): resets keep level and origin."""
    from oracle import shifu_oracle as so
    from shifu_b200.sim.synthetic import a1_snapshot
    n = 32 * 11 + 7
    hs, origins, types, env_origins = _terrain(n)
    p, st = util.make_oracle_a1(n, hs, origins, types, env_origins, curriculum=False)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, curriculum=False)
    so.a1_reset(p, st, a1_snapshot(8, 0, n, p_base=0.2))
    hp.reset_idx(None)
    util.cuda_a1_step(hp, a1_snapshot(8, 0, n, p_base=0.2), torch.zeros(n, 12))
    for t in range(1, 4):
        snap = a1_snapshot(8, t, n, p_base=0.2)
        so.a1_step(p, st, snap.actions, snap)
        util.cuda_a1_step(hp, snap, snap.actions)
        util.compare_a1(util.cuda_a1_outputs(hp), util.oracle_a1_outputs(st), f"no-curriculum/s{t}")
    assert int(st.reset.sum()) > 0 and int(st.terrain_levels.abs().sum()) == 0


def test_asymmetric_point_grid_matches_oracle():
    """The pipelined kernel rotates once per point PAIR, which needs measured_points symmetric about the
    base; any other 17x11 grid (here: shifted forward, uneven rows) must be routed to the phased kernel
    and still match the oracle cell for cell."""
    from oracle import shifu_oracle as so
    from shifu_b200.sim.synthetic import a1_snapshot
    n = 32 * 6 + 3
    hs, origins, types, env_origins = _terrain(n)
    px = [round(-0.6 + 0.1 * i, 3) for i in range(17)]            # -0.6 .. 1.0: looks further ahead
    py = [-0.5, -0.4, -0.3, -0.2, -0.1, 0., 0.1, 0.25, 0.4, 0.55, 0.7]
    p, st = util.make_oracle_a1(n, hs, origins, types, env_origins, points_x=px, points_y=py)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, points_x=px, points_y=py)
    so.a1_reset(p, st, a1_snapshot(6, 0, n, p_base=0.05))
    hp.reset_idx(None)
    util.cuda_a1_step(hp, a1_snapshot(6, 0, n, p_base=0.05), torch.zeros(n, 12))
    for t in range(1, 3):
        snap = a1_snapshot(6, t, n, p_base=0.05)
        so.a1_step(p, st, snap.actions, snap)
        util.cuda_a1_step(hp, snap, snap.actions)
        util.compare_a1(util.cuda_a1_outputs(hp), util.oracle_a1_outputs(st), f"asym-grid/s{t}")


def _instantiations_agree(monkeypatch, term_kw, snap_kw):
    from shifu_b200.sim.synthetic import a1_snapshot
    n = 32 * 40 + 9
    hs, origins, types, env_origins = _terrain(n)

    def run(**kw):
        hp = util.make_cuda_a1(n, hs, origins, types, env_origins, **kw, **term_kw)
        hp.reset_idx(None)
        util.cuda_a1_step(hp, a1_snapshot(9, 0, n, **snap_kw), torch.zeros(n, 12))
        hp.ep_len.copy_(torch.from_numpy(np.random.RandomState(1).randint(0, 500, size=n)))
        outs = []
        for t in range(1, 4):
            snap = a1_snapshot(9, t, n, **snap_kw)
            util.cuda_a1_step(hp, snap, snap.actions)
            outs.append(util.cuda_a1_outputs(hp))
        return outs

    base = run()
    lean = run(want_measured_heights=False)
    monkeypatch.setenv("SHIFU_A1_KERNEL", "phased")
    phased = run()
    for t, (a, b, c) in enumerate(zip(base, lean, phased), 1):
        assert "measured_heights" in a and "measured_heights" not in b
        assert "swing_time" in a and "last_contacts" in a
        for k, v in a.items():
            if k in b:
                assert np.array_equal(v, b[k]), f"no-measured-heights instantiation differs: {k} step {t}"
            assert np.array_equal(v, c[k]), f"phased kernel differs: {k} step {t}"


def test_kernel_instantiations_agree(monkeypatch):
    """The pipelined kernel with / without measured_heights and the barrier-phased kernel are the
    same function: bit-identical outputs on the same inputs (the bench runs without
    measured_heights, the parity tests with)."""
    _instantiations_agree(monkeypatch, {}, dict(p_base=0.05))


@pytest.mark.parametrize("terms", ["L1", "L2"])
def test_kernel_instantiations_agree_term_lists(monkeypatch, terms):
    """The same for the legged_gym-style term lists (tests/util.py::term_list): the HAS_EXTRA
    instantiation of the pipelined kernel; L2 carries the feet-air-time state, compared too.  Legs touch
    more often (p_leg) so the feet land."""
    _instantiations_agree(monkeypatch, util.term_list(terms), dict(p_base=0.05, p_leg=0.3))


def test_full_size_properties_1m():
    """BASELINE config 3 size (1M envs): properties that need no oracle run."""
    from shifu_b200.sim.synthetic import a1_snapshot
    n = 1 << 20
    hs, origins, types, env_origins = _terrain(n)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins)
    snap = a1_snapshot(3, 1, n, gen_device="cuda", p_base=0.01)
    hp.ep_len.copy_(torch.randint(0, 500, (n,), device="cuda"))
    hp.command.uniform_(-1, 1)
    util.cuda_a1_step(hp, snap, snap.actions)
    ids = hp.reset_id_list()
    # ids == nonzero(reset_buf), ascending
    assert torch.equal(ids, hp.reset_buf.nonzero().flatten())
    # fused heights == stand-alone heights on the pre-reset pose is not recoverable after reset;
    # check non-reset envs only
    keep = ~hp.reset_buf
    mh_fused = hp.measured_heights.clone()
    mh_alone = torch.empty_like(mh_fused)
    hp.get_heights(out=mh_alone)
    assert torch.equal(mh_fused[keep], mh_alone[keep])
    # obs columns 72.. are clip((z-0.5) - h, +-1) of those heights
    want = torch.clip((hp.root_state[:, 2:3] - 0.5) - mh_fused, -1, 1)
    assert torch.equal(hp.obs_buf[:, 72:], want)
    # reset envs: ep_len 0, history = [a,0,0], dof at default, obs dof columns 0
    r = hp.reset_buf
    assert int(hp.ep_len[r].abs().sum()) == 0
    assert torch.equal(hp.history[r][..., 0], hp.actions[r]) and float(hp.history[r][..., 1:].abs().sum()) == 0
    assert float(hp.obs_buf[r][:, 12:24].abs().sum()) == 0
    # stats: n_reset and the level sum agree with the tensors
    assert int(hp.stats[8].item()) == int(r.sum())
    assert int(hp.stats[9].item()) == int(hp.terrain_levels.sum())
    # a second step with no new simulator state is deterministic (same ids)
    n1 = int(hp.n_reset.item())
    assert n1 > 0


# ---------------------------------------------------------------------------------------------
# Parity at the benchmarked sizes and instantiations (VERDICT r1: the oracle comparison stopped at
# 38 407 envs and never saw carry=True / no measured_heights or a non-zero env_offset on CUDA)
# ---------------------------------------------------------------------------------------------

def _oracle_vs_cuda_sharded(n, shards, steps, *, carry, want_heights, seed=91):
    """CUDA run over n envs against the CPU oracle run shard by shard (contiguous env ranges with
    their env_offset, so the oracle's memory stays bounded at 1 Mi envs)."""
    from oracle import shifu_oracle as so
    hs, origins, _, _ = _terrain(64)
    world = util.world_state(n, seed, steps, origins)
    types, levels0, ep0, cmd0, env_origins, snaps, root0 = world
    hp = util.world_shard_cuda(world, slice(0, n), hs, origins, carry=carry, want_heights=want_heights)
    got = []
    for t in range(1, steps + 1):
        util.cuda_a1_step(hp, snaps[t], snaps[t].actions)
        got.append(util.cuda_a1_outputs(hp))
    m = n // shards
    skip = {"base_lin_vel", "base_ang_vel", "projected_gravity"} if carry else set()
    skip |= {k for k in got[0] if k.startswith("extras/")} | {"reset_ids"}    # whole-world means / ids: below
    for s_ in range(shards):
        sl = slice(s_ * m, (s_ + 1) * m)
        p, st = util.make_oracle_a1(m, hs, origins, types[sl], env_origins[sl], env_offset=s_ * m)
        st.ep_len[:] = ep0[sl]
        st.command[:] = cmd0[sl]
        st.terrain_levels[:] = levels0[sl]
        st.root_state[:] = root0[sl]
        for t in range(1, steps + 1):
            so.a1_step(p, st, snaps[t].actions[sl], util.slice_snap(snaps[t], sl))
            want = util.oracle_a1_outputs(st)
            part = {k: (v[sl] if v.shape[:1] == (n,) else v) for k, v in got[t - 1].items()}
            part["dof_state"] = got[t - 1]["dof_state"].reshape(n, 12, 2)[sl].reshape(-1, 2)
            util.compare_a1(part, want, f"n{n}/shard{s_}/s{t}", skip=skip)
            ids = got[t - 1]["reset_ids"]
            local = ids[(ids >= s_ * m) & (ids < (s_ + 1) * m)] - s_ * m
            assert np.array_equal(local, st.reset_ids.numpy()), f"reset ids differ: shard {s_} step {t}"
    return hp, got, world


@pytest.mark.parametrize("n,shards,carry,want_heights", [
    (65536, 1, True, False),           # the benchmarked instantiation (carry, no measured_heights)
    (262144, 2, True, False),
    (262144, 2, False, True),
    (1 << 20, 8, True, False),         # BASELINE configs[2] size, benchmarked instantiation
])
def test_oracle_parity_benchmark_sizes(n, shards, carry, want_heights):
    _oracle_vs_cuda_sharded(n, shards, 2, carry=carry, want_heights=want_heights)


def test_env_offset_on_cuda():
    """Sharded layout on the CUDA path: a shard created with env_offset = r*n draws the Philox
    samples / terrain types of global envs r*n ..., so (i) the whole world matches the oracle run
    shard by shard with those offsets and (ii) four CUDA shards of the 4n-env world concatenate to
    the single 4n-env CUDA run bit for bit."""
    n, k = 8192, 4
    whole, got_w, world = _oracle_vs_cuda_sharded(n * k, k, 2, carry=True, want_heights=False, seed=17)
    hs, origins, _, _ = _terrain(64)
    snaps = world[5]
    for r in range(k):
        sl = slice(r * n, (r + 1) * n)
        hp = util.world_shard_cuda(world, sl, hs, origins, carry=True, want_heights=False)
        for t in (1, 2):
            util.cuda_a1_step(hp, util.slice_snap(snaps[t], sl), snaps[t].actions[sl])
            got = util.cuda_a1_outputs(hp)
            for key in ("obs", "rew", "reset", "time_out", "ep_len", "terrain_levels", "command", "root_state",
                        "env_origins", "history", "rand_force"):
                w = got_w[t - 1][key]
                assert np.array_equal(got[key], w[sl]), f"shard {r} step {t}: {key} differs from the 1-process run"
            ids_w = got_w[t - 1]["reset_ids"]
            assert np.array_equal(got["reset_ids"] + r * n, ids_w[(ids_w >= r * n) & (ids_w < (r + 1) * n)])


def test_two_rank_nccl_matches_one_rank(tmp_path):
    """2 ranks over NCCL (skipped on a 1-GPU box): concatenated obs / reset ids / levels and the
    all-reduced extras equal the 1-rank run."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = tmp_path / "ranks"
    out.mkdir()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29571", os.path.join(root, "tests", "nccl_two_rank_worker.py"), str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    one = np.load(out / "world1.npz")
    parts = [np.load(out / f"rank{i}.npz") for i in range(2)]
    for key in ("obs", "rew", "reset", "terrain_levels", "ep_len"):
        assert np.array_equal(np.concatenate([p[key] for p in parts]), one[key]), key
    n = parts[0]["obs"].shape[0]
    ids = np.concatenate([p["reset_ids"] + i * n for i, p in enumerate(parts)])
    assert np.array_equal(ids, one["reset_ids"])
    np.testing.assert_allclose(parts[0]["extras"], one["extras"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(parts[1]["extras"], one["extras"], rtol=1e-5, atol=1e-6)
