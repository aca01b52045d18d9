"""Blind A1 tasks on the B200: the 72-column observation without the height scan.  The fused blind step
against the oracle's obs[:, :72] (phased kernel, pipelined kernel + ragged tail, the benchmarked layout),
blind == sighted on the same state for every output, both blind kernels bit for bit, a sharded run against
the single-process one, and the class API (explicit fused task, refused hooks, heights on demand;
automatic fusion of the reference class edited to be blind where the reference examples are present)."""
import numpy as np
import pytest
import torch

from tests import obs_layouts, obs_noise, util
from tests.test_dropin_gpu import needs_examples
from tests.test_reward_terms_gpu import SNAP_KW, _terrain

pytestmark = pytest.mark.gpu
SEED = 0x5EED                                       # hotpath.a1_desc's default rng_seed
BLIND = 72


def _snap(seed, t, n):
    from shifu_b200.sim.synthetic import a1_snapshot
    return a1_snapshot(seed, t, n, **SNAP_KW)


def _blind_noisy():
    """legged_gym's layout + noise without the height noise (a blind observation has no height columns)."""
    lay = obs_noise.legged_gym_noisy()
    from shifu_b200.hotpath import ObsLayout
    return ObsLayout(lay.slots, lay.scales, lay.height_scale, lay.noise, 0.0)


LAYOUTS = {"reference": lambda: None, "legged_gym": obs_layouts.legged_gym, "legged_gym_noisy": _blind_noisy}


def _oracle_obs(p, st, lay, step):
    if lay is None:
        return util.oracle_a1_outputs(st)["obs"][:, :BLIND]
    if lay.has_noise():
        return obs_noise.oracle_obs_noisy(p, st, lay, SEED, step).numpy()[:, :BLIND]
    return obs_layouts.oracle_obs(p, st, lay).numpy()[:, :BLIND]


# ---------------------------------------------------------------------------------------------
# 1. the blind fused step against the oracle's obs[:, :72]
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("n,carry,terms,kernel", [
    (33, False, None, "phased"),             # the barrier-phased kernel only (full tile + tail)
    (32 * 1200 + 7, False, "L1", None),      # pipelined blind kernel (HAS_EXTRA) + the phased kernel on the tail
    (65536, True, None, None),               # the benchmarked configuration (carried body frame)
])
def test_blind_step_vs_oracle(layout, n, carry, terms, kernel, monkeypatch, steps=3, seed=43):
    if kernel is None:
        monkeypatch.delenv("SHIFU_A1_KERNEL", raising=False)
    else:
        monkeypatch.setenv("SHIFU_A1_KERNEL", kernel)
    lay = LAYOUTS[layout]()
    kw = util.term_list(terms)
    hs, origins, types, env_origins = _terrain(n)
    p, st = util.make_oracle_a1(n, hs, origins, types, env_origins, **kw)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=carry, want_measured_heights=False, obs=lay,
                           num_obs=BLIND, **kw)
    assert hp.blind and tuple(hp.obs_buf.shape) == (n, BLIND) and hp.measured_heights is None
    from oracle import shifu_oracle as so
    snap = _snap(seed, 0, n)
    so.a1_reset(p, st, snap)
    hp.reset_idx(None)
    if carry:
        hp.body_frame()
    util.cuda_a1_step(hp, snap, torch.zeros(n, 12))
    skip = ("base_lin_vel", "base_ang_vel", "projected_gravity") if carry else ()

    def want():
        out = util.oracle_a1_outputs(st)
        out.pop("measured_heights", None)
        out["obs"] = _oracle_obs(p, st, lay, hp.step_counter)
        return out

    util.compare_a1(util.cuda_a1_outputs(hp), want(), f"blind/{layout}/n{n}/reset", skip=skip)
    ep = torch.from_numpy(np.random.RandomState(n).randint(0, 500, size=n))
    st.ep_len[:] = ep
    hp.ep_len.copy_(ep)
    resets = 0
    for t in range(1, steps + 1):
        snap = _snap(seed, t, n)
        so.a1_step(p, st, snap.actions, snap)
        util.cuda_a1_step(hp, snap, snap.actions)
        got = util.cuda_a1_outputs(hp)
        util.compare_a1(got, want(), f"blind/{layout}/n{n}/s{t}", skip=skip)
        assert np.array_equal(got["reset_ids"], st.reset_ids.numpy())
        resets += int(st.reset.sum())
    assert resets > 0                                   # not vacuous: envs reset


# ---------------------------------------------------------------------------------------------
# 2. blind == sighted on the same state, every output, bit for bit
# ---------------------------------------------------------------------------------------------

def _run(n, num_obs, lay, carry, kernel, monkeypatch, seed=11, steps=3):
    if kernel is None:
        monkeypatch.delenv("SHIFU_A1_KERNEL", raising=False)
    else:
        monkeypatch.setenv("SHIFU_A1_KERNEL", kernel)
    hs, origins, types, env_origins = _terrain(n)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=carry, want_measured_heights=False, obs=lay,
                           num_obs=num_obs)
    hp.reset_idx(None)
    outs = []
    for t in range(steps):
        snap = _snap(seed, t, n)
        util.cuda_a1_step(hp, snap, snap.actions)
        outs.append(util.cuda_a1_outputs(hp))
    monkeypatch.delenv("SHIFU_A1_KERNEL", raising=False)
    return outs


@pytest.mark.parametrize("layout", ["reference", "legged_gym_noisy"])
@pytest.mark.parametrize("carry", [False, True])
def test_blind_equals_sighted(layout, carry, monkeypatch):
    n = 32 * 400 + 9
    lay = LAYOUTS[layout]()
    if lay is not None and lay.has_noise():
        sighted_lay = obs_noise.legged_gym_noisy()      # the same head noise; its height noise lands in 72..258
    else:
        sighted_lay = lay
    blind = _run(n, BLIND, lay, carry, None, monkeypatch)
    sighted = _run(n, 259, sighted_lay, carry, None, monkeypatch)
    resets = 0
    for t, (b, s) in enumerate(zip(blind, sighted)):
        assert b.keys() == s.keys()
        for k in b:
            want = np.ascontiguousarray(s[k][:, :BLIND]) if k == "obs" else s[k]
            assert b[k].tobytes() == want.tobytes(), f"step {t}: {k}"
        resets += int(b["reset"].sum())
    assert resets > 0


# ---------------------------------------------------------------------------------------------
# 3. the pipelined and the phased blind kernels agree bit for bit
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("layout", ["reference", "legged_gym", "legged_gym_noisy"])
def test_blind_pipelined_and_phased_kernels_agree(layout, monkeypatch):
    n = 32 * 300 + 5
    lay = LAYOUTS[layout]()
    a = _run(n, BLIND, lay, True, None, monkeypatch)
    b = _run(n, BLIND, lay, True, "phased", monkeypatch)
    for t, (x, y) in enumerate(zip(a, b)):
        for k in x:
            assert x[k].tobytes() == y[k].tobytes(), f"step {t}: {k}"


def test_blind_runs_the_blind_kernels():
    from torch.profiler import ProfilerActivity, profile
    n = 32 * 100 + 3
    hs, origins, types, env_origins = _terrain(n)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=True, want_measured_heights=False,
                           num_obs=BLIND)
    hp.reset_idx(None)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        util.cuda_a1_step(hp, _snap(3, 0, n), torch.zeros(n, 12))
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if "a1_post_physics" in e.name}
    assert any("a1_post_physics_blind_kernel" in x for x in names), names
    assert not any("a1_post_physics_tma_kernel" in x for x in names), names
    assert not any("get_heights" in e.name for e in prof.events())


# ---------------------------------------------------------------------------------------------
# 4. noise is keyed by the global env id: two shards reproduce the single run
# ---------------------------------------------------------------------------------------------

def test_blind_sharded_noise_matches_the_single_run():
    n, half = 32 * 200 + 10, 32 * 100 + 3           # the first shard has a ragged tail, the second starts mid-tile
    lay = _blind_noisy()
    hs, origins, _, _ = _terrain(64)
    world = util.world_state(n, 29, 2, origins)
    types, levels0, ep0, cmd0, env_origins, snaps, root0 = world

    def shard(sl):
        m = sl.stop - sl.start
        hp = util.make_cuda_a1(m, hs, origins, types[sl], env_origins[sl], carry=True, want_measured_heights=False,
                               env_offset=sl.start, obs=lay, num_obs=BLIND)
        hp.ep_len.copy_(ep0[sl])
        hp.command.copy_(cmd0[sl])
        hp.terrain_levels.copy_(levels0[sl])
        hp.sync_level_sum()
        hp.root_state.copy_(root0[sl].to(hp.device))
        hp.body_frame()
        return hp

    parts = [slice(0, n), slice(0, half), slice(half, n)]
    hps = [shard(sl) for sl in parts]
    for t in (1, 2):
        got = []
        for hp, sl in zip(hps, parts):
            util.cuda_a1_step(hp, util.slice_snap(snaps[t], sl), snaps[t].actions[sl])
            got.append(util.cuda_a1_outputs(hp))
        for key in ("obs", "rew", "reset", "command", "history"):
            both = np.concatenate([got[1][key], got[2][key]])
            assert both.tobytes() == got[0][key].tobytes(), f"step {t}: {key}"
    assert int(got[0]["reset"].sum()) > 0


# ---------------------------------------------------------------------------------------------
# 5. the class API: a blind A1Conditional subclass, fused vs hooks; refusals
# ---------------------------------------------------------------------------------------------

def _blind_obs(self):
    """A proprioceptive-only compute_observations: the reference head without the height columns."""
    rb = self.robot
    self.obs_buf = torch.cat([self.command_buf, rb.base_lin_vel, rb.base_ang_vel, rb.gravity_vec,
                              rb.dof_pos - rb.default_dof_pos, rb.dof_vel, self.actions_recorder.flatten()], dim=1)


def _blind_obs_reading_heights(self):
    """72 columns, but the last one follows the mean terrain height under the robot."""
    _blind_obs(self)
    self.obs_buf[:, 71] = self.obs_buf[:, 71] + self.isg_env.measured_heights.mean(dim=1)


def _blind_cfg(n, terrain, measure_heights=False, store=False):
    from tests.test_env_api_gpu import _install
    _install()
    from shifu_b200.tasks.a1_walking import A1EnvConfig
    cfg = A1EnvConfig()
    cfg.num_envs, cfg.device, cfg.num_obs = n, "cuda:0", BLIND
    for k, v in (terrain or {}).items():
        setattr(cfg.terrain, k, v)
    cfg.terrain.measure_heights = measure_heights
    cfg.store_measured_heights = store
    np.random.seed(0)
    torch.manual_seed(0)
    return cfg


def _blind_task(obs_fn=_blind_obs):
    from shifu_b200.tasks.a1_walking import A1Conditional
    return type("BlindA1", (A1Conditional,), {"compute_observations": obs_fn})


def _task_outputs(env):
    """``test_env_api_gpu._env_outputs`` of a blind task, which keeps no measured heights."""
    from tests.test_env_api_gpu import _env_outputs
    isg = env.isg_env
    assert isg.measured_heights is None                 # neither mode measures heights
    isg.measured_heights = torch.zeros(1)
    try:
        out = _env_outputs(env)
    finally:
        isg.measured_heights = None
    del out["measured_heights"]
    return out


@pytest.mark.parametrize("carry", [False, True])
def test_blind_task_fused_vs_hooks(carry):
    from shifu_b200.sim.synthetic import A1Replay
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    cls = _blind_task()
    envs = [cls(_blind_cfg(n, meta["terrain"]), fused=fused, carry_body_frame=carry) for fused in (True, False)]
    assert envs[0].hot is not None and envs[0].hot.blind and envs[0].hot.desc.num_obs == BLIND
    assert envs[1].hot is None
    replays = []
    for env in envs:
        class Replay(A1Replay):
            def begin_step(self, step):
                self.snap = util.golden_snap(z, step)
                self._dof_i = 0
                self.enabled = True
                return self.snap.actions
        r = Replay(0, n, lambda env=env: env.isg_env.env_origins)
        env.isg_env.sim.provider = r
        replays.append(r)
    skip = ("base_lin_vel", "base_ang_vel", "projected_gravity") if carry else ()
    for env, r in zip(envs, replays):
        r.begin_step(0)
        env.reset()
        env.episode_length_buf = torch.from_numpy(z["ep_len_init"]).cuda()
        env.terrain_levels[:] = torch.from_numpy(z["levels_init"]).cuda()
    envs[0].hot.sync_level_sum()
    resets = 0
    for t in range(1, meta["steps"] + 1):
        outs = []
        for env, r in zip(envs, replays):
            env.step(r.begin_step(t).cuda())
            out = _task_outputs(env)
            assert out["obs"].shape == (n, BLIND)
            outs.append(out)
        util.compare_a1(outs[0], outs[1], f"blind-task/s{t}", skip=skip)
        resets += int(outs[0]["reset"].sum())
    assert resets > 0


def test_blind_task_graph_replay_vs_hooks():
    """Resident state: the fused blind task steps by CUDA-graph replay; fused=False runs the hooks."""
    n = 32 * 64 + 5
    cls = _blind_task()
    envs = [cls(_blind_cfg(n, None), fused=fused, carry_body_frame=True) for fused in (True, False)]
    for env in envs:
        env.reset()
    g = torch.Generator().manual_seed(5)
    for t in range(6):
        a = (torch.rand(n, 12, generator=g) * 2 - 1).cuda()
        outs = []
        for env in envs:
            env.step(a)
            outs.append(_task_outputs(env))
        util.compare_a1(outs[0], outs[1], f"blind-graph/s{t}",
                        skip=("base_lin_vel", "base_ang_vel", "projected_gravity"))
    assert envs[0].hot._graph is not None               # the fused steps replayed the captured graph


@pytest.mark.parametrize("grid", [((0.0,), (0.0,)), (tuple(0.1 * i for i in range(-10, 11)), (-0.5, 0.0, 0.5))])
def test_blind_task_with_another_grid_fuses(grid):
    """A blind task's measured-point grid is not read by the fused step: a config with another grid fuses
    (the 17x11 grid stays what the sighted step requires)."""
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    cls = _blind_task()

    def cfg():
        c = _blind_cfg(n, meta["terrain"])
        c.terrain.measured_points_x, c.terrain.measured_points_y = list(grid[0]), list(grid[1])
        return c

    env = cls(cfg(), fused=True)
    assert env.hot.blind and (env.hot.desc.num_points_x, env.hot.desc.num_points_y) == (17, 11)
    env.reset()
    env.step(torch.zeros(n, 12, device="cuda:0"))
    assert env.obs_buf.shape == (n, BLIND) and torch.isfinite(env.obs_buf).all()
    auto = _auto_env(_auto_blind_class(), cfg(), True)                # the automatic path fuses it too
    assert auto.fusion_report == "fused: a1", auto.fusion_report
    assert (auto.hot.desc.num_points_x, auto.hot.desc.num_points_y) == (17, 11)


def test_blind_task_refuses_store_measured_heights():
    z, meta = util.load_golden("a1_small")
    with pytest.raises(NotImplementedError, match="store_measured_heights"):
        _blind_task()(_blind_cfg(meta["n"], meta["terrain"], measure_heights=True), fused=True,
                      store_measured_heights=True)


def test_blind_task_refuses_a_hook_that_reads_heights():
    z, meta = util.load_golden("a1_small")
    cls = _blind_task(_blind_obs_reading_heights)
    with pytest.raises(NotImplementedError, match="measured_heights"):
        cls(_blind_cfg(meta["n"], meta["terrain"], measure_heights=True), fused=True)
    env = cls(_blind_cfg(meta["n"], meta["terrain"], measure_heights=True), fused=False)
    assert env.hot is None                              # user-hook mode runs it
    env.reset()
    env.step(torch.zeros(meta["n"], 12, device="cuda:0"))
    assert env.obs_buf.shape == (meta["n"], BLIND)


@pytest.mark.parametrize("measure_heights", [False, True])
def test_blind_task_measured_heights_on_demand(measure_heights):
    """A fused blind task keeps no heights; with measure_heights set the stand-alone scan fills
    isg.measured_heights on demand, otherwise it stays None as in user-hook mode."""
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    env = _blind_task()(_blind_cfg(n, meta["terrain"], measure_heights=measure_heights), fused=True)
    assert env.hot.blind and env.hot.measured_heights is None
    env.reset()
    env.step(torch.zeros(n, 12, device="cuda:0"))
    isg = env.isg_env
    if measure_heights:
        h = isg.measured_heights
        assert h is not None and tuple(h.shape) == (n, isg.num_height_points)
        assert torch.equal(h, isg.get_heights())
    else:
        assert isg.measured_heights is None


def test_blind_autofusion_refuses_store_measured_heights():
    from shifu_b200.gym import autofuse
    z, meta = util.load_golden("a1_small")
    env = _blind_task()(_blind_cfg(meta["n"], meta["terrain"], measure_heights=True, store=True), fused=False)
    with pytest.raises(autofuse.NotFusable, match="store_measured_heights"):
        autofuse.fuse_a1(env)


# ---------------------------------------------------------------------------------------------
# 6. automatic fusion of a blind ShifuVecEnv subclass (shaped like the reference task, not the reference's)
# ---------------------------------------------------------------------------------------------

def torch_rand_float(lower, upper, shape, device):
    """The draw site of the reference-shaped hooks below; the user-hook run replaces it with the kernels'
    counter-based draws (tests/test_dropin_gpu._philox_draws)."""
    return (upper - lower) * torch.rand(*shape, device=device) + lower


def _auto_blind_class(obs_fn=_blind_obs):
    """An A1Conditional subclass in user-hook mode whose reset pieces have the reference's shape
    (a1_conditional.py:43-50, 77-87, 194-221), so that automatic fusion recognises them."""
    import sys
    from shifu_b200.tasks.a1_walking import A1Conditional, A1Robot
    mod = sys.modules[__name__]

    class RefShapedA1Robot(A1Robot):
        def _reset_root_state(self, env_ids):
            rows = self.root_indices[env_ids]
            self.env.root_state[rows, :3] = self.default_base_pose[:3] + self.env.env_origins[env_ids]
            self.env.root_state[rows, :2] += mod.torch_rand_float(-1., 1., (len(env_ids), 2), self.device)
            self.env.root_state[rows, 3:7] = self.default_base_pose[3:7]
            self.env.root_state[rows, 7:] = 0.

        def reset_idx(self, env_ids):
            super(A1Robot, self).reset_idx(env_ids)
            self.rand_force_buf[env_ids, self.rigid_body_dict['base']] = mod.torch_rand_float(
                -5., 5., (len(env_ids), 3), self.device)

    class AutoBlindA1(A1Conditional):
        def __init__(self, cfg):
            super().__init__(cfg, fused=False)
            self.robot.__class__ = RefShapedA1Robot
            self.auto_fuse = True

        def sample_command(self, env_ids):
            n = len(env_ids)
            self.command_buf[env_ids, 0] = mod.torch_rand_float(*self.cmd_lin_vel_x, (n, 1), self.device).squeeze(1)
            self.command_buf[env_ids, 1] = mod.torch_rand_float(*self.cmd_lin_vel_y, (n, 1), self.device).squeeze(1)
            self.command_buf[env_ids, 2] = mod.torch_rand_float(*self.cmd_ang_vel_yaw, (n, 1), self.device).squeeze(1)

        def update_terrain_curriculum(self, env_ids):
            if not self.isg_env.init_done or len(env_ids) == 0:
                return
            dist = torch.norm(self.robot.base_pose[env_ids, :2] - self.isg_env.env_origins[env_ids, :2], dim=1)
            move_up = dist > self.isg_env.terrain.env_length / 2
            move_down = (dist < torch.norm(self.command_buf[env_ids, :2], dim=1) * self.max_episode_length_s * 0.5) \
                * ~move_up
            self.terrain_levels[env_ids] += 1 * move_up - 1 * move_down
            self.terrain_levels[env_ids] = torch.where(
                self.terrain_levels[env_ids] >= self.isg_env.max_terrain_level,
                torch.randint_like(self.terrain_levels[env_ids], self.isg_env.max_terrain_level),
                torch.clip(self.terrain_levels[env_ids], 0))
            self.isg_env.update_terrain_level(env_ids, self.terrain_levels)

    AutoBlindA1.compute_observations = obs_fn
    return AutoBlindA1


def _auto_env(cls, cfg, fuse):
    env = cls(cfg)
    env.auto_fuse = fuse
    env._maybe_fuse()
    return env


def test_blind_shifu_vec_env_autofuses_and_matches_hooks():
    import sys
    from shifu_b200.sim.synthetic import A1Replay
    from tests.test_dropin_gpu import _philox_draws
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    cls = _auto_blind_class()
    fused, hooks = (_auto_env(cls, _blind_cfg(n, meta["terrain"]), fuse) for fuse in (True, False))
    assert fused.fusion_report == "fused: a1", fused.fusion_report
    assert fused.hot.blind and fused.hot.desc.num_obs == BLIND and fused.obs_buf.shape == (n, BLIND)
    assert hooks.hot is None
    replays = []
    for env in (fused, hooks):
        class Replay(A1Replay):
            def begin_step(self, step):
                self.snap = util.golden_snap(z, step)
                self._dof_i = 0
                self.enabled = True
                return self.snap.actions
        r = Replay(0, n, lambda env=env: env.isg_env.env_origins)
        env.isg_env.sim.provider = r
        replays.append(r)
    seed = getattr(hooks.cfg, "rng_seed", 0x5EED)
    with _philox_draws(sys.modules[__name__], hooks, seed):
        for env, r in zip((fused, hooks), replays):
            r.begin_step(0)
            env.reset()
            env.episode_length_buf = torch.from_numpy(z["ep_len_init"]).cuda()
            env.terrain_levels[:] = torch.from_numpy(z["levels_init"]).cuda()
        fused.hot.sync_level_sum()
        resets = 0
        for t in range(1, meta["steps"] + 1):
            outs = []
            for env, r in zip((fused, hooks), replays):
                env.step(r.begin_step(t).cuda())
                outs.append(_task_outputs(env))
            util.compare_a1(outs[0], outs[1], f"auto-blind/s{t}",
                            skip=("base_lin_vel", "base_ang_vel", "projected_gravity"))
            resets += int(outs[0]["reset"].sum())
    assert resets > 0


def test_blind_shifu_vec_env_refusals():
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    env = _auto_env(_auto_blind_class(_blind_obs_reading_heights),
                    _blind_cfg(n, meta["terrain"], measure_heights=True), True)
    assert env.hot is None and env.fusion_report.startswith("user-hook mode"), env.fusion_report
    assert "measured_heights" in env.fusion_report, env.fusion_report
    env.reset()
    env.step(torch.zeros(n, 12, device="cuda:0"))        # the hooks run
    env = _auto_env(_auto_blind_class(), _blind_cfg(n, meta["terrain"], measure_heights=True, store=True), True)
    assert env.hot is None and "store_measured_heights" in env.fusion_report, env.fusion_report


def _blind_ref_class(a1, reads_heights=False):
    class BlindRef(a1.A1Conditional):
        def compute_observations(self):
            rb = self.robot
            self.obs_buf = torch.cat([self.command_buf, rb.base_lin_vel, rb.base_ang_vel, rb.gravity_vec,
                                      rb.dof_pos - rb.default_dof_pos, rb.dof_vel,
                                      self.actions_recorder.flatten()], dim=1)
            if reads_heights:
                self.obs_buf[:, 71] += self.isg_env.measured_heights.mean(dim=1)
    return BlindRef


def _ref_env(a1, cls, n, terrain, measure_heights=False, store=False):
    from shifu_b200.sim import fake_isaacgym
    fake_isaacgym.reset_gym()
    cfg = a1.A1EnvConfig()
    cfg.num_envs, cfg.device, cfg.num_obs = n, "cuda:0", BLIND
    for k, v in terrain.items():
        setattr(cfg.terrain, k, v)
    cfg.terrain.measure_heights = measure_heights
    cfg.store_measured_heights = store
    np.random.seed(0)
    env = cls(cfg)
    env._maybe_fuse()
    return env


@needs_examples
def test_reference_a1_edited_to_be_blind_autofuses():
    from tests.test_dropin_gpu import _examples
    a1, _ = _examples()
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    env = _ref_env(a1, _blind_ref_class(a1), n, meta["terrain"])
    assert env.fusion_report == "fused: a1", env.fusion_report
    assert env.hot.blind and env.obs_buf.shape == (n, BLIND)
    env = _ref_env(a1, _blind_ref_class(a1, reads_heights=True), n, meta["terrain"], measure_heights=True)
    assert env.hot is None and "measured_heights" in env.fusion_report, env.fusion_report
    env = _ref_env(a1, _blind_ref_class(a1), n, meta["terrain"], measure_heights=True, store=True)
    assert env.hot is None and "store_measured_heights" in env.fusion_report, env.fusion_report
