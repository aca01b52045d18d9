"""The action head on the B200: legged_gym's own observation, whose 48-column head ends with the step's
actions (235 columns with the heights, 48 blind).  The fused step against the oracle (phased kernel,
pipelined kernel + ragged tail with a HAS_EXTRA term list, the benchmarked size with the carried body
frame, and the stored measured heights), the 235 / 259 / 48 identities with every other output byte-equal,
pipelined == phased, sharded noise, the kernels that run, and the class API (an explicit legged_gym-shaped
task through event launches and graph replay, automatic fusion of a ShifuVecEnv subclass, refusals)."""
import numpy as np
import pytest
import torch

from tests import action_head, util
from tests.test_blind_gpu import _auto_env, _auto_blind_class, _blind_cfg, _task_outputs
from tests.test_reward_terms_gpu import SNAP_KW, _terrain

pytestmark = pytest.mark.gpu
SEED = 0x5EED                                       # hotpath.a1_desc's default rng_seed
HEAD, SIGHTED = 48, 235


def _snap(seed, t, n):
    from shifu_b200.sim.synthetic import a1_snapshot
    return a1_snapshot(seed, t, n, **SNAP_KW)


def _layout(name, num_obs):
    lay = action_head.LAYOUTS[name]()
    return action_head.blind(lay) if num_obs == HEAD else lay


def _kernel(monkeypatch, kernel):
    if kernel is None:
        monkeypatch.delenv("SHIFU_A1_KERNEL", raising=False)
    else:
        monkeypatch.setenv("SHIFU_A1_KERNEL", kernel)


# ---------------------------------------------------------------------------------------------
# 1. the fused step against the oracle
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("layout", list(action_head.LAYOUTS))
@pytest.mark.parametrize("num_obs", [SIGHTED, HEAD])
@pytest.mark.parametrize("n,carry,terms,kernel,mrow", [
    (33, False, None, "phased", False),            # the barrier-phased kernel only (full tile + tail)
    (32 * 1200 + 7, False, "L1", None, False),     # pipelined kernel (HAS_EXTRA) + the phased kernel on the tail
    (65536, True, None, None, False),              # the benchmarked size (carried body frame)
    (32 * 1200 + 7, True, None, None, True),       # 235 with store_measured_heights (HAS_MROW)
])
def test_action_head_step_vs_oracle(layout, num_obs, n, carry, terms, kernel, mrow, monkeypatch, steps=3, seed=43):
    if mrow and (num_obs == HEAD or layout == "loud"):
        pytest.skip("stored heights: the 235-column step with legged_gym's layouts")
    _kernel(monkeypatch, kernel)
    lay = _layout(layout, num_obs)
    kw = util.term_list(terms)
    hs, origins, types, env_origins = _terrain(n)
    p, st = util.make_oracle_a1(n, hs, origins, types, env_origins, **kw)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=carry, want_measured_heights=mrow, obs=lay,
                           num_obs=num_obs, **kw)
    assert tuple(hp.obs_buf.shape) == (n, num_obs) and hp.blind == (num_obs == HEAD)
    from oracle import shifu_oracle as so
    snap = _snap(seed, 0, n)
    so.a1_reset(p, st, snap)
    hp.reset_idx(None)
    if carry:
        hp.body_frame()
    util.cuda_a1_step(hp, snap, torch.zeros(n, 12))
    skip = ("base_lin_vel", "base_ang_vel", "projected_gravity") if carry else ()

    def check(tag):
        got = util.cuda_a1_outputs(hp)
        want = util.oracle_a1_outputs(st)
        if not mrow:
            want.pop("measured_heights", None)
        else:                                           # the stored heights: bit for bit
            util.assert_close(f"{tag}:measured_heights", got["measured_heights"], want.pop("measured_heights"),
                              exact=True)
        want["obs"] = action_head.oracle_obs(p, st, lay, SEED, hp.step_counter).numpy()[:, :num_obs]
        util.compare_a1(got, want, tag, skip=skip)
        return got

    check(f"act/{layout}/{num_obs}/n{n}/reset")
    ep = torch.from_numpy(np.random.RandomState(n).randint(0, 500, size=n))
    st.ep_len[:] = ep
    hp.ep_len.copy_(ep)
    resets = 0
    for t in range(1, steps + 1):
        snap = _snap(seed, t, n)
        so.a1_step(p, st, snap.actions, snap)
        util.cuda_a1_step(hp, snap, snap.actions)
        got = check(f"act/{layout}/{num_obs}/n{n}/s{t}")
        assert np.array_equal(got["reset_ids"], st.reset_ids.numpy())
        resets += int(st.reset.sum())
    assert resets > 0                                   # not vacuous: envs reset


# ---------------------------------------------------------------------------------------------
# 2. the 235 / 259 / 48 identities, pipelined == phased, every output byte for byte
# ---------------------------------------------------------------------------------------------

def _run(n, num_obs, lay, carry, kernel, monkeypatch, seed=11, steps=3, mrow=False):
    _kernel(monkeypatch, kernel)
    hs, origins, types, env_origins = _terrain(n)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=carry, want_measured_heights=mrow, obs=lay,
                           num_obs=num_obs)
    hp.reset_idx(None)
    outs = []
    for t in range(steps):
        snap = _snap(seed, t, n)
        util.cuda_a1_step(hp, snap, snap.actions)
        outs.append(util.cuda_a1_outputs(hp))
    monkeypatch.delenv("SHIFU_A1_KERNEL", raising=False)
    return outs


@pytest.mark.parametrize("layout", list(action_head.LAYOUTS))
@pytest.mark.parametrize("carry,kernel", [(False, None), (True, None), (True, "phased")])
def test_action_head_identities(layout, carry, kernel, monkeypatch):
    n = 32 * 400 + 9
    lay = action_head.LAYOUTS[layout]()
    act = _run(n, SIGHTED, lay, carry, kernel, monkeypatch, mrow=True)
    ref = _run(n, 259, action_head.with_history(lay), carry, kernel, monkeypatch, mrow=True)
    blind = _run(n, HEAD, action_head.blind(lay), carry, kernel, monkeypatch)
    resets = 0
    for t, (a, r, b) in enumerate(zip(act, ref, blind)):
        assert a.keys() == r.keys() and set(b) == set(a) - {"measured_heights"}
        for k in a:
            if k == "obs":
                assert a[k][:, :36].tobytes() == r[k][:, :36].tobytes(), f"step {t}: obs 0-35"
                assert a[k][:, 48:].tobytes() == r[k][:, 72:].tobytes(), f"step {t}: heights"
                assert b[k].tobytes() == np.ascontiguousarray(a[k][:, :HEAD]).tobytes(), f"step {t}: 48 == 235[:48]"
                continue
            assert a[k].tobytes() == r[k].tobytes(), f"step {t}: {k}"
            if k in b:
                assert b[k].tobytes() == a[k].tobytes(), f"step {t}: blind {k}"
        resets += int(a["reset"].sum())
    assert resets > 0


@pytest.mark.parametrize("num_obs", [SIGHTED, HEAD])
@pytest.mark.parametrize("layout", ["legged_gym", "loud"])
def test_action_head_pipelined_and_phased_kernels_agree(num_obs, layout, monkeypatch):
    n = 32 * 300 + 5
    lay = _layout(layout, num_obs)
    a = _run(n, num_obs, lay, True, None, monkeypatch)
    b = _run(n, num_obs, lay, True, "phased", monkeypatch)
    for t, (x, y) in enumerate(zip(a, b)):
        for k in x:
            assert x[k].tobytes() == y[k].tobytes(), f"step {t}: {k}"


@pytest.mark.parametrize("num_obs,kernel", [(SIGHTED, "a1_post_physics_tma_kernel"),
                                            (HEAD, "a1_post_physics_blind_kernel")])
def test_action_head_runs_its_kernel(num_obs, kernel):
    from torch.profiler import ProfilerActivity, profile
    n = 32 * 100 + 3
    hs, origins, types, env_origins = _terrain(n)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=True, want_measured_heights=False,
                           obs=_layout("legged_gym_noisy", num_obs), num_obs=num_obs)
    hp.reset_idx(None)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        util.cuda_a1_step(hp, _snap(3, 0, n), torch.zeros(n, 12))
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if "a1_post_physics" in e.name}
    assert any(kernel + "_act<" in x for x in names), names         # the action-head instantiation
    other = {"a1_post_physics_tma_kernel", "a1_post_physics_blind_kernel"} - {kernel}
    assert not any(o in x for o in other for x in names), names


# ---------------------------------------------------------------------------------------------
# 3. noise is keyed by the global env id: two shards reproduce the single run
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("num_obs", [SIGHTED, HEAD])
def test_action_head_sharded_noise_matches_the_single_run(num_obs):
    n, half = 32 * 200 + 10, 32 * 100 + 3           # the first shard has a ragged tail, the second starts mid-tile
    lay = _layout("loud", num_obs)
    hs, origins, _, _ = _terrain(64)
    types, levels0, ep0, cmd0, env_origins, snaps, root0 = util.world_state(n, 29, 2, origins)

    def shard(sl):
        m = sl.stop - sl.start
        hp = util.make_cuda_a1(m, hs, origins, types[sl], env_origins[sl], carry=True, want_measured_heights=False,
                               env_offset=sl.start, obs=lay, num_obs=num_obs)
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
# 4. the class API: legged_gym's compute_observations on an A1Conditional subclass
# ---------------------------------------------------------------------------------------------

def _lg_noise_vec(self, width):
    """legged_gym's _get_noise_scale_vec (noise_level 1; the actions get none)."""
    vec = torch.zeros(width, device=self.device)
    vec[:3], vec[3:6], vec[6:9] = 0.1 * 2.0, 0.2 * 0.25, 0.05
    vec[12:24], vec[24:36] = 0.01, 1.5 * 0.05
    vec[48:] = 0.1 * 5.0
    return vec


def _lg_obs(self, noise=True):
    """legged_gym's compute_observations: its order and obs_scales, the step's actions, the heights when the
    observation has them, and its uniform noise."""
    rb = self.robot
    cs = torch.tensor([2.0, 2.0, 0.25], device=self.device)
    cols = [rb.base_lin_vel * 2.0, rb.base_ang_vel * 0.25, rb.projected_gravity, self.command_buf * cs,
            (rb.dof_pos - rb.default_dof_pos) * 1.0, rb.dof_vel * 0.05, self.actions]
    if self.num_obs == SIGHTED:
        cols.append(torch.clip(rb.base_pose[:, 2].unsqueeze(1) - 0.5 - self.isg_env.measured_heights, -1, 1.) * 5.0)
    self.obs_buf = torch.cat(cols, dim=-1)
    if noise:
        self.obs_buf += (2 * torch.rand_like(self.obs_buf) - 1) * _lg_noise_vec(self, self.obs_buf.shape[1])


def _obs_class(obs_fn=_lg_obs, base=None):
    from shifu_b200.tasks.a1_walking import A1Conditional
    return type("LeggedGymObsA1", (base or A1Conditional,), {"compute_observations": obs_fn})


def _cfg(n, terrain, num_obs, store=None):
    """The task config; a sighted task stores the kernel's measured heights, so that they compare with the
    heights the hooks measure (the on-demand scan sees the post-reset pose of an env that reset)."""
    store = num_obs == SIGHTED if store is None else store
    cfg = _blind_cfg(n, terrain, measure_heights=num_obs == SIGHTED, store=store)
    cfg.num_obs = num_obs
    return cfg


def _kernel_draws(monkeypatch, env):
    """torch.rand_like of the observation -> the fused kernel's noise draws at the env's step counter."""
    from shifu_b200.utils import philox
    orig = torch.rand_like
    seed = getattr(env, "rng_seed", SEED)

    def rand_like(t, *a, **kw):
        if tuple(t.shape) != (env.num_envs, env.num_obs):
            return orig(t, *a, **kw)
        ids = torch.arange(env.num_envs, device=t.device) + int(getattr(env, "env_offset", 0))
        u = philox.obs_noise_u01(seed, ids, int(env.common_step_counter), head=HEAD)
        return u[:, :env.num_obs].to(t.dtype)

    monkeypatch.setattr(torch, "rand_like", rand_like)


def _outputs(env):
    if env.num_obs == HEAD:
        return _task_outputs(env)
    from tests.test_env_api_gpu import _env_outputs
    return _env_outputs(env)


def _replays(envs, z, n):
    from shifu_b200.sim.synthetic import A1Replay
    out = []
    for env in envs:
        class Replay(A1Replay):
            def begin_step(self, step):
                self.snap = util.golden_snap(z, step)
                self._dof_i = 0
                self.enabled = True
                return self.snap.actions
        r = Replay(0, n, lambda env=env: env.isg_env.env_origins)
        env.isg_env.sim.provider = r
        out.append(r)
    return out


@pytest.mark.parametrize("num_obs", [SIGHTED, HEAD])
@pytest.mark.parametrize("carry", [False, True])
def test_legged_gym_task_fused_vs_hooks(num_obs, carry, monkeypatch):
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    cls = _obs_class()
    envs = [cls(_cfg(n, meta["terrain"], num_obs), fused=fused, carry_body_frame=carry,
                store_measured_heights=num_obs == SIGHTED) for fused in (True, False)]
    d = envs[0].hot.desc
    assert d.num_obs == num_obs and d.obs_layout == 1 and envs[0].hot.blind == (num_obs == HEAD)
    assert list(d.obs_scale[36:48]) == [1.0] * 12 and list(d.obs_noise[36:48]) == [0.0] * 12
    assert envs[1].hot is None
    _kernel_draws(monkeypatch, envs[1])
    replays = _replays(envs, z, n)
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
            outs.append(_outputs(env))
        assert outs[0]["obs"].shape == (n, num_obs)
        util.compare_a1(outs[0], outs[1], f"lg-task/{num_obs}/s{t}", skip=skip)
        resets += int(outs[0]["reset"].sum())
    assert resets > 0


@pytest.mark.parametrize("num_obs", [SIGHTED, HEAD])
def test_legged_gym_task_graph_replay_vs_hooks(num_obs, monkeypatch):
    """Resident state: the fused task steps by CUDA-graph replay; fused=False runs the hooks."""
    n = 32 * 64 + 5
    cls = _obs_class()
    envs = [cls(_cfg(n, None, num_obs), fused=fused, carry_body_frame=True, store_measured_heights=num_obs == SIGHTED)
            for fused in (True, False)]
    _kernel_draws(monkeypatch, envs[1])
    for env in envs:
        env.reset()
    g = torch.Generator().manual_seed(5)
    for t in range(6):
        a = (torch.rand(n, 12, generator=g) * 2 - 1).cuda()
        outs = []
        for env in envs:
            env.step(a)
            outs.append(_outputs(env))
        util.compare_a1(outs[0], outs[1], f"lg-graph/{num_obs}/s{t}",
                        skip=("base_lin_vel", "base_ang_vel", "projected_gravity"))
    assert envs[0].hot._graph is not None               # the fused steps replayed the captured graph


def test_legged_gym_shifu_vec_env_autofuses_and_matches_hooks():
    """A ShifuVecEnv subclass shaped like the reference task, with legged_gym's observation (235 columns, no
    noise: the automatic path's draws are checked by the class test above) fuses automatically and matches
    the same class in user-hook mode."""
    from tests.test_dropin_gpu import _philox_draws
    import tests.test_blind_gpu as blind_mod
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    cls = _auto_blind_class(lambda self: _lg_obs(self, noise=False))
    fused, hooks = (_auto_env(cls, _cfg(n, meta["terrain"], SIGHTED), fuse) for fuse in (True, False))
    assert fused.fusion_report == "fused: a1", fused.fusion_report
    assert fused.hot.desc.num_obs == SIGHTED and fused.obs_buf.shape == (n, SIGHTED)
    assert hooks.hot is None
    replays = _replays((fused, hooks), z, n)
    with _philox_draws(blind_mod, hooks, getattr(hooks.cfg, "rng_seed", SEED)):
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
                outs.append(_outputs(env))
            util.compare_a1(outs[0], outs[1], f"auto-lg/s{t}", skip=("base_lin_vel", "base_ang_vel", "projected_gravity"))
            resets += int(outs[0]["reset"].sum())
    assert resets > 0


# ---------------------------------------------------------------------------------------------
# 5. refusals, with their reasons
# ---------------------------------------------------------------------------------------------

def _mixed_obs(self):
    """The action head with the last history slot in place of three action columns."""
    _lg_obs(self, noise=False)
    self.obs_buf[:, 45:48] = self.actions_recorder.get_last(2)[:, 9:12]


def _actions_in_72(self):
    """A 72-column head whose first history slot is the step's actions."""
    rb = self.robot
    self.obs_buf = torch.cat([self.command_buf, rb.base_lin_vel, rb.base_ang_vel, rb.gravity_vec,
                              rb.dof_pos - rb.default_dof_pos, rb.dof_vel, self.actions,
                              self.actions_recorder.flatten()[:, 12:]], dim=1)


def _tanh_actions(self):
    _lg_obs(self, noise=False)
    self.obs_buf[:, 36:48] = torch.tanh(self.actions)


@pytest.mark.parametrize("obs_fn,num_obs,reason", [
    (_mixed_obs, HEAD, "actions_recorder"),
    (_mixed_obs, SIGHTED, "actions_recorder"),
    (_actions_in_72, 72, "actions_recorder"),
    (_tanh_actions, SIGHTED, "no other function"),
])
def test_refusals(obs_fn, num_obs, reason):
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    with pytest.raises(NotImplementedError, match=reason) as exc:
        _obs_class(obs_fn)(_cfg(n, meta["terrain"], num_obs), fused=True)
    assert "actions" in str(exc.value)
    env = _auto_env(_auto_blind_class(obs_fn), _cfg(n, meta["terrain"], num_obs), True)
    assert env.hot is None and env.fusion_report.startswith("user-hook mode"), env.fusion_report
    assert reason in env.fusion_report, env.fusion_report
    env.reset()
    env.step(torch.zeros(n, 12, device="cuda:0"))        # the hooks run
    assert env.obs_buf.shape == (n, num_obs)


def test_blind_action_head_refuses_store_measured_heights():
    from shifu_b200.gym import autofuse
    z, meta = util.load_golden("a1_small")
    cfg = _cfg(meta["n"], meta["terrain"], HEAD)
    cfg.terrain.measure_heights = True
    with pytest.raises(NotImplementedError, match="store_measured_heights"):
        _obs_class()(cfg, fused=True, store_measured_heights=True)
    cfg = _cfg(meta["n"], meta["terrain"], HEAD, store=True)
    cfg.terrain.measure_heights = True
    env = _obs_class()(cfg, fused=False)
    with pytest.raises(autofuse.NotFusable, match="store_measured_heights with a 48-column"):
        autofuse.fuse_a1(env)


def test_history_depth_other_than_3_is_refused_with_its_reason():
    from shifu_b200.gym import autofuse
    z, meta = util.load_golden("a1_small")
    env = _obs_class()(_cfg(meta["n"], meta["terrain"], SIGHTED), fused=False)
    env.cfg.num_actions_history = 1
    with pytest.raises(autofuse.NotFusable, match="num_actions_history = 1"):
        autofuse.fuse_a1(env)
