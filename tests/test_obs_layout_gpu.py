"""The fused observation layout on the B200: the fused step under non-reference layouts against the oracle
(phased kernel, pipelined kernel + ragged tail, the benchmarked layout), the pre-step projected gravity,
both kernels bit for bit, the reference layout on the default instantiation, and the observation compiler
through the class API (explicit fused task and the reference's own class)."""
import numpy as np
import pytest
import torch

from tests import obs_layouts, util
from tests.test_dropin_gpu import needs_examples
from tests.test_reward_terms_gpu import SNAP_KW, _terrain

pytestmark = pytest.mark.gpu


def _snap(seed, t, n):
    from shifu_b200.sim.synthetic import a1_snapshot
    return a1_snapshot(seed, t, n, **SNAP_KW)


# ---------------------------------------------------------------------------------------------
# 1. the fused step against the oracle
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("layout", ["d1", "legged_gym", "extreme"])
@pytest.mark.parametrize("n,carry,heights,terms", [
    (33, False, True, None),                 # the barrier-phased kernel only
    (32 * 1200 + 7, False, True, "L1"),      # pipelined OBS kernel (HAS_EXTRA) + the phased kernel on the tail
    (65536, True, False, None),              # the benchmarked layout (carried body frame, no measured_heights)
])
def test_fused_step_obs_layout_vs_oracle(layout, n, carry, heights, terms, steps=3, seed=43):
    lay = obs_layouts.LAYOUTS[layout]()
    kw = util.term_list(terms)
    hs, origins, types, env_origins = _terrain(n)
    p, st = util.make_oracle_a1(n, hs, origins, types, env_origins, **kw)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=carry, want_measured_heights=heights, obs=lay,
                           **kw)
    assert hp.desc.obs_layout == 1
    from oracle import shifu_oracle as so
    snap = _snap(seed, 0, n)
    so.a1_reset(p, st, snap)
    hp.reset_idx(None)
    if carry:
        hp.body_frame()
    util.cuda_a1_step(hp, snap, torch.zeros(n, 12))
    skip = ("base_lin_vel", "base_ang_vel", "projected_gravity") if carry else ()

    def want():                                         # the oracle's step, observed under the layout
        out = util.oracle_a1_outputs(st)
        out["obs"] = obs_layouts.oracle_obs(p, st, lay).numpy()
        return out

    util.compare_a1(util.cuda_a1_outputs(hp), want(), f"{layout}/n{n}/reset", skip=skip)
    ep = torch.from_numpy(np.random.RandomState(n).randint(0, 500, size=n))
    st.ep_len[:] = ep
    hp.ep_len.copy_(ep)
    resets = at_clip = 0
    for t in range(1, steps + 1):
        snap = _snap(seed, t, n)
        so.a1_step(p, st, snap.actions, snap)
        util.cuda_a1_step(hp, snap, snap.actions)
        got = util.cuda_a1_outputs(hp)
        util.compare_a1(got, want(), f"{layout}/n{n}/s{t}", skip=skip)
        assert np.array_equal(got["reset_ids"], st.reset_ids.numpy())
        resets += int(st.reset.sum())
        at_clip += int((np.abs(got["obs"]) == np.float32(100.0)).sum())
    assert resets > 0                                   # not vacuous: envs reset
    if layout == "extreme":
        assert at_clip > 0                              # columns pushed past clip_obs sit at +-clip_obs


# ---------------------------------------------------------------------------------------------
# 2. PROJECTED_GRAVITY is the value at the start of the step
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [32 * 64, 32 * 64 + 5])
def test_projected_gravity_is_the_pre_step_value(n):
    hs, origins, types, env_origins = _terrain(n)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=True, want_measured_heights=False,
                           obs=obs_layouts.d1_fix())
    hp.reset_idx(None)
    changed = 0
    for t in range(4):
        seen = {}
        snap = _snap(5, t, n)
        util.cuda_a1_step(hp, snap, snap.actions, before_post=lambda h: seen.__setitem__("pg", h.projected_gravity.clone()))
        assert torch.equal(hp.obs_buf[:, 9:12], seen["pg"]), f"step {t}"
        changed += int((hp.projected_gravity != seen["pg"]).any(dim=1).sum())
    assert changed > n // 2                             # the kernel did write the next step's values


# ---------------------------------------------------------------------------------------------
# 3. the pipelined and the phased kernel agree bit for bit
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("heights", [True, False])
def test_pipelined_and_phased_kernels_agree(heights, monkeypatch):
    n = 32 * 300
    hs, origins, types, env_origins = _terrain(n)
    outs = []
    for kern in (None, "phased"):
        if kern is None:
            monkeypatch.delenv("SHIFU_A1_KERNEL", raising=False)
        else:
            monkeypatch.setenv("SHIFU_A1_KERNEL", kern)
        hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=True, want_measured_heights=heights,
                               obs=obs_layouts.legged_gym())
        hp.reset_idx(None)
        steps = []
        for t in range(3):
            snap = _snap(11, t, n)
            util.cuda_a1_step(hp, snap, snap.actions)
            steps.append(util.cuda_a1_outputs(hp))
        outs.append(steps)
    for t, (a, b) in enumerate(zip(*outs)):
        assert a.keys() == b.keys()
        for k in a:
            assert a[k].tobytes() == b[k].tobytes(), f"step {t}: {k}"


# ---------------------------------------------------------------------------------------------
# 4. the reference layout runs the default instantiation
# ---------------------------------------------------------------------------------------------

def _tma_instantiations(hp, snap):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        util.cuda_a1_step(hp, snap, snap.actions)
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if "a1_post_physics_tma_kernel" in e.name}


def _obs_flag(name):
    """The OBS template argument of an a1_post_physics_tma_kernel instantiation, demangled or not."""
    if "<" in name:
        return name.split("<")[1].split(">")[0].split(",")[3].strip() == "true"
    flags = name.split("a1_post_physics_tma_kernel")[1].split("ILb")[1].split("ELb")    # _Z...ILb0ELb0ELb0ELb1EE...
    return flags[3][0] == "1"


def test_reference_layout_takes_the_default_path(monkeypatch):
    from shifu_b200 import hotpath
    n = 32 * 100 + 3
    hs, origins, types, env_origins = _terrain(n)
    runs, names = [], []
    orig = hotpath.a1_desc

    def layout_one_reference(*a, **kw):                 # obs_layout = 1 holding exactly the reference layout
        d = orig(*a, **kw)
        d.obs_layout = 1
        for i in range(4):
            d.obs_vec_src[i] = i
        for j in range(72):
            d.obs_scale[j] = 1.0
        d.obs_height_scale = 1.0
        return d

    for mode in ("none", "explicit", "layout1", "custom"):
        obs = {"explicit": hotpath.ObsLayout(), "custom": obs_layouts.d1_fix()}.get(mode)
        if mode == "layout1":
            monkeypatch.setattr(hotpath, "a1_desc", layout_one_reference)
        hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=True, want_measured_heights=False, obs=obs)
        monkeypatch.setattr(hotpath, "a1_desc", orig)
        assert hp.desc.obs_layout == (1 if mode in ("layout1", "custom") else 0)
        hp.reset_idx(None)
        util.cuda_a1_step(hp, _snap(3, 0, n), torch.zeros(n, 12))
        names.append(_tma_instantiations(hp, _snap(3, 1, n)))
        runs.append(util.cuda_a1_outputs(hp))
    for got, mode in zip(names, ("none", "explicit", "layout1", "custom")):
        assert len(got) == 1, got
        assert _obs_flag(next(iter(got))) == (mode == "custom"), (mode, got)
    for other in runs[1:3]:
        for k in runs[0]:
            assert runs[0][k].tobytes() == other[k].tobytes(), k
    assert not np.array_equal(runs[0]["obs"], runs[3]["obs"])


# ---------------------------------------------------------------------------------------------
# 5-6. the explicit fused task compiles an edited compute_observations, or refuses it
# ---------------------------------------------------------------------------------------------

def _lg_obs(self):
    """legged_gym's compute_observations (order and obs_scales) on the A1 task's tensors."""
    rb = self.robot
    cs = torch.tensor([2.0, 2.0, 0.25], device=self.device)
    heights = torch.clip(rb.base_pose[:, 2].unsqueeze(1) - 0.5 - self.isg_env.measured_heights, -1, 1.) * 5.0
    self.obs_buf = torch.cat([rb.base_lin_vel * 2.0, rb.base_ang_vel * 0.25, rb.projected_gravity,
                              self.command_buf * cs, (rb.dof_pos - rb.default_dof_pos) * 1.0, rb.dof_vel * 0.05,
                              self.actions_recorder.flatten(), heights], dim=1)


def _task_class(obs_fn):
    from shifu_b200.tasks.a1_walking import A1Conditional
    return type("EditedObs", (A1Conditional,), {"compute_observations": obs_fn})


def _make_task(cls, n, terrain, fused, carry=True):
    from tests.test_env_api_gpu import _install
    _install()
    from shifu_b200.tasks.a1_walking import A1EnvConfig
    cfg = A1EnvConfig()
    cfg.num_envs, cfg.device = n, "cuda:0"
    for k, v in (terrain or {}).items():
        setattr(cfg.terrain, k, v)
    np.random.seed(0)
    torch.manual_seed(0)
    return cls(cfg, fused=fused, carry_body_frame=carry, store_measured_heights=True)


@pytest.mark.parametrize("carry", [False, True])
def test_task_with_legged_gym_observation_fused_vs_hooks(carry):
    from shifu_b200 import _native as nv
    from shifu_b200.sim.synthetic import A1Replay
    from shifu_b200.tasks.a1_walking import A1Conditional
    from tests.test_env_api_gpu import _env_outputs
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    cls = _task_class(_lg_obs)
    envs = [_make_task(cls, n, meta["terrain"], fused, carry) for fused in (True, False)]
    d = envs[0].hot.desc
    assert d.obs_layout == 1
    assert list(d.obs_vec_src) == [nv.OBS_BASE_LIN_VEL, nv.OBS_BASE_ANG_VEL, nv.OBS_PROJECTED_GRAVITY, nv.OBS_COMMAND]
    assert np.array_equal(np.array(d.obs_scale, np.float32), np.array(obs_layouts.legged_gym().scales, np.float32))
    assert np.float32(d.obs_height_scale) == np.float32(5.0)
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
            outs.append(_env_outputs(env))
        util.compare_a1(outs[0], outs[1], f"lg-task/s{t}", skip=skip)
        resets += int(outs[0]["reset"].sum())
    assert resets > 0
    plain = _make_task(A1Conditional, n, meta["terrain"], True)
    assert plain.hot.desc.obs_layout == 0


def _bad_obs(kind):
    def obs(self):
        rb = self.robot
        h = rb.base_pose[:, 2].unsqueeze(1) - 0.5 - self.isg_env.measured_heights
        heights = torch.clip(h, -1, 1.)
        dv = rb.dof_vel
        dp = rb.dof_pos - rb.default_dof_pos
        vec = [self.command_buf, rb.base_lin_vel, rb.base_ang_vel, rb.gravity_vec]
        if kind == "tanh":
            dv = torch.tanh(dv)
        elif kind == "sum":
            vec[1] = rb.base_lin_vel + self.command_buf
        elif kind == "absolute":
            dp = rb.dof_pos
        elif kind == "scale_first":
            heights = torch.clip(h * 5.0, -1, 1.)
        elif kind == "offset":
            dv = rb.dof_vel * 0.05 + 0.1
        self.obs_buf = torch.cat(vec + [dp, dv, self.actions_recorder.flatten(), heights], dim=1)
    return obs


@pytest.mark.parametrize("kind", ["tanh", "sum", "absolute", "scale_first", "offset"])
def test_task_refuses_an_observation_the_kernel_cannot_build(kind):
    z, meta = util.load_golden("a1_small")
    with pytest.raises(NotImplementedError, match="compute_observations"):
        _make_task(_task_class(_bad_obs(kind)), meta["n"], meta["terrain"], True)
    env = _make_task(_task_class(_bad_obs(kind)), meta["n"], meta["terrain"], False)    # user-hook mode runs it
    assert env.hot is None


# ---------------------------------------------------------------------------------------------
# 7. the reference's own class with a legged_gym observation auto-fuses
# ---------------------------------------------------------------------------------------------

@needs_examples
def test_reference_a1_with_legged_gym_observation_autofuses():
    from tests.test_dropin_gpu import _examples, _philox_draws
    from shifu_b200.sim import fake_isaacgym
    from shifu_b200.sim.synthetic import A1Replay
    a1, _ = _examples()
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    cls = type("LeggedGymObs", (a1.A1Conditional,), {"compute_observations": _lg_obs})

    def make(fuse):
        fake_isaacgym.reset_gym()
        cfg = a1.A1EnvConfig()
        cfg.num_envs, cfg.device, cfg.rng_seed, cfg.carry_body_frame = n, "cuda:0", meta["rng_seed"], False
        for k, v in meta["terrain"].items():
            setattr(cfg.terrain, k, v)
        np.random.seed(0)
        env = cls(cfg)
        env.auto_fuse = fuse

        class Replay(A1Replay):
            def begin_step(self, step):
                self.snap = util.golden_snap(z, step)
                self._dof_i = 0
                self.enabled = True
                return self.snap.actions

        env.replay = Replay(0, n, lambda: env.isg_env.env_origins)
        env.isg_env.sim.provider = env.replay
        return env

    fused, hooks = make(True), make(False)
    fused.replay.begin_step(0)
    fused.reset()
    assert fused.fusion_report == "fused: a1", fused.fusion_report
    assert fused.hot.desc.obs_layout == 1
    with _philox_draws(a1, hooks, meta["rng_seed"]):
        hooks.replay.begin_step(0)
        hooks.reset()
        for env in (fused, hooks):
            env.episode_length_buf = torch.from_numpy(z["ep_len_init"]).cuda()
            env.terrain_levels[:] = torch.from_numpy(z["levels_init"]).cuda()
        fused.hot.sync_level_sum()
        for t in range(1, meta["steps"] + 1):
            out = []
            for env in (fused, hooks):
                obs, _, rew, dones, _ = env.step(env.replay.begin_step(t).cuda())
                out.append(dict(obs=obs.clone(), rew=rew.clone(), dones=dones.clone()))
            for k in out[0]:
                a, b = out[0][k].float(), out[1][k].float()
                assert torch.allclose(a, b, rtol=1e-5, atol=1e-6), (t, k, float((a - b).abs().max()))
