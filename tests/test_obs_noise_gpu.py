"""Observation noise on the B200: the fused step with legged_gym's uniform noise against the oracle (phased
kernel, pipelined kernel + ragged tail, the benchmarked layout), both kernels bit for bit, a sharded run
against the single-process one, the NOISE instantiation choice, and the observation compiler through the
class API (explicit fused task, refused hooks, the reference's own class)."""
import numpy as np
import pytest
import torch

from tests import obs_layouts, obs_noise, util
from tests.test_dropin_gpu import needs_examples
from tests.test_obs_layout_gpu import _lg_obs, _make_task, _task_class, _tma_instantiations
from tests.test_reward_terms_gpu import SNAP_KW, _terrain

pytestmark = pytest.mark.gpu
SEED = 0x5EED                                       # hotpath.a1_desc's default rng_seed


def _snap(seed, t, n):
    from shifu_b200.sim.synthetic import a1_snapshot
    return a1_snapshot(seed, t, n, **SNAP_KW)


# ---------------------------------------------------------------------------------------------
# 1. the fused step against the oracle + noise
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("layout", ["legged_gym", "loud"])
@pytest.mark.parametrize("n,carry,heights,terms", [
    (33, False, True, None),                 # the barrier-phased kernel only
    (32 * 1200 + 7, False, True, "L1"),      # pipelined NOISE kernel (HAS_EXTRA) + the phased kernel on the tail
    (65536, True, False, None),              # the benchmarked layout (carried body frame, no measured_heights)
])
def test_fused_step_noisy_obs_vs_oracle(layout, n, carry, heights, terms, steps=3, seed=43):
    lay = obs_noise.NOISY[layout]()
    kw = util.term_list(terms)
    hs, origins, types, env_origins = _terrain(n)
    p, st = util.make_oracle_a1(n, hs, origins, types, env_origins, **kw)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=carry, want_measured_heights=heights, obs=lay,
                           **kw)
    assert hp.desc.obs_layout == 1 and hp.desc.obs_height_noise == lay.height_noise
    from oracle import shifu_oracle as so
    snap = _snap(seed, 0, n)
    so.a1_reset(p, st, snap)
    hp.reset_idx(None)
    if carry:
        hp.body_frame()
    util.cuda_a1_step(hp, snap, torch.zeros(n, 12))
    skip = ("base_lin_vel", "base_ang_vel", "projected_gravity") if carry else ()

    def want():                                         # the oracle's step, observed under the layout + noise
        out = util.oracle_a1_outputs(st)
        out["obs"] = obs_noise.oracle_obs_noisy(p, st, lay, SEED, hp.step_counter).numpy()
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
        assert not np.array_equal(got["obs"], obs_layouts.oracle_obs(p, st, lay).numpy())    # the noise is there
        resets += int(st.reset.sum())
        at_clip += int((np.abs(got["obs"]) == np.float32(100.0)).sum())
    assert resets > 0                                   # not vacuous: envs reset
    if layout == "loud":
        assert at_clip > 0                              # columns noised past clip_obs sit at +-clip_obs


# ---------------------------------------------------------------------------------------------
# 2. the pipelined and the phased kernel agree bit for bit
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("heights", [True, False])
def test_noisy_pipelined_and_phased_kernels_agree(heights, monkeypatch):
    n = 32 * 300 + 5
    hs, origins, types, env_origins = _terrain(n)
    outs = []
    for kern in (None, "phased"):
        if kern is None:
            monkeypatch.delenv("SHIFU_A1_KERNEL", raising=False)
        else:
            monkeypatch.setenv("SHIFU_A1_KERNEL", kern)
        hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=True, want_measured_heights=heights,
                               obs=obs_noise.legged_gym_noisy())
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
# 3. noise is keyed by the global env id: two shards reproduce the single run
# ---------------------------------------------------------------------------------------------

def test_sharded_noise_matches_the_single_run():
    n, half = 32 * 200 + 10, 32 * 100 + 3           # the first shard has a ragged tail, the second starts mid-tile
    lay = obs_noise.legged_gym_noisy()
    hs, origins, _, _ = _terrain(64)
    world = util.world_state(n, 29, 2, origins)
    types, levels0, ep0, cmd0, env_origins, snaps, root0 = world

    def shard(sl):
        m = sl.stop - sl.start
        hp = util.make_cuda_a1(m, hs, origins, types[sl], env_origins[sl], carry=True, want_measured_heights=False,
                               env_offset=sl.start, obs=lay)
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
# 4. noise runs the NOISE instantiation; zero noise the noiseless one, with identical results
# ---------------------------------------------------------------------------------------------

def _flags(name):
    """The five template arguments of an a1_post_physics_tma_kernel instantiation, demangled or not."""
    if "<" in name:
        return [f.strip() == "true" for f in name.split("<")[1].split(">")[0].split(",")]
    flags = name.split("a1_post_physics_tma_kernel")[1].split("ILb")[1].split("ELb")    # _Z...ILb0ELb0ELb0ELb1ELb1EE...
    return [f[0] == "1" for f in flags]


def test_noise_selects_the_noise_instantiation(monkeypatch):
    from shifu_b200 import hotpath
    n = 32 * 100 + 3
    hs, origins, types, env_origins = _terrain(n)
    orig = hotpath.a1_desc

    def signed_zero_noise(*a, **kw):                    # noise fields written, every one -0.0
        d = orig(*a, **kw)
        for j in range(72):
            d.obs_noise[j] = -0.0
        d.obs_height_noise = -0.0
        return d

    modes = ("plain", "zero", "noisy")
    runs, names = [], []
    for mode in modes:
        lay = obs_noise.legged_gym_noisy() if mode == "noisy" else obs_layouts.legged_gym()
        if mode == "zero":
            monkeypatch.setattr(hotpath, "a1_desc", signed_zero_noise)
        hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=True, want_measured_heights=False, obs=lay)
        monkeypatch.setattr(hotpath, "a1_desc", orig)
        hp.reset_idx(None)
        util.cuda_a1_step(hp, _snap(3, 0, n), torch.zeros(n, 12))
        names.append(_tma_instantiations(hp, _snap(3, 1, n)))
        runs.append(util.cuda_a1_outputs(hp))
    for got, mode in zip(names, modes):
        assert len(got) == 1, got
        flags = _flags(next(iter(got)))
        assert len(flags) == 5 and flags[3], (mode, got)                       # OBS
        assert flags[4] == (mode == "noisy"), (mode, got)                     # NOISE
    for k in runs[0]:
        assert runs[0][k].tobytes() == runs[1][k].tobytes(), k
    assert not np.array_equal(runs[0]["obs"], runs[2]["obs"])
    assert np.array_equal(runs[0]["rew"], runs[2]["rew"])


# ---------------------------------------------------------------------------------------------
# 5-6. the explicit fused task compiles a noisy compute_observations, or refuses it
# ---------------------------------------------------------------------------------------------

def _lg_noise_scale_vec(self):
    """legged_gym's _get_noise_scale_vec (noise_level 1, obs_scales of tests/obs_layouts.LG)."""
    vec = torch.zeros(259, device=self.device)
    vec[:3] = 0.1 * 1.0 * 2.0
    vec[3:6] = 0.2 * 1.0 * 0.25
    vec[6:9] = 0.05 * 1.0
    vec[9:12] = 0.0
    vec[12:24] = 0.01 * 1.0 * 1.0
    vec[24:36] = 1.5 * 1.0 * 0.05
    vec[36:72] = 0.0
    vec[72:] = 0.1 * 1.0 * 5.0
    return vec


def _lg_noisy_obs(self):
    """legged_gym's compute_observations with cfg.noise.add_noise = True."""
    _lg_obs(self)
    self.obs_buf += (2 * torch.rand_like(self.obs_buf) - 1) * self._get_noise_scale_vec()


def _noisy_class(base, obs_fn=_lg_noisy_obs, name="NoisyObs"):
    return type(name, (base,), {"compute_observations": obs_fn, "_get_noise_scale_vec": _lg_noise_scale_vec})


def _kernel_draws(monkeypatch, env, seed):
    """torch.rand_like of the observation -> the fused kernel's noise draws at the env's step counter."""
    from shifu_b200.utils import philox
    orig = torch.rand_like

    def rand_like(t, *a, **kw):
        if tuple(t.shape) != (env.num_envs, 259):
            return orig(t, *a, **kw)
        ids = torch.arange(env.num_envs, device=t.device) + int(getattr(env, "env_offset", 0))
        return philox.obs_noise_u01(seed, ids, int(env.common_step_counter)).to(t.dtype)

    monkeypatch.setattr(torch, "rand_like", rand_like)


@pytest.mark.parametrize("carry", [False, True])
def test_task_with_noisy_legged_gym_observation_fused_vs_hooks(carry, monkeypatch):
    from shifu_b200.sim.synthetic import A1Replay
    from shifu_b200.tasks.a1_walking import A1Conditional
    from tests.test_env_api_gpu import _env_outputs
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    cls = _noisy_class(A1Conditional)
    envs = [_make_task(cls, n, meta["terrain"], fused, carry) for fused in (True, False)]
    d = envs[0].hot.desc
    assert d.obs_layout == 1
    assert np.array_equal(np.array(d.obs_noise, np.float32), np.array(obs_noise.LG_NOISE, np.float32))
    assert np.float32(d.obs_height_noise) == np.float32(0.5)
    assert np.array_equal(np.array(d.obs_scale, np.float32), np.array(obs_layouts.legged_gym().scales, np.float32))
    _kernel_draws(monkeypatch, envs[1], envs[1].rng_seed)
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
        util.compare_a1(outs[0], outs[1], f"noisy-task/s{t}", skip=skip)
        resets += int(outs[0]["reset"].sum())
    assert resets > 0


def _bad_noise(kind):
    def obs(self):
        _lg_obs(self)
        vec = self._get_noise_scale_vec()
        if kind == "gaussian":
            self.obs_buf += torch.randn_like(self.obs_buf) * vec
        elif kind == "slice":
            self.obs_buf[:, :48] += (2 * torch.rand_like(self.obs_buf[:, :48]) - 1) * vec[:48]
        elif kind == "per_point":
            vec[72:] = torch.linspace(0.1, 0.5, 187, device=vec.device)
            self.obs_buf += (2 * torch.rand_like(self.obs_buf) - 1) * vec
        elif kind == "inside_clip":
            rb = self.robot
            u = 2 * torch.rand_like(self.obs_buf) - 1
            h = rb.base_pose[:, 2].unsqueeze(1) - 0.5 - self.isg_env.measured_heights + u[:, 72:] * 0.1
            self.obs_buf[:, 72:] = torch.clip(h, -1, 1.) * 5.0
            self.obs_buf[:, :72] += u[:, :72] * vec[:72]
    return obs


@pytest.mark.parametrize("kind", ["gaussian", "slice", "per_point", "inside_clip"])
def test_task_refuses_noise_the_kernel_cannot_draw(kind):
    from shifu_b200.tasks.a1_walking import A1Conditional
    z, meta = util.load_golden("a1_small")
    with pytest.raises(NotImplementedError, match="compute_observations"):
        _make_task(_noisy_class(A1Conditional, _bad_noise(kind)), meta["n"], meta["terrain"], True)
    env = _make_task(_noisy_class(A1Conditional, _bad_noise(kind)), meta["n"], meta["terrain"], False)
    assert env.hot is None                              # user-hook mode runs it


# ---------------------------------------------------------------------------------------------
# 7. the reference's own class with a noisy legged_gym observation auto-fuses
# ---------------------------------------------------------------------------------------------

@needs_examples
def test_reference_a1_with_noisy_legged_gym_observation_autofuses(monkeypatch):
    from tests.test_dropin_gpu import _examples, _philox_draws
    from shifu_b200.sim import fake_isaacgym
    from shifu_b200.sim.synthetic import A1Replay
    a1, _ = _examples()
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    cls = _noisy_class(a1.A1Conditional, name="NoisyLeggedGymObs")

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
    d = fused.hot.desc
    assert d.obs_layout == 1 and np.float32(d.obs_height_noise) == np.float32(0.5)
    _kernel_draws(monkeypatch, hooks, meta["rng_seed"])
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
