"""GPU tests of the drop-in class API (ShifuVecEnv / Unit mirror + tasks) on the stand-in simulator:
the same call sequence the reference harness used to record the golden fixtures
(env.reset(), then env.step(actions) with replayed simulator snapshots)."""
import numpy as np
import pytest
import torch

from tests import util

pytestmark = pytest.mark.gpu


def _install():
    from shifu_b200.sim import fake_isaacgym
    fake_isaacgym.install("cuda:0")
    fake_isaacgym.reset_gym()
    fake_isaacgym.set_default_device("cuda:0")
    return fake_isaacgym


def _make_a1(n, terrain, fused=True, carry=False):
    _install()
    from shifu_b200.tasks.a1_walking import A1Conditional, A1EnvConfig
    cfg = A1EnvConfig()
    cfg.num_envs = n
    cfg.device = "cuda:0"
    for k, v in (terrain or {}).items():
        setattr(cfg.terrain, k, v)
    np.random.seed(0)
    torch.manual_seed(0)
    return A1Conditional(cfg, fused=fused, carry_body_frame=carry, store_measured_heights=True)


def _env_outputs(env):
    isg, rb = env.isg_env, env.robot
    d = dict(obs=env.obs_buf, rew=env.rew_buf, reset=env.reset_buf.to(torch.uint8),
             time_out=env.time_out_buf.to(torch.uint8), contact_term=env.contact_terminate_buf.to(torch.uint8),
             ep_len=env.episode_length_buf, terrain_levels=env.terrain_levels, env_origins=isg.env_origins,
             command=env.command_buf, history=env.actions_recorder.history_buf, actions=env.actions,
             root_state=isg.root_state, dof_state=isg.dof_state, dof_targets=rb.dof_targets,
             rand_force=rb.rand_force_buf, torques=rb.torques, base_lin_vel=rb.base_lin_vel,
             base_ang_vel=rb.base_ang_vel, projected_gravity=rb.projected_gravity,
             measured_heights=isg.measured_heights)
    for k, v in env.episode_rewards.items():
        d["ep_sum/" + k] = v
    for k, v in env.extras.get("episode", {}).items():
        d["extras/" + k] = torch.as_tensor(v)
    return {k: v.detach().cpu().numpy().copy() for k, v in d.items()}


@pytest.mark.parametrize("fused,carry", [(True, False), (True, True), (False, False)])
def test_a1_class_api_replays_golden(fused, carry):
    from shifu_b200.sim.synthetic import A1Replay
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    env = _make_a1(n, meta["terrain"], fused=fused, carry=carry)
    isg = env.isg_env
    assert np.array_equal(isg.height_samples.cpu().numpy(), z["height_samples"])
    assert np.array_equal(isg.env_origins.cpu().numpy(), z["env_origins_init"])
    assert np.array_equal(isg.terrain_types.cpu().numpy(), z["terrain_types"])

    class Replay(A1Replay):              # serve the fixture's recorded snapshots
        def begin_step(self, step):
            self.snap = util.golden_snap(z, step)
            self._dof_i = 0
            self.enabled = True
            return self.snap.actions

    replay = Replay(0, n, lambda: isg.env_origins)
    isg.sim.provider = replay
    skip = ("base_lin_vel", "base_ang_vel", "projected_gravity") if carry else ()
    replay.begin_step(0)
    env.reset()
    util.compare_a1(_env_outputs(env), util.golden_out(z, 0), "api/reset", skip=skip)
    env.episode_length_buf = torch.from_numpy(z["ep_len_init"]).cuda()       # rsl_rl-style re-binding
    env.terrain_levels[:] = torch.from_numpy(z["levels_init"]).cuda()
    if fused:
        env.hot.sync_level_sum()
    for t in range(1, meta["steps"] + 1):
        actions = replay.begin_step(t)
        obs, priv, rew, dones, extras = env.step(actions.cuda())
        assert priv is None and obs.shape == (n, 259) and dones.dtype == torch.bool
        util.compare_a1(_env_outputs(env), util.golden_out(z, t), f"api/s{t}", skip=skip)
        assert torch.equal(extras["time_outs"].cpu(), torch.from_numpy(z[f"s{t}/out/time_out"]).bool())


def test_abb_class_api_replays_golden():
    _install()
    from shifu_b200.sim.synthetic import AbbReplay
    from shifu_b200.tasks.abb_pushbox import AbbPushBox, PriorStageEnvConfig
    z, meta = util.load_golden("abb_small")
    n = meta["n"]
    cfg = PriorStageEnvConfig()
    cfg.num_envs = n
    cfg.device = "cuda:0"
    env = AbbPushBox(cfg, rng_seed=meta["rng_seed"])

    class Replay(AbbReplay):
        def begin_step(self, step):
            self.snap = util.golden_snap(z, step, "abb")
            self.enabled = True
            return self.snap.actions

    replay = Replay(0, n)
    env.isg_env.sim.provider = replay
    env.episode_length_buf = torch.from_numpy(z["ep_len_init"]).cuda()
    for t in range(1, meta["steps"] + 1):
        actions = replay.begin_step(t)
        obs, _, rew, dones, extras = env.step(actions.cuda())
        want = util.golden_out(z, t)
        got = dict(obs=obs, rew=rew, reset=dones.to(torch.uint8), time_out=env.time_out_buf.to(torch.uint8),
                   success=env.success_buf.to(torch.uint8), ep_len=env.episode_length_buf,
                   root_state=env.isg_env.root_state, dof_state=env.isg_env.dof_state)
        for k, v in env.episode_rewards.items():
            got["ep_sum/" + k] = v
        for k, v in extras["episode"].items():
            got["extras/" + k] = v
        got = {k: v.detach().cpu().numpy() for k, v in got.items()}
        util.compare_a1(got, want, f"abb api/s{t}", skip=("dof_targets",))


def test_task_classes_carry_the_reference_descriptor():
    """The fused task classes on their default configs hand the kernel exactly the reference's constants:
    the descriptor builders they share with automatic fusion read every value off the env, its robot,
    its scene and its config, and the default config has the constants ``a1_desc`` / ``abb_desc`` default to."""
    from shifu_b200 import hotpath
    n, offset, seed = 64, 4096, 99
    _install()
    from shifu_b200.tasks.a1_walking import A1Conditional, A1EnvConfig
    cfg = A1EnvConfig()
    cfg.num_envs, cfg.device = n, "cuda:0"
    env = A1Conditional(cfg, rng_seed=seed, env_offset=offset, num_envs_global=offset + n)
    assert bytes(env.hot.desc) == bytes(hotpath.a1_desc(n, env_offset=offset, rng_seed=seed))
    _install()
    from shifu_b200.tasks.abb_pushbox import AbbPushBox, PriorStageEnvConfig
    cfg = PriorStageEnvConfig()
    cfg.num_envs, cfg.device = n, "cuda:0"
    env = AbbPushBox(cfg, rng_seed=seed, env_offset=offset)
    assert bytes(env.hot.desc) == bytes(hotpath.abb_desc(n, env_offset=offset, rng_seed=seed))


def test_abb_robot_step_uses_arm_ik_kernel():
    """AbbRobot.step (a_prior_stage.py:67-73) through the class API == oracle restatement."""
    import json, os
    from oracle import shifu_oracle as so
    _install()
    from shifu_b200.tasks.abb_pushbox import AbbPushBox, PriorStageEnvConfig
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "arm_ik.npz"))
    meta = json.loads(bytes(z["meta"]).decode())
    d = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("in/")}
    cfg = PriorStageEnvConfig()
    cfg.num_envs, cfg.device = meta["n"], "cuda:0"
    env = AbbPushBox(cfg)
    rb = env.robot
    assert abs(float(rb.env.dt) - meta["dt"]) < 1e-9 and rb._jacobian.is_contiguous()
    rb.body_state[:, int(rb.ee_indices[0]), :7] = d["ee_pose"].cuda()
    rb.dof_pos[:] = d["dof_pos"].cuda()
    rb._jacobian[:, rb._ee_link] = d["j_ee"].cuda()
    rb.step(d["actions"].cuda())
    want = torch.from_numpy(z["out/dof_targets_step"])
    goal = so.arm_goal_from_actions(d["ee_pose"][:, :3], d["actions"], meta["ee_velocity"], meta["dt"],
                                    meta["min_ee_pos"], meta["max_ee_pos"], meta["tar_quat"])
    o64 = so.arm_ik(d["dof_pos"].double(), d["ee_pose"].double(), d["j_ee"].double(), goal.double(), meta["damping"])
    err_ref = float((want.double() - o64).abs().max())
    assert float((rb.dof_targets.cpu() - want).abs().max()) <= 3.0 * err_ref + 1e-6
    # the generic entry: inverse_kinematics(goal_pose)
    got = rb.inverse_kinematics(d["goal_pose"].cuda()).cpu()
    assert float((got - torch.from_numpy(z["out/dof_targets_goal"])).abs().max()) <= 3.0 * err_ref + 1e-6


def test_no_cpu_fallback():
    """The product path must fail loudly off-GPU (ShifuNativeError), never fall back to torch."""
    from shifu_b200 import _native as nv, hotpath
    with pytest.raises(nv.ShifuNativeError):
        hotpath.EnvKernels("cpu", 16)
    with pytest.raises(nv.ShifuNativeError):
        nv.ptr(torch.zeros(4))


def test_abb_env_reset_and_reset_idx():
    """ADVICE r1 (high): AbbPushBox.reset() / reset_idx() — what rsl_rl's OnPolicyRunner and the
    reference's run_policy call first (policy_runner.py:22,33; env.py:108-130).  The reset state is
    compared with the oracle's abb_reset_idx driven by the same Philox streams."""
    from oracle import shifu_oracle as so
    _install()
    from shifu_b200.sim.synthetic import AbbReplay, abb_snapshot
    from shifu_b200.tasks.abb_pushbox import AbbPushBox, PriorStageEnvConfig
    n = 1000
    cfg = PriorStageEnvConfig()
    cfg.num_envs, cfg.device = n, "cuda:0"
    env = AbbPushBox(cfg, rng_seed=99)
    p = so.AbbParams(n=n, rng_seed=99)
    st = so.abb_new_state(p)
    st.success = torch.zeros(n, dtype=torch.bool)          # the env's success_buf before the first step
    # --- reset(): reset_idx(all) at step counter 0 ...
    extras_id = id(env.extras)
    env.reset_idx(None)
    so.abb_reset_idx(p, st, torch.arange(n))
    util.assert_close("root after reset_idx", env.isg_env.root_state.cpu().numpy(), st.root_state.numpy(), exact=False)
    util.assert_close("dof after reset_idx", env.isg_env.dof_state.cpu().numpy(), st.dof_state.numpy(), exact=True)
    cube = env.isg_env.root_state.view(n, 4, 13)[:, 2]
    goal = env.isg_env.root_state.view(n, 4, 13)[:, 3]
    assert float((cube[:, :2] - goal[:, :2]).norm(dim=1).min()) > 0.0     # not the default (coincident) poses
    assert float(cube[:, :2].abs().max()) <= 0.1 + 1e-6 and float(env.episode_length_buf.abs().sum()) == 0
    assert id(env.extras) == extras_id and set(env.extras["episode"]) == {"reward_reaching", "reward_success",
                                                                          "success_rate"}
    # ... then a zero-action step; the full reset() is what a runner calls
    env.isg_env.sim.provider = AbbReplay(3, n)
    obs, priv = env.reset()
    assert obs.shape == (n, 6) and priv is None and torch.isfinite(obs).all()
    # --- reset_idx(ids) mid-run: only those envs change, their episode sums are logged and zeroed
    env.isg_env.sim.provider.enabled = False
    env.episode_rewards["reward_reaching"].fill_(2.0)
    before = env.isg_env.root_state.clone()
    ids = torch.tensor([3, 10, 500], device="cuda")
    env.reset_idx(ids)
    keep = torch.ones(n, dtype=torch.bool, device="cuda")
    keep[ids] = False
    assert torch.equal(env.isg_env.root_state.view(n, 4, 13)[keep], before.view(n, 4, 13)[keep])
    assert float(env.episode_rewards["reward_reaching"][ids].abs().sum()) == 0
    assert abs(float(env.extras["episode"]["reward_reaching"]) - 2.0 / 20.0) < 1e-6      # mean / max_episode_length_s
    assert int(env.episode_length_buf[ids].abs().sum()) == 0


def test_extras_of_each_step_keep_their_own_storage():
    """ADVICE r1 (medium): rsl_rl appends infos['episode'] every step and reduces the list at the end
    of the iteration; the reference allocates fresh tensors per resetting step (env.py:124-130)."""
    from shifu_b200.sim.synthetic import A1Replay
    z, meta = util.load_golden("a1_small")
    env = _make_a1(meta["n"], meta["terrain"], fused=True, carry=True)
    replay = A1Replay(5, meta["n"], lambda: env.isg_env.env_origins, p_base=0.3)
    env.isg_env.sim.provider = replay
    env.reset()
    kept, values = [], []
    for t in range(1, 9):
        actions = replay.begin_step(t)
        _, _, _, dones, extras = env.step(actions.cuda())
        kept.append(extras["episode"])
        values.append({k: float(v) for k, v in extras["episode"].items()})
    assert len({id(d) for d in kept}) == len(kept)
    ptrs = {d["tracking_lin_vel"].data_ptr() for d in kept}
    assert len(ptrs) == len(kept), "every step's extras must live in its own slot"
    for d, v in zip(kept, values):                                  # later steps did not overwrite earlier ones
        assert {k: float(x) for k, x in d.items()} == v
    assert len({v["tracking_lin_vel"] for v in values}) > 1
