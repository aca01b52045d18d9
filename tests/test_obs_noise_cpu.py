"""Observation noise on a CPU-only checkout: descriptor and ObsLayout validation, the draw map of the
numpy oracle and the torch implementation, and the test oracle's noisy observation."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from tests import obs_layouts, obs_noise, util


def _create(d):
    from shifu_b200 import _native as nv
    lib = nv.load()
    out = C.c_void_p()
    return lib.shifu_ctx_create(0, C.byref(d), None, C.byref(out)), lib.shifu_last_error().decode()


@pytest.mark.parametrize("field,value", [
    ("obs_noise", math.nan), ("obs_noise", math.inf), ("obs_noise", -math.inf),
    ("obs_height_noise", math.nan), ("obs_height_noise", -math.inf),
])
def test_non_finite_noise_is_rejected_before_the_device_check(field, value):
    from shifu_b200 import _native as nv, hotpath
    d = hotpath.a1_desc(64, obs=obs_noise.legged_gym_noisy())
    if field == "obs_noise":
        d.obs_noise[30] = value
    else:
        d.obs_height_noise = value
    rc, msg = _create(d)
    assert rc == nv.E_RANGE, (rc, msg)
    assert field in msg


@pytest.mark.parametrize("field", ["obs_noise", "obs_height_noise"])
def test_noise_without_a_layout_is_rejected(field):
    from shifu_b200 import _native as nv, hotpath
    d = hotpath.a1_desc(64)
    assert d.obs_layout == 0
    if field == "obs_noise":
        d.obs_noise[5] = 0.1
    else:
        d.obs_height_noise = 0.1
    rc, msg = _create(d)
    assert rc == nv.E_RANGE, (rc, msg)
    assert "obs_layout" in msg


def test_noisy_layout_passes_validation():
    from shifu_b200 import _native as nv, hotpath
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: the descriptor would create a context")
    for make in obs_noise.NOISY.values():
        assert _create(hotpath.a1_desc(64, obs=make()))[0] == nv.E_NODEVICE


def test_obs_layout_noise_values():
    from shifu_b200 import hotpath
    from shifu_b200.hotpath import ObsLayout
    lay = obs_noise.legged_gym_noisy()
    assert lay.has_noise() and not lay.is_reference()
    assert lay.noise[24] == float(np.float32(0.075)) and lay.height_noise == 0.5
    assert ObsLayout(height_noise=0.1).has_noise() and not ObsLayout(height_noise=0.1).is_reference()
    assert ObsLayout(noise=(0.0,) * 72, height_noise=0.0) == ObsLayout()
    for bad in (dict(noise=(0.1,) * 71), dict(noise=(math.nan,) * 72), dict(height_noise=math.inf)):
        with pytest.raises(ValueError):
            ObsLayout(**bad)
    d = hotpath.a1_desc(8, obs=lay)
    assert d.obs_layout == 1
    assert np.array_equal(np.array(d.obs_noise, np.float32), np.array(obs_noise.LG_NOISE, np.float32))
    assert np.float32(d.obs_height_noise) == np.float32(0.5)
    # a zero noise leaves the descriptor byte for byte that of the layout without noise
    quiet = ObsLayout(lay.slots, lay.scales, lay.height_scale, (0.0,) * 72, 0.0)
    assert bytes(hotpath.a1_desc(8, obs=quiet)) == bytes(hotpath.a1_desc(8, obs=obs_layouts.legged_gym()))
    d = hotpath.a1_desc(8, obs=ObsLayout(height_noise=0.25))         # noise alone makes a layout-1 descriptor
    assert d.obs_layout == 1 and d.obs_height_noise == 0.25 and list(d.obs_scale) == [1.0] * 72


def test_draw_map_covers_every_column_once_in_65_words():
    from oracle import obs_noise_np as onp
    from shifu_b200.utils import philox
    word, lane = onp.obs_noise_map()
    assert word.min() == 0 and word.max() == 64                     # 65 evaluations per env and step
    assert len(set(zip(word.tolist(), lane.tolist()))) == 259       # no (word, lane) serves two columns
    assert (lane >= 0).all() and (lane < 4).all()
    # only the centre point's mirror slot (word 64, lane w) is unused
    assert set((w, l) for w in range(65) for l in range(4)) - set(zip(word.tolist(), lane.tolist())) == {(64, 3)}
    tw, tl = philox.obs_noise_slots()
    assert np.array_equal(tw.numpy(), word) and np.array_equal(tl.numpy(), lane)
    # the head words of the pipelined kernel's lane pairs (d = 2i, 2i+1 write columns d + 12m)
    for i in range(6):
        cols = [d + 12 * m for d in (2 * i, 2 * i + 1) for m in range(6)]
        assert sorted(set(word[cols].tolist())) == [3 * i, 3 * i + 1, 3 * i + 2]


@pytest.mark.parametrize("seed", [0, 0x5EED, (1 << 40) + 12345])
def test_numpy_and_torch_draws_agree(seed):
    from oracle import obs_noise_np as onp, philox_np as px
    from shifu_b200.utils import philox
    ids = np.array([0, 1, 2, 31, 32, 1000, (1 << 20) + 3, (1 << 31) + 7, (1 << 32) - 1], dtype=np.int64)
    for step in (0, 1, 7, 500, (1 << 32) + 5):
        want = onp.obs_noise_u01(seed, ids, step)
        got = philox.obs_noise_u01(seed, torch.from_numpy(ids), step).numpy()
        assert want.shape == got.shape == (len(ids), 259) and want.dtype == got.dtype == np.float32
        assert np.array_equal(want, got), step
        # word 0 lane x of the map is the plain stream-8 draw with word 0
        assert np.array_equal(want[:, 0], px.u01_f32(px.draw_u32(seed, ids, step, onp.STREAM_OBS_NOISE)[0]))
    a, b = onp.obs_noise_u01(seed, ids, 3), onp.obs_noise_u01(seed, ids, 4)
    assert not np.array_equal(a, b) and len(np.unique(a)) > 0.99 * a.size


def _oracle_state(n=6):
    from oracle import shifu_oracle as so
    p = so.A1Params(n=n, env_offset=1000)
    st = so.a1_new_state(p, torch.zeros(2, 2, dtype=torch.int16), torch.zeros(1, 1, 3), torch.zeros(n, dtype=torch.long),
                         torch.zeros(n, 3))
    g = torch.Generator().manual_seed(0)
    for name in ("command", "base_lin_vel", "base_ang_vel", "projected_gravity", "history"):
        getattr(st, name).copy_(torch.randn(getattr(st, name).shape, generator=g))
    st.dof_state.copy_(torch.randn(st.dof_state.shape, generator=g))
    st.root_state[:, 2] = torch.tensor([0.5, 2.0, -2.0, 0.7, 0.1, 0.45])[:n]
    st.measured_heights = torch.zeros(n, 187)
    so.a1_compute_observations(p, st)
    return p, st


def test_oracle_noise_zero_is_the_layout_observation():
    from shifu_b200.hotpath import ObsLayout
    p, st = _oracle_state()
    for lay in (obs_layouts.legged_gym(), ObsLayout()):
        got = obs_noise.oracle_obs_noisy(p, st, lay, 0x5EED, 3)
        assert got.numpy().tobytes() == obs_layouts.oracle_obs(p, st, lay).numpy().tobytes()


@pytest.mark.parametrize("layout", ["legged_gym", "loud"])
def test_oracle_applies_the_noise(layout):
    """fl(fl(x_j * scale_j) + fl((2u - 1) * noise_j)), heights fl(fl(clip(d, +-1) * hs) + n), then the clip."""
    from oracle import obs_noise_np as onp
    p, st = _oracle_state()
    lay = obs_noise.NOISY[layout]()
    seed, step = 77, 12
    got = obs_noise.oracle_obs_noisy(p, st, lay, seed, step).numpy()
    u = onp.obs_noise_u01(seed, np.arange(p.n) + p.env_offset, step)
    scale = np.array(lay.noise + (lay.height_noise,) * 187, np.float32)
    n = ((np.float32(2) * u - np.float32(1)) * scale).astype(np.float32)
    dof = st.dof_state.view(p.n, 12, 2).numpy()
    src = {"COMMAND": st.command, "BASE_LIN_VEL": st.base_lin_vel, "BASE_ANG_VEL": st.base_ang_vel,
           "GRAVITY_VEC": st.gravity_vec, "PROJECTED_GRAVITY": st.projected_gravity}
    x = np.concatenate([src[s].numpy() for s in lay.slots] + [dof[..., 0] - p.q0.numpy(), dof[..., 1],
                       st.obs[:, 36:72].numpy()], axis=1).astype(np.float32)
    head = (x * np.array(lay.scales, np.float32)).astype(np.float32) + n[:, :72]
    hts = np.clip(st.obs[:, 72:].numpy(), -1, 1) * np.float32(lay.height_scale) + n[:, 72:]
    want = np.clip(np.concatenate([head, hts], axis=1), -p.clip_obs, p.clip_obs).astype(np.float32)
    assert got.tobytes() == want.tobytes()
    if layout == "loud":
        assert (np.abs(got) == np.float32(p.clip_obs)).sum() > 50         # columns noised past +-clip_obs
        assert (got == -p.clip_obs).any() and (got == p.clip_obs).any()
    else:
        assert not np.array_equal(got, obs_layouts.oracle_obs(p, st, lay).numpy())
