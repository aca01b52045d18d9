"""The observation layout on a CPU-only checkout: descriptor validation happens before any device check,
hotpath.a1_desc writes the layout it is given, and the oracle's layout-aware observation reproduces the
reference's with an explicit reference layout."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from tests import obs_layouts, util


def _create(d):
    from shifu_b200 import _native as nv
    lib = nv.load()
    out = C.c_void_p()
    return lib.shifu_ctx_create(0, C.byref(d), None, C.byref(out)), lib.shifu_last_error().decode()


@pytest.mark.parametrize("field,value", [
    ("obs_layout", 2), ("obs_layout", -1),
    ("obs_vec_src", -1), ("obs_vec_src", 5),
    ("obs_scale", math.nan), ("obs_scale", math.inf), ("obs_scale", -math.inf),
    ("obs_height_scale", math.nan), ("obs_height_scale", math.inf),
])
def test_bad_layout_is_rejected_before_the_device_check(field, value):
    from shifu_b200 import _native as nv, hotpath
    d = hotpath.a1_desc(64, obs=obs_layouts.legged_gym())
    assert d.obs_layout == 1
    if field in ("obs_layout", "obs_height_scale"):
        setattr(d, field, value)
    elif field == "obs_vec_src":
        d.obs_vec_src[2] = value
    else:
        d.obs_scale[40] = value
    rc, msg = _create(d)
    assert rc == nv.E_RANGE, (rc, msg)
    assert field in msg


def test_valid_layout_passes_validation():
    """A valid layout-1 descriptor gets past the argument checks (to the device check, or to a context)."""
    from shifu_b200 import _native as nv, hotpath
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: the descriptor would create a context")
    for make in obs_layouts.LAYOUTS.values():
        assert _create(hotpath.a1_desc(64, obs=make()))[0] == nv.E_NODEVICE


def test_a1_desc_writes_the_layout():
    from shifu_b200 import _native as nv, hotpath
    assert hotpath.a1_desc(8).obs_layout == 0
    assert hotpath.a1_desc(8, obs=None).obs_layout == 0
    ref = hotpath.ObsLayout()
    assert ref.is_reference() and hotpath.a1_desc(8, obs=ref).obs_layout == 0
    d = hotpath.a1_desc(8, obs=obs_layouts.legged_gym())
    assert d.obs_layout == 1
    assert list(d.obs_vec_src) == [nv.OBS_BASE_LIN_VEL, nv.OBS_BASE_ANG_VEL, nv.OBS_PROJECTED_GRAVITY, nv.OBS_COMMAND]
    want = np.array([2, 2, 2, .25, .25, .25, 1, 1, 1, 2, 2, .25] + [1] * 12 + [0.05] * 12 + [1] * 36, np.float32)
    assert np.array_equal(np.array(d.obs_scale, np.float32), want)
    assert d.obs_height_scale == 5.0
    d1 = hotpath.a1_desc(8, obs=obs_layouts.d1_fix())
    assert d1.obs_layout == 1 and d1.obs_vec_src[3] == nv.OBS_PROJECTED_GRAVITY
    assert list(d1.obs_scale) == [1.0] * 72 and d1.obs_height_scale == 1.0


def test_obs_layout_values():
    from shifu_b200.hotpath import ObsLayout
    lay = ObsLayout(scales=(0.1,) * 72)
    assert lay.scales[0] == float(np.float32(0.1)) and not lay.is_reference()
    for bad in (dict(slots=("COMMAND",) * 3), dict(slots=("COMMAND", "X", "COMMAND", "COMMAND")),
                dict(scales=(1.0,) * 71), dict(height_scale=math.nan)):
        with pytest.raises(ValueError):
            ObsLayout(**bad)


def test_oracle_reference_layout_is_the_reference_observation_on_a1_small():
    """The layout observation of the test oracle (obs_layouts.oracle_obs), with the reference layout, is
    the oracle's own observation bit for bit on every step of the a1_small replay (and that is the
    fixture's)."""
    from oracle import shifu_oracle as so
    from shifu_b200.hotpath import ObsLayout
    z, meta = util.load_golden("a1_small")
    n = meta["n"]
    p, st = util.make_oracle_a1(n, z["height_samples"], z["terrain_origins"], z["terrain_types"],
                                z["env_origins_init"], border_size=int(meta["border_size"]),
                                max_terrain_level=meta["max_terrain_level"], num_cols=meta["num_cols"],
                                rng_seed=meta["rng_seed"])
    so.a1_reset(p, st, util.golden_snap(z, 0))
    st.ep_len[:] = torch.from_numpy(z["ep_len_init"])
    st.terrain_levels[:] = torch.from_numpy(z["levels_init"])
    for t in range(meta["steps"] + 1):
        if t > 0:
            snap = util.golden_snap(z, t)
            so.a1_step(p, st, snap.actions, snap)
        assert np.array_equal(st.obs.numpy(), z[f"s{t}/out/obs"])
        got = obs_layouts.oracle_obs(p, st, ObsLayout())
        assert got.numpy().tobytes() == st.obs.numpy().tobytes(), f"step {t}"


def test_oracle_applies_a_layout():
    """The test oracle's layout: slot sources, one fp32 rounding per multiply, heights clipped then scaled,
    the final clip."""
    from oracle import shifu_oracle as so
    n = 5
    lay = obs_layouts.legged_gym()
    p = so.A1Params(n=n)
    st = so.a1_new_state(p, torch.zeros(2, 2, dtype=torch.int16), torch.zeros(1, 1, 3), torch.zeros(n, dtype=torch.long),
                         torch.zeros(n, 3))
    g = torch.Generator().manual_seed(0)
    for name in ("command", "base_lin_vel", "base_ang_vel", "projected_gravity", "history"):
        getattr(st, name).copy_(torch.randn(getattr(st, name).shape, generator=g))
    st.dof_state.copy_(torch.randn(st.dof_state.shape, generator=g))
    st.root_state[:, 2] = torch.tensor([0.5, 2.0, -2.0, 0.7, 0.1])
    st.measured_heights = torch.zeros(n, 187)
    so.a1_compute_observations(p, st)
    got = obs_layouts.oracle_obs(p, st, lay)
    sc = torch.tensor(lay.scales)
    assert torch.equal(got[:, 0:3], st.base_lin_vel * sc[0:3])
    assert torch.equal(got[:, 6:9], st.projected_gravity)
    assert torch.equal(got[:, 9:12], st.command * sc[9:12])
    assert torch.equal(got[:, 24:36], st.dof_state.view(n, 12, 2)[..., 1] * np.float32(0.05))
    assert torch.equal(got[:, 36:72], st.obs[:, 36:72])
    assert torch.allclose(got[:, 72], torch.tensor([0.0, 5.0, -5.0, 0.2 * 5, -0.4 * 5]), atol=1e-6)
    big = obs_layouts.extreme()
    assert float(obs_layouts.oracle_obs(p, st, big).abs().max()) == p.clip_obs
