"""The action head (legged_gym's own observation: 235 columns, or 48 blind) on a CPU-only checkout:
descriptor validation before any device check, ``ObsLayout`` and ``a1_desc`` widths, and the noise map of
the 235-column observation."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from tests import action_head, obs_layouts


def _create(d):
    from shifu_b200 import _native as nv
    lib = nv.load()
    out = C.c_void_p()
    return lib.shifu_ctx_create(0, C.byref(d), None, C.byref(out)), lib.shifu_last_error().decode()


def _no_gpu():
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: the descriptor would create a context")


@pytest.mark.parametrize("num_obs", [235, 48])
def test_action_head_needs_obs_layout_1(num_obs):
    from shifu_b200 import _native as nv, hotpath
    d = hotpath.a1_desc(64, num_obs=num_obs, obs=action_head.blind(action_head.legged_gym()))
    assert d.obs_layout == 1
    d.obs_layout = 0
    rc, msg = _create(d)
    assert rc == nv.E_RANGE, (rc, msg)
    assert "obs_layout = 1" in msg and str(num_obs) in msg, msg
    with pytest.raises(ValueError, match="ObsLayout"):
        hotpath.a1_desc(64, num_obs=num_obs)


def test_blind_action_head_with_height_noise_is_rejected():
    from shifu_b200 import _native as nv, hotpath
    d = hotpath.a1_desc(64, num_obs=48, obs=action_head.blind(action_head.legged_gym_noisy()))
    d.obs_height_noise = 0.1
    rc, msg = _create(d)
    assert rc == nv.E_RANGE, (rc, msg)
    assert "obs_height_noise" in msg and "blind" in msg, msg
    with pytest.raises(ValueError, match="height"):
        hotpath.a1_desc(64, num_obs=48, obs=action_head.legged_gym_noisy())


@pytest.mark.parametrize("num_obs", [0, 47, 49, 60, 234, 236, 258])
def test_other_widths_are_rejected(num_obs):
    from shifu_b200 import _native as nv, hotpath
    d = hotpath.a1_desc(64, num_obs=235, obs=action_head.legged_gym())
    d.num_obs = num_obs
    rc, msg = _create(d)
    assert rc == nv.E_RANGE, (rc, msg)
    assert "235 or 48 with the action head" in msg and f" {num_obs} " in msg, msg
    with pytest.raises(ValueError, match="num_obs"):
        hotpath.a1_desc(64, num_obs=num_obs, obs=action_head.legged_gym())


def test_action_head_descriptors_pass_validation():
    from shifu_b200 import _native as nv, hotpath
    _no_gpu()
    for num_obs, lay in ((235, action_head.legged_gym()), (235, action_head.legged_gym_noisy()),
                         (235, action_head.loud()), (48, action_head.blind(action_head.legged_gym_noisy()))):
        d = hotpath.a1_desc(64, num_obs=num_obs, obs=lay)
        assert _create(d)[0] == nv.E_NODEVICE, num_obs            # validation passed: only the device is missing


def test_action_head_reads_the_first_48_scales_and_noise_scales():
    from shifu_b200 import _native as nv, hotpath
    _no_gpu()
    d = hotpath.a1_desc(64, num_obs=235, obs=action_head.legged_gym())
    assert list(d.obs_scale[48:]) == [0.0] * 24 and list(d.obs_noise[48:]) == [0.0] * 24
    for j in (48, 60, 71):
        d.obs_scale[j], d.obs_noise[j] = math.nan, math.inf         # not read
    assert _create(d)[0] == nv.E_NODEVICE
    d.obs_noise[47] = math.nan                                      # read
    rc, msg = _create(d)
    assert rc == nv.E_RANGE and "obs_noise[47]" in msg, msg


def test_obs_layout_widths():
    from shifu_b200 import hotpath
    from shifu_b200.hotpath import ObsLayout
    lay = action_head.legged_gym()
    assert lay.head == 48 and len(lay.scales) == 48 and len(lay.noise) == 48
    assert ObsLayout().head == 72 and len(ObsLayout().noise) == 72
    assert ObsLayout(scales=(1.0,) * 48).noise == (0.0,) * 48
    # never the reference observation: identity scales and reference slots still write obs_layout = 1
    ident = ObsLayout(scales=(1.0,) * 48)
    assert not ident.is_reference()
    d = hotpath.a1_desc(8, num_obs=235, obs=ident)
    assert d.obs_layout == 1 and d.num_obs == 235
    for bad in (dict(scales=(1.0,) * 60), dict(scales=(1.0,) * 48, noise=(0.0,) * 72),
                dict(scales=(1.0,) * 72, noise=(0.0,) * 48)):
        with pytest.raises(ValueError):
            ObsLayout(**bad)


def test_a1_desc_widths():
    from shifu_b200 import hotpath
    lay = action_head.legged_gym_noisy()
    d = hotpath.a1_desc(8, num_obs=235, obs=lay)
    assert d.num_obs == 235 and d.obs_layout == 1
    assert np.array_equal(np.array(d.obs_scale[:48], np.float32), np.array(lay.scales, np.float32))
    assert np.array_equal(np.array(d.obs_noise[:48], np.float32), np.array(lay.noise, np.float32))
    assert np.float32(d.obs_height_noise) == np.float32(lay.height_noise)
    assert hotpath.a1_desc(8, num_obs=48, obs=action_head.blind(lay)).num_obs == 48
    with pytest.raises(ValueError, match="the layout has 48 columns"):
        hotpath.a1_desc(8, num_obs=259, obs=lay)                   # a 48-column layout, a 72-column head
    with pytest.raises(ValueError, match="72 columns"):
        hotpath.a1_desc(8, num_obs=235, obs=obs_layouts.legged_gym())
    # the 235 descriptor equals the 259 one except num_obs and the scales / noise of columns 36-71
    lay72 = action_head.with_history(lay)
    a, b = hotpath.a1_desc(8, num_obs=235, obs=lay), hotpath.a1_desc(8, obs=lay72)
    for j in range(36, 72):
        b.obs_scale[j] = a.obs_scale[j]
        b.obs_noise[j] = a.obs_noise[j]
    b.num_obs = 235
    assert bytes(a) == bytes(b)


def test_235_noise_map_covers_every_column_once():
    from shifu_b200.utils import philox
    word, lane = action_head.noise_map()
    assert len(word) == 235
    head_words = {3 * i + r for i in range(6) for r in (0, 1)}
    assert set(word[:48].tolist()) == head_words
    assert set(word[48:].tolist()) == set(range(18, 65))
    assert len(set(word.tolist())) == 12 + 47                       # 59 evaluations per env and step
    assert not any(w % 3 == 2 and w < 18 for w in word.tolist())    # words 3i + 2 are not drawn
    pairs = list(zip(word.tolist(), lane.tolist()))
    assert len(set(pairs)) == 235                                   # no two columns share a (word, lane)
    # the kernels' width-aware formula (shifu_b200.utils.philox) gives the same map
    w, ln = philox.obs_noise_slots(48)
    assert np.array_equal(w.numpy(), word) and np.array_equal(ln.numpy(), lane)
    # and the 48-column observation is the first 48 columns of it
    assert np.array_equal(w[:48].numpy(), word[:48])


@pytest.mark.parametrize("seed,step", [(0x5EED, 1), (2**40 + 17, 2**33 + 5)])
def test_numpy_and_torch_draws_agree(seed, step):
    from shifu_b200.utils import philox
    ids = np.array([0, 1, 31, 32, 1000, 2**31 + 3])
    want = action_head.noise_u01(seed, ids, step)
    got = philox.obs_noise_u01(seed, torch.from_numpy(ids), step, head=48).numpy()
    assert got.shape == (len(ids), 235)
    assert np.array_equal(got, want)
    # the 235-column draws are columns 0-47 and 72-258 of the 259-column ones
    full = philox.obs_noise_u01(seed, torch.from_numpy(ids), step).numpy()
    assert np.array_equal(got, full[:, action_head.KEPT])
