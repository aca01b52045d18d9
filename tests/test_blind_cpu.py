"""Blind A1 descriptors on a CPU-only checkout: num_obs must be 72 or 259, and a blind observation takes no
height noise.  Both are checked before any device check."""
import ctypes as C

import pytest
import torch

from tests import obs_layouts, obs_noise


def _create(d):
    from shifu_b200 import _native as nv
    lib = nv.load()
    out = C.c_void_p()
    return lib.shifu_ctx_create(0, C.byref(d), None, C.byref(out)), lib.shifu_last_error().decode()


@pytest.mark.parametrize("num_obs", [0, 71, 73, 187, 258, 260, 331])
def test_num_obs_other_than_72_or_259_is_rejected(num_obs):
    from shifu_b200 import _native as nv, hotpath
    d = hotpath.a1_desc(64)
    d.num_obs = num_obs
    rc, msg = _create(d)
    assert rc == nv.E_RANGE, (rc, msg)
    assert "obs=259 or 72" in msg and f" {num_obs} " in msg, msg
    with pytest.raises(ValueError, match="num_obs"):
        hotpath.a1_desc(64, num_obs=num_obs)


def test_blind_with_height_noise_is_rejected():
    from shifu_b200 import _native as nv, hotpath
    d = hotpath.a1_desc(64, num_obs=72, obs=obs_layouts.legged_gym())
    assert d.num_obs == 72 and d.obs_layout == 1
    d.obs_height_noise = 0.1
    rc, msg = _create(d)
    assert rc == nv.E_RANGE, (rc, msg)
    assert "obs_height_noise" in msg and "blind" in msg, msg
    with pytest.raises(ValueError, match="height"):
        hotpath.a1_desc(64, num_obs=72, obs=obs_noise.legged_gym_noisy())


def test_blind_descriptors_pass_validation():
    from shifu_b200 import _native as nv, hotpath
    from shifu_b200.hotpath import ObsLayout
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: the descriptor would create a context")
    lay = obs_noise.legged_gym_noisy()
    blind_noisy = ObsLayout(lay.slots, lay.scales, lay.height_scale, lay.noise, 0.0)
    for obs in (None, obs_layouts.legged_gym(), blind_noisy):
        d = hotpath.a1_desc(64, num_obs=72, obs=obs)
        assert _create(d)[0] == nv.E_NODEVICE
    # the blind descriptor differs from the sighted one in num_obs alone
    a, b = hotpath.a1_desc(64, num_obs=72, obs=blind_noisy), hotpath.a1_desc(64, obs=blind_noisy)
    b.num_obs = 72
    assert bytes(a) == bytes(b)


def test_blind_does_not_read_the_height_scale():
    import math
    from shifu_b200 import _native as nv, hotpath
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: the descriptor would create a context")
    for v in (math.nan, math.inf, 5.0):
        d = hotpath.a1_desc(64, num_obs=72, obs=obs_layouts.legged_gym())
        d.obs_height_scale = v
        assert _create(d)[0] == nv.E_NODEVICE, v          # validation passed: only the device is missing
        d.num_obs = 259
        if not math.isfinite(v):
            assert _create(d)[0] == nv.E_RANGE            # the sighted step reads it
