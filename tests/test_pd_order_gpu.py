"""The PD substep's sweep order changes no result.

``shifu_pd_torque`` sweeps the envs upward or downward depending on the decimation substep it is
given (so that consecutive substeps reuse what the previous one left in L2).  Every substep must
write every quad of ``torques`` (and of ``actions`` when it clips raw actions) exactly once, with
the values substep 0 computes.  The sizes put the grid-stride tail at both ends of the range.
"""

import numpy as np
import pytest
import torch

from tests import util

pytestmark = pytest.mark.gpu

SUBSTEPS = range(4)


def _hot_path(n):
    z, meta = util.load_golden("a1_small")
    rs = np.random.RandomState(n % 9973)
    types = torch.from_numpy(rs.randint(0, meta["num_cols"], size=n)).long()
    levels = torch.from_numpy(rs.randint(0, meta["max_terrain_level"], size=n)).long()
    origins = torch.from_numpy(z["terrain_origins"]).float()
    return util.make_cuda_a1(n, z["height_samples"], origins, types, origins[levels, types],
                             border_size=int(meta["border_size"]), max_terrain_level=meta["max_terrain_level"],
                             num_cols=meta["num_cols"], want_measured_heights=False)


def _pd(hp, a_in, a_out, substep):
    from shifu_b200 import _native as nv
    return hp.lib.shifu_pd_torque(hp.ctx.handle, nv.ptr(a_in), nv.ptr(a_out), nv.ptr(hp.dof_state),
                                  nv.ptr(hp.torques), substep, nv.current_stream())


@pytest.mark.parametrize("n", [1, 2, 33, 4099, 100003, 1 << 20])
def test_every_substep_matches_substep_zero(n):
    from shifu_b200 import _native as nv
    hp = _hot_path(n)
    g = torch.Generator(device="cuda").manual_seed(n)
    raw = (torch.randn(n, 12, device="cuda", generator=g) * 3).contiguous()     # some beyond the clip
    hp.dof_state.copy_(torch.randn(n * 12, 2, device="cuda", generator=g))
    nan = float("nan")

    # substep 0 on raw actions: clipped actions + torques
    hp.torques.fill_(nan)
    hp.actions.fill_(nan)
    nv.check(_pd(hp, raw, hp.actions, 0))
    want_act, want_tau_raw = hp.actions.clone(), hp.torques.clone()
    assert not torch.isnan(want_act).any() and not torch.isnan(want_tau_raw).any()
    # substep 0 on the clipped actions (what the later substeps read)
    hp.torques.fill_(nan)
    nv.check(_pd(hp, want_act, None, 0))
    want_tau = hp.torques.clone()
    assert not torch.isnan(want_tau).any()

    for s in SUBSTEPS:
        hp.torques.fill_(nan)
        hp.actions.fill_(nan)
        nv.check(_pd(hp, raw, hp.actions, s))
        torch.cuda.synchronize()
        assert torch.equal(hp.actions, want_act), f"actions, substep {s}"
        assert torch.equal(hp.torques, want_tau_raw), f"torques from raw actions, substep {s}"

        hp.torques.fill_(nan)
        nv.check(_pd(hp, want_act, None, s))
        torch.cuda.synchronize()
        assert torch.equal(hp.torques, want_tau), f"torques, substep {s}"


def test_negative_substep_is_rejected():
    from shifu_b200 import _native as nv
    hp = _hot_path(64)
    hp.torques.fill_(float("nan"))
    assert _pd(hp, hp.actions, None, -1) == nv.E_RANGE
    assert b"substep" in hp.lib.shifu_last_error()
    torch.cuda.synchronize()
    assert torch.isnan(hp.torques).all()          # nothing was launched
