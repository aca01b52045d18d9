"""The oracle's reward terms (oracle/shifu_oracle.py, fp32 torch on CPU) against the float64 reference
of every A1 opcode (oracle/a1_terms_f64.py), on seeded and crafted states.  The reference's six terms are
pinned by the golden replays of test_oracle_cpu.py; the legged_gym-style terms and non-default constants
have no recorded reference, so this is what pins them before the CUDA kernels are compared with both."""
import numpy as np
import pytest
import torch

from oracle import a1_terms_f64 as f64
from oracle import shifu_oracle as so
from tests import util

def all_terms(track_p1, leg_thr):
    """Every A1 opcode once; tracking / leg-collision constants edited."""
    params = {**so.A1_TERM_PARAMS, **util.EXTRA_TERM_PARAMS, "tracking_lin_vel": (1.0, track_p1),
              "tracking_ang_vel": (0.5, track_p1), "leg_collision": (-1.0, leg_thr)}
    return [(k, *params[k]) for k in (*so.A1_REWARD_TERMS, *so.A1_EXTRA_TERMS)]


def oracle_terms(n, s, terms, limits, feet, **kw):
    p = so.A1Params(n=n, terms=terms, feet_bodies=feet,
                    dof_pos_limits=None if limits is None else torch.from_numpy(limits), **kw)
    st = util.oracle_term_state(p, s)
    return p, st, so.a1_reward_terms(p, st)


def air_time_counts(n, s, feet, **kw):
    """Discrete parts of the oracle's feet_air_time, made visible through its value: with p1 = -1000 every
    first-contact foot adds 1000 + air (air < 1), so round(value / 1000) = #first_contact * moving; with
    every foot primed (swing > 0, last_contacts set) it is #feet * moving."""
    probe = [("feet_air_time", 1.0, -1000.0)]
    _, _, v = oracle_terms(n, s, probe, None, feet, **kw)
    primed = {**s, "swing": np.full_like(s["swing"], 0.5), "last": np.ones_like(s["last"])}
    _, _, w = oracle_terms(n, primed, probe, None, feet, **kw)
    return (np.rint(v["feet_air_time"].numpy() / 1000).astype(int),
            np.rint(w["feet_air_time"].numpy() / 1000).astype(int) == len(feet))


@pytest.mark.parametrize("n", [1, 33, 4099])
@pytest.mark.parametrize("track_p1,leg_thr", [(0.25, 0.1), (0.3, 0.37), (0.1, 1.0)])
@pytest.mark.parametrize("limits,feet", [("custom", (4, 8, 12, 16)), ("default", (4, 8, 12, 16)),
                                         ("custom", (8, 16)), ("default", (4, 12, 16))])
def test_oracle_terms_match_float64(n, track_p1, leg_thr, limits, feet):
    lim = util.dof_limits() if limits == "custom" else None
    consts = util.term_consts(lim, feet=feet)
    s = util.term_inputs(n, 1000 + n, leg_thr=leg_thr, limits=np.stack([consts["dof_lo"], consts["dof_hi"]], 1),
                         feet=feet)
    terms = all_terms(track_p1, leg_thr)
    p, st, got = oracle_terms(n, s, terms, lim, feet)
    leg_norm = torch.norm(torch.from_numpy(s["contact"][:, list(util.LEG_BODIES)]), dim=-1).numpy()
    want, mag, disc, swing, last = f64.eval_terms_f64(terms, s, consts, leg_norm=leg_norm)
    assert list(got) == [t[0] for t in terms]
    for q, (name, _, _) in enumerate(terms):
        f64.assert_within_bound(f"oracle:{name}", got[name].numpy(), want[q], mag[q], f64.BOUND_C[name])
    # discrete parts, exactly
    assert np.array_equal(-got["leg_collision"].numpy(), disc["leg_count"])
    assert np.array_equal(st.swing_time.numpy(), swing) and np.array_equal(st.last_contacts.numpy(), last)
    n_first, moving = air_time_counts(n, s, feet)
    assert np.array_equal(moving, disc["moving"])
    assert np.array_equal(n_first, disc["first_contact"].sum(1) * disc["moving"])
    if n > 100:            # the crafted rows reached both sides of every edge
        assert 0 < disc["leg_count"].sum() and (leg_norm == np.float32(leg_thr)).any()
        assert disc["dof_outside"].any() and disc["first_contact"].any() and not disc["moving"].all()
        assert (got["feet_air_time"].numpy() != 0).any()


def test_oracle_default_terms_unchanged():
    """The default term list is the reference's six terms with its literals, in its order."""
    p = so.A1Params(n=2)
    assert p.terms == [("tracking_lin_vel", 1.0, 0.25), ("tracking_ang_vel", 0.5, 0.25),
                       ("stabilizing_base", -2.0, -0.005), ("smoothing_action", -0.005, 0.0),
                       ("leg_collision", -1.0, 0.1), ("torques_penalize", -2e-5, 0.0)]


def test_oracle_reset_clears_air_time_state():
    n = 6
    p = so.A1Params(n=n, curriculum=False)
    st = util.oracle_term_state(p, util.term_inputs(n, 3))
    st.swing_time[:] = 0.3
    st.last_contacts[:] = True
    so.a1_reset_idx(p, st, torch.tensor([1, 4]))
    assert st.swing_time[[1, 4]].abs().sum() == 0 and not st.last_contacts[[1, 4]].any()
    assert (st.swing_time[[0, 2, 3, 5]] == np.float32(0.3)).all() and st.last_contacts[[0, 2, 3, 5]].all()
    p.air_time_reset = False
    so.a1_reset_idx(p, st, torch.tensor([0]))
    assert st.swing_time[0].eq(np.float32(0.3)).all() and st.last_contacts[0].all()
