"""The reward-term library on the B200: every A1 opcode of ``shifu_a1_eval_terms`` against the float64
reference (oracle/a1_terms_f64.py) and the fp32 oracle; the fused step with non-default term lists
(both instantiations of the pipelined kernel, the phased kernel, the ragged tail) against the extended
oracle; and the property the term compiler's safety check relies on: the kernel it verifies computes,
bit for bit, what the fused step accumulates."""
import functools

import numpy as np
import pytest
import torch

from oracle import a1_terms_f64 as f64
from oracle import shifu_oracle as so
from tests import util

pytestmark = pytest.mark.gpu

ALL_TERMS = (*so.A1_REWARD_TERMS, *so.A1_EXTRA_TERMS)


@functools.lru_cache(maxsize=1)
def _height_map():
    from shifu_b200.sim import fake_isaacgym
    fake_isaacgym.install("cpu")
    from shifu_b200.configs import TerrainEnvConfig
    from shifu_b200.utils.heightmap import Terrain
    np.random.seed(0)
    ter = Terrain(TerrainEnvConfig().terrain, 64)
    return ter.heightsamples, torch.from_numpy(ter.env_origins).float()


def _terrain(n):
    hs, origins = _height_map()
    types = torch.div(torch.arange(n), n / origins.shape[1], rounding_mode='floor').to(torch.long)
    levels0 = torch.from_numpy(np.random.RandomState(3).randint(0, 6, size=n))
    return hs, origins, types, origins[levels0, types]


# ---------------------------------------------------------------------------------------------
# (a) shifu_a1_eval_terms, opcode by opcode
# ---------------------------------------------------------------------------------------------

def _load_inputs(hp, s):
    n, nf = hp.n, s["swing"].shape[1]
    c = lambda k: torch.from_numpy(np.ascontiguousarray(s[k])).to(hp.device)
    hp.command.copy_(c("command"))
    hp.base_lin_vel.copy_(c("lin"))
    hp.base_ang_vel.copy_(c("ang"))
    hp.projected_gravity.copy_(c("pg"))
    hp.dof_state.view(n, 12, 2).copy_(c("dof"))
    hp.history.copy_(c("hist"))
    hp.actions.copy_(c("act"))
    hp.torques.copy_(c("tau"))
    hp.contact_state.view(n, 17, 3).copy_(c("contact"))
    hp.root_state[:, 2] = c("base_z")
    hp.swing_time[:, :nf] = c("swing")
    hp.last_contacts[:, :nf] = c("last")


def _eval_kernel(n, s, terms, lim, feet):
    """shifu_a1_eval_terms of ``terms`` [(name, p0, p1)] on ``s``: values and the air-time state it leaves."""
    hp = util.make_cuda_a1(n, np.zeros((4, 4), np.int16), torch.zeros(1, 1, 3), torch.zeros(n, dtype=torch.long),
                           torch.zeros(n, 3), terms=[t[0] for t in terms],
                           term_params={t[0]: (t[1], t[2]) for t in terms}, dof_pos_limits=lim, feet_bodies=feet)
    _load_inputs(hp, s)
    out = hp.eval_terms().cpu().numpy()
    nf = len(feet)
    return out, hp.swing_time[:, :nf].cpu().numpy(), hp.last_contacts[:, :nf].cpu().numpy()


def _lists(track_p1, leg_thr):
    params = {**so.A1_TERM_PARAMS, **util.EXTRA_TERM_PARAMS, "tracking_lin_vel": (1.0, track_p1),
              "tracking_ang_vel": (0.5, track_p1), "leg_collision": (-1.0, leg_thr)}
    one = lambda names: [(k, *params[k]) for k in names]
    # every opcode alone, then two lists of SHIFU_MAX_REWARD_TERMS = 8 that cover all 14 between them
    return ([one([k]) for k in ALL_TERMS] + [one(ALL_TERMS[:8]), one(ALL_TERMS[6:])])


@pytest.mark.parametrize("n", [1, 31, 33, 4099])
@pytest.mark.parametrize("track_p1,leg_thr,limits,feet", [(0.25, 0.1, "custom", (4, 8, 12, 16)),
                                                          (0.3, 0.37, "default", (4, 8, 12, 16)),
                                                          (0.1, 1.0, "custom", (8, 16))])
def test_eval_terms_vs_float64(n, track_p1, leg_thr, limits, feet):
    lim = util.dof_limits() if limits == "custom" else None
    consts = util.term_consts(lim, feet=feet)
    s = util.term_inputs(n, 2000 + n, leg_thr=leg_thr, limits=np.stack([consts["dof_lo"], consts["dof_hi"]], 1),
                         feet=feet)
    leg_norm = torch.norm(torch.from_numpy(s["contact"][:, list(util.LEG_BODIES)]), dim=-1).numpy()
    seen = {}
    for terms in _lists(track_p1, leg_thr):
        names = [t[0] for t in terms]
        got, swing, last = _eval_kernel(n, s, terms, lim, feet)
        assert got.shape == (len(terms), n)
        want, mag, disc, want_swing, want_last = f64.eval_terms_f64(terms, s, consts, leg_norm=leg_norm)
        p = so.A1Params(n=n, terms=terms, feet_bodies=feet, dof_pos_limits=None if lim is None else torch.from_numpy(lim))
        st = util.oracle_term_state(p, s)
        ora = so.a1_reward_terms(p, st)
        for q, name in enumerate(names):
            f64.assert_within_bound(f"{names}:{name}", got[q], want[q], mag[q], f64.BOUND_C[name])
            util.assert_close(f"{names}:{name} vs oracle", got[q], ora[name].numpy(), exact=False)
        if "leg_collision" in names:
            assert np.array_equal(-got[names.index("leg_collision")], disc["leg_count"])
        # the air-time state the call leaves (unchanged unless the term is listed)
        assert np.array_equal(swing, want_swing) and np.array_equal(last, want_last)
        assert np.array_equal(swing, st.swing_time.numpy()) and np.array_equal(last, st.last_contacts.numpy())
        seen.update(disc)
    # first_contact and the moving gate: with p1 = -1000 each first-contact foot adds 1000 + air (air < 1)
    probe = [("feet_air_time", 1.0, -1000.0)]
    got, _, _ = _eval_kernel(n, s, probe, lim, feet)
    _, _, disc, _, _ = f64.eval_terms_f64(probe, s, consts)
    assert np.array_equal(np.rint(got[0] / 1000).astype(int), disc["first_contact"].sum(1) * disc["moving"])
    primed = {**s, "swing": np.full_like(s["swing"], 0.5), "last": np.ones_like(s["last"])}
    got, _, _ = _eval_kernel(n, primed, probe, lim, feet)
    assert np.array_equal(np.rint(got[0] / 1000).astype(int) == len(feet), disc["moving"])
    if n > 100:            # the crafted rows reached both sides of every edge
        assert (leg_norm == np.float32(leg_thr)).any() and seen["leg_count"].any() and not seen["leg_count"].all()
        assert seen["first_contact"].any() and seen["moving"].any() and not seen["moving"].all()
        assert seen["dof_outside"].any()


# ---------------------------------------------------------------------------------------------
# (b) the fused step with non-default term lists against the extended oracle
# ---------------------------------------------------------------------------------------------

SNAP_KW = dict(p_base=0.05, p_leg=0.3)


def _edge_contacts(snap, leg_thr, step):
    """Overwrite part of the snapshot's contact rows: leg forces with fp32 norm exactly ``leg_thr`` and
    one ulp either side, base forces exactly at the termination threshold 1.0 and one ulp either side."""
    n = snap.contact.shape[0]
    legs = util.norm_edge_forces(leg_thr, 64, seed=step)
    base = util.norm_edge_forces(1.0, 64, seed=100 + step)
    for i in range(0, n, 5):
        j = i // 5
        snap.contact[i, util.LEG_BODIES[j % 8]] = torch.from_numpy(legs[j % 3][(j // 3) % 64])
        if j % 4 == 0:
            snap.contact[i, 0] = torch.from_numpy(base[(j // 4) % 3][(j // 12) % 64])


def _fused_vs_oracle(list_name, n, carry, heights, steps=3, seed=41):
    kw = util.term_list(list_name)
    hs, origins, types, env_origins = _terrain(n)
    p, st = util.make_oracle_a1(n, hs, origins, types, env_origins, **kw)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=carry, want_measured_heights=heights, **kw)
    leg_thr = dict(zip(kw["terms"], [p1 for _, _, p1 in p.terms])).get("leg_collision", 0.1)

    def snap_at(t):
        from shifu_b200.sim.synthetic import a1_snapshot
        snap = a1_snapshot(seed, t, n, **SNAP_KW)
        if list_name == "L3":
            _edge_contacts(snap, leg_thr, t)
        return snap

    snap = snap_at(0)
    so.a1_reset(p, st, snap)
    hp.reset_idx(None)
    if carry:
        hp.body_frame()
    util.cuda_a1_step(hp, snap, torch.zeros(n, 12))
    skip = ("base_lin_vel", "base_ang_vel", "projected_gravity") if carry else ()
    util.compare_a1(util.cuda_a1_outputs(hp), util.oracle_a1_outputs(st), f"{list_name}/n{n}/reset", skip=skip)
    ep = torch.from_numpy(np.random.RandomState(n).randint(0, 500, size=n))
    st.ep_len[:] = ep
    hp.ep_len.copy_(ep)
    seen = dict(air=0, reset_swing=0, dof_out=0, leg_over=0, leg_edge=0, base_edge=0)
    feet = list(p.feet_bodies)
    lo, hi = p.dof_pos_limits[:, 0], p.dof_pos_limits[:, 1]
    for t in range(1, steps + 1):
        snap = snap_at(t)
        # what the air-time update leaves before reset_idx clears it: non-zero unless the foot touches
        left = ~((snap.contact[:, feet, 2] > p.feet_contact_force) | st.last_contacts)
        so.a1_step(p, st, snap.actions, snap)
        util.cuda_a1_step(hp, snap, snap.actions)
        got = util.cuda_a1_outputs(hp)
        util.compare_a1(got, util.oracle_a1_outputs(st), f"{list_name}/n{n}/s{t}", skip=skip)
        assert np.array_equal(got["reset_ids"], st.reset_ids.numpy()), f"reset ids differ at step {t}"
        assert sorted(k[len("ep_sum/"):] for k in got if k.startswith("ep_sum/")) == sorted(kw["terms"])
        if "feet_air_time" in kw["terms"]:
            seen["air"] += int((st.ep_sums["feet_air_time"] != 0).sum())
            seen["reset_swing"] += int(left[st.reset_ids].any(dim=1).sum())
        q = snap.dof[4][..., 0]
        seen["dof_out"] += int(((q < lo) | (q > hi)).sum())
        nrm = torch.norm(snap.contact[:, list(util.LEG_BODIES)], dim=-1)
        seen["leg_over"] += int((nrm > np.float32(leg_thr)).sum())
        seen["leg_edge"] += int((nrm == np.float32(leg_thr)).sum())
        seen["base_edge"] += int((torch.norm(snap.contact[:, 0], dim=-1) == 1.0).sum())
    # the run was not vacuous
    assert seen["leg_over"] > 0
    if "feet_air_time" in kw["terms"]:
        assert seen["air"] > 0 and seen["reset_swing"] > 0, seen
    if "dof_pos_limits" in kw["terms"]:
        assert seen["dof_out"] > 0
    if list_name == "L3":
        assert seen["leg_edge"] > 0 and seen["base_edge"] > 0, seen
    return hp, st


@pytest.mark.parametrize("list_name", ["L1", "L2", "L3"])
@pytest.mark.parametrize("n,carry,heights", [
    (33, False, True),                 # the barrier-phased kernel only
    (32 * 1200 + 7, False, True),      # pipelined kernel on full tiles + the phased kernel on the ragged tail
    (65536, True, False),              # the benchmarked layout (carried body frame, no measured_heights)
])
def test_fused_step_term_lists_vs_oracle(list_name, n, carry, heights):
    _fused_vs_oracle(list_name, n, carry, heights)


# ---------------------------------------------------------------------------------------------
# (d) the term compiler verifies the kernel the step runs
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("list_name", ["L1", "L2", "L3"])
def test_eval_terms_is_what_the_step_accumulates(list_name):
    """terms.verify_a1_terms compares user hooks with shifu_a1_eval_terms; full tiles of a step run the
    pipelined kernel, which stages its rows and accumulates the terms its own way (both evaluate
    a1_reward_term).  On the simulator state of a live step, every non-reset env's episode sums must grow
    by exactly the eval_terms values, and rew must be their sum."""
    from shifu_b200.sim.synthetic import a1_snapshot
    n = 32 * 300                                     # full tiles only: every env goes through the pipelined kernel
    kw = util.term_list(list_name)
    hs, origins, types, env_origins = _terrain(n)
    hp = util.make_cuda_a1(n, hs, origins, types, env_origins, carry=True, want_measured_heights=False, **kw)
    hp.reset_idx(None)
    util.cuda_a1_step(hp, a1_snapshot(7, 0, n, **SNAP_KW), torch.zeros(n, 12))
    hp.ep_len.copy_(torch.from_numpy(np.random.RandomState(2).randint(0, 500, size=n)))
    fired = 0
    for t in range(1, 4):
        saved = {}

        def verify(hp):
            saved["sums"] = {k: v.clone() for k, v in hp.ep_sums.items()}
            sw, lc = hp.swing_time.clone(), hp.last_contacts.clone()
            saved["terms"] = hp.eval_terms()
            saved["swing"] = hp.swing_time.clone()
            hp.swing_time.copy_(sw)
            hp.last_contacts.copy_(lc)

        snap = a1_snapshot(7, t, n, **SNAP_KW)
        util.cuda_a1_step(hp, snap, snap.actions, before_post=verify)
        ev, keep = saved["terms"], ~hp.reset_buf
        rew = torch.zeros(n, device=hp.device)
        for q, k in enumerate(hp.terms):
            want = saved["sums"][k] + ev[q]
            bad = (want != hp.ep_sums[k]) & keep
            assert not bad.any(), f"{list_name} step {t}: {k} differs at {int(bad.sum())} envs"
            rew = rew + ev[q]
        assert torch.equal(rew, hp.rew_buf), f"{list_name} step {t}: rew is not the sum of eval_terms"
        if "feet_air_time" in hp.terms:
            fired += int((ev[hp.terms.index("feet_air_time")] != 0).sum())
            kept = keep.unsqueeze(1).expand_as(hp.swing_time)
            assert torch.equal(saved["swing"][kept], hp.swing_time[kept])
        assert int(keep.sum()) > n // 2 and int((~keep).sum()) > 0
    if "feet_air_time" in hp.terms:
        assert fired > 0
