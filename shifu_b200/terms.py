"""Reward / observation term compiler (SURVEY.md §8f row N1): ``build_reward_functions()`` lists -> fused term
descriptors, ``compute_observations`` -> the fused observation layout (:func:`compile_a1_obs`).

The reference's "registry" is a plain list of bound methods whose weights are literals inside each
body (``shifu/gym/env.py:78-80,160-166,180-185``; ``a1_conditional.py:152-192``).  To fuse such a
list the kernel needs, per term, an opcode of its term library (``enum ShifuRewardTerm``) and the
term's constants.  This module gets both WITHOUT reading source text:

1. **match** — the method name (``fn.__name__``, prefixes ``_reward_`` / ``reward_`` / ``rew_`` stripped)
   selects a library entry; every entry is a parametric form ``f(state; p0, p1)``;
2. **fit** — the user's Python hook is evaluated on a handful of crafted device states (all zeros
   except one input) which determine ``p0`` / ``p1`` exactly or — for the two constants that only
   come out of a logarithm — up to rounding, in which case the value is snapped to the matching
   literal in the method's ``co_consts``;
3. **verify** — the hook and the kernel (``shifu_a1_eval_terms``) are evaluated on the same seeded
   random state; any term that disagrees beyond the parity tolerance makes the compiler refuse
   (the env then stays in user-hook mode: torch hooks on CUDA tensors).

So a user who edits a literal inside a known term gets the edited constant in the fused kernel, and
a user who changes the *shape* of a term gets a loud refusal instead of silently different rewards.
"""
from __future__ import annotations

import math
from contextlib import contextmanager
from dataclasses import dataclass
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch

from . import _native as nv
from .hotpath import OBS_SOURCES, ObsLayout

RTOL, ATOL = 2e-5, 2e-6


class TermMismatch(Exception):
    """The user's hook is not (numerically) the library term it was matched to."""


class NotFusable(Exception):
    """A hook of the env is not what the fused kernel computes; the message names the hook and the reason."""


def check_close(a: torch.Tensor, b: torch.Tensor, what: str, rtol=1e-6, atol=1e-7):
    """Raise NotFusable unless the hook's result ``a`` is the fused definition ``b``."""
    if a.shape != b.shape:
        raise NotFusable(f"{what}: shape {tuple(a.shape)} != {tuple(b.shape)}")
    if a.dtype == torch.bool or b.dtype == torch.bool:
        bad = int((a.bool() != b.bool()).sum())
    else:
        bad = int(((a.float() - b.float()).abs() > atol + rtol * b.float().abs()).sum())
    if bad:
        raise NotFusable(f"{what}: the Python hook differs from the fused kernel's definition on {bad} entries")


@dataclass
class CompiledTerm:
    name: str
    code: int
    p0: float
    p1: float
    extra: Optional[dict] = None        # descriptor-level constants of the term (a1_desc keyword -> value)


def _strip(name: str) -> str:
    for prefix in ("_reward_", "reward_", "rew_"):
        if name.startswith(prefix):
            return name[len(prefix):]
    return name


# name -> opcode (a1_conditional.py names + the legged_gym vocabulary)
A1_NAMES: Dict[str, int] = {
    "tracking_lin_vel": nv.REW_TRACKING_LIN_VEL, "tracking_ang_vel": nv.REW_TRACKING_ANG_VEL,
    "stabilizing_base": nv.REW_STABILIZING_BASE, "smoothing_action": nv.REW_SMOOTHING_ACTION,
    "leg_collision": nv.REW_LEG_COLLISION, "collision": nv.REW_LEG_COLLISION,
    "torques_penalize": nv.REW_TORQUES, "torques": nv.REW_TORQUES,
    "lin_vel_z": nv.REW_LIN_VEL_Z, "ang_vel_xy": nv.REW_ANG_VEL_XY, "orientation": nv.REW_ORIENTATION,
    "dof_vel": nv.REW_DOF_VEL, "action_rate": nv.REW_ACTION_RATE, "base_height": nv.REW_BASE_HEIGHT,
    "dof_pos_limits": nv.REW_DOF_POS_LIMITS, "feet_air_time": nv.REW_FEET_AIR_TIME,
}


def air_time_state(env):
    """(swing_time, last_contacts) of an env that carries the legged_gym feet-air-time state, else None."""
    swing = getattr(env, "swing_time", None)
    swing = getattr(env, "feet_air_time", None) if swing is None else swing
    last = getattr(env, "last_contacts", None)
    if torch.is_tensor(swing) and torch.is_tensor(last):
        return swing, last
    return None


def dof_limits(env) -> torch.Tensor:
    """(num_dof, 2) limits a dof-limit term reads: ``env.dof_pos_limits`` (legged_gym's soft limits) when the
    env defines it, else the asset limits of the robot (units/robot.py:39-40)."""
    lim = getattr(env, "dof_pos_limits", None)
    if torch.is_tensor(lim):
        return lim
    rb = env.robot
    return torch.stack([rb.dof_lower_limits, rb.dof_upper_limits], dim=1)


class A1Probe:
    """Crafted states for an A1-shaped env: every tensor a reward / observation / termination hook may
    read is saved, overwritten and restored.  Works on the env's OWN tensors (the hooks close over
    them), so it must run before the first real step or between steps."""

    def __init__(self, env):
        self.env, self.robot, self.isg = env, env.robot, env.isg_env
        rb, isg = self.robot, self.isg
        self.tensors = {
            "command": env.command_buf, "lin": rb.base_lin_vel, "ang": rb.base_ang_vel, "pg": rb.projected_gravity,
            "gvec": rb.gravity_vec,
            "history": env.actions_recorder.history_buf, "contact": isg.contact_state, "torques": rb.torques,
            "dof": isg.dof_state, "root": isg.root_state, "actions": env.actions,
            "ep_len": env.episode_length_buf,
        }
        if getattr(isg, "measured_heights", None) is not None:
            self.tensors["heights"] = isg.measured_heights
        air = air_time_state(env)
        if air is not None:
            self.tensors["swing_time"], self.tensors["last_contacts"] = air
        self._saved = None
        self._attrs = ("obs_buf", "reset_buf", "time_out_buf", "contact_terminate_buf", "rew_buf")

    def __enter__(self):
        self._saved = {k: t.clone() for k, t in self.tensors.items()}
        self._saved_attrs = {a: getattr(self.env, a, None) for a in self._attrs}
        self._saved_torques_obj = self.robot.torques
        return self

    def __exit__(self, *exc):
        for k, t in self.tensors.items():
            t.copy_(self._saved[k])
        for a, v in self._saved_attrs.items():
            if v is not None:
                setattr(self.env, a, v)
        self.robot.torques = self._saved_torques_obj
        return False

    def zero(self):
        for k, t in self.tensors.items():
            t.zero_()
        self.isg.root_state[:, 6] = 1.0            # identity quaternion

    def randomize(self, seed: int = 1234):
        g = torch.Generator(device=self.env.device).manual_seed(seed)
        for k, t in self.tensors.items():
            if t.dtype.is_floating_point:
                t.copy_(torch.randn(t.shape, generator=g, device=t.device) * (0.6 if k != "contact" else 0.4))
            elif t.dtype == torch.bool:
                t.copy_(torch.rand(t.shape, generator=g, device=t.device) < 0.5)
            else:
                t.copy_(torch.randint(0, int(self.env.max_episode_length) + 40, t.shape, generator=g, device=t.device))
        q = self.isg.root_state[:, 3:7]
        q.copy_(q / q.norm(dim=1, keepdim=True).clamp_min(1e-6))

    def value(self, fn: Callable) -> float:
        return float(fn()[0])


def _snap(value: float, fn: Callable, rel: float = 1e-3) -> float:
    """The literal of the method body nearest to a fitted constant (exact user value when present)."""
    consts = []
    code = getattr(fn, "__code__", None) or getattr(getattr(fn, "__func__", None), "__code__", None)
    for c in (code.co_consts if code is not None else ()):
        if isinstance(c, (int, float)) and not isinstance(c, bool):
            consts += [float(c), -float(c)]
    best = min(consts, key=lambda c: abs(c - value), default=None)
    if best is not None and abs(best - value) <= rel * max(abs(value), 1e-12):
        return best
    return value


def _fit_exp(pr: A1Probe, fn, setter) -> Tuple[float, float]:
    pr.zero()
    p0 = pr.value(fn)                               # exp(0) = 1
    if p0 == 0.0:
        raise TermMismatch("term is identically zero")
    pr.zero()
    setter(0.5)                                     # squared error 0.25
    r = pr.value(fn)
    ratio = r / p0
    if not (0.0 < ratio < 1.0):
        raise TermMismatch("not of the form p0*exp(-err/p1)")
    return p0, _snap(-0.25 / math.log(ratio), fn)


def fit_a1_term(pr: A1Probe, fn: Callable, code: int) -> Tuple[float, float]:
    env, rb, t = pr.env, pr.robot, pr.tensors
    one = lambda name, idx: (pr.zero(), t[name].__setitem__(idx, 1.0), pr.value(fn))[2]
    if code == nv.REW_TRACKING_LIN_VEL:
        return _fit_exp(pr, fn, lambda v: t["command"].__setitem__((0, 0), v))
    if code == nv.REW_TRACKING_ANG_VEL:
        return _fit_exp(pr, fn, lambda v: t["command"].__setitem__((0, 2), v))
    if code == nv.REW_STABILIZING_BASE:
        return one("lin", (0, 2)), one("ang", (0, 0))
    if code == nv.REW_SMOOTHING_ACTION:
        return one("history", (0, 0, 0)) / 2.0, 0.0             # |a1-a0|^2 + |a2-2a1+a0|^2 = 1 + 1
    if code == nv.REW_TORQUES:
        return one("torques", (0, 0)), 0.0
    if code == nv.REW_LIN_VEL_Z:
        return one("lin", (0, 2)), 0.0
    if code == nv.REW_ANG_VEL_XY:
        return one("ang", (0, 0)), 0.0
    if code == nv.REW_ORIENTATION:
        return one("pg", (0, 0)), 0.0
    if code == nv.REW_DOF_VEL:
        return one("dof", (0, 1)), 0.0                           # dof_state row 0 = (pos, vel) of dof 0
    if code == nv.REW_ACTION_RATE:
        return one("actions", (0, 0)), 0.0
    if code == nv.REW_BASE_HEIGHT:
        vals = []
        for z in (0.0, 1.0, 2.0):
            pr.zero()
            rows = rb.root_indices[0]
            t["root"][rows, 2] = z
            vals.append(pr.value(fn))
        d1, d2 = vals[1] - vals[0], vals[2] - vals[1]
        p0 = (d2 - d1) / 2.0
        if p0 == 0.0:
            raise TermMismatch("not quadratic in the base height")
        return _snap(p0, fn), _snap((1.0 - d1 / p0) / 2.0, fn)
    if code == nv.REW_LEG_COLLISION:
        n_leg = int(rb.leg_indices.numel())
        cf = t["contact"].view(env.num_envs, -1, 3)

        def count_at(force):
            pr.zero()
            cf[0, :, 0] = force
            return pr.value(fn)

        p0 = count_at(1e4) / n_leg
        if p0 == 0.0:
            raise TermMismatch("term is identically zero")
        lo, hi = 0.0, 1e4                           # threshold by bisection, then snapped to the literal
        for _ in range(60):
            mid = 0.5 * (lo + hi)
            if count_at(mid) != 0.0:
                hi = mid
            else:
                lo = mid
        return p0, _snap(0.5 * (lo + hi), fn)
    if code == nv.REW_DOF_POS_LIMITS:
        lim = dof_limits(env)
        if tuple(lim.shape) != (rb.num_dof, 2):
            raise TermMismatch("dof limits are not a (num_dof, 2) tensor")
        vals = []
        for over in (1.0, 2.0):                     # dof 0 that far above its upper limit; the rest unchanged
            pr.zero()
            t["dof"].view(env.num_envs, -1, 2)[0, 0, 0] = float(lim[0, 1]) + over
            vals.append(pr.value(fn))
        return (_snap(vals[1] - vals[0], fn), 0.0,
                {"dof_pos_limits": [(float(lo), float(hi)) for lo, hi in lim.tolist()]})
    if code == nv.REW_FEET_AIR_TIME:
        if "swing_time" not in t:
            raise TermMismatch("feet_air_time needs env.swing_time (N, feet) and env.last_contacts (N, feet) bool")
        feet = [int(b) for b in rb.ee_indices.tolist()]
        if tuple(t["swing_time"].shape) != (env.num_envs, len(feet)) or len(feet) > 4:
            raise TermMismatch("swing_time is not (num_envs, num_feet<=4)")
        cf = t["contact"].view(env.num_envs, -1, 3)

        def landing(air, force=100.0, cmd=1.0):     # foot 0 lands after `air` seconds in the air
            pr.zero()
            t["command"][0, 0] = cmd
            t["swing_time"][0, 0] = air
            cf[0, feet[0], 2] = force
            return pr.value(fn)

        r1, r2 = landing(1.0), landing(2.0)
        p0 = r2 - r1
        if p0 == 0.0:
            raise TermMismatch("term does not respond to a landing foot")
        dt = float(t["swing_time"][0, 1]) if len(feet) > 1 else float(pr.isg.dt)   # a foot in the air gained dt
        p0 = _snap(p0, fn)
        p1 = _snap(1.0 + dt - r1 / p0, fn)

        def bisect(lo, hi, responds):
            for _ in range(60):
                mid = 0.5 * (lo + hi)
                lo, hi = (lo, mid) if responds(mid) else (mid, hi)
            return 0.5 * (lo + hi)

        force_thr = _snap(bisect(0.0, 100.0, lambda f: landing(2.0, force=f) != 0.0), fn)
        cmd_thr = _snap(bisect(0.0, 1.0, lambda c: landing(2.0, cmd=c) != 0.0), fn)
        return p0, p1, {"feet_bodies": tuple(feet), "feet_contact_force": force_thr, "air_time_cmd_min": cmd_thr,
                        "air_time_dt": dt}
    raise TermMismatch(f"no fitting rule for term code {code}")


def compile_a1_terms(env, functions: Sequence[Callable], names: Optional[Dict[str, int]] = None) -> List[CompiledTerm]:
    """match + fit (steps 1-2).  Raises TermMismatch / KeyError with the offending term's name."""
    names = names or A1_NAMES
    if len(functions) == 0:
        raise TermMismatch("build_reward_functions() returned no term (env.py:161)")
    if len(functions) > nv.MAX_TERMS:
        raise TermMismatch(f"{len(functions)} terms: at most {nv.MAX_TERMS} fused reward terms are supported")
    out = []
    with A1Probe(env) as pr:
        for fn in functions:
            key = _strip(fn.__name__)
            if key not in names:
                raise KeyError(f"reward term {fn.__name__!r} has no fused implementation; known: {sorted(names)}")
            p0, p1, *extra = fit_a1_term(pr, fn, names[key])
            out.append(CompiledTerm(fn.__name__, names[key], float(p0), float(p1), extra[0] if extra else None))
    return out


def desc_extras(terms: Sequence[CompiledTerm]) -> dict:
    """The a1_desc keywords the compiled terms carry (feet, thresholds, dof limits)."""
    out = {}
    for term in terms:
        out.update(term.extra or {})
    return out


def verify_a1_terms(env, hot, functions: Sequence[Callable], terms: Sequence[CompiledTerm], seed: int = 1234):
    """Step 3: user hooks (torch) vs the kernel's term library on the same random state."""
    with A1Probe(env) as pr:
        pr.randomize(seed)
        stateful = [pr.tensors[k] for k in ("swing_time", "last_contacts") if k in pr.tensors]
        if stateful:
            pr.tensors["swing_time"].abs_()
        before = [t.clone() for t in stateful]
        want = torch.stack([fn().to(torch.float) for fn in functions])
        after_hooks = [t.clone() for t in stateful]
        for t, b in zip(stateful, before):          # a stateful term advanced its state: rewind for the kernel's turn
            t.copy_(b)
        got = hot.eval_terms()
        for t, a, name in zip(stateful, after_hooks, ("swing_time", "last_contacts")):
            if not torch.allclose(t.to(torch.float), a.to(torch.float), rtol=RTOL, atol=ATOL):
                raise TermMismatch(f"feet_air_time: {name} after the Python hook and after the fused term differ")
    for i, term in enumerate(terms):
        err = (got[i] - want[i]).abs()
        tol = ATOL + RTOL * want[i].abs()
        bad = int((err > tol).sum())
        if bad:
            raise TermMismatch(f"reward term {term.name!r}: the Python hook and the fused term (code {term.code}, "
                               f"p0={term.p0:g}, p1={term.p1:g}) differ on {bad} of {err.numel()} envs "
                               f"(max abs err {float(err.max()):.3e})")


# ---------------------------------------------------------------------------------------------
# Observation layout (ObsLayout): which source feeds each vector slot, and every column's scale
# ---------------------------------------------------------------------------------------------

_OBS_PROBE = {"COMMAND": ("command", "command_buf"), "BASE_LIN_VEL": ("lin", "base_lin_vel"),
              "BASE_ANG_VEL": ("ang", "base_ang_vel"), "GRAVITY_VEC": ("gvec", "gravity_vec"),
              "PROJECTED_GRAVITY": ("pg", "projected_gravity")}
assert set(_OBS_PROBE) == set(OBS_SOURCES)


def _exact_offset(q0: float) -> float:
    """A power of two v with fp32 (q0 + v) - q0 == v: a dof-position probe whose dof_pos - q0 is exact."""
    q = torch.tensor(q0, dtype=torch.float)
    for k in range(0, 40):
        v = 2.0 ** -k
        if float((q + v) - q) == v:
            return v
    raise NotFusable(f"compute_observations: no exact dof-position probe around {q0}")


class _NoHeights:
    """Stands in for ``measured_heights`` while a blind (72-column) observation hook runs: the fused blind
    step does not scan the terrain, so any use of the heights refuses the hook."""
    REASON = ("compute_observations: the blind (72- or 48-column) observation reads measured_heights; the fused "
              "blind step does not scan the terrain")

    def __init__(self):
        self.touched = False

    def _refuse(self, *args, **kwargs):
        object.__setattr__(self, "touched", True)
        raise NotFusable(self.REASON)

    @classmethod
    def __torch_function__(cls, func, types, args=(), kwargs=None):
        for a in (*args, *(kwargs or {}).values()):
            if isinstance(a, _NoHeights):
                a._refuse()
        raise NotFusable(cls.REASON)

    def __getattr__(self, name):
        self._refuse()

    __getitem__ = __len__ = __iter__ = __array__ = _refuse
    __add__ = __radd__ = __sub__ = __rsub__ = __mul__ = __rmul__ = __truediv__ = __rtruediv__ = __neg__ = _refuse


def _blind_hook(env, heights):
    """Runs ``compute_observations`` with ``heights`` (a ``_NoHeights``) as the measured heights; an error
    the heights caused becomes NotFusable with the reason."""
    env.isg_env.measured_heights = heights
    try:
        env.compute_observations()
    except NotFusable:
        raise
    except Exception as exc:
        if heights.touched:
            raise NotFusable(_NoHeights.REASON) from exc
        raise


@contextmanager
def _obs_draws(env, u, width: Optional[int] = None):
    """While ``compute_observations`` runs: ``torch.rand_like`` of the whole observation returns ``u`` (a
    number or a tensor of that shape), once per call; any other draw raises NotFusable.  legged_gym's noise
    is ``obs_buf += (2 * torch.rand_like(obs_buf) - 1) * noise_scale_vec``, which the fused kernel adds.
    ``width``: the observation's columns (default 72 + the height points)."""
    shape = (env.num_envs, width if width is not None else nv.OBS_HEAD + env.isg_env.num_height_points)
    calls = []

    def rand_like(t, *args, **kwargs):
        if tuple(t.shape) != shape:
            raise NotFusable(f"compute_observations: torch.rand_like of a {tuple(t.shape)} tensor; the fused noise "
                             f"draws one u per column of the whole {shape} observation")
        calls.append(1)
        if len(calls) > 1:
            raise NotFusable("compute_observations: torch.rand_like is called more than once; the fused noise draws "
                             "one u per column")
        dtype = t.dtype if t.dtype.is_floating_point else torch.float
        if isinstance(u, torch.Tensor):
            return u.to(device=t.device, dtype=dtype)
        return torch.full(shape, float(u), device=t.device, dtype=dtype)

    def refuse(name):
        def draw(*args, **kwargs):
            raise NotFusable(f"compute_observations: draws with torch.{name}; the fused observation noise is "
                             "uniform: (2 * torch.rand_like(obs_buf) - 1) * scale")
        return draw

    saved = {name: getattr(torch, name) for name in ("rand_like", "randn_like", "rand", "randn", "normal")}
    patched = {name: (rand_like if name == "rand_like" else refuse(name)) for name in saved}
    try:
        for name, fn in patched.items():
            setattr(torch, name, fn)
        yield
    finally:
        for name, fn in saved.items():
            setattr(torch, name, fn)


def compile_a1_obs(env, num_obs: Optional[int] = None) -> ObsLayout:
    """``env.compute_observations`` -> ObsLayout, by probing.  At the zero state (every input zero,
    dof_pos = default_dof_pos, base 0.5 above flat terrain) the observation must be all zeros; then each
    input is set alone to a power of two and must reach exactly one column of its block, the three
    components of a vector in order in one slot; the column's value over the input is its scale.  The
    heights are probed at z - 0.5 - h = 0.5 and 3, which fixes their scale and the clip-then-scale order.
    Every probe so far runs with ``torch.rand_like`` at u = 0.5, where uniform noise vanishes.  Then, at the
    zero state, u = 1 gives each column's noise scale and u = 0 must give its negative; the heights share
    one scale, added after their clip and scale (probed at z - 0.5 - h = 3).
    A hook that returns (N, 72) is blind: the same head probes run with the measured heights replaced by
    a stand-in whose every use refuses the hook, and there are no height probes (the layout keeps height
    scale 1 and no height noise).
    A 48-column head (num_obs 48 + the height points, or 48 blind) is the action head, legged_gym's own
    observation: each ``env.actions[:, d]`` must reach column 36 + d alone, as a scale times the action, and
    the action history none; in a 72-column head the step's actions must reach no column.  The heights and
    their noise then start at column 48.  ``num_obs``: the width the hook must return (default: the
    hook's own width when it is one of these four, else 72 + the height points).
    Anything else raises NotFusable naming the column and the reason."""
    rb, isg = env.robot, env.isg_env
    widths = [h + p for h in (nv.OBS_HEAD, nv.OBS_HEAD_ACT) for p in (isg.num_height_points, 0)]
    if num_obs is not None and num_obs not in widths:
        raise NotFusable(f"observation width {num_obs} is none of {widths} (72 or 48 head columns, with or "
                         "without the height points)")
    had = isg.__dict__.get("_measured_heights")
    with A1Probe(env) as pr:
        t = pr.tensors
        heights = torch.zeros(env.num_envs, isg.num_height_points, device=env.device)
        dof = t["dof"].view(env.num_envs, -1, 2)
        q0 = rb.default_dof_pos
        rows0 = rb.root_indices[0]

        def zero_state():
            pr.zero()
            dof[:, :, 0] = q0
            t["root"][rb.root_indices, 2] = 0.5
            heights.zero_()

        width = num_obs
        if width is None:                           # the hook's own width: a head, or a head + the heights
            zero_state()
            isg.measured_heights = heights
            with _obs_draws(env, 0.5, env.obs_buf.shape[1]):
                env.compute_observations()
            shape = tuple(env.obs_buf.shape)
            width = shape[1] if len(shape) == 2 and shape[0] == env.num_envs and shape[1] in widths \
                else nv.OBS_HEAD + heights.shape[1]
        n_head = nv.OBS_HEAD_ACT if width in (nv.OBS_HEAD_ACT, nv.OBS_HEAD_ACT + heights.shape[1]) else nv.OBS_HEAD
        blind = width == n_head

        def observe(u=0.5):
            with _obs_draws(env, u, width):
                if blind:
                    _blind_hook(env, _NoHeights())
                else:
                    isg.measured_heights = heights
                    env.compute_observations()
            obs = env.obs_buf
            if tuple(obs.shape) != (env.num_envs, width):
                raise NotFusable(f"compute_observations: shape {tuple(obs.shape)}, the fused observation is "
                                 f"({env.num_envs}, {width})")
            return obs[0].float().cpu()

        def lit(o, lo=0, hi=n_head):
            return [(j, float(o[j])) for j in torch.nonzero(o[lo:hi]).flatten().add(lo).tolist()]

        try:
            zero_state()
            for j, v in lit(observe(), 0, None):
                raise NotFusable(f"compute_observations: column {j} is {v:g} with every input at zero (dof_pos = "
                                 "default_dof_pos, base height 0.5 above the terrain): the fused observation has "
                                 "no additive offsets")
            slots, scales = [None] * 4, [None] * n_head
            for name, (key, label) in _OBS_PROBE.items():
                cols = []
                for c in range(3):
                    zero_state()
                    t[key][0, c] = 1.0
                    cols.append(lit(observe(), 0, None))
                if not any(cols):
                    continue                                        # source not observed
                for c, hits in enumerate(cols):
                    if len(hits) != 1:
                        raise NotFusable(f"compute_observations: {label}[:, {c}] reaches columns "
                                         f"{[j for j, _ in hits]}; it must reach exactly one column")
                    j = hits[0][0]
                    if j >= 12 or j % 3 != c or j // 3 != cols[0][0][0] // 3:
                        raise NotFusable(f"compute_observations: column {j} reads {label}[:, {c}]; the fused "
                                         "observation takes a vector whole, in order, into one of the slots at "
                                         "columns 0-2, 3-5, 6-8, 9-11")
                slot = cols[0][0][0] // 3
                if slots[slot] is not None:
                    raise NotFusable(f"compute_observations: columns {3 * slot}-{3 * slot + 2} read both "
                                     f"{_OBS_PROBE[slots[slot]][1]} and {label}; a column takes one source")
                slots[slot] = name
                for c in range(3):
                    scales[3 * slot + c] = cols[c][0][1]
            for i, src in enumerate(slots):
                if src is None:
                    raise NotFusable(f"compute_observations: columns {3 * i}-{3 * i + 2} follow none of "
                                     f"{[label for _, label in _OBS_PROBE.values()]}")
            # dof positions (dof_pos - default_dof_pos), dof velocities, then the step's actions (48-column
            # head) or the history slot-major (72-column head); col None: the input must reach no column
            act = n_head == nv.OBS_HEAD_ACT
            probes = []
            for d in range(12):
                probes.append((12 + d, f"dof_pos[:, {d}] - default_dof_pos[{d}]", ("dof", d, 0)))
                probes.append((24 + d, f"dof_vel[:, {d}]", ("dof", d, 1)))
                probes.append((36 + d if act else None, f"actions[:, {d}]", ("actions", 0, d)))
                for h in range(3):
                    probes.append((None if act else 36 + 12 * h + d, f"actions_recorder.get_last({h})[:, {d}]",
                                   ("history", d, h)))
            mixed = (f"the {n_head}-column head observes "
                     + ("the step's actions (env.actions, column 36 + d), not the action history (actions_recorder)"
                        if act else "the action history (actions_recorder), not the step's actions (env.actions): "
                        "the step's actions are the 48-column action head (num_obs 235 or 48)"))

            def probe(key, a, b, x):
                zero_state()
                if key == "dof" and b == 0:
                    dof[0, a, 0] = float(torch.tensor(float(q0[a]), dtype=torch.float) + x)
                elif key == "actions":
                    t["actions"][0, b] = x
                else:
                    (dof if key == "dof" else t["history"])[0, a, b] = x
                return lit(observe(), 0, None)

            for col, label, (key, a, b) in probes:
                x = _exact_offset(float(q0[a])) if key == "dof" and b == 0 else 1.0
                hits = probe(key, a, b, x)
                if col is None:
                    if hits:
                        raise NotFusable(f"compute_observations: {label} reaches columns {[j for j, _ in hits]}; "
                                         + mixed)
                    continue
                if len(hits) != 1 or hits[0][0] != col:
                    raise NotFusable(f"compute_observations: {label} reaches columns {[j for j, _ in hits]}; the "
                                     f"fused observation has it in column {col} alone"
                                     + (f" ({mixed})" if key in ("actions", "history") else ""))
                scales[col] = hits[0][1] / x
                if key == "actions":                    # a scale times the action: half the input, half the value
                    half = probe(key, a, b, 0.5 * x)
                    if len(half) != 1 or half[0][0] != col or half[0][1] != 0.5 * hits[0][1]:
                        raise NotFusable(f"compute_observations: column {col} is {hits[0][1]:g} at {label} = 1 "
                                         f"and {half[0][1] if half else 0.0:g} at 0.5; the fused observation takes "
                                         "the step's actions times a scale, no other function of them")
            if blind:                                       # no height columns: no height probes
                zero_state()
                up, down = observe(1.0), observe(0.0)
                bad = torch.nonzero(down != -up).flatten().tolist()
                if bad:
                    j = bad[0]
                    raise NotFusable(f"compute_observations: column {j} is {float(up[j]):g} at u = 1 and "
                                     f"{float(down[j]):g} at u = 0 with every input at zero; the fused noise is "
                                     "(2u - 1) * scale with u = torch.rand_like(obs_buf)")
                return ObsLayout(tuple(slots), tuple(scales), 1.0, tuple(float(v) for v in up), 0.0)
            # heights: clip(z - 0.5 - h, +-1) * height_scale
            zero_state()
            heights[0] = -0.5
            o = observe()
            for j, v in lit(o):
                raise NotFusable(f"compute_observations: column {j} follows the measured heights")
            hv = o[n_head:]
            hs = float(hv[0]) / 0.5
            if hs == 0.0 or not bool((hv == hv[0]).all()):
                raise NotFusable("compute_observations: the height columns are not one scale times "
                                 "clip(base z - 0.5 - measured_heights, -1, 1)")
            heights[0] = -3.0
            hv = observe()[n_head:]
            bad = torch.nonzero(hv != hs).flatten().tolist()
            if bad:
                raise NotFusable(f"compute_observations: height column {n_head + bad[0]} is {float(hv[bad[0]]):g} at "
                                 f"z - 0.5 - h = 3, not clip(3, -1, 1) * {hs:g}: heights must be clipped to +-1 "
                                 "before they are scaled")
            # noise: clean + (2u - 1) * s, so +s at u = 1 and -s at u = 0 on the all-zero observation
            zero_state()
            up, down = observe(1.0), observe(0.0)
            bad = torch.nonzero(down != -up).flatten().tolist()
            if bad:
                j = bad[0]
                raise NotFusable(f"compute_observations: column {j} is {float(up[j]):g} at u = 1 and {float(down[j]):g} "
                                 "at u = 0 with every input at zero; the fused noise is (2u - 1) * scale with "
                                 "u = torch.rand_like(obs_buf)")
            hn = float(up[n_head])
            bad = torch.nonzero(up[n_head:] != hn).flatten().tolist()
            if bad:
                raise NotFusable(f"compute_observations: height column {n_head + bad[0]} has noise scale "
                                 f"{float(up[n_head + bad[0]]):g}, height column {n_head} {hn:g}; the fused observation "
                                 "has one noise scale for all height columns")
            if hn != 0.0:
                heights[0] = -3.0
                for u, sign in ((1.0, 1.0), (0.0, -1.0)):
                    want = torch.tensor(hs, dtype=torch.float) + torch.tensor(sign * hn, dtype=torch.float)
                    hv = observe(u)[n_head:]
                    bad = torch.nonzero(hv != want).flatten().tolist()
                    if bad:
                        raise NotFusable(f"compute_observations: height column {n_head + bad[0]} is "
                                         f"{float(hv[bad[0]]):g} at z - 0.5 - h = 3 and u = {u:g}, not "
                                         f"clip(3, -1, 1) * {hs:g} {'+' if sign > 0 else '-'} {hn:g}: the noise must "
                                         "be added after the heights are clipped and scaled")
            noise = tuple(float(v) for v in up[:n_head])
        finally:
            if had is None:
                del isg.measured_heights
            else:
                isg.measured_heights = had
    return ObsLayout(tuple(slots), tuple(scales), hs, noise, hn)


def a1_obs_definition(env, layout: ObsLayout, u: Optional[torch.Tensor] = None, blind: bool = False) -> torch.Tensor:
    """The observation the fused kernel builds under ``layout``, in torch on the env's tensors (before the
    final clip to +-clip_obs that the base class applies).  ``u``: the noise draws, (num_envs, head + 259 -
    72), or (num_envs, head) when ``blind`` (the head columns alone).  A 48-column layout (the action head)
    ends its head with the step's ``env.actions``, a 72-column one with ``actions_recorder.flatten()``."""
    rb, isg = env.robot, env.isg_env
    src = {name: getattr(rb if key != "command" else env, label) for name, (key, label) in _OBS_PROBE.items()}
    last = env.actions if layout.head == nv.OBS_HEAD_ACT else env.actions_recorder.flatten()
    head = torch.cat([src[name] for name in layout.slots] + [rb.dof_pos - rb.default_dof_pos, rb.dof_vel, last],
                     dim=1)
    head = head * torch.tensor(layout.scales, dtype=torch.float, device=head.device)
    if blind:
        if u is not None and layout.has_noise():
            head = head + (2 * u - 1) * torch.tensor(layout.noise, dtype=torch.float, device=head.device)
        return head
    heights = torch.clip(rb.base_pose[:, 2].unsqueeze(1) - 0.5 - isg.measured_heights, -1, 1.) * layout.height_scale
    obs = torch.cat([head, heights], dim=1)
    if u is not None and layout.has_noise():
        scale = torch.tensor(layout.noise + (layout.height_noise,) * heights.shape[1], dtype=torch.float,
                             device=obs.device)
        obs = obs + (2 * u - 1) * scale
    return obs


def verify_a1_obs(env, layout: ObsLayout, seed: int = 4321, num_obs: Optional[int] = None):
    """``env.compute_observations`` against the layout's definition (noise included) on a seeded random
    state, with the same seeded draws given to the hook's ``torch.rand_like`` and to the definition.
    ``num_obs = layout.head``: the blind observation, with the heights replaced by a stand-in that refuses
    any use."""
    isg = env.isg_env
    blind = num_obs == layout.head
    width = layout.head + (0 if blind else isg.num_height_points)
    had = isg.__dict__.get("_measured_heights")
    with A1Probe(env) as pr:
        pr.randomize(seed)
        g = torch.Generator(device=env.device).manual_seed(seed)
        heights = torch.randn(env.num_envs, isg.num_height_points, generator=g, device=env.device)
        u = torch.rand(env.num_envs, width, generator=g, device=env.device)
        try:
            with _obs_draws(env, u, width):
                if blind:
                    _blind_hook(env, _NoHeights())
                else:
                    isg.measured_heights = heights
                    env.compute_observations()
            check_close(env.obs_buf, a1_obs_definition(env, layout, u, blind), "compute_observations")
        finally:
            if had is None:
                del isg.measured_heights
            else:
                isg.measured_heights = had
