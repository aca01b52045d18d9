"""ORACLE — test infrastructure, NOT product code.

A float64 numpy evaluation of every A1 reward opcode (``enum ShifuRewardTerm`` in
``include/shifu_b200.h``), written from the formulas in the enum comments and independent of torch
and of ``shifu_oracle.py``.  The fp32 implementations (the CUDA kernels and the torch oracle) are
measured against it with a per-term error bound ``c * 2**-24 * M``: ``M`` (returned next to each
value) is the sum of the magnitudes of the term's intermediate products, ``c`` (``BOUND_C``) comes
from the term's count of rounded operations.

Inputs are the fp32 arrays the kernels read; constants are passed as the fp32 values the kernel's
descriptor holds, so only the arithmetic is done in float64.
"""
from __future__ import annotations

from typing import Dict, Sequence, Tuple

import numpy as np

U = 2.0 ** -24          # unit roundoff of fp32
TINY = 2.0 ** -126      # below this a fp32 result may be subnormal: absolute error up to 2^-149 per op

# c of the bound, per term: (rounded ops that feed the result, counting a correctly rounded square,
# product, sum or difference as one unit roundoff of its magnitude; a sequential sum of k terms as
# k - 1; CUDA's expf as 2 ulp = 4 unit roundoffs of its result)
BOUND_C = {
    # exp(-x) * p0, x = err / p1: the argument carries <= 5 u relative error (sub, square, add, div),
    # which exp turns into 5u|x| of the result; expf 4u, the product with p0 1u.  M = |v| (1 + |x|)
    "tracking_lin_vel": 5, "tracking_ang_vel": 5,
    # p0 vz^2 + p1 (wx^2 + wy^2): square, product, add on each side, final add.  M = sum of the products
    "stabilizing_base": 4,
    # sum over 12 dofs of d1^2 and d2^2 (d2 = (a2 - 2 a1) + a0 carries its two roundings, which enter
    # M as |d2| |a2 - 2 a1|), two 12-term sums, their sum, product with p0
    "smoothing_action": 16,
    # p0 * integer count: one rounding
    "leg_collision": 1,
    # 12 squares, 11 sequential adds, product with p0
    "torques_penalize": 13, "dof_vel": 13,
    "lin_vel_z": 2,                       # square, product
    "ang_vel_xy": 3, "orientation": 3,    # squares, add, product
    "action_rate": 15,                    # difference, square (3 u), 11 adds, product
    "base_height": 4,                     # difference, square, product
    "dof_pos_limits": 14,                 # difference, clip (exact), add with the other side (exact), 11 adds, product
    # per foot: swing + dt, - p1; up to 3 adds of the feet; product with p0.  M = |p0| sum(|air| + |p1|)
    "feet_air_time": 6,
}


def norm_f64(v: np.ndarray) -> np.ndarray:
    return np.sqrt(np.sum(np.square(v.astype(np.float64)), axis=-1))


def eval_terms_f64(terms: Sequence[Tuple[str, float, float]], s: Dict[str, np.ndarray], c: Dict,
                   leg_norm: np.ndarray = None):
    """Evaluate ``terms`` [(name, p0, p1)] on the state ``s`` (fp32 arrays, see below) in float64.

    ``s``: command (N,3), lin (N,3) / ang (N,3) body-frame velocities, pg (N,3) projected gravity,
    dof (N,12,2) pos/vel, hist (N,12,3) action history (slot 0 = a_{t-1}), act (N,12), tau (N,12),
    contact (N,17,3), base_z (N,), swing (N,F), last (N,F) bool.
    ``c``: leg_bodies, dof_lo (12), dof_hi (12), feet (F bodies), feet_thr, air_cmd_min, air_dt.
    ``leg_norm`` (N, legs): the fp32 norms that define ``|F| > p1`` of leg_collision (aten's fp32
    norm); float64 norms when None.

    Returns (values (T,N) f64, M (T,N) f64, discrete dict, swing (N,F) fp32, last (N,F) bool), the
    last two being the feet-air-time state after the call (unchanged when the term is not listed).
    """
    f8 = lambda k: s[k].astype(np.float64)
    n = s["command"].shape[0]
    vals, mags, disc = [], [], {}
    swing, last = s["swing"].copy(), s["last"].copy()
    for name, p0, p1 in terms:
        p0, p1 = float(np.float32(p0)), float(np.float32(p1))
        if name == "tracking_lin_vel":
            x = np.sum(np.square(f8("command")[:, :2] - f8("lin")[:, :2]), axis=1) / p1
            v = p0 * np.exp(-x)
            m = np.abs(v) * (1 + np.abs(x))
        elif name == "tracking_ang_vel":
            x = np.square(f8("command")[:, 2] - f8("ang")[:, 2]) / p1
            v = p0 * np.exp(-x)
            m = np.abs(v) * (1 + np.abs(x))
        elif name == "stabilizing_base":
            a = p0 * np.square(f8("lin")[:, 2])
            b = p1 * np.sum(np.square(f8("ang")[:, :2]), axis=1)
            v, m = a + b, np.abs(a) + np.abs(b)
        elif name == "smoothing_action":
            h = f8("hist")
            d1 = h[..., 1] - h[..., 0]
            d2 = h[..., 2] - 2 * h[..., 1] + h[..., 0]
            v = p0 * np.sum(d1 * d1 + d2 * d2, axis=1)
            m = abs(p0) * np.sum(d1 * d1 + d2 * d2 + np.abs(d2) * np.abs(h[..., 2] - 2 * h[..., 1]), axis=1)
        elif name == "leg_collision":
            nrm = norm_f64(s["contact"][:, list(c["leg_bodies"])]) if leg_norm is None else leg_norm.astype(np.float64)
            cnt = np.sum(nrm > p1, axis=1)
            disc["leg_count"] = cnt
            v = p0 * cnt
            m = np.abs(v)
        elif name in ("torques_penalize", "dof_vel"):
            x = f8("tau") if name == "torques_penalize" else f8("dof")[..., 1]
            v = p0 * np.sum(x * x, axis=1)
            m = np.abs(v)
        elif name == "lin_vel_z":
            v = p0 * np.square(f8("lin")[:, 2])
            m = np.abs(v)
        elif name in ("ang_vel_xy", "orientation"):
            x = f8("ang" if name == "ang_vel_xy" else "pg")[:, :2]
            v = p0 * np.sum(x * x, axis=1)
            m = np.abs(v)
        elif name == "action_rate":
            d = f8("hist")[..., 0] - f8("act")
            v = p0 * np.sum(d * d, axis=1)
            m = np.abs(v)
        elif name == "base_height":
            v = p0 * np.square(f8("base_z") - p1)
            m = np.abs(v)
        elif name == "dof_pos_limits":
            q = f8("dof")[..., 0]
            lo = np.asarray(c["dof_lo"], np.float32).astype(np.float64)
            hi = np.asarray(c["dof_hi"], np.float32).astype(np.float64)
            out = -np.minimum(q - lo, 0.0) + np.maximum(q - hi, 0.0)
            disc["dof_outside"] = (q < lo) | (q > hi)
            v = p0 * np.sum(out, axis=1)
            m = np.abs(v)
        elif name == "feet_air_time":
            # STATEFUL (legged_gym _reward_feet_air_time): contact = F_z > thr; filt = contact | last;
            # first = (swing > 0) & filt; swing += dt; rew = sum (swing - p1) [first] [|cmd_xy| > cmd_min];
            # swing = 0 where filt; last = contact
            fz = s["contact"][:, list(c["feet"]), 2].astype(np.float64)
            contact = fz > float(np.float32(c["feet_thr"]))
            filt = contact | s["last"]
            first = (s["swing"] > 0) & filt
            air = s["swing"].astype(np.float64) + float(np.float32(c["air_dt"]))
            cmd = f8("command")
            moving = np.sqrt(cmd[:, 0] ** 2 + cmd[:, 1] ** 2) > float(np.float32(c["air_cmd_min"]))
            v = p0 * np.sum(np.where(first, air - p1, 0.0), axis=1) * moving
            m = abs(p0) * np.sum(np.where(first, np.abs(air) + abs(p1), 0.0), axis=1) * moving
            # the state: swing + dt is ONE fp32 add
            air32 = (s["swing"] + np.float32(c["air_dt"])).astype(np.float32)
            swing = np.where(filt, np.float32(0), air32).astype(np.float32)
            last = contact.copy()
            disc.update(contact=contact, first_contact=first, moving=moving)
        else:
            raise KeyError(f"no A1 opcode named {name!r}")
        vals.append(np.broadcast_to(np.asarray(v, np.float64), (n,)))
        mags.append(np.broadcast_to(np.asarray(m, np.float64), (n,)))
    return np.stack(vals), np.stack(mags), disc, swing, last


def assert_within_bound(tag: str, got: np.ndarray, want: np.ndarray, mag: np.ndarray, c: float):
    """|got - want| <= c * 2^-24 * M (+ 2^-126 for results in fp32's subnormal range)."""
    got = np.asarray(got, np.float64)
    err = np.abs(got - want)
    tol = c * U * mag + TINY
    bad = np.flatnonzero(~(err <= tol))
    assert bad.size == 0, (f"{tag}: {bad.size} of {got.size} values outside {c}*2^-24*M; first env {bad[0]}: "
                           f"got {got[bad[0]]!r} want {want[bad[0]]!r} M {mag[bad[0]]!r} "
                           f"(err/M = {err[bad[0]] / max(mag[bad[0]], 1e-300) / U:.2f} u)")
