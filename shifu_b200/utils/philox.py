"""Philox4x32-10 on torch int64 tensors (any device) for USER-HOOK tasks that want the same
counter-based reset draws as the fused kernels (``csrc/philox.cuh``): counter =
(env_id_global, step, stream, 0), key = (seed_lo, seed_hi).  The fused path never calls this.
``obs_noise_u01`` gives the observation-noise draws (stream 8, one counter word per column group)."""
from __future__ import annotations

import torch

_M0, _M1, _W0, _W1, _MASK = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85, 0xFFFFFFFF


def _mulhilo(m: int, c: torch.Tensor):
    """(hi32, lo32) of m*c for a 32-bit constant m and c in [0, 2^32) held in int64."""
    p_lo = m * (c & 0xFFFF)
    p_hi = m * (c >> 16)
    low = p_lo + ((p_hi & 0xFFFF) << 16)
    return (p_hi >> 16) + (low >> 32), low & _MASK


def philox4x32_10(c0, c1, c2, c3, k0: int, k1: int):
    for _ in range(10):
        hi0, lo0 = _mulhilo(_M0, c0)
        hi1, lo1 = _mulhilo(_M1, c2)
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0, k1 = (k0 + _W0) & _MASK, (k1 + _W1) & _MASK
    return c0, c1, c2, c3


def _lanes(seed: int, env_ids: torch.Tensor, step: int, stream: int):
    e = env_ids.to(torch.int64) & _MASK
    z = torch.zeros_like(e)
    return philox4x32_10(e, z + (step & _MASK), z + stream, z, seed & _MASK, (seed >> 32) & _MASK)


def draw_u01(seed: int, env_ids: torch.Tensor, step: int, stream: int, lanes: int) -> torch.Tensor:
    """(R, lanes) float32 in [0,1) on the 24-bit grid: (x >> 8) * 2^-24."""
    out = _lanes(seed, env_ids, step, stream)[:lanes]
    return torch.stack([(x >> 8).to(torch.float32) * (2.0 ** -24) for x in out], dim=1)


def draw_randint(seed: int, env_ids: torch.Tensor, step: int, stream: int, high: int) -> torch.Tensor:
    x = _lanes(seed, env_ids, step, stream)[0]
    return ((x >> 8) * high) >> 24


STREAM_OBS_NOISE, OBS_COLS, OBS_HEAD = 8, 259, 72


def obs_noise_slots():
    """(word, lane) int64 tensors of the 259 observation columns (map: include/shifu_b200.h)."""
    col = torch.arange(OBS_COLS)
    m, d = col // 12, col % 12
    pt = (col - OBS_HEAD).clamp(min=0)
    k = torch.minimum(pt, 186 - pt)
    head = col < OBS_HEAD
    word = torch.where(head, 3 * (d >> 1) + (m >> 1), 18 + (k >> 1))
    lane = torch.where(head, (d & 1) + 2 * (m & 1), 2 * (k & 1) + (pt != k).long())
    return word, lane


def obs_noise_u01(seed: int, env_ids: torch.Tensor, step: int) -> torch.Tensor:
    """(R, 259) float32 u of the fused kernels' observation noise for global env ids ``env_ids`` at ``step``
    (the step the same step's reset draws use): a user-hook ``compute_observations`` that takes
    ``torch.rand_like(obs_buf)`` from here adds the noise the kernel adds."""
    word, lane = (t.to(env_ids.device) for t in obs_noise_slots())
    n_words = int(word.max()) + 1
    e = (env_ids.to(torch.int64) & _MASK).unsqueeze(1)
    z = torch.zeros(e.shape[0], n_words, dtype=torch.int64, device=env_ids.device)
    out = torch.stack(philox4x32_10(e + z, z + (step & _MASK), z + STREAM_OBS_NOISE,
                                    z + torch.arange(n_words, device=env_ids.device), seed & _MASK,
                                    (seed >> 32) & _MASK))            # (4, R, words)
    x = out[lane, :, word].T
    return (x >> 8).to(torch.float32) * (2.0 ** -24)
