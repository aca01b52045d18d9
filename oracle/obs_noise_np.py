"""ORACLE (test infrastructure, not product code): the observation-noise draws in numpy.

Stream 8 of ``philox_np`` (counter (env, step, 8, word), key = the seed), one word per group of up to
four observation columns, 65 words for the 259 columns.  The map is enumerated here word by word as
``include/shifu_b200.h`` states it, independently of the kernels' and ``shifu_b200.utils.philox``'s
column-by-column formula.
"""
from __future__ import annotations

import numpy as np

from oracle.philox_np import philox4x32_10, u01_f32

STREAM_OBS_NOISE = 8
OBS_COLS, OBS_HEAD, OBS_POINTS = 259, 72, 187


def obs_noise_map():
    """(word, lane) of each of the 259 observation columns, enumerated word by word as
    include/shifu_b200.h states it: head word 3i + r holds columns 2i + 24r, 2i + 1 + 24r, 2i + 24r + 12,
    2i + 1 + 24r + 12; height word 18 + (k >> 1) holds point k and its mirror 186 - k in (x, y) for even
    k and (z, w) for odd k, the centre point 93 in z alone."""
    word = np.full(OBS_COLS, -1, dtype=np.int64)
    lane = np.full(OBS_COLS, -1, dtype=np.int64)
    for i in range(6):
        for r in range(3):
            for l, c in enumerate((2 * i + 24 * r, 2 * i + 1 + 24 * r, 2 * i + 24 * r + 12, 2 * i + 1 + 24 * r + 12)):
                word[c], lane[c] = 3 * i + r, l
    for k in range(OBS_POINTS // 2 + 1):
        w, base = 18 + (k >> 1), 2 * (k & 1)
        word[OBS_HEAD + k], lane[OBS_HEAD + k] = w, base
        if k != OBS_POINTS - 1 - k:
            word[OBS_HEAD + OBS_POINTS - 1 - k], lane[OBS_HEAD + OBS_POINTS - 1 - k] = w, base + 1
    return word, lane


def obs_noise_u01(seed: int, env_ids, step: int):
    """(R, 259) float32 u of the observation noise of envs ``env_ids`` (global ids) at ``step``."""
    word, lane = obs_noise_map()
    n_words = int(word.max()) + 1
    ids = np.asarray(env_ids, dtype=np.uint32)[:, None]
    z = np.zeros((ids.shape[0], n_words), dtype=np.uint32)
    out = philox4x32_10(ids + z, z + np.uint32(step & 0xFFFFFFFF), z + np.uint32(STREAM_OBS_NOISE),
                        z + np.arange(n_words, dtype=np.uint32), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    x = np.stack(out, axis=0)                     # (4, R, words)
    return u01_f32(x[lane, :, word].T)
