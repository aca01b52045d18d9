// Philox4x32-10 (Salmon et al., SC'11), counter = (env_id_global, step, stream, 0),
// key = (seed_lo, seed_hi).  Same function as oracle/philox_np.py (pinned to the Random123
// known-answer vectors); the reference draws its reset samples from torch's / numpy's global
// generators (SURVEY.md D2), parity is defined on these injected per-env draws (§8d).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace shifu {

enum : uint32_t {
  STREAM_LEVEL = 0,     // a1_conditional.py:219  terrain-level re-draw
  STREAM_XY = 1,        // a1_conditional.py:47   reset xy offset
  STREAM_FORCE = 2,     // a1_conditional.py:86   random push force
  STREAM_CMD = 3,       // a1_conditional.py:195-199 commands
  STREAM_CUBE_POS = 4,  // a_prior_stage.py:41
  STREAM_CUBE_EUL = 5,  // a_prior_stage.py:44
  STREAM_GOAL_POS = 6,
  STREAM_GOAL_EUL = 7,
  STREAM_OBS_NOISE = 8  // observation noise: counter (env, step, 8, word); the word map is SHIFU_STREAM_OBS_NOISE's
};

struct U4 {
  uint32_t x, y, z, w;
};

__device__ __forceinline__ U4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                            uint32_t k0, uint32_t k1) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
    const uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += W0; k1 += W1;
  }
  return U4{c0, c1, c2, c3};
}

__device__ __forceinline__ U4 draw(uint64_t seed, int64_t env_global, int64_t step, uint32_t stream) {
  return philox4x32_10((uint32_t)env_global, (uint32_t)step, stream, 0u, (uint32_t)seed,
                       (uint32_t)(seed >> 32));
}

// uint32 -> [0,1) on torch.rand's 24-bit grid
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-8f; }
__device__ __forceinline__ double u01d(uint32_t x) { return (double)(x >> 8) * 5.9604644775390625e-8; }
// 2u - 1 for u = u01(x), exactly: (x >> 8) - 2^23 is an integer of at most 24 bits
__device__ __forceinline__ float u_pm1(uint32_t x) {
  return (float)((int)(x >> 8) - 0x800000) * 1.1920928955078125e-7f;
}

// Observation-noise word of env `gid` (counter (gid, step, STREAM_OBS_NOISE, word)).
__device__ __forceinline__ U4 obs_noise_word(uint64_t seed, int64_t gid, int64_t step, uint32_t word) {
  return philox4x32_10((uint32_t)gid, (uint32_t)step, STREAM_OBS_NOISE, word, (uint32_t)seed, (uint32_t)(seed >> 32));
}

// The (word, lane) of observation column `col` < head + 187 (the map of include/shifu_b200.h).  head: the
// head width, 72 or 48 (the action head: its column d + 12m, m < 4, keeps the word and lane it has at 72).
__device__ __forceinline__ void obs_noise_slot(int col, uint32_t& word, int& lane, int head = 72) {
  if (col < head) {                                 // head: column d + 12m, lane pair d = 2i, 2i+1
    const int m = col / 12, d = col - 12 * m;
    word = 3 * (d >> 1) + (m >> 1);
    lane = (d & 1) + 2 * (m & 1);
  } else {                                          // heights: point pair k = (pt, 186 - pt)
    const int pt = col - head, k = min(pt, 186 - pt);
    word = 18 + (k >> 1);
    lane = 2 * (k & 1) + (pt != k ? 1 : 0);
  }
}

__device__ __forceinline__ uint32_t u4_lane(const U4& u, int lane) {
  return lane == 0 ? u.x : lane == 1 ? u.y : lane == 2 ? u.z : u.w;
}

// floor(u * high) in integers
__device__ __forceinline__ int64_t randint(uint32_t x, int32_t high) {
  return (int64_t)(((uint64_t)(x >> 8) * (uint64_t)high) >> 24);
}

}  // namespace shifu
