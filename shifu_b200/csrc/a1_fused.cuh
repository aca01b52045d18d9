// K-main: the fused A1 post-physics step (ShifuVecEnv.post_step, shifu/gym/env.py:93-106, with
// the A1 task hooks, + the obs clip of env.py:90).  Rows a5-a7, a9-a14 of SURVEY.md §8(a).
//
// One CTA = A1_TILE (32) consecutive envs, 6 warps.  Phases (separated by CTA barriers):
//   A   coalesced 128-bit loads of the tile's root / dof / contact / history / torque / action
//       rows into shared memory; warp 0 prefetches the per-env scalars (lane = env)
//   B1  warp w evaluates reward terms j = w, w+6, ... for all 32 envs (lane = env); warp 0 also
//       does termination, warp 5 the yaw-quaternion normalisation for the height scan
//   B2  warp 0 (lane = env): ordered reward / episode-sum accumulation, flag and ep_len stores,
//       reset of flagged envs (curriculum, Philox draws, state rewrite), per-step log sums
//   B3  all threads: obs head (72 columns, laid out and scaled by A1Obs), history push, carried
//       body-frame velocities
//   D   coalesced write-back of the obs head and the history tile
//   C   thread t owns scan point t: 187-point height scan per env, obs columns 72..258 streamed
//       straight to HBM (a warp writes 128 contiguous bytes per env)
// HBM traffic is the algorithmic minimum (every state row read once, obs written once); the scan
// table (banded min-of-3 map, 5.4 MB) lives in L2/L1.
#pragma once
#include "a1_kernels.cuh"

namespace shifu {

struct A1Smem {
  float root[A1_TILE][13];
  float dof[A1_TILE][A1_DOF * 2];
  float contact[A1_TILE][A1_BODIES * 3];
  float hist[A1_TILE][A1_DOF * A1_HIST];
  float tau[A1_TILE][A1_DOF];
  float act[A1_TILE][A1_DOF];
  float head[A1_TILE][A1_HEAD];
  float rterm[SHIFU_MAX_REWARD_TERMS][A1_TILE];   // reward term values, [term][env]
  float cla[3][A1_TILE][3];                         // command (post-reset), base lin vel, base ang vel
  ScanEnv ev[A1_TILE];                              // yaw and xy of the PRE-reset pose
  float zb[A1_TILE];                                // z_postreset - h_off
};

// Copy `n` floats global -> shared with float4 when both sides are 16-byte aligned.
__device__ __forceinline__ void load_span(float* __restrict__ dst, const float* __restrict__ src, int n,
                                          int tid, int nthreads) {
  if ((((uintptr_t)src | (uintptr_t)dst) & 15u) == 0) {
    const int n4 = n >> 2;
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* d4 = reinterpret_cast<float4*>(dst);
    for (int i = tid; i < n4; i += nthreads) d4[i] = __ldg(s4 + i);
    for (int i = (n4 << 2) + tid; i < n; i += nthreads) dst[i] = __ldg(src + i);
  } else {
    for (int i = tid; i < n; i += nthreads) dst[i] = __ldg(src + i);
  }
}

__device__ __forceinline__ void store_span(float* __restrict__ dst, const float* __restrict__ src, int n,
                                           int tid, int nthreads) {
  if ((((uintptr_t)src | (uintptr_t)dst) & 15u) == 0) {
    const int n4 = n >> 2;
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* d4 = reinterpret_cast<float4*>(dst);
    for (int i = tid; i < n4; i += nthreads) d4[i] = s4[i];
    for (int i = (n4 << 2) + tid; i < n; i += nthreads) dst[i] = src[i];
  } else {
    for (int i = tid; i < n; i += nthreads) dst[i] = src[i];
  }
}

// Staging of phase A: the tile's root / dof / contact / history / torque / action rows -> shared memory.
__device__ __forceinline__ void a1_stage_rows(A1Smem& s, const A1K& k, const ShifuA1StepIO& io, int e0, int ne, int t) {
  if (k.root_stride == 1 && k.root_offset == 0) {
    load_span(&s.root[0][0], io.root_state + (long long)e0 * 13, ne * 13, t, A1_THREADS);
  } else {
    for (int i = t; i < ne * 13; i += A1_THREADS) {
      const int e = i / 13, c = i % 13;
      s.root[e][c] = io.root_state[((long long)(e0 + e) * k.root_stride + k.root_offset) * 13 + c];
    }
  }
  load_span(&s.dof[0][0], io.dof_state + (long long)e0 * (A1_DOF * 2), ne * A1_DOF * 2, t, A1_THREADS);
  load_span(&s.contact[0][0], io.contact_state + (long long)e0 * (A1_BODIES * 3), ne * A1_BODIES * 3, t, A1_THREADS);
  load_span(&s.hist[0][0], io.history + (long long)e0 * (A1_DOF * A1_HIST), ne * A1_DOF * A1_HIST, t, A1_THREADS);
  load_span(&s.tau[0][0], io.torques + (long long)e0 * A1_DOF, ne * A1_DOF, t, A1_THREADS);
  load_span(&s.act[0][0], io.actions + (long long)e0 * A1_DOF, ne * A1_DOF, t, A1_THREADS);
}

// |f| > thr for a force row f, tested as "sum of squares > thr_sq" with thr_sq = sqrt_threshold(thr)
// from the host: sqrt_rn is correctly rounded and monotonic, so this equals norm3_fma(f) > thr exactly.
__device__ __forceinline__ bool force_exceeds(const float* f, float thr_sq) {
  return fma_rn(f[2], f[2], fma_rn(f[1], f[1], mul_rn(f[0], f[0]))) > thr_sq;
}

// Terms 8-15 (legged_gym-style, see enum ShifuRewardTerm).  Everything a term may read for one env:
struct TermCtx {
  const float *cmd, *lin, *ang, *pg;      // command, body-frame velocities, projected gravity (this step's)
  const float *dof_row, *hist_row, *act_row, *contact_row;
  float base_z;
  float* swing;                           // (num_feet) feet-air-time state of the env (global memory), or nullptr
  unsigned char* last;                    // (num_feet) last_contacts
};

__device__ __noinline__ float a1_extra_term(int code, float p0, float p1, const A1K& k, const TermCtx& c) {
  switch (code) {
    case SHIFU_REW_LIN_VEL_Z:
      return mul_rn(p0, mul_rn(c.lin[2], c.lin[2]));
    case SHIFU_REW_ANG_VEL_XY:
      return mul_rn(p0, add_rn(mul_rn(c.ang[0], c.ang[0]), mul_rn(c.ang[1], c.ang[1])));
    case SHIFU_REW_ORIENTATION:
      return mul_rn(p0, add_rn(mul_rn(c.pg[0], c.pg[0]), mul_rn(c.pg[1], c.pg[1])));
    case SHIFU_REW_DOF_VEL: {
      float acc = 0.0f;
#pragma unroll
      for (int d = 0; d < A1_DOF; ++d) acc = add_rn(acc, mul_rn(c.dof_row[2 * d + 1], c.dof_row[2 * d + 1]));
      return mul_rn(p0, acc);
    }
    case SHIFU_REW_ACTION_RATE: {
      float acc = 0.0f;
#pragma unroll
      for (int d = 0; d < A1_DOF; ++d) {
        const float df = sub_rn(c.hist_row[d * A1_HIST], c.act_row[d]);
        acc = add_rn(acc, mul_rn(df, df));
      }
      return mul_rn(p0, acc);
    }
    case SHIFU_REW_BASE_HEIGHT: {
      const float df = sub_rn(c.base_z, p1);
      return mul_rn(p0, mul_rn(df, df));
    }
    case SHIFU_REW_DOF_POS_LIMITS: {          // -(q - lo).clip(max=0) + (q - hi).clip(min=0), summed over the dofs
      float acc = 0.0f;
#pragma unroll
      for (int d = 0; d < A1_DOF; ++d) {
        const float q = c.dof_row[2 * d];
        const float under = -fminf(sub_rn(q, k.dof_lo[d]), 0.0f), over = fmaxf(sub_rn(q, k.dof_hi[d]), 0.0f);
        acc = add_rn(acc, add_rn(under, over));
      }
      return mul_rn(p0, acc);
    }
    case SHIFU_REW_FEET_AIR_TIME: {           // legged_gym _reward_feet_air_time on swing_time / last_contacts
      if (c.swing == nullptr) return 0.0f;
      float rew = 0.0f;
      for (int f = 0; f < k.n_feet; ++f) {
        const bool contact = c.contact_row[k.feet[f] * 3 + 2] > k.feet_thr;
        const bool filt = contact | (c.last[f] != 0);
        c.last[f] = contact ? 1 : 0;
        float air = c.swing[f];
        const bool first = (air > 0.0f) & filt;
        air = add_rn(air, k.air_dt);
        rew = add_rn(rew, first ? sub_rn(air, p1) : 0.0f);
        c.swing[f] = filt ? 0.0f : air;
      }
      const bool moving = norm2_fma(c.cmd[0], c.cmd[1]) > k.air_cmd_min;
      return mul_rn(p0, moving ? rew : 0.0f);
    }
    default:
      return 0.0f;
  }
}

// One reward term for env e of a staged tile: V3In (pipelined kernel) or A1Smem (phased and eval-terms
// kernels), which both hold root / dof / contact / hist / tau / act rows and cla = command, base lin vel,
// base ang vel.  a1_conditional.py:162-192; every op rounds like the aten elementwise op it stands for.
// Two forms restate the reference exactly: x / p1 is RN(x * rp_inv) when p1 is a power of two (1/p1 is
// then exact), and the leg-force norm test is force_exceeds.
// HAS_EXTRA: the term list may hold a code >= SHIFU_REW_LIN_VEL_Z.
template <bool HAS_EXTRA, class Tile>
__device__ __forceinline__ float a1_reward_term(int code, int q, float p0, float p1, const A1K& k, const Tile& in, int e,
                                                const ShifuA1StepIO& io, long long ge) {
  const float* cmd = in.cla[0][e];
  const float* lin = in.cla[1][e];
  const float* ang = in.cla[2][e];
  if (HAS_EXTRA && code >= SHIFU_REW_LIN_VEL_Z) {   // legged_gym-style terms: pg / air-time state straight from global memory
    const TermCtx c{cmd, lin, ang, io.projected_gravity + ge * 3, in.dof[e], in.hist[e], in.act[e], in.contact[e],
                    in.root[e][2], io.swing_time ? io.swing_time + ge * k.n_feet : nullptr,
                    io.last_contacts ? io.last_contacts + ge * k.n_feet : nullptr};
    return a1_extra_term(code, p0, p1, k, c);
  }
  switch (code) {
    case SHIFU_REW_TRACKING_LIN_VEL: {
      const float dx = sub_rn(cmd[0], lin[0]), dy = sub_rn(cmd[1], lin[1]);
      const float ne = -add_rn(mul_rn(dx, dx), mul_rn(dy, dy));
      return mul_rn(p0, expf(k.rp_pow2[q] ? mul_rn(ne, k.rp_inv[q]) : div_rn(ne, p1)));
    }
    case SHIFU_REW_TRACKING_ANG_VEL: {
      const float d = sub_rn(cmd[2], ang[2]);
      const float ne = -mul_rn(d, d);
      return mul_rn(p0, expf(k.rp_pow2[q] ? mul_rn(ne, k.rp_inv[q]) : div_rn(ne, p1)));
    }
    case SHIFU_REW_STABILIZING_BASE:
      return add_rn(mul_rn(p0, mul_rn(lin[2], lin[2])),
                    mul_rn(p1, add_rn(mul_rn(ang[0], ang[0]), mul_rn(ang[1], ang[1]))));
    case SHIFU_REW_SMOOTHING_ACTION: {
      float f1 = 0.0f, f2 = 0.0f;
#pragma unroll
      for (int d = 0; d < A1_DOF; ++d) {
        const float a0 = in.hist[e][d * A1_HIST + 0], a1 = in.hist[e][d * A1_HIST + 1],
                    a2 = in.hist[e][d * A1_HIST + 2];
        const float d1 = sub_rn(a1, a0);
        const float d2 = add_rn(sub_rn(a2, mul_rn(2.0f, a1)), a0);
        f1 = add_rn(f1, mul_rn(d1, d1));
        f2 = add_rn(f2, mul_rn(d2, d2));
      }
      return mul_rn(p0, add_rn(f1, f2));
    }
    case SHIFU_REW_LEG_COLLISION: {
      int cnt = 0;
      for (int b = 0; b < k.n_leg; ++b)   // rolled on purpose: unrolled, the pipelined kernel's B warps spill (0.4376 vs 0.4289 ms)
        cnt += force_exceeds(&in.contact[e][k.leg[b] * 3], k.rp_thr_sq[q]) ? 1 : 0;
      return mul_rn(p0, (float)cnt);
    }
    case SHIFU_REW_TORQUES: {
      float acc = 0.0f;
#pragma unroll
      for (int d = 0; d < A1_DOF; ++d) acc = add_rn(acc, mul_rn(in.tau[e][d], in.tau[e][d]));
      return mul_rn(p0, acc);
    }
    default:
      return 0.0f;
  }
}

// Term q of the descriptor's list, out of line: the phased and eval-terms kernels call it from a rolled loop.
__device__ __noinline__ float a1_eval_term(int q, const A1K& k, const A1Smem& s, int e, const ShifuA1StepIO& io,
                                           long long ge) {
  return a1_reward_term<true>(k.terms[q], q, k.rp[q][0], k.rp[q][1], k, s, e, io, ge);
}

// The observation layout `o` is applied at run time for every layout (this kernel takes the ragged tail
// and the fallback layouts); for the reference layout it is the identity, and x * 1.0f plus the
// composed clips are exact, so the reference observation comes out unchanged.  NOISE (the host sets it
// when o.noisy): observation noise from the same words as the pipelined kernel, one evaluation per
// column; a compile-time flag, so that the noiseless instantiations keep their registers and code.
// The kernel starts at tile first_tile (the tiles before it are the pipelined kernel's); env indices
// stay absolute, so k and io describe all k.n envs.
// BLIND: the head without the height scan (no phase C, obs rows of HEAD floats); EXACT_DIV does not apply.
// HEAD: the head width, A1_HEAD or A1_HEAD_ACT (the action head, a1_post_physics_kernel_act: columns 36 + d
// are the step's actions in place of the three history slots; heights at HEAD + point).
#define A1_PHASED_KERNEL a1_post_physics_kernel
#define A1_PHASED_HEAD A1_HEAD
#include "a1_fused_kernel.inc"
#undef A1_PHASED_KERNEL
#undef A1_PHASED_HEAD

// The action head (num_obs = 235, or 48 with BLIND).
#define A1_PHASED_KERNEL a1_post_physics_kernel_act
#define A1_PHASED_HEAD A1_HEAD_ACT
#include "a1_fused_kernel.inc"
#undef A1_PHASED_KERNEL
#undef A1_PHASED_HEAD

// Row a7 stand-alone (shifu_a1_eval_terms): the descriptor's term list on the current tensors, one
// CTA per 32 envs with the rows staged like phase A of the fused kernel; writes nothing but out.
__global__ void __launch_bounds__(A1_THREADS)
a1_eval_terms_kernel(const __grid_constant__ A1K k, const __grid_constant__ ShifuA1StepIO io, float* __restrict__ out) {
  __shared__ __align__(16) A1Smem s;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  for (int e0 = blockIdx.x * A1_TILE; e0 < k.n; e0 += gridDim.x * A1_TILE) {
    const int ne = min(A1_TILE, k.n - e0);
    const int ge = e0 + lane;
    __syncthreads();
    a1_stage_rows(s, k, io, e0, ne, t);
    if (warp == 0 && lane < ne) {
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        s.cla[0][lane][j] = io.command[ge * 3LL + j];
        s.cla[1][lane][j] = io.base_lin_vel[ge * 3LL + j];
        s.cla[2][lane][j] = io.base_ang_vel[ge * 3LL + j];
      }
    }
    __syncthreads();
    if (lane < ne)
#pragma unroll 1
      for (int j = warp; j < k.n_terms; j += A1_THREADS / 32) out[(long long)j * k.n + ge] = a1_eval_term(j, k, s, lane, io, ge);
  }
}

}  // namespace shifu
