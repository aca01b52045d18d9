// A1 conditional-walking kernels (sm_100a).  Rows a2, a3, a5-a7, a9-a14 of SURVEY.md §8(a).
//
// Everything here is HBM-/LSU-bound fp32 + integer work; there is no contraction, so no
// tensor-core path.  The design rules that matter: one pass over every state tensor with
// coalesced 128-bit loads, the obs row written once with streaming stores, grids sized by the
// SM count, and the 187-point height scan served from an L2-resident banded table.
#pragma once
#include "exact_math.cuh"
#include "philox.cuh"
#include "../../include/shifu_b200.h"

namespace shifu {

// Compile-time shape of the A1 task (validated against the descriptor in shifu_ctx_create).
constexpr int A1_DOF = 12, A1_BODIES = 17, A1_HIST = 3, A1_OBS = 259;
constexpr int A1_NX = 17, A1_NY = 11, A1_POINTS = A1_NX * A1_NY;   // 187
constexpr int A1_HEAD = A1_OBS - A1_POINTS;                          // 72 non-height obs columns
constexpr int A1_TILE = 32;       // envs per CTA
constexpr int A1_THREADS = 192;   // 6 warps: 187 scan points + 5 idle lanes
constexpr int TILE_SHIFT = 3;     // scan table stored in bands of 8 map rows: a 128-B line = 8x8 cells

// Kernel-side constants (passed by value as a __grid_constant__ parameter: constant bank).
constexpr int A1K_TERM_WARPS = 4;     // the pipelined kernel splits the term list over up to this many warps

struct A1K {
  int n;
  long long env_offset;
  unsigned long long seed;
  int base_body, n_leg, leg[SHIFU_MAX_LEG_BODIES], force_body;
  int root_stride, root_offset;
  float q0[A1_DOF], kp[A1_DOF], kd[A1_DOF], tau_max[A1_DOF];
  float action_scale, clip_actions, clip_obs;
  float px[A1_NX], py[A1_NY];
  float border;
  ConstDiv hdiv;          // horizontal_scale and its rounded reciprocal
  int exact_div;          // 1: use __fdiv_rn instead of the 3-op constant division
  float vscale, h_off, h_clip;
  long long max_len;
  float max_len_s, contact_thr;
  float root0[7];
  float xy_span, xy_low, force_span, force_low, cmd_span[3], cmd_low[3];
  int curriculum, max_level, n_types;
  float up_dist, down_factor;
  int n_terms, terms[SHIFU_MAX_REWARD_TERMS];
  float rp[SHIFU_MAX_REWARD_TERMS][2];
  float rp_inv[SHIFU_MAX_REWARD_TERMS];   // 1/p1 when p1 is a power of two: x/p1 == x*rp_inv exactly
  int rp_pow2[SHIFU_MAX_REWARD_TERMS];
  // largest s with sqrt_rn(s) <= threshold: "norm > thr" == "sum of squares > thr_sq" exactly
  float rp_thr_sq[SHIFU_MAX_REWARD_TERMS];
  // constants of the row-N1 terms (dof-limit, feet-air-time)
  float dof_lo[A1_DOF], dof_hi[A1_DOF];
  int n_feet, feet[4];
  float feet_thr, air_cmd_min, air_dt;
  int air_reset;
  // term lists of the B warps of the pipelined kernel (host-side cost balance)
  int term_count[A1K_TERM_WARPS], term_list[A1K_TERM_WARPS][SHIFU_MAX_REWARD_TERMS];
  float contact_thr_sq;
  // scan table
  const short* table;     // banded min-of-3 table T[px>>3][py][px&7]: a 128-B line = 8x8 cells
  int trows, tcols;       // valid index range: px in [0, trows-1], py in [0, tcols-1]
  int band_w;             // entries per map row inside a band (tcols padded to 8)
  double* stats;          // SHIFU_NUM_STATS accumulators
  float neg_zero;         // -0.0f, opaque to ptxas: see the fma(a, b, -0) products in scan_pairs.cuh
};

// Observation layout of the fused step (ShifuA1Desc.obs_layout = 1): a separate __grid_constant__
// parameter appended after the existing ones, so that A1K and the parameter offsets of the
// reference-layout instantiations stay as they are.  Identity (src = 0, 1, 2, 3, every scale 1) for
// the reference observation.
static_assert(A1_HEAD == SHIFU_OBS_HEAD, "observation head width");
struct A1Obs {
  int src[4];             // enum ShifuObsVec of columns 3i..3i+2
  float scale[A1_HEAD];   // obs[j] = clip(x_j * scale[j], +-clip_obs)
  float h_scale;          // heights: clip(clip(z - h_off - h, +-h_clip) * h_scale, +-clip_obs)
  float h_bound;          // min(h_clip * |h_scale|, clip_obs): the same heights as clip((z - h_off - h) * h_scale,
                          // +-h_bound), because rounding the product is monotonic and sign-symmetric
  int uses_pg;            // some slot reads projected_gravity
  // uniform noise, added before the clip to +-clip_obs (0 everywhere: none).  With noise the heights are
  // clip(clip(clip(z - h_off - h, +-h_clip) * h_scale + n, +-clip_obs)): h_bound does not apply.
  float noise[A1_HEAD];   // head column j: n = (2u - 1) * noise[j]
  float h_noise;          // every height column
  int noisy;              // some noise scale is non-zero
};
static_assert(STREAM_OBS_NOISE == SHIFU_STREAM_OBS_NOISE, "observation-noise stream");

// Head width of the action head (ShifuA1Desc.num_obs = 235 or 48): the slots, dof_pos - q0, dof_vel and the
// step's actions, where the 72-column head has the three history slots.
constexpr int A1_HEAD_ACT = 48;
static_assert(A1_HEAD_ACT == SHIFU_OBS_HEAD_ACT, "action head width");

// Noise n = (2u - 1) * s of head column j < HEAD or height column j >= HEAD of env gid (the phased kernel's
// form: one Philox evaluation per column; the pipelined kernel shares the words between lanes).
template <int HEAD = A1_HEAD>
__device__ __forceinline__ float obs_noise_at(const A1Obs& o, unsigned long long seed, long long gid, long long step,
                                              int j) {
  uint32_t word;
  int lane;
  obs_noise_slot(j, word, lane, HEAD);
  return mul_rn(u_pm1(u4_lane(obs_noise_word(seed, gid, step, word), lane)), j < HEAD ? o.noise[j] : o.h_noise);
}

// Value of head column j < 12 of env e: slot j / 3, component j % 3.  cla = command, base lin vel,
// base ang vel of the env; pg = component j % 3 of its projected gravity when the step started.
template <class Cla>
__device__ __forceinline__ float a1_obs_vec(const A1Obs& o, int j, const Cla& cla, int e, float pg) {
  const int c = j % 3;
  switch (o.src[j / 3]) {
    case SHIFU_OBS_COMMAND: return cla[0][e][c];
    case SHIFU_OBS_BASE_LIN_VEL: return cla[1][e][c];
    case SHIFU_OBS_BASE_ANG_VEL: return cla[2][e][c];
    case SHIFU_OBS_GRAVITY_VEC: return c == 2 ? -1.0f : 0.0f;
    default: return pg;
  }
}

__device__ __forceinline__ int table_index(unsigned px, unsigned py, const A1K& k) {
  // (px>>3)*8*W + py*8 + (px&7)  ==  (px & ~7)*(W-1) + px + 8*py      (3 integer ops)
  return (int)((px & ~7u) * (unsigned)(k.band_w - 1) + px + (py << TILE_SHIFT));
}

// ------------------------------------------------------------------------------------------
// Scan-table build: T[px][py] = min(H[px][py], H[px+1][py], H[px][py+1])
// (shifu/gym/isaac_gym.py:427-431 folded; the map is static after create_ground()).
// ------------------------------------------------------------------------------------------
__global__ void build_scan_table_kernel(const short* __restrict__ H, int rows, int cols,
                                        short* __restrict__ T, int band_w) {
  const int trows = rows - 1, tcols = cols - 1;
  const long long total = (long long)trows * tcols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int px = (int)(i / tcols), py = (int)(i % tcols);
    const short a = H[(long long)px * cols + py];
    const short b = H[(long long)(px + 1) * cols + py];
    const short c = H[(long long)px * cols + py + 1];
    T[(long long)(px >> TILE_SHIFT) * 8 * band_w + (long long)py * 8 + (px & 7)] = min(min(a, b), c);
  }
}

// ------------------------------------------------------------------------------------------
// Row a1/a2: (optional) action scale+clip, then one PD substep.
//   tau = clip(kp*((a + q0) - q) - kd*qd, +-tau_max)       a1_conditional.py:66-67
// One thread per group of 4 consecutive dofs (3 groups per env): one 128-bit action load, two
// 128-bit dof_state loads (4 x (pos, vel)), one 128-bit torque store — all fully coalesced.
// Pure streaming: 192 B/env per substep (240 B when the clipped actions are written too).
// descending != 0 sweeps the quads from the last one down (loop counter i processes quad
// total-1-i), so a launch can start on the rows the launch before it touched last, which are
// still in L2.  A warp still covers a contiguous span, so the accesses stay coalesced; which
// launch sweeps which way is decided in capi.cu (shifu_pd_torque).  The first half of every
// sweep is the half the next, reversed sweep reaches last, long after it has left L2: its loads
// and stores carry an L2 evict_first policy, so that the second half, which the next sweep
// starts on, keeps more of L2.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float pd_one(float a, float q0, float kp, float kd, float lim, float q, float qd) {
  const float e = sub_rn(add_rn(a, q0), q);
  return clampf(sub_rn(mul_rn(kp, e), mul_rn(kd, qd)), -lim, lim);
}

__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
  unsigned long long p;
  asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ unsigned long long l2_policy_evict_normal() {
  unsigned long long p;
  asm("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// read-only (non-coherent) 128-bit load / 128-bit store with an L2 cache policy
__device__ __forceinline__ float4 ldg_l2(const float4* p, unsigned long long pol) {
  float4 v;
  asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ void stg_l2(float4* p, float4 v, unsigned long long pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;"
               :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}

__global__ void __launch_bounds__(256)
pd_torque_kernel(const __grid_constant__ A1K k, const float4* __restrict__ a_in, float4* __restrict__ a_out,
                 const float4* __restrict__ dof, float4* __restrict__ tau, int descending) {
  __shared__ __align__(16) float c_q0[A1_DOF], c_kp[A1_DOF], c_kd[A1_DOF], c_lim[A1_DOF];
  if (threadIdx.x < A1_DOF) {
    c_q0[threadIdx.x] = k.q0[threadIdx.x];
    c_kp[threadIdx.x] = k.kp[threadIdx.x];
    c_kd[threadIdx.x] = k.kd[threadIdx.x];
    c_lim[threadIdx.x] = k.tau_max[threadIdx.x];
  }
  __syncthreads();
  const unsigned total = (unsigned)k.n * (A1_DOF / 4);          // <= 3 * 2^31 / 4 quads
  const float sc = k.action_scale, ca = k.clip_actions;
  const unsigned long long pol_first = l2_policy_evict_first(), pol_normal = l2_policy_evict_normal();
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const unsigned q = descending ? total - 1u - i : i;           // the quad this iteration processes
    const unsigned g = q % 3u;                                    // which third of the env's 12 dofs
    const unsigned long long pol = i < total / 2u ? pol_first : pol_normal;
    float4 a = ldg_l2(a_in + q, pol);
    if (a_out != nullptr) {                                       // a1_conditional.py:123, env.py:87
      a.x = clampf(mul_rn(a.x, sc), -ca, ca); a.y = clampf(mul_rn(a.y, sc), -ca, ca);
      a.z = clampf(mul_rn(a.z, sc), -ca, ca); a.w = clampf(mul_rn(a.w, sc), -ca, ca);
      stg_l2(a_out + q, a, pol);
    }
    const float4 s0 = ldg_l2(dof + 2 * (size_t)q, pol), s1 = ldg_l2(dof + 2 * (size_t)q + 1, pol);
    const float4 q0 = reinterpret_cast<const float4*>(c_q0)[g], kp = reinterpret_cast<const float4*>(c_kp)[g];
    const float4 kd = reinterpret_cast<const float4*>(c_kd)[g], lm = reinterpret_cast<const float4*>(c_lim)[g];
    float4 t;
    t.x = pd_one(a.x, q0.x, kp.x, kd.x, lm.x, s0.x, s0.y);
    t.y = pd_one(a.y, q0.y, kp.y, kd.y, lm.y, s0.z, s0.w);
    t.z = pd_one(a.z, q0.z, kp.z, kd.z, lm.z, s1.x, s1.y);
    t.w = pd_one(a.w, q0.w, kp.w, kd.w, lm.w, s1.z, s1.w);
    stg_l2(tau + q, t, pol);
  }
}

// quat_rotate_inverse (isaacgym.torch_utils): a = v(2w^2-1); b = 2w(q x v); c = 2q(q.v); a - b + c
__device__ __forceinline__ void rotate_inverse(const float* q, float vx, float vy, float vz, float* out) {
  const float qx = q[0], qy = q[1], qz = q[2], qw = q[3];
  const float s = sub_rn(mul_rn(2.0f, mul_rn(qw, qw)), 1.0f);
  const float cx = fma_rn(qy, vz, -mul_rn(qz, vy));   // torch CPU cross uses fma(a,b,-fl(c*d))
  const float cy = fma_rn(qz, vx, -mul_rn(qx, vz));
  const float cz = fma_rn(qx, vy, -mul_rn(qy, vx));
  const float dot = add_rn(add_rn(mul_rn(qx, vx), mul_rn(qy, vy)), mul_rn(qz, vz));
  const float v[3] = {vx, vy, vz}, c[3] = {cx, cy, cz}, qq[3] = {qx, qy, qz};
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const float a = mul_rn(v[i], s);
    const float b = mul_rn(mul_rn(c[i], qw), 2.0f);
    const float cc = mul_rn(mul_rn(qq[i], dot), 2.0f);
    out[i] = add_rn(sub_rn(a, b), cc);
  }
}

// ------------------------------------------------------------------------------------------
// Row a3: LeggedRobot.post_step (shifu/units/robot.py:222-229), one thread per env.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
body_frame_kernel(int n, int root_stride, int root_offset, const float* __restrict__ root, float* __restrict__ lin,
                  float* __restrict__ ang, float* __restrict__ pg, float* __restrict__ gvec) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    const float* r = root + ((long long)e * root_stride + root_offset) * 13;
    float row[13];
#pragma unroll
    for (int j = 0; j < 13; ++j) row[j] = r[j];
    float o[3];
    rotate_inverse(row + 3, row[7], row[8], row[9], o);
    lin[e * 3 + 0] = o[0]; lin[e * 3 + 1] = o[1]; lin[e * 3 + 2] = o[2];
    rotate_inverse(row + 3, row[10], row[11], row[12], o);
    ang[e * 3 + 0] = o[0]; ang[e * 3 + 1] = o[1]; ang[e * 3 + 2] = o[2];
    rotate_inverse(row + 3, 0.0f, 0.0f, -1.0f, o);
    pg[e * 3 + 0] = o[0]; pg[e * 3 + 1] = o[1]; pg[e * 3 + 2] = o[2];
    if (gvec != nullptr) { gvec[e * 3 + 0] = 0.0f; gvec[e * 3 + 1] = 0.0f; gvec[e * 3 + 2] = -1.0f; }
  }
}

// ------------------------------------------------------------------------------------------
// The height scan of ONE point (rows a5): yaw-rotate (bx,by), translate, to cell index, gather.
//   quat_apply_yaw: shifu/utils/terrain.py:202-206; get_heights: shifu/gym/isaac_gym.py:416-433
// ev = {2*zq, zq, wq, pos_x, pos_y} with (zq, wq) the normalised yaw quaternion.
// Every op keeps the rounding of the aten elementwise op it stands for.
// ------------------------------------------------------------------------------------------
struct ScanEnv {
  float z2, z, w, x, y;
};

__device__ __forceinline__ ScanEnv make_scan_env(const float* root_row) {
  const float qz = root_row[5], qw = root_row[6];
  // normalize((0,0,qz,qw)): x / clamp(sqrt(fl(qz^2)+fl(qw^2)), 1e-9)
  float nrm = sqrt_rn(add_rn(mul_rn(qz, qz), mul_rn(qw, qw)));
  nrm = fmaxf(nrm, 1e-9f);
  ScanEnv ev;
  ev.z = div_rn(qz, nrm);
  ev.w = div_rn(qw, nrm);
  ev.z2 = mul_rn(ev.z, 2.0f);
  ev.x = root_row[0];
  ev.y = root_row[1];
  return ev;
}

// EXACT_DIV: / horizontal_scale as __fdiv_rn (A1K::exact_div), else the 3-op constant division
template <bool EXACT_DIV>
__device__ __forceinline__ float scan_point(const ScanEnv& ev, float bx, float by, const A1K& k,
                                            unsigned* opx, unsigned* opy) {
  // t = 2*(q_xyz x b) with q_xyz = (0,0,z), b = (bx,by,0)  ->  (-2z*by, 2z*bx, 0)
  const float tx = -mul_rn(ev.z2, by);
  const float ty = mul_rn(ev.z2, bx);
  // b + w*t + q_xyz x t ;  q_xyz x t = (-z*ty, z*tx, 0)
  const float rx = add_rn(add_rn(bx, mul_rn(ev.w, tx)), -mul_rn(ev.z, ty));
  const float ry = add_rn(add_rn(by, mul_rn(ev.w, ty)), mul_rn(ev.z, tx));
  // + base xy, + border, / horizontal_scale, .long() (trunc), clip to [0, dim-2]
  const float ax = add_rn(add_rn(rx, ev.x), k.border);
  const float ay = add_rn(add_rn(ry, ev.y), k.border);
  const float fx = EXACT_DIV ? div_rn(ax, k.hdiv.d) : div_const(ax, k.hdiv);
  const float fy = EXACT_DIV ? div_rn(ay, k.hdiv.d) : div_const(ay, k.hdiv);
  // float->unsigned conversion truncates toward zero and saturates (negatives -> 0)
  const unsigned px = min(__float2uint_rz(fx), (unsigned)(k.trows - 1));
  const unsigned py = min(__float2uint_rz(fy), (unsigned)(k.tcols - 1));
  *opx = px; *opy = py;
  const short h = __ldg(k.table + table_index(px, py, k));
  return mul_rn((float)h, k.vscale);
}

// Stand-alone get_heights (for user-hook tasks and the index parity tests): one CTA per
// A1_TILE envs, thread t < 187 owns scan point t.
__global__ void __launch_bounds__(A1_THREADS)
get_heights_kernel(const __grid_constant__ A1K k, const float* __restrict__ root, float* __restrict__ mh,
                   int* __restrict__ cell_idx) {
  __shared__ ScanEnv s_ev[A1_TILE];
  const int t = threadIdx.x;
  const float bx = k.px[t % A1_NX], by = k.py[(t / A1_NX) % A1_NY];
  for (int e0 = blockIdx.x * A1_TILE; e0 < k.n; e0 += gridDim.x * A1_TILE) {
    const int ne = min(A1_TILE, k.n - e0);
    __syncthreads();
    if (t < ne) s_ev[t] = make_scan_env(root + ((long long)(e0 + t) * k.root_stride + k.root_offset) * 13);
    __syncthreads();
    if (t < A1_POINTS) {
      for (int e = 0; e < ne; ++e) {
        unsigned px, py;
        const float h = k.exact_div ? scan_point<true>(s_ev[e], bx, by, k, &px, &py)
                                    : scan_point<false>(s_ev[e], bx, by, k, &px, &py);
        const long long o = (long long)(e0 + e) * A1_POINTS + t;
        mh[o] = h;
        if (cell_idx != nullptr) { cell_idx[2 * o] = (int)px; cell_idx[2 * o + 1] = (int)py; }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// Reset of ONE env (rows a9-a11): A1Conditional.reset_idx, a1_conditional.py:116-120, i.e.
// update_terrain_curriculum (:204-221) -> ShifuVecEnv.reset_idx (env.py:114-130) ->
// IsaacGymEnv.reset_idx / A1Robot.reset_idx (isaac_gym.py:54-73, robot.py:74-86,
// a1_conditional.py:43-50,77-87) -> sample_command (:194-200).
// root_row / dof_row / hist_row are the env's rows wherever the caller keeps them (shared memory
// inside K-main, global memory in the stand-alone kernel); with MIRROR the root/dof rows are
// additionally written through to the flat gym tensors.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// PARTS: 1 = state rewrite (curriculum, dof / root rows, push force, history, command), 2 = episode
// bookkeeping (length, episode sums -> log sums); the pipelined kernel runs the two on different warps.
template <bool MIRROR, int PARTS = 3, bool AIR = true>
__device__ __forceinline__ void a1_reset_env(const A1K& k, const ShifuA1StepIO& io, long long step, int ge,
                                             float* root_row, float* dof_row, float* hist_row,
                                             float (&cmd)[3], float (&esum)[SHIFU_MAX_REWARD_TERMS],
                                             long long& len, double (&st_sum)[SHIFU_MAX_REWARD_TERMS],
                                             long long& level_delta, float ox, float oy, float oz,
                                             long long old_level, long long ty) {
  // (ox, oy, oz) = env_origins[ge], old_level = terrain_levels[ge], ty = terrain_types[ge]: read by
  // the caller (global memory, or the shared-memory stage the pipelined kernel bulk-loads them into)
  const long long gid = k.env_offset + ge;
  if (PARTS & 2) {                                                       // env.py:119-122 ; log_info, env.py:149-153
    len = 0;
#pragma unroll
    for (int j = 0; j < SHIFU_MAX_REWARD_TERMS; ++j) {
      if (j < k.n_terms) { st_sum[j] = (double)esum[j]; esum[j] = 0.0f; }
    }
  }
  if (!(PARTS & 1)) return;
  if (k.curriculum) {                                                    // a1_conditional.py:204-221
    const float dist = norm2_fma(sub_rn(root_row[0], ox), sub_rn(root_row[1], oy));
    const bool up = dist > k.up_dist;
    const float need = mul_rn(mul_rn(norm2_fma(cmd[0], cmd[1]), k.max_len_s), k.down_factor);
    const bool down = (dist < need) && !up;
    long long level = old_level + (up ? 1 : 0) - (down ? 1 : 0);
    const long long rnd = randint(draw(k.seed, gid, step, STREAM_LEVEL).x, k.max_level);
    level = (level >= k.max_level) ? rnd : (level < 0 ? 0 : level);
    io.terrain_levels[ge] = level;
    level_delta = level - old_level;
    const float* org = io.terrain_origins + (level * k.n_types + ty) * 3;   // isaac_gym.py:387-391
    ox = org[0]; oy = org[1]; oz = org[2];
    io.env_origins[ge * 3LL + 0] = ox; io.env_origins[ge * 3LL + 1] = oy; io.env_origins[ge * 3LL + 2] = oz;
  }
  // Robot._reset_dof_state, shifu/units/robot.py:74-77
#pragma unroll
  for (int d = 0; d < A1_DOF; ++d) {
    dof_row[2 * d] = k.q0[d];
    dof_row[2 * d + 1] = 0.0f;
    io.dof_targets[ge * (long long)A1_DOF + d] = k.q0[d];
  }
  if (MIRROR) {
    float4* drow = reinterpret_cast<float4*>(io.dof_state + (long long)ge * (A1_DOF * 2));
    const float4* srow = reinterpret_cast<const float4*>(dof_row);
#pragma unroll
    for (int j = 0; j < A1_DOF * 2 / 4; ++j) drow[j] = srow[j];
  }
  // A1Robot._reset_root_state, a1_conditional.py:43-50
  const U4 uxy = draw(k.seed, gid, step, STREAM_XY);
  float rr[13];
  rr[0] = add_rn(add_rn(k.root0[0], ox), add_rn(mul_rn(k.xy_span, u01(uxy.x)), k.xy_low));
  rr[1] = add_rn(add_rn(k.root0[1], oy), add_rn(mul_rn(k.xy_span, u01(uxy.y)), k.xy_low));
  rr[2] = add_rn(k.root0[2], oz);
  rr[3] = k.root0[3]; rr[4] = k.root0[4]; rr[5] = k.root0[5]; rr[6] = k.root0[6];
#pragma unroll
  for (int j = 7; j < 13; ++j) rr[j] = 0.0f;
  float* grow = io.root_state + ((long long)ge * k.root_stride + k.root_offset) * 13;
#pragma unroll
  for (int j = 0; j < 13; ++j) {
    root_row[j] = rr[j];
    if (MIRROR) grow[j] = rr[j];
  }
  // update_rand_force_buf, a1_conditional.py:82-87
  const U4 uf = draw(k.seed, gid, step, STREAM_FORCE);
  float* fr = io.rand_force + ((long long)ge * A1_BODIES + k.force_body) * 3;
  fr[0] = add_rn(mul_rn(k.force_span, u01(uf.x)), k.force_low);
  fr[1] = add_rn(mul_rn(k.force_span, u01(uf.y)), k.force_low);
  fr[2] = add_rn(mul_rn(k.force_span, u01(uf.z)), k.force_low);
  // HistoryRecorder.reset_idx, train.py:16-17
#pragma unroll
  for (int j = 0; j < A1_DOF * A1_HIST; ++j) hist_row[j] = 0.0f;
  if (AIR && k.air_reset && io.swing_time != nullptr) {                      // legged_gym reset_idx: feet_air_time[env_ids] = 0
    for (int f = 0; f < k.n_feet; ++f) {
      io.swing_time[(long long)ge * k.n_feet + f] = 0.0f;
      io.last_contacts[(long long)ge * k.n_feet + f] = 0;
    }
  }
  // sample_command, a1_conditional.py:194-200
  const U4 uc = draw(k.seed, gid, step, STREAM_CMD);
  cmd[0] = add_rn(mul_rn(k.cmd_span[0], u01(uc.x)), k.cmd_low[0]);
  cmd[1] = add_rn(mul_rn(k.cmd_span[1], u01(uc.y)), k.cmd_low[1]);
  cmd[2] = add_rn(mul_rn(k.cmd_span[2], u01(uc.z)), k.cmd_low[2]);
  io.command[ge * 3LL + 0] = cmd[0]; io.command[ge * 3LL + 1] = cmd[1]; io.command[ge * 3LL + 2] = cmd[2];
}

// Warp-level reduction of the per-step log sums (env.py:149-153) -> one set of atomics per warp.
template <int PARTS = 3>
__device__ __forceinline__ void a1_log_sums(const A1K& k, bool reset, const double (&st_sum)[SHIFU_MAX_REWARD_TERMS],
                                            long long level_delta, int lane) {
  const unsigned any = __ballot_sync(0xffffffffu, reset);
  if (!any) return;
  if (PARTS != 3) {              // split form (pipelined kernel): direct reductions only
    if (reset) {
      if (PARTS & 2) {
#pragma unroll
        for (int j = 0; j < SHIFU_MAX_REWARD_TERMS; ++j)
          if (j < k.n_terms) atomicAdd(k.stats + SHIFU_STAT_TERM0 + j, st_sum[j]);
        atomicAdd(k.stats + SHIFU_STAT_NRESET, 1.0);
      }
      if ((PARTS & 1) && level_delta != 0) atomicAdd(k.stats + SHIFU_STAT_LEVEL_SUM, (double)level_delta);
    }
    return;
  }
  if (__popc(any) <= 4) {
    // sparse resets (the steady state, ~1 % of envs): a handful of fire-and-forget reductions is
    // cheaper for the latency-critical warp than seven 5-step double-precision warp reductions
    if (reset) {
#pragma unroll
      for (int j = 0; j < SHIFU_MAX_REWARD_TERMS; ++j)
        if (j < k.n_terms) atomicAdd(k.stats + SHIFU_STAT_TERM0 + j, st_sum[j]);
      atomicAdd(k.stats + SHIFU_STAT_NRESET, 1.0);
      if (level_delta != 0) atomicAdd(k.stats + SHIFU_STAT_LEVEL_SUM, (double)level_delta);
    }
    return;
  }
  const double cnt = warp_sum(reset ? 1.0 : 0.0);
  const double dl = warp_sum((double)level_delta);
#pragma unroll
  for (int j = 0; j < SHIFU_MAX_REWARD_TERMS; ++j) {
    if (j < k.n_terms) {
      const double v = warp_sum(st_sum[j]);
      if (lane == 0) atomicAdd(k.stats + SHIFU_STAT_TERM0 + j, v);
    }
  }
  if (lane == 0) {
    atomicAdd(k.stats + SHIFU_STAT_NRESET, cnt);
    if (dl != 0.0) atomicAdd(k.stats + SHIFU_STAT_LEVEL_SUM, dl);
  }
}

// Stand-alone reset_idx(env_ids) (user calls / ShifuVecEnv.reset, env.py:108-112): one thread per id;
// ids == nullptr means arange(n_ids).
__global__ void __launch_bounds__(128)
a1_reset_idx_kernel(const __grid_constant__ A1K k, const __grid_constant__ ShifuA1StepIO io,
                    const long long* __restrict__ ids, int n_ids) {
  const long long step = (io.step_dev != nullptr) ? *io.step_dev : io.step;
  const int lane = threadIdx.x & 31;
  for (int i0 = blockIdx.x * blockDim.x; i0 < n_ids; i0 += gridDim.x * blockDim.x) {
    const int i = i0 + threadIdx.x;
    bool reset = false;
    double st_sum[SHIFU_MAX_REWARD_TERMS];
#pragma unroll
    for (int j = 0; j < SHIFU_MAX_REWARD_TERMS; ++j) st_sum[j] = 0.0;
    long long level_delta = 0;
    if (i < n_ids) {
      const int ge = (ids != nullptr) ? (int)ids[i] : i;
      if (ge >= 0 && ge < k.n) {
        reset = true;
        float cmd[3], esum[SHIFU_MAX_REWARD_TERMS];
#pragma unroll
        for (int j = 0; j < 3; ++j) cmd[j] = io.command[ge * 3LL + j];
#pragma unroll
        for (int j = 0; j < SHIFU_MAX_REWARD_TERMS; ++j) esum[j] = (j < k.n_terms) ? io.ep_sums[j][ge] : 0.0f;
        long long len = 0;
        a1_reset_env<false>(k, io, step, ge, io.root_state + ((long long)ge * k.root_stride + k.root_offset) * 13,
                            io.dof_state + (long long)ge * (A1_DOF * 2),
                            io.history + (long long)ge * (A1_DOF * A1_HIST), cmd, esum, len, st_sum, level_delta,
                            io.env_origins[ge * 3LL + 0], io.env_origins[ge * 3LL + 1], io.env_origins[ge * 3LL + 2],
                            k.curriculum ? io.terrain_levels[ge] : 0, k.curriculum ? io.terrain_types[ge] : 0);
        io.ep_len[ge] = 0;
        io.reset_buf[ge] = 1;
#pragma unroll
        for (int j = 0; j < SHIFU_MAX_REWARD_TERMS; ++j)
          if (j < k.n_terms) io.ep_sums[j][ge] = 0.0f;
      }
    }
    a1_log_sums(k, reset, st_sum, level_delta, lane);
  }
}
}  // namespace shifu
