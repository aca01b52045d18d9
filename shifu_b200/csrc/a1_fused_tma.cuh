// K-main, pipelined form (the default for full 32-env tiles): persistent CTAs (2 per SM, 512 threads =
// the whole register file at 64 registers) with three warp roles that never meet at a CTA-wide barrier —
//
//   DMA warp (1 lane)    bulk-TMA loads (cp.async.bulk -> mbarrier, SASS UBLKCP) of everything the
//                        tile reads — the root / dof / contact / history / torque / action rows
//                        and the per-env scalars (ep_len, command, carried velocities, episode
//                        sums) — into a ring of three shared-memory stages, refilled as soon as the
//                        tile's head phase is over; bulk-TMA stores of the pushed history tile and of
//                        the carried body-frame rows
//   B group (3 warps; lane = env)
//                        yaw normalisation for the scan (warp 0, first: the scan group starts on
//                        e_done), the reward-term list (split over the three warps by a host-side cost
//                        balance; warp 2 does nothing else and runs ahead into the next tile's terms)
//                        + episode sums, termination, reset (curriculum, Philox draws, state rewrite
//                        and the carried body-frame velocities of the post-reset pose — warp 1,
//                        while warp 0 does the ordered accumulation and the flags), per-step log
//                        sums — the scalar game logic of ShifuVecEnv.post_step (env.py:93-106);
//                        reads only the stage (plus env origin / terrain level / type of the ~1 % of
//                        envs that reset)
//   scan group (12 warps; thread = scan point + its mirror point, warp w: point pairs 32*(w%3)..,
//                        env pairs 4*(w/3) .. +3 in two items of 4 envs)
//                        first item's index arithmetic + gathers, then the obs head from the
//                        post-reset rows (a1_conditional.py:131-144, or the A1Obs layout with OBS),
//                        history push (train.py:12-14),
//                        then the rest of the 187-point height scan (isaac_gym.py:393-433) with
//                        packed fp32x2 arithmetic (two envs per instruction, one yaw rotation per
//                        point pair), streamed with st.global.cs
//
// mbarriers hand a stage round DMA -> B -> scan -> DMA; every thread of the producing group
// arrives itself, so fast warps never wait for slow siblings.  The per-env scalars the scan needs
// travel through a 4-deep ring, which lets the B group run ahead of the scan group.
#pragma once
#include "a1_fused.cuh"
#include "scan_pairs.cuh"
#include "tma_pipe.cuh"

namespace shifu {

constexpr int V3_STAGES = 3;                      // input stages per CTA (the scalar ring holds 4)
constexpr int V3_CTAS_PER_SM = 2;
constexpr int V3_BG_WARPS = 3;                    // warps 0, 1: terms + B2; warp 2: terms only
constexpr int V3_SCAN_WARPS = 12;
static_assert(V3_BG_WARPS <= A1K_TERM_WARPS, "A1K holds a term list per B warp");
constexpr int V3_B_THREADS = 32 * V3_BG_WARPS, V3_B2_THREADS = 64;
constexpr int V3_C_THREADS = 32 * V3_SCAN_WARPS;
constexpr int V3_DMA_THREADS = 32;
constexpr int V3_THREADS = V3_B_THREADS + V3_C_THREADS + V3_DMA_THREADS;
constexpr int V3_SCAN_BASE = V3_B_THREADS;
constexpr int V3_DMA_BASE = V3_B_THREADS + V3_C_THREADS;
constexpr uint32_t V3_OBS_CHUNK_BYTES = 8 * A1_OBS * 4;      // 8288 = 16 * 518

struct alignas(128) V3In {            // one tile of simulator/env rows, each member 16-B aligned
  float root[A1_TILE][13];            //  1664 B
  float dof[A1_TILE][A1_DOF * 2];     //  3072 B
  float contact[A1_TILE][A1_BODIES * 3];   // 6528 B
  float hist[A1_TILE][A1_DOF * A1_HIST];   // 4608 B  (pushed in place, then bulk-stored back)
  float tau[A1_TILE][A1_DOF];         //  1536 B
  float act[A1_TILE][A1_DOF];         //  1536 B
  // per-env scalars: bulk-loaded with the rows, so the B warps issue no global loads of their own
  long long ep_len[A1_TILE];          //   256 B
  float cla[3][A1_TILE][3];           //  1152 B  command (rewritten on reset), base lin vel, base ang vel
  float esum[SHIFU_MAX_REWARD_TERMS][A1_TILE];   // 1024 B  (the first n_terms rows are loaded)
  // output rows: carried body-frame velocities / projected gravity of the POST-reset pose, written by
  // the B group and bulk-stored by the DMA lane together with the pushed history
  float cout[3][A1_TILE][3];          //  1152 B
};
static_assert(sizeof(V3In) == 22528 && offsetof(V3In, ep_len) == 18944 && offsetof(V3In, cout) % 16 == 0, "tile layout");

struct alignas(128) V3Smem {
  V3In in[V3_STAGES];
  // per-env scan scalars, laid out per env PAIR (e, e+1) so that one 128-bit broadcast load yields
  // two packed fp32x2 operands: sA = (2zq_e, 2zq_e1, zq_e, zq_e1), sB = (wq_e, wq_e1, x_e, x_e1),
  // sC = (y_e, y_e1, zb_e, zb_e1); (zq, wq) = normalised yaw quaternion of the PRE-reset pose,
  // zb = z_postreset - 0.5
  // (4-deep ring: the B group may run ahead of the scan group without an extra hand-shake)
  float4 sA[4][A1_TILE / 2];
  float4 sB[4][A1_TILE / 2];
  float4 sC[4][A1_TILE / 2];
  // double-buffered on the tile parity: warp 1 may start the next tile's terms while warp 0 still
  // accumulates this tile's
  float rterm[2][SHIFU_MAX_REWARD_TERMS][A1_TILE];
  uint64_t full_in[V3_STAGES], e_done[V3_STAGES], b_done[V3_STAGES], h_done[V3_STAGES];
};

constexpr uint32_t V3_ROW_BYTES = offsetof(V3In, ep_len);
constexpr uint32_t V3_HIST_BYTES = A1_TILE * A1_DOF * A1_HIST * 4;

// with_hist = false leaves the history rows out (their stage buffer is still being read by the
// bulk store of the pushed history); v3_issue_hist_load follows once that read has finished.
__device__ __forceinline__ void v3_issue_hist_load(V3In& in, const ShifuA1StepIO& io, long long e0, uint64_t* bar) {
  pipe::bulk_load(in.hist, io.history + e0 * (A1_DOF * A1_HIST), sizeof(in.hist), bar);
}

__device__ __forceinline__ void v3_issue_loads(V3In& in, const A1K& k, const ShifuA1StepIO& io, long long e0,
                                               uint64_t* bar, bool with_hist) {
  const uint32_t scalars = sizeof(in.ep_len) + sizeof(in.cla) + k.n_terms * sizeof(in.esum[0]);
  pipe::mbar_arrive_expect_tx(bar, V3_ROW_BYTES + scalars);
  pipe::bulk_load(in.root, io.root_state + e0 * 13, sizeof(in.root), bar);
  pipe::bulk_load(in.dof, io.dof_state + e0 * (A1_DOF * 2), sizeof(in.dof), bar);
  pipe::bulk_load(in.contact, io.contact_state + e0 * (A1_BODIES * 3), sizeof(in.contact), bar);
  if (with_hist) v3_issue_hist_load(in, io, e0, bar);
  pipe::bulk_load(in.tau, io.torques + e0 * A1_DOF, sizeof(in.tau), bar);
  pipe::bulk_load(in.act, io.actions + e0 * A1_DOF, sizeof(in.act), bar);
  pipe::bulk_load(in.ep_len, io.ep_len + e0, sizeof(in.ep_len), bar);
  pipe::bulk_load(in.cla[0], io.command + e0 * 3, sizeof(in.cla[0]), bar);
  pipe::bulk_load(in.cla[1], io.base_lin_vel + e0 * 3, sizeof(in.cla[1]), bar);
  pipe::bulk_load(in.cla[2], io.base_ang_vel + e0 * 3, sizeof(in.cla[2]), bar);
  for (int q = 0; q < k.n_terms; ++q) pipe::bulk_load(in.esum[q], io.ep_sums[q] + e0, sizeof(in.esum[q]), bar);
}

// With noise: the M head noise values of column d + 12m (m < M) of env gid, words 3(d>>1) .. of
// SHIFU_STREAM_OBS_NOISE; M = 6 for the 72-column head, 4 for the action head (words 3(d>>1) + 2 not drawn).
// The lanes of columns d and d^1 (lane ^ 1) share the words: each evaluates one of 3(d>>1), 3(d>>1)+1 and
// swaps halves with its neighbour; with M = 6 both evaluate 3(d>>1)+2.  hns: the M scales.
template <int M>
__device__ __forceinline__ void head_noise(const A1K& k, long long gid, long long step, int d, const float (&hns)[M],
                                           float (&hn)[M]) {
  static_assert(M == 6 || M == 4, "a 72- or 48-column head");
  const int c = d & 1;
  const U4 wa = obs_noise_word(k.seed, gid, step, 3 * (d >> 1) + c);
  const U4 wc = M == 6 ? obs_noise_word(k.seed, gid, step, 3 * (d >> 1) + 2) : U4{0u, 0u, 0u, 0u};
  const uint32_t r0 = __shfl_xor_sync(~0u, c ? wa.x : wa.y, 1), r1 = __shfl_xor_sync(~0u, c ? wa.z : wa.w, 1);
  const uint32_t o0 = c ? wa.y : wa.x, o1 = c ? wa.w : wa.z;
  const uint32_t x[6] = {c ? r0 : o0, c ? r1 : o1, c ? o0 : r0, c ? o1 : r1, c ? wc.y : wc.x, c ? wc.w : wc.z};
#pragma unroll
  for (int m = 0; m < M; ++m) hn[m] = mul_rn(u_pm1(x[m]), hns[m]);
}

// The B group (warps 0 .. V3_BG_WARPS-1, lane = env) of the pipelined kernels: the reward-term list
// (split over the three warps by a host-side cost balance; warp 2 does nothing else and runs ahead into
// the next tile's terms) + episode sums, termination, reset (curriculum, Philox draws, state rewrite and
// the carried body-frame velocities of the post-reset pose — warp 1, while warp 0 does the ordered
// accumulation and the flags), per-step log sums — the scalar game logic of ShifuVecEnv.post_step
// (env.py:93-106).  Reads only the stage (plus env origin / terrain level / type of the ~1 % of envs that
// reset); arrives on b_done when the tile's post-reset rows are final.
// SCAN (the sighted kernel): warp 0 first publishes the pre-reset yaw / xy of the tile's envs to the scan
// ring and arrives on e_done, warp 1 the post-reset base z.
template <bool HAS_EXTRA, bool SCAN, int STAGES, class Smem>
__device__ __forceinline__ void v3_b_group(const A1K& k, const ShifuA1StepIO& io, Smem& s, int my_tiles, int first,
                                           int stride, long long step, int t) {
  const int warp = t >> 5, lane = t & 31;

  for (int j = 0; j < my_tiles; ++j) {
    const int b = j % STAGES;
    const uint32_t par = (j / STAGES) & 1;
    const long long e0 = (long long)(first + j * stride) * A1_TILE;
    const long long ge = e0 + lane;
    auto& in = s.in[b];
    const int rb = j & 3;                                   // scalar ring stage (see V3Smem)
    pipe::mbar_wait<64>(&s.full_in[b], par);                // tile rows + per-env scalars have landed

    // ---- B1: yaw normalisation for the scan first (warp 0; the scan group starts its index
    //          arithmetic as soon as e_done completes), then the reward terms, split over the
    //          B warps by the host-side cost balance k.term_list
    if constexpr (SCAN) {
      if (warp == 0) {
        // heights are measured at the PRE-reset pose (isaac_gym.py:320-322 runs before post_step)
        publish_scan_env(make_scan_env(in.root[lane]), lane, s.sA[rb], s.sB[rb], s.sC[rb]);
        pipe::mbar_arrive(&s.e_done[b]);
      }
    }
#pragma unroll 1
    for (int i = 0; i < k.term_count[warp]; ++i) {
      const int q = k.term_list[warp][i];
      s.rterm[j & 1][q][lane] = a1_reward_term<HAS_EXTRA>(k.terms[q], q, k.rp[q][0], k.rp[q][1], k, in, lane, io, ge);
    }
    pipe::named_barrier(1, V3_B_THREADS);
    if (warp >= 2) continue;                                // a terms-only warp: on to the next tile's terms

    // ---- B2: both warps decide termination (a1_conditional.py:146-150); warp 0 does the ordered
    //          accumulation, flags and episode bookkeeping, warp 1 the state rewrite of resetting envs
    long long len = in.ep_len[lane] + 1;                                 // env.py:95
    const bool contact_term = force_exceeds(&in.contact[lane][k.base_body * 3], k.contact_thr_sq);
    const bool time_out = len > k.max_len;
    const bool reset = contact_term | time_out;
    double st_sum[SHIFU_MAX_REWARD_TERMS];
#pragma unroll
    for (int q = 0; q < SHIFU_MAX_REWARD_TERMS; ++q) st_sum[q] = 0.0;
    long long level_delta = 0;
    float esum[SHIFU_MAX_REWARD_TERMS];
    float cmd[3];
    if (warp == 0) {
#pragma unroll
      for (int q = 0; q < SHIFU_MAX_REWARD_TERMS; ++q) esum[q] = (q < k.n_terms) ? in.esum[q][lane] : 0.0f;
      float rew = 0.0f;                                                  // env.py:180-185
#pragma unroll
      for (int q = 0; q < SHIFU_MAX_REWARD_TERMS; ++q) {
        if (q < k.n_terms) {
          const float r = s.rterm[j & 1][q][lane];
          esum[q] = add_rn(esum[q], r);
          rew = add_rn(rew, r);
        }
      }
      io.rew_buf[ge] = rew;
      io.reset_buf[ge] = reset ? 1 : 0;
      io.time_out_buf[ge] = time_out ? 1 : 0;
      io.contact_term_buf[ge] = contact_term ? 1 : 0;
      if (reset)                                                         // env.py:101-102, bookkeeping part
        a1_reset_env<true, 2>(k, io, step, (int)ge, nullptr, nullptr, nullptr, cmd, esum, len, st_sum, level_delta,
                              0.0f, 0.0f, 0.0f, 0, 0);
      io.ep_len[ge] = len;
#pragma unroll
      for (int q = 0; q < SHIFU_MAX_REWARD_TERMS; ++q)
        if (q < k.n_terms) io.ep_sums[q][ge] = esum[q];
      a1_log_sums<2>(k, reset, st_sum, level_delta, lane);
    } else {
      if (reset) {                                                       // state part
        cmd[0] = in.cla[0][lane][0]; cmd[1] = in.cla[0][lane][1]; cmd[2] = in.cla[0][lane][2];
        a1_reset_env<true, 1, HAS_EXTRA>(k, io, step, (int)ge, in.root[lane], in.dof[lane], in.hist[lane], cmd, esum, len,
                              st_sum, level_delta, io.env_origins[ge * 3 + 0], io.env_origins[ge * 3 + 1],
                              io.env_origins[ge * 3 + 2], k.curriculum ? io.terrain_levels[ge] : 0,
                              k.curriculum ? io.terrain_types[ge] : 0);     // ~1 % of the envs: not worth a stage row
        in.cla[0][lane][0] = cmd[0]; in.cla[0][lane][1] = cmd[1]; in.cla[0][lane][2] = cmd[2];
      }
      if constexpr (SCAN)
        reinterpret_cast<float*>(&s.sC[rb][lane >> 1])[2 + (lane & 1)] =
            sub_rn(in.root[lane][2], k.h_off);                            // post-reset base z (D8)
      if (io.carry_body_frame) {
        // carried body-frame velocities for the next control step (robot.py:222-229, D7), from the
        // post-reset root row of this lane's env; the rows leave with the DMA lane's bulk stores
        const float* r = in.root[lane];
#pragma unroll
        for (int v = 0; v < 3; ++v) {
          float o[3];
          rotate_inverse(r + 3, v == 2 ? 0.0f : r[7 + 3 * v], v == 2 ? 0.0f : r[8 + 3 * v],
                         v == 2 ? -1.0f : r[9 + 3 * v], o);
          in.cout[v][lane][0] = o[0]; in.cout[v][lane][1] = o[1]; in.cout[v][lane][2] = o[2];
        }
        pipe::fence_proxy_async();                           // -> visible to the bulk stores
      }
      a1_log_sums<1>(k, reset, st_sum, level_delta, lane);
    }
    // post-reset rows / command / zb are final: hand the tile to the scan group
    pipe::mbar_arrive(&s.b_done[b]);
  }
}

// Processes tiles [0, num_tiles) of 32 envs each (the ragged tail, if any, is a separate launch of
// the barrier-phased kernel).  Requires root_stride == 1 and 16-byte aligned tensors.
// HAS_EXTRA: the term list holds a code >= SHIFU_REW_LIN_VEL_Z.  The reference's own six terms run the
// instantiation without that code (its presence alone cost the B group 5-10 % of the kernel).
// OBS: the observation follows the layout `o` (slot sources, column scales, height scale); without it
// `o` is not read and the reference observation is built.
// NOISE (only with OBS): uniform noise o.noise / o.h_noise is added before the clip to +-clip_obs, drawn
// on STREAM_OBS_NOISE with the word map of include/shifu_b200.h.
// HEAD (A1_HEAD_ACT only with OBS; a1_post_physics_tma_kernel_act): the action head.  A scan thread's head
// item writes 4 columns, the last the step's action in.act[e][d] (read before the stage is released); the
// heights follow at column 48 of a 235-column row.
#define A1_TMA_KERNEL a1_post_physics_tma_kernel
#define A1_TMA_HEAD A1_HEAD
#include "a1_fused_tma_kernel.inc"
#undef A1_TMA_KERNEL
#undef A1_TMA_HEAD

// The action head (num_obs = 235): instantiated with OBS = true only.
#define A1_TMA_KERNEL a1_post_physics_tma_kernel_act
#define A1_TMA_HEAD A1_HEAD_ACT
#include "a1_fused_tma_kernel.inc"
#undef A1_TMA_KERNEL
#undef A1_TMA_HEAD

// ===================================================================================================
// Blind form (72-column observation, no height scan): a streaming kernel.  Without the scan there is
// nothing to hide gathers under, so the CTA is small and an SM holds several: DMA warp (1 lane) + the
// B group above (3 warps, shared with the sighted kernel) + a head group of 3 warps (thread = (dof d,
// env group g): the 4 envs g, g+8, g+16, g+24 of the tile).  The head group builds the tile's 72-column
// observation in shared memory and pushes the history in place; the 288-B rows make the tile's
// observation one contiguous 9 216-B block, which the DMA lane bulk-stores with the history and the
// carried rows.  Every observation value is computed like the sighted kernel's head, so the blind obs
// equals columns 0-71 of the sighted obs bit for bit.
constexpr int VB_STAGES = 2;
constexpr int VB_CTAS_PER_SM = 3;
constexpr int VB_HEAD_WARPS = 3;
constexpr int VB_H_THREADS = 32 * VB_HEAD_WARPS;
constexpr int VB_HEAD_BASE = V3_B_THREADS;
constexpr int VB_DMA_BASE = V3_B_THREADS + VB_H_THREADS;
constexpr int VB_THREADS = VB_DMA_BASE + 32;
constexpr int VB_ENVS_PER_THREAD = A1_TILE * A1_DOF / VB_H_THREADS;      // 4
static_assert(VB_H_THREADS % A1_DOF == 0 && A1_TILE % (VB_H_THREADS / A1_DOF) == 0, "head group: (dof, env group) threads");

struct alignas(128) VBIn : V3In {     // the sighted stage + the tile's observation block
  float obs[A1_TILE][A1_HEAD];        //  9216 B
};
static_assert(sizeof(VBIn) == 31744 && sizeof(V3In) % 16 == 0, "blind tile layout: obs follows the stage, 16-B aligned");

struct alignas(128) VBSmem {
  VBIn in[VB_STAGES];
  float rterm[2][SHIFU_MAX_REWARD_TERMS][A1_TILE];
  uint64_t full_in[VB_STAGES], b_done[VB_STAGES], h_done[VB_STAGES];
};

// Processes tiles [0, num_tiles) like the sighted kernel (the ragged tail is the phased kernel's).
// HAS_EXTRA, OBS, NOISE and HEAD as above; EXACT_DIV and HAS_MROW do not apply.  Noise uses words 0-17
// (the action head: words 3i and 3i + 1).  With HEAD = A1_HEAD_ACT the tile's observation is a 32 x 48
// block (6 144 B) at the start of the stage's obs buffer (a1_post_physics_blind_kernel_act).
template <bool HAS_EXTRA, bool OBS, bool NOISE, int HEAD>
__device__ __forceinline__ void a1_post_physics_blind_body(const A1K& k, const ShifuA1StepIO& io, int num_tiles,
                                                           const A1Obs& o) {
  static_assert(HEAD == A1_HEAD || (OBS && HEAD == A1_HEAD_ACT), "the action head is an OBS layout");
  constexpr int NM = HEAD / 12;                               // head columns per (env, dof) item
  extern __shared__ __align__(128) unsigned char smem_raw[];
  VBSmem& s = *reinterpret_cast<VBSmem*>(smem_raw);
  const int t = threadIdx.x;
  const long long step = (io.step_dev != nullptr) ? *io.step_dev : io.step;
  const int first = blockIdx.x, stride = gridDim.x;
  const int my_tiles = (first < num_tiles) ? (num_tiles - first + stride - 1) / stride : 0;

  if (threadIdx.x == 0) {
#pragma unroll
    for (int b = 0; b < VB_STAGES; ++b) {
      pipe::mbar_init(&s.full_in[b], 1);
      pipe::mbar_init(&s.b_done[b], V3_B2_THREADS);
      pipe::mbar_init(&s.h_done[b], VB_H_THREADS);
    }
    pipe::fence_barrier_init();
  }
  __syncthreads();

  if (t >= VB_DMA_BASE) {
    // ---------------- DMA warp ----------------
    if (t != VB_DMA_BASE) return;
    for (int j = 0; j < VB_STAGES && j < my_tiles; ++j)
      v3_issue_loads(s.in[j], k, io, (long long)(first + j * stride) * A1_TILE, &s.full_in[j], true);
    for (int j = 0; j < my_tiles; ++j) {
      const int b = j % VB_STAGES;
      const uint32_t par = (j / VB_STAGES) & 1;
      const long long e0 = (long long)(first + j * stride) * A1_TILE;
      pipe::mbar_wait<64>(&s.h_done[b], par);
      pipe::bulk_store(io.obs_buf + e0 * HEAD, s.in[b].obs, A1_TILE * HEAD * 4);
      pipe::bulk_store(io.history + e0 * (A1_DOF * A1_HIST), s.in[b].hist, V3_HIST_BYTES);
      if (io.carry_body_frame) {                              // robot.py:222-229 for the next control step (D7)
        pipe::bulk_store(io.base_lin_vel + e0 * 3, s.in[b].cout[0], sizeof(s.in[b].cout[0]));
        pipe::bulk_store(io.base_ang_vel + e0 * 3, s.in[b].cout[1], sizeof(s.in[b].cout[1]));
        pipe::bulk_store(io.projected_gravity + e0 * 3, s.in[b].cout[2], sizeof(s.in[b].cout[2]));
      }
      pipe::bulk_commit();
      // the rows the stores do not read are dead: refill them while the stores still read hist / obs
      // (the head group writes this stage's obs again only after the hist load below has landed)
      const long long en = (long long)(first + (j + VB_STAGES) * stride) * A1_TILE;
      if (j + VB_STAGES < my_tiles) v3_issue_loads(s.in[b], k, io, en, &s.full_in[b], false);
      pipe::bulk_wait_read_all();
      if (j + VB_STAGES < my_tiles) v3_issue_hist_load(s.in[b], io, en, &s.full_in[b]);
    }
    pipe::bulk_wait_all();                                    // global writes done before exit
    return;
  }

  if (t < V3_B_THREADS) {
    v3_b_group<HAS_EXTRA, false, VB_STAGES>(k, io, s, my_tiles, first, stride, step, t);
    return;
  }

  // ---------------- head group: thread = (dof d, env group g) ----------------
  const int p = t - VB_HEAD_BASE;
  const int d = p % A1_DOF, g = p / A1_DOF;
  constexpr int NG = VB_H_THREADS / A1_DOF;                   // env groups: envs g + NG*r
  float hns[NM];                                              // this thread's noise scales (columns d + 12m)
  if (NOISE) {
#pragma unroll
    for (int m = 0; m < NM; ++m) hns[m] = o.noise[d + 12 * m];
  }
  const bool pg_slot = OBS && o.src[d / 3] == SHIFU_OBS_PROJECTED_GRAVITY;
  for (int j = 0; j < my_tiles; ++j) {
    const int b = j % VB_STAGES;
    const uint32_t par = (j / VB_STAGES) & 1;
    const long long e0 = (long long)(first + j * stride) * A1_TILE;
    // with OBS, a slot of projected_gravity reads its pre-step value from global memory: this tile's rows
    // are bulk-stored over only after this thread's h_done arrival
    float pgv[VB_ENVS_PER_THREAD];
#pragma unroll
    for (int r = 0; r < VB_ENVS_PER_THREAD; ++r)
      pgv[r] = pg_slot ? io.projected_gravity[(e0 + g + NG * r) * 3 + d % 3] : 0.0f;
    pipe::mbar_wait<32>(&s.b_done[b], par);
    VBIn& in = s.in[b];
    const float c = k.clip_obs;
#pragma unroll
    for (int r = 0; r < VB_ENVS_PER_THREAD; ++r) {
      // obs head (a1_conditional.py:131-144) + history push (train.py:12-14) of env e, from the post-reset rows
      const int e = g + NG * r;
      float hn[NM];
      if (NOISE) head_noise<NM>(k, k.env_offset + e0 + e, step, d, hns, hn);
      const float2 qd = *reinterpret_cast<const float2*>(&in.dof[e][2 * d]);
      const float a0 = in.hist[e][d * A1_HIST + 0], a1 = in.hist[e][d * A1_HIST + 1],
                  a2 = in.hist[e][d * A1_HIST + 2];
      const float v = OBS ? a1_obs_vec(o, d, in.cla, e, pgv[r])
                          : (d < 9) ? in.cla[d / 3][e][d % 3] : ((d == 11) ? -1.0f : 0.0f);
      in.hist[e][d * A1_HIST + 2] = a1;                       // HistoryRecorder.add (train.py:12-14)
      in.hist[e][d * A1_HIST + 1] = a0;
      in.hist[e][d * A1_HIST + 0] = in.act[e][d];
      auto sc = [&](float x, int m) {
        const float y = OBS ? mul_rn(x, o.scale[d + 12 * m]) : x;
        return NOISE ? add_rn(y, hn[m]) : y;
      };
      float* h = HEAD == A1_HEAD ? in.obs[e] : &in.obs[0][0] + e * HEAD;
      h[d] = clampf(sc(v, 0), -c, c);
      h[12 + d] = clampf(sc(sub_rn(qd.x, k.q0[d]), 1), -c, c);
      h[24 + d] = clampf(sc(qd.y, 2), -c, c);
      if constexpr (HEAD == A1_HEAD) {
        h[36 + d] = clampf(sc(a0, 3), -c, c);                // HistoryRecorder.flatten: slot-major
        h[48 + d] = clampf(sc(a1, 4), -c, c);
        h[60 + d] = clampf(sc(a2, 5), -c, c);
      } else {
        h[36 + d] = clampf(sc(in.act[e][d], 3), -c, c);      // legged_gym's self.actions
      }
    }
    pipe::fence_proxy_async();                                // obs block + pushed history -> the TMA stores
    pipe::mbar_arrive(&s.h_done[b]);
  }
}

template <bool HAS_EXTRA, bool OBS, bool NOISE>
__global__ void __launch_bounds__(VB_THREADS, VB_CTAS_PER_SM)
a1_post_physics_blind_kernel(const __grid_constant__ A1K k, const __grid_constant__ ShifuA1StepIO io, int num_tiles,
                             const __grid_constant__ A1Obs o) {
  a1_post_physics_blind_body<HAS_EXTRA, OBS, NOISE, A1_HEAD>(k, io, num_tiles, o);
}

// The 48-column action head (num_obs = 48): always an OBS layout.
template <bool HAS_EXTRA, bool NOISE>
__global__ void __launch_bounds__(VB_THREADS, VB_CTAS_PER_SM)
a1_post_physics_blind_kernel_act(const __grid_constant__ A1K k, const __grid_constant__ ShifuA1StepIO io,
                                 int num_tiles, const __grid_constant__ A1Obs o) {
  a1_post_physics_blind_body<HAS_EXTRA, true, NOISE, A1_HEAD_ACT>(k, io, num_tiles, o);
}

}  // namespace shifu
