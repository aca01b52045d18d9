// C-ABI entry points of libshifu_b200.so (see include/shifu_b200.h for the contract).
// Host side only validates arguments, fills the kernel constant blocks and enqueues launches
// on the caller's stream.  nvcc -gencode arch=compute_100a,code=sm_100a --fmad=false.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include <cstdarg>
#include <cmath>
#include <new>

#include "../../include/shifu_b200.h"
#include "a1_kernels.cuh"
#include "a1_fused.cuh"
#include "a1_fused_tma.cuh"
#include "scan_pairs.cuh"
#include "abb_kernels.cuh"
#include "arm_ik.cuh"
#include "camera_gather.cuh"
#include "common_kernels.cuh"
#include "terrain_gen.cuh"

using namespace shifu;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CUDA_TRY(expr)                                                                      \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) return fail((int)_e, "%s: %s", #expr, cudaGetErrorString(_e));  \
  } while (0)

#define REQUIRE_PTR(p)                                                      \
  do {                                                                      \
    if ((p) == nullptr) return fail(SHIFU_E_NULL, "%s is NULL", #p);        \
  } while (0)

#define REQUIRE_ALIGNED(p, a)                                                                    \
  do {                                                                                           \
    if ((reinterpret_cast<uintptr_t>(p) & ((a) - 1)) != 0)                                       \
      return fail(SHIFU_E_ALIGN, "%s must be %d-byte aligned", #p, (int)(a));                    \
  } while (0)

struct ShifuCtx {
  int device = 0;
  int sm_count = 0;
  bool is_a1 = false, is_abb = false;
  ShifuA1Desc a1{};
  ShifuAbbDesc abb{};
  A1K a1k{};
  A1Obs a1o{};                     // observation layout (identity for the reference observation)
  bool obs_custom = false;         // a1o differs from the reference: the OBS instantiations of the pipelined kernel
  AbbK abbk{};
  short* d_table = nullptr;
  double* d_stats = nullptr;         // SHIFU_NUM_STATS accumulators + [SHIFU_NUM_STATS] = level sum
  unsigned long long* d_chain = nullptr;
  unsigned* d_ticket = nullptr;      // [0] ticket, [1] retired CTAs
  int chain_len = 0;
  unsigned epoch = 0;
  int a1_grid = 0;
  int a1_occ = 0;
  int tma_occ = 0;
  bool use_tma = true;
  bool grid_symmetric = false;     // measured-point grid is point-symmetric (what the pipelined scan assumes)
  bool blind = false;              // num_obs = SHIFU_OBS_HEAD or SHIFU_OBS_HEAD_ACT: no height columns, no scan
  bool act_head = false;           // num_obs = 235 or 48: the action head (SHIFU_OBS_HEAD_ACT columns)
  int blind_occ = 0;
};

static inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// the pipelined kernel's instantiations, index = 8*(OBS + NOISE) + 4*EXACT_DIV + 2*HAS_MROW + HAS_EXTRA
// (NOISE only with OBS), then the action head's (always OBS): 24 + 8*NOISE + 4*EXACT_DIV + 2*HAS_MROW + HAS_EXTRA
constexpr int A1_TMA_VARIANTS = 40;
template <bool OBS, bool NOISE>
static void a1_tma_fill(const void** t) {
  t[0] = (const void*)a1_post_physics_tma_kernel<false, false, false, OBS, NOISE>;
  t[1] = (const void*)a1_post_physics_tma_kernel<false, false, true, OBS, NOISE>;
  t[2] = (const void*)a1_post_physics_tma_kernel<false, true, false, OBS, NOISE>;
  t[3] = (const void*)a1_post_physics_tma_kernel<false, true, true, OBS, NOISE>;
  t[4] = (const void*)a1_post_physics_tma_kernel<true, false, false, OBS, NOISE>;
  t[5] = (const void*)a1_post_physics_tma_kernel<true, false, true, OBS, NOISE>;
  t[6] = (const void*)a1_post_physics_tma_kernel<true, true, false, OBS, NOISE>;
  t[7] = (const void*)a1_post_physics_tma_kernel<true, true, true, OBS, NOISE>;
}
template <bool NOISE>
static void a1_tma_act_fill(const void** t) {
  t[0] = (const void*)a1_post_physics_tma_kernel_act<false, false, false, true, NOISE>;
  t[1] = (const void*)a1_post_physics_tma_kernel_act<false, false, true, true, NOISE>;
  t[2] = (const void*)a1_post_physics_tma_kernel_act<false, true, false, true, NOISE>;
  t[3] = (const void*)a1_post_physics_tma_kernel_act<false, true, true, true, NOISE>;
  t[4] = (const void*)a1_post_physics_tma_kernel_act<true, false, false, true, NOISE>;
  t[5] = (const void*)a1_post_physics_tma_kernel_act<true, false, true, true, NOISE>;
  t[6] = (const void*)a1_post_physics_tma_kernel_act<true, true, false, true, NOISE>;
  t[7] = (const void*)a1_post_physics_tma_kernel_act<true, true, true, true, NOISE>;
}
// the blind pipelined kernel's instantiations, index = 2*(OBS + NOISE) + HAS_EXTRA (NOISE only with OBS),
// then the 48-column action head's: 6 + 2*NOISE + HAS_EXTRA
constexpr int A1_BLIND_VARIANTS = 10;
static const void* const* a1_blind_variants() {
  static const void* const table[A1_BLIND_VARIANTS] = {
      (const void*)a1_post_physics_blind_kernel<false, false, false>, (const void*)a1_post_physics_blind_kernel<true, false, false>,
      (const void*)a1_post_physics_blind_kernel<false, true, false>, (const void*)a1_post_physics_blind_kernel<true, true, false>,
      (const void*)a1_post_physics_blind_kernel<false, true, true>, (const void*)a1_post_physics_blind_kernel<true, true, true>,
      (const void*)a1_post_physics_blind_kernel_act<false, false>, (const void*)a1_post_physics_blind_kernel_act<true, false>,
      (const void*)a1_post_physics_blind_kernel_act<false, true>, (const void*)a1_post_physics_blind_kernel_act<true, true>};
  return table;
}
static const void* const* a1_tma_variants() {
  static const void* table[A1_TMA_VARIANTS];
  static const bool filled = (a1_tma_fill<false, false>(table), a1_tma_fill<true, false>(table + 8),
                              a1_tma_fill<true, true>(table + 16), a1_tma_act_fill<false>(table + 24),
                              a1_tma_act_fill<true>(table + 32), true);
  (void)filled;
  return table;
}

extern "C" const char* shifu_last_error(void) { return g_err; }
extern "C" int shifu_abi_version(void) { return SHIFU_ABI_VERSION; }

// Largest float s with sqrtf(s) <= thr (sqrtf is correctly rounded and monotonic), so that
// "sqrt_rn(s) > thr" can be tested as "s > sqrt_threshold(thr)" with identical results.
static float sqrt_threshold(float thr) {
  if (!(thr >= 0.0f) || std::isinf(thr)) return thr;
  float s = thr * thr;
  while (s > 0.0f && std::sqrt(s) > thr) s = std::nextafter(s, 0.0f);
  while (std::sqrt(std::nextafter(s, INFINITY)) <= thr) s = std::nextafter(s, INFINITY);
  return s;
}

// Observation layout of the descriptor -> o (identity for layout 0); custom = it differs from the reference.
// The action head (num_obs = 235 or 48) reads obs_scale / obs_noise for j < SHIFU_OBS_HEAD_ACT only and is
// always custom: it is never the reference observation.
static int fill_a1obs(const ShifuA1Desc& d, A1Obs& o, bool& custom) {
  if (d.obs_layout != 0 && d.obs_layout != 1) return fail(SHIFU_E_RANGE, "obs_layout=%d must be 0 or 1", d.obs_layout);
  const bool act = d.num_obs == A1_HEAD_ACT + A1_POINTS || d.num_obs == A1_HEAD_ACT;
  const int head = act ? A1_HEAD_ACT : A1_HEAD;
  if (act && d.obs_layout != 1)
    return fail(SHIFU_E_RANGE, "num_obs = %d (the action head) needs obs_layout = 1: it is never the reference "
                "observation", d.num_obs);
  std::memset(&o, 0, sizeof(o));
  for (int i = 0; i < 4; ++i) o.src[i] = i;                // COMMAND, BASE_LIN_VEL, BASE_ANG_VEL, GRAVITY_VEC
  for (int j = 0; j < A1_HEAD; ++j) o.scale[j] = 1.0f;
  o.h_scale = 1.0f;
  o.h_bound = std::fmin(d.height_clip, d.clip_obs);
  custom = false;
  for (int j = 0; j <= head; ++j) {
    const float v = j < head ? d.obs_noise[j] : d.obs_height_noise;
    if (!std::isfinite(v))
      return j < head ? fail(SHIFU_E_RANGE, "obs_noise[%d]=%g is not finite", j, (double)v)
                      : fail(SHIFU_E_RANGE, "obs_height_noise=%g is not finite", (double)v);
    if (v != 0.0f && d.obs_layout == 0)
      return fail(SHIFU_E_RANGE, "observation noise needs obs_layout = 1 (obs_layout = 0 ignores the layout fields)");
  }
  if ((d.num_obs == A1_HEAD || d.num_obs == A1_HEAD_ACT) && d.obs_height_noise != 0.0f)
    return fail(SHIFU_E_RANGE, "obs_height_noise=%g with num_obs = %d: a blind observation has no height columns",
                (double)d.obs_height_noise, d.num_obs);
  if (d.obs_layout == 0) return SHIFU_OK;
  for (int i = 0; i < 4; ++i) {
    if (d.obs_vec_src[i] < 0 || d.obs_vec_src[i] >= SHIFU_OBS_VEC_COUNT)
      return fail(SHIFU_E_RANGE, "obs_vec_src[%d]=%d is not an enum ShifuObsVec value", i, d.obs_vec_src[i]);
    custom |= d.obs_vec_src[i] != i;
    o.src[i] = d.obs_vec_src[i];
    o.uses_pg |= d.obs_vec_src[i] == SHIFU_OBS_PROJECTED_GRAVITY;
  }
  custom |= act;
  for (int j = 0; j < head; ++j) {
    if (!std::isfinite(d.obs_scale[j])) return fail(SHIFU_E_RANGE, "obs_scale[%d]=%g is not finite", j, (double)d.obs_scale[j]);
    custom |= d.obs_scale[j] != 1.0f;
    o.scale[j] = d.obs_scale[j];
  }
  if (d.num_obs != A1_HEAD && d.num_obs != A1_HEAD_ACT) {  // a blind observation has no height columns
    if (!std::isfinite(d.obs_height_scale))
      return fail(SHIFU_E_RANGE, "obs_height_scale=%g is not finite", (double)d.obs_height_scale);
    custom |= d.obs_height_scale != 1.0f;
    o.h_scale = d.obs_height_scale;
    o.h_bound = std::fmin(d.height_clip * std::fabs(o.h_scale), d.clip_obs);
  }
  for (int j = 0; j < head; ++j) { o.noise[j] = d.obs_noise[j]; o.noisy |= d.obs_noise[j] != 0.0f; }
  o.h_noise = d.obs_height_noise;
  o.noisy |= d.obs_height_noise != 0.0f;
  custom |= o.noisy != 0;
  return SHIFU_OK;
}

static int fill_a1k(const ShifuA1Desc& d, A1K& k) {
  if (d.abi_version != SHIFU_ABI_VERSION) return fail(SHIFU_E_RANGE, "ShifuA1Desc.abi_version %d != %d", d.abi_version, SHIFU_ABI_VERSION);
  if (d.num_envs <= 0) return fail(SHIFU_E_RANGE, "num_envs must be > 0 (got %d)", d.num_envs);
  if (d.num_dof != A1_DOF || d.num_bodies != A1_BODIES || d.num_hist != A1_HIST ||
      (d.num_obs != A1_OBS && d.num_obs != A1_HEAD && d.num_obs != A1_HEAD_ACT + A1_POINTS && d.num_obs != A1_HEAD_ACT) ||
      d.num_points_x != A1_NX || d.num_points_y != A1_NY)
    return fail(SHIFU_E_RANGE,
                "this build is specialised for dof=%d bodies=%d hist=%d obs=%d or %d (%d or %d with the action head) "
                "grid=%dx%d (got %d %d %d %d %dx%d)",
                A1_DOF, A1_BODIES, A1_HIST, A1_OBS, A1_HEAD, A1_HEAD_ACT + A1_POINTS, A1_HEAD_ACT, A1_NX, A1_NY,
                d.num_dof, d.num_bodies, d.num_hist, d.num_obs, d.num_points_x, d.num_points_y);
  if (d.base_body < 0 || d.base_body >= A1_BODIES || d.force_body < 0 || d.force_body >= A1_BODIES)
    return fail(SHIFU_E_RANGE, "base_body/force_body out of range");
  if (d.num_leg_bodies < 0 || d.num_leg_bodies > SHIFU_MAX_LEG_BODIES) return fail(SHIFU_E_RANGE, "num_leg_bodies out of range");
  for (int i = 0; i < d.num_leg_bodies; ++i)
    if (d.leg_bodies[i] < 0 || d.leg_bodies[i] >= A1_BODIES) return fail(SHIFU_E_RANGE, "leg_bodies[%d] out of range", i);
  if (d.num_reward_terms < 0 || d.num_reward_terms > SHIFU_MAX_REWARD_TERMS) return fail(SHIFU_E_RANGE, "num_reward_terms out of range");
  for (int i = 0; i < d.num_reward_terms; ++i)
    if (d.reward_terms[i] < 0 || d.reward_terms[i] >= SHIFU_REW_COUNT ||
        d.reward_terms[i] == SHIFU_REW_ABB_REACHING || d.reward_terms[i] == SHIFU_REW_ABB_SUCCESS)
      return fail(SHIFU_E_RANGE, "reward_terms[%d]=%d is not an A1 term", i, d.reward_terms[i]);
  if (d.root_stride < 1 || d.root_offset < 0 || d.root_offset >= d.root_stride) return fail(SHIFU_E_RANGE, "root_stride/root_offset invalid");
  if (!(d.horizontal_scale > 0.f) || d.max_terrain_level < 1 || d.num_terrain_types < 1) return fail(SHIFU_E_RANGE, "terrain constants invalid");
  std::memset(&k, 0, sizeof(k));
  k.n = d.num_envs;
  k.env_offset = d.env_offset;
  k.seed = d.rng_seed;
  k.base_body = d.base_body;
  k.n_leg = d.num_leg_bodies;
  for (int i = 0; i < d.num_leg_bodies; ++i) k.leg[i] = d.leg_bodies[i];
  k.force_body = d.force_body;
  k.root_stride = d.root_stride;
  k.root_offset = d.root_offset;
  for (int i = 0; i < A1_DOF; ++i) { k.q0[i] = d.q0[i]; k.kp[i] = d.kp[i]; k.kd[i] = d.kd[i]; k.tau_max[i] = d.torque_limit[i]; }
  k.action_scale = d.action_scale; k.clip_actions = d.clip_actions; k.clip_obs = d.clip_obs;
  for (int i = 0; i < A1_NX; ++i) k.px[i] = d.points_x[i];
  for (int i = 0; i < A1_NY; ++i) k.py[i] = d.points_y[i];
  k.border = d.border_size;
  k.hdiv.d = d.horizontal_scale;
  k.hdiv.r = 1.0f / d.horizontal_scale;
  // The 3-op constant division is proven (exhaustively) for 0.1f only; anything else divides.
  k.exact_div = (d.horizontal_scale == 0.1f) ? 0 : 1;
  k.vscale = d.vertical_scale; k.h_off = d.height_offset; k.h_clip = d.height_clip;
  k.max_len = d.max_episode_length; k.max_len_s = d.max_episode_length_s; k.contact_thr = d.contact_term_force;
  for (int i = 0; i < 7; ++i) k.root0[i] = d.default_root[i];
  // torch_rand_float(lo, hi): (hi - lo) * u + lo with (hi - lo) formed in Python double arithmetic
  k.xy_span = (float)((double)d.reset_xy_range - (double)(-d.reset_xy_range)); k.xy_low = -d.reset_xy_range;
  k.force_span = (float)((double)d.push_force_max - (double)(-d.push_force_max)); k.force_low = -d.push_force_max;
  for (int i = 0; i < 3; ++i) { k.cmd_span[i] = (float)((double)d.cmd_high[i] - (double)d.cmd_low[i]); k.cmd_low[i] = d.cmd_low[i]; }
  k.neg_zero = -0.0f;
  k.curriculum = d.curriculum; k.max_level = d.max_terrain_level; k.n_types = d.num_terrain_types;
  k.up_dist = d.level_up_distance; k.down_factor = d.level_down_factor;
  k.n_terms = d.num_reward_terms;
  for (int i = 0; i < d.num_reward_terms; ++i) {
    k.terms[i] = d.reward_terms[i]; k.rp[i][0] = d.reward_params[i][0]; k.rp[i][1] = d.reward_params[i][1];
    int ex = 0;
    const float p1 = d.reward_params[i][1];
    const bool pow2 = (p1 > 0.0f) && (std::frexp(p1, &ex) == 0.5f) && ex > -100 && ex < 100;
    k.rp_pow2[i] = pow2 ? 1 : 0;
    k.rp_inv[i] = pow2 ? 1.0f / p1 : 0.0f;
    k.rp_thr_sq[i] = sqrt_threshold(p1);
  }
  k.contact_thr_sq = sqrt_threshold(d.contact_term_force);
  // constants of the dof-limit / feet-air-time terms
  for (int i = 0; i < A1_DOF; ++i) { k.dof_lo[i] = d.dof_pos_limit_low[i]; k.dof_hi[i] = d.dof_pos_limit_high[i]; }
  if (d.num_feet < 0 || d.num_feet > 4) return fail(SHIFU_E_RANGE, "num_feet=%d out of range", d.num_feet);
  k.n_feet = d.num_feet;
  for (int i = 0; i < 4; ++i) {
    if (i < d.num_feet && (d.feet_bodies[i] < 0 || d.feet_bodies[i] >= A1_BODIES))
      return fail(SHIFU_E_RANGE, "feet_bodies[%d]=%d out of range", i, d.feet_bodies[i]);
    k.feet[i] = d.feet_bodies[i];
  }
  k.feet_thr = d.feet_contact_force; k.air_cmd_min = d.air_time_cmd_min; k.air_dt = d.air_time_dt; k.air_reset = d.air_time_reset;
  static const int term_cost[SHIFU_REW_COUNT] = {30, 25, 12, 135, 70, 40, 20, 20, 8, 10, 10, 40, 60, 8, 70, 90};
  // longest-processing-time split of the term list over the B warps of the pipelined kernel.  Warp 0
  // starts loaded with the yaw normalisation it does first (~115 on the scale of term_cost, from the
  // phase timers); warps 0 and 1 also carry their B2 halves (~100 and ~160 with the carried
  // body-frame rows), which the terms-only warp 2 overlaps with the next tile's terms.  The preloads
  // were tuned on the B200 (profiles/README.md: a dozen other splits of the reference's six terms
  // are 0.5-8 % slower).
  int load[A1K_TERM_WARPS] = {215, 160, 0, 0}, order[SHIFU_MAX_REWARD_TERMS];
  for (int i = 0; i < k.n_terms; ++i) order[i] = i;
  auto cost_of = [&](int q) { const int c = k.terms[q]; return (c >= 0 && c < SHIFU_REW_COUNT) ? term_cost[c] : 40; };
  for (int i = 0; i < k.n_terms; ++i)
    for (int j = i + 1; j < k.n_terms; ++j)
      if (cost_of(order[j]) > cost_of(order[i])) { const int t = order[i]; order[i] = order[j]; order[j] = t; }
  for (int w = 0; w < A1K_TERM_WARPS; ++w) k.term_count[w] = 0;
  for (int i = 0; i < k.n_terms; ++i) {
    int w = 0;
    for (int v = 1; v < V3_BG_WARPS; ++v) if (load[v] < load[w]) w = v;
    k.term_list[w][k.term_count[w]++] = order[i];
    load[w] += cost_of(order[i]);
  }
  return SHIFU_OK;
}

static int fill_abbk(const ShifuAbbDesc& d, AbbK& k) {
  if (d.abi_version != SHIFU_ABI_VERSION) return fail(SHIFU_E_RANGE, "ShifuAbbDesc.abi_version %d != %d", d.abi_version, SHIFU_ABI_VERSION);
  if (d.num_envs <= 0) return fail(SHIFU_E_RANGE, "num_envs must be > 0 (got %d)", d.num_envs);
  if (d.num_actors < 1 || d.num_bodies < 1 || d.num_dof < 0 || d.num_dof > SHIFU_MAX_DOF) return fail(SHIFU_E_RANGE, "actor/body/dof counts invalid");
  const int acts[4] = {d.robot_actor, d.table_actor, d.cube_actor, d.goal_actor};
  for (int i = 0; i < 4; ++i) if (acts[i] < 0 || acts[i] >= d.num_actors) return fail(SHIFU_E_RANGE, "actor index %d out of range", i);
  if (d.ee_body < 0 || d.ee_body >= d.num_bodies) return fail(SHIFU_E_RANGE, "ee_body out of range");
  if (d.num_reward_terms < 0 || d.num_reward_terms > SHIFU_MAX_REWARD_TERMS) return fail(SHIFU_E_RANGE, "num_reward_terms out of range");
  for (int i = 0; i < d.num_reward_terms; ++i)
    if (d.reward_terms[i] != SHIFU_REW_ABB_REACHING && d.reward_terms[i] != SHIFU_REW_ABB_SUCCESS)
      return fail(SHIFU_E_RANGE, "reward_terms[%d]=%d is not an ABB term", i, d.reward_terms[i]);
  std::memset(&k, 0, sizeof(k));
  k.n = d.num_envs; k.env_offset = d.env_offset; k.seed = d.rng_seed;
  k.n_actors = d.num_actors; k.n_bodies = d.num_bodies; k.n_dof = d.num_dof; k.ee_body = d.ee_body;
  k.robot_actor = d.robot_actor; k.table_actor = d.table_actor; k.cube_actor = d.cube_actor; k.goal_actor = d.goal_actor;
  for (int i = 0; i < 2; ++i) { k.min_xy[i] = d.min_ee_pos[i]; k.max_xy[i] = d.max_ee_pos[i]; }
  for (int i = 0; i < d.num_dof; ++i) k.q0[i] = d.q0[i];
  for (int i = 0; i < 7; ++i) { k.robot_root[i] = d.robot_root[i]; k.table_root[i] = d.table_root[i]; }
  for (int i = 0; i < 3; ++i) { k.pos_low[i] = d.box_pos_low[i]; k.pos_high[i] = d.box_pos_high[i]; }
  k.goal_z = d.goal_z; k.success_dist = d.success_distance;
  k.max_len = d.max_episode_length; k.max_len_s = d.max_episode_length_s; k.clip_obs = d.clip_obs;
  k.n_terms = d.num_reward_terms;
  for (int i = 0; i < d.num_reward_terms; ++i) { k.terms[i] = d.reward_terms[i]; k.rp[i][0] = d.reward_params[i][0]; k.rp[i][1] = d.reward_params[i][1]; }
  return SHIFU_OK;
}

static int ctx_create_impl(int device, const ShifuA1Desc* a1, const ShifuAbbDesc* abb, int util_envs, ShifuCtx** out);

extern "C" int shifu_ctx_create(int device, const ShifuA1Desc* a1, const ShifuAbbDesc* abb, ShifuCtx** out) {
  REQUIRE_PTR(out);
  *out = nullptr;
  if ((a1 == nullptr) == (abb == nullptr)) return fail(SHIFU_E_NULL, "exactly one of a1 / abb must be given");
  return ctx_create_impl(device, a1, abb, 0, out);
}

extern "C" int shifu_ctx_create_util(int device, int32_t num_envs, ShifuCtx** out) {
  REQUIRE_PTR(out);
  *out = nullptr;
  if (num_envs <= 0) return fail(SHIFU_E_RANGE, "num_envs must be > 0 (got %d)", num_envs);
  return ctx_create_impl(device, nullptr, nullptr, num_envs, out);
}

static int ctx_create_impl(int device, const ShifuA1Desc* a1, const ShifuAbbDesc* abb, int util_envs, ShifuCtx** out) {
  // validate the descriptor before touching the device so argument errors surface without a GPU
  A1K a1k; AbbK abbk; A1Obs a1o; bool obs_custom = false;
  if (a1 != nullptr) {
    int rc = fill_a1k(*a1, a1k);
    if (rc == SHIFU_OK) rc = fill_a1obs(*a1, a1o, obs_custom);
    if (rc) return rc;
  }
  else if (abb != nullptr) { int rc = fill_abbk(*abb, abbk); if (rc) return rc; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
    cudaGetLastError();
    return fail(SHIFU_E_NODEVICE, "no CUDA device: libshifu_b200 has no CPU fallback");
  }
  if (device < 0 || device >= ndev) return fail(SHIFU_E_RANGE, "device %d out of range (%d devices)", device, ndev);
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(SHIFU_E_NODEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
  ShifuCtx* c = new (std::nothrow) ShifuCtx();
  if (c == nullptr) return fail(SHIFU_E_STATE, "out of host memory");
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  int n = 0;
  if (a1 != nullptr) {
    c->is_a1 = true; c->a1 = *a1; c->a1k = a1k; c->a1o = a1o; c->obs_custom = obs_custom; n = a1->num_envs;
    c->blind = a1->num_obs == A1_HEAD || a1->num_obs == A1_HEAD_ACT;
    c->act_head = a1->num_obs == A1_HEAD_ACT + A1_POINTS || a1->num_obs == A1_HEAD_ACT;
    c->grid_symmetric = true;
    for (int i = 0; i < A1_NX; ++i) c->grid_symmetric &= (a1k.px[i] == -a1k.px[A1_NX - 1 - i]);
    for (int i = 0; i < A1_NY; ++i) c->grid_symmetric &= (a1k.py[i] == -a1k.py[A1_NY - 1 - i]);
  }
  else if (abb != nullptr) { c->is_abb = true; c->abb = *abb; c->abbk = abbk; n = abb->num_envs; }
  else n = util_envs;
  cudaError_t e = cudaMalloc(&c->d_stats, sizeof(double) * (SHIFU_NUM_STATS + 1));
  if (e == cudaSuccess) e = cudaMemset(c->d_stats, 0, sizeof(double) * (SHIFU_NUM_STATS + 1));
  c->chain_len = (n + COMPACT_CHUNK - 1) / COMPACT_CHUNK + 1;
  if (e == cudaSuccess) e = cudaMalloc(&c->d_chain, sizeof(unsigned long long) * c->chain_len);
  if (e == cudaSuccess) e = cudaMemset(c->d_chain, 0, sizeof(unsigned long long) * c->chain_len);
  if (e == cudaSuccess) e = cudaMalloc(&c->d_ticket, sizeof(unsigned) * 2);
  if (e == cudaSuccess) e = cudaMemset(c->d_ticket, 0, sizeof(unsigned) * 2);
  if (e == cudaSuccess && c->is_a1) {
    // all four instantiations share resources; ask for the full shared-memory carve-out so the
    // resident-CTA count is bounded by registers/threads, not by the default L1/smem split
    const void* variants[12] = {
        (const void*)a1_post_physics_kernel<false, false, false>, (const void*)a1_post_physics_kernel<true, false, false>,
        (const void*)a1_post_physics_kernel<false, true, false>, (const void*)a1_post_physics_kernel<true, true, false>,
        (const void*)a1_post_physics_kernel<false, false, true>, (const void*)a1_post_physics_kernel<false, true, true>,
        (const void*)a1_post_physics_kernel_act<false, false, false>, (const void*)a1_post_physics_kernel_act<true, false, false>,
        (const void*)a1_post_physics_kernel_act<false, true, false>, (const void*)a1_post_physics_kernel_act<true, true, false>,
        (const void*)a1_post_physics_kernel_act<false, false, true>, (const void*)a1_post_physics_kernel_act<false, true, true>};
    for (int v = 0; v < 12 && e == cudaSuccess; ++v)
      e = cudaFuncSetAttribute(variants[v], cudaFuncAttributePreferredSharedMemoryCarveout, 75);
    int occ = 0;
    if (e == cudaSuccess)
      e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, a1_post_physics_kernel<false, false, false>, A1_THREADS, 0);
    const int tiles = (n + A1_TILE - 1) / A1_TILE;
    const int cap = c->sm_count * (occ > 0 ? occ : 1);
    c->a1_grid = tiles < cap ? tiles : cap;
    c->a1_occ = occ;
    // pipelined TMA variants: opt in to the large dynamic shared-memory footprint
    const void* const* tma_variants = a1_tma_variants();
    // Ask for just enough shared memory for V3_CTAS_PER_SM resident CTAs (+1 KB the runtime reserves
    // per CTA) and leave the rest of the 256 KB array to L1, which serves the scan-table gathers:
    // 164 KB / 92 KB L1 measured 1.7 % faster than the maximum carve-out (228 KB / 28 KB L1).
    int smem_sm = 0;
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, device);
    int carve = 100;
    if (e == cudaSuccess && smem_sm > 0) {
      const long long need = (long long)V3_CTAS_PER_SM * ((long long)sizeof(V3Smem) + 1024);
      carve = (int)((need * 100 + smem_sm - 1) / smem_sm);
      if (carve > 100) carve = 100;
    }
    for (int v = 0; v < A1_TMA_VARIANTS && e == cudaSuccess; ++v) {
      e = cudaFuncSetAttribute(tma_variants[v], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(V3Smem));
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(tma_variants[v], cudaFuncAttributePreferredSharedMemoryCarveout, carve);
    }
    int tocc = 0;
    if (e == cudaSuccess)
      e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&tocc, a1_post_physics_tma_kernel<false, false, false, false, false>, V3_THREADS,
                                                        sizeof(V3Smem));
    c->tma_occ = tocc;
    // blind pipelined variants: VB_CTAS_PER_SM CTAs of VBSmem each; no scan table, so L1 keeps the rest
    if (e == cudaSuccess && smem_sm > 0) {
      const long long need = (long long)VB_CTAS_PER_SM * ((long long)sizeof(VBSmem) + 1024);
      carve = (int)((need * 100 + smem_sm - 1) / smem_sm);
      if (carve > 100) carve = 100;
    }
    const void* const* blind_variants = a1_blind_variants();
    for (int v = 0; v < A1_BLIND_VARIANTS && e == cudaSuccess; ++v) {
      e = cudaFuncSetAttribute(blind_variants[v], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(VBSmem));
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(blind_variants[v], cudaFuncAttributePreferredSharedMemoryCarveout, carve);
    }
    int bocc = 0;
    if (e == cudaSuccess)
      e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bocc, a1_post_physics_blind_kernel<false, false, false>, VB_THREADS,
                                                        sizeof(VBSmem));
    c->blind_occ = bocc;
    const char* kern = getenv("SHIFU_A1_KERNEL");
    c->use_tma = !(kern != nullptr && strcmp(kern, "phased") == 0);
  }
  if (e != cudaSuccess) {
    int rc = fail((int)e, "shifu_ctx_create: %s", cudaGetErrorString(e));
    shifu_ctx_destroy(c);
    return rc;
  }
  c->a1k.stats = c->d_stats;
  c->abbk.stats = c->d_stats;
  CUDA_TRY(cudaDeviceSynchronize());
  *out = c;
  return SHIFU_OK;
}

extern "C" int shifu_ctx_destroy(ShifuCtx* c) {
  if (c == nullptr) return SHIFU_OK;
  cudaFree(c->d_table);
  cudaFree(c->d_stats);
  cudaFree(c->d_chain);
  cudaFree(c->d_ticket);
  delete c;
  return SHIFU_OK;
}

static inline int grid_for(long long work_items, int threads, int sm_count, int per_sm) {
  long long g = (work_items + threads - 1) / threads;
  const long long cap = (long long)sm_count * per_sm;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

extern "C" int shifu_set_height_map(ShifuCtx* c, const int16_t* hs, int32_t rows, int32_t cols, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(hs);
  if (!c->is_a1) return fail(SHIFU_E_STATE, "height map only applies to an A1 ctx");
  if (rows < 2 || cols < 2 || (long long)rows * cols > (1LL << 30)) return fail(SHIFU_E_RANGE, "map %dx%d out of range", rows, cols);
  const int trows = rows - 1, tcols = cols - 1;
  // banded layout T[px>>3][py][px&7]: the 8 rows of a band are interleaved per column, so a 128-B
  // line still holds an 8x8-cell patch of the map while the index needs 3 integer ops
  const int bands = (trows + 7) / 8, band_w = ((tcols + 7) / 8) * 8;
  const size_t elems = (size_t)bands * 8 * band_w;
  CUDA_TRY(cudaStreamSynchronize(S(stream)));
  if (c->d_table != nullptr) { cudaFree(c->d_table); c->d_table = nullptr; }
  CUDA_TRY(cudaMalloc(&c->d_table, elems * sizeof(short)));
  CUDA_TRY(cudaMemsetAsync(c->d_table, 0, elems * sizeof(short), S(stream)));
  build_scan_table_kernel<<<grid_for((long long)trows * tcols, 256, c->sm_count, 8), 256, 0, S(stream)>>>(
      hs, rows, cols, c->d_table, band_w);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaStreamSynchronize(S(stream)));
  c->a1k.table = c->d_table;
  c->a1k.trows = trows; c->a1k.tcols = tcols; c->a1k.band_w = band_w;
  return SHIFU_OK;
}

extern "C" int shifu_set_level_sum(ShifuCtx* c, const int64_t* levels, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(levels);
  if (!c->is_a1) return fail(SHIFU_E_STATE, "terrain levels only apply to an A1 ctx");
  CUDA_TRY(cudaMemsetAsync(c->d_stats + SHIFU_NUM_STATS, 0, sizeof(double), S(stream)));
  level_sum_kernel<<<grid_for(c->a1.num_envs, 256, c->sm_count, 2), 256, 0, S(stream)>>>(
      reinterpret_cast<const long long*>(levels), c->a1.num_envs, c->d_stats + SHIFU_NUM_STATS);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_pd_torque(ShifuCtx* c, const float* a_in, float* a_out, const float* dof, float* tau,
                               int32_t substep, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(a_in); REQUIRE_PTR(dof); REQUIRE_PTR(tau);
  if (!c->is_a1) return fail(SHIFU_E_STATE, "shifu_pd_torque needs an A1 ctx");
  if (substep < 0) return fail(SHIFU_E_RANGE, "shifu_pd_torque: substep must be >= 0 (got %d)", substep);
  REQUIRE_ALIGNED(dof, 16); REQUIRE_ALIGNED(a_in, 16); REQUIRE_ALIGNED(tau, 16);
  if (a_out != nullptr) REQUIRE_ALIGNED(a_out, 16);
  const long long quads = (long long)c->a1.num_envs * (A1_DOF / 4);
  // The four substeps and the fused kernel all stream the same dof_state / actions / torques
  // (~200 MB at 1 Mi envs, more than L2).  Odd substeps sweep downward, so each launch starts on
  // the rows the previous one touched last, and the last substep ends on env 0, where the fused
  // kernel's first tiles start.
  const int descending = substep & 1;
  pd_torque_kernel<<<grid_for(quads, 256, c->sm_count, 8), 256, 0, S(stream)>>>(
      c->a1k, reinterpret_cast<const float4*>(a_in), reinterpret_cast<float4*>(a_out),
      reinterpret_cast<const float4*>(dof), reinterpret_cast<float4*>(tau), descending);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_body_frame(ShifuCtx* c, const float* root, int32_t n, int32_t root_stride, int32_t root_offset,
                                float* lin, float* ang, float* pg, float* gvec, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(root); REQUIRE_PTR(lin); REQUIRE_PTR(ang); REQUIRE_PTR(pg);
  if (n <= 0 || root_stride < 1 || root_offset < 0 || root_offset >= root_stride)
    return fail(SHIFU_E_RANGE, "shifu_body_frame: n=%d stride=%d offset=%d invalid", n, root_stride, root_offset);
  body_frame_kernel<<<grid_for(n, 256, c->sm_count, 8), 256, 0, S(stream)>>>(n, root_stride, root_offset, root, lin,
                                                                            ang, pg, gvec);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_get_heights(ShifuCtx* c, const float* root, float* mh, int32_t* cell_idx, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(root); REQUIRE_PTR(mh);
  if (!c->is_a1) return fail(SHIFU_E_STATE, "shifu_get_heights needs an A1 ctx");
  if (c->d_table == nullptr) return fail(SHIFU_E_STATE, "call shifu_set_height_map first");
  const int tiles = (c->a1.num_envs + A1_TILE - 1) / A1_TILE;
  if (cell_idx == nullptr && !c->a1k.exact_div && c->grid_symmetric && c->use_tma) {
    const int cap4 = c->sm_count * 4;                   // packed, one rotation per point pair (scan_pairs.cuh)
    get_heights_pairs_kernel<<<tiles < cap4 ? tiles : cap4, SP_THREADS, 0, S(stream)>>>(c->a1k, root, mh);
    CUDA_TRY(cudaGetLastError());
    return SHIFU_OK;
  }
  const int cap = c->sm_count * 8;
  get_heights_kernel<<<tiles < cap ? tiles : cap, A1_THREADS, 0, S(stream)>>>(c->a1k, root, mh, cell_idx);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_a1_eval_terms(ShifuCtx* c, const ShifuA1StepIO* io, float* out, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(io); REQUIRE_PTR(out);
  if (!c->is_a1) return fail(SHIFU_E_STATE, "shifu_a1_eval_terms needs an A1 ctx");
  REQUIRE_PTR(io->root_state); REQUIRE_PTR(io->dof_state); REQUIRE_PTR(io->contact_state); REQUIRE_PTR(io->actions);
  REQUIRE_PTR(io->torques); REQUIRE_PTR(io->history); REQUIRE_PTR(io->command); REQUIRE_PTR(io->base_lin_vel);
  REQUIRE_PTR(io->base_ang_vel); REQUIRE_PTR(io->projected_gravity);
  const int tiles = (c->a1.num_envs + A1_TILE - 1) / A1_TILE;
  const int cap = c->sm_count * 8;
  a1_eval_terms_kernel<<<tiles < cap ? tiles : cap, A1_THREADS, 0, S(stream)>>>(c->a1k, *io, out);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_a1_post_physics(ShifuCtx* c, const ShifuA1StepIO* io, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(io);
  if (!c->is_a1) return fail(SHIFU_E_STATE, "shifu_a1_post_physics needs an A1 ctx");
  if (!c->blind && c->d_table == nullptr) return fail(SHIFU_E_STATE, "call shifu_set_height_map first");
  if (c->blind && io->measured_heights != nullptr)
    return fail(SHIFU_E_RANGE, "measured_heights must be NULL with num_obs = %d (no height scan)", c->a1.num_obs);
  REQUIRE_PTR(io->root_state); REQUIRE_PTR(io->dof_state); REQUIRE_PTR(io->contact_state);
  REQUIRE_PTR(io->actions); REQUIRE_PTR(io->torques); REQUIRE_PTR(io->history); REQUIRE_PTR(io->command);
  REQUIRE_PTR(io->ep_len); REQUIRE_PTR(io->base_lin_vel); REQUIRE_PTR(io->base_ang_vel);
  REQUIRE_PTR(io->projected_gravity); REQUIRE_PTR(io->env_origins); REQUIRE_PTR(io->terrain_levels);
  REQUIRE_PTR(io->terrain_types); REQUIRE_PTR(io->terrain_origins); REQUIRE_PTR(io->dof_targets);
  REQUIRE_PTR(io->rand_force); REQUIRE_PTR(io->obs_buf); REQUIRE_PTR(io->rew_buf); REQUIRE_PTR(io->reset_buf);
  REQUIRE_PTR(io->time_out_buf); REQUIRE_PTR(io->contact_term_buf);
  for (int j = 0; j < c->a1.num_reward_terms; ++j)
    if (io->ep_sums[j] == nullptr) return fail(SHIFU_E_NULL, "ep_sums[%d] is NULL", j);
  REQUIRE_ALIGNED(io->dof_state, 16);
  const bool exact = c->a1k.exact_div != 0;
  const int n = c->a1.num_envs;

  // Pipelined TMA kernel for the full 32-env tiles when the layout allows bulk copies
  // (contiguous root rows, 16-byte aligned tensors); the barrier-phased kernel takes the ragged
  // tail (< 32 envs) or everything when bulk copies are not possible.
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
  // the pipelined scan rotates once per point pair: it needs the point-symmetric grid (else: phased kernel)
  const bool can_tma = c->use_tma && (c->grid_symmetric || c->blind) && c->a1k.root_stride == 1 && c->a1k.root_offset == 0 && al16(io->root_state) &&
                       al16(io->dof_state) && al16(io->contact_state) && al16(io->history) && al16(io->torques) &&
                       al16(io->actions) && al16(io->obs_buf) && al16(io->ep_len) && al16(io->command) &&
                       al16(io->base_lin_vel) && al16(io->base_ang_vel) && al16(io->projected_gravity) &&
                       [&] { for (int q = 0; q < c->a1k.n_terms; ++q) if (!al16(io->ep_sums[q])) return false; return true; }();
  const int full_tiles = can_tma ? n / A1_TILE : 0;
  if (full_tiles > 0 && c->blind) {
    const int cap = c->sm_count * (c->blind_occ > 0 ? c->blind_occ : 1);
    const dim3 grid(full_tiles < cap ? full_tiles : cap), block(VB_THREADS);
    bool extra = false;
    for (int q = 0; q < c->a1k.n_terms; ++q) extra |= c->a1k.terms[q] >= SHIFU_REW_LIN_VEL_Z;
    int tiles_arg = full_tiles;
    void* args[4] = {(void*)&c->a1k, const_cast<ShifuA1StepIO*>(io), (void*)&tiles_arg, (void*)&c->a1o};
    const int variant = c->act_head ? 6 + (c->a1o.noisy ? 2 : 0) + (extra ? 1 : 0)
                                    : (c->obs_custom ? 2 : 0) + (c->a1o.noisy ? 2 : 0) + (extra ? 1 : 0);
    CUDA_TRY(cudaLaunchKernel(a1_blind_variants()[variant], grid, block, args, sizeof(VBSmem), S(stream)));
  } else if (full_tiles > 0) {
    const int cap = c->sm_count * (c->tma_occ > 0 ? c->tma_occ : 1);
    const dim3 grid(full_tiles < cap ? full_tiles : cap), block(V3_THREADS);
    const size_t smem = sizeof(V3Smem);
    const bool mrow = io->measured_heights != nullptr;
    bool extra = false;
    for (int q = 0; q < c->a1k.n_terms; ++q) extra |= c->a1k.terms[q] >= SHIFU_REW_LIN_VEL_Z;
    int tiles_arg = full_tiles;
    void* args[4] = {(void*)&c->a1k, const_cast<ShifuA1StepIO*>(io), (void*)&tiles_arg, (void*)&c->a1o};
    const int variant = (c->act_head ? 24 : c->obs_custom ? 8 : 0) + (c->a1o.noisy ? 8 : 0) + (exact ? 4 : 0) +
                        (mrow ? 2 : 0) + (extra ? 1 : 0);
    CUDA_TRY(cudaLaunchKernel(a1_tma_variants()[variant], grid, block, args, smem, S(stream)));
  }
  const int tiles = (n + A1_TILE - 1) / A1_TILE - full_tiles;    // the ragged tail, or every tile
  if (tiles > 0) {
    const int cap = c->sm_count * (c->a1_occ > 0 ? c->a1_occ : 1);
    const dim3 grid(tiles < cap ? tiles : cap), block(A1_THREADS);
    const A1K& k = c->a1k;
    const A1Obs& o = c->a1o;
    if (c->act_head) {
      if (c->blind) {
        if (o.noisy) a1_post_physics_kernel_act<false, true, true><<<grid, block, 0, S(stream)>>>(k, *io, o, full_tiles);
        else a1_post_physics_kernel_act<false, false, true><<<grid, block, 0, S(stream)>>>(k, *io, o, full_tiles);
      } else if (o.noisy) {
        if (exact) a1_post_physics_kernel_act<true, true, false><<<grid, block, 0, S(stream)>>>(k, *io, o, full_tiles);
        else a1_post_physics_kernel_act<false, true, false><<<grid, block, 0, S(stream)>>>(k, *io, o, full_tiles);
      } else {
        if (exact) a1_post_physics_kernel_act<true, false, false><<<grid, block, 0, S(stream)>>>(k, *io, o, full_tiles);
        else a1_post_physics_kernel_act<false, false, false><<<grid, block, 0, S(stream)>>>(k, *io, o, full_tiles);
      }
    } else if (c->blind) {
      if (o.noisy) a1_post_physics_kernel<false, true, true><<<grid, block, 0, S(stream)>>>(k, *io, o, full_tiles);
      else a1_post_physics_kernel<false, false, true><<<grid, block, 0, S(stream)>>>(k, *io, o, full_tiles);
    } else if (o.noisy) {
      if (exact) a1_post_physics_kernel<true, true, false><<<grid, block, 0, S(stream)>>>(k, *io, o, full_tiles);
      else a1_post_physics_kernel<false, true, false><<<grid, block, 0, S(stream)>>>(k, *io, o, full_tiles);
    } else {
      if (exact) a1_post_physics_kernel<true, false, false><<<grid, block, 0, S(stream)>>>(k, *io, o, full_tiles);
      else a1_post_physics_kernel<false, false, false><<<grid, block, 0, S(stream)>>>(k, *io, o, full_tiles);
    }
    CUDA_TRY(cudaGetLastError());
  }
  return SHIFU_OK;
}

extern "C" int shifu_abb_post_physics(ShifuCtx* c, const ShifuAbbStepIO* io, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(io);
  if (!c->is_abb) return fail(SHIFU_E_STATE, "shifu_abb_post_physics needs an ABB ctx");
  REQUIRE_PTR(io->root_state); REQUIRE_PTR(io->body_state); REQUIRE_PTR(io->dof_state); REQUIRE_PTR(io->dof_targets);
  REQUIRE_PTR(io->ep_len); REQUIRE_PTR(io->obs_buf); REQUIRE_PTR(io->rew_buf); REQUIRE_PTR(io->reset_buf);
  REQUIRE_PTR(io->time_out_buf); REQUIRE_PTR(io->success_buf);
  for (int j = 0; j < c->abb.num_reward_terms; ++j)
    if (io->ep_sums[j] == nullptr) return fail(SHIFU_E_NULL, "ep_sums[%d] is NULL", j);
  abb_post_physics_kernel<<<grid_for(c->abb.num_envs, 128, c->sm_count, 16), 128, 0, S(stream)>>>(c->abbk, *io);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_abb_reset_idx(ShifuCtx* c, const ShifuAbbStepIO* io, const int64_t* ids, int32_t n_ids, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(io);
  if (c->is_a1) return fail(SHIFU_E_STATE, "shifu_abb_reset_idx needs an ABB ctx");
  if (n_ids < 0 || n_ids > c->abb.num_envs) return fail(SHIFU_E_RANGE, "n_ids=%d out of range", n_ids);
  if (n_ids == 0) return SHIFU_OK;                    // shifu/gym/env.py:115-116
  REQUIRE_PTR(io->root_state); REQUIRE_PTR(io->dof_state); REQUIRE_PTR(io->dof_targets); REQUIRE_PTR(io->ep_len);
  REQUIRE_PTR(io->reset_buf); REQUIRE_PTR(io->success_buf);
  for (int j = 0; j < c->abb.num_reward_terms; ++j)
    if (io->ep_sums[j] == nullptr) return fail(SHIFU_E_NULL, "ep_sums[%d] is NULL", j);
  abb_reset_idx_kernel<<<grid_for(n_ids, 128, c->sm_count, 16), 128, 0, S(stream)>>>(
      c->abbk, *io, reinterpret_cast<const long long*>(ids), n_ids);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_compact_reset_ids(ShifuCtx* c, const uint8_t* flags, int32_t n, int64_t* ids, int32_t* n_out, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(flags); REQUIRE_PTR(ids); REQUIRE_PTR(n_out);
  if (n <= 0) return fail(SHIFU_E_RANGE, "n must be > 0 (got %d)", n);
  const int chunks = (n + COMPACT_CHUNK - 1) / COMPACT_CHUNK;
  if (chunks > c->chain_len) return fail(SHIFU_E_RANGE, "n=%d exceeds the ctx's num_envs", n);
  c->epoch += 1;
  compact_ids_kernel<<<chunks, COMPACT_THREADS, 0, S(stream)>>>(flags, n, reinterpret_cast<long long*>(ids), n_out,
                                                               c->d_chain, c->d_ticket, c->epoch);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_history_add(ShifuCtx* c, float* hist, const float* x, int32_t n, int32_t a, int32_t h, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(hist); REQUIRE_PTR(x);
  if (n <= 0 || a <= 0 || h <= 0) return fail(SHIFU_E_RANGE, "history shape (%d,%d,%d) invalid", n, a, h);
  const long long rows = (long long)n * a;
  history_add_kernel<<<grid_for(rows, 256, c->sm_count, 8), 256, 0, S(stream)>>>(hist, x, rows, h);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_arm_ik(ShifuCtx* c, const ShifuArmIkIO* io, int32_t n, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(io); REQUIRE_PTR(io->body_state); REQUIRE_PTR(io->jacobian); REQUIRE_PTR(io->dof_state);
  REQUIRE_PTR(io->dof_targets);
  if ((io->goal_pose == nullptr) == (io->actions == nullptr))
    return fail(SHIFU_E_RANGE, "shifu_arm_ik: exactly one of goal_pose / actions must be given");
  if (n <= 0) return fail(SHIFU_E_RANGE, "num_envs must be > 0");
  if (io->num_dof < 1 || io->num_dof > SHIFU_MAX_DOF) return fail(SHIFU_E_RANGE, "num_dof=%d out of range", io->num_dof);
  if (io->ee_body < 0 || io->ee_body >= io->num_bodies || io->ee_link < 0 || io->ee_link >= io->num_links)
    return fail(SHIFU_E_RANGE, "end-effector body/link index out of range");
  arm_ik_kernel<<<grid_for(n, 128, c->sm_count, 16), 128, 0, S(stream)>>>(*io, n);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_camera_gather(ShifuCtx* c, const ShifuCameraGatherIO* io, int32_t n, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(io);
  if (n <= 0 || io->height <= 0 || io->width <= 0) return fail(SHIFU_E_RANGE, "num_envs, height and width must be > 0");
  if ((io->color_src && !io->color_out) || (io->depth_src && !io->depth_out) || (io->seg_src && !io->seg_out) ||
      (io->flow_src && !io->flow_out))
    return fail(SHIFU_E_NULL, "shifu_camera_gather: an image type has a source table but no output buffer");
  if (!io->color_src && !io->depth_src && !io->seg_src && !io->flow_src) return SHIFU_OK;
  const long long px = (long long)io->height * io->width;
  // the per-env OUTPUT bases must stay 16-byte aligned for the vector path (px % 4, px % 8 for int16)
  if (px % 8 != 0) return fail(SHIFU_E_RANGE, "height*width=%lld must be a multiple of 8", px);
  int bx = (int)((px / 4 + 255) / 256);
  if (bx > 8) bx = 8;
  const dim3 grid(bx, n < 65535 ? n : 65535);
  camera_gather_kernel<<<grid, 256, 0, S(stream)>>>(*io, n);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_clip(ShifuCtx* c, const float* in, float* out, int64_t count, float lim, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(in); REQUIRE_PTR(out);
  if (count <= 0) return fail(SHIFU_E_RANGE, "count must be > 0");
  clip_kernel<<<grid_for((count + 3) / 4, 256, c->sm_count, 8), 256, 0, S(stream)>>>(in, out, count, lim);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_a1_reset_idx(ShifuCtx* c, const ShifuA1StepIO* io, const int64_t* ids, int32_t n_ids, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(io);
  if (!c->is_a1) return fail(SHIFU_E_STATE, "shifu_a1_reset_idx needs an A1 ctx");
  if (n_ids < 0 || n_ids > c->a1.num_envs) return fail(SHIFU_E_RANGE, "n_ids=%d out of range", n_ids);
  if (n_ids == 0) return SHIFU_OK;                    // shifu/gym/env.py:115-116
  REQUIRE_PTR(io->root_state); REQUIRE_PTR(io->dof_state); REQUIRE_PTR(io->history); REQUIRE_PTR(io->command);
  REQUIRE_PTR(io->ep_len); REQUIRE_PTR(io->env_origins); REQUIRE_PTR(io->terrain_levels);
  REQUIRE_PTR(io->terrain_types); REQUIRE_PTR(io->terrain_origins); REQUIRE_PTR(io->dof_targets);
  REQUIRE_PTR(io->rand_force); REQUIRE_PTR(io->reset_buf);
  for (int j = 0; j < c->a1.num_reward_terms; ++j)
    if (io->ep_sums[j] == nullptr) return fail(SHIFU_E_NULL, "ep_sums[%d] is NULL", j);
  a1_reset_idx_kernel<<<grid_for(n_ids, 128, c->sm_count, 16), 128, 0, S(stream)>>>(
      c->a1k, *io, reinterpret_cast<const long long*>(ids), n_ids);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_collect_stats(ShifuCtx* c, double* out, int64_t* step_dev, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(out);
  const double n = c->is_a1 ? c->a1.num_envs : c->abb.num_envs;
  collect_stats_kernel<<<1, 32, 0, S(stream)>>>(c->d_stats, c->d_stats + SHIFU_NUM_STATS, out, 1, 0, n,
                                                reinterpret_cast<long long*>(step_dev));
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_collect_stats_ring(ShifuCtx* c, double* ring, int32_t slots, int32_t slot, int64_t* step_dev, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(ring);
  if (slots < 1 || slot >= slots) return fail(SHIFU_E_RANGE, "slot %d outside the ring of %d", slot, slots);
  if (slot < 0 && step_dev == nullptr) return fail(SHIFU_E_NULL, "slot < 0 needs the device step counter");
  const double n = c->is_a1 ? c->a1.num_envs : c->abb.num_envs;
  collect_stats_kernel<<<1, 32, 0, S(stream)>>>(c->d_stats, c->d_stats + SHIFU_NUM_STATS, ring, slots, slot, n,
                                                reinterpret_cast<long long*>(step_dev));
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_publish_extras(ShifuCtx* c, const double* stats, float* extras, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(stats); REQUIRE_PTR(extras);
  const float ls = c->is_a1 ? c->a1.max_episode_length_s : c->abb.max_episode_length_s;
  const int nt = c->is_a1 ? c->a1.num_reward_terms : c->abb.num_reward_terms;
  publish_extras_kernel<<<1, 32, 0, S(stream)>>>(stats, extras, 1, 0, nullptr, ls, nt);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_publish_extras_ring(ShifuCtx* c, const double* stats, float* ring, int32_t slots, int32_t slot,
                                         const int64_t* step_dev, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(stats); REQUIRE_PTR(ring);
  if (slots < 1) return fail(SHIFU_E_RANGE, "slots must be >= 1 (got %d)", slots);
  if (slot >= slots) return fail(SHIFU_E_RANGE, "slot %d outside the ring of %d", slot, slots);
  if (slot < 0 && step_dev == nullptr) return fail(SHIFU_E_NULL, "slot < 0 needs the device step counter");
  const float ls = c->is_a1 ? c->a1.max_episode_length_s : c->abb.max_episode_length_s;
  const int nt = c->is_a1 ? c->a1.num_reward_terms : c->abb.num_reward_terms;
  publish_extras_kernel<<<1, 32, 0, S(stream)>>>(stats, ring, slots, slot, reinterpret_cast<const long long*>(step_dev),
                                                 ls, nt);
  CUDA_TRY(cudaGetLastError());
  return SHIFU_OK;
}

extern "C" int shifu_terrain_generate(ShifuCtx* c, const ShifuTerrainDesc* d, const ShifuTerrainTile* tiles, int32_t n_tiles,
                                      const double* table, int32_t n_table, int16_t* map, double* origins, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(d); REQUIRE_PTR(tiles); REQUIRE_PTR(map); REQUIRE_PTR(origins);
  if (n_tiles <= 0 || n_tiles > d->num_rows * d->num_cols) return fail(SHIFU_E_RANGE, "n_tiles=%d out of range", n_tiles);
  if (n_table < 0 || (n_table > 0 && table == nullptr)) return fail(SHIFU_E_NULL, "table is NULL");
  if (d->width_px <= 1 || d->length_px <= 1 || d->width_px != d->length_px)
    return fail(SHIFU_E_RANGE, "tiles must be square (terrain.py:100-104 builds SubTerrain(width, width))");
  const int tot_rows = d->num_rows * d->length_px + 2 * d->border_px, tot_cols = d->num_cols * d->width_px + 2 * d->border_px;
  ShifuTerrainTile* d_tiles = nullptr; double* d_table = nullptr;
  CUDA_TRY(cudaMalloc(&d_tiles, sizeof(ShifuTerrainTile) * n_tiles));
  cudaError_t e = cudaMalloc(&d_table, sizeof(double) * (n_table > 0 ? n_table : 1));
  if (e != cudaSuccess) { cudaFree(d_tiles); return fail((int)e, "cudaMalloc: %s", cudaGetErrorString(e)); }
  cudaMemcpyAsync(d_tiles, tiles, sizeof(ShifuTerrainTile) * n_tiles, cudaMemcpyHostToDevice, S(stream));
  if (n_table > 0) cudaMemcpyAsync(d_table, table, sizeof(double) * n_table, cudaMemcpyHostToDevice, S(stream));
  cudaMemsetAsync(map, 0, sizeof(int16_t) * (size_t)tot_rows * tot_cols, S(stream));
  const int px = d->width_px * d->length_px;
  terrain_raster_kernel<<<dim3(n_tiles, (px + 255) / 256 > 8 ? 8 : (px + 255) / 256), 256, 0, S(stream)>>>(
      d_tiles, d_table, d->width_px, d->length_px, d->border_px, tot_cols, map);
  const double hs = d->horizontal_scale;                       // window of terrain.py:166-169
  const int wx1 = (int)((d->env_length / 2. - 1) / hs), wx2 = (int)((d->env_length / 2. + 1) / hs);
  const int wy1 = (int)((d->env_width / 2. - 1) / hs), wy2 = (int)((d->env_width / 2. + 1) / hs);
  terrain_origins_kernel<<<n_tiles, 32, 0, S(stream)>>>(d_tiles, map, d->width_px, d->length_px, d->border_px, tot_cols,
                                                        d->num_cols, d->env_length, d->env_width, wx1, wx2, wy1, wy2,
                                                        d->vertical_scale, origins);
  e = cudaGetLastError();
  cudaStreamSynchronize(S(stream));                            // one-time init: the staging buffers go away here
  cudaFree(d_tiles); cudaFree(d_table);
  if (e != cudaSuccess) return fail((int)e, "terrain kernels: %s", cudaGetErrorString(e));
  return SHIFU_OK;
}

extern "C" int shifu_read_stats_host(ShifuCtx* c, double* host, void* stream) {
  REQUIRE_PTR(c); REQUIRE_PTR(host);
  CUDA_TRY(cudaMemcpyAsync(host, c->d_stats, sizeof(double) * SHIFU_NUM_STATS, cudaMemcpyDeviceToHost, S(stream)));
  CUDA_TRY(cudaStreamSynchronize(S(stream)));
  return SHIFU_OK;
}
