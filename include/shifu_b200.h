/*
 * shifu_b200 — C ABI of the B200-native post-physics hot path of 42jaylonw/shifu.
 *
 * The reference has no FFI: its "operator API" for this path is a set of Python methods on
 * ShifuVecEnv / Unit subclasses (SURVEY.md §8b).  Each entry point below replaces the torch
 * code of the cited reference lines (paths relative to the reference root) and is what a
 * maintainer binds with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C, no torch types; every pointer is a DEVICE pointer borrowed from the caller
 *     (tensor.data_ptr()) unless the name ends in _host; it must stay alive until `stream`
 *     reaches the call.  The library allocates nothing after shifu_ctx_create().
 *   - every call only ENQUEUES work on `stream` (a cudaStream_t passed as void*); no call
 *     synchronises except shifu_ctx_create / shifu_set_height_map / shifu_read_stats_host.
 *   - return value: 0 = OK, >0 = cudaError_t, <0 = SHIFU_E_* argument error.  No exceptions or
 *     aborts cross the ABI; shifu_last_error() returns a thread-local message.
 *   - a ctx is not re-entrant; distinct ctxs (one per GPU / process) are independent.
 *   - flat tensor layouts are Isaac Gym's (shifu/gym/isaac_gym.py:110-130):
 *       root_state (n_actors*N, 13) = pos3, quat xyzw 4, linvel 3, angvel 3
 *       dof_state  (dofs*N, 2)      = pos, vel
 *       contact    (bodies*N, 3)
 */
#ifndef SHIFU_B200_H
#define SHIFU_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SHIFU_ABI_VERSION 5

#define SHIFU_MAX_DOF 12
#define SHIFU_MAX_LEG_BODIES 8
#define SHIFU_MAX_POINTS_X 17
#define SHIFU_MAX_POINTS_Y 11
#define SHIFU_MAX_REWARD_TERMS 8
#define SHIFU_NUM_STATS 16
#define SHIFU_OBS_HEAD 72       /* observation columns before the 187 heights */
#define SHIFU_OBS_HEAD_ACT 48   /* the action head (num_obs = 235 or 48): columns 0-35 as in the 72-column head,
                                   then column 36 + d = the step's actions[d] (legged_gym's observation) */

/* Philox stream of the observation noise (ShifuA1Desc.obs_noise / obs_height_noise).  Counter
 * (global env id, step, SHIFU_STREAM_OBS_NOISE, word), key rng_seed, u = (x >> 8) * 2^-24 like every other
 * draw; step is the one the step's reset draws use.  65 words (0-64) cover the 259 columns:
 *   head, words 0-17: column d + 12m (d < 12, m < 6) is lane (d & 1) + 2 (m & 1) of word 3 (d >> 1) + (m >> 1),
 *     i.e. word 3i + r holds columns 2i + 24r, 2i + 1 + 24r, 2i + 24r + 12, 2i + 1 + 24r + 12 in x, y, z, w;
 *   heights, words 18-64: point pair k = (point k, point 186 - k), k = 0..93, is word 18 + (k >> 1): for even
 *     k, x = point k and y = point 186 - k; for odd k, z = point k and w = point 186 - k; the centre point 93
 *     uses z only.
 * The map follows the pipelined kernel's work split.  The two scan lanes of head columns d = 2i, 2i+1 each
 * evaluate one of words 3i, 3i+1 and swap halves; both evaluate word 3i+2 and each uses its half (a warp
 * issues that evaluation in the same slots whether one lane or two run it): 24 evaluations for the 18 head
 * words.  The two lanes of height point pairs k, k^1 each evaluate word 18 + (k >> 1) for one env of an env
 * pair and swap halves, so every lane of those evaluations is used; the two idle scan lanes evaluate word 64
 * for nothing.
 * A 72-column (blind, num_obs = SHIFU_OBS_HEAD) observation draws words 0-17 only, with the same map.
 * The action head (num_obs = 235 or 48, head width SHIFU_OBS_HEAD_ACT) keeps every position: head column
 * d + 12m (m < 4) uses the word and lane it has in the 72-column map (so the action column 36 + d uses the
 * word and lane of history column 36 + d), words 3i + 2 are not drawn, and height point k (column 48 + k)
 * uses word 18 + ... exactly as above.  The 235-column observation draws 12 + 47 = 59 words (0, 1, 3, 4, ...,
 * 15, 16 and 18-64), the 48-column one 12. */
#define SHIFU_STREAM_OBS_NOISE 8

enum {
  SHIFU_OK = 0,
  SHIFU_E_NULL = -1,       /* required pointer is NULL */
  SHIFU_E_RANGE = -2,      /* size / index out of the supported range */
  SHIFU_E_STATE = -3,      /* call order (e.g. height map not set) */
  SHIFU_E_NODEVICE = -4,   /* no CUDA device / not an sm_100 part */
  SHIFU_E_ALIGN = -5       /* pointer not aligned for vector access */
};

/* Reward-term registry: the compiled form of build_reward_functions()
 * (shifu/gym/env.py:78-80,160-166; examples/a1_conditional/a1_conditional.py:152-192;
 *  examples/abb_pushbox_vision/a_prior_stage.py:112-127).  Term order = accumulation order. */
enum ShifuRewardTerm {
  SHIFU_REW_TRACKING_LIN_VEL = 0, /* p0*exp(-|cmd_xy - v_xy|^2 / p1)            a1_conditional.py:162-164 */
  SHIFU_REW_TRACKING_ANG_VEL = 1, /* p0*exp(-(cmd_yaw - w_z)^2 / p1)            :166-168 */
  SHIFU_REW_STABILIZING_BASE = 2, /* p0*v_z^2 + p1*|w_xy|^2                     :170-174 */
  SHIFU_REW_SMOOTHING_ACTION = 3, /* p0*(|a1-a0|^2 + |a2-2a1+a0|^2)             :182-189 */
  SHIFU_REW_LEG_COLLISION = 4,    /* p0*#{leg bodies with |F| > p1}             :176-180 */
  SHIFU_REW_TORQUES = 5,          /* p0*|tau|^2                                 :191-192 */
  SHIFU_REW_ABB_REACHING = 6,     /* [|ee-cube|<p0] * exp(-|goal-cube|^2 / p1)  a_prior_stage.py:118-123 */
  SHIFU_REW_ABB_SUCCESS = 7,      /* p0*[|goal-cube| < p1]                      :125-131 */
  /* legged_gym-style terms for user task lists (SURVEY.md 8f row N1; shifu/gym/env.py:160-185 accepts any
   * list; the buffers of a1_conditional.py:100-103 / robot.py:215 hint at them) */
  SHIFU_REW_LIN_VEL_Z = 8,        /* p0*v_z^2                         torch.square(base_lin_vel[:, 2]) */
  SHIFU_REW_ANG_VEL_XY = 9,       /* p0*|w_xy|^2                      sum(square(base_ang_vel[:, :2])) */
  SHIFU_REW_ORIENTATION = 10,     /* p0*|g_xy|^2                      sum(square(projected_gravity[:, :2])), robot.py:215 */
  SHIFU_REW_DOF_VEL = 11,         /* p0*|qd|^2                        sum(square(dof_vel)) */
  SHIFU_REW_ACTION_RATE = 12,     /* p0*|a_{t-1} - a_t|^2             sum(square(actions_recorder.get_last(0) - actions)) */
  SHIFU_REW_BASE_HEIGHT = 13,     /* p0*(z - p1)^2                    square(base_pose[:, 2] - p1) */
  SHIFU_REW_DOF_POS_LIMITS = 14,  /* p0*sum(-(q - lo).clip(max=0) + (q - hi).clip(min=0))   lo/hi = dof_pos_limit_low/high */
  SHIFU_REW_FEET_AIR_TIME = 15,   /* p0*sum((air_time + dt - p1) * first_contact) * [|cmd_xy| > air_time_cmd_min];
                                     STATEFUL: swing_time / last_contacts (a1_conditional.py:99-102) are
                                     updated exactly like legged_gym's _reward_feet_air_time */
  SHIFU_REW_COUNT = 16
};

/* Source of one 3-column vector slot of the A1 observation (columns 3i..3i+2, i < 4) when
 * ShifuA1Desc.obs_layout == 1.  The reference observation is COMMAND, BASE_LIN_VEL, BASE_ANG_VEL,
 * GRAVITY_VEC (a1_conditional.py:131-144). */
enum ShifuObsVec {
  SHIFU_OBS_COMMAND = 0,            /* command_buf */
  SHIFU_OBS_BASE_LIN_VEL = 1,       /* base_lin_vel (the carried S_prev value, D7) */
  SHIFU_OBS_BASE_ANG_VEL = 2,       /* base_ang_vel */
  SHIFU_OBS_GRAVITY_VEC = 3,        /* the constant (0, 0, -1) */
  SHIFU_OBS_PROJECTED_GRAVITY = 4,  /* projected_gravity as it is when the step starts (robot.py:222-229 on S_prev) */
  SHIFU_OBS_VEC_COUNT = 5
};

/* Index of each statistic in the stats vector (double[SHIFU_NUM_STATS]) that
 * shifu_*_post_physics accumulates and shifu_finalize_step publishes.  This vector is the
 * payload of the multi-GPU all-reduce (SURVEY.md §8e). */
enum {
  SHIFU_STAT_TERM0 = 0,        /* [0..7]  sum over resetting envs of episode_rewards[term k] (shifu/gym/env.py:149-153) */
  SHIFU_STAT_NRESET = 8,       /* number of resetting envs */
  SHIFU_STAT_LEVEL_SUM = 9,    /* sum over ALL envs of terrain_levels (a1_conditional.py:126-129) */
  SHIFU_STAT_SUCCESS = 10,     /* sum over resetting envs of success_buf (a_prior_stage.py:92-93) */
  SHIFU_STAT_NENVS = 11        /* number of envs contributing (so the reduced vector carries N_global) */
};

typedef struct ShifuCtx ShifuCtx;

/* ------------------------------------------------------------------------------------------
 * A1 conditional walking task constants.  Replaces the attribute reads scattered over
 * A1Conditional.__init__/A1Robot.__init__ (examples/a1_conditional/a1_conditional.py:22-114),
 * examples/a1_conditional/task_config.py and shifu/configs/env_config.py:77-102.
 * ------------------------------------------------------------------------------------------ */
typedef struct ShifuA1Desc {
  int32_t abi_version;          /* SHIFU_ABI_VERSION */
  int32_t num_envs;             /* local N (this GPU) */
  int64_t env_offset;           /* global id of local env 0: Philox counters, SURVEY.md §8e */
  uint64_t rng_seed;            /* Philox key (lo, hi) */
  int32_t num_dof;              /* 12 */
  int32_t num_bodies;           /* 17: contact rows per env */
  int32_t num_hist;             /* 3  (cfg.num_actions_history) */
  int32_t num_obs;              /* 259, or SHIFU_OBS_HEAD (72) for a blind task: obs_buf is (N,72), the
                                   measured heights are neither scanned nor written (measured_heights must be
                                   NULL), obs_height_scale is not read, obs_height_noise must be 0, and
                                   shifu_a1_post_physics needs no shifu_set_height_map.
                                   235 (SHIFU_OBS_HEAD_ACT + 187) or 48: the action head (legged_gym's
                                   observation), which needs obs_layout = 1; obs_scale[j] and obs_noise[j]
                                   are read for j < 48 only, column 36 + d is clip(actions[d] * obs_scale[36 + d]
                                   [+ noise], +-clip_obs), and the heights follow at column 48.  48 is blind
                                   like 72.  Anything else: SHIFU_E_RANGE */
  int32_t base_body;            /* contact_terminate_indices, a1_conditional.py:98-99 */
  int32_t num_leg_bodies;       /* 8 */
  int32_t leg_bodies[SHIFU_MAX_LEG_BODIES]; /* a1_conditional.py:59-61 */
  int32_t force_body;           /* rigid_body_dict['base'], a1_conditional.py:85 */
  int32_t root_stride;          /* actors per env (root row of env e = root_offset + e*root_stride) */
  int32_t root_offset;
  float q0[SHIFU_MAX_DOF];      /* default_dof_pos, task_config.py:17-20 */
  float kp[SHIFU_MAX_DOF];      /* task_config.py:22 */
  float kd[SHIFU_MAX_DOF];      /* task_config.py:23 */
  float torque_limit[SHIFU_MAX_DOF]; /* a1.urdf:95,137,165 via shifu/units/robot.py:42 */
  float action_scale;           /* 0.5, a1_conditional.py:123 */
  float clip_actions;           /* 1.0, shifu/gym/env.py:87 */
  float clip_obs;               /* 100, shifu/gym/env.py:90 */
  int32_t num_points_x;         /* 17 */
  int32_t num_points_y;         /* 11 */
  float points_x[SHIFU_MAX_POINTS_X]; /* env_config.py:87-88 */
  float points_y[SHIFU_MAX_POINTS_Y]; /* env_config.py:89 */
  float border_size;            /* 25, env_config.py:80 */
  float horizontal_scale;       /* 0.1 */
  float vertical_scale;         /* 0.005 */
  float height_offset;          /* 0.5, a1_conditional.py:132 */
  float height_clip;            /* 1.0, a1_conditional.py:133 */
  int64_t max_episode_length;   /* 500 = ceil(10/0.02), env.py:42; reset when ep_len > this */
  float max_episode_length_s;   /* 10 */
  float contact_term_force;     /* 1.0, a1_conditional.py:148 */
  float default_root[7];        /* default_pos + default_quat, task_config.py:15-16 */
  float reset_xy_range;         /* 1.0, a1_conditional.py:47 */
  float push_force_max;         /* 5.0, a1_conditional.py:83 */
  float cmd_low[3];             /* a1_conditional.py:110-112 */
  float cmd_high[3];
  int32_t curriculum;           /* cfg.terrain.curriculum */
  int32_t max_terrain_level;    /* 10 = cfg.terrain.num_rows, isaac_gym.py:345 */
  int32_t num_terrain_types;    /* 20 = cfg.terrain.num_cols */
  float level_up_distance;      /* env_length/2 = 4, a1_conditional.py:210 */
  float level_down_factor;      /* 0.5, a1_conditional.py:212-213 (x max_episode_length_s x |cmd|) */
  int32_t num_reward_terms;
  int32_t reward_terms[SHIFU_MAX_REWARD_TERMS];     /* enum ShifuRewardTerm, list order */
  float reward_params[SHIFU_MAX_REWARD_TERMS][2];   /* (p0, p1) per listed term */
  /* constants of the row-N1 terms that need more than (p0, p1) */
  float dof_pos_limit_low[SHIFU_MAX_DOF];           /* robot.dof_lower_limits (robot.py:35-45) */
  float dof_pos_limit_high[SHIFU_MAX_DOF];
  int32_t num_feet;                                 /* <= 4 */
  int32_t feet_bodies[4];                           /* robot.ee_indices (end_effector_names, task_config.py:21) */
  float feet_contact_force;                         /* a foot touches when F_z > this (1.0) */
  float air_time_cmd_min;                           /* term is 0 unless |cmd_xy| > this (0.1) */
  float air_time_dt;                                /* control dt added to swing_time every step (isaac_gym.py:26) */
  int32_t air_time_reset;                           /* !=0: reset_idx zeroes swing_time / last_contacts of the env */
  /* observation layout (legged_gym's obs_scales / commands_scale, projected gravity, slot order) */
  int32_t obs_layout;                               /* 0: the reference observation (a1_conditional.py:131-144); the
                                                       fields below are ignored.  1: as below */
  int32_t obs_vec_src[4];                           /* enum ShifuObsVec, source of columns 3i..3i+2 */
  float obs_scale[SHIFU_OBS_HEAD];                  /* obs[j] = clip(x_j * obs_scale[j], +-clip_obs), j < 72;
                                                       x_j of the dof-position columns is dof_pos - q0 */
  float obs_height_scale;                           /* heights = clip(clip(z - height_offset - h, +-height_clip) * this,
                                                       +-clip_obs) */
  /* uniform observation noise (legged_gym's noise_scale_vec), added before the clip to +-clip_obs:
   * obs[j] = clip(x_j * obs_scale[j] + (2u_j - 1) * obs_noise[j], +-clip_obs), heights likewise with
   * obs_height_noise, u_j drawn on SHIFU_STREAM_OBS_NOISE.  All zero: no noise.  Needs obs_layout = 1. */
  float obs_noise[SHIFU_OBS_HEAD];
  float obs_height_noise;
} ShifuA1Desc;

/* Tensors of one A1 step.  "rw" = read and written in place. */
typedef struct ShifuA1StepIO {
  float* root_state;              /* rw (n_actors*N,13): S_new; reset rows rewritten (isaac_gym.py:54-73) */
  float* dof_state;               /* rw (N*12,2) */
  const float* contact_state;     /* (N*17,3) */
  const float* actions;           /* (N,12) env.actions = clip(0.5*a, +-1)  (env.py:87) */
  const float* torques;           /* (N,12) last PD substep (a1_conditional.py:66-67) */
  float* history;                 /* rw (N,12,3) HistoryRecorder.history_buf (shifu/utils/train.py) */
  float* command;                 /* rw (N,3) */
  int64_t* ep_len;                /* rw (N) episode_length_buf; incremented here (env.py:95) */
  float* ep_sums[SHIFU_MAX_REWARD_TERMS]; /* rw (N) each, in reward_terms order (env.py:162-166) */
  float* base_lin_vel;            /* rw (N,3) carried body-frame velocity (D7) */
  float* base_ang_vel;            /* rw (N,3) */
  float* projected_gravity;       /* rw (N,3) */
  float* env_origins;             /* rw (N,3) */
  int64_t* terrain_levels;        /* rw (N) */
  const int64_t* terrain_types;   /* (N) */
  const float* terrain_origins;   /* (levels, types, 3) */
  float* dof_targets;             /* w on reset (N,12) (robot.py:75) */
  float* rand_force;              /* w on reset (N,17,3) (a1_conditional.py:82-87) */
  float* obs_buf;                 /* w (N,num_obs) already clipped to +-clip_obs */
  float* rew_buf;                 /* w (N) */
  uint8_t* reset_buf;             /* w (N) bool */
  uint8_t* time_out_buf;          /* w (N) bool */
  uint8_t* contact_term_buf;      /* w (N) bool */
  float* measured_heights;        /* optional w (N,187), may be NULL; must be NULL when num_obs = 72 or 48 */
  int64_t step;                   /* common_step_counter AFTER its increment (env.py:96): Philox counter */
  const int64_t* step_dev;        /* optional: when non-NULL the step is read from this device word
                                     instead (lets a captured CUDA graph replay with a moving
                                     counter; shifu_collect_stats can advance it) */
  float* swing_time;              /* rw (N, num_feet), only read when SHIFU_REW_FEET_AIR_TIME is listed (may be NULL otherwise) */
  uint8_t* last_contacts;         /* rw (N, num_feet) bool, same */
  int32_t carry_body_frame;      /* !=0: also write next step's base_lin/ang_vel, projected_gravity
                                     from the post-reset root row (== LeggedRobot.post_step of the
                                     next control step, robot.py:222-229, as long as nobody else
                                     writes root_state in between) */
} ShifuA1StepIO;

/* ------------------------------------------------------------------------------------------
 * ABB push-box prior stage (examples/abb_pushbox_vision/a_prior_stage.py, task_config.py:49-91)
 * ------------------------------------------------------------------------------------------ */
typedef struct ShifuAbbDesc {
  int32_t abi_version;
  int32_t num_envs;
  int64_t env_offset;
  uint64_t rng_seed;
  int32_t num_actors;           /* 4: robot, table, cube, goal */
  int32_t num_bodies;           /* 10 per env */
  int32_t num_dof;              /* 6 */
  int32_t ee_body;              /* 6 (tip0), robot.py:119-120 */
  int32_t robot_actor, table_actor, cube_actor, goal_actor; /* 0,1,2,3 */
  float min_ee_pos[3];          /* task_config.py:63 */
  float max_ee_pos[3];          /* task_config.py:64 */
  float q0[SHIFU_MAX_DOF];      /* task_config.py:56 */
  float robot_root[7];          /* task_config.py:54-55 */
  float table_root[7];          /* task_config.py:15-16 */
  double box_pos_low[3];        /* a_prior_stage.py:30-33 (float64: numpy draws) */
  double box_pos_high[3];
  double goal_z;                /* task_config.py:38 via GoalBox, a_prior_stage.py:57-58 */
  float success_distance;       /* 0.02, a_prior_stage.py:129-131 */
  int64_t max_episode_length;   /* 200 */
  float max_episode_length_s;   /* 20 */
  float clip_obs;               /* 10 */
  int32_t num_reward_terms;
  int32_t reward_terms[SHIFU_MAX_REWARD_TERMS];
  float reward_params[SHIFU_MAX_REWARD_TERMS][2];
} ShifuAbbDesc;

typedef struct ShifuAbbStepIO {
  float* root_state;            /* rw (4N,13) */
  const float* body_state;      /* (10N,13) */
  float* dof_state;             /* rw (6N,2) */
  float* dof_targets;           /* w on reset (N,6) */
  int64_t* ep_len;              /* rw */
  float* ep_sums[SHIFU_MAX_REWARD_TERMS];
  float* obs_buf;               /* w (N,6) clipped */
  float* rew_buf;
  uint8_t* reset_buf;
  uint8_t* time_out_buf;
  uint8_t* success_buf;
  int64_t step;
  const int64_t* step_dev;      /* optional device-resident step counter, see ShifuA1StepIO */
} ShifuAbbStepIO;

/* ---- context ------------------------------------------------------------------------------ */

/* Replaces the buffer/constant set-up of ShifuVecEnv.__init__ (shifu/gym/env.py:19-63).
 * Exactly one of a1 / abb may be non-NULL per ctx.  `device` is the CUDA ordinal. */
int shifu_ctx_create(int device, const ShifuA1Desc* a1, const ShifuAbbDesc* abb, ShifuCtx** out);
/* Task-less context for envs whose hooks stay user-written torch code: only the generic rows
 * (shifu_compact_reset_ids, shifu_history_add, shifu_clip) may be called on it. */
int shifu_ctx_create_util(int device, int32_t num_envs, ShifuCtx** out);
int shifu_ctx_destroy(ShifuCtx* ctx);
const char* shifu_last_error(void);
int shifu_abi_version(void);

/* Upload the static int16 height map (TerrainGymEnv.height_samples, isaac_gym.py:384-385) and
 * build the scan table from it: T[px][py] = min(H[px][py], H[px+1][py], H[px][py+1]) — the three
 * gathers + two mins of isaac_gym.py:427-431 folded into one table, stored in 8x8-cell tiles so a
 * rotated 17x11 footprint touches ~10 cache lines.  Call again if the map is edited. */
int shifu_set_height_map(ShifuCtx* ctx, const int16_t* height_samples, int32_t rows, int32_t cols, void* stream);

/* Seed the persistent all-env terrain-level sum (SHIFU_STAT_LEVEL_SUM) from the current levels. */
int shifu_set_level_sum(ShifuCtx* ctx, const int64_t* terrain_levels, void* stream);

/* ---- row a1/a2: action clip + PD torque substep --------------------------------------------
 * a1_conditional.py:66-67 (+ :123 and env.py:87 when actions_out != NULL: actions_out =
 * clip(action_scale*actions_in, +-clip_actions) is written and used; otherwise actions_in is used
 * as is).  Called once per decimation substep; PhysX runs between calls.  substep is the 0-based
 * decimation substep (negative: SHIFU_E_RANGE).  It changes no result: the library uses it only
 * to choose the order in which the envs are swept, so that consecutive substeps reuse what the
 * previous one left in L2. */
int shifu_pd_torque(ShifuCtx* ctx, const float* actions_in, float* actions_out, const float* dof_state,
                    float* torques, int32_t substep, void* stream);

/* ---- row a3: LeggedRobot.post_step (shifu/units/robot.py:222-229) -------------------------- */
/* Root row of env e = root_state[(root_offset + e*root_stride)*13 ..]; works on any ctx. */
int shifu_body_frame(ShifuCtx* ctx, const float* root_state, int32_t num_envs, int32_t root_stride,
                     int32_t root_offset, float* base_lin_vel, float* base_ang_vel,
                     float* projected_gravity, float* gravity_vec, void* stream);

/* ---- row a5: TerrainGymEnv.get_heights (shifu/gym/isaac_gym.py:393-433) --------------------
 * cell_idx (optional, (N*P,2) int32 = clipped px,py) exposes the integer cell indices for the
 * bit-exactness tests. */
int shifu_get_heights(ShifuCtx* ctx, const float* root_state, float* measured_heights, int32_t* cell_idx,
                      void* stream);

/* ---- rows a5-a7, a9-a14: the fused A1 post-physics step ------------------------------------
 * ShifuVecEnv.post_step (env.py:93-106) + obs clip (env.py:90) with the A1 task hooks. */
int shifu_a1_post_physics(ShifuCtx* ctx, const ShifuA1StepIO* io, void* stream);

/* ---- row a7 stand-alone / N1 self-check: the listed reward terms on the CURRENT tensors ------
 * terms_out[k*N + e] = value of term k of the descriptor for env e (no accumulation, no writes to
 * the env state).  The host-side term compiler calls the user's Python hook on the same tensors and
 * refuses to fuse when the two disagree (shifu/gym/env.py:180-185). */
int shifu_a1_eval_terms(ShifuCtx* ctx, const ShifuA1StepIO* io, float* terms_out, void* stream);

/* ---- rows a9-a11 stand-alone: A1Conditional.reset_idx(env_ids) ------------------------------
 * (a1_conditional.py:116-120; used by ShifuVecEnv.reset, env.py:108-112, and by user code).
 * env_ids: device int64 (n_ids), NULL = arange(n_ids).  Draws use io->step / io->step_dev. */
int shifu_a1_reset_idx(ShifuCtx* ctx, const ShifuA1StepIO* io, const int64_t* env_ids, int32_t n_ids,
                       void* stream);

/* ---- row a16 stand-alone: ShifuVecEnv.reset_idx(env_ids) of the ABB push-box scene -----------
 * (env.py:114-130 with RandPosBox._reset_root_state, a_prior_stage.py:39-51; used by
 * ShifuVecEnv.reset, env.py:108-112).  env_ids: device int64 (n_ids), NULL = arange(n_ids).
 * Adds the episode sums / success flags of the ids to the statistics accumulators. */
int shifu_abb_reset_idx(ShifuCtx* ctx, const ShifuAbbStepIO* io, const int64_t* env_ids, int32_t n_ids,
                        void* stream);

/* ---- row a16 -------------------------------------------------------------------------------- */
int shifu_abb_post_physics(ShifuCtx* ctx, const ShifuAbbStepIO* io, void* stream);

/* ---- row N2 (SURVEY.md 8f): the arm's PRE-physics action path --------------------------------
 * ArmRobot.inverse_kinematics (shifu/units/robot.py:156-182; same math as the stand-alone
 * shifu/utils/torch_utils.py:41-58): damped least squares
 *     u = J^T (J J^T + damping^2 I)^-1 [pos_err ; orn_err],   dof_targets = dof_pos + u
 * with orn_err = xyz(goal_quat * conj(ee_quat)) * sign(w) (robot.py:150-154, torch_utils.py:12-38).
 * When `actions` is non-NULL the goal is built first, as AbbRobot.step does
 * (examples/abb_pushbox_vision/a_prior_stage.py:67-73):
 *     goal_pos = clip(ee_pos + actions * ee_velocity * dt, min_ee_pos, max_ee_pos), goal_quat = tar_quat.
 * Floating-point row: the 6x6 system is solved by Cholesky instead of torch.inverse (LU); results
 * agree with the reference to the conditioning of J J^T + damping^2 I (tests state the tolerance). */
typedef struct ShifuArmIkIO {
  const float* body_state;      /* (N*num_bodies,13) gym rigid-body state; ee pose = row ee_body, cols 0:7 */
  const float* jacobian;        /* (N,num_links,6,num_dof) gym jacobian tensor; j_ee = [:, ee_link] (robot.py:125-128) */
  const float* dof_state;       /* (N*num_dof,2); dof_pos = [:,0] */
  const float* goal_pose;       /* (N,7) pos + quat(xyzw), or NULL when actions is given */
  const float* actions;         /* (N,3) or NULL */
  float* dof_targets;           /* w (N,num_dof) */
  int32_t num_bodies;           /* rigid bodies per env in body_state */
  int32_t ee_body;              /* end-effector body index inside the env */
  int32_t num_links;            /* links per env in the jacobian tensor */
  int32_t ee_link;              /* ee_body - 1 for a fixed-base arm (robot.py:128) */
  int32_t num_dof;              /* 1..SHIFU_MAX_DOF */
  float ee_velocity;            /* task_config.py:60 (0.2) */
  float dt;                     /* env.dt = sim.dt * decimation */
  float min_ee_pos[3];          /* task_config.py:63 */
  float max_ee_pos[3];          /* task_config.py:64 */
  float tar_quat[4];            /* a_prior_stage.py:70 (0,1,0,0) */
  float damping;                /* robot.py:156 (0.05) */
} ShifuArmIkIO;
int shifu_arm_ik(ShifuCtx* ctx, const ShifuArmIkIO* io, int32_t num_envs, void* stream);

/* ---- row N4 (SURVEY.md 8f): CameraSensor.refresh_image_tensors ------------------------------
 * shifu/units/sensors.py:165-188 copies one small image per env and image type inside a Python
 * loop over the envs.  Here one launch gathers every env's per-env interop tensors (addresses in a
 * device-resident pointer table, fixed after the sensors are created) into the batched buffers:
 *   color  (H,W,4) u8  -> color_out (N,H,W,3) f32 = rgba[..., :3] / 255   (normalize_color,
 *                         shifu/utils/image.py:12-15) or (N,H,W,4) u8 verbatim (sensors.py:171)
 *   depth  (H,W) f32   -> depth_out (N,H,W) = -depth                      (sensors.py:174-177)
 *   seg    (H,W) i32   -> seg_out   (N,H,W) verbatim                      (sensors.py:179-182)
 *   flow   (H,W) i16   -> flow_out  (N,H,W) verbatim                      (sensors.py:184-187)
 * A NULL *_src table skips that image type.  Every image must be 16-byte aligned. */
typedef struct ShifuCameraGatherIO {
  const void* const* color_src;   /* device array of N device pointers, or NULL */
  const void* const* depth_src;
  const void* const* seg_src;
  const void* const* flow_src;
  void* color_out;
  float* depth_out;
  int32_t* seg_out;
  int16_t* flow_out;
  int32_t height, width;
  int32_t normalize_color;        /* cfg.image_normalization */
} ShifuCameraGatherIO;
int shifu_camera_gather(ShifuCtx* ctx, const ShifuCameraGatherIO* io, int32_t num_envs, void* stream);

/* ---- row a8: reset_buf.nonzero().flatten() (env.py:101) -------------------------------------
 * ids_out (N) int64 ascending, n_out device int32.  Stand-alone so user-written
 * compute_termination hooks can use it too. */
int shifu_compact_reset_ids(ShifuCtx* ctx, const uint8_t* reset_buf, int32_t n, int64_t* ids_out,
                            int32_t* n_out, void* stream);

/* ---- rows a13/a14 for user-hook (unfused) tasks --------------------------------------------- */
/* HistoryRecorder.add (shifu/utils/train.py:12-14): history (N,A,H) shift + slot 0 = x (N,A). */
int shifu_history_add(ShifuCtx* ctx, float* history, const float* x, int32_t n, int32_t a, int32_t h, void* stream);
/* torch.clip(x, -c, c) (env.py:87,90), in place or out of place. */
int shifu_clip(ShifuCtx* ctx, const float* in, float* out, int64_t count, float c, void* stream);

/* ---- row N3 (SURVEY.md 8f): Terrain height map on the device ---------------------------------
 * Replaces the tile-by-tile numpy assembly of shifu/utils/terrain.py:42-173 (make_terrain 106-152,
 * add_terrain_to_map 154-173, gap_terrain / pit_terrain 176-198).  The caller lists one record per
 * tile; generators that draw random numbers (coarse noise grid, obstacle rectangles, stone heights)
 * find them in `table` (float64), written by the host in the generator's own draw order. */
enum ShifuTerrainKind {
  SHIFU_TERRAIN_PYRAMID = 0,        /* p = {peak, platform half-width px}                 pyramid_sloped_terrain */
  SHIFU_TERRAIN_PYRAMID_NOISE = 1,  /* p = {peak, half, nx, ny}; table: nx*ny coarse heights   + random_uniform_terrain */
  SHIFU_TERRAIN_STAIRS = 2,         /* p = {step width px, step height units, platform px}     pyramid_stairs_terrain */
  SHIFU_TERRAIN_OBSTACLES = 3,      /* p = {num rects, platform px}; table: (sx, sy, w, l, h) per rect */
  SHIFU_TERRAIN_STONES = 4,         /* p = {stone px, distance px, platform px, depth units}; table: height per stone */
  SHIFU_TERRAIN_GAP = 5,            /* p = {gap px, platform px}                          terrain.py:176-187 */
  SHIFU_TERRAIN_PIT = 6             /* p = {depth units, platform half px}                terrain.py:190-198 */
};
typedef struct ShifuTerrainTile {
  int32_t kind;        /* enum ShifuTerrainKind */
  int32_t i, j;        /* curriculum level (row of tiles) and terrain type (column of tiles) */
  int32_t p[4];
  int32_t table_off;   /* first entry of this tile in `table` */
} ShifuTerrainTile;
typedef struct ShifuTerrainDesc {
  int32_t num_rows, num_cols;          /* tiles */
  int32_t width_px, length_px;         /* tile size in cells (terrain.py:59-60) */
  int32_t border_px;                   /* terrain.py:62 */
  double env_length, env_width;        /* metres */
  double horizontal_scale, vertical_scale;
} ShifuTerrainDesc;
/* tiles / table: HOST arrays (n_tiles records, n_table doubles); height_map: device int16
 * (tot_rows x tot_cols, zero-filled border included); origins: device float64 (num_rows, num_cols, 3). */
int shifu_terrain_generate(ShifuCtx* ctx, const ShifuTerrainDesc* desc, const ShifuTerrainTile* tiles, int32_t n_tiles,
                           const double* table, int32_t n_table, int16_t* height_map, double* origins, void* stream);

/* ---- step statistics (row a11 logging, §8e collective payload) ------------------------------
 * After *_post_physics: move the step's stats (double[SHIFU_NUM_STATS]) into stats_out and clear
 * the accumulator; when step_dev_to_advance != NULL that device counter is incremented (the
 * common_step_counter += 1 of env.py:96 for graph-replayed steps).  Between this call and shifu_publish_extras a multi-GPU caller all-reduces
 * stats_out (sum over ranks; the host layer does it with torch.distributed over NCCL — the only
 * collective on the path, SURVEY.md C1 / §8e). */
int shifu_collect_stats(ShifuCtx* ctx, double* stats_out, int64_t* step_dev_to_advance, void* stream);
/* Same, into slot `slot` of a ring double[slots][SHIFU_NUM_STATS] (slot < 0: *step_dev % slots, read
 * before the increment): every step owns its vector, so a sharded run can all-reduce step t on a side
 * stream while step t+1 already runs (SURVEY.md §5: "overlap it on a side stream so it never gates the
 * next step"), also for steps replayed from a CUDA graph. */
int shifu_collect_stats_ring(ShifuCtx* ctx, double* ring, int32_t slots, int32_t slot, int64_t* step_dev_to_advance,
                             void* stream);

/* extras["episode"][term k] = mean over reset envs / max_episode_length_s, terrain_levels mean,
 * success_rate; values are left unchanged when no env reset this step (env.py:115-116).
 * extras_out: float[SHIFU_NUM_STATS] persistent device array:
 *   [k] term k mean, [8] n_reset (as float), [9] terrain_levels mean, [10] success_rate. */
int shifu_publish_extras(ShifuCtx* ctx, const double* stats, float* extras_out, void* stream);
/* Same, into slot `slot` of a ring of `slots` such arrays (float[slots][SHIFU_NUM_STATS]): every step
 * gets its own array, so the extras dicts of earlier steps that a caller still holds (rsl_rl keeps one
 * per rollout step; the reference allocates fresh tensors on every resetting step, env.py:124-130)
 * are not overwritten; a step without resets copies the previous slot.  slot < 0: the slot is
 * (*step_dev - 1) % slots, for graph-replayed steps whose counter lives on the device, and `stats` is
 * then the ring base shifu_collect_stats_ring wrote (same slot). */
int shifu_publish_extras_ring(ShifuCtx* ctx, const double* stats, float* ring, int32_t slots, int32_t slot,
                              const int64_t* step_dev, void* stream);

/* Synchronising convenience for tests: copy the accumulator as it stands to the host. */
int shifu_read_stats_host(ShifuCtx* ctx, double* stats_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SHIFU_B200_H */
