/*
 * hrl_b200.h - C-ABI of the B200-native batched env-step for hrl_pybullet_envs.
 *
 * This is the drop-in boundary (SURVEY.md 8b).  The reference reaches its physics through
 * per-env pybullet C-API calls; the batched replacement exposes ONE handle per device that
 * owns N envs.  Every entry point cites the reference interface it replaces (paths relative
 * to /root/reference/hrl_pybullet_envs).
 *
 * Conventions
 *   - plain C types only; no torch types.  All pointers named d_* are DEVICE pointers owned
 *     by the caller (e.g. tensor.data_ptr()), h_* are HOST pointers.
 *   - `stream` is a cudaStream_t passed as void* (0 = default stream); calls are asynchronous
 *     on that stream unless documented otherwise; calls on one handle must be stream-ordered.
 *   - return value: 0 = ok, <0 = error (HRL_E_*); hrl_last_error() gives text.  Nothing throws.
 */
#ifndef HRL_B200_H
#define HRL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- env families: the ids registered in __init__.py:9-16 (+ AntMjEnv, envs/MjAnt.py:31) */
enum {
  HRL_ANT_GATHER = 0,   /* envs/gather/ant_gather_env.py:12      obs 46, act 8 */
  HRL_ANT_MAZE = 1,     /* envs/ant_maze/ant_maze_bullet_env.py:17 obs 38, act 8 */
  HRL_ANT_FLAGRUN = 2,  /* envs/ant_flagrun/ant_flagrun_env.py:11 obs 28, act 8 */
  HRL_ANT_MJ = 3,       /* envs/MjAnt.py:31 (AntMjEnv)            obs 29, act 8 */
  HRL_POINT_GATHER = 4, /* envs/gather/point_gather_env.py:7      obs 18, act 2 */
  HRL_ANT_MAZE_MJ = 5   /* envs/ant_maze/ant_maze_mj_env.py:17    obs 60, act 8 */
};

enum {
  HRL_OK = 0,
  HRL_E_INVALID = -1, /* bad argument / config */
  HRL_E_CUDA = -2,    /* CUDA runtime error (text in hrl_last_error) */
  HRL_E_NOMEM = -3
};

#define HRL_MAX_ITEMS 16   /* 8 food + 8 poison (ant_gather_env.py:17-18 defaults) */
#define HRL_MAX_TARGETS 8  /* maze goal table (ant_maze_bullet_env.py:13-14: 4, ant_maze_mj_env.py:13-14: 5) */
#define HRL_MAX_BINS 16

/* ---- saved-state layout (hrl_get_state / hrl_set_state), one row per env ------------- */
#define HRL_STATE_F 72
enum {
  HRL_SF_POS = 0,      /* torso origin xyz (world)                                   */
  HRL_SF_QUAT = 3,     /* torso orientation x,y,z,w                                  */
  HRL_SF_LINVEL = 7,   /* world-frame linear velocity of the torso origin            */
  HRL_SF_ANGVEL = 10,  /* world-frame angular velocity                               */
  HRL_SF_Q = 13,       /* hip_1, ankle_1, ..., hip_4, ankle_4 (rad)                  */
  HRL_SF_QD = 21,      /* same order (rad/s)                                         */
  HRL_SF_INITIAL_Z = 29,
  HRL_SF_POTENTIAL = 30,
  HRL_SF_TARGET = 31,  /* walk target x,y                                            */
  HRL_SF_WTD = 33,     /* cached walk_target_dist of the last calc_state             */
  HRL_SF_FEET = 34,    /* 4 feet-contact flags shown in the NEXT obs (quirk Q2)      */
  HRL_SF_ITEMS = 38,   /* 16 x (x,y): food 0-7 then poison 8-15                      */
  HRL_SF_RETURN = 70,      /* return of the running episode (SURVEY.md section 5: metrics / logging)   */
  HRL_SF_RETURN_SUM = 71   /* sum of the returns of the episodes this env has finished                */
};
#define HRL_STATE_I 8
enum {
  HRL_SI_T = 0,          /* steps taken in this episode (TimeLimit counter)          */
  HRL_SI_EPISODE = 1,    /* number of resets so far                                  */
  HRL_SI_STEPS = 2,      /* steps taken since creation (RNG draw index of respawns)  */
  HRL_SI_GOALS_LEFT = 3, /* Flagrun: goals still in the list                         */
  HRL_SI_SINCE = 4,      /* Flagrun: steps_since_goal_change (survives reset)        */
  HRL_SI_REWARDED = 5,   /* Flagrun: _rewarded                                       */
  HRL_SI_GOAL_GEN = 6    /* Flagrun: create_targets() calls so far (each draws fresh goals, ant_flagrun_env.py:91-96); 7 spare */
};

/* ---- configuration: the reference's ctor kwargs + the recalled third-party constants --- */
typedef struct hrl_config {
  int32_t env_kind;
  int32_t num_envs;
  uint64_t seed;            /* env e uses RNG key (seed, env_index_offset + e)            */
  int32_t env_index_offset; /* global index of local env 0 (multi-GPU shards)             */
  int32_t max_episode_steps;/* 2000 (__init__.py:15); <=0 disables the TimeLimit          */
  int32_t auto_reset;       /* 1: done envs are reset inside hrl_step                     */
  /* physics [3P-MEM], SURVEY.md A.2/A.3 */
  float gravity;            /* 9.8 (ant_gather_env.py:58)                                 */
  float dt;                 /* 0.0165 control step                                        */
  int32_t substeps;         /* 4                                                          */
  int32_t solver_iters;     /* 5                                                          */
  float contact_erp;        /* 0.9  (setDefaultContactERP)                                */
  float limit_erp;          /* 0.2                                                        */
  float lin_damping;        /* 0.04 (btMultiBody default)                                 */
  float ang_damping;        /* 0.04                                                       */
  float friction;           /* combined mu robot-vs-scene: 1.5*0.8 (ant), 0.1*0.8 (point) */
  float limit_max_impulse;  /* 100                                                        */
  float max_coord_vel;      /* 100                                                        */
  float contact_margin;     /* 0.02 contact breaking threshold                            */
  float torque_scale;       /* power*power_coef = 2.5*100 (ant); 500 N (point_bot.py:29)  */
  int32_t torque_first_substep_only; /* SURVEY.md A.3 item 3                              */
  /* scene (sizeable_enclosed_scene.py:14-61, maze_scene.py:9-38) */
  float world_size[2];
  float ground_z;           /* top of the slab: 0.005 (plane.xml), 0 for the AntMj stadium */
  int32_t has_walls;
  int32_t has_box;          /* maze obstacle */
  float box_lo[3], box_hi[3];
  float start_pos[3];       /* base pose after reset                                      */
  int32_t n_scene_parts;    /* quirk Q1: scene bodies averaged into body_xyz              */
  float scene_parts_sum[2]; /* sum of their xy                                            */
  /* gather (ant_gather_env.py:16-29, gather_base.py:15-29) */
  int32_t n_food, n_poison, n_bins;
  float sensor_range, sensor_span, robot_coll_dist, robot_object_spacing, dying_cost;
  int32_t respawn, use_sensor;
  /* maze (ant_maze_bullet_env.py:23-25) / flagrun (ant_flagrun_env.py:14-16) */
  int32_t n_targets;
  float targets[HRL_MAX_TARGETS][2];
  float tol;
  int32_t done_at_target;
  float inner_rew_weight;
  int32_t target_encoding;  /* utils.py PositionEncoding: 0 normed_vec, 1 angle           */
  int32_t sense_walls;
  int32_t flag_max_targets; /* 100 */
  int32_t flag_timeout;     /* 200 */
  float flag_size;          /* 10  */
  float goal_reach_rew;     /* 5000 (ant_flagrun_env.py:160) */
  uint64_t flag_seed;       /* 123: goal stream shared by all envs (ant_flagrun_env.py:39) */
  /* reward weights of the third-party walker step (SURVEY.md 3P-5) */
  float electricity_cost, stall_torque_cost, joints_at_limit_cost;
  /* non-default ctor kwargs (SURVEY.md 8f item 3); appended so that the layout above is stable */
  int32_t sense_target;      /* ant_maze_bullet_env.py:24,135-178: goal sector sensor replaces the 2-d goal vector */
  int32_t maze_max_steps;    /* ant_maze_bullet_env.py:25,86-91: max_steps, -1 = off                        */
  int32_t targ_dist_rew;     /* ant_maze_bullet_env.py:25,93-94                                               */
  int32_t flag_use_sensor;   /* ant_flagrun_env.py:15,122-130: wall lidar appended (n_bins, sensor_span, sensor_range) */
  int32_t flag_switch_on_collision; /* ant_flagrun_env.py:16,187-194, default 1                               */
  float flag_max_target_dist;/* ant_flagrun_env.py:14,80-89: create_close_target when flag_max_targets <= 0   */
  /* food / poison cubes as colliders (assets/food.xml:17-22, gather_scene.py:62,66): static 0.25^3 boxes at z = 0.1.
   * On by default for AntGather, like the reference; required by the contact-based pickup (robot_coll_dist <= 0,
   * ant_gather_env.py:113-116).  With the distance-based pickup a cube is respawned once the torso is within 1 m,
   * so leg-vs-cube contacts are rare (the candidate mask is almost always empty: < 0.5 % of the step time). */
  int32_t item_contacts;
  float item_friction;       /* 1.5 (ant.xml:9) x 0.5 (Bullet default of the cube URDF) [3P-MEM]               */
  float item_half;           /* 0.125                                                                         */
  float item_z;              /* 0.1 (gather_scene.py:62)                                                      */
  int32_t flag_manual_goals; /* ant_flagrun_env.py:16,150-153 manual_goal_creation: reset() draws no goals and keeps the
                              * current walk target; the caller sets goals (VecEnv.set_target / create_targets)    */
} hrl_config;

typedef struct hrl_handle hrl_handle;

/* Fill `cfg` with the reference defaults of `env_kind` (ctor kwarg defaults cited above). */
int hrl_default_config(int32_t env_kind, int32_t num_envs, hrl_config* cfg);

/* obs / action widths of a config (observation_space.shape, action_space.shape). */
int hrl_obs_dim(const hrl_config* cfg);
int hrl_act_dim(const hrl_config* cfg);

/* Replaces env construction + the per-env BulletClient (pybullet.connect DIRECT). */
int hrl_create(const hrl_config* cfg, int32_t device, hrl_handle** out);
int hrl_destroy(hrl_handle* h);

/* Replaces env.reset() (ant_gather_env.py:68-74, ant_maze_bullet_env.py:104-121,
 * ant_flagrun_env.py:132-155, gather_base.py:67-72).  d_mask: u8[N] or NULL (= all).
 * d_obs: f32[N, obs_dim]; only rows of reset envs are written. */
int hrl_reset(hrl_handle* h, const uint8_t* d_mask, float* d_obs, void* stream);

/* Replaces env.step(a) (ant_gather_env.py:76-119, ant_maze_bullet_env.py:77-97,
 * ant_flagrun_env.py:162-204, MjAnt.py:36-97, gather_base.py:74-109) for all N envs.
 *   d_actions f32[N, act_dim]; d_obs f32[N, obs_dim]; d_rew f32[N]; d_done u8[N];
 *   d_info    f32[N, 4] or NULL: (food_rew | inner reward, dead_rew | goals_left, flags, episode length);
 *             flags: bit 0 = TimeLimit.truncated, bit 1 (Flagrun) = the walk target changed in this step, i.e. the
 *             reference sets info['target'] (ant_flagrun_env.py:188-191,199)
 *   d_terminal_obs f32[N, obs_dim] or NULL: pre-reset observation of envs that finished. */
int hrl_step(hrl_handle* h, const float* d_actions, float* d_obs, float* d_rew, uint8_t* d_done,
             float* d_info, float* d_terminal_obs, void* stream);

/* Same as hrl_step but with HOST buffers (pinned or pageable): copies actions H2D, steps,
 * copies obs/rew/done (and info if non-NULL) D2H and synchronises the stream - the call a
 * gym-style user makes with numpy arrays. */
int hrl_step_host(hrl_handle* h, const float* h_actions, float* h_obs, float* h_rew, uint8_t* h_done,
                  float* h_info, void* stream);

/* How hrl_step_host moves data (the reference has no device boundary: env.step(a) takes and returns
 * numpy arrays, ant_gather_env.py:76-119, so this is the whole cost of being a drop-in for it):
 *   HRL_HOST_COPY      H2D copy of the actions, kernel, D2H copies (ONE copy when the four output
 *                      buffers are carved out of one allocation as hrl_host_layout says), sync;
 *   HRL_HOST_ZEROCOPY  the output buffers must be pinned: the kernel writes them over PCIe while
 *                      it computes (transfers overlap the step), sync;
 *   HRL_HOST_AUTO      zero-copy when all output buffers are pinned, else copy (default).
 * h_info may also be a DEVICE pointer: the per-step info columns then stay on the device (16 of the 205 bytes per env the
 * host path would otherwise move) and the caller fetches them only when somebody looks (VecEnv does).
 * In the last two modes a pinned action array is read in place over PCIe; a pageable one (the
 * array a gym-style caller hands over) is copied H2D first - it is asked afresh on every call.
 * The handle caches which host pointers are pinned; calling hrl_set_host_mode (any mode) clears
 * that cache - do so after freeing a pinned buffer that was passed to hrl_step_host.
 * Calls on one handle must not overlap (the reference env is single-threaded too). */
#define HRL_HOST_AUTO 0
#define HRL_HOST_COPY 1
#define HRL_HOST_ZEROCOPY 2
int hrl_set_host_mode(hrl_handle* h, int32_t mode);
/* Byte offsets of rew / info / done inside one packed host allocation that starts with obs
 * (obs f32[N,D] | rew f32[N] | info f32[N,4] | done u8[N], 256-byte aligned sections); total bytes. */
int hrl_host_layout(const hrl_config* cfg, size_t* off_rew, size_t* off_info, size_t* off_done, size_t* total);

/* Fused rollout with an in-kernel policy (SURVEY.md 8f item 4, "policy-inference fusion"; no counterpart in the reference,
 * whose users call step() once per action: README.md:20-37).  ONE launch runs T consecutive env steps of all N Ant envs;
 * the action of every step is computed in the kernel from the observation the previous step produced, by the MLP
 *     a = tanh(W3 tanh(W2 tanh(W1 obs + b1) + b2) + b3) + sigma * N(0, 1)           (then clipped like any action)
 * so neither observations nor actions leave the SM between steps and the robot state stays in registers.
 *   d_weights f32, packed INPUT-major: W1[obs_dim][H] b1[H] W2[H][H] b2[H] W3[H][8] b3[8], H = hidden = 32 or 64
 *   d_obs f32[T+1, N, obs_dim] (slot 0 = the observation before the first step), d_act f32[T, N, 8] (the actions taken,
 *   before clipping), d_rew f32[T, N], d_done u8[T, N].  Auto-reset as in hrl_step; info / terminal observations are not
 *   produced.  noise_seed keys the counter RNG of the exploration noise (addressed by env and step count). */
int hrl_rollout_mlp(hrl_handle* h, int32_t T, const float* d_weights, int32_t hidden, float sigma, uint64_t noise_seed,
                    float* d_obs, float* d_act, float* d_rew, uint8_t* d_done, void* stream);

/* hrl_rollout_mlp for training (hrl_rollout_mlp is this call with d_sigma, d_info and d_terminal_obs NULL).  Every env
 * family, PointGather included (act_dim A = 2: W3[H][2] b3[2]; Ant: A = 8).  The buffers a trainer needs besides those above:
 *   d_sigma        f32[A] or NULL: action component c gets noise d_sigma[c] * N(0, 1) (the same draw as for the scalar
 *                  sigma, so d_sigma filled with s gives the actions of sigma = s); entries must be finite and >= 0, which
 *                  the caller checks (reading them here would cost a synchronisation).  NULL: the scalar sigma for all.
 *   d_info         f32[T, N, 4] or NULL: slot t holds what hrl_step writes to d_info for step t (bit 0 of column 2 tells a
 *                  TimeLimit truncation from a termination).
 *   d_terminal_obs f32[T, N, obs_dim] or NULL: row e of slot t is written only when env e finished in step t, with its
 *                  observation from before the auto-reset (d_obs[t + 1] already holds the reset observation); other rows
 *                  are left untouched, as in hrl_step.
 * d_act f32[T, N, A]; T >= 1; hidden = 32 or 64. */
int hrl_rollout_mlp_ex(hrl_handle* h, int32_t T, const float* d_weights, int32_t hidden, float sigma, const float* d_sigma,
                       uint64_t noise_seed, float* d_obs, float* d_act, float* d_rew, uint8_t* d_done, float* d_info,
                       float* d_terminal_obs, void* stream);

/* hrl_rollout_mlp_ex with a normalized policy input (hrl_rollout_mlp_ex is this call with NULL, NULL, 0).
 *   d_obs_mean, d_obs_rstd f32[obs_dim]: both NULL (the raw observation, as hrl_rollout_mlp_ex) or both non-NULL.  The
 *   policy then reads, for obs component i,
 *       x_i = fminf(fmaxf((o_i - mean_i) * rstd_i, -obs_clip), obs_clip)       (float32; subtract, multiply, clamp)
 *   so torch.clamp((obs - mean) * rstd, -obs_clip, obs_clip) gives the same bits for finite observations.  obs_clip must be
 *   finite and > 0 when the statistics are given.  The statistics are read once per launch: they are frozen for the T steps.
 *   d_obs and d_terminal_obs still receive the RAW observations.
 * The one difference from SB3 VecNormalize: SB3 updates the observation statistics every step, so step t + 1's input is
 * normalized with statistics that already include it.  Here the statistics are frozen for a rollout and updated from its
 * observations afterwards (hrl_obs_moments), as GPU-batched PPO implementations do. */
int hrl_rollout_mlp_norm(hrl_handle* h, int32_t T, const float* d_weights, int32_t hidden, float sigma, const float* d_sigma,
                         uint64_t noise_seed, const float* d_obs_mean, const float* d_obs_rstd, float obs_clip,
                         float* d_obs, float* d_act, float* d_rew, uint8_t* d_done, float* d_info, float* d_terminal_obs,
                         void* stream);

/* Score a population of P MLP policies by their episodes, in ONE launch and without per-step buffers (evolution
 * strategies, population-based training, comparing checkpoints).  The policy, noise and auto-reset are those of
 * hrl_rollout_mlp_norm; what differs is that each env runs its member's weights and that only per-env results are written.
 *   d_weights  f32[P][nw]: P rows in the packed layout of hrl_rollout_mlp, nw = D*H + H + H*H + H + H*A + A.
 *   Env e runs member e / M, M = N / P.  P = 1: any N.  P > 1: N must be a multiple of P and M a multiple of the envs
 *   one CTA runs, 16 for the Ant families and 8 for PointGather (a CTA stages one member's weights); otherwise
 *   HRL_E_INVALID.
 *   sigma, d_sigma, noise_seed, d_obs_mean, d_obs_rstd, obs_clip: as in hrl_rollout_mlp_norm, shared by every member (the
 *   same noise draw for the same seed, global env index and step count; the statistics frozen for the launch).
 * T steps run from the current state; nothing per step is written.  Per env:
 *   d_ret      f32[N]: the sum of the rewards from the launch's first step up to and including the env's first done,
 *              accumulated in float32 in step order (ret += rew);
 *   d_len      i32[N]: the number of those steps;
 *   d_finished u8[N]:  1 if a done came within the T steps; else 0, and d_ret / d_len cover all T steps.
 * The env state afterwards is the state after T steps, the one hrl_rollout_mlp would leave.  To score whole episodes, reset
 * first (hrl_reset): a launch that starts mid-episode scores the remainder of that episode.  T >= 1, P >= 1, hidden = 32 or
 * 64, and the three result pointers are required. */
int hrl_evaluate_mlp(hrl_handle* h, int32_t T, int32_t P, const float* d_weights, int32_t hidden, float sigma, const float* d_sigma,
                     uint64_t noise_seed, const float* d_obs_mean, const float* d_obs_rstd, float obs_clip, float* d_ret,
                     int32_t* d_len, uint8_t* d_finished, void* stream);

/* Replaces saveState/restoreState (used as the reset mechanism by pybullet_envs) and gives
 * the "identical saved states" hook the one-step parity tests need.
 *   d_fstate f32[N, HRL_STATE_F], d_istate i32[N, HRL_STATE_I]. */
int hrl_get_state(hrl_handle* h, float* d_fstate, int32_t* d_istate, void* stream);
int hrl_set_state(hrl_handle* h, const float* d_fstate, const int32_t* d_istate, void* stream);
/* Observation of the current state without stepping (reset()'s return path). */
int hrl_observe(hrl_handle* h, float* d_obs, void* stream);

/* AntFlagrunBulletEnv.next_target() (ant_flagrun_env.py:112-120) for the envs with d_mask[e] != 0 (NULL: all): pop the
 * next pre-drawn goal (or draw a close one when max_targets <= 0), clear `_rewarded`, restart the potential
 * (steps_since_goal_change is left alone, like the reference's method).  With manual_goal_creation (hrl_config.flag_manual_goals) this, together with writing
 * HRL_SF_TARGET / HRL_SI_GOALS_LEFT through hrl_set_state (set_target :98-110, create_targets :91-96), is how the
 * caller drives the goals; envs with an empty goal list are left untouched (the reference raises IndexError). */
int hrl_flagrun_next_target(hrl_handle* h, const uint8_t* d_mask, void* stream);

/* ---- stand-alone parity entry points (stateless) --------------------------------------- */
/* Gather sector sensor, ant_gather_env.py:128-177 / gather_base.py:118-168.
 *   d_xy f32[M,2] torso xy, d_yaw f32[M], d_items f32[M,16,2] -> d_food/d_poison f32[M,n_bins],
 *   d_bins i32[M,16] bin index of each item or -1 when not sensed. */
int hrl_gather_sensor(int32_t M, int32_t n_bins, float sensor_range, float sensor_span, const float* d_xy,
                      const float* d_yaw, const float* d_items, float* d_food, float* d_poison,
                      int32_t* d_bins, void* stream);
/* Wall lidar, sizeable_enclosed_scene.py:63-97.  d_bounds f32[n_lines,4] (x1,y1,x2,y2). */
int hrl_sense_walls(int32_t M, int32_t n_bins, float span, float range, int32_t n_lines,
                    const float* d_bounds, const float* d_xy, const float* d_yaw, float* d_out, void* stream);
/* GAE(lambda) over a rollout buffer (no counterpart in the reference; DESIGN.md section 4, kernel 7).  Stateless, no handle;
 * runs on the current device.  ONE launch, no atomics: the same inputs give the same bytes on every call.
 *   d_rew f32[T,N], d_done u8[T,N], d_values f32[T+1,N] (V of obs[0..T]),
 *   d_info f32[T,N,4] and d_terminal_values f32[T,N]: both NULL (every done terminates) or both non-NULL,
 *   d_adv f32[T,N], d_ret f32[T,N] or NULL.  0 <= gamma, lam <= 1.  Asynchronous on `stream`, no host synchronisation.
 * For env e and step t:
 *   next_t  = d_terminal_values[t,e] if done and bit 0 (TimeLimit truncation) of int(d_info[t,e,2]) is set,
 *             0 if done otherwise (bit 1, the Flagrun goal switch, is ignored), d_values[t+1,e] if not done;
 *   delta_t = rew + gamma next_t - values[t,e];  A_t = delta_t + gamma lam (1 - done_t) A_{t+1}, A_T = 0;  ret_t = A_t + values[t,e].
 * Values that are not selected are never operands: stale terminal-value rows and the value after a termination may hold
 * anything, NaN included.  d_adv / d_ret must not overlap the inputs. */
int hrl_gae(int32_t T, int32_t N, float gamma, float lam, const float* d_rew, const uint8_t* d_done, const float* d_info,
            const float* d_values, const float* d_terminal_values, float* d_adv, float* d_ret, void* stream);
/* Running observation statistics (SB3 RunningMeanStd; DESIGN.md section 4, kernel 8).  Stateless, current device.
 * Merges the batch d_x f32[M, D] into d_moments f64[1 + 2D] = {count, mean[D], var[D]} with SB3's update_from_moments:
 *   delta = bmean - mean;  tot = count + M;  mean += delta * M / tot;
 *   var = (var * count + bvar * M + delta^2 * count * M / tot) / tot;  count = tot        (bvar: population variance)
 * then writes d_mean_f[i] = (float)mean[i] and d_rstd_f[i] = (float)(1 / sqrt(var[i] + eps)), the two arrays
 * hrl_rollout_mlp_norm reads.  The initial state is the caller's (SB3: count = 1e-4, mean = 0, var = 1).
 * Accumulates in float64 (deviations from a sample inside a thread, Chan merges above it, in a fixed order); ONE launch of
 * one thread-block cluster, no atomics, no scratch memory: the same inputs give the same bytes on every call, and calls on
 * different streams may overlap.  No host synchronisation, no allocation: capturable in a CUDA graph.
 * 1 <= M, 1 <= D <= 64, eps > 0, no NULL pointer. */
int hrl_obs_moments(int32_t M, int32_t D, const float* d_x, double* d_moments, float eps, float* d_mean_f, float* d_rstd_f,
                    void* stream);
/* Return-based reward scaling with SB3 VecNormalize's sequential semantics (step_wait, _update_reward, normalize_reward).
 * Stateless, current device.  For t = 0 .. T-1:
 *   R[e]      = gamma * R[e] + rew[t, e]                                (d_returns f64[N], carried across calls)
 *   moments   = merge(moments, mean_e R, population-var_e R, count N)    (d_ret_moments f64[3] = {count, mean, var})
 *   s_t       = (float)(1 / sqrt(var + eps))
 *   out[t, e] = fminf(fmaxf(rew[t, e] * s_t, -clip), clip)              (float32)
 *   R[e]      = 0 where done[t, e]                                       (truncations included, as in SB3)
 * R is kept in float64; the per-step mean and variance are taken over R rounded to float32 (a relative difference of at
 * most 2^-24 per value).  d_rew f32[T, N], d_done u8[T, N], d_work f64 scratch of >= 2 T entries (contents on entry do not
 * matter), d_out f32[T, N], which must not overlap the inputs.  1 <= T, N; 0 <= gamma <= 1; clip, eps > 0.
 * THREE launches (a scan over T per env, one cluster for the statistics and the chain over t, the scaling), no atomics:
 * the same bytes on every call.  No host synchronisation, capturable in a CUDA graph. */
int hrl_reward_scale(int32_t T, int32_t N, float gamma, float clip, float eps, const float* d_rew, const uint8_t* d_done,
                     double* d_returns, double* d_ret_moments, double* d_work, float* d_out, void* stream);
/* `n_sub` physics sub-steps on the handle's current state (no task logic, no reset):
 * replaces scene.global_step() -> p.stepSimulation() (ant_gather_env.py:78). */
int hrl_substeps(hrl_handle* h, const float* d_actions, int32_t n_sub, void* stream);

/* Lane mapping of the fused Ant kernels (a tuning knob, not part of the reference's surface): 4 lanes per env
 * (8 envs per warp), 8 (4 envs per warp) or 16 (2 envs per warp); results are identical up to float rounding.
 * New handles take the library default, or HRL_B200_LANES from the environment.  DESIGN.md section 4. */
int hrl_set_lanes_per_env(hrl_handle* h, int32_t lanes);
int hrl_get_lanes_per_env(const hrl_handle* h);
/* Solver-row layout of the 4-lane Ant kernel: 14-wide rows, or compact rows (the 8 non-zeros of a row + its leg index,
 * expanded to 14 wide on load; smaller shared memory, so 7 CTAs per SM instead of 6).  Results agree up to float32
 * rounding: the compiler contracts a few multiply-adds differently in the two kernels.
 * hrl_create picks compact when it saves a whole wave of CTAs at the device's SM count; HRL_B200_COMPACT=0|1 in the
 * environment overrides that for new handles.  set: any handle (HRL_E_INVALID for NULL).  get: 1 iff the next step,
 * reset, observe or substeps launch uses the compact rows (an Ant env with 4 lanes per env and the flag set), 0 if not,
 * -1 for NULL.  The fused rollout (hrl_rollout_mlp*) always uses the 14-wide rows. */
int hrl_set_compact_rows(hrl_handle* h, int32_t on);
int hrl_get_compact_rows(const hrl_handle* h);

/* In-kernel counters feeding the FLOP model of bench.py (SURVEY.md section 5 "in-kernel optional counters"):
 * out = {contacts, joint-limit rows, env-substeps, reserved} accumulated since the last reset; synchronises. */
int hrl_get_stats(hrl_handle* h, unsigned long long out[4], int reset);

/* Measurement aid (bench.py): work enqueued on `stream` after this call waits ON THE DEVICE until the 32-bit word at
 * d_flag (pinned host memory the device can address, or device memory) equals `expect`, or `timeout_ns` elapsed.
 * Lets a caller queue a batch of steps with their timing events and release them at once, so that no host-side
 * launch gap can fall between an event pair.  Not part of the reference's surface. */
int hrl_stream_gate(const uint32_t* d_flag, uint32_t expect, uint64_t timeout_ns, void* stream);

/* Number of kernels this library has launched since load (bench's gpu_launches claim). */
int64_t hrl_launch_count(void);
const char* hrl_last_error(void);
const char* hrl_version(void);

#ifdef __cplusplus
}
#endif
#endif /* HRL_B200_H */
