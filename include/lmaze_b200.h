/*
 * lmaze_b200.h -- C ABI of the B200-native batched LMaze step/reset path.
 *
 * The reference (gkm2708/gym-lmaze) has no FFI layer: its hot path sits behind
 * gym's Python Env protocol -- `reset() -> obs`, `step(a) -> (obs, reward, done,
 * info)` on one maze (reference gym_lmaze/envs/lmaze_env.py:64,146,237;
 * lmaze_env_v3.py:134,220,398-402).  This header is the boundary a maintainer
 * would bind instead (ctypes stub in INTEGRATION.md): the same operations over N
 * independent mazes whose state and outputs live in GPU memory.
 *
 * Conventions
 *   - every function returns 0 on success or a negative lmz_status; the message
 *     for the calling thread's last failure is lmz_last_error()
 *   - no exceptions, aborts or hidden synchronisation: work is enqueued on the
 *     caller's CUDA stream (`stream` is a cudaStream_t passed as void*; NULL =
 *     the legacy default stream); asynchronous CUDA faults surface on a later call
 *   - the caller owns every buffer; pointers are DEVICE pointers unless the
 *     name says `_host`; the handle owns only its small per-env state arrays
 *   - the `_dl` forms take borrowed `DLManagedTensor*` (include/lmz_dlpack.h),
 *     validate device / dtype / shape / contiguity / alignment and forward to the
 *     plain-pointer forms.  They never call the tensor's deleter.
 *   - one handle <-> one device; calls on one handle must be serialised by the caller
 *
 * There is no CPU implementation behind this ABI.
 */
#ifndef LMAZE_B200_H
#define LMAZE_B200_H

#include <stdint.h>
#include "lmz_dlpack.h"

#ifdef __cplusplus
extern "C" {
#endif

#define LMZ_ABI_VERSION 1

typedef struct lmz_env lmz_env;   /* opaque handle */

typedef enum {
  LMZ_OK = 0,
  LMZ_ERR_INVALID = -1,    /* bad argument (NULL, range, shape, dtype, alignment) */
  LMZ_ERR_CUDA = -2,       /* a CUDA runtime call failed; message has the cudaError */
  LMZ_ERR_STATE = -3,      /* call not legal in the handle's state (e.g. step before bind) */
  LMZ_ERR_UNSUPPORTED = -4
} lmz_status;

/* Maze variants (reference class each one replaces). */
typedef enum {
  LMZ_V0 = 0,   /* LmazeEnv     'lmaze-v0', 12x12, obs f32 (4,84,84)  -- lmaze_env.py:11-256    */
  LMZ_V2 = 2,   /* LmazeEnv_v2  'lmaze-v2', 5 mazes of 18x18, Discrete(25), obs f32 (5,35,35) -- lmaze_env_v2.py:17-405 */
  LMZ_V3 = 3,   /* LmazeEnv_v3  'lmaze-v3', 18x18, obs f32 (3,72,72)  -- lmaze_env_v3.py:17-402 */
  LMZ_V4 = 4,   /* LmazeEnv_v4  'lmaze-v4', v2 + float visit layer, obs f32 (7,35,35) -- lmaze_env_v4.py:17-482 */
  LMZ_V5 = 5    /* LmazeEnv_v5 / LmazeEnv_v6  'lmaze-v5', 'lmaze-v6': planner / actor env, foveal obs f32 (7,35,35)
                   + local obs f32 (4,35,35) -- lmaze_env_v5.py:17-712; v6 adds safeFovealGoal, lmaze_env_v6.py:505-523 */
} lmz_variant;

/* How the fused kernel writes the observation tensor. */
typedef enum {
  LMZ_RENDER_TMA = 0,     /* bulk async shared->global copies (cp.async.bulk) of template segments */
  LMZ_RENDER_ST128 = 1,   /* 128-bit vector stores (st.global.v4) fed from the shared-memory template */
  LMZ_RENDER_INCREMENTAL = 2  /* v0/v3: the bound obs tensor persists, so a step only erases the ball's old ExE block
                             and draws the new one (2*E*E floats instead of the whole image); the tensor stays
                             bit-identical to a full render.  Full renders (TMA) are used for reset / render calls
                             and whenever the tensor may be stale (after bind, set_window, set_state).  The caller
                             must not write into obs. */
} lmz_render_mode;

/* What the observation tensor holds. */
typedef enum {
  LMZ_OBS_FULL = 0,       /* f32 [N,C,G*E,G*E]: the reference's upsampled image (lmaze_env.py:217-234), bit-exact */
  LMZ_OBS_COMPACT = 1,    /* u8  [N,C,G,G]: the same layers BEFORE the xE upsample (lmaze_env.py:208-215);
                             the reference image is exactly repeat_interleave(compact, E) on both axes.
                             Foveal variants (v2, v4, v5): f32 [N,C,5,5] -- the 5x5 crops before the x7 upsample
                             (lmaze_env_v2.py:185-203); v5's local obs is then f32 [N,4,5,5] */
  LMZ_OBS_BITS = 2        /* v0 / v3: u8 [N,R]: the compact layers at ONE BIT per cell -- every value of those layers is
                             0.0 or 1.0 (lmaze_env.py:80,92-107) -- bit k of the flattened [C][G][G] layers is bit k%8 of
                             byte k/8 (little-endian bit order), rows padded to whole 32-bit words: R = 72 (v0, 576 bits),
                             124 (v3, 972 bits + 20 zero pad bits).  The observation for a HOST consumer: 72 B instead of
                             112,896 B per env over PCIe; unpacking + xE replication gives the reference image exactly. */
} lmz_obs_mode;

/* Element type of an action buffer. */
typedef enum { LMZ_ACT_U8 = 0, LMZ_ACT_I32 = 1, LMZ_ACT_I64 = 2 } lmz_action_dtype;

typedef struct lmz_config {
  int32_t  struct_size;   /* = sizeof(lmz_config); guards against header/library skew */
  int32_t  variant;       /* lmz_variant */
  int64_t  num_envs;      /* N: mazes owned by this handle (this rank's shard) */
  int64_t  env_id0;       /* global id of env 0; the device RNG is keyed by global id so
                             trajectories do not depend on how envs are sharded over GPUs */
  uint64_t seed;
  int32_t  device;        /* CUDA device ordinal */
  int32_t  autoreset;     /* 1: an env that finishes is re-spawned inside the same step and the
                             returned obs is the new episode's first obs (terminal reward/done kept);
                             0: reference behaviour, stepping past done is legal (lmaze_env.py:246-249) */
  int32_t  random_ball;   /* RANDOM_BALL  (lmaze_env.py:25, lmaze_env_v3.py:103); 0 => spawn on 'S' */
  int32_t  random_goal;   /* RANDOM_GOAL  (lmaze_env_v3.py:104); ignored by v0 */
  int32_t  render_mode;   /* lmz_render_mode */
  int32_t  tune[4];       /* launch tuning for the TMA render path, 0 = library default:
                             [0] threads per CTA (TMA path: 32/64/128/256 issuing warps x32; ST128 path: 256/512/1024;
                                 foveal render kernels: 128 (default), 160, 192, 224, 256, 512, 1024;
                                 compact foveal kernel: 64, 128 (default), 256)
                             [1] L2 policy of the obs stores: 1 evict_first, 2 evict_normal, 3 evict_last, 4 none
                             [2] resident CTAs per SM (0 = library default)
                             [3] split bulk copies into pieces of at most this many bytes (multiple of 16) */
  int32_t  obs_mode;      /* lmz_obs_mode */
  int32_t  reserved[2];   /* must be zero */
} lmz_config;

/* Episode statistics kept on the device as integer counters (lmz_stats). */
enum {
  LMZ_STAT_STEPS = 0,     /* env-steps executed */
  LMZ_STAT_EPISODES,      /* done flags raised */
  LMZ_STAT_GOALS,         /* reward == 100.0 */
  LMZ_STAT_TIMEOUTS,      /* done without a goal */
  LMZ_STAT_WALL_BUMPS,    /* 'W' branch  (lmaze_env.py:172-174) */
  LMZ_STAT_MOVES,         /* 'B'/'X' branches (lmaze_env.py:176-195) */
  LMZ_STAT_STALE,         /* 'S' target: no branch, reward kept (v0 quirk) */
  LMZ_STAT_EPLEN_SUM,     /* sum of stepCount over finished episodes */
  LMZ_NUM_STATS
};

/* Columns of the unpacked per-env state exchanged by lmz_get_state / lmz_set_state. */
enum {
  LMZ_ST_X = 0, LMZ_ST_Y, LMZ_ST_GOAL_X, LMZ_ST_GOAL_Y, LMZ_ST_STEP_COUNT,
  LMZ_ST_REWARD_CODE,     /* 0: -0.0  1: -1.0  2: -0.01  3: 100.0  (last reward, lmaze_env.py:109,174-194) */
  LMZ_ST_GOAL_COUNT,      /* goalCount, survives reset (lmaze_env.py:24,195) */
  LMZ_ST_EPISODE,         /* resets performed so far (device RNG counter) */
  LMZ_ST_COLS
};

/* ---- library ---- */
int         lmz_abi_version(void);
const char *lmz_last_error(void);
void        lmz_default_config(lmz_config *cfg);                    /* fills struct_size + defaults */
/* Static facts about a variant: obs shape (C,H,W) -- observation_space of
 * lmaze_env.py:20 / lmaze_env_v3.py:91 -- and grid side. */
int         lmz_obs_shape(int32_t variant, int64_t shape[3]);
int         lmz_grid_size(int32_t variant);
/* Shape (C,H,W) and element size of one env's observation in the given obs_mode. */
int         lmz_obs_desc(int32_t variant, int32_t obs_mode, int64_t shape[3], int32_t *elem_bytes);
/* Copies the maze rows (G*G cell letters, row-major, no terminator) -- lmaze_env.py:37-48. */
int         lmz_layout(int32_t variant, char *cells);
/* Variants with several mazes (v2: 5, lmaze_env_v2.py:303-405): index is 1-based. */
int         lmz_num_layouts(int32_t variant);
int         lmz_layout_ex(int32_t variant, int32_t index, char *cells);
/* n of the variant's Discrete(n) action space (lmaze_env.py:16, lmaze_env_v2.py:39). */
int         lmz_num_actions(int32_t variant);

/* ---- handle lifecycle: replaces LmazeEnv.__init__ (lmaze_env.py:14-53) minus its first reset ---- */
int lmz_create(const lmz_config *cfg, lmz_env **out);
int lmz_destroy(lmz_env *env);

/* ---- observation memory ---- */
/* Device memory for an observation tensor, bound like any other buffer.  With LMZ_OBS_MEM_COMPRESSIBLE it is memory
 * the L2 may keep compressed in DRAM (cuMemCreate with generic compression, on devices that support it): lossless and
 * invisible to kernels, copies and DLPack consumers, and an observation is largely whole lines of zeros, so fewer
 * bytes reach DRAM.  *compressed_bytes (may be NULL) returns how many bytes the driver made compressible; 0 means
 * plain cudaMalloc memory (not asked for, not supported, or refused).  The memory belongs to the caller, not to any
 * handle: lmz_destroy never frees it.  lmz_free_obs waits for the device, then releases it. */
enum { LMZ_OBS_MEM_COMPRESSIBLE = 1 };
int lmz_alloc_obs(int32_t device, int64_t bytes, int32_t flags, void **ptr, int64_t *compressed_bytes);
int lmz_free_obs(void *ptr);

/* Bind the output buffers every later call writes: obs (f32 [N,C,H,W], or u8 [N,C,G,G] in
 * compact mode; may be NULL: transition only, nothing rendered), reward f32 [N], done u8 [N].
 * obs must be 16-byte aligned. */
int lmz_bind(lmz_env *env, void *obs, float *reward, uint8_t *done);
int lmz_bind_dl(lmz_env *env, DLManagedTensor *obs, DLManagedTensor *reward, DLManagedTensor *done);

/* Render window: re-point obs at a buffer of env_count rows that stands for envs
 * [env_lo, env_lo + env_count).  Steps still advance EVERY env but only render the window;
 * lmz_render re-renders whatever window is current, so a batch whose full observation tensor
 * does not fit in HBM (8M v3 envs = 498 GB) is consumed window by window. */
int lmz_set_window(lmz_env *env, void *obs, int64_t env_lo, int64_t env_count);
int lmz_set_window_dl(lmz_env *env, DLManagedTensor *obs, int64_t env_lo);

/* reset(): replaces LmazeEnv.reset (lmaze_env.py:64-141) / LmazeEnv_v3.reset
 * (lmaze_env_v3.py:134-206) for every env whose mask byte is non-zero (mask NULL =
 * all).  spawn NULL => device RNG; else int32 [N][4] = ball_x, ball_y, goal_x,
 * goal_y (the cells the reference's rejection loop would have accepted; goal
 * ignored by v0; for v2 the last column is goal_y | new_layout << 5, because its
 * reset also re-rolls the maze, lmaze_env_v2.py:90-92).  Re-renders obs for the
 * envs it resets.  v3: a row with LMZ_SPAWN_FORCE added to goal_x overrides RANDOM_BALL /
 * RANDOM_GOAL = 0 -- the priority reset(mode="test") has in lmaze_env_v3.py:145-146,154-155. */
#define LMZ_SPAWN_FORCE 64
int lmz_reset(lmz_env *env, const uint8_t *mask, const int32_t *spawn, void *stream);
int lmz_reset_dl(lmz_env *env, DLManagedTensor *mask, DLManagedTensor *spawn, void *stream);

/* step(): replaces LmazeEnv.step (lmaze_env.py:146-237) / LmazeEnv_v3.step
 * (lmaze_env_v3.py:220-402): one fused kernel -- action decode, wall lookup,
 * move, reward, done, optional auto-reset, obs render, statistics.  actions is
 * [N] of `action_dtype`; codes 0..3 move, any other value takes the reference's
 * unmatched branch (offset 0,0).  spawn as for lmz_reset, consumed only by envs
 * that auto-reset in this step. */
int lmz_step(lmz_env *env, const void *actions, int32_t action_dtype, const int32_t *spawn, void *stream);
int lmz_step_dl(lmz_env *env, DLManagedTensor *actions, DLManagedTensor *spawn, void *stream);

/* Host-buffer form of step() (the end-to-end call): copies actions H2D, runs the
 * fused step, copies reward/done (and obs when obs_host != NULL) D2H and waits
 * for the stream.  Host buffers should be pinned for the copies to be asynchronous. */
int lmz_step_host(lmz_env *env, const void *actions_host, int32_t action_dtype,
                  float *reward_host, uint8_t *done_host, void *obs_host, void *stream);

/* Double-buffered form for a host consumer (pipeline depth 2).  _async enqueues the H2D copy of the actions, the
 * fused step and -- on an internal copy stream -- the D2H copies of reward / done / obs into the given host
 * buffers, and returns at once with *ticket (0 or 1); _wait blocks until that step's copies have landed.  The
 * copies of step k overlap the H2D + kernel of step k+1; a third _async call reuses the first ticket's device
 * buffers, so wait for ticket t before submitting the second step after it.  All host buffers (actions included)
 * must stay untouched until the step's _wait returns.  The step's outputs are written to handle-owned device
 * buffers, NOT to the tensors given to lmz_bind; obs_host is only available for obs_mode compact / bits. */
int lmz_step_host_async(lmz_env *env, const void *actions_host, int32_t action_dtype, float *reward_host,
                        uint8_t *done_host, void *obs_host, void *stream, int32_t *ticket);
int lmz_step_host_wait(lmz_env *env, int32_t ticket);

/* Render the current state into the bound obs without stepping (the
 * upsample loop of lmaze_env.py:208-234 on its own). */
int lmz_render(lmz_env *env, void *stream);

/* T fused steps with state in registers and no per-step observation:
 * rewards f32 [T][N], dones u8 [T][N].  actions NULL => device-side random
 * actions (Philox keyed by seed, global env id, step index); else [T][N].
 * v0 / v3: lmaze_env.py:146-237 / lmaze_env_v3.py:220-402 looped; v2 / v4: lmaze_env_v2.py:127-225 /
 * lmaze_env_v4.py:155-275 looped (Discrete(25) actions; v4's visit layer is kept up to date in HBM).
 * v5 / v6 roll out through lmz_hier_rollout. */
int lmz_rollout(lmz_env *env, int32_t T, const void *actions, int32_t action_dtype,
                float *rewards, uint8_t *dones, void *stream);
int lmz_rollout_dl(lmz_env *env, int32_t T, DLManagedTensor *actions, DLManagedTensor *rewards,
                   DLManagedTensor *dones, void *stream);
/* The same rollout with the rewards written as 1-byte CODES u8 [T][N] -- a reward takes only four values
 * (lmaze_env.py:21-23,109): 0: -0.0, 1: -1.0 (wall), 2: -0.01 (move), 3: 100.0 (goal) -- 2 B instead of 5 B per env-step. */
int lmz_rollout_codes(lmz_env *env, int32_t T, const void *actions, int32_t action_dtype,
                      uint8_t *reward_codes, uint8_t *dones, void *stream);
int lmz_rollout_codes_dl(lmz_env *env, int32_t T, DLManagedTensor *actions, DLManagedTensor *reward_codes,
                         DLManagedTensor *dones, void *stream);

/* Unpacked per-env state, int32 [N][LMZ_ST_COLS] on the device (checkpoint /
 * resume, and how parity tests start both sides from the same state).  For v2 columns
 * 5 and 6 are: layout (1..5), and prev_x | prev_y << 5 | last_action << 10 | action_valid << 15
 * (the position of the previous crop and the action plane of the current obs).
 * lmz_set_state never repairs a row silently: a row the env could not be in (coordinate outside the
 * grid interior, ball on a wall (v0/v3), v3 goal on a wall, reward code / maze / action out of range,
 * negative counters) is clamped so that the kernels stay in bounds AND counted in lmz_stats' error counter. */
/* For v5/v6 the rows are int32 [N][LMZ_ST_COLS_HIER] (see lmz_state_cols). */
int lmz_get_state(lmz_env *env, int32_t *out, void *stream);
int lmz_set_state(lmz_env *env, const int32_t *in, void *stream);
int lmz_get_state_dl(lmz_env *env, DLManagedTensor *out, void *stream);
int lmz_set_state_dl(lmz_env *env, DLManagedTensor *in, void *stream);

/* lmaze-v4 / v5 / v6: the float visit layer state[2] of every env (lmaze_env_v4.py:106-113,211-214; lmaze_env_v5.py:308-312),
 * f32 [N][18][18] on the device -- part of the checkpoint next to lmz_get_state.  The handle itself keeps the layer as
 * its HISTORY (the window centre of every averaging since the reset, 64 bytes per env; DESIGN.md section 3.5) and
 * computes the values from it; lmz_get_visit materialises them.  A layer written with lmz_set_visit has no history:
 * that env averages its layer in memory with the literal full pass until its next reset. */
int lmz_get_visit(lmz_env *env, float *out, void *stream);
int lmz_set_visit(lmz_env *env, const float *in, void *stream);
int lmz_get_visit_dl(lmz_env *env, DLManagedTensor *out, void *stream);
int lmz_set_visit_dl(lmz_env *env, DLManagedTensor *in, void *stream);

/* ---- lmaze-v5 / lmaze-v6: the planner / actor protocol ------------------------------------------
 * reset()             -> lmz_reset: foveal obs into the tensor bound as `obs`      (lmaze_env_v5.py:102-153)
 * plannerStep(goal)   -> lmz_planner_step: local obs into `loc_obs`                (:158-182)
 * step(action)        -> lmz_step: the reference's 8-tuple (:285-292) lands in
 *                          obs (foveal), loc_obs, reward (globalReward), local_reward (originalReward),
 *                          done (globalDone), local_done (localDone), foveal_goal (hot cell of fovealGoal);
 *                          the 8th element is the caller's own action.
 * Actions 0..3 are (+1,0) (-1,0) (0,+1) (0,-1) on (row, col) (:205-217) -- NOT v0's map; other values do not move.
 * With autoreset an env whose globalDone is raised is reset inside the same step: both observation rows
 * then show the new episode (what reset() / buildLocalObservation() would return), the flags and rewards
 * stay the terminal ones, and the caller's next lmz_planner_step mask is local_done | done.
 * Where the reference's buildLocalObservation raises IndexError (the actor is 3 cells right of / below the
 * planner-time fovea, :365-366) the local row is written as zeros, loc_err[i] = 1 and the error counter of
 * lmz_stats is bumped; negative indices wrap exactly like numpy's.
 * lmz_set_window and lmz_step_host are not available for this variant; its rollout is lmz_hier_rollout. */
#define LMZ_ST_COLS_HIER 17   /* x, y, prev_x, prev_y, fovea_x1, fovea_y1, goal_x, goal_y, fgoal_x, fgoal_y, last_x, last_y,
                                 fgoal_action, step_count, foveal_step_count, globalDone | localDone << 1 | layout << 4, episode */
int lmz_state_cols(int32_t variant);                               /* LMZ_ST_COLS, or LMZ_ST_COLS_HIER for v5 */
int lmz_local_obs_shape(int32_t variant, int64_t shape[3]);        /* (4,35,35), lmaze_env_v5.py:357-358 */
/* loc_obs f32 [N,4,35,35] (16-byte aligned; may be NULL), local_reward f32 [N], local_done u8 [N],
 * loc_err u8 [N] (may be NULL), foveal_goal u8 [N] (may be NULL). */
int lmz_bind_local(lmz_env *env, float *loc_obs, float *local_reward, uint8_t *local_done, uint8_t *loc_err,
                   uint8_t *foveal_goal);
int lmz_bind_local_dl(lmz_env *env, DLManagedTensor *loc_obs, DLManagedTensor *local_reward,
                      DLManagedTensor *local_done, DLManagedTensor *loc_err, DLManagedTensor *foveal_goal);
/* plannerStep() for every env whose mask byte is non-zero (mask NULL = all): goals [N] in 0..24 of
 * `goal_dtype` (lmz_action_dtype); out-of-range goals (IndexError in the reference) are clamped and counted. */
int lmz_planner_step(lmz_env *env, const void *goals, int32_t goal_dtype, const uint8_t *mask, void *stream);
int lmz_planner_step_dl(lmz_env *env, DLManagedTensor *goals, DLManagedTensor *mask, void *stream);
/* The same with the mask derived on the device: plannerStep for every env that is WAITING for its planner --
 * localDone is set, or no plannerStep happened since its last reset (which includes envs that auto-reset in the
 * previous step).  This is the loop `if localDone: plannerStep(...)` of a hierarchical agent without a host
 * round trip, and it makes the planner + step pair capturable in a CUDA graph. */
int lmz_planner_step_auto(lmz_env *env, const void *goals, int32_t goal_dtype, void *stream);
int lmz_planner_step_auto_dl(lmz_env *env, DLManagedTensor *goals, void *stream);
/* Host-buffer form of one planner + actor step (the end-to-end call): copies goals and actions H2D, runs
 * lmz_planner_step_auto and lmz_step, copies globalReward / originalReward / globalDone / localDone D2H and waits
 * for the stream.  Observations stay in the bound device tensors. */
int lmz_hier_step_host(lmz_env *env, const void *goals_host, const void *actions_host, int32_t dtype,
                       float *global_reward_host, float *local_reward_host, uint8_t *global_done_host,
                       uint8_t *local_done_host, void *stream);
/* T fused planner + actor steps with no per-step observation (lmaze_env_v5.py:158-292 looped).  One step =
 * plannerStep(goals[t]) for the envs that are waiting for their planner (the device-side mask of
 * lmz_planner_step_auto) followed by step(actions[t]); with autoreset an env whose globalDone is raised is reset.
 * Outputs [T][N]: globalReward, originalReward (f32), globalDone, localDone (u8).  goals and actions are [T][N] of
 * the same dtype, or both NULL: device-side random goals (0..24) and actions (0..3). */
int lmz_hier_rollout(lmz_env *env, int32_t T, const void *goals, const void *actions, int32_t dtype,
                     float *global_rewards, float *local_rewards, uint8_t *global_dones, uint8_t *local_dones,
                     void *stream);
int lmz_hier_rollout_dl(lmz_env *env, int32_t T, DLManagedTensor *goals, DLManagedTensor *actions,
                        DLManagedTensor *global_rewards, DLManagedTensor *local_rewards,
                        DLManagedTensor *global_dones, DLManagedTensor *local_dones, void *stream);

/* lmaze-v6 safeFovealGoal() (lmaze_env_v6.py:505-523): goals_out u8 [N] = a cell 0..24 of the 5x5 window around
 * the ball that is not a wall.  draws NULL => device RNG, exactly uniform over the non-wall cells (the
 * distribution of the reference's rejection loop); else int64 [N][n_draws] are the values its
 * np.random.randint(0, 25) calls would return: the first non-wall one wins, used_out i32 [N] (may be NULL)
 * receives how many were consumed, and goals_out is 255 if none qualified. */
int lmz_safe_goal(lmz_env *env, const int64_t *draws, int32_t n_draws, uint8_t *goals_out, int32_t *used_out,
                  void *stream);
int lmz_safe_goal_dl(lmz_env *env, DLManagedTensor *draws, DLManagedTensor *goals_out, DLManagedTensor *used_out,
                     void *stream);

/* Copies the device counters to out_host[LMZ_NUM_STATS] (synchronises `stream`).
 * *errors_host (may be NULL) receives the number of rejected injected spawns, out-of-range actions
 * (v2/v4/v5), IndexError rows (v5 local obs) and invalid lmz_set_state rows. */
int lmz_stats(lmz_env *env, int64_t *out_host, int64_t *errors_host, void *stream);
int lmz_stats_reset(lmz_env *env, void *stream);

/* Launch bookkeeping for benchmarks: kernels launched by this handle so far. */
int64_t lmz_launch_count(const lmz_env *env);

#ifdef __cplusplus
}
#endif
#endif
