// lmz_kernels.cuh -- sm_100a kernels of the batched LMaze step/reset path.
//
//   lmz_env_tma_kernel  fused reset / step / render: one thread per env does the
//   lmz_env_st_kernel   transition (lmaze_env.py:146-196,246-249; lmaze_env_v3.py:
//                       220-265,398), warp ballots feed the episode statistics, and
//                       the observation (lmaze_env.py:208-234) is emitted either as
//                       bulk async shared->global copies (TMA engine) or as 128-bit
//                       vector stores, both sourced from a template blob that one
//                       cp.async.bulk load stages into shared memory per CTA.
//   lmz_rollout_kernel  T fused steps, state in registers, no per-step obs,
//                       optional device-side Philox actions.
//   lmz_state_kernel    pack / unpack of the per-env state for get/set_state.
//
// Nothing here is GEMM-shaped: the path is a pure HBM streaming write (112,896 B
// per env-step for v0), so tensor cores / TMEM are deliberately unused.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "lmz_variants.h"

// tiles per grab of the small-observation kernels (tools/small_bench.py sweep: compact v0 8.6 -> 9.9 G env-steps/s and
// transition-only 43 -> 116 G with 4; v3 / incremental are instruction-bound and flat)
#ifndef LMZ_G_COMPACT_V0
#define LMZ_G_COMPACT_V0 4
#endif
#ifndef LMZ_G_COMPACT_V3
#define LMZ_G_COMPACT_V3 2
#endif
#ifndef LMZ_G_INCR
#define LMZ_G_INCR 2
#endif

namespace lmz {

enum : int { MODE_STEP = 0, MODE_RESET = 1, MODE_RENDER = 2, MODE_PLANNER = 3 };
enum : int { ACT_U8 = 0, ACT_I32 = 1, ACT_I64 = 2 };
enum : int { RENDER_TMA = 0, RENDER_ST128 = 1, RENDER_INCREMENTAL = 2 };
enum : int { OBS_FULL = 0, OBS_COMPACT = 1, OBS_BITS = 2 };
enum : int {
  STAT_STEPS = 0, STAT_EPISODES, STAT_GOALS, STAT_TIMEOUTS, STAT_WALL_BUMPS, STAT_MOVES, STAT_STALE,
  STAT_EPLEN_SUM, NUM_STATS
};

struct KParams {
  int64_t n;                    // envs in this handle
  int mode;                     // MODE_*
  const void *actions;          // [n] (step) or [T][n] (rollout); may be null in rollout
  int action_dtype;
  const int4 *spawn;            // optional injected spawn: sx, sy, gx, gy
  const uint8_t *mask;          // reset only, optional
  uint32_t *state;              // packed per-env state
  uint32_t *goal_count;         // goalCount per env (v0; lmaze_env.py:24,195)
  uint32_t *episode;            // resets so far (RNG counter)
  float *visit;                 // v4 / v5: state[2] visit layer, f32 [n][18*18] -- holds the layer of envs in DIRECT mode only
  uint8_t *hist;                // v4 / v5: visit history, u8 [n][64]: the window centre of each averaging since the reset
  void *obs;                    // f32 [win_n][C][S][S], or u8 [win_n][C][G][G] (compact), or null
  int64_t win_lo, win_n;        // obs rows hold envs [win_lo, win_lo + win_n)
  int64_t tile_begin, tile_end; // tiles (32 envs) this launch visits
  float *reward;                // [n] or [T][n]
  uint8_t *done;                // [n] or [T][n]
  uint8_t *reward_code;         // rollout only: RC_* codes u8 [T][n] instead of the f32 rewards, or null
  int obs_bits;                 // compact kernel: the observation is the bit-packed form (OBS_BITS)
  const uint8_t *blob;          // template blob in global memory
  unsigned long long *stats;    // [NUM_STATS]
  unsigned int *errors;         // rejected injected spawns
  uint64_t seed, env_id0;
  uint64_t t0;                  // rollout: global index of the first step
  int T;                        // rollout length
  int autoreset, random_ball, random_goal;
  int n_cand;                   // entries in the spawn-candidate table
  int s_cell;                   // linear index of the 'S' cell
  int l2_policy;                // L2_* policy of the obs stores (TMA path)
  unsigned long long *work;     // [2]: next tile to hand out, grabbers finished (self re-arming)
  uint32_t bulk_split;          // 0, or the largest single bulk copy in bytes
  // ---- lmaze-v5 / v6 (planner / actor env, lmz_v5.cuh)
  uint32_t *aux2;               // third packed state word
  void *obs2;                   // local observation f32 [n][4][35][35], or null
  float *reward2;               // originalReward (the actor's reward) [n]
  uint8_t *done2;               // localDone [n]
  uint8_t *loc_err;             // 1 where the reference's buildLocalObservation raises IndexError [n], or null
  uint8_t *fgoal_out;           // hot cell of fovealGoal [n], or null
  int auto_mask;                // plannerStep: act on the envs that are waiting for their planner
  const void *goals;            // v5 rollout: planner goals [T][n] (same dtype as the actions), or null with actions
};

enum : int { L2_EVICT_FIRST = 1, L2_EVICT_NORMAL = 2, L2_EVICT_LAST = 3, L2_NONE = 4 };
constexpr int DEFAULT_L2_POLICY = L2_EVICT_FIRST;   // the obs is streamed out once (sweep: +0.3 % over no hint)

// ------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_addr(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_addr(bar)),
      "r"(parity)
      : "memory");
}
// global -> shared bulk async copy (TMA engine), completion on an mbarrier
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_addr(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_addr(bar))
               : "memory");
}
// shared -> global bulk async copy (TMA engine), tracked by the thread's bulk group
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, uint32_t src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(src_smem),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_s2g_hint(void *dst_gmem, uint32_t src_smem, uint32_t bytes, uint64_t policy) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst_gmem),
               "r"(src_smem), "r"(bytes), "l"(policy)
               : "memory");
}
__device__ __forceinline__ uint64_t make_l2_policy(int kind) {
  uint64_t pol = 0;
  if (kind == L2_EVICT_FIRST) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  else if (kind == L2_EVICT_LAST) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// streaming 128-bit store: the obs is written once and not re-read by this kernel
__device__ __forceinline__ void st_stream_v4(void *p, const uint4 &v) {
  asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
__device__ __forceinline__ uint4 lds_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

// ------------------------------------------------------------------ RNG (spec in DESIGN.md; CPU twin in oracle/)
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

constexpr uint32_t TAG_SPAWN = 0x53u, TAG_ACTION = 0x41u;
constexpr int SPAWN_FORCE = 64;      // added to an injected spawn row's goal_x: the row overrides RANDOM_BALL / RANDOM_GOAL (v3 test mode)

struct WordStream {   // words 4a..4a+3 come from Philox block `a` of (seed, env, episode)
  uint32_t c0, c1, c2, k0, k1, attempt, buf[4];
  int have;
  __device__ __forceinline__ void init(uint64_t seed, uint64_t gid, uint32_t episode) {
    c0 = (uint32_t)gid; c1 = (uint32_t)(gid >> 32); c2 = episode;
    k0 = (uint32_t)seed; k1 = (uint32_t)(seed >> 32); attempt = 0; have = 0;
  }
  __device__ __forceinline__ uint32_t next() {
    if (have == 0) {
      philox4x32_10(c0, c1, c2, (attempt << 8) | TAG_SPAWN, k0, k1, buf);
      attempt += 1; have = 4;
    }
    const int i = 4 - have;
    have -= 1;
    return i == 0 ? buf[0] : i == 1 ? buf[1] : i == 2 ? buf[2] : buf[3];
  }
  // exactly uniform in [0, n): multiply-shift, rejecting the short low range
  __device__ __forceinline__ uint32_t uniform(uint32_t n) {
    const uint32_t thresh = (uint32_t)(0x100000000ull % n);
    for (;;) {
      const uint64_t m = (uint64_t)next() * (uint64_t)n;
      if ((uint32_t)m >= thresh) return (uint32_t)(m >> 32);
    }
  }
};

// ------------------------------------------------------------------ transition
__device__ __forceinline__ long long load_action(const void *base, int dtype, int64_t idx) {
  if (dtype == ACT_U8) return (long long)((const uint8_t *)base)[idx];
  if (dtype == ACT_I32) return (long long)((const int32_t *)base)[idx];
  return ((const long long *)base)[idx];
}

__device__ __forceinline__ uint32_t reward_bits(int rc) {
  // float32 images of the reference's four possible rewards (lmaze_env.py:21-23,109)
  return rc == RC_NEG_ZERO ? 0x80000000u : rc == RC_WALL ? 0xBF800000u : rc == RC_MOVE ? 0xBC23D70Au : 0x42C80000u;
}

struct StepOut {
  int cls;      // branch taken: CLS_W wall, CLS_B move, CLS_X goal, CLS_S none
  bool done;
};

// One reference step() on registers.  `cls` is the G*G cell-class table in shared memory.
template <class V>
__device__ __forceinline__ StepOut transition(EnvRegs &r, long long a, const uint8_t *cls, uint32_t &goal_hits) {
  StepOut o;
  r.step = r.step < V::STEP_SAT ? r.step + 1 : V::STEP_SAT;                 // lmaze_env.py:151
  int ox = 0, oy = 0;                                                       // lmaze_env.py:153-170
  if (a == 0) ox = -1; else if (a == 1) ox = 1; else if (a == 2) oy = -1; else if (a == 3) oy = 1;
  const int t = cls[(r.x + ox) * V::G + (r.y + oy)];
  if (V::ID == 0) {
    if (t == CLS_W) { r.rcode = RC_WALL; }                                   // :172-174
    else if (t == CLS_B) { r.x += ox; r.y += oy; r.rcode = RC_MOVE; }        // :176-184
    else if (t == CLS_X) { r.x += ox; r.y += oy; r.rcode = RC_GOAL; goal_hits += 1; }  // :186-195
    /* CLS_S: no branch -- position and reward keep their previous values */
    o.cls = t;
    o.done = (r.rcode == RC_GOAL) || (r.step == (uint32_t)V::STEP_LIMIT);    // :246-249 (equality)
  } else {
    if (t == CLS_W) { r.rcode = RC_WALL; o.cls = CLS_W; }                    // lmaze_env_v3.py:251-252
    else {                                                                   // :255-265
      r.x += ox; r.y += oy; r.rcode = RC_MOVE; o.cls = CLS_B;
      if (r.x + ox == r.gx && r.y + oy == r.gy) { r.rcode = RC_GOAL; o.cls = CLS_X; }   // look-ahead
    }
    o.done = (r.rcode == RC_GOAL) || (r.step > (uint32_t)V::STEP_LIMIT);     // :398 (strictly greater)
  }
  return o;
}

// reset(): new spawn (injected or device RNG), stepCount 0, reward -0.0
// (lmaze_env.py:70-80,109-110; lmaze_env_v3.py:143-164).
template <class V>
__device__ __forceinline__ void respawn(EnvRegs &r, const KParams &p, int64_t e, uint32_t &episode,
                                        const uint8_t *cls, const uint16_t *cand) {
  int sx, sy, gx = r.gx, gy = r.gy;
  const int s_x = p.s_cell / V::G, s_y = p.s_cell % V::G;
  bool forced = false;
  if (p.spawn) {
    int4 s = p.spawn[e];
    // v3 reset(mode="test") (lmaze_env_v3.py:145-146,154-155): the fixed goal / ball take priority over
    // RANDOM_GOAL / RANDOM_BALL.  The row says so with SPAWN_FORCE added to its goal_x column.
    forced = V::ID == 3 && s.z >= SPAWN_FORCE;
    if (forced) s.z -= SPAWN_FORCE;
    sx = s.x; sy = s.y;
    bool ok = true;
    if (V::ID == 3 && (p.random_goal || forced) && s.z >= 0) {
      const bool gok = s.z >= 1 && s.z <= V::G - 2 && s.w >= 1 && s.w <= V::G - 2 && cls[s.z * V::G + s.w] != CLS_W;
      if (gok) { gx = s.z; gy = s.w; } else ok = false;
    }
    if (p.random_ball || forced) {
      bool bok = sx >= 1 && sx <= V::G - 2 && sy >= 1 && sy <= V::G - 2;
      if (bok) {
        const int c = cls[sx * V::G + sy];
        bok = (V::ID == 0) ? (c != CLS_W && c != CLS_X) : (c != CLS_W && !(sx == gx && sy == gy));
      }
      if (!bok) { ok = false; sx = s_x; sy = s_y; }
    }
    if (!ok) atomicAdd(p.errors, 1u);
  } else {
    WordStream ws;
    ws.init(p.seed, p.env_id0 + (uint64_t)e, episode);
    if (V::ID == 0) {
      const int k = cand[ws.uniform((uint32_t)p.n_cand)];
      sx = k / V::G; sy = k % V::G;
    } else {
      const uint32_t gi = ws.uniform((uint32_t)p.n_cand);
      uint32_t bi = ws.uniform((uint32_t)p.n_cand - 1u);
      if (bi >= gi) bi += 1;
      if (p.random_goal) { gx = cand[gi] / V::G; gy = cand[gi] % V::G; }
      // if the goal is pinned the ball must still avoid it (lmaze_env_v3.py:157)
      sx = cand[bi] / V::G; sy = cand[bi] % V::G;
      if (!p.random_goal && sx == gx && sy == gy) { sx = cand[gi] / V::G; sy = cand[gi] % V::G; }
    }
  }
  if (!p.random_ball && !forced) { sx = s_x; sy = s_y; }                    // lmaze_env.py:82-89
  r.x = sx; r.y = sy; r.gx = gx; r.gy = gy;
  r.step = 0; r.rcode = RC_NEG_ZERO;
  episode += 1;
}

// ------------------------------------------------------------------ fused reset / step / render
// Everything one env does in a fused call except writing its observation.
struct LaneOut {
  uint32_t st;        // packed state after the call
  uint32_t st_old;    // packed state before the call (the incremental render erases its blocks)
  bool render;        // obs row must be (re)written
  bool done;
  int cls;            // branch taken by the transition (-1: no step)
  uint32_t eplen;     // stepCount of an episode that finished in this call
  // what a lane without an env (past the end of the batch) reports
  __device__ static __forceinline__ LaneOut blank() {
    LaneOut o;
    o.st = 0; o.st_old = 0; o.render = false; o.done = false; o.cls = -1; o.eplen = 0;
    return o;
  }
};

// One env of a v0 / v3 tile kernel.  `st_old` and `a` are the env's packed state and action, loaded by the caller (so
// that a kernel can have the loads of several tiles in flight before it needs any of them).
template <class V>
__device__ __forceinline__ LaneOut tile_lane(const KParams &p, int64_t e, uint32_t st_old, long long a,
                                             const uint8_t *cls, const uint16_t *cand) {
  LaneOut o = LaneOut::blank();
  o.st_old = st_old;
  EnvRegs r = V::unpack(o.st_old);
  bool reset_now = false;
  if (p.mode == MODE_STEP) {
    uint32_t hits = 0;
    const StepOut so = transition<V>(r, a, cls, hits);
    if (V::ID == 0 && hits) p.goal_count[e] += hits;
    o.done = so.done; o.cls = so.cls;
    p.reward[e] = __uint_as_float(reward_bits(r.rcode));
    p.done[e] = so.done ? 1 : 0;
    if (so.done) o.eplen = r.step;
    reset_now = so.done && p.autoreset;
    o.render = true;
  } else if (p.mode == MODE_RESET) {
    reset_now = (p.mask == nullptr) || (p.mask[e] != 0);
    o.render = reset_now;
  } else {
    o.render = true;
  }
  if (reset_now) {
    uint32_t ep = p.episode[e];
    respawn<V>(r, p, e, ep, cls, cand);
    p.episode[e] = ep;
  }
  o.st = V::pack(r);
  if (p.mode != MODE_RENDER) p.state[e] = o.st;
  o.render = o.render && p.obs != nullptr && e >= p.win_lo && e < p.win_lo + p.win_n;   // render window
  return o;
}

// Latency-tolerant tile pipeline of the small-observation kernels (compact, incremental, transition-only).
// Under a saturated write stream a global load or atomic takes several microseconds, and a warp that
// grabs a tile, loads its 32 states and only then works is bound by that chain (ncu: long_scoreboard is
// the top stall, ~17 us per tile per warp).  So every warp grabs GROUPS of G consecutive tiles with ONE
// atomic, keeps the loads of a whole group in flight, and runs two groups ahead: the group being
// rendered was loaded one iteration ago and grabbed two iterations ago.
template <int G>
struct TileGroup {
  uint32_t st[G];
  int act[G];           // action, clamped to 0..255 (anything outside 0..3 is the same no-op)
};
template <int G>
__device__ __forceinline__ void preload_group(const KParams &p, int64_t tile0, int lane, int64_t tiles, TileGroup<G> &g) {
#pragma unroll
  for (int k = 0; k < G; ++k) {
    const int64_t e = (tile0 + k) * 32 + lane;
    g.st[k] = 0; g.act[k] = 255;
    if (tile0 + k < tiles && e < p.n) {
      g.st[k] = p.state[e];
      if (p.mode == MODE_STEP) {
        const long long a = load_action(p.actions, p.action_dtype, e);
        g.act[k] = (a < 0 || a > 255) ? 255 : (int)a;
      }
    }
  }
}
// Episode statistics of one warp: a ballot + popc per counter (the counts are warp-uniform
// registers), a shuffle reduction for the episode-length sum, one atomicAdd per counter at the end.
struct WarpStats {
  uint32_t steps = 0, ep = 0, goal = 0, wall = 0, move = 0, stale = 0;
  unsigned long long len = 0;
  __device__ __forceinline__ void add(bool valid, const LaneOut &o) {
    steps += __popc(__ballot_sync(0xffffffffu, valid && o.cls >= 0));
    ep += __popc(__ballot_sync(0xffffffffu, valid && o.done));
    goal += __popc(__ballot_sync(0xffffffffu, valid && o.done && o.cls == CLS_X));
    wall += __popc(__ballot_sync(0xffffffffu, valid && o.cls == CLS_W));
    move += __popc(__ballot_sync(0xffffffffu, valid && (o.cls == CLS_B || o.cls == CLS_X)));
    stale += __popc(__ballot_sync(0xffffffffu, valid && o.cls == CLS_S));
    if (valid) len += o.eplen;
  }
  __device__ __forceinline__ void flush(unsigned long long *stats, int lane) {
    unsigned long long v = len;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    if (lane != 0 || steps == 0) return;
    atomicAdd(&stats[STAT_STEPS], (unsigned long long)steps);
    if (ep) {
      atomicAdd(&stats[STAT_EPISODES], (unsigned long long)ep);
      if (ep - goal) atomicAdd(&stats[STAT_TIMEOUTS], (unsigned long long)(ep - goal));
      atomicAdd(&stats[STAT_EPLEN_SUM], v);
    }
    if (goal) atomicAdd(&stats[STAT_GOALS], (unsigned long long)goal);
    if (wall) atomicAdd(&stats[STAT_WALL_BUMPS], (unsigned long long)wall);
    if (move) atomicAdd(&stats[STAT_MOVES], (unsigned long long)move);
    if (stale) atomicAdd(&stats[STAT_STALE], (unsigned long long)stale);
  }
};

// Stage the template blob (static channels, zero rows, band table, cell classes, spawn
// candidates) with ONE bulk async load; the TMA engine signals the mbarrier.
template <class V>
__device__ __forceinline__ void stage_blob(unsigned char *smem, uint64_t *bar, const uint8_t *blob) {
  if (threadIdx.x == 0) { mbar_init(bar, 1); fence_mbar_init(); }
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, V::BLOB_BYTES);
    bulk_g2s(smem, blob, V::BLOB_BYTES, bar);
  }
  mbar_wait(bar, 0);
}

// Dynamic work distribution.  A B200's SMs do NOT get equal shares of a saturated write path
// (tools/wbench.cu: with a static env->SM split the first SM finishes ~5 ms of 16 ms before the
// last and the chip averages 6.4 TB/s; with tiles handed out by an atomic counter the spread is
// 0.02 ms and the same copies reach 7.5 TB/s).  So tiles of 32 consecutive envs are grabbed from
// work[0]; work[1] counts finished grabbers and the last one re-arms both for the next launch
// (self-contained, so the launch is also safe to replay from a CUDA graph).
__device__ __forceinline__ int64_t grab_tiles(unsigned long long *work, int count) {
  return (int64_t)atomicAdd(&work[0], (unsigned long long)count);
}
// Lane 0 grabs `count` consecutive tiles for the whole warp; every lane gets the first one's index.
__device__ __forceinline__ int64_t warp_grab(const KParams &p, int lane, int count) {
  int64_t t = 0;
  if (lane == 0) t = p.tile_begin + grab_tiles(p.work, count);
  return __shfl_sync(0xffffffffu, t, 0);
}
// The same grab as inline PTX: the compiler aggregates a result-returning atomicAdd across the warp and broadcasts the
// result with a shuffle RIGHT BEHIND the atomic, which makes every grab synchronous; this form lets the result be
// touched a tile later (lane 0 calls it alone).
__device__ __forceinline__ int64_t grab_tile_async(unsigned long long *work) {
  unsigned long long r;
  asm volatile("atom.global.add.u64 %0, [%1], 1;" : "=l"(r) : "l"(work) : "memory");
  return (int64_t)r;
}
__device__ __forceinline__ void finish_grabber(unsigned long long *work, unsigned long long grabbers) {
  __threadfence();
  if (atomicAdd(&work[1], 1ull) == grabbers - 1) { work[0] = 0; work[1] = 0; }
}

// ---- render path 1: the TMA engine writes the observation ------------------------------------
// Warp-granular: each lane owns one env of the warp's 32-env tile.  The loop is software
// pipelined: the NEXT tile is grabbed and its transitions (loads, table lookups, stores) run
// while the TMA engine is still draining the copies issued for the previous tile; then lane 0
// issues, env by env, one cp.async.bulk shared->global copy per blob segment.
template <class V, int THREADS>
__global__ void __launch_bounds__(THREADS, 1) lmz_env_tma_kernel(const KParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar;
  constexpr int WARPS = THREADS / 32;
  const int lane = threadIdx.x & 31;
  stage_blob<V>(smem, &bar, p.blob);
  const uint8_t *cls = smem + V::CLS_OFF;
  const uint16_t *cand = reinterpret_cast<const uint16_t *>(smem + V::CAND_OFF);
  const uint32_t blob_s = smem_addr(smem);
  const uint64_t l2pol = (p.l2_policy != L2_NONE) ? make_l2_policy(p.l2_policy) : 0;
  const int64_t tiles = p.tile_end;
  WarpStats ws;

  auto step_tile = [&](int64_t tl, bool &valid) {        // this lane's env of tile `tl`: load, step, count
    const int64_t e = tl * 32 + lane;
    valid = tl < tiles && e < p.n;
    LaneOut o = LaneOut::blank();
    if (valid) {
      const uint32_t st = p.state[e];
      const long long a = (p.mode == MODE_STEP) ? load_action(p.actions, p.action_dtype, e) : 0;
      o = tile_lane<V>(p, e, st, a, cls, cand);
    }
    if (p.mode == MODE_STEP) ws.add(valid, o);
    return o;
  };
  int64_t tile = warp_grab(p, lane, 1);
  bool valid;
  LaneOut o = step_tile(tile, valid);
  while (tile < tiles) {
    const int64_t ntile = warp_grab(p, lane, 1);
    bool nvalid;
    const LaneOut no = step_tile(ntile, nvalid);
    // ---- observation render (lmaze_env.py:208-234): the env's image is NSEG blob segments
    unsigned rmask = __ballot_sync(0xffffffffu, valid && o.render);
    while (rmask) {
      const int l = __ffs(rmask) - 1;
      rmask &= rmask - 1;
      const uint32_t s = __shfl_sync(0xffffffffu, o.st, l);
      if (lane == 0) {
        unsigned char *dst = reinterpret_cast<unsigned char *>(p.obs) + (size_t)(tile * 32 + l - p.win_lo) * V::OBS_BYTES;
        Seg sg[V::NSEG];
        V::segments(V::unpack(s), sg);
#pragma unroll
        for (int k = 0; k < V::NSEG; ++k) {
          uint32_t off = 0, left = sg[k].len;
          while (left) {
            const uint32_t len = (p.bulk_split && left > p.bulk_split) ? p.bulk_split : left;
            if (p.l2_policy != L2_NONE) bulk_s2g_hint(dst + sg[k].dst + off, blob_s + sg[k].src + off, len, l2pol);
            else bulk_s2g(dst + sg[k].dst + off, blob_s + sg[k].src + off, len);
            off += len; left -= len;
          }
        }
      }
    }
    tile = ntile; o = no; valid = nvalid;
  }
  // the blob must outlive every copy that reads it; wait_group 0 also covers the global writes
  bulk_commit();
  bulk_wait_all();
  if (p.mode == MODE_STEP) ws.flush(p.stats, lane);
  if (lane == 0) finish_grabber(p.work, (unsigned long long)gridDim.x * WARPS);
}

// ---- render path 2: 128-bit vector stores -----------------------------------------------------
// CTA-cooperative.  Warp 0 grabs a 32-env tile and runs its transitions (one env per lane),
// parking the packed states in shared memory; then ALL threads copy the tile's observations env
// by env with LDS.128 -> st.global.cs.v4 (consecutive threads, consecutive 16-byte words) while
// warp 0 is already working on the next tile (double-buffered, one __syncthreads per tile).
template <class V, int THREADS>
__global__ void __launch_bounds__(THREADS, 1) lmz_env_st_kernel(const KParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t s_st[2][32];
  __shared__ long long s_tile[2];
  constexpr uint32_t NO_RENDER = 0xffffffffu;           // not a packable state (x would be 31)
  constexpr uint32_t OBS16 = V::OBS_BYTES / 16;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  stage_blob<V>(smem, &bar, p.blob);
  const uint8_t *cls = smem + V::CLS_OFF;
  const uint16_t *cand = reinterpret_cast<const uint16_t *>(smem + V::CAND_OFF);
  const uint32_t blob_s = smem_addr(smem);
  const int64_t tiles = p.tile_end;
  WarpStats ws;

  auto produce = [&](int buf) {                          // warp 0 only
    const int64_t t = warp_grab(p, lane, 1), e = t * 32 + lane;
    const bool valid = t < tiles && e < p.n;
    LaneOut o = LaneOut::blank();
    if (valid) {
      const uint32_t st = p.state[e];
      const long long a = (p.mode == MODE_STEP) ? load_action(p.actions, p.action_dtype, e) : 0;
      o = tile_lane<V>(p, e, st, a, cls, cand);
    }
    if (p.mode == MODE_STEP) ws.add(valid, o);
    s_st[buf][lane] = (valid && o.render) ? o.st : NO_RENDER;
    if (lane == 0) s_tile[buf] = t;
  };
  if (warp == 0) produce(0);
  for (int buf = 0;; buf ^= 1) {
    __syncthreads();                                     // s_st[buf] ready; s_st[buf^1] free again
    const int64_t tile = s_tile[buf];
    if (tile >= tiles) break;
    if (warp == 0) produce(buf ^ 1);
    for (int k = 0; k < 32; ++k) {
      const uint32_t s = s_st[buf][k];
      if (s == NO_RENDER) continue;
      unsigned char *dst = reinterpret_cast<unsigned char *>(p.obs) + (size_t)(tile * 32 + k - p.win_lo) * V::OBS_BYTES;
      Seg sg[V::NSEG];
      V::segments(V::unpack(s), sg);
      // 16-byte word f of the obs comes from blob byte 16*f + delta[q], q = the segment holding f
      uint32_t bnd[V::NSEG];
      int32_t delta[V::NSEG];
#pragma unroll
      for (int q = 0; q < V::NSEG; ++q) { bnd[q] = sg[q].dst >> 4; delta[q] = (int32_t)sg[q].src - (int32_t)sg[q].dst; }
      auto src_of = [&](uint32_t f) {
        int32_t d = delta[0];
#pragma unroll
        for (int q = 1; q < V::NSEG; ++q) d = (f >= bnd[q]) ? delta[q] : d;
        return blob_s + (uint32_t)((int32_t)(f << 4) + d);
      };
      uint32_t f = tid;
      for (; f + 3 * THREADS < OBS16; f += 4 * THREADS) {     // 4 independent 16-byte moves in flight
        const uint4 v0 = lds_v4(src_of(f)), v1 = lds_v4(src_of(f + THREADS));
        const uint4 v2 = lds_v4(src_of(f + 2 * THREADS)), v3 = lds_v4(src_of(f + 3 * THREADS));
        st_stream_v4(dst + ((size_t)f << 4), v0);
        st_stream_v4(dst + ((size_t)(f + THREADS) << 4), v1);
        st_stream_v4(dst + ((size_t)(f + 2 * THREADS) << 4), v2);
        st_stream_v4(dst + ((size_t)(f + 3 * THREADS) << 4), v3);
      }
      for (; f < OBS16; f += THREADS) st_stream_v4(dst + ((size_t)f << 4), lds_v4(src_of(f)));
    }
  }
  if (warp == 0) {
    if (p.mode == MODE_STEP) ws.flush(p.stats, lane);
    if (lane == 0) finish_grabber(p.work, (unsigned long long)gridDim.x);
  }
}

// ---- render path 3: compact observation (u8, un-expanded layers) -------------------------------
// obs_mode OBS_COMPACT: the env's observation is written as uint8 [C][G][G] -- the reference's
// `state` layers before its xE upsample (lmaze_env.py:208-215) -- 576 B (v0) / 972 B (v3) per env
// instead of 112,896 / 62,208.  The reference image is exactly repeat_interleave(compact, E) on both
// axes.  Small CTAs (hardware-scheduled), one warp per 32-env tile, one thread per env for the
// transition; the tile's compact rows are then stored row by row as 32-bit words, lanes on
// consecutive words (coalesced 128 B per warp store), static words held in registers.
template <class V, int THREADS>
__global__ void __launch_bounds__(THREADS) lmz_env_compact_kernel(const KParams p) {
  __shared__ __align__(16) unsigned char tab[V::TABLES_BYTES];
  constexpr int WARPS = THREADS / 32;
  constexpr uint32_t W = V::COMPACT_BYTES / 4;           // 32-bit words per env (v0 144, v3 243)
  constexpr int K = (W + 31) / 32;
  const int lane = threadIdx.x & 31;
  for (uint32_t i = threadIdx.x; i < V::TABLES_BYTES / 4; i += THREADS)
    reinterpret_cast<uint32_t *>(tab)[i] = reinterpret_cast<const uint32_t *>(p.blob + V::TABLES_OFF)[i];
  __syncthreads();
  const uint8_t *cls = tab;
  const uint16_t *cand = reinterpret_cast<const uint16_t *>(tab + (V::CAND_OFF - V::TABLES_OFF));
  const uint32_t *tmpl = reinterpret_cast<const uint32_t *>(tab + (V::COMPACT_OFF - V::TABLES_OFF));
  // Lane l owns words l, l+32, l+64, ... of EVERY env row: the static layer words live in registers,
  // and per env the only per-word work is "does this word hold the env's hot byte?" + one store.
  uint32_t base[K];
#pragma unroll
  for (int k = 0; k < K; ++k) base[k] = (lane + 32 * k < (int)W) ? tmpl[lane + 32 * k] : 0u;
  const int64_t tiles = p.tile_end;
  WarpStats ws;
  // persistent warps; groups of G tiles handed out dynamically, two groups ahead (see TileGroup)
  constexpr int G = (V::ID == 0) ? LMZ_G_COMPACT_V0 : LMZ_G_COMPACT_V3;
  int64_t t0 = warp_grab(p, lane, G), t1 = warp_grab(p, lane, G);
  TileGroup<G> pre;
  preload_group<G>(p, t0, lane, tiles, pre);
  while (t0 < tiles) {
    const int64_t t2 = warp_grab(p, lane, G);                 // needed two iterations from now
    uint32_t st[G];
    unsigned rmask[G];
#pragma unroll
    for (int k = 0; k < G; ++k) {                    // transitions of the group loaded one iteration ago
      const int64_t e = (t0 + k) * 32 + lane;
      const bool valid = t0 + k < tiles && e < p.n;
      LaneOut o = LaneOut::blank();
      if (valid) o = tile_lane<V>(p, e, pre.st[k], pre.act[k], cls, cand);
      if (p.mode == MODE_STEP) ws.add(valid, o);
      st[k] = o.st;
      rmask[k] = __ballot_sync(0xffffffffu, valid && o.render);
    }
    preload_group<G>(p, t1, lane, tiles, pre);       // next group's loads fly while this group's rows are stored
    if (p.obs_bits) {
      // bit-packed rows (OBS_BITS): BW words per env, the tile's 32 rows are ONE flat run of 32 * BW words; lane l
      // stores words l, l+32, ... of the run (coalesced), each the static template word with the env's hot bit(s)
      constexpr uint32_t BW = V::BITS_WORDS;
      const uint32_t *btmpl = reinterpret_cast<const uint32_t *>(tab + (V::BITS_OFF - V::TABLES_OFF));
#pragma unroll
      for (int k = 0; k < G; ++k) {
        if (!rmask[k]) continue;
        uint32_t hot[V::NHOT];
        V::hot_bytes(V::unpack(st[k]), hot);
        uint32_t *dst = reinterpret_cast<uint32_t *>(p.obs) + ((t0 + k) * 32 - p.win_lo) * (int64_t)BW;
#pragma unroll
        for (uint32_t j = 0; j < BW; ++j) {
          const uint32_t w = lane + 32 * j, env = w / BW, kk = w - env * BW;
          uint32_t v = btmpl[kk];
#pragma unroll
          for (int q = 0; q < V::NHOT; ++q) {
            const uint32_t h = __shfl_sync(0xffffffffu, hot[q], env);
            v |= ((h >> 5) == kk) ? (1u << (h & 31)) : 0u;
          }
          if ((rmask[k] >> env) & 1u) __stcs(dst + w, v);
        }
      }
      t0 = t1; t1 = t2;
      continue;
    }
#pragma unroll
    for (int k = 0; k < G; ++k) {
      if (!rmask[k]) continue;
      uint32_t hot[V::NHOT];
      V::hot_bytes(V::unpack(st[k]), hot);
      uint32_t *dst = reinterpret_cast<uint32_t *>(p.obs) + (size_t)((t0 + k) * 32 - p.win_lo) * W;
      for (unsigned m = rmask[k]; m; m &= m - 1) {
        const int env = __ffs(m) - 1;
        uint32_t h[V::NHOT];
#pragma unroll
        for (int q = 0; q < V::NHOT; ++q) h[q] = __shfl_sync(0xffffffffu, hot[q], env);
        uint32_t *row = dst + (size_t)env * W;
#pragma unroll
        for (int kk = 0; kk < K; ++kk) {
          const uint32_t w = lane + 32 * kk;
          uint32_t v = base[kk];
#pragma unroll
          for (int q = 0; q < V::NHOT; ++q) v |= ((h[q] >> 2) == w) ? (1u << (8 * (h[q] & 3))) : 0u;
          if (w < W) __stcs(row + w, v);
        }
      }
    }
    t0 = t1; t1 = t2;
  }
  if (p.mode == MODE_STEP) ws.flush(p.stats, lane);
  if (lane == 0) finish_grabber(p.work, (unsigned long long)gridDim.x * WARPS);
}

// ---- render path 4: incremental patches into a persistent observation ---------------------------
// LMZ_RENDER_INCREMENTAL.  The bound obs tensor persists between calls, and a step changes at most
// the ball's ExE block (v3: also the goal block, on a reset): walls / goal / blank channels never
// change (lmaze_env.py:92-107), and ch0 is one block of ones on a zero plane.  So once the tensor
// holds a full render, a step only has to erase the old block and draw the new one -- 2*E*E floats
// (392 B for v0) instead of 112,896 B, with the tensor bit-identical to a full re-render afterwards.
// The host only selects this kernel for MODE_STEP and only while the tensor is known to be in sync
// (after a full reset / render through the same handle); otherwise it falls back to the full render.
// One thread per env for the transition; then, env by env, the warp rewrites the sectors around the old
// and the new block in ONE pass of E iterations (half-warp per block, no per-element divide).
template <class V, int THREADS>
__global__ void __launch_bounds__(THREADS) lmz_env_incr_kernel(const KParams p) {
  __shared__ __align__(16) unsigned char tab[V::TABLES_BYTES];
  constexpr int WARPS = THREADS / 32;
  constexpr int NBLK = (V::ID == 0) ? 1 : 2;                // v0: ball in ch0; v3: ball in ch1, goal in ch2
  const int lane = threadIdx.x & 31;
  for (uint32_t i = threadIdx.x; i < V::TABLES_BYTES / 4; i += THREADS)
    reinterpret_cast<uint32_t *>(tab)[i] = reinterpret_cast<const uint32_t *>(p.blob + V::TABLES_OFF)[i];
  __syncthreads();
  const uint8_t *cls = tab;
  const uint16_t *cand = reinterpret_cast<const uint16_t *>(tab + (V::CAND_OFF - V::TABLES_OFF));
  const int64_t tiles = p.tile_end;
  WarpStats ws;
  // block b of a packed state: channel and top-left element
  auto block_of = [](uint32_t st, int b, int &ch, int &row, int &col) {
    const EnvRegs r = V::unpack(st);
    if (V::ID == 0) { ch = 0; row = r.x * V::E; col = r.y * V::E; }
    else if (b == 0) { ch = 1; row = r.x * V::E; col = r.y * V::E; }
    else { ch = 2; row = r.gx * V::E; col = r.gy * V::E; }
  };
  constexpr int G = LMZ_G_INCR;
  int64_t t0 = warp_grab(p, lane, G), t1 = warp_grab(p, lane, G);
  TileGroup<G> pre;
  preload_group<G>(p, t0, lane, tiles, pre);
  while (t0 < tiles) {
    const int64_t t2 = warp_grab(p, lane, G);
    uint32_t st_new[G], st_old[G];
    unsigned mmask[G];
#pragma unroll
    for (int k = 0; k < G; ++k) {
      const int64_t e = (t0 + k) * 32 + lane;
      const bool valid = t0 + k < tiles && e < p.n;
      LaneOut o = LaneOut::blank();
      if (valid) o = tile_lane<V>(p, e, pre.st[k], pre.act[k], cls, cand);
      ws.add(valid, o);
      // which envs of the tile have a block that moved?
      bool moved = false;
      if (valid && o.render) {
#pragma unroll
        for (int b = 0; b < NBLK; ++b) {
          int c0, r0, q0, c1, r1, q1;
          block_of(o.st_old, b, c0, r0, q0); block_of(o.st, b, c1, r1, q1);
          moved = moved || r0 != r1 || q0 != q1;
        }
      }
      st_new[k] = o.st; st_old[k] = o.st_old;
      mmask[k] = __ballot_sync(0xffffffffu, moved);
    }
    preload_group<G>(p, t1, lane, tiles, pre);
#pragma unroll
    for (int k = 0; k < G; ++k) {
      for (unsigned m = mmask[k]; m; m &= m - 1) {
        const int l = __ffs(m) - 1;
        const uint32_t so = __shfl_sync(0xffffffffu, st_old[k], l), sn = __shfl_sync(0xffffffffu, st_new[k], l);
        float *img = reinterpret_cast<float *>(p.obs) + (size_t)((t0 + k) * 32 + l - p.win_lo) * (V::OBS_BYTES / 4);
#pragma unroll
        for (int b = 0; b < NBLK; ++b) {
          int ch, r0, q0, r1, q1;
          block_of(so, b, ch, r0, q0); block_of(sn, b, ch, r1, q1);
          if (r0 == r1 && q0 == q1) continue;
          // The plane holds ONE block of ones, so every element's value follows from the new position.  Rewrite
          // whole aligned 32-byte sectors around the old and the new block (values computed, not read): full-sector
          // writes need no read-modify-write in L2/DRAM, and where the two regions share a sector both write the
          // same values.  ONE loop covers both blocks.  A sector may reach into the neighbouring row; those floats lie in
          // the maze's border columns, which a block never touches (the border cells are walls), so "column relative
          // to this row" decides the value with no divide.
          float *plane = img + (size_t)ch * V::S * V::S;            // 32-byte aligned (plane = 28,224 / 20,736 B)
          auto put = [&](int brow, int rr, int bcol, int width, int q) {
            const int first = (brow + rr) * V::S + bcol;            // the row segment [first, first + width)
            const int lo = first & ~7, hi = (first + width + 7) & ~7;
            const int e = lo + 4 * q;
            if (e < hi) {
              const int c = e - first + bcol;                       // column of the float4's first float (may run over: border)
              const bool row_in = (unsigned)(brow + rr - r1) < (unsigned)V::E;
              float4 v;
              v.x = (row_in && (unsigned)(c - q1) < (unsigned)V::E) ? 1.0f : 0.0f;
              v.y = (row_in && (unsigned)(c + 1 - q1) < (unsigned)V::E) ? 1.0f : 0.0f;
              v.z = (row_in && (unsigned)(c + 2 - q1) < (unsigned)V::E) ? 1.0f : 0.0f;
              v.w = (row_in && (unsigned)(c + 3 - q1) < (unsigned)V::E) ? 1.0f : 0.0f;
              *reinterpret_cast<float4 *>(plane + e) = v;
            }
          };
          if (r0 == r1 && (q0 - q1 == V::E || q1 - q0 == V::E)) {
            // a one-cell move along the row: the two blocks are side by side -- ONE box of E rows x 2E floats
            // (<= 24 floats = 6 float4s per row, 8 lanes per row): a third fewer sectors than two separate boxes,
            // and the step is bound by the number of scattered 32-byte sectors it writes
            const int bcol = q0 < q1 ? q0 : q1;
#pragma unroll
            for (int it = 0; it < (V::E * 8 + 31) / 32; ++it) {
              const int idx = it * 32 + lane, rr = idx >> 3;
              if (rr < V::E) put(r0, rr, bcol, 2 * V::E, idx & 7);
            }
          } else {
            // 2 * E rows (E of the old block, then E of the new one), each a span of <= 16 floats = <= 4 float4s:
            // 4 lanes per row, 8 rows per warp pass
#pragma unroll
            for (int it = 0; it < (2 * V::E * 4 + 31) / 32; ++it) {
              const int idx = it * 32 + lane, rid = idx >> 2;
              const bool nw = rid >= V::E;                          // this row belongs to the new block
              if (rid < 2 * V::E) put(nw ? r1 : r0, nw ? rid - V::E : rid, nw ? q1 : q0, V::E, idx & 3);
            }
          }
        }
      }
    }
    t0 = t1; t1 = t2;
  }
  ws.flush(p.stats, lane);
  if (lane == 0) finish_grabber(p.work, (unsigned long long)gridDim.x * WARPS);
}

// ------------------------------------------------------------------ T-step rollout, no per-step obs
// One thread per env, state in registers for all T steps.  This kernel is issue-bound, not
// HBM-bound (5.25 B of output per env-step), so the per-step path is kept to a few dozen
// instructions: linear cell index + delta, branch-free move / reward code (CLS_* + 1 == RC_*),
// reward bits from a 4-entry constant table, pointer-bumped [T][N] stores, and the next spawn
// drawn ONCE before the loop so the divergent Philox path only runs when an env finishes a
// second episode inside the same rollout.
__constant__ uint32_t c_reward_bits[4] = {0x80000000u, 0xBF800000u, 0xBC23D70Au, 0x42C80000u};

template <class V>
__device__ __forceinline__ void draw_spawn(const KParams &p, uint64_t gid, uint32_t episode, const uint16_t *cand,
                                           int &ball, int &goal) {
  WordStream ws;
  ws.init(p.seed, gid, episode);
  if (V::ID == 0) {
    ball = cand[ws.uniform((uint32_t)p.n_cand)];
    goal = -1;
  } else {
    const uint32_t gi = ws.uniform((uint32_t)p.n_cand);
    uint32_t bi = ws.uniform((uint32_t)p.n_cand - 1u);
    if (bi >= gi) bi += 1;
    goal = cand[gi]; ball = cand[bi];
  }
}

template <class V, int THREADS>
__global__ void __launch_bounds__(THREADS, 3) lmz_rollout_kernel(const KParams p) {
  __shared__ uint8_t cls[V::G * V::G];
  __shared__ uint16_t cand[V::MAX_CAND];
  __shared__ unsigned long long blk_stats[NUM_STATS];
  for (int i = threadIdx.x; i < V::G * V::G; i += THREADS) cls[i] = p.blob[V::CLS_OFF + i];
  for (int i = threadIdx.x; i < V::MAX_CAND; i += THREADS)
    cand[i] = reinterpret_cast<const uint16_t *>(p.blob + V::CAND_OFF)[i];
  if (threadIdx.x < NUM_STATS) blk_stats[threadIdx.x] = 0;
  __syncthreads();

  uint32_t c_ep = 0, c_goal = 0, c_wall = 0, c_stale = 0, c_steps = 0;
  unsigned long long c_len = 0;
  const uint32_t k0 = (uint32_t)p.seed, k1 = (uint32_t)(p.seed >> 32);
  const bool fast_spawn = p.autoreset && p.spawn == nullptr && p.random_ball && (V::ID == 0 || p.random_goal);

  for (int64_t e = (int64_t)blockIdx.x * THREADS + threadIdx.x; e < p.n; e += (int64_t)gridDim.x * THREADS) {
    EnvRegs r = V::unpack(p.state[e]);
    uint32_t ep = p.episode[e];
    uint32_t hits = 0;
    const uint64_t gid = p.env_id0 + (uint64_t)e;
    int pos = r.x * V::G + r.y, gpos = r.gx * V::G + r.gy, rcode = r.rcode;
    uint32_t step = r.step;
    int nball = 0, ngoal = 0;
    bool have_next = false;
    if (fast_spawn) { draw_spawn<V>(p, gid, ep, cand, nball, ngoal); have_next = true; }
    float *rp = p.reward + e;
    uint8_t *dp = p.done + e;
    uint8_t *cp = p.reward_code + e;    // (only dereferenced when reward codes were asked for)
    // action source: a [T][N] buffer, or Philox (one block = 64 two-bit actions, consumed 2 bits a step)
    uint32_t w[4] = {0, 0, 0, 0}, cur = 0;
    int left = 0;                       // actions left in `cur`
    uint64_t tg = p.t0;
    constexpr int CH = 8;               // caller-supplied actions are fetched CH steps ahead (independent loads)
    long long abuf[CH];
    for (int t = 0; t < p.T; ++t, ++tg, rp += p.n, dp += p.n, cp += p.n) {
      int d;                            // linear offset of the move: -G, +G, -1, +1 or 0 (lmaze_env.py:153-170)
      if (p.actions) {
        if ((t & (CH - 1)) == 0) {
#pragma unroll
          for (int k = 0; k < CH; ++k)
            abuf[k] = (t + k < p.T) ? load_action(p.actions, p.action_dtype, (int64_t)(t + k) * p.n + e) : 0;
        }
        long long a = abuf[0];
#pragma unroll
        for (int k = 1; k < CH; ++k) a = ((t & (CH - 1)) == k) ? abuf[k] : a;
        d = a == 0 ? -V::G : a == 1 ? V::G : a == 2 ? -1 : a == 3 ? 1 : 0;
      } else {
        if (left == 0) {
          const uint32_t slot = (uint32_t)(tg & 63);
          if (slot == 0 || t == 0) {
            const uint64_t blk = tg >> 6;
            philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)blk,
                          ((uint32_t)(blk >> 32) << 8) | TAG_ACTION, k0, k1, w);
          }
          const uint32_t wi = slot >> 4;
          cur = (wi == 0 ? w[0] : wi == 1 ? w[1] : wi == 2 ? w[2] : w[3]) >> (2 * (slot & 15));
          left = 16 - (int)(slot & 15);
        }
        const uint32_t a = cur & 3u;
        cur >>= 2; left -= 1;
        d = (a & 2u) ? ((a & 1u) ? 1 : -1) : ((a & 1u) ? V::G : -V::G);
      }
      step = step < V::STEP_SAT ? step + 1 : V::STEP_SAT;
      const int tcls = cls[pos + d];
      bool done;
      int branch;                       // CLS_W wall, CLS_B move, CLS_X goal, CLS_S none
      if (V::ID == 0) {
        // W: stay, -1 | B: move, -0.01 | X: move, 100 | S: nothing, reward kept (lmaze_env.py:172-196)
        pos += (tcls == CLS_B || tcls == CLS_X) ? d : 0;
        rcode = (tcls == CLS_S) ? rcode : tcls + 1;
        hits += (tcls == CLS_X);
        branch = tcls;
        done = (rcode == RC_GOAL) || (step == (uint32_t)V::STEP_LIMIT);
      } else {
        // W: stay, -1 | else move, -0.01, and 100 if one more step would reach the goal (lmaze_env_v3.py:251-265)
        const bool wall = tcls == CLS_W;
        pos += wall ? 0 : d;
        const bool goal = !wall && (pos + d == gpos);
        rcode = wall ? RC_WALL : goal ? RC_GOAL : RC_MOVE;
        branch = wall ? CLS_W : goal ? CLS_X : CLS_B;
        done = goal || (step > (uint32_t)V::STEP_LIMIT);
      }
      if (p.reward_code) __stcs(cp, (uint8_t)rcode);               // 1 B instead of 4: the reward takes four values
      else __stcs(rp, __uint_as_float(c_reward_bits[rcode]));
      __stcs(dp, (uint8_t)(done ? 1 : 0));
      c_wall += (branch == CLS_W); c_stale += (branch == CLS_S);
      if (done) {
        c_ep += 1; c_len += step; c_goal += (branch == CLS_X);
        if (p.autoreset) {
          if (have_next) {              // the pre-drawn spawn of episode `ep`
            pos = nball; if (V::ID == 3) gpos = ngoal;
            step = 0; rcode = RC_NEG_ZERO; ep += 1; have_next = false;
          } else {                      // slow path: injected spawns, pinned ball/goal, or a 2nd reset in this rollout
            r.x = pos / V::G; r.y = pos % V::G; r.gx = gpos / V::G; r.gy = gpos % V::G; r.step = step; r.rcode = rcode;
            respawn<V>(r, p, e, ep, cls, cand);
            pos = r.x * V::G + r.y; gpos = r.gx * V::G + r.gy; step = r.step; rcode = r.rcode;
          }
        }
      }
    }
    c_steps += (uint32_t)p.T;
    r.x = pos / V::G; r.y = pos % V::G; r.gx = gpos / V::G; r.gy = gpos % V::G; r.step = step; r.rcode = rcode;
    p.state[e] = V::pack(r);
    p.episode[e] = ep;
    if (V::ID == 0 && hits) p.goal_count[e] += hits;
  }
  // statistics: warp reduce -> shared atomics -> one global atomic per counter per CTA
  unsigned long long v[NUM_STATS] = {c_steps, c_ep, c_goal, (unsigned long long)(c_ep - c_goal), c_wall,
                                     (unsigned long long)(c_steps - c_wall - c_stale), c_stale, c_len};
#pragma unroll
  for (int k = 0; k < NUM_STATS; ++k) {
    unsigned long long x = v[k];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x += __shfl_down_sync(0xffffffffu, x, off);
    if ((threadIdx.x & 31) == 0 && x) atomicAdd(&blk_stats[k], x);
  }
  __syncthreads();
  if (threadIdx.x < NUM_STATS && blk_stats[threadIdx.x]) atomicAdd(&p.stats[threadIdx.x], blk_stats[threadIdx.x]);
}

// ------------------------------------------------------------------ state exchange (get/set_state)
// cols: x, y, goal_x, goal_y, step_count, reward_code, goal_count, episode
// set: a row the env could never be in -- a coordinate outside the grid interior (it is clamped so that the
// kernels' +-1 lookups stay inside the table), the ball on a wall, v3's goal on a wall, a reward code
// outside 0..3 -- is COUNTED in the handle's error counter (lmz_stats errors), never fixed silently.
template <class V>
__global__ void lmz_state_kernel(int64_t n, uint32_t *state, uint32_t *goal_count, uint32_t *episode, int32_t *io,
                                 int set, const uint8_t *blob, unsigned int *errors) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  int32_t *row = io + e * 8;
  if (set) {
    EnvRegs r;
    auto clampi = [](int v) { return v < 1 ? 1 : (v > V::G - 2 ? V::G - 2 : v); };   // keep +-1 lookups in the table
    r.x = clampi(row[0]); r.y = clampi(row[1]); r.gx = clampi(row[2]); r.gy = clampi(row[3]);
    r.step = (uint32_t)row[4] < V::STEP_SAT ? (uint32_t)row[4] : V::STEP_SAT;
    r.rcode = row[5] & 3;
    const uint8_t *cls = blob + V::CLS_OFF;
    bool bad = r.x != row[0] || r.y != row[1] || row[4] < 0 || cls[r.x * V::G + r.y] == CLS_W;
    if (V::ID == 0) bad = bad || row[5] < 0 || row[5] > 3;                            // v0 has no goal columns (always 5,5)
    else bad = bad || r.gx != row[2] || r.gy != row[3] || cls[r.gx * V::G + r.gy] == CLS_W;
    if (bad) atomicAdd(errors, 1u);
    state[e] = V::pack(r);
    goal_count[e] = (uint32_t)row[6];
    episode[e] = (uint32_t)row[7];
  } else {
    const EnvRegs r = V::unpack(state[e]);
    row[0] = r.x; row[1] = r.y; row[2] = r.gx; row[3] = r.gy; row[4] = (int32_t)r.step; row[5] = r.rcode;
    row[6] = (int32_t)goal_count[e]; row[7] = (int32_t)episode[e];
  }
}

}  // namespace lmz
