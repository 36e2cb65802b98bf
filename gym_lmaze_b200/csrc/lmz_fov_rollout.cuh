// lmz_fov_rollout.cuh -- T fused steps of the FOVEAL variants with no per-step observation:
// lmaze-v2 / lmaze-v4 (lmaze_env_v2.py:127-225, lmaze_env_v4.py:155-275) and the planner / actor env lmaze-v5 / v6
// (lmaze_env_v5.py:158-292), the counterpart of lmz_rollout_kernel (v0 / v3) in lmz_kernels.cuh.
//
// One thread per env, the packed state words in registers for all T steps, the per-maze tables (cell classes,
// spawn candidate lists) in shared memory, per-step reward f32 (or 1-byte reward code) and done u8 [T][N] streaming
// stores, coalesced across envs.  Actions come from a [T][N] device buffer or from Philox.  The same transition
// functions as the fused step kernel run here (v2_step_core, v5_planner_core, v5_step_core, v2_respawn): there is
// one statement of the env logic.  v4 / v5 keep their float visit layer in HBM in the SCALED form (lmz_v2.cuh): an
// averaging step is 25 read-modify-writes on the window around the ball, by the env's own thread.
//
// v5 / v6: one rollout step = plannerStep for the envs that are waiting for their planner (localDone set, or no
// plannerStep since the last reset -- the device-side mask of lmz_planner_step_auto) followed by step(); outputs
// are globalReward, originalReward, globalDone, localDone per step.
#pragma once
#include "lmz_fov.cuh"

namespace lmz {

constexpr uint32_t TAG_ACTION25 = 0x42u, TAG_HIER = 0x48u;

// The visit layer during a rollout.  Nobody looks at the layer while a rollout runs, so in history mode (lmz_v2.cuh,
// "visit layer") an averaging only APPENDS its window centre to the env's 64-byte history -- kept in shared memory for
// the whole launch (one row per thread, 68-byte stride: no bank conflicts) -- and a reset sets the length to 0.  No
// float is touched.  An env in DIRECT mode (history full, or a layer set through lmz_set_visit) averages its layer
// in global memory with the literal full pass, by its own thread; the step that finds the history full
// materialises the layer from it first.
constexpr int HIST_STRIDE = 68;                            // bytes between two threads' history rows in shared memory

template <class W>
__device__ __forceinline__ void visit_thread(float *layer, uint8_t *hrow, uint32_t vinfo, int bx, int by) {
  const uint32_t op = vinfo & 7u;
  const int tpre = (vinfo >> 3) & 127, tpost = (vinfo >> 10) & 127;
  if (op == VOP_AVG || (op == VOP_RESET && W::VT_RESET == 1)) { hrow[tpost - 1] = (uint8_t)visit_entry(bx, by); return; }
  if (op != VOP_FULL) return;
  for (int cell = 0; cell < W::G * W::G; ++cell) {
    const int x = cell / W::G, y = cell - x * W::G;
    float v;
    if (tpre == VT_DIRECT) v = __ldcg(layer + cell);
    else {                                                 // the history is full: this cell's value from it
      v = 0.0f;
      for (int k = 0; k < tpre; ++k) {
        const int hx = (hrow[k] >> 4) + 2, hy = (hrow[k] & 15) + 2;
        v = visit_avg1(v, (unsigned)(x - hx + 2) < 5u && (unsigned)(y - hy + 2) < 5u);
      }
    }
    __stcg(layer + cell, visit_average(v, (unsigned)(x - bx + 2) < 5u && (unsigned)(y - by + 2) < 5u));
  }
}

struct RolloutCounters {
  uint32_t steps = 0, ep = 0, goal = 0, wall = 0, move = 0, stale = 0;
  unsigned long long len = 0;
};

__device__ __forceinline__ void rollout_store_reward(const KParams &p, int64_t off, int rcode) {
  if (p.reward_code) __stcs(p.reward_code + off, (uint8_t)rcode);
  else __stcs(p.reward + off, __uint_as_float(reward_bits(rcode)));
}

// ---- lmaze-v2 / lmaze-v4 ------------------------------------------------------------------------------------
// Philox action of env g at global rollout step t: word t & 3 of philox(ctr = (g_lo, g_hi, b_lo, (b_hi << 8) | 0x42)),
// b = t >> 2; action = (word * 25) >> 32.
template <class W>
__device__ __forceinline__ void rollout_env_v2(const KParams &p, int64_t e, const FovTables<W> &t, RolloutCounters &c,
                                               uint8_t *hrow) {
  V2Regs r = v2_unpack(p.state[e], p.goal_count[e]);
  uint32_t ep = p.episode[e];
  const uint64_t gid = p.env_id0 + (uint64_t)e;
  uint32_t w[4] = {0, 0, 0, 0};
  float *layer = W::NVIS > 0 ? p.visit + e * (W::G * W::G) : nullptr;
  uint64_t tg = p.t0;
  int64_t off = e;
  for (int s = 0; s < p.T; ++s, ++tg, off += p.n) {
    long long a;
    if (p.actions) a = load_action(p.actions, p.action_dtype, off);
    else {
      if ((tg & 3) == 0 || s == 0) {
        const uint64_t blk = tg >> 2;
        philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)blk, ((uint32_t)(blk >> 32) << 8) | TAG_ACTION25,
                      (uint32_t)p.seed, (uint32_t)(p.seed >> 32), w);
      }
      const uint32_t k = (uint32_t)(tg & 3);
      a = __umulhi(k == 0 ? w[0] : k == 1 ? w[1] : k == 2 ? w[2] : w[3], 25u);
    }
    int rcode, cls = -1;
    const bool done = v2_step_core<W>(r, a, t, p.errors, rcode, cls);
    rollout_store_reward(p, off, rcode);
    __stcs(p.done + off, (uint8_t)(done ? 1 : 0));
    c.wall += (cls == CLS_W); c.move += (cls == CLS_B || cls == CLS_X); c.stale += (cls == CLS_S);
    int want = 1;                                          // v4: every step averages the layer (lmaze_env_v4.py:211-214)
    if (done) {
      c.ep += 1; c.len += r.step; c.goal += (cls == CLS_X);
      if (p.autoreset) { v2_respawn<W>(r, p, e, ep, t); want = 2; }
    }
    if (W::NVIS > 0) visit_thread<W>(layer, hrow, visit_plan<W>(want, r.vt), r.x, r.y);
  }
  c.steps += (uint32_t)p.T;
  uint32_t w0, w1;
  v2_pack(r, w0, w1);
  p.state[e] = w0; p.goal_count[e] = w1; p.episode[e] = ep;
}

// ---- lmaze-v5 / lmaze-v6 ------------------------------------------------------------------------------------
// Philox goal / action of env g at global rollout step t: philox(ctr = (g_lo, g_hi, t_lo, (t_hi << 8) | 0x48));
// goal = (word0 * 25) >> 32, action = word1 >> 30.
template <class W>
__device__ __forceinline__ void rollout_env_v5(const KParams &p, int64_t e, const FovTables<W> &t, const unsigned char *sb,
                                               RolloutCounters &c, uint8_t *hrow) {
  V5Regs r = v5_unpack(p.state[e], p.goal_count[e], p.aux2[e]);
  uint32_t ep = p.episode[e];
  const uint64_t gid = p.env_id0 + (uint64_t)e;
  float *layer = p.visit + e * (W::G * W::G);
  uint64_t tg = p.t0;
  int64_t off = e;
  for (int s = 0; s < p.T; ++s, ++tg, off += p.n) {
    long long a, g;
    if (p.actions) {
      a = load_action(p.actions, p.action_dtype, off);
      g = load_action(p.goals, p.action_dtype, off);
    } else {
      uint32_t w[4];
      philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)tg, ((uint32_t)(tg >> 32) << 8) | TAG_HIER,
                    (uint32_t)p.seed, (uint32_t)(p.seed >> 32), w);
      g = __umulhi(w[0], 25u);
      a = w[1] >> 30;
    }
    if (r.ld != 0 || r.fstep == 0) v5_planner_core<W>(r, g, p.errors);      // plannerStep for the envs waiting for it
    int lcode, gcode, cls = -1;
    const bool done = v5_step_core<W>(r, a, t, lcode, gcode, cls);
    int want = r.ld ? 1 : 0;                                                 // lmaze_env_v5.py:308-312
    if (r.fstep == 0 || r.ld) { r.lx = r.x; r.ly = r.y; }                    // :327-328, :351-352
    __stcs(p.reward + off, __uint_as_float(reward_bits(gcode)));
    __stcs(p.reward2 + off, __uint_as_float(reward_bits(lcode)));
    __stcs(p.done + off, (uint8_t)r.gd);
    __stcs(p.done2 + off, (uint8_t)r.ld);
    c.wall += (cls == CLS_W); c.move += (cls == CLS_B || cls == CLS_X);
    if (done) { c.ep += 1; c.len += r.fstep; c.goal += (cls == CLS_X); }
    if (r.gd && p.autoreset) { v5_respawn<W>(r, p, e, ep, t, sb); want = 2; }
    visit_thread<W>(layer, hrow, visit_plan<W>(want, r.vt), r.x, r.y);
  }
  c.steps += (uint32_t)p.T;
  uint32_t w0, w1, w2;
  v5_pack(r, w0, w1, w2);
  p.state[e] = w0; p.goal_count[e] = w1; p.aux2[e] = w2; p.episode[e] = ep;
  if (p.fgoal_out) p.fgoal_out[e] = (uint8_t)r.fga;
}

template <class W, int THREADS>
__global__ void __launch_bounds__(THREADS) lmz_fov_rollout_kernel(const KParams p) {
  extern __shared__ __align__(128) unsigned char smem[];         // the per-maze tables (blob from ROWBITS_OFF on) + the history rows
  __shared__ unsigned long long blk_stats[NUM_STATS];
  using FS = FovSmall<W>;
  for (uint32_t i = threadIdx.x; i < (W::BLOB_BYTES - FS::STAGE_OFF) / 4; i += THREADS)
    reinterpret_cast<uint32_t *>(smem)[i] = reinterpret_cast<const uint32_t *>(p.blob + FS::STAGE_OFF)[i];
  if (threadIdx.x < NUM_STATS) blk_stats[threadIdx.x] = 0;
  __syncthreads();
  const unsigned char *sb = smem - FS::STAGE_OFF;
  const FovTables<W> t(sb);
  uint8_t *hrow = smem + FS::TAB_BYTES + threadIdx.x * HIST_STRIDE;  // this thread's visit history (v4 / v5)
  RolloutCounters c;
  for (int64_t e = (int64_t)blockIdx.x * THREADS + threadIdx.x; e < p.n; e += (int64_t)gridDim.x * THREADS) {
    if (W::NVIS > 0) {                                           // history in: 64 contiguous bytes per env
      const uint32_t *src = reinterpret_cast<const uint32_t *>(p.hist + e * HIST_MAX);
#pragma unroll
      for (int k = 0; k < HIST_MAX / 4; ++k) reinterpret_cast<uint32_t *>(hrow)[k] = __ldcs(src + k);
    }
    if constexpr (W::HAS_LOC) rollout_env_v5<W>(p, e, t, sb, c, hrow);
    else rollout_env_v2<W>(p, e, t, c, hrow);
    if (W::NVIS > 0) {                                           // ... and out
      uint32_t *dst = reinterpret_cast<uint32_t *>(p.hist + e * HIST_MAX);
#pragma unroll
      for (int k = 0; k < HIST_MAX / 4; ++k) __stcs(dst + k, reinterpret_cast<const uint32_t *>(hrow)[k]);
    }
  }
  unsigned long long v[NUM_STATS] = {c.steps, c.ep, c.goal, (unsigned long long)(c.ep - c.goal), c.wall, c.move, c.stale, c.len};
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

}  // namespace lmz
