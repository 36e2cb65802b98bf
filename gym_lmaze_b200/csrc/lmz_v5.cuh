// lmz_v5.cuh -- lmaze-v5 / lmaze-v6: the two-level planner / actor env
// (reference gym_lmaze/envs/lmaze_env_v5.py; v6 = v5 + safeFovealGoal(), lmaze_env_v6.py:505-523).
//
// Protocol (SURVEY 8f #4):  reset() -> foveal obs (7,35,35)                       lmaze_env_v5.py:102-153
//                           plannerStep(goal25) -> local obs (4,35,35)            :158-182
//                           step(action4) -> foveal obs, local obs, globalReward, originalReward,
//                                            globalDone, localDone, fovealGoal, action   :187-292
// What shapes the kernel:
//   * the five 18x18 mazes of v2/v4 and v4's float visit layer state[2], but the layer is averaged with
//     the window around the ball only while the LOCAL episode is over (:308-312), and reset() zeroes it;
//   * two observation tensors per step: the foveal one has v4's structure (crop at the ball of free /
//     goal / visit, the fovealGoal one-hot, retStatelast = crop of the LIVE state where the last local
//     episode ended, :314-333,351-352); the local one is four 5x5 bit planes (free crop, ball and previous
//     ball relative to the planner-time fovea WITH numpy's negative-index wrap-around, fovealGoal,
//     :356-380).  Both are x7 upsampled and written as flat runs of float4 per 32-env tile, like v2/v4;
//   * ~80 bits of per-env state in three packed words.
// The kernel itself is the generic foveal kernel of lmz_fov.cuh; this file supplies the per-env logic.
// Where the reference raises IndexError (ball 3 cells right of / below the planner-time fovea, :365-366)
// the local obs row is written as all zeros, loc_err[e] = 1 and the error counter is bumped.
#pragma once
#include "lmz_v2.cuh"

namespace lmz {

struct V5 {
  static constexpr int ID = 5;
  static constexpr int G = 18, E = 7, F = 5, C = 7, CL = 4, S = F * E;       // lmaze_env_v5.py:25-37,357-358
  static constexpr int NLAYOUT = 5, MAX_CAND = 80;
  static constexpr int NBIT = 9;      // bit planes: free, goal, fovealGoal, last free, last goal, ball rel, previous ball rel,
                                      // + the local obs's own copies of free / fovealGoal (all-zero on an IndexError row)
  static constexpr int NVIS = 2;      // float planes: visit crop at the ball, visit crop at retStatelast's window
  static constexpr bool HAS_LOC = true;
  // 5x5 value planes per env: slots 0-6 are the foveal channels -- crop(free, goal, visit), fovealGoal,
  // retStatelast(free, goal, visit) (:314-333) -- 7/8 the ball / previous ball relative to the planner-time fovea,
  // 9/10 the local obs's free crop / fovealGoal; the local obs (:356-380) is slots 9, 7, 8, 10
  static constexpr int NSLOT = 11;
  static constexpr int VALS = NSLOT * 25;
  static constexpr int VIS_SLOT0 = 2, VIS_SLOT1 = 6;
  __host__ __device__ static constexpr int bit_slot(int b) { return b < 2 ? b : (b < 5 ? b + 1 : b + 2); }   // 0 1 3 4 5 7 8 9 10
  __device__ static __forceinline__ float visit_reset(bool) { return 0.0f; }   // self.state = zeros (:134), no averaging
  static constexpr int VT_RESET = 0;
  static constexpr bool MAZE_FIRST = true;                                   // reset(): setGrid() first (:104,115-116)
  static constexpr uint32_t OBS_FLOATS = C * S * S;                          // 8,575 (foveal)
  static constexpr uint32_t OBS_BYTES = OBS_FLOATS * 4;                      // 34,300
  static constexpr uint32_t LOC_FLOATS = CL * S * S;                         // 4,900 (local)
  static constexpr uint32_t LOC_BYTES = LOC_FLOATS * 4;                      // 19,600
  static constexpr int STEP_LIMIT = 10, FSTEP_LIMIT = 50;                    // :47-48
  static constexpr uint32_t STEP_SAT = 255;
  // blob layout (bytes)
  static constexpr uint32_t LUT_OFF = 0;                                     // u32 [8575]: float4 entries of a 4-env group, foveal obs
  static constexpr uint32_t LOCLUT_OFF = align16(OBS_FLOATS * 4);                   // u32 [1225]: float4 entries of one env, local obs
  static constexpr uint32_t ROWBITS_OFF = LOCLUT_OFF + align16(LOC_FLOATS); // u32 [5][18]
  static constexpr uint32_t CLS_OFF = ROWBITS_OFF + align16(NLAYOUT * G * 4);
  static constexpr uint32_t GCAND_OFF = CLS_OFF + align16(NLAYOUT * G * G);
  static constexpr uint32_t BCAND_OFF = GCAND_OFF + NLAYOUT * MAX_CAND * 2;
  static constexpr uint32_t BRANK_OFF = BCAND_OFF + NLAYOUT * MAX_CAND * 2;
  static constexpr uint32_t COUNT_OFF = BRANK_OFF + align16(NLAYOUT * G * G); // u8 ng[5], nb[5]; u16 xcell[5] at +16
  static constexpr uint32_t XCELL_OFF = COUNT_OFF + 16;
  static constexpr uint32_t BLOB_BYTES = COUNT_OFF + 32;
  static constexpr uint32_t SMEM_BYTES = BLOB_BYTES + 2 * 32 * VALS * 4;
};

struct V5Regs {
  int L, x, y, gx, gy;        // maze, ball (= fovea_x0/y0), global goal
  int x1, y1;                 // previous ball            (lmaze_env_v5.py:192-193)
  int fx1, fy1;               // planner-time fovea       (:176-178)
  int fgx, fgy;               // f_goal_x0 / f_goal_y0    (:170-171)
  int lx, ly;                 // where retStatelast was taken (:327-328,351-352)
  int fga;                    // hot cell of fovealGoal   (:166-168; 12 after reset, :131-132)
  uint32_t step, fstep;       // stepCount, fovealStepCount (saturating; only >= 10 / >= 50 / == 0 matter)
  int ld, gd;                 // localDone, globalDone
  int vt;                     // entries in the visit history, or VT_DIRECT (lmz_v2.cuh, "visit layer")
};

// w0: L:3 | x:5 | y:5 | gx:5 | gy:5 | ld:1 | gd:1 | visit T:7      w1: x1:5 | y1:5 | fx1:5 | fy1:5 | fgx:5 | fgy:5
// w2: lx:5 | ly:5 | fga:5 | step:8 | fstep:8
__host__ __device__ inline V5Regs v5_unpack(uint32_t w0, uint32_t w1, uint32_t w2) {
  V5Regs r;
  r.L = w0 & 7; r.x = (w0 >> 3) & 31; r.y = (w0 >> 8) & 31; r.gx = (w0 >> 13) & 31; r.gy = (w0 >> 18) & 31;
  r.ld = (w0 >> 23) & 1; r.gd = (w0 >> 24) & 1; r.vt = (w0 >> 25) & 127;
  r.x1 = w1 & 31; r.y1 = (w1 >> 5) & 31; r.fx1 = (w1 >> 10) & 31; r.fy1 = (w1 >> 15) & 31;
  r.fgx = (w1 >> 20) & 31; r.fgy = (w1 >> 25) & 31;
  r.lx = w2 & 31; r.ly = (w2 >> 5) & 31; r.fga = (w2 >> 10) & 31; r.step = (w2 >> 15) & 255; r.fstep = (w2 >> 23) & 255;
  return r;
}
__host__ __device__ inline void v5_pack(const V5Regs &r, uint32_t &w0, uint32_t &w1, uint32_t &w2) {
  w0 = (uint32_t)r.L | ((uint32_t)r.x << 3) | ((uint32_t)r.y << 8) | ((uint32_t)r.gx << 13) | ((uint32_t)r.gy << 18) |
       ((uint32_t)r.ld << 23) | ((uint32_t)r.gd << 24) | ((uint32_t)r.vt << 25);
  w1 = (uint32_t)r.x1 | ((uint32_t)r.y1 << 5) | ((uint32_t)r.fx1 << 10) | ((uint32_t)r.fy1 << 15) |
       ((uint32_t)r.fgx << 20) | ((uint32_t)r.fgy << 25);
  w2 = (uint32_t)r.lx | ((uint32_t)r.ly << 5) | ((uint32_t)r.fga << 10) | (r.step << 15) | (r.fstep << 23);
}

// reset() (lmaze_env_v5.py:102-153): new maze, goal, ball; every history field collapses onto the ball
template <class W>
__device__ __forceinline__ void v5_respawn(V5Regs &r, const KParams &p, int64_t e, uint32_t &episode,
                                           const FovTables<W> &t, const unsigned char *smem) {
  V2Regs v;
  v.L = r.L; v.x = r.x; v.y = r.y; v.gx = r.gx; v.gy = r.gy; v.px = v.py = 0; v.a = -1; v.step = 0; v.vt = 0;
  v2_respawn<W>(v, p, e, episode, t);                     // MAZE_FIRST: maze, then goal, then ball (as v4); RANDOM_* flags
  r.L = v.L; r.x = v.x; r.y = v.y; r.gx = v.gx; r.gy = v.gy;
  r.x1 = r.fx1 = r.fgx = r.lx = r.x;                      // :139-148, and retStatelast = observation (:327-328)
  r.y1 = r.fy1 = r.fgy = r.ly = r.y;
  r.fga = 12;                                             // fovealGoal[0,2,2] = 1 (:131-132)
  r.step = 0; r.fstep = 0; r.ld = 0; r.gd = 0;            // :109-113
}

// numpy index of a 5-long axis: 0..4 direct, -5..-1 wrap, anything else raises IndexError (:365-366)
__device__ __forceinline__ bool v5_np_index(int &i) {
  if (i < -5 || i > 4) return false;
  if (i < 0) i += 5;
  return true;
}

// step() on registers (lmaze_env_v5.py:187-262 minus the observations): returns "globalDone was raised by this
// step"; leaves the local / global reward codes and the branch taken.
template <class W>
__device__ __forceinline__ bool v5_step_core(V5Regs &r, long long a, const FovTables<W> &t, int &lcode, int &gcode, int &cls) {
  r.x1 = r.x; r.y1 = r.y;                                                            // :192-193
  r.step = r.step < W::STEP_SAT ? r.step + 1 : W::STEP_SAT;                          // :196
  int dx = 0, dy = 0;                                                                // :203-217
  if (a == 0) dx = 1; else if (a == 1) dx = -1; else if (a == 2) dy = 1; else if (a == 3) dy = -1;
  const int nx = r.x + dx, ny = r.y + dy;
  const int tc = t.cls[(r.L - 1) * W::G * W::G + nx * W::G + ny];
  const bool at_fgoal = (nx == r.fgx && ny == r.fgy);
  const int was_gd = r.gd;
  lcode = RC_NEG_ZERO;                                                               // :195
  if (tc == CLS_W) { lcode = RC_WALL; cls = CLS_W; }                                 // :223-224
  else if (at_fgoal) { lcode = RC_GOAL; r.x = nx; r.y = ny; r.ld = 1; cls = CLS_B; } // :226-230
  else {                                                                             // :232-242 (B, S or X)
    if (nx < r.fx1 - 3 || nx > r.fx1 + 2 || ny < r.fy1 - 3 || ny > r.fy1 + 2) r.ld = 1;
    lcode = RC_MOVE; r.x = nx; r.y = ny; cls = CLS_B;
  }
  if (nx == r.gx && ny == r.gy) { gcode = RC_GOAL; r.gd = 1; cls = CLS_X; }          // :245-247
  else if (at_fgoal) gcode = RC_MOVE;                                                // :248-249
  else gcode = RC_WALL;                                                              // :250-251
  if (r.step >= (uint32_t)W::STEP_LIMIT) r.ld = 1;                                   // :257-258
  if (r.fstep >= (uint32_t)W::FSTEP_LIMIT) { r.gd = 1; r.ld = 1; }                   // :260-262
  return r.gd && !was_gd;
}

// plannerStep() on registers (lmaze_env_v5.py:158-182 minus the local observation)
template <class W>
__device__ __forceinline__ void v5_planner_core(V5Regs &r, long long g, unsigned int *errors) {
  if (g < 0 || g > 24) { atomicAdd(errors, 1u); g = g < 0 ? 0 : 24; }               // the reference raises IndexError (:168)
  r.step = 0; r.ld = 0;                                                              // :161-163
  r.fga = (int)g;                                                                    // :165-168
  r.fgx = r.x + (int)g / 5 - 2; r.fgy = r.y + (int)g % 5 - 2;                        // :170-171
  if (r.fstep > 0) { r.fx1 = r.x; r.fy1 = r.y; }                                     // :176-178 (fovea_x0 is the ball)
  r.fstep = r.fstep < W::STEP_SAT ? r.fstep + 1 : W::STEP_SAT;                       // :180
}

using V5Lane = FovLane<V5::NBIT>;   // info: x | y | shown retStatelast x | y | visit op (0 read, 1 average, 2 zero) | loc_err

template <class W>
__device__ __forceinline__ V5Lane v5_lane(const KParams &p, int64_t e, const FovTables<W> &t, const unsigned char *smem,
                                         const FovPre &pre) {
  V5Lane out;
  LaneOut &o = out.o;
  o.st_old = 0; o.render = false; o.done = false; o.cls = -1; o.eplen = 0;
  out.rfov = false; out.rloc = false;
  V5Regs r = v5_unpack(pre.w0, pre.w1, pre.w2);
  bool reset_now = false, write_state = false;
  int visit_want = 0;
  int slx = r.lx, sly = r.ly;                       // the retStatelast window the FOVEAL obs of this call shows
  if (p.mode == MODE_STEP) {
    int lcode, gcode;
    o.done = v5_step_core<W>(r, pre.act, t, lcode, gcode, o.cls);
    visit_want = r.ld ? 1 : 0;                                                       // buildFovealObservation, :308-312
    if (r.fstep == 0) { r.lx = r.x; r.ly = r.y; }                                    // :327-328
    slx = r.lx; sly = r.ly;
    if (r.ld) { r.lx = r.x; r.ly = r.y; }                                            // :351-352, after the obs was built
    p.reward[e] = __uint_as_float(reward_bits(gcode));
    p.reward2[e] = __uint_as_float(reward_bits(lcode));
    p.done[e] = (uint8_t)r.gd;
    p.done2[e] = (uint8_t)r.ld;
    if (o.done) o.eplen = r.fstep;
    reset_now = r.gd && p.autoreset;
    out.rfov = out.rloc = true;
    write_state = true;
  } else if (p.mode == MODE_PLANNER) {
    // auto mask: the envs that are waiting for their planner -- local episode over, or no plannerStep since reset()
    const bool take = p.auto_mask ? (r.ld != 0 || r.fstep == 0) : (p.mask == nullptr || p.mask[e] != 0);
    if (take) {
      v5_planner_core<W>(r, pre.act, p.errors);
      out.rloc = true;
      write_state = true;
    }
  } else if (p.mode == MODE_RESET) {
    reset_now = (p.mask == nullptr) || (p.mask[e] != 0);
    out.rfov = reset_now;
  } else {
    out.rfov = out.rloc = true;
  }
  if (reset_now) {
    uint32_t ep = p.episode[e];
    v5_respawn<W>(r, p, e, ep, t, smem);
    p.episode[e] = ep;
    visit_want = 2;                                 // self.state = zeros (:134); no averaging: localDone is False
    slx = r.lx; sly = r.ly;
    write_state = true;
  }
  // local observation (:356-380)
  int i0 = r.x - r.fx1 + 2, i1 = r.y - r.fy1 + 2, j0 = r.x1 - r.fx1 + 2, j1 = r.y1 - r.fy1 + 2;
  const bool loc_ok = v5_np_index(i0) & v5_np_index(i1) & v5_np_index(j0) & v5_np_index(j1);
  if (out.rloc) {
    if (!loc_ok) atomicAdd(p.errors, 1u);
    if (p.loc_err) p.loc_err[e] = loc_ok ? 0 : 1;
  }
  out.vinfo = visit_plan<W>(visit_want, r.vt);
  if (write_state) {
    uint32_t w0, w1, w2;
    v5_pack(r, w0, w1, w2);
    p.state[e] = w0; p.goal_count[e] = w1; p.aux2[e] = w2;
    if (p.fgoal_out) p.fgoal_out[e] = (uint8_t)r.fga;
  }
  o.st = 0;
  out.info = (uint32_t)r.x | ((uint32_t)r.y << 5) | ((uint32_t)slx << 10) | ((uint32_t)sly << 15) |
             (loc_ok ? 0u : (1u << 22));
  out.rfov = out.rfov && p.obs != nullptr;
  out.rloc = out.rloc && p.obs2 != nullptr;
  out.mask[0] = v2_free_crop<W>(t, r.L, r.x, r.y);                                   // state[0] crop at the fovea
  out.mask[1] = v2_goal_crop(r.x, r.y, r.gx, r.gy);                                  // state[1] crop
  out.mask[2] = 1u << r.fga;                                                         // fovealGoal
  out.mask[3] = v2_free_crop<W>(t, r.L, slx, sly);                                   // retStatelast (a view of state)
  out.mask[4] = v2_goal_crop(slx, sly, r.gx, r.gy);
  out.mask[5] = loc_ok ? (1u << (i0 * 5 + i1)) : 0u;                                 // :365
  out.mask[6] = loc_ok ? (1u << (j0 * 5 + j1)) : 0u;                                 // :366
  out.mask[7] = loc_ok ? out.mask[0] : 0u;                                           // :360, local copy
  out.mask[8] = loc_ok ? out.mask[2] : 0u;                                           // :368, local copy
  return out;
}

// plannerStep on its own (lmaze_env_v5.py:158-182).  Only the envs whose local episode is over take part and
// only their local observation is re-rendered, so the work per tile is small and the CTA-cooperative render
// kernel would spend its time on the one producer warp's per-tile latency chain.  Here every WARP is
// independent: it grabs a tile from the work counter, runs the 32 planner updates (one env per lane) and then
// writes the 19,600-byte local rows of the envs that took part, one env at a time, as float4 runs.
template <class W, int THREADS>
__global__ void __launch_bounds__(THREADS) lmz_planner_kernel(const KParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ float s_vals[THREADS / 32][W::VALS];          // one env's value planes per warp
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  stage_blob<W>(smem, &bar, p.blob);
  const FovTables<W> t(smem);
  const uint32_t *loclut = reinterpret_cast<const uint32_t *>(smem + W::LOCLUT_OFF);
  constexpr uint32_t PER = W::LOC_FLOATS / 4;
  float *mv = s_vals[warp];
  for (;;) {
    const int64_t tl = warp_grab(p, lane, 1);
    if (tl >= p.tile_end) break;
    const int64_t e = tl * 32 + lane;
    const bool valid = e < p.n;
    V5Lane v;
    v.rloc = false; v.info = 0; v.vinfo = 0;
#pragma unroll
    for (int b = 0; b < W::NBIT; ++b) v.mask[b] = 0;
    if (valid) v = v5_lane<W>(p, e, t, smem, fov_preload<W>(p, e));
    unsigned flags = __ballot_sync(0xffffffffu, valid && v.rloc);
    while (flags) {
      const int src = __ffs(flags) - 1;
      flags &= flags - 1;
      // local obs planes (lmaze_env_v5.py:360-368): free crop (value plane 0), ball (7), previous ball (8), fovealGoal (3)
      const uint32_t m0 = __shfl_sync(0xffffffffu, v.mask[0], src), m5 = __shfl_sync(0xffffffffu, v.mask[5], src);
      const uint32_t m6 = __shfl_sync(0xffffffffu, v.mask[6], src), m2 = __shfl_sync(0xffffffffu, v.mask[2], src);
      const bool err = (__shfl_sync(0xffffffffu, v.info, src) >> 22) & 1u;
      __syncwarp();
      if (lane < 25) {
        mv[9 * 25 + lane] = ((m0 >> lane) & 1u) ? 1.0f : 0.0f;
        mv[7 * 25 + lane] = ((m5 >> lane) & 1u) ? 1.0f : 0.0f;
        mv[8 * 25 + lane] = ((m6 >> lane) & 1u) ? 1.0f : 0.0f;
        mv[10 * 25 + lane] = ((m2 >> lane) & 1u) ? 1.0f : 0.0f;
      }
      __syncwarp();
      unsigned char *dst = reinterpret_cast<unsigned char *>(p.obs2) + (tl * 32 + src - p.win_lo) * (int64_t)W::LOC_BYTES;
#pragma unroll 4
      for (uint32_t q = lane; q < PER; q += 32) {
        uint4 val = make_uint4(0u, 0u, 0u, 0u);              // IndexError in the reference: the row is all zero
        if (!err) val = f4_pick(loclut[q], mv);
        st_stream_v4(dst + ((size_t)q << 4), val);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) finish_grabber(p.work, (unsigned long long)gridDim.x);
}

// v6 safeFovealGoal() (lmaze_env_v6.py:505-523): a foveal goal whose window cell is not a wall.
// draws != null: int64 [n][n_draws] values the reference's np.random.randint(0, 25) would have returned;
// the first non-wall one wins (used[e] = how many were consumed; goal -1 if none qualified).
// draws == null: exactly uniform over the window's non-wall cells (the distribution the rejection loop
// has), Philox keyed by (seed, global env id, episode, fovealStepCount).
constexpr uint32_t TAG_SAFE = 0x47u;
template <class W>
__global__ void lmz_safe_goal_kernel(int64_t n, const uint32_t *state, const uint32_t *aux2, const uint32_t *episode,
                                     const uint8_t *blob, const long long *draws, int n_draws, uint8_t *goal_out,
                                     int32_t *used_out, uint64_t seed, uint64_t env_id0) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const uint32_t w0 = state[e];
  const int L = w0 & 7, x = (w0 >> 3) & 31, y = (w0 >> 8) & 31;
  const uint32_t *rowbits = reinterpret_cast<const uint32_t *>(blob + W::ROWBITS_OFF);
  uint32_t m = 0;                                               // smallGrid != 'W', bit i*5+j
#pragma unroll
  for (int i = 0; i < 5; ++i) m |= ((rowbits[(L - 1) * W::G + x - 2 + i] >> (y - 2)) & 31u) << (5 * i);
  int goal = -1, used = 0;
  if (draws) {
    for (int k = 0; k < n_draws; ++k) {
      const long long a = draws[e * n_draws + k];
      used = k + 1;
      if (a >= 0 && a < 25 && ((m >> a) & 1u)) { goal = (int)a; break; }
    }
  } else {
    const int cnt = __popc(m);                                  // >= 1: the ball's own cell is never a wall
    const uint32_t fstep = (aux2[e] >> 23) & 255u;
    const uint64_t gid = env_id0 + (uint64_t)e;
    uint32_t out[4];
    uint32_t k = 0;
    for (uint32_t attempt = 0;; ++attempt) {
      philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), episode[e], (attempt << 16) | (fstep << 8) | TAG_SAFE,
                    (uint32_t)seed, (uint32_t)(seed >> 32), out);
      const uint32_t thresh = (uint32_t)(0x100000000ull % (uint32_t)cnt);
      bool got = false;
#pragma unroll
      for (int i = 0; i < 4 && !got; ++i) {
        const uint64_t mm = (uint64_t)out[i] * (uint64_t)cnt;
        if ((uint32_t)mm >= thresh) { k = (uint32_t)(mm >> 32); got = true; }
      }
      if (got) break;
    }
    uint32_t mm = m;
    for (uint32_t i = 0; i < k; ++i) mm &= mm - 1;              // k-th set bit
    goal = __ffs(mm) - 1;
  }
  goal_out[e] = (uint8_t)(goal < 0 ? 255 : goal);
  if (used_out) used_out[e] = used;
}

// get/set_state for v5/v6.  int32 [n][16]: x, y, x1, y1, fx1, fy1, gx, gy, fgx, fgy, last_x, last_y, fgoal_action,
// step, foveal_step, flags (globalDone | localDone << 1 | layout << 4);
// the episode counter travels in a 17th column.
// set: positions outside [2, 15], goals outside 0..31, a foveal-goal cell outside 0..24 or a maze outside 1..5 are
// clamped AND counted in the error counter.
__global__ void lmz_state_v5_kernel(int64_t n, uint32_t *state, uint32_t *aux1, uint32_t *aux2, uint32_t *episode,
                                    int32_t *io, int set, unsigned int *errors) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  int32_t *row = io + e * 17;
  if (set) {
    auto pos = [](int v) { return v < 2 ? 2 : (v > V5::G - 3 ? V5::G - 3 : v); };     // 5x5 crops stay inside the grid
    V5Regs r;
    r.x = pos(row[0]); r.y = pos(row[1]); r.x1 = pos(row[2]); r.y1 = pos(row[3]); r.fx1 = pos(row[4]); r.fy1 = pos(row[5]);
    r.gx = row[6] & 31; r.gy = row[7] & 31; r.fgx = row[8] & 31; r.fgy = row[9] & 31; r.lx = pos(row[10]); r.ly = pos(row[11]);
    r.fga = row[12] < 0 ? 0 : (row[12] > 24 ? 24 : row[12]);
    r.step = (uint32_t)row[13] < V5::STEP_SAT ? (uint32_t)row[13] : V5::STEP_SAT;
    r.fstep = (uint32_t)row[14] < V5::STEP_SAT ? (uint32_t)row[14] : V5::STEP_SAT;
    r.gd = row[15] & 1; r.ld = (row[15] >> 1) & 1;
    const int L = (row[15] >> 4) & 7;
    r.L = L < 1 ? 1 : (L > 5 ? 5 : L);
    const bool bad = r.x != row[0] || r.y != row[1] || r.x1 != row[2] || r.y1 != row[3] || r.fx1 != row[4] ||
                     r.fy1 != row[5] || r.gx != row[6] || r.gy != row[7] || r.fgx != row[8] || r.fgy != row[9] ||
                     r.lx != row[10] || r.ly != row[11] || r.fga != row[12] || row[13] < 0 || row[14] < 0 || r.L != L;
    if (bad) atomicAdd(errors, 1u);
    r.vt = (state[e] >> 25) & 127;                  // the visit history length is not part of the row: kept
    uint32_t w0, w1, w2;
    v5_pack(r, w0, w1, w2);
    state[e] = w0; aux1[e] = w1; aux2[e] = w2; episode[e] = (uint32_t)row[16];
  } else {
    const V5Regs r = v5_unpack(state[e], aux1[e], aux2[e]);
    row[0] = r.x; row[1] = r.y; row[2] = r.x1; row[3] = r.y1; row[4] = r.fx1; row[5] = r.fy1; row[6] = r.gx; row[7] = r.gy;
    row[8] = r.fgx; row[9] = r.fgy; row[10] = r.lx; row[11] = r.ly; row[12] = r.fga; row[13] = (int32_t)r.step;
    row[14] = (int32_t)r.fstep; row[15] = r.gd | (r.ld << 1) | (r.L << 4); row[16] = (int32_t)episode[e];
  }
}

}  // namespace lmz
