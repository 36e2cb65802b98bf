// lmz_v2.cuh -- lmaze-v2: multi-layout foveal env (reference gym_lmaze/envs/lmaze_env_v2.py).
//
// Differences from v0/v3 that shape the kernel:
//   * five 18x18 mazes, one re-rolled per episode (lmaze_env_v2.py:92,303-405): the per-layout
//     tables (row bitmasks, cell classes, goal / ball candidate lists) are staged into shared
//     memory with the same single bulk async (TMA) load as the other variants' blob;
//   * Discrete(25) "teleport the fovea" actions (:39,151-169), reward by the cell the fovea was
//     pointed at (:175-180), done at reward 100 or stepCount > 50 (:222);
//   * the observation is five 5x5 planes -- free-cell crop and goal crop around the ball, the
//     action one-hot, and the previous step's two crops (:185-193) -- each upsampled x7 to 35x35
//     floats: 6,125 floats = 24,500 B per env.  24,500 is not a multiple of 16, so neither bulk
//     copies nor per-env vector stores are possible; instead a TILE of 32 envs (784,000 B, which
//     IS 16-byte aligned) is written as one flat run of float4 stores by the generic foveal kernel
//     in lmz_fov.cuh, which this file feeds with the per-env transition (v2_lane).
#pragma once
#include "lmz_kernels.cuh"

namespace lmz {

// Shared blob layout of the foveal variants (v2, v4); only the LUT length differs.
template <int ID_, int C_>
struct Fov {
  static constexpr int ID = ID_;
  static constexpr int G = 18, E = 7, F = 5, C = C_, S = F * E;       // lmaze_env_v2.py:26-37, lmaze_env_v4.py:26-40
  static constexpr int NLAYOUT = 5, MAX_CAND = 80;
  static constexpr int NBIT = 5;                                       // bit planes: free, goal, action, prev free, prev goal
  static constexpr int NVIS = (C_ == 7) ? 2 : 0;                       // v4: float visit crop at the ball and at the previous window
  static constexpr bool HAS_LOC = false;                               // no second observation tensor
  static constexpr int NSLOT = C_;                                     // 5x5 value planes per env = obs channels
  static constexpr int VALS = NSLOT * 25;
  static constexpr int VIS_SLOT0 = 2, VIS_SLOT1 = 6;                   // v4 channel order: crop(free, goal, visit), action,
                                                                       // retStatelast(free, goal, visit) -- lmaze_env_v4.py:37-40,236-239
  __host__ __device__ static constexpr int bit_slot(int b) {           // channel fed by bit plane b
    return C_ == 7 ? (b < 2 ? b : b + 1) : b;
  }
  __device__ static __forceinline__ float visit_reset(bool in_cur) { return in_cur ? 0.5f : 0.0f; }   // zeros, then :110-113
  static constexpr bool MAZE_FIRST = (ID_ == 4);                       // v4 re-rolls the maze BEFORE drawing goal/ball (:91-98)
  static constexpr uint32_t OBS_FLOATS = C * S * S;                    // 6,125 (v2) / 8,575 (v4)
  static constexpr uint32_t OBS_BYTES = OBS_FLOATS * 4;                // 24,500 / 34,300
  static constexpr uint32_t LOC_FLOATS = 0;
  static constexpr int STEP_LIMIT = 50;                                // lmaze_env_v2.py:43, lmaze_env_v4.py:48
  static constexpr uint32_t STEP_SAT = 63;
  // blob layout (bytes)
  static constexpr uint32_t LUT_OFF = 0;                               // u32 [OBS_FLOATS]: one entry per float4 of a 4-env group (lmz_fov.cuh)
  static constexpr uint32_t LOCLUT_OFF = align16(OBS_FLOATS * 4);
  static constexpr uint32_t ROWBITS_OFF = LOCLUT_OFF;                  // u32 [5][18]: bit y = cell (x,y) is B/S/X
  static constexpr uint32_t CLS_OFF = ROWBITS_OFF + align16(NLAYOUT * G * 4);     // u8 [5][324]
  static constexpr uint32_t GCAND_OFF = CLS_OFF + align16(NLAYOUT * G * G);       // u16 [5][80] cells not in {W,S}
  static constexpr uint32_t BCAND_OFF = GCAND_OFF + NLAYOUT * MAX_CAND * 2;       // u16 [5][80] cells not in {W,X}
  static constexpr uint32_t BRANK_OFF = BCAND_OFF + NLAYOUT * MAX_CAND * 2;       // i8 [5][324] index in BCAND or -1
  static constexpr uint32_t COUNT_OFF = BRANK_OFF + align16(NLAYOUT * G * G);     // u8 ng[5], nb[5]
  static constexpr uint32_t XCELL_OFF = COUNT_OFF + 16;                           // u16 [5]: each maze's 'X' cell
  static constexpr uint32_t BLOB_BYTES = COUNT_OFF + 32;
  static constexpr uint32_t SMEM_BYTES = BLOB_BYTES + 2 * 32 * VALS * 4;   // + the double-buffered per-env value planes
  static constexpr int VT_RESET = 1;                                   // v4 reset(): zeros, then ONE averaging (lmaze_env_v4.py:110-119)
};
using V2 = Fov<2, 5>;
using V4 = Fov<4, 7>;

struct V2Regs {
  int L, x, y, gx, gy, px, py, a;     // a: last action, -1 right after a reset (action plane all zero)
  uint32_t step;
  int vt;                             // v4: entries in the visit history, or VT_DIRECT (see "visit layer" below)
};

// ---- the float visit layer of v4 / v5, kept as its HISTORY -----------------------------------------------------------
// Reference: state[2] = (state[2] + visitMap) / 2 over all 324 cells, visitMap = 1 on the 5x5 window around the ball
// (lmaze_env_v4.py:116-119,211-214; lmaze_env_v5.py:308-312), starting from zeros at reset().  EVERY cell changes on
// every averaging, so a literal implementation reads and writes the whole 1,296-byte layer per env-step, and any
// implementation that keeps the layer in memory has to touch the env's own scattered piece of it every step -- which
// is what limits a kernel whose job is a saturated write stream (DESIGN.md 3.5: ~2.5 KB of streaming per request).
// But the layer is a pure function of WHERE the ball was at each averaging since the reset:
//     v_cell = fold over the averagings k = 0 .. T-1 of   v <- RN32((v + [cell in window_k]) / 2),   v = 0 before k = 0
// so per env only those window centres are stored: hist u8 [N][64], byte k = (x_k - 2) << 4 | (y_k - 2), T in the state
// word.  An averaging APPENDS one byte; a reset sets T = 0 (v4: and appends the spawn cell, its reset averages once);
// an observation needs the layer at 50 cells (the window at the ball and the previous window) and gets them by
// running the fold over the T <= 64 entries in registers -- the same float32 operation sequence as the reference
// (RN32((v + m) / 2) = fma(v, 0.5, m / 2) exactly, denormals included), so the values are bit-identical.  The 32 rows of
// a tile are 2 KB of contiguous memory, read together with the state words a tile ahead.
// An env whose history is full (64 averagings without a reset: only by stepping on far past `done` with autoreset
// off) or whose layer was set through lmz_set_visit (arbitrary values have no history) falls back to DIRECT mode
// (T field = VT_DIRECT): its layer lives in `visit f32 [N][324]` and every averaging is the literal full pass;
// reset() returns to the history form.  lmz_get_visit / lmz_set_visit exchange the layer itself.
constexpr int HIST_MAX = 64, VT_DIRECT = 127;
enum : uint32_t { VOP_READ = 0, VOP_AVG = 1, VOP_RESET = 2, VOP_FULL = 3 };
// want: 0 nothing, 1 average with the window at the ball, 2 reset.  vinfo = op:3 | T before:7 | T after:7
// VOP_FULL with T before != VT_DIRECT: the history is full -- materialise the layer from it first, then the full pass.
template <class W>
__device__ __forceinline__ uint32_t visit_plan(int want, int &vt) {
  const int tpre = vt;
  uint32_t op = VOP_READ;
  if (want == 2) { op = VOP_RESET; vt = W::VT_RESET; }
  else if (want == 1) {
    if (vt >= HIST_MAX) { op = VOP_FULL; vt = VT_DIRECT; }        // direct mode, or the step that converts to it
    else { op = VOP_AVG; vt = vt + 1; }
  }
  return op | ((uint32_t)tpre << 3) | ((uint32_t)vt << 10);
}
// one averaging of one cell: RN32((v + m) / 2) -- v / 2 is exact inside the fma, one rounding, as in the reference's
// float64 expression rounded to float32 (lmz_fov.cuh, visit_average)
__device__ __forceinline__ float visit_avg1(float v, bool in_window) { return __fmaf_rn(v, 0.5f, in_window ? 0.5f : 0.0f); }

// state word: L:3 | x:5 | y:5 | gx:5 | gy:5 | step:6 ; aux word: px:5 | py:5 | a:5 | a_valid:1 | visit T:7 (v4)
__host__ __device__ inline V2Regs v2_unpack(uint32_t s, uint32_t aux) {
  V2Regs r;
  r.L = s & 7; r.x = (s >> 3) & 31; r.y = (s >> 8) & 31; r.gx = (s >> 13) & 31; r.gy = (s >> 18) & 31;
  r.step = (s >> 23) & 63;
  r.px = aux & 31; r.py = (aux >> 5) & 31; r.a = ((aux >> 15) & 1) ? (int)((aux >> 10) & 31) : -1;
  r.vt = (aux >> 16) & 127;
  return r;
}
__host__ __device__ inline void v2_pack(const V2Regs &r, uint32_t &s, uint32_t &aux) {
  s = (uint32_t)r.L | ((uint32_t)r.x << 3) | ((uint32_t)r.y << 8) | ((uint32_t)r.gx << 13) | ((uint32_t)r.gy << 18) |
      (r.step << 23);
  aux = (uint32_t)r.px | ((uint32_t)r.py << 5) | (r.a >= 0 ? (((uint32_t)r.a << 10) | (1u << 15)) : 0u) |
        ((uint32_t)r.vt << 16);
}

template <class W>
struct FovTables {
  const uint32_t *lut;
  const uint32_t *rowbits;
  const uint8_t *cls;
  const uint16_t *gcand, *bcand;
  const int8_t *brank;
  const uint8_t *count;      // ng[0..4], nb[5..9]
  const uint16_t *xcell;     // the 'X' cell of each maze
  __device__ __forceinline__ explicit FovTables(const unsigned char *smem)
      : lut(reinterpret_cast<const uint32_t *>(smem + W::LUT_OFF)), rowbits(reinterpret_cast<const uint32_t *>(smem + W::ROWBITS_OFF)),
        cls(smem + W::CLS_OFF), gcand(reinterpret_cast<const uint16_t *>(smem + W::GCAND_OFF)),
        bcand(reinterpret_cast<const uint16_t *>(smem + W::BCAND_OFF)),
        brank(reinterpret_cast<const int8_t *>(smem + W::BRANK_OFF)), count(smem + W::COUNT_OFF),
        xcell(reinterpret_cast<const uint16_t *>(smem + W::XCELL_OFF)) {}
};

// One float4 of an x7-upsampled image from its table entry (A:11 | B:11 | k:3, built by the host: the first k
// floats show value-plane entry A, the rest entry B) -- see lmz_fov.cuh.  (Byte offsets instead of indices were
// tried and were slower: the casts cost the compiler the shared-memory address space of the loads.)
__device__ __forceinline__ uint4 f4_pick(uint32_t en, const float *gv) {
  const uint32_t va = __float_as_uint(gv[en & 2047u]), vb = __float_as_uint(gv[(en >> 11) & 2047u]), k = en >> 22;
  return make_uint4(va, k > 1 ? va : vb, k > 2 ? va : vb, k > 3 ? va : vb);
}

// a 25-bit plane (bit c = cell c of a 5x5 window) as 25 floats 1.0 / 0.0
__device__ __forceinline__ void expand_plane(uint32_t m, float *dst) {
#pragma unroll
  for (int c = 0; c < 25; ++c) dst[c] = ((m >> c) & 1u) ? 1.0f : 0.0f;
}

// 5x5 crop of the free-cell layer around (x,y) as 25 bits, bit i*5+j = cell (x-2+i, y-2+j)
template <class W>
__device__ __forceinline__ uint32_t v2_free_crop(const FovTables<W> &t, int L, int x, int y) {
  uint32_t m = 0;
#pragma unroll
  for (int i = 0; i < 5; ++i) m |= ((t.rowbits[(L - 1) * V2::G + x - 2 + i] >> (y - 2)) & 31u) << (5 * i);
  return m;
}
__device__ __forceinline__ uint32_t v2_goal_crop(int x, int y, int gx, int gy) {
  const int dx = gx - (x - 2), dy = gy - (y - 2);
  return (dx >= 0 && dx < 5 && dy >= 0 && dy < 5) ? (1u << (dx * 5 + dy)) : 0u;
}

// reset().  v2: goal and ball are drawn on the maze of the episode that just ended, THEN the maze is
// re-rolled (lmaze_env_v2.py:90-92,277-299).  v4: the maze is re-rolled first and goal/ball are drawn
// on the new one (lmaze_env_v4.py:91-98).  Injected spawn: sx, sy, gx, gy | new_layout << 5.
template <class W>
__device__ __forceinline__ void v2_respawn(V2Regs &r, const KParams &p, int64_t e, uint32_t &episode,
                                           const FovTables<W> &t) {
  int sx, sy, gx, gy, nl;
  int Ld;                                         // the maze setGoal() / setBall() look at
  if (p.spawn) {
    const int4 s = p.spawn[e];
    sx = s.x; sy = s.y; gx = s.z; gy = s.w & 31; nl = s.w >> 5;
    bool ok = nl >= 1 && nl <= 5;
    Ld = W::MAZE_FIRST ? (ok ? nl : 1) : r.L;
    const uint8_t *cls = t.cls + (Ld - 1) * W::G * W::G;
    if (!p.random_goal) { gx = t.xcell[Ld - 1] / W::G; gy = t.xcell[Ld - 1] % W::G; }   // the injected goal is ignored
    if (!p.random_ball) { sx = 4; sy = 4; }
    if (ok) ok = gx >= 1 && gx <= W::G - 2 && gy >= 1 && gy <= W::G - 2 && sx >= 1 && sx <= W::G - 2 && sy >= 1 &&
                 sy <= W::G - 2;
    if (ok) {
      const int gc = cls[gx * W::G + gy], bc = cls[sx * W::G + sy];
      if (p.random_goal) ok = gc != CLS_W && gc != CLS_S;
      if (ok && p.random_ball) ok = bc != CLS_W && bc != CLS_X && !(sx == gx && sy == gy);
    }
    if (!ok) {                                    // rejected: count it, fall back to the S / X cells of maze 1
      atomicAdd(p.errors, 1u);
      sx = 4; sy = 4; gx = 8; gy = 8; nl = 1;
    }
  } else {
    WordStream ws;
    ws.init(p.seed, p.env_id0 + (uint64_t)e, episode);
    int L0;
    if (W::MAZE_FIRST) { nl = 1 + (int)ws.uniform(5); L0 = nl - 1; }
    else {
      if (episode == 0) r.L = 1 + (int)ws.uniform(5);              // the maze the constructor rolled (:75)
      L0 = r.L - 1;
    }
    Ld = L0 + 1;
    const int g = t.gcand[L0 * W::MAX_CAND + ws.uniform(t.count[L0])];
    const int rank = t.brank[L0 * W::G * W::G + g];
    const uint32_t nb = t.count[5 + L0];
    uint32_t k;
    if (rank >= 0) { k = ws.uniform(nb - 1); if ((int)k >= rank) k += 1; }
    else k = ws.uniform(nb);
    const int b = t.bcand[L0 * W::MAX_CAND + k];
    gx = g / W::G; gy = g % W::G; sx = b / W::G; sy = b % W::G;
    if (!W::MAZE_FIRST) nl = 1 + (int)ws.uniform(5);
    // RANDOM_GOAL / RANDOM_BALL False (lmaze_env_v2.py:278-299): the draws above are still consumed (the stream
    // layout does not depend on the flags) and then replaced by the maze's 'X' / 'S' cell
    if (!p.random_goal) { gx = t.xcell[Ld - 1] / W::G; gy = t.xcell[Ld - 1] % W::G; }
    if (!p.random_ball) { sx = 4; sy = 4; }       // 'S' is (4,4) in all five mazes
  }
  r.L = nl; r.x = sx; r.y = sy; r.gx = gx; r.gy = gy; r.px = sx; r.py = sy; r.a = -1; r.step = 0;
  episode += 1;
}

// What one env hands to the renderer: NB 25-bit planes, and where / how its visit layer is touched.
template <int NB>
struct FovLane {
  LaneOut o;
  uint32_t mask[NB];
  uint32_t info;            // x:5 | y:5 | px:5 | py:5 | (2 unused bits) | local-obs error:1
  uint32_t vinfo;           // visit layer: op:3 (VOP_*) | T before:7 | T after:7   (visit_plan)
  bool rfov, rloc;          // which observation rows this call writes
};
using V2Lane = FovLane<5>;  // free, goal, action, previous free, previous goal

// An env's packed state words and its action / goal, loaded ahead of time by the kernel (lmz_fov.cuh keeps
// the loads of the NEXT tile in flight while it works on the current one).
struct FovPre {
  uint32_t w0, w1, w2;
  long long act;
  uint4 h[4];               // v4 / v5: the env's 64 visit-history bytes
};
template <class W>
__device__ __forceinline__ FovPre fov_preload(const KParams &p, int64_t e) {
  FovPre q;
  q.w0 = p.state[e]; q.w1 = p.goal_count[e]; q.w2 = W::HAS_LOC ? p.aux2[e] : 0u;
  q.act = (p.mode == MODE_STEP || p.mode == MODE_PLANNER) ? load_action(p.actions, p.action_dtype, e) : 0;
  if (W::NVIS > 0 && p.mode != MODE_PLANNER) {
    const uint4 *hp = reinterpret_cast<const uint4 *>(p.hist + e * HIST_MAX);
#pragma unroll
    for (int k = 0; k < 4; ++k) q.h[k] = __ldcg(hp + k);
  }
  return q;
}

// One reference step() on registers (lmaze_env_v2.py:127-225 minus the observation): returns done, leaves the
// reward code and the branch taken (CLS_X goal, CLS_W wall, CLS_B blank / start, CLS_S: an 'X' cell that is not the goal).
template <class W>
__device__ __forceinline__ bool v2_step_core(V2Regs &r, long long a64, const FovTables<W> &t, unsigned int *errors,
                                             int &reward_code, int &cls) {
  if (a64 < 0 || a64 > 24) { atomicAdd(errors, 1u); a64 = a64 < 0 ? 0 : 24; }       // reference raises IndexError
  const int a = (int)a64;
  reward_code = RC_NEG_ZERO;                                                         // :146
  r.step = r.step < W::STEP_SAT ? r.step + 1 : W::STEP_SAT;                          // :148
  const int fx = r.x + a / 5 - 2, fy = r.y + a % 5 - 2;                              // :151-152
  r.px = r.x; r.py = r.y; r.a = a;                                                   // this obs shows the old crop
  if (fx < W::G - 2 && fx > 1 && fy < W::G - 2 && fy > 1) { r.x = fx; r.y = fy; }    // :157-159
  else {                                                                             // :160-169 per-axis clamp
    if (fx >= W::G - 2) r.x = W::G - 3;
    if (fx <= 1) r.x = 2;
    if (fy >= W::G - 2) r.y = W::G - 3;
    if (fy <= 1) r.y = 2;
  }
  const int tc = t.cls[(r.L - 1) * W::G * W::G + fx * W::G + fy];
  if (fx == r.gx && fy == r.gy) { reward_code = RC_GOAL; cls = CLS_X; }              // :175-176
  else if (tc == CLS_W) { reward_code = RC_WALL; cls = CLS_W; }                      // :177-178
  else if (tc == CLS_B || tc == CLS_S) { reward_code = RC_MOVE; cls = CLS_B; }       // :179-180
  else cls = CLS_S;                                                                  // 'X' not the goal: -0.0
  return (reward_code == RC_GOAL) || (r.step > (uint32_t)W::STEP_LIMIT);            // :222
}

template <class W>
__device__ __forceinline__ V2Lane v2_lane(const KParams &p, int64_t e, const FovTables<W> &t, const FovPre &pre) {
  V2Lane out;
  LaneOut &o = out.o;
  o.st_old = 0; o.render = false; o.done = false; o.cls = -1; o.eplen = 0;
  V2Regs r = v2_unpack(pre.w0, pre.w1);
  bool reset_now = false;
  int reward_code = RC_NEG_ZERO;
  int visit_want = 0;
  if (p.mode == MODE_STEP) {
    visit_want = 1;                                                                  // lmaze_env_v4.py:211-214
    o.done = v2_step_core<W>(r, pre.act, t, p.errors, reward_code, o.cls);
    p.reward[e] = __uint_as_float(reward_bits(reward_code));
    p.done[e] = o.done ? 1 : 0;
    if (o.done) o.eplen = r.step;
    reset_now = o.done && p.autoreset;
    o.render = true;
  } else if (p.mode == MODE_RESET) {
    reset_now = (p.mask == nullptr) || (p.mask[e] != 0);
    o.render = reset_now;
  } else {
    o.render = true;
  }
  if (reset_now) {
    uint32_t ep = p.episode[e];
    v2_respawn<W>(r, p, e, ep, t);
    p.episode[e] = ep;
    visit_want = 2;
  }
  out.info = (uint32_t)r.x | ((uint32_t)r.y << 5) | ((uint32_t)r.px << 10) | ((uint32_t)r.py << 15);
  out.vinfo = (W::NVIS > 0) ? visit_plan<W>(visit_want, r.vt) : 0u;
  uint32_t s, aux;
  v2_pack(r, s, aux);
  o.st = s;
  if (p.mode != MODE_RENDER) { p.state[e] = s; p.goal_count[e] = aux; }
  o.render = o.render && p.obs != nullptr && e >= p.win_lo && e < p.win_lo + p.win_n;
  out.rfov = o.render; out.rloc = false;
  out.mask[0] = v2_free_crop<W>(t, r.L, r.x, r.y);                                   // :185-186
  out.mask[1] = v2_goal_crop(r.x, r.y, r.gx, r.gy);
  out.mask[2] = r.a >= 0 ? (1u << r.a) : 0u;                                         // :136-137 / :87
  out.mask[3] = v2_free_crop<W>(t, r.L, r.px, r.py);                                 // retStatelast (:193)
  out.mask[4] = v2_goal_crop(r.px, r.py, r.gx, r.gy);
  return out;
}

// get/set_state for v2.  cols: x, y, goal_x, goal_y, step_count, layout, aux, episode
// aux = prev_x | prev_y << 5 | last_action << 10 | action_valid << 15
// set: rows the env could never be in (ball / previous ball outside [2, 15], goal outside 0..31, maze outside 1..5,
// action > 24) are clamped AND counted in the error counter.  (The ball MAY sit on a wall: lmaze_env_v2.py:157-159.)
__global__ void lmz_state_v2_kernel(int64_t n, uint32_t *state, uint32_t *auxw, uint32_t *episode, int32_t *io, int set,
                                    unsigned int *errors) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  int32_t *row = io + e * 8;
  if (set) {
    auto clampi = [](int v) { return v < 2 ? 2 : (v > V2::G - 3 ? V2::G - 3 : v); };   // ball stays in [2, 15]
    V2Regs r;
    r.x = clampi(row[0]); r.y = clampi(row[1]); r.gx = row[2] & 31; r.gy = row[3] & 31;
    r.step = (uint32_t)row[4] < V2::STEP_SAT ? (uint32_t)row[4] : V2::STEP_SAT;
    r.L = row[5] < 1 ? 1 : (row[5] > 5 ? 5 : row[5]);
    r.px = clampi(row[6] & 31); r.py = clampi((row[6] >> 5) & 31);
    r.a = ((row[6] >> 15) & 1) ? ((row[6] >> 10) & 31) : -1;
    bool bad = r.x != row[0] || r.y != row[1] || r.gx != row[2] || r.gy != row[3] || row[4] < 0 || r.L != row[5] ||
               r.px != (row[6] & 31) || r.py != ((row[6] >> 5) & 31) || r.a > 24;
    if (bad) atomicAdd(errors, 1u);
    if (r.a > 24) r.a = 24;
    r.vt = (auxw[e] >> 16) & 127;                 // the visit history length is not part of the row: kept
    uint32_t s, aux;
    v2_pack(r, s, aux);
    state[e] = s; auxw[e] = aux; episode[e] = (uint32_t)row[7];
  } else {
    const V2Regs r = v2_unpack(state[e], auxw[e]);
    row[0] = r.x; row[1] = r.y; row[2] = r.gx; row[3] = r.gy; row[4] = (int32_t)r.step; row[5] = r.L;
    row[6] = (int32_t)(auxw[e] & 0xFFFFu); row[7] = (int32_t)episode[e];
  }
}

}  // namespace lmz
