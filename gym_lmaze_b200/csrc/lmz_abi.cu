// lmz_abi.cu -- C-ABI shim of the batched LMaze path (include/lmaze_b200.h).
//
// Host side only does bookkeeping: handle lifecycle, argument / DLPack
// validation, template-blob construction and kernel launches on the caller's
// stream.  No torch types, no exceptions across the boundary, no hidden syncs on
// the step path, and NO CPU implementation of the env -- if there is no CUDA
// device lmz_create fails.
#include <cuda.h>           // driver API types only: lmz_alloc_obs fetches its entry points at run time (no -lcuda)
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <type_traits>
#include <vector>

#include "../../include/lmaze_b200.h"
#include "lmz_kernels.cuh"
#include "lmz_fov.cuh"
#include "lmz_fov_rollout.cuh"

namespace {

// ------------------------------------------------------------------ error plumbing
thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define LMZ_CUDA(expr)                                                                           \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess)                                                                       \
      return fail(LMZ_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

// ------------------------------------------------------------------ mazes
// Cell letters as in the reference: W wall, B blank, S start, X goal.
// v0: lmaze_env.py:37-48.  v3: lmaze_env_v3.py:26-43.  tests/test_abi_cpu.py
// (test_static_queries_and_layouts) checks both against the golden extraction
// from the reference (tests/golden/layouts.npz).
const char V0_CELLS[] =
    "WWWWWWWWWWWW" "WSBBBBBBBBBW" "WBWWBWWWWWBW" "WBBBWBBBBBBW" "WBBWBBBWWWBW" "WBWBWXWBBBBW"
    "WBBBWBBWWBBW" "WBWBWBBBBWBW" "WBWBBBWBBBBW" "WBBWWWBBWWBW" "WBBBBBBBBBBW" "WWWWWWWWWWWW";
const char V3_CELLS[] =
    "WWWWWWWWWWWWWWWWWW" "WWWWWWWWWWWWWWWWWW" "WWWWWWWWWWWWWWWWWW" "WWWWWWWWWWWWWWWWWW"
    "WWWWSBBBWBBBBBWWWW" "WWWWBWWWWBWWBBWWWW" "WWWWBWBBBBBWBBWWWW" "WWWWBWBBBBBWBBWWWW"
    "WWWWBBBBXBBWWWWWWW" "WWWWBWBBBBBWBBWWWW" "WWWWBWBBBBBWBBWWWW" "WWWWBWBBBBBWBBWWWW"
    "WWWWBWWWWWBWBBWWWW" "WWWWBBBBWBBBBBWWWW" "WWWWWWWWWWWWWWWWWW" "WWWWWWWWWWWWWWWWWW"
    "WWWWWWWWWWWWWWWWWW" "WWWWWWWWWWWWWWWWWW";

// v2: lmaze_env_v2.py:303-405.  Five 18x18 mazes whose rows/cols 0-3 and 14-17 are all wall; only the
// 10x10 active region (rows 4..13, cols 4..13) is listed, row-major.
const char *const V2_ACTIVE[5] = {
    "SBBBWBBBBB" "BWWWWBWWBB" "BWBWBBBWBB" "BWBWBWBWBB" "BBBWXWBWWW" "BWBWBWBWBB" "BWBWBWBWBB" "BWBBBWBWBB" "BWWWWWBWBB" "BBBBWBBBBB",
    "SBBBBBBBBB" "BWWWBWWWWB" "BWBBBBBWWB" "BWBWBWBWWB" "BWBWXWBWWB" "BWBWWWBWWB" "BWBWWWBBBB" "BWBBBBBWWB" "BWWWBWWWWB" "BBBBBBBBBB",
    "SBBBBBBBBB" "BWBWWWWWBB" "BWBBBWBBBB" "BWBBBWBWBB" "BWBWXWBWBB" "BWBWBBBWBB" "BWBWBWBWBB" "BBBWBBBBBB" "BWWWWWWWBB" "BBBBBBBBBB",
    "SBBBBBBBBB" "BBWWWBWWBB" "BBBWBBBWBB" "BWBWBWBWBB" "BWBWXWBWBB" "BWBWBWBWBB" "BWBWBWBBBB" "BWBBBWBWBB" "BWBWWWWWBB" "BBBBBBBBBB",
    "SBBBBBBBBB" "BWWWWBWWBB" "BBWBBBBWBB" "BBBBWWBWBB" "BWWXWWWWBB" "BWWBWWBWBB" "BWWBWWBWBB" "BWBBBBBWBB" "BWBWWBWWBB" "BBBBBBBBBB",
};

void v2_cells(int layout, char *cells) {     // layout 1..5 -> 324 letters
  memset(cells, 'W', 18 * 18);
  for (int x = 0; x < 10; ++x) memcpy(cells + (x + 4) * 18 + 4, V2_ACTIVE[layout - 1] + 10 * x, 10);
}

int cls_of(char c) {
  switch (c) {
    case 'W': return lmz::CLS_W;
    case 'B': return lmz::CLS_B;
    case 'X': return lmz::CLS_X;
    default: return lmz::CLS_S;
  }
}

// Host construction of the template blob (layout documented in lmz_variants.h).
template <class V>
void build_blob(const char *cells, std::vector<unsigned char> &blob, int &n_cand, int &s_cell, int &x_cell) {
  blob.assign(V::BLOB_BYTES, 0);
  auto plane = [&](uint32_t off, auto pred) {   // upsampled ExE mask of `pred(cell)`
    float *f = reinterpret_cast<float *>(blob.data() + off);
    for (int i = 0; i < V::G; ++i)
      for (int j = 0; j < V::G; ++j)
        if (pred(cells[i * V::G + j]))
          for (int ii = 0; ii < V::E; ++ii)
            for (int jj = 0; jj < V::E; ++jj) f[(i * V::E + ii) * V::S + j * V::E + jj] = 1.0f;
  };
  if (V::ID == 0) {
    plane(V::STATIC_OFF + 0 * V::PLANE_BYTES, [](char c) { return c == 'W'; });   // lmaze_env.py:92-94
    plane(V::STATIC_OFF + 1 * V::PLANE_BYTES, [](char c) { return c == 'X'; });   // :96-98
    plane(V::STATIC_OFF + 2 * V::PLANE_BYTES, [](char c) { return c == 'B'; });   // :105-107
  } else {
    plane(V::STATIC_OFF, [](char c) { return c == 'B' || c == 'S' || c == 'X'; });  // lmaze_env_v3.py:166
  }
  for (int y = 0; y < V::G; ++y) {   // band table: E rows with ones in columns [E*y, E*y+E)
    float *f = reinterpret_cast<float *>(blob.data() + V::BAND_OFF + y * V::BAND_BYTES);
    for (int ii = 0; ii < V::E; ++ii)
      for (int jj = 0; jj < V::E; ++jj) f[ii * V::S + y * V::E + jj] = 1.0f;
  }
  uint16_t *cand = reinterpret_cast<uint16_t *>(blob.data() + V::CAND_OFF);
  unsigned char *compact = blob.data() + V::COMPACT_OFF;   // u8 [C][G][G]: the un-expanded static layers
  n_cand = 0; s_cell = 0; x_cell = 0;
  for (int i = 0; i < V::G * V::G; ++i) {
    const char c = cells[i];
    if (V::ID == 0) {
      compact[1 * V::G * V::G + i] = (c == 'W'); compact[2 * V::G * V::G + i] = (c == 'X');
      compact[3 * V::G * V::G + i] = (c == 'B');
    } else {
      compact[i] = (c == 'B' || c == 'S' || c == 'X');
    }
    blob[V::CLS_OFF + i] = (unsigned char)cls_of(c);
    for (int ch = 0; ch < V::C; ++ch)                    // the same static layers, one bit per cell
      if (compact[ch * V::G * V::G + i]) {
        const int k = ch * V::G * V::G + i;
        reinterpret_cast<uint32_t *>(blob.data() + V::BITS_OFF)[k >> 5] |= 1u << (k & 31);
      }
    if (c == 'S' && s_cell == 0) s_cell = i;
    if (c == 'X' && x_cell == 0) x_cell = i;
    // spawn candidates: v0 not in {W,X} (lmaze_env.py:73); v3 not W (lmaze_env_v3.py:148,157)
    const bool ok = (V::ID == 0) ? (c != 'W' && c != 'X') : (c != 'W');
    if (ok && n_cand < V::MAX_CAND) cand[n_cand++] = (uint16_t)i;
  }
}

// One table entry per float4 of a run of x7-upsampled 5x5 planes (lmz_fov.cuh): the four floats take at most two
// different cell values -- the first k from value A, the rest from value B.  entry = A | B << 11 | k << 22, A and B
// indexing [env in group][slot][cell] value planes (< 2048 entries).  `slot_of(channel)` maps an obs channel to its value plane.
template <class V, class SlotOf>
void build_f4_lut(uint32_t *lut, uint32_t floats_per_env, uint32_t n_entries, SlotOf slot_of) {
  auto code = [&](uint32_t g) -> uint32_t {
    const uint32_t env = g / floats_per_env, r = g % floats_per_env;
    const uint32_t c = r / (V::S * V::S), row = (r / V::S) % V::S, col = r % V::S;
    return env * V::VALS + (uint32_t)slot_of((int)c) * 25u + (row / V::E) * V::F + col / V::E;   // lmaze_env_v2.py:197-203
  };
  for (uint32_t q = 0; q < n_entries; ++q) {
    const uint32_t c[4] = {code(4 * q), code(4 * q + 1), code(4 * q + 2), code(4 * q + 3)};
    uint32_t k = 1;
    while (k < 4 && c[k] == c[0]) ++k;
    const uint32_t b = k < 4 ? c[k] : c[0];
    for (uint32_t j = k; j < 4; ++j)
      if (c[j] != b) { fprintf(stderr, "lmaze_b200: float4 table: more than two values in one float4\n"); abort(); }
    lut[q] = c[0] | (b << 11) | (k << 22);
  }
}

template <class V>
void build_blob_fov(const char *, std::vector<unsigned char> &blob, int &, int &s_cell, int &x_cell) {
  blob.assign(V::BLOB_BYTES, 0);
  s_cell = 4 * 18 + 4; x_cell = 8 * 18 + 8;        // maze 1's 'S' and 'X'; spawn candidates are per maze in the blob
  // the obs channels ARE the first C value planes (v2: free, goal, action, prev free, prev goal; v4/v5:
  // crop(free, goal, visit), action / fovealGoal, retStatelast(free, goal, visit)); a group of 4 envs = OBS_FLOATS float4s
  build_f4_lut<V>(reinterpret_cast<uint32_t *>(blob.data() + V::LUT_OFF), V::OBS_FLOATS, V::OBS_FLOATS,
                  [](int c) { return c; });
  uint32_t *rowbits = reinterpret_cast<uint32_t *>(blob.data() + V::ROWBITS_OFF);
  uint16_t *gcand = reinterpret_cast<uint16_t *>(blob.data() + V::GCAND_OFF);
  uint16_t *bcand = reinterpret_cast<uint16_t *>(blob.data() + V::BCAND_OFF);
  signed char *brank = reinterpret_cast<signed char *>(blob.data() + V::BRANK_OFF);
  for (int L = 0; L < V::NLAYOUT; ++L) {
    char cells[18 * 18];
    v2_cells(L + 1, cells);
    int ng = 0, nb = 0;
    for (int i = 0; i < V::G * V::G; ++i) {
      const char c = cells[i];
      blob[V::CLS_OFF + L * V::G * V::G + i] = (unsigned char)cls_of(c);
      if (c != 'W') rowbits[L * V::G + i / V::G] |= 1u << (i % V::G);                 // state[0], :94
      brank[L * V::G * V::G + i] = -1;
      if (c != 'W' && c != 'S' && ng < V::MAX_CAND) gcand[L * V::MAX_CAND + ng++] = (uint16_t)i;   // setGoal, :280
      if (c != 'W' && c != 'X' && nb < V::MAX_CAND) {                                 // setBall, :293
        brank[L * V::G * V::G + i] = (signed char)nb;
        bcand[L * V::MAX_CAND + nb++] = (uint16_t)i;
      }
    }
    blob[V::COUNT_OFF + L] = (unsigned char)ng;
    blob[V::COUNT_OFF + 5 + L] = (unsigned char)nb;
    for (int i = 0; i < V::G * V::G; ++i)
      if (cells[i] == 'X') reinterpret_cast<uint16_t *>(blob.data() + V::XCELL_OFF)[L] = (uint16_t)i;
  }
}

// v5/v6: v4's foveal tables + the local observation's LUT (lmaze_env_v5.py:356-380) + each maze's 'X' cell
void build_blob_v5(const char *cells, std::vector<unsigned char> &blob, int &n_cand, int &s_cell, int &x_cell) {
  using V = lmz::V5;
  build_blob_fov<V>(cells, blob, n_cand, s_cell, x_cell);
  // local obs channels (lmaze_env_v5.py:360-368): free crop (value plane 9), ball rel. fovea_x1 (7), previous ball (8),
  // fovealGoal (10) -- the local copies are all zero on an IndexError row; one env row = 1,225 float4s exactly
  build_f4_lut<V>(reinterpret_cast<uint32_t *>(blob.data() + V::LOCLUT_OFF), V::LOC_FLOATS, V::LOC_FLOATS / 4,
                  [](int c) { static const int plane[4] = {9, 7, 8, 10}; return plane[c]; });
}

// ------------------------------------------------------------------ variants
// What the host needs to know of each built variant.  Byte counts are per env.
struct VariantInfo {
  int32_t id;
  int G, C, S, CL;               // maze side, obs channels, obs side, local obs channels (0: no local observation)
  uint32_t obs_bytes;            // full f32 observation
  uint32_t compact_bytes;        // compact observation: u8 [C][G][G], or f32 [C][5][5] for the foveal variants
  uint32_t bits_bytes;           // bit-packed observation (0: not built)
  int num_actions, num_layouts, state_cols;
  bool foveal;                   // the observation is a crop around the ball (v2, v4, v5)
  bool hier;                     // planner / actor levels and the local observation (v5)
  bool has_visit;                // float visit layer (v4, v5)
  const char *cells;             // the one maze of the full-view variants (null: five mazes, v2_cells)
  void (*build_blob)(const char *cells, std::vector<unsigned char> &blob, int &n_cand, int &s_cell, int &x_cell);
};

// actions: lmaze_env.py:16, lmaze_env_v3.py:92; v2 lmaze_env_v2.py:39 (commented out in v4, :43-44); v5's step()
// moves by one cell (lmaze_env_v5.py:205-217), plannerStep takes 25.  Layouts: lmaze_env_v2.py:306, lmaze_env_v4.py:351.
const VariantInfo VARIANTS[] = {
    {LMZ_V0, lmz::V0::G, lmz::V0::C, lmz::V0::S, 0, lmz::V0::OBS_BYTES, lmz::V0::COMPACT_BYTES,
     lmz::V0::BITS_WORDS * 4, 4, 1, LMZ_ST_COLS, false, false, false, V0_CELLS, build_blob<lmz::V0>},
    {LMZ_V2, lmz::V2::G, lmz::V2::C, lmz::V2::S, 0, lmz::V2::OBS_BYTES, lmz::V2::C * 25 * 4,
     0, 25, 5, LMZ_ST_COLS, true, false, false, nullptr, build_blob_fov<lmz::V2>},
    {LMZ_V3, lmz::V3::G, lmz::V3::C, lmz::V3::S, 0, lmz::V3::OBS_BYTES, lmz::V3::COMPACT_BYTES,
     lmz::V3::BITS_WORDS * 4, 4, 1, LMZ_ST_COLS, false, false, false, V3_CELLS, build_blob<lmz::V3>},
    {LMZ_V4, lmz::V4::G, lmz::V4::C, lmz::V4::S, 0, lmz::V4::OBS_BYTES, lmz::V4::C * 25 * 4,
     0, 25, 5, LMZ_ST_COLS, true, false, true, nullptr, build_blob_fov<lmz::V4>},
    {LMZ_V5, lmz::V5::G, lmz::V5::C, lmz::V5::S, lmz::V5::CL, lmz::V5::OBS_BYTES, lmz::V5::C * 25 * 4,   // CL: lmaze_env_v5.py:357-358
     0, 4, 5, LMZ_ST_COLS_HIER, true, true, true, nullptr, build_blob_v5},
};

const VariantInfo *variant_info(int32_t variant) {   // null for a variant that is not built
  for (const VariantInfo &v : VARIANTS)
    if (v.id == variant) return &v;
  return nullptr;
}

int unknown_variant(int32_t variant) { return fail(LMZ_ERR_UNSUPPORTED, "unknown variant %d", variant); }

}  // namespace

// ------------------------------------------------------------------ handle
struct lmz_env {
  lmz_config cfg;
  const VariantInfo *var;        // cfg.variant's entry of VARIANTS
  int num_sms;
  // device memory owned by the handle
  uint32_t *state, *goal_count, *episode;
  float *visit;                  // v4 / v5: f32 [N][324] (the layer of envs in direct mode)
  uint8_t *hist;                 // v4 / v5: u8 [N][64] visit history
  uint32_t *aux2;                // v5: third packed state word
  // v5 local outputs (caller-owned), lmz_bind_local
  float *loc_obs, *reward2;
  uint8_t *done2, *loc_err, *fgoal_out;
  bool local_bound;
  unsigned char *blob;
  unsigned long long *stats;     // NUM_STATS counters + 1 error counter + 2 work-distribution words
  void *act_stage;               // lmz_step_host staging, lazily allocated (N * 8 bytes)
  // bound outputs (caller-owned)
  void *obs;                     // f32 [win_n][C][S][S] or u8 [win_n][C][G][G]
  float *reward;
  uint8_t *done;
  bool bound;
  int64_t win_lo, win_n;         // obs rows hold envs [win_lo, win_lo + win_n)
  bool obs_synced;               // incremental render: obs currently holds a full render of the window
  int n_cand, s_cell, x_cell;
  uint64_t rollout_t;            // rollout steps taken so far (keys the action RNG)
  int64_t launches;
  // double-buffered host pipeline (lmz_step_host_async / lmz_step_host_wait), lazily created
  struct {
    bool init;
    cudaStream_t copy;           // D2H stream: step k's copies overlap step k+1's H2D + kernel
    cudaEvent_t ready[2];        // step outputs of slot s are complete on the caller's stream
    cudaEvent_t drained[2];      // the D2H copies out of slot s have finished
    bool inflight[2];
    void *act[2];                // device staging of the host actions
    void *obs[2];                // device obs buffers the kernel writes in pipelined mode (compact / bits rows)
    float *reward[2];
    uint8_t *done[2];
    uint64_t k;                  // steps submitted
  } pipe;
};

namespace {

struct DeviceGuard {   // run on the handle's device, restore the caller's on exit
  int prev;
  bool changed;
  explicit DeviceGuard(int dev) : prev(-1), changed(false) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) changed = (cudaSetDevice(dev) == cudaSuccess);
  }
  ~DeviceGuard() {
    if (changed) cudaSetDevice(prev);
  }
};

lmz::KParams base_params(lmz_env *h) {
  lmz::KParams p;
  memset(&p, 0, sizeof(p));
  p.n = h->cfg.num_envs;
  p.state = h->state; p.goal_count = h->goal_count; p.episode = h->episode; p.visit = h->visit; p.hist = h->hist;
  p.obs = h->obs; p.reward = h->reward; p.done = h->done;
  p.win_lo = h->win_lo; p.win_n = h->win_n;
  p.tile_begin = 0; p.tile_end = (p.n + 31) / 32;
  p.blob = h->blob; p.stats = h->stats;
  p.errors = reinterpret_cast<unsigned int *>(h->stats + lmz::NUM_STATS);
  p.seed = h->cfg.seed; p.env_id0 = (uint64_t)h->cfg.env_id0;
  p.autoreset = h->cfg.autoreset; p.random_ball = h->cfg.random_ball; p.random_goal = h->cfg.random_goal;
  p.n_cand = h->n_cand; p.s_cell = h->s_cell;
  p.l2_policy = h->cfg.tune[1] ? h->cfg.tune[1] : lmz::DEFAULT_L2_POLICY;
  p.work = h->stats + lmz::NUM_STATS + 1;
  p.bulk_split = (uint32_t)h->cfg.tune[3];
  p.aux2 = h->aux2; p.obs2 = h->loc_obs; p.reward2 = h->reward2; p.done2 = h->done2; p.loc_err = h->loc_err;
  p.fgoal_out = h->fgoal_out;
  p.obs_bits = h->cfg.obs_mode == LMZ_OBS_BITS;
  return p;
}

// bytes of one env's row in the bound obs tensor
size_t obs_row_bytes(const lmz_env *h) {
  if (h->cfg.obs_mode == LMZ_OBS_COMPACT) return h->var->compact_bytes;
  if (h->cfg.obs_mode == LMZ_OBS_BITS) return h->var->bits_bytes;
  return h->var->obs_bytes;
}

// Resident CTAs per SM of KERN with `threads` threads and `smem` bytes of dynamic shared memory (>= 1), or an LMZ_ERR
// code.  Queried once per device and thread; `raise_smem` first lifts the kernel's dynamic shared memory limit to `smem`.
template <auto KERN>
int resident_ctas(lmz_env *h, int threads, int smem, bool raise_smem, const char *what) {
  static thread_local int configured_dev = -1;
  static thread_local int ctas_per_sm = 1;
  if (configured_dev != h->cfg.device) {
    if (raise_smem) LMZ_CUDA(cudaFuncSetAttribute(KERN, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LMZ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, KERN, threads, smem));
    if (ctas_per_sm < 1) return fail(LMZ_ERR_CUDA, "%s does not fit on an SM", what);
    configured_dev = h->cfg.device;
  }
  return ctas_per_sm;
}

// CTAs per SM of a persistent launch: the tune[2] cap when set, else `dflt`; never more than `fit`
int ctas_per_sm(const lmz_env *h, int dflt, int fit) {
  const int per_sm = h->cfg.tune[2] > 0 ? h->cfg.tune[2] : dflt;
  return per_sm < fit ? per_sm : fit;
}

// `per_sm` CTAs on every SM, but no more CTAs than `work` units
int64_t persistent_grid(const lmz_env *h, int per_sm, int64_t work) {
  const int64_t grid = (int64_t)h->num_sms * per_sm;
  return grid < work ? grid : work;
}

int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Every kernel launch of the handle: at least one CTA, the launch error checked, the launch counted.
template <class Kern, class... Args>
int launch(lmz_env *h, Kern kern, int64_t grid, int threads, int smem, cudaStream_t s, Args... args) {
  if (grid < 1) grid = 1;
  kern<<<(unsigned)grid, threads, smem, s>>>(args...);
  LMZ_CUDA(cudaGetLastError());
  h->launches += 1;
  return LMZ_OK;
}

constexpr int TMA_THREADS = 32;      // one warp per SM issues the bulk copies: the TMA engine does the moving
constexpr int ST_THREADS = 1024;     // 32 warps of vector stores per SM

template <class V, int RENDER, int THREADS>
int launch_env_t(lmz_env *h, const lmz::KParams &p, cudaStream_t s) {
  constexpr auto kern = (RENDER == lmz::RENDER_TMA) ? lmz::lmz_env_tma_kernel<V, THREADS> : lmz::lmz_env_st_kernel<V, THREADS>;
  const int fit = resident_ctas<kern>(h, THREADS, V::BLOB_BYTES, true, "env kernel");
  if (fit < 0) return fit;
  // persistent grid: a whole number of CTAs per SM, never more CTAs than tiles
  // TMA render: ONE issuing CTA per SM even where two fit (v3: 7,528 vs 7,481 GB/s, tools/v3_sweep.py)
  const int per_sm = ctas_per_sm(h, RENDER == lmz::RENDER_TMA ? 1 : fit, fit);
  return launch(h, kern, persistent_grid(h, per_sm, p.tile_end - p.tile_begin), THREADS, V::BLOB_BYTES, s, p);
}

// transition-only (no obs bound) and compact-obs launches: persistent 128-thread CTAs, dynamic tiles
template <class V>
int launch_compact(lmz_env *h, const lmz::KParams &p, cudaStream_t s) {
  constexpr int THREADS = 128;
  constexpr auto kern = lmz::lmz_env_compact_kernel<V, THREADS>;
  const int fit = resident_ctas<kern>(h, THREADS, 0, false, "compact env kernel");
  if (fit < 0) return fit;
  // resident CTAs per SM (tools/small_bench.py): with observations to write, TWO 4-warp CTAs per SM stream more
  // (10.9 vs 9.9 G env-steps/s on v0) than the 8 that fit -- fewer storing warps, higher write bandwidth; the
  // transition-only launch (14 B per env, latency-bound) wants them all
  const int per_sm = ctas_per_sm(h, p.obs != nullptr ? 2 : fit, fit);
  return launch(h, kern, persistent_grid(h, per_sm, ceil_div(p.tile_end - p.tile_begin, THREADS / 32)), THREADS, 0, s, p);
}

// incremental render (LMZ_RENDER_INCREMENTAL): only the ball / goal blocks that moved are rewritten
template <class V>
int launch_incremental(lmz_env *h, const lmz::KParams &p, cudaStream_t s) {
  constexpr int THREADS = 128;
  constexpr auto kern = lmz::lmz_env_incr_kernel<V, THREADS>;
  const int fit = resident_ctas<kern>(h, THREADS, 0, false, "incremental env kernel");
  if (fit < 0) return fit;
  const int per_sm = ctas_per_sm(h, V::ID == 0 ? 4 : 6, fit);      // tools/small_bench.py: +10 % over full occupancy
  return launch(h, kern, persistent_grid(h, per_sm, ceil_div(p.tile_end - p.tile_begin, THREADS / 32)), THREADS, 0, s, p);
}

template <class V>
int launch_env_v(lmz_env *h, const lmz::KParams &p, cudaStream_t s) {
  if (p.obs == nullptr || h->cfg.obs_mode == LMZ_OBS_COMPACT || h->cfg.obs_mode == LMZ_OBS_BITS)
    return launch_compact<V>(h, p, s);
  if (h->cfg.render_mode == LMZ_RENDER_INCREMENTAL) {
    if (p.mode == lmz::MODE_STEP && h->obs_synced) return launch_incremental<V>(h, p, s);
    // not in sync yet (first call after bind / set_window / set_state), or a reset / render call:
    // full TMA render.  A call that renders every env of the window leaves the tensor in sync.
    const int rc = launch_env_t<V, lmz::RENDER_TMA, TMA_THREADS>(h, p, s);
    if (rc == LMZ_OK && (p.mode != lmz::MODE_RESET || p.mask == nullptr)) h->obs_synced = true;
    return rc;
  }
  if (h->cfg.render_mode == LMZ_RENDER_ST128) {
    if (h->cfg.tune[0] == 512) return launch_env_t<V, lmz::RENDER_ST128, 512>(h, p, s);
    if (h->cfg.tune[0] == 256) return launch_env_t<V, lmz::RENDER_ST128, 256>(h, p, s);
    return launch_env_t<V, lmz::RENDER_ST128, ST_THREADS>(h, p, s);
  }
  switch (h->cfg.tune[0]) {
    case 64: return launch_env_t<V, lmz::RENDER_TMA, 64>(h, p, s);
    case 128: return launch_env_t<V, lmz::RENDER_TMA, 128>(h, p, s);
    case 256: return launch_env_t<V, lmz::RENDER_TMA, 256>(h, p, s);
    default: return launch_env_t<V, lmz::RENDER_TMA, TMA_THREADS>(h, p, s);
  }
}

// default CTA size of the foveal render kernel per variant (1 producer warp + the rendering warps)
#ifndef LMZ_FOV_THREADS
#define LMZ_FOV_THREADS(id) 128      /* v2, v4, v5 alike: 1 producer + 3 rendering warps (tools/fov_sweep2.py) */
#endif

template <class W, int THREADS>
int launch_fov_t(lmz_env *h, const lmz::KParams &p, cudaStream_t s) {
  constexpr auto kern = lmz::lmz_env_fov_kernel<W, THREADS>;
  const int fit = resident_ctas<kern>(h, THREADS, W::SMEM_BYTES, true, "foveal env kernel");
  if (fit < 0) return fit;
  const int per_sm = ctas_per_sm(h, 1, fit);          // default: ONE persistent CTA per SM
  return launch(h, kern, persistent_grid(h, per_sm, p.tile_end - p.tile_begin), THREADS, W::SMEM_BYTES, s, p);
}

template <class W>
int launch_fov(lmz_env *h, const lmz::KParams &p, cudaStream_t s) {
  if (W::HAS_LOC && !h->local_bound)
    return fail(LMZ_ERR_STATE, "lmaze-v5/v6: local outputs not bound: call lmz_bind_local first");
  // CTA size and CTAs per SM (tools/fov_sweep2.py).  FEWER storing warps reach a HIGHER write bandwidth on a B200:
  // v2 with ONE 128-thread CTA per SM (1 producer warp + 3 rendering warps) streams 7.47 TB/s, the pure-write
  // ceiling, against 7.0 TB/s with 1024 threads and 6.3 TB/s with two 128-thread CTAs per SM.  v4 / v5 run the
  // same organisation since round 2 (the scaled visit layer needs no producer warps of its own).
  const int t = h->cfg.tune[0] ? h->cfg.tune[0] : LMZ_FOV_THREADS(W::ID);
  switch (t) {
    case 128: return launch_fov_t<W, 128>(h, p, s);
    case 160: return launch_fov_t<W, 160>(h, p, s);
    case 192: return launch_fov_t<W, 192>(h, p, s);
    case 224: return launch_fov_t<W, 224>(h, p, s);
    case 256: return launch_fov_t<W, 256>(h, p, s);
    case 512: return launch_fov_t<W, 512>(h, p, s);
    case 1024: return launch_fov_t<W, 1024>(h, p, s);
    default: break;
  }
  return fail(LMZ_ERR_INVALID, "foveal kernels are built for tune[0] = 128, 160, 192, 224, 256, 512 or 1024 threads (got %d)", t);
}

// compact observations / nothing to render (foveal variants): warp-granular kernel, several small CTAs per SM
template <class W, int THREADS>
int launch_fov_small_t(lmz_env *h, const lmz::KParams &p, cudaStream_t s) {
  if (W::HAS_LOC && !h->local_bound)
    return fail(LMZ_ERR_STATE, "lmaze-v5/v6: local outputs not bound: call lmz_bind_local first");
  constexpr auto kern = lmz::lmz_fov_small_kernel<W, THREADS>;
  constexpr int SMEM = (int)lmz::FovSmall<W>::smem_bytes(THREADS);      // tables + one 32-env tile of rows per warp
  const int fit = resident_ctas<kern>(h, THREADS, SMEM, true, "foveal compact kernel");
  if (fit < 0) return fit;
  // resident CTAs per SM (tools/fov_compact_sweep.py): v2 writes through the TMA engine only, and ONE 4-warp CTA per
  // SM streams more (11.5 G env-steps/s) than the three that fit (9.2 G) -- fewer writers, higher write bandwidth;
  // the visit variants and the launches that write nothing are latency-bound and want every CTA that fits
  const int per_sm = ctas_per_sm(h, (W::NVIS == 0 && p.obs != nullptr) ? 1 : fit, fit);
  return launch(h, kern, persistent_grid(h, per_sm, ceil_div(p.tile_end - p.tile_begin, THREADS / 32)), THREADS, SMEM, s, p);
}

template <class W>
int launch_fov_small(lmz_env *h, const lmz::KParams &p, cudaStream_t s) {
  if (h->cfg.tune[0] == 64) return launch_fov_small_t<W, 64>(h, p, s);       // (tuning: 2 warps per CTA)
  if (h->cfg.tune[0] == 256) return launch_fov_small_t<W, 256>(h, p, s);     // (tuning: 8 warps per CTA)
  return launch_fov_small_t<W, 128>(h, p, s);
}

template <class W>
int launch_fov_any(lmz_env *h, const lmz::KParams &p, cudaStream_t s) {
  const bool nothing_to_render = p.obs == nullptr && (!W::HAS_LOC || p.obs2 == nullptr);
  if (h->cfg.obs_mode == LMZ_OBS_COMPACT || nothing_to_render) return launch_fov_small<W>(h, p, s);
  return launch_fov<W>(h, p, s);
}

// plannerStep (lmaze-v5/v6): warp-granular kernel, several small CTAs per SM
int launch_planner(lmz_env *h, const lmz::KParams &p, cudaStream_t s) {
  using W = lmz::V5;
  constexpr int THREADS = 128;
  if (!h->local_bound) return fail(LMZ_ERR_STATE, "lmaze-v5/v6: local outputs not bound: call lmz_bind_local first");
  constexpr auto kern = lmz::lmz_planner_kernel<W, THREADS>;
  const int fit = resident_ctas<kern>(h, THREADS, W::BLOB_BYTES, true, "planner kernel");
  if (fit < 0) return fit;
  // every CTA that fits, whatever tune[2] says
  return launch(h, kern, persistent_grid(h, fit, ceil_div(p.tile_end - p.tile_begin, THREADS / 32)), THREADS, W::BLOB_BYTES, s, p);
}

int launch_env(lmz_env *h, const lmz::KParams &p, cudaStream_t s) {
  if (h->cfg.variant == LMZ_V5 && p.mode == lmz::MODE_PLANNER && h->cfg.obs_mode == LMZ_OBS_FULL && p.obs2 != nullptr)
    return launch_planner(h, p, s);
  if (h->cfg.variant == LMZ_V5) return launch_fov_any<lmz::V5>(h, p, s);
  if (h->cfg.variant == LMZ_V2) return launch_fov_any<lmz::V2>(h, p, s);
  if (h->cfg.variant == LMZ_V4) return launch_fov_any<lmz::V4>(h, p, s);
  if (h->cfg.variant == LMZ_V0) return launch_env_v<lmz::V0>(h, p, s);
  return launch_env_v<lmz::V3>(h, p, s);
}

template <class V>
int launch_rollout_v(lmz_env *h, const lmz::KParams &p, cudaStream_t s) {
  constexpr int THREADS = 256;
  // 8 resident CTAs of 256 threads per SM
  return launch(h, lmz::lmz_rollout_kernel<V, THREADS>, persistent_grid(h, 8, ceil_div(p.n, THREADS)), THREADS, 0, s, p);
}

template <class W>
int launch_fov_rollout(lmz_env *h, const lmz::KParams &p, cudaStream_t s) {
  constexpr int THREADS = 128;
  constexpr int TAB = (int)((W::BLOB_BYTES - W::ROWBITS_OFF + 15u) & ~15u);
  constexpr int SMEM = TAB + THREADS * lmz::HIST_STRIDE;               // tables + one visit-history row per thread
  constexpr auto kern = lmz::lmz_fov_rollout_kernel<W, THREADS>;
  const int fit = resident_ctas<kern>(h, THREADS, SMEM, false, "foveal rollout kernel");
  if (fit < 0) return fit;
  return launch(h, kern, persistent_grid(h, fit, ceil_div(p.n, THREADS)), THREADS, SMEM, s, p);
}

int check_handle(lmz_env *h) {
  if (!h) return fail(LMZ_ERR_INVALID, "env handle is NULL");
  return LMZ_OK;
}

int check_bound(lmz_env *h) {
  if (!h->bound) return fail(LMZ_ERR_STATE, "output buffers not bound: call lmz_bind first");
  return LMZ_OK;
}

// bytes of one action (goal) of LMZ_ACT_* dtype `d`; 0 for an unknown dtype
size_t action_bytes(int32_t d) { return d == LMZ_ACT_U8 ? 1 : d == LMZ_ACT_I32 ? 4 : d == LMZ_ACT_I64 ? 8 : 0; }

int check_action_dtype(int32_t d, const char *what) {
  if (!action_bytes(d)) return fail(LMZ_ERR_INVALID, "unknown %s %d", what, d);
  return LMZ_OK;
}

// ---- DLPack validation -----------------------------------------------------
constexpr uint8_t ANY_INT = 255;   // Want::code of an action-like tensor: uint8, int32 or int64

struct Want {
  const char *name;
  uint8_t code;      // DLDataTypeCode, or ANY_INT
  uint8_t bits;
  int ndim;
  int64_t shape[4];
  int align;        // required alignment of the data pointer in bytes
};

// a per-env vector [n] and a per-step matrix [T, n], aligned to their element
Want per_env(const lmz_env *h, const char *name, uint8_t code, uint8_t bits = 0) {
  return Want{name, code, bits, 1, {h->cfg.num_envs, 0, 0, 0}, code == ANY_INT ? 1 : bits / 8};
}

Want per_step(const lmz_env *h, const char *name, int32_t T, uint8_t code, uint8_t bits = 0) {
  return Want{name, code, bits, 2, {T, h->cfg.num_envs, 0, 0}, code == ANY_INT ? 1 : bits / 8};
}

int check_dl(const lmz_env *h, const DLManagedTensor *mt, const Want &w, void **data, int *action_dtype = nullptr) {
  if (!mt) return fail(LMZ_ERR_INVALID, "%s: DLManagedTensor is NULL", w.name);
  const DLTensor &t = mt->dl_tensor;
  if (t.device.device_type != kDLCUDA && t.device.device_type != kDLCUDAManaged)
    return fail(LMZ_ERR_INVALID, "%s: tensor must live on the CUDA device (device_type %d)", w.name,
                t.device.device_type);
  if (t.device.device_id != h->cfg.device)
    return fail(LMZ_ERR_INVALID, "%s: tensor is on cuda:%d, env is on cuda:%d", w.name, t.device.device_id,
                h->cfg.device);
  if (t.dtype.lanes != 1) return fail(LMZ_ERR_INVALID, "%s: vector dtypes not supported", w.name);
  if (w.code == ANY_INT) {
    int ad = -1;
    if ((t.dtype.code == kDLUInt || t.dtype.code == kDLBool) && t.dtype.bits == 8) ad = LMZ_ACT_U8;
    else if (t.dtype.code == kDLInt && t.dtype.bits == 32) ad = LMZ_ACT_I32;
    else if (t.dtype.code == kDLInt && t.dtype.bits == 64) ad = LMZ_ACT_I64;
    if (ad < 0)
      return fail(LMZ_ERR_INVALID, "%s: dtype must be uint8, int32 or int64 (got code %d bits %d)", w.name,
                  t.dtype.code, t.dtype.bits);
    if (action_dtype) *action_dtype = ad;
  } else {
    const bool u8_like = (w.code == kDLUInt && w.bits == 8) &&
                         ((t.dtype.code == kDLUInt || t.dtype.code == kDLBool) && t.dtype.bits == 8);
    if (!u8_like && (t.dtype.code != w.code || t.dtype.bits != w.bits))
      return fail(LMZ_ERR_INVALID, "%s: wrong dtype (got code %d bits %d, want code %d bits %d)", w.name,
                  t.dtype.code, t.dtype.bits, w.code, w.bits);
  }
  if (t.ndim != w.ndim) return fail(LMZ_ERR_INVALID, "%s: ndim %d, want %d", w.name, t.ndim, w.ndim);
  int64_t expect_stride = 1;
  for (int d = w.ndim - 1; d >= 0; --d) {
    if (t.shape[d] != w.shape[d])
      return fail(LMZ_ERR_INVALID, "%s: shape[%d] = %lld, want %lld", w.name, d, (long long)t.shape[d],
                  (long long)w.shape[d]);
    if (t.strides && t.shape[d] > 1 && t.strides[d] != expect_stride)
      return fail(LMZ_ERR_INVALID, "%s: tensor must be contiguous (stride[%d] = %lld, want %lld)", w.name, d,
                  (long long)t.strides[d], (long long)expect_stride);
    expect_stride *= t.shape[d];
  }
  unsigned char *ptr = static_cast<unsigned char *>(t.data) + t.byte_offset;
  if ((reinterpret_cast<uintptr_t>(ptr) % (uintptr_t)w.align) != 0)
    return fail(LMZ_ERR_INVALID, "%s: data pointer must be %d-byte aligned", w.name, w.align);
  *data = ptr;
  return LMZ_OK;
}

// Frees whatever the host pipeline holds -- all of it, or what a failed set-up got to create -- and marks it
// not set up.
void release_pipe(lmz_env *h) {
  auto &pp = h->pipe;
  if (pp.copy) cudaStreamSynchronize(pp.copy);
  for (int i = 0; i < 2; ++i) {
    if (pp.ready[i]) cudaEventDestroy(pp.ready[i]);
    if (pp.drained[i]) cudaEventDestroy(pp.drained[i]);
    cudaFree(pp.act[i]); cudaFree(pp.obs[i]); cudaFree(pp.reward[i]); cudaFree(pp.done[i]);
  }
  if (pp.copy) cudaStreamDestroy(pp.copy);
  memset(&pp, 0, sizeof(pp));
}

// Creates the host pipeline's copy stream, events and staging buffers for n envs.  On failure the caller releases
// what was created.
int setup_pipe(lmz_env *h, size_t n) {
  auto &pp = h->pipe;
  LMZ_CUDA(cudaStreamCreateWithFlags(&pp.copy, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    LMZ_CUDA(cudaEventCreateWithFlags(&pp.ready[i], cudaEventDisableTiming));
    LMZ_CUDA(cudaEventCreateWithFlags(&pp.drained[i], cudaEventDisableTiming));
    LMZ_CUDA(cudaMalloc(&pp.act[i], n * 8));
    LMZ_CUDA(cudaMalloc(&pp.reward[i], n * sizeof(float)));
    LMZ_CUDA(cudaMalloc(&pp.done[i], n));
  }
  pp.init = true;
  return LMZ_OK;
}

// n copies of `value` to device memory, through a host buffer of at most 2^20 words
cudaError_t fill_u32(uint32_t *dst, size_t n, uint32_t value) {
  const std::vector<uint32_t> chunk(n < (1u << 20) ? n : (1u << 20), value);
  cudaError_t e = cudaSuccess;
  for (size_t off = 0; off < n && e == cudaSuccess; off += chunk.size()) {
    const size_t cnt = (n - off < chunk.size()) ? n - off : chunk.size();
    e = cudaMemcpy(dst + off, chunk.data(), cnt * sizeof(uint32_t), cudaMemcpyHostToDevice);
  }
  return e;
}

// ------------------------------------------------------------------ observation memory (lmz_alloc_obs)
// The driver's virtual-memory calls, fetched through the runtime so that the library keeps linking cudart only.
struct DriverVmm {
  decltype(&cuDeviceGetAttribute) attribute = nullptr;
  decltype(&cuMemGetAllocationGranularity) granularity = nullptr;
  decltype(&cuMemCreate) create = nullptr;
  decltype(&cuMemGetAllocationPropertiesFromHandle) properties = nullptr;
  decltype(&cuMemAddressReserve) reserve = nullptr;
  decltype(&cuMemMap) map = nullptr;
  decltype(&cuMemSetAccess) set_access = nullptr;
  decltype(&cuMemUnmap) unmap = nullptr;
  decltype(&cuMemRelease) release = nullptr;
  decltype(&cuMemAddressFree) address_free = nullptr;
  bool ok = false;
};

const DriverVmm &vmm() {
  static const DriverVmm d = [] {
    DriverVmm v;
    auto get = [](const char *name, auto &fn) {
      void *p = nullptr;
      cudaDriverEntryPointQueryResult q;
      if (cudaGetDriverEntryPointByVersion(name, &p, 12000, cudaEnableDefault, &q) != cudaSuccess ||
          q != cudaDriverEntryPointSuccess)
        p = nullptr;
      fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(p);
      return p != nullptr;
    };
    v.ok = get("cuDeviceGetAttribute", v.attribute) && get("cuMemGetAllocationGranularity", v.granularity) &&
           get("cuMemCreate", v.create) && get("cuMemGetAllocationPropertiesFromHandle", v.properties) &&
           get("cuMemAddressReserve", v.reserve) && get("cuMemMap", v.map) && get("cuMemSetAccess", v.set_access) &&
           get("cuMemUnmap", v.unmap) && get("cuMemRelease", v.release) && get("cuMemAddressFree", v.address_free);
    return v;
  }();
  return d;
}

// One lmz_alloc_obs allocation: `chunks` empty = cudaMalloc memory, else the physical chunks mapped back to back
// from `ptr`.
struct ObsAlloc {
  void *ptr = nullptr;
  int device = 0;
  size_t size = 0;
  std::vector<std::pair<CUmemGenericAllocationHandle, size_t>> chunks;
};
std::mutex g_obs_mu;
std::vector<ObsAlloc> g_obs;

void release_vmm(ObsAlloc &a) {
  const DriverVmm &d = vmm();
  const CUdeviceptr base = reinterpret_cast<CUdeviceptr>(a.ptr);
  size_t off = 0;
  for (const auto &c : a.chunks) {
    d.unmap(base + off, c.second);
    d.release(c.first);
    off += c.second;
  }
  d.address_free(base, a.size);
  a.chunks.clear();
}

// Compressible memory (cuMemCreate with generic compression) for `bytes`, rounded up to the granularity: physical
// chunks of at most OBS_CHUNK_BYTES mapped into one reserved range.  Returns the bytes the driver made compressible;
// on 0 nothing is kept and `a` is untouched.
constexpr size_t OBS_CHUNK_BYTES = size_t(1) << 30;
int64_t alloc_compressible(int device, size_t bytes, ObsAlloc &a) {
  const DriverVmm &d = vmm();
  int supported = 0;
  if (!d.ok || d.attribute(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, device) != CUDA_SUCCESS ||
      !supported)
    return 0;
  CUmemAllocationProp prop;
  memset(&prop, 0, sizeof(prop));
  prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
  prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
  prop.location.id = device;
  prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
  size_t gran = 0;
  if (d.granularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || gran == 0) return 0;
  ObsAlloc v;
  v.device = device;
  v.size = (bytes + gran - 1) / gran * gran;
  CUdeviceptr base = 0;
  if (d.reserve(&base, v.size, gran, 0, 0) != CUDA_SUCCESS) return 0;
  v.ptr = reinterpret_cast<void *>(base);
  int64_t granted = 0;
  for (size_t off = 0; off < v.size;) {
    const size_t sz = v.size - off < OBS_CHUNK_BYTES ? v.size - off : OBS_CHUNK_BYTES;
    CUmemGenericAllocationHandle hd;
    if (d.create(&hd, sz, &prop, 0) != CUDA_SUCCESS) break;
    if (d.map(base + off, sz, 0, hd, 0) != CUDA_SUCCESS) {
      d.release(hd);
      break;
    }
    v.chunks.push_back({hd, sz});
    CUmemAllocationProp got;
    if (d.properties(&got, hd) == CUDA_SUCCESS && got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC)
      granted += (int64_t)sz;
    off += sz;
  }
  size_t mapped = 0;
  for (const auto &c : v.chunks) mapped += c.second;
  CUmemAccessDesc acc;
  memset(&acc, 0, sizeof(acc));
  acc.location = prop.location;
  acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
  if (mapped != v.size || d.set_access(base, v.size, &acc, 1) != CUDA_SUCCESS || granted == 0) {
    release_vmm(v);
    return 0;
  }
  a = std::move(v);
  return granted;
}

}  // namespace

// ================================================================== exports
extern "C" {

int lmz_abi_version(void) { return LMZ_ABI_VERSION; }

const char *lmz_last_error(void) { return g_err; }

void lmz_default_config(lmz_config *cfg) {
  if (!cfg) return;
  memset(cfg, 0, sizeof(*cfg));
  cfg->struct_size = (int32_t)sizeof(lmz_config);
  cfg->variant = LMZ_V0;
  cfg->num_envs = 1;
  cfg->autoreset = 1;
  cfg->random_ball = 1;     // lmaze_env.py:25
  cfg->random_goal = 1;     // lmaze_env_v3.py:104
  cfg->render_mode = LMZ_RENDER_TMA;
}

int lmz_obs_shape(int32_t variant, int64_t shape[3]) {
  if (!shape) return fail(LMZ_ERR_INVALID, "shape is NULL");
  const VariantInfo *v = variant_info(variant);
  if (!v) return unknown_variant(variant);
  shape[0] = v->C; shape[1] = shape[2] = v->S;
  return LMZ_OK;
}

int lmz_local_obs_shape(int32_t variant, int64_t shape[3]) {
  if (!shape) return fail(LMZ_ERR_INVALID, "shape is NULL");
  const VariantInfo *v = variant_info(variant);
  if (!v || !v->CL) return fail(LMZ_ERR_UNSUPPORTED, "only lmaze-v5/v6 have a local observation");
  shape[0] = v->CL; shape[1] = shape[2] = v->S;
  return LMZ_OK;
}

int lmz_state_cols(int32_t variant) {
  const VariantInfo *v = variant_info(variant);
  return v ? v->state_cols : unknown_variant(variant);
}

int lmz_num_actions(int32_t variant) {
  const VariantInfo *v = variant_info(variant);
  return v ? v->num_actions : unknown_variant(variant);
}

int lmz_num_layouts(int32_t variant) {
  const VariantInfo *v = variant_info(variant);
  return v ? v->num_layouts : unknown_variant(variant);
}

int lmz_layout_ex(int32_t variant, int32_t index, char *cells) {
  if (!cells) return fail(LMZ_ERR_INVALID, "cells is NULL");
  const int nl = lmz_num_layouts(variant);
  if (nl < 0) return nl;
  if (index < 1 || index > nl) return fail(LMZ_ERR_INVALID, "layout index %d outside 1..%d", index, nl);
  if (!variant_info(variant)->cells) { v2_cells(index, cells); return LMZ_OK; }
  return lmz_layout(variant, cells);
}

int lmz_obs_desc(int32_t variant, int32_t obs_mode, int64_t shape[3], int32_t *elem_bytes) {
  if (!shape) return fail(LMZ_ERR_INVALID, "shape is NULL");
  if (int rc = lmz_obs_shape(variant, shape)) return rc;
  const VariantInfo *v = variant_info(variant);
  if (obs_mode == LMZ_OBS_COMPACT) {
    shape[1] = shape[2] = v->foveal ? 5 : v->G;        // foveal variants: the 5x5 crops, as float32
    if (elem_bytes) *elem_bytes = v->foveal ? 4 : 1;
  } else if (obs_mode == LMZ_OBS_BITS) {
    if (!v->bits_bytes)
      return fail(LMZ_ERR_UNSUPPORTED, "bit-packed observations exist for the full-view variants (v0, v3) only");
    shape[0] = v->bits_bytes;                          // one row of bytes per env
    shape[1] = shape[2] = 1;
    if (elem_bytes) *elem_bytes = 1;
  } else if (obs_mode == LMZ_OBS_FULL) {
    if (elem_bytes) *elem_bytes = 4;
  } else {
    return fail(LMZ_ERR_INVALID, "unknown obs_mode %d", obs_mode);
  }
  return LMZ_OK;
}

int lmz_grid_size(int32_t variant) {
  const VariantInfo *v = variant_info(variant);
  return v ? v->G : unknown_variant(variant);
}

int lmz_layout(int32_t variant, char *cells) {
  const VariantInfo *v = variant_info(variant);
  if (!v) return unknown_variant(variant);
  if (!v->cells) return lmz_layout_ex(variant, 1, cells);
  if (!cells) return fail(LMZ_ERR_INVALID, "cells is NULL");
  memcpy(cells, v->cells, (size_t)v->G * v->G);
  return LMZ_OK;
}

int lmz_create(const lmz_config *cfg, lmz_env **out) {
  if (!cfg || !out) return fail(LMZ_ERR_INVALID, "cfg/out is NULL");
  *out = nullptr;
  if (cfg->struct_size != (int32_t)sizeof(lmz_config))
    return fail(LMZ_ERR_INVALID, "lmz_config.struct_size %d != %d: header/library mismatch", cfg->struct_size,
                (int)sizeof(lmz_config));
  const VariantInfo *v = variant_info(cfg->variant);
  if (!v)
    return fail(LMZ_ERR_UNSUPPORTED,
                "variant %d is not built (supported: 0 = lmaze-v0, 2 = lmaze-v2, 3 = lmaze-v3, 4 = lmaze-v4, "
                "5 = lmaze-v5/v6)", cfg->variant);
  if (cfg->num_envs < 1) return fail(LMZ_ERR_INVALID, "num_envs must be >= 1 (got %lld)", (long long)cfg->num_envs);
  if (cfg->env_id0 < 0) return fail(LMZ_ERR_INVALID, "env_id0 must be >= 0");
  if (cfg->render_mode != LMZ_RENDER_TMA && cfg->render_mode != LMZ_RENDER_ST128 &&
      cfg->render_mode != LMZ_RENDER_INCREMENTAL)
    return fail(LMZ_ERR_INVALID, "unknown render_mode %d", cfg->render_mode);
  if (cfg->render_mode == LMZ_RENDER_INCREMENTAL && v->foveal)
    return fail(LMZ_ERR_UNSUPPORTED, "incremental render needs a full-view variant (v0, v3): a foveal crop changes entirely every step");
  for (int i = 0; i < 2; ++i)
    if (cfg->reserved[i] != 0) return fail(LMZ_ERR_INVALID, "lmz_config.reserved must be zero");
  if (cfg->obs_mode != LMZ_OBS_FULL && cfg->obs_mode != LMZ_OBS_COMPACT && cfg->obs_mode != LMZ_OBS_BITS)
    return fail(LMZ_ERR_INVALID, "unknown obs_mode %d", cfg->obs_mode);
  if (cfg->obs_mode == LMZ_OBS_BITS && !v->bits_bytes)
    return fail(LMZ_ERR_UNSUPPORTED, "bit-packed observations exist for the full-view variants (v0, v3) only");
  {
    const int t = cfg->tune[0];
    if (t < 0 || t > 1024 || (t & 31))
      return fail(LMZ_ERR_INVALID, "tune[0] (threads per CTA) must be 0 or a multiple of 32 up to 1024");
    if (cfg->tune[1] < 0 || cfg->tune[1] > 4) return fail(LMZ_ERR_INVALID, "tune[1] (L2 policy) must be 0..4");
    if (cfg->tune[2] < 0 || cfg->tune[2] > 32) return fail(LMZ_ERR_INVALID, "tune[2] (CTAs per SM cap) must be 0..32");
    if (cfg->tune[3] < 0 || (cfg->tune[3] & 15)) return fail(LMZ_ERR_INVALID, "tune[3] (bulk split) must be a multiple of 16");
  }
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0)
    return fail(LMZ_ERR_CUDA, "no CUDA device available (%s); this library has no CPU path",
                ce == cudaSuccess ? "device count is 0" : cudaGetErrorString(ce));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(LMZ_ERR_INVALID, "device %d out of range", cfg->device);
  DeviceGuard guard(cfg->device);
  cudaDeviceProp prop;
  LMZ_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major < 10)
    return fail(LMZ_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a only", cfg->device,
                prop.major, prop.minor);

  lmz_env *h = new (std::nothrow) lmz_env();
  if (!h) return fail(LMZ_ERR_INVALID, "out of host memory");
  memset(h, 0, sizeof(*h));
  h->cfg = *cfg;
  h->num_sms = prop.multiProcessorCount;
  h->win_lo = 0; h->win_n = cfg->num_envs;
  h->var = v;
  std::vector<unsigned char> blob;
  v->build_blob(v->cells, blob, h->n_cand, h->s_cell, h->x_cell);
  const size_t n = (size_t)cfg->num_envs;
  // The per-env state arrays are padded to whole 32-env tiles: the compact foveal kernel fetches a tile's words as
  // fixed-size bulk copies (lmz_fov.cuh).  The padding is zeroed so that those copies read defined words.
  const size_t n32 = (n + 31) & ~(size_t)31;
  cudaError_t e = cudaSuccess;
  auto alloc_zero = [&](auto **ptr, size_t bytes) {
    if (e == cudaSuccess) e = cudaMalloc(ptr, bytes);
    if (e == cudaSuccess) e = cudaMemset(*ptr, 0, bytes);
  };
  alloc_zero(&h->state, n32 * sizeof(uint32_t));
  alloc_zero(&h->goal_count, n32 * sizeof(uint32_t));
  alloc_zero(&h->episode, n * sizeof(uint32_t));
  alloc_zero(&h->stats, (lmz::NUM_STATS + 3) * sizeof(unsigned long long));
  if (v->hier) alloc_zero(&h->aux2, n32 * sizeof(uint32_t));
  if (v->has_visit) {
    alloc_zero(&h->visit, n * 324 * sizeof(float));     // state[2], the float visit layer (lmaze_env_v4.py:106-113)
    alloc_zero(&h->hist, n32 * 64);                     // the visit history (lmz_v2.cuh): empty = an all-zero layer
  }
  if (e == cudaSuccess) e = cudaMalloc(&h->blob, blob.size());
  if (e == cudaSuccess) e = cudaMemcpy(h->blob, blob.data(), blob.size(), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    // Before the first reset every env sits on the 'S' cell with the goal on 'X'
    // (lmaze_env_v3.py:119-123 starts at 0,0; any in-range cell keeps the kernels' +-1 lookups in the table).
    lmz::EnvRegs r;
    r.x = h->s_cell / v->G; r.y = h->s_cell % v->G; r.gx = h->x_cell / v->G; r.gy = h->x_cell % v->G;
    r.step = 0; r.rcode = lmz::RC_NEG_ZERO;
    uint32_t packed = (cfg->variant == LMZ_V0) ? lmz::V0::pack(r) : lmz::V3::pack(r);
    if (v->hier) {                         // maze 1, everything on 'S', goal on 'X' (the state reset() would leave there)
      lmz::V5Regs r5;
      r5.L = 1; r5.x = r5.x1 = r5.fx1 = r5.fgx = r5.lx = 4; r5.y = r5.y1 = r5.fy1 = r5.fgy = r5.ly = 4; r5.gx = 8; r5.gy = 8;
      r5.fga = 12; r5.step = 0; r5.fstep = 0; r5.ld = 0; r5.gd = 0; r5.vt = 0;
      uint32_t w1, w2;
      lmz::v5_pack(r5, packed, w1, w2);
      if (e == cudaSuccess) e = fill_u32(h->goal_count, n, w1);
      if (e == cudaSuccess) e = fill_u32(h->aux2, n, w2);
    } else if (v->foveal) {                // maze 1, ball on 'S', goal on 'X', no previous action
      lmz::V2Regs r2;
      r2.L = 1; r2.x = r2.px = 4; r2.y = r2.py = 4; r2.gx = 8; r2.gy = 8; r2.a = -1; r2.step = 0; r2.vt = 0;
      uint32_t aux;
      lmz::v2_pack(r2, packed, aux);
      if (e == cudaSuccess) e = fill_u32(h->goal_count, n, aux);
    }
    if (e == cudaSuccess) e = fill_u32(h->state, n, packed);
  }
  if (e != cudaSuccess) {
    fail(LMZ_ERR_CUDA, "device allocation/initialisation failed: %s", cudaGetErrorString(e));
    lmz_destroy(h);
    return LMZ_ERR_CUDA;
  }
  *out = h;
  return LMZ_OK;
}

int lmz_destroy(lmz_env *h) {
  if (!h) return LMZ_OK;
  DeviceGuard guard(h->cfg.device);
  cudaFree(h->state); cudaFree(h->goal_count); cudaFree(h->episode); cudaFree(h->blob); cudaFree(h->stats);
  cudaFree(h->act_stage); cudaFree(h->visit); cudaFree(h->hist); cudaFree(h->aux2);
  release_pipe(h);
  delete h;
  return LMZ_OK;
}

int lmz_alloc_obs(int32_t device, int64_t bytes, int32_t flags, void **ptr, int64_t *compressed_bytes) {
  if (!ptr || bytes <= 0) return fail(LMZ_ERR_INVALID, "lmz_alloc_obs: ptr must not be NULL and bytes must be > 0");
  if (flags & ~LMZ_OBS_MEM_COMPRESSIBLE) return fail(LMZ_ERR_INVALID, "lmz_alloc_obs: unknown flags 0x%x", flags);
  *ptr = nullptr;
  if (compressed_bytes) *compressed_bytes = 0;
  int count = 0;
  LMZ_CUDA(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count) return fail(LMZ_ERR_INVALID, "lmz_alloc_obs: no CUDA device %d", device);
  DeviceGuard guard(device);
  LMZ_CUDA(cudaFree(nullptr));      // the device's primary context, current for the driver calls
  ObsAlloc a;
  const int64_t granted = (flags & LMZ_OBS_MEM_COMPRESSIBLE) ? alloc_compressible(device, (size_t)bytes, a) : 0;
  if (granted == 0) {               // not asked for, not supported, or refused: plain memory
    a.device = device;
    a.size = (size_t)bytes;
    LMZ_CUDA(cudaMalloc(&a.ptr, a.size));
  }
  *ptr = a.ptr;
  if (compressed_bytes) *compressed_bytes = granted;
  std::lock_guard<std::mutex> lock(g_obs_mu);
  g_obs.push_back(std::move(a));
  return LMZ_OK;
}

int lmz_free_obs(void *ptr) {
  if (!ptr) return LMZ_OK;
  ObsAlloc a;
  {
    std::lock_guard<std::mutex> lock(g_obs_mu);
    auto it = g_obs.begin();
    while (it != g_obs.end() && it->ptr != ptr) ++it;
    if (it == g_obs.end()) return fail(LMZ_ERR_INVALID, "lmz_free_obs: %p was not returned by lmz_alloc_obs", ptr);
    a = std::move(*it);
    g_obs.erase(it);
  }
  DeviceGuard guard(a.device);
  if (a.chunks.empty()) {
    LMZ_CUDA(cudaFree(a.ptr));
    return LMZ_OK;
  }
  LMZ_CUDA(cudaDeviceSynchronize());      // as cudaFree does: work still writing the memory finishes first
  release_vmm(a);
  return LMZ_OK;
}

int lmz_bind(lmz_env *h, void *obs, float *reward, uint8_t *done) {
  if (int rc = check_handle(h)) return rc;
  if (!reward || !done) return fail(LMZ_ERR_INVALID, "reward/done must not be NULL");
  if ((reinterpret_cast<uintptr_t>(obs) & 15u) != 0) return fail(LMZ_ERR_INVALID, "obs must be 16-byte aligned");
  if ((reinterpret_cast<uintptr_t>(reward) & 3u) != 0) return fail(LMZ_ERR_INVALID, "reward must be 4-byte aligned");
  h->obs = obs; h->reward = reward; h->done = done; h->bound = true;
  h->win_lo = 0; h->win_n = h->cfg.num_envs;
  h->obs_synced = false;
  return LMZ_OK;
}

static int check_obs_dl(lmz_env *h, DLManagedTensor *obs, int64_t rows, void **po) {
  int64_t shape[3];
  int32_t elem = 0;
  if (int rc = lmz_obs_desc(h->cfg.variant, h->cfg.obs_mode, shape, &elem)) return rc;
  // f32 [rows][C][side][side] or u8 [rows][C][G][G]; bit-packed rows are u8 [rows][bytes]
  const bool bits = h->cfg.obs_mode == LMZ_OBS_BITS;
  const Want w{"obs", elem == 4 ? (uint8_t)kDLFloat : (uint8_t)kDLUInt, (uint8_t)(8 * elem), bits ? 2 : 4,
               {rows, shape[0], shape[1], shape[2]}, 16};
  return check_dl(h, obs, w, po);
}

int lmz_bind_dl(lmz_env *h, DLManagedTensor *obs, DLManagedTensor *reward, DLManagedTensor *done) {
  if (int rc = check_handle(h)) return rc;
  const int64_t n = h->cfg.num_envs;
  void *po = nullptr, *pr = nullptr, *pd = nullptr;
  if (obs)
    if (int rc = check_obs_dl(h, obs, n, &po)) return rc;
  if (int rc = check_dl(h, reward, per_env(h, "reward", kDLFloat, 32), &pr)) return rc;
  if (int rc = check_dl(h, done, per_env(h, "done", kDLUInt, 8), &pd)) return rc;
  return lmz_bind(h, po, static_cast<float *>(pr), static_cast<uint8_t *>(pd));
}

int lmz_set_window(lmz_env *h, void *obs, int64_t env_lo, int64_t env_count) {
  if (int rc = check_handle(h)) return rc;
  if (int rc = check_bound(h)) return rc;
  if (h->var->hier) return fail(LMZ_ERR_UNSUPPORTED, "lmz_set_window is not built for lmaze-v5/v6");
  if (!obs) return fail(LMZ_ERR_INVALID, "obs is NULL");
  if ((reinterpret_cast<uintptr_t>(obs) & 15u) != 0) return fail(LMZ_ERR_INVALID, "obs must be 16-byte aligned");
  if (env_lo < 0 || env_count < 1 || env_lo + env_count > h->cfg.num_envs)
    return fail(LMZ_ERR_INVALID, "window [%lld, %lld) outside [0, %lld)", (long long)env_lo,
                (long long)(env_lo + env_count), (long long)h->cfg.num_envs);
  h->obs = obs; h->win_lo = env_lo; h->win_n = env_count;
  h->obs_synced = false;
  return LMZ_OK;
}

int lmz_set_window_dl(lmz_env *h, DLManagedTensor *obs, int64_t env_lo) {
  if (int rc = check_handle(h)) return rc;
  if (!obs) return fail(LMZ_ERR_INVALID, "obs: DLManagedTensor is NULL");
  if (obs->dl_tensor.ndim < 1) return fail(LMZ_ERR_INVALID, "obs: ndim %d, want 4", obs->dl_tensor.ndim);
  const int64_t rows = obs->dl_tensor.shape[0];
  void *po = nullptr;
  if (int rc = check_obs_dl(h, obs, rows, &po)) return rc;
  return lmz_set_window(h, po, env_lo, rows);
}

int lmz_reset(lmz_env *h, const uint8_t *mask, const int32_t *spawn, void *stream) {
  if (int rc = check_handle(h)) return rc;
  if (int rc = check_bound(h)) return rc;
  if ((reinterpret_cast<uintptr_t>(spawn) & 15u) != 0) return fail(LMZ_ERR_INVALID, "spawn must be 16-byte aligned");
  DeviceGuard guard(h->cfg.device);
  lmz::KParams p = base_params(h);
  p.mode = lmz::MODE_RESET; p.mask = mask; p.spawn = reinterpret_cast<const int4 *>(spawn);
  return launch_env(h, p, static_cast<cudaStream_t>(stream));
}

int lmz_reset_dl(lmz_env *h, DLManagedTensor *mask, DLManagedTensor *spawn, void *stream) {
  if (int rc = check_handle(h)) return rc;
  const int64_t n = h->cfg.num_envs;
  void *pm = nullptr, *ps = nullptr;
  if (mask)
    if (int rc = check_dl(h, mask, per_env(h, "mask", kDLUInt, 8), &pm)) return rc;
  if (spawn) {
    const Want w{"spawn", kDLInt, 32, 2, {n, 4, 0, 0}, 16};
    if (int rc = check_dl(h, spawn, w, &ps)) return rc;
  }
  return lmz_reset(h, static_cast<const uint8_t *>(pm), static_cast<const int32_t *>(ps), stream);
}

int lmz_step(lmz_env *h, const void *actions, int32_t action_dtype, const int32_t *spawn, void *stream) {
  if (int rc = check_handle(h)) return rc;
  if (int rc = check_bound(h)) return rc;
  if (!actions) return fail(LMZ_ERR_INVALID, "actions is NULL");
  if (int rc = check_action_dtype(action_dtype, "action dtype")) return rc;
  if ((reinterpret_cast<uintptr_t>(spawn) & 15u) != 0) return fail(LMZ_ERR_INVALID, "spawn must be 16-byte aligned");
  DeviceGuard guard(h->cfg.device);
  lmz::KParams p = base_params(h);
  p.mode = lmz::MODE_STEP; p.actions = actions; p.action_dtype = action_dtype;
  p.spawn = reinterpret_cast<const int4 *>(spawn);
  return launch_env(h, p, static_cast<cudaStream_t>(stream));
}

int lmz_step_dl(lmz_env *h, DLManagedTensor *actions, DLManagedTensor *spawn, void *stream) {
  if (int rc = check_handle(h)) return rc;
  const int64_t n = h->cfg.num_envs;
  void *pa = nullptr, *ps = nullptr;
  int ad = 0;
  if (int rc = check_dl(h, actions, per_env(h, "actions", ANY_INT), &pa, &ad)) return rc;
  if (spawn) {
    const Want w{"spawn", kDLInt, 32, 2, {n, 4, 0, 0}, 16};
    if (int rc = check_dl(h, spawn, w, &ps)) return rc;
  }
  return lmz_step(h, pa, ad, static_cast<const int32_t *>(ps), stream);
}

int lmz_step_host(lmz_env *h, const void *actions_host, int32_t action_dtype, float *reward_host,
                  uint8_t *done_host, void *obs_host, void *stream) {
  if (int rc = check_handle(h)) return rc;
  if (int rc = check_bound(h)) return rc;
  if (!actions_host || !reward_host || !done_host) return fail(LMZ_ERR_INVALID, "host buffers must not be NULL");
  if (int rc = check_action_dtype(action_dtype, "action dtype")) return rc;
  if (obs_host && !h->obs) return fail(LMZ_ERR_STATE, "obs_host given but no device obs buffer is bound");
  if (h->var->hier) return fail(LMZ_ERR_UNSUPPORTED, "lmz_step_host is not built for lmaze-v5/v6");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t n = (size_t)h->cfg.num_envs;
  if (!h->act_stage) LMZ_CUDA(cudaMalloc(&h->act_stage, n * 8));
  LMZ_CUDA(cudaMemcpyAsync(h->act_stage, actions_host, n * action_bytes(action_dtype), cudaMemcpyHostToDevice, s));
  if (int rc = lmz_step(h, h->act_stage, action_dtype, nullptr, stream)) return rc;
  LMZ_CUDA(cudaMemcpyAsync(reward_host, h->reward, n * sizeof(float), cudaMemcpyDeviceToHost, s));
  LMZ_CUDA(cudaMemcpyAsync(done_host, h->done, n, cudaMemcpyDeviceToHost, s));
  if (obs_host) {
    LMZ_CUDA(cudaMemcpyAsync(obs_host, h->obs, (size_t)h->win_n * obs_row_bytes(h), cudaMemcpyDeviceToHost, s));
  }
  LMZ_CUDA(cudaStreamSynchronize(s));
  return LMZ_OK;
}

// Double-buffered host step.  Slot s = k & 1 owns a device staging buffer for the actions and device buffers for
// reward / done / (compact or bit-packed) obs that the kernel of step k writes DIRECTLY; the D2H copies of step k run
// on the handle's copy stream while the caller's stream already carries step k+1's H2D + kernel into the other slot.
int lmz_step_host_async(lmz_env *h, const void *actions_host, int32_t action_dtype, float *reward_host,
                        uint8_t *done_host, void *obs_host, void *stream, int32_t *ticket) {
  if (int rc = check_handle(h)) return rc;
  if (int rc = check_bound(h)) return rc;
  if (!actions_host || !reward_host || !done_host || !ticket) return fail(LMZ_ERR_INVALID, "host buffers / ticket must not be NULL");
  if (int rc = check_action_dtype(action_dtype, "action dtype")) return rc;
  if (h->var->hier) return fail(LMZ_ERR_UNSUPPORTED, "lmz_step_host_async is not built for lmaze-v5/v6");
  if (obs_host && h->cfg.obs_mode == LMZ_OBS_FULL)
    return fail(LMZ_ERR_UNSUPPORTED, "the full f32 observation is not double-buffered (2 x N x %zu bytes of HBM): a host "
                "consumer takes obs_mode compact or bits; pass obs_host = NULL to keep the observation on the device",
                (size_t)h->var->obs_bytes);
  if (obs_host && h->win_n != h->cfg.num_envs) return fail(LMZ_ERR_STATE, "obs_host needs the whole batch bound, not a render window");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t n = (size_t)h->cfg.num_envs;
  const size_t row = obs_row_bytes(h);
  auto &pp = h->pipe;
  if (!pp.init)
    if (int rc = setup_pipe(h, n)) {
      release_pipe(h);
      return rc;
    }
  const int slot = (int)(pp.k & 1);
  if (obs_host && !pp.obs[slot]) LMZ_CUDA(cudaMalloc(&pp.obs[slot], n * row));
  if (pp.inflight[slot]) LMZ_CUDA(cudaStreamWaitEvent(s, pp.drained[slot], 0));   // slot's previous copies must be out
  LMZ_CUDA(cudaMemcpyAsync(pp.act[slot], actions_host, n * action_bytes(action_dtype), cudaMemcpyHostToDevice, s));
  lmz::KParams p = base_params(h);
  p.mode = lmz::MODE_STEP; p.actions = pp.act[slot]; p.action_dtype = action_dtype;
  p.reward = pp.reward[slot]; p.done = pp.done[slot];
  if (obs_host) p.obs = pp.obs[slot];                       // compact / bits rows are rewritten whole every step
  if (int rc = launch_env(h, p, s)) return rc;
  LMZ_CUDA(cudaEventRecord(pp.ready[slot], s));
  LMZ_CUDA(cudaStreamWaitEvent(pp.copy, pp.ready[slot], 0));
  LMZ_CUDA(cudaMemcpyAsync(reward_host, pp.reward[slot], n * sizeof(float), cudaMemcpyDeviceToHost, pp.copy));
  LMZ_CUDA(cudaMemcpyAsync(done_host, pp.done[slot], n, cudaMemcpyDeviceToHost, pp.copy));
  if (obs_host) LMZ_CUDA(cudaMemcpyAsync(obs_host, pp.obs[slot], n * row, cudaMemcpyDeviceToHost, pp.copy));
  LMZ_CUDA(cudaEventRecord(pp.drained[slot], pp.copy));
  pp.inflight[slot] = true;
  pp.k += 1;
  *ticket = slot;
  return LMZ_OK;
}

int lmz_step_host_wait(lmz_env *h, int32_t ticket) {
  if (int rc = check_handle(h)) return rc;
  if (ticket < 0 || ticket > 1 || !h->pipe.init || !h->pipe.inflight[ticket])
    return fail(LMZ_ERR_STATE, "no step in flight for ticket %d", ticket);
  DeviceGuard guard(h->cfg.device);
  LMZ_CUDA(cudaEventSynchronize(h->pipe.drained[ticket]));
  return LMZ_OK;
}

int lmz_render(lmz_env *h, void *stream) {
  if (int rc = check_handle(h)) return rc;
  if (int rc = check_bound(h)) return rc;
  if (!h->obs) return fail(LMZ_ERR_STATE, "no obs buffer bound");
  DeviceGuard guard(h->cfg.device);
  lmz::KParams p = base_params(h);
  p.mode = lmz::MODE_RENDER;
  p.tile_begin = h->win_lo / 32;                     // only the tiles that intersect the window
  p.tile_end = (h->win_lo + h->win_n + 31) / 32;
  return launch_env(h, p, static_cast<cudaStream_t>(stream));
}

static int rollout_impl(lmz_env *h, int32_t T, const void *actions, int32_t action_dtype, float *rewards,
                        uint8_t *reward_codes, uint8_t *dones, void *stream);

int lmz_rollout(lmz_env *h, int32_t T, const void *actions, int32_t action_dtype, float *rewards, uint8_t *dones,
                void *stream) {
  if (!rewards) return fail(LMZ_ERR_INVALID, "rewards/dones must not be NULL");
  return rollout_impl(h, T, actions, action_dtype, rewards, nullptr, dones, stream);
}

int lmz_rollout_codes(lmz_env *h, int32_t T, const void *actions, int32_t action_dtype, uint8_t *reward_codes,
                      uint8_t *dones, void *stream) {
  if (!reward_codes) return fail(LMZ_ERR_INVALID, "reward_codes/dones must not be NULL");
  return rollout_impl(h, T, actions, action_dtype, nullptr, reward_codes, dones, stream);
}

static int rollout_impl(lmz_env *h, int32_t T, const void *actions, int32_t action_dtype, float *rewards,
                        uint8_t *reward_codes, uint8_t *dones, void *stream) {
  if (int rc = check_handle(h)) return rc;
  if (T < 1) return fail(LMZ_ERR_INVALID, "T must be >= 1 (got %d)", T);
  if (h->var->hier)
    return fail(LMZ_ERR_UNSUPPORTED, "lmaze-v5/v6 roll out through lmz_hier_rollout (planner goals + actor actions)");
  if (!dones) return fail(LMZ_ERR_INVALID, "rewards/dones must not be NULL");
  if (actions)
    if (int rc = check_action_dtype(action_dtype, "action dtype")) return rc;
  DeviceGuard guard(h->cfg.device);
  lmz::KParams p = base_params(h);
  p.mode = lmz::MODE_STEP; p.actions = actions; p.action_dtype = action_dtype;
  p.reward = rewards; p.reward_code = reward_codes; p.done = dones; p.obs = nullptr; p.T = T; p.t0 = h->rollout_t;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int rc = h->cfg.variant == LMZ_V0   ? launch_rollout_v<lmz::V0>(h, p, s)
           : h->cfg.variant == LMZ_V3 ? launch_rollout_v<lmz::V3>(h, p, s)
           : h->cfg.variant == LMZ_V2 ? launch_fov_rollout<lmz::V2>(h, p, s)
                                      : launch_fov_rollout<lmz::V4>(h, p, s);
  if (rc == LMZ_OK) {
    h->rollout_t += (uint64_t)T;
    h->obs_synced = false;               // every ball / goal moved and nothing was rendered (incremental render)
  }
  return rc;
}

// rewards as f32 [T, n], or (codes) as u8 reward codes [T, n]
static int rollout_dl(lmz_env *h, int32_t T, DLManagedTensor *actions, DLManagedTensor *rewards, bool codes,
                      DLManagedTensor *dones, void *stream) {
  if (int rc = check_handle(h)) return rc;
  void *pa = nullptr, *pr = nullptr, *pd = nullptr;
  int ad = 0;
  if (actions)
    if (int rc = check_dl(h, actions, per_step(h, "actions", T, ANY_INT), &pa, &ad)) return rc;
  const Want wr = codes ? per_step(h, "reward_codes", T, kDLUInt, 8) : per_step(h, "rewards", T, kDLFloat, 32);
  if (int rc = check_dl(h, rewards, wr, &pr)) return rc;
  if (int rc = check_dl(h, dones, per_step(h, "dones", T, kDLUInt, 8), &pd)) return rc;
  if (codes) return lmz_rollout_codes(h, T, pa, ad, static_cast<uint8_t *>(pr), static_cast<uint8_t *>(pd), stream);
  return lmz_rollout(h, T, pa, ad, static_cast<float *>(pr), static_cast<uint8_t *>(pd), stream);
}

int lmz_rollout_dl(lmz_env *h, int32_t T, DLManagedTensor *actions, DLManagedTensor *rewards, DLManagedTensor *dones,
                   void *stream) {
  return rollout_dl(h, T, actions, rewards, false, dones, stream);
}

int lmz_rollout_codes_dl(lmz_env *h, int32_t T, DLManagedTensor *actions, DLManagedTensor *reward_codes,
                         DLManagedTensor *dones, void *stream) {
  return rollout_dl(h, T, actions, reward_codes, true, dones, stream);
}

static int state_xfer(lmz_env *h, int32_t *io, int set, void *stream) {
  if (int rc = check_handle(h)) return rc;
  if (!io) return fail(LMZ_ERR_INVALID, "state buffer is NULL");
  DeviceGuard guard(h->cfg.device);
  const int64_t n = h->cfg.num_envs;
  const int64_t blocks = ceil_div(n, 256);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  unsigned int *errors = reinterpret_cast<unsigned int *>(h->stats + lmz::NUM_STATS);
  if (h->var->hier)
    return launch(h, lmz::lmz_state_v5_kernel, blocks, 256, 0, s, n, h->state, h->goal_count, h->aux2, h->episode, io,
                  set, errors);
  if (h->var->foveal)
    return launch(h, lmz::lmz_state_v2_kernel, blocks, 256, 0, s, n, h->state, h->goal_count, h->episode, io, set, errors);
  return launch(h, h->cfg.variant == LMZ_V0 ? lmz::lmz_state_kernel<lmz::V0> : lmz::lmz_state_kernel<lmz::V3>, blocks,
                256, 0, s, n, h->state, h->goal_count, h->episode, io, set, h->blob, errors);
}

int lmz_get_state(lmz_env *h, int32_t *out, void *stream) { return state_xfer(h, out, 0, stream); }
int lmz_set_state(lmz_env *h, const int32_t *in, void *stream) {
  if (h) h->obs_synced = false;            // positions change behind the obs tensor's back
  return state_xfer(h, const_cast<int32_t *>(in), 1, stream);
}

static int state_xfer_dl(lmz_env *h, DLManagedTensor *t, int set, void *stream) {
  if (int rc = check_handle(h)) return rc;
  void *pt = nullptr;
  const Want w{"state", kDLInt, 32, 2, {h->cfg.num_envs, h->var->state_cols, 0, 0}, 4};
  if (int rc = check_dl(h, t, w, &pt)) return rc;
  return state_xfer(h, static_cast<int32_t *>(pt), set, stream);
}
int lmz_get_state_dl(lmz_env *h, DLManagedTensor *out, void *stream) { return state_xfer_dl(h, out, 0, stream); }
int lmz_set_state_dl(lmz_env *h, DLManagedTensor *in, void *stream) {
  if (h) h->obs_synced = false;
  return state_xfer_dl(h, in, 1, stream);
}

static int visit_xfer(lmz_env *h, float *buf, int set, void *stream) {
  if (int rc = check_handle(h)) return rc;
  if (!h->var->has_visit) return fail(LMZ_ERR_UNSUPPORTED, "only lmaze-v4/v5/v6 have a visit layer");
  if (!buf) return fail(LMZ_ERR_INVALID, "visit buffer is NULL");
  DeviceGuard guard(h->cfg.device);
  // the handle keeps the layer as its history (lmz_v2.cuh, "visit layer"); it crosses the ABI as values
  const int64_t n = h->cfg.num_envs;
  const bool v5 = h->var->hier;
  return launch(h, lmz::lmz_visit_xfer_kernel, ceil_div(n * 324, 256), 256, 0, static_cast<cudaStream_t>(stream), n,
                h->visit, h->hist, v5 ? h->state : h->goal_count, v5 ? 25 : 16, buf, set);
}
int lmz_get_visit(lmz_env *h, float *out, void *stream) { return visit_xfer(h, out, 0, stream); }
int lmz_set_visit(lmz_env *h, const float *in, void *stream) { return visit_xfer(h, const_cast<float *>(in), 1, stream); }
static int visit_xfer_dl(lmz_env *h, DLManagedTensor *t, int set, void *stream) {
  if (int rc = check_handle(h)) return rc;
  void *pt = nullptr;
  const Want w{"visit", kDLFloat, 32, 3, {h->cfg.num_envs, 18, 18, 0}, 4};
  if (int rc = check_dl(h, t, w, &pt)) return rc;
  return visit_xfer(h, static_cast<float *>(pt), set, stream);
}
int lmz_get_visit_dl(lmz_env *h, DLManagedTensor *out, void *stream) { return visit_xfer_dl(h, out, 0, stream); }
int lmz_set_visit_dl(lmz_env *h, DLManagedTensor *in, void *stream) { return visit_xfer_dl(h, in, 1, stream); }

// ---- lmaze-v5 / v6 -------------------------------------------------------------------------------
int lmz_bind_local(lmz_env *h, float *loc_obs, float *local_reward, uint8_t *local_done, uint8_t *loc_err,
                   uint8_t *foveal_goal) {
  if (int rc = check_handle(h)) return rc;
  if (!h->var->hier) return fail(LMZ_ERR_UNSUPPORTED, "lmz_bind_local: only lmaze-v5/v6 have local outputs");
  if (!local_reward || !local_done) return fail(LMZ_ERR_INVALID, "local_reward/local_done must not be NULL");
  if ((reinterpret_cast<uintptr_t>(loc_obs) & 15u) != 0) return fail(LMZ_ERR_INVALID, "loc_obs must be 16-byte aligned");
  if ((reinterpret_cast<uintptr_t>(local_reward) & 3u) != 0)
    return fail(LMZ_ERR_INVALID, "local_reward must be 4-byte aligned");
  h->loc_obs = loc_obs; h->reward2 = local_reward; h->done2 = local_done; h->loc_err = loc_err;
  h->fgoal_out = foveal_goal; h->local_bound = true;
  return LMZ_OK;
}

int lmz_bind_local_dl(lmz_env *h, DLManagedTensor *loc_obs, DLManagedTensor *local_reward, DLManagedTensor *local_done,
                      DLManagedTensor *loc_err, DLManagedTensor *foveal_goal) {
  if (int rc = check_handle(h)) return rc;
  const int64_t n = h->cfg.num_envs;
  void *po = nullptr, *pr = nullptr, *pd = nullptr, *pe = nullptr, *pg = nullptr;
  if (loc_obs) {
    const int64_t side = h->cfg.obs_mode == LMZ_OBS_COMPACT ? 5 : lmz::V5::S;
    const Want w{"loc_obs", kDLFloat, 32, 4, {n, lmz::V5::CL, side, side}, 16};
    if (int rc = check_dl(h, loc_obs, w, &po)) return rc;
  }
  if (int rc = check_dl(h, local_reward, per_env(h, "local_reward", kDLFloat, 32), &pr)) return rc;
  if (int rc = check_dl(h, local_done, per_env(h, "local_done", kDLUInt, 8), &pd)) return rc;
  if (loc_err)
    if (int rc = check_dl(h, loc_err, per_env(h, "loc_err", kDLUInt, 8), &pe)) return rc;
  if (foveal_goal)
    if (int rc = check_dl(h, foveal_goal, per_env(h, "foveal_goal", kDLUInt, 8), &pg)) return rc;
  return lmz_bind_local(h, static_cast<float *>(po), static_cast<float *>(pr), static_cast<uint8_t *>(pd),
                        static_cast<uint8_t *>(pe), static_cast<uint8_t *>(pg));
}

// plannerStep on the envs of `mask` (null: all), or with auto_mask on the envs whose foveal goal is done
static int planner_step(const char *fn, lmz_env *h, const void *goals, int32_t goal_dtype, const uint8_t *mask,
                        bool auto_mask, void *stream) {
  if (int rc = check_handle(h)) return rc;
  if (!h->var->hier) return fail(LMZ_ERR_UNSUPPORTED, "%s: only lmaze-v5/v6 have a planner level", fn);
  if (int rc = check_bound(h)) return rc;
  if (!goals) return fail(LMZ_ERR_INVALID, "goals is NULL");
  if (int rc = check_action_dtype(goal_dtype, "goal dtype")) return rc;
  DeviceGuard guard(h->cfg.device);
  lmz::KParams p = base_params(h);
  p.mode = lmz::MODE_PLANNER; p.actions = goals; p.action_dtype = goal_dtype; p.mask = mask; p.auto_mask = auto_mask;
  return launch_env(h, p, static_cast<cudaStream_t>(stream));
}

int lmz_planner_step(lmz_env *h, const void *goals, int32_t goal_dtype, const uint8_t *mask, void *stream) {
  return planner_step("lmz_planner_step", h, goals, goal_dtype, mask, false, stream);
}

int lmz_planner_step_auto(lmz_env *h, const void *goals, int32_t goal_dtype, void *stream) {
  return planner_step("lmz_planner_step_auto", h, goals, goal_dtype, nullptr, true, stream);
}

int lmz_planner_step_auto_dl(lmz_env *h, DLManagedTensor *goals, void *stream) {
  if (int rc = check_handle(h)) return rc;
  void *pg = nullptr;
  int ad = 0;
  if (int rc = check_dl(h, goals, per_env(h, "goals", ANY_INT), &pg, &ad)) return rc;
  return lmz_planner_step_auto(h, pg, ad, stream);
}

int lmz_hier_step_host(lmz_env *h, const void *goals_host, const void *actions_host, int32_t dtype,
                       float *global_reward_host, float *local_reward_host, uint8_t *global_done_host,
                       uint8_t *local_done_host, void *stream) {
  if (int rc = check_handle(h)) return rc;
  if (!h->var->hier) return fail(LMZ_ERR_UNSUPPORTED, "lmz_hier_step_host: only lmaze-v5/v6");
  if (int rc = check_bound(h)) return rc;
  if (!h->local_bound) return fail(LMZ_ERR_STATE, "local outputs not bound: call lmz_bind_local first");
  if (!goals_host || !actions_host || !global_reward_host || !local_reward_host || !global_done_host || !local_done_host)
    return fail(LMZ_ERR_INVALID, "host buffers must not be NULL");
  if (int rc = check_action_dtype(dtype, "dtype")) return rc;
  DeviceGuard guard(h->cfg.device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t n = (size_t)h->cfg.num_envs;
  if (!h->act_stage) LMZ_CUDA(cudaMalloc(&h->act_stage, n * 16));       // goals | actions
  const size_t esz = action_bytes(dtype);
  unsigned char *stage = static_cast<unsigned char *>(h->act_stage);
  LMZ_CUDA(cudaMemcpyAsync(stage, goals_host, n * esz, cudaMemcpyHostToDevice, s));
  LMZ_CUDA(cudaMemcpyAsync(stage + n * 8, actions_host, n * esz, cudaMemcpyHostToDevice, s));
  if (int rc = lmz_planner_step_auto(h, stage, dtype, stream)) return rc;
  if (int rc = lmz_step(h, stage + n * 8, dtype, nullptr, stream)) return rc;
  LMZ_CUDA(cudaMemcpyAsync(global_reward_host, h->reward, n * sizeof(float), cudaMemcpyDeviceToHost, s));
  LMZ_CUDA(cudaMemcpyAsync(local_reward_host, h->reward2, n * sizeof(float), cudaMemcpyDeviceToHost, s));
  LMZ_CUDA(cudaMemcpyAsync(global_done_host, h->done, n, cudaMemcpyDeviceToHost, s));
  LMZ_CUDA(cudaMemcpyAsync(local_done_host, h->done2, n, cudaMemcpyDeviceToHost, s));
  LMZ_CUDA(cudaStreamSynchronize(s));
  return LMZ_OK;
}

int lmz_hier_rollout(lmz_env *h, int32_t T, const void *goals, const void *actions, int32_t dtype, float *global_rewards,
                     float *local_rewards, uint8_t *global_dones, uint8_t *local_dones, void *stream) {
  if (int rc = check_handle(h)) return rc;
  if (!h->var->hier) return fail(LMZ_ERR_UNSUPPORTED, "lmz_hier_rollout: only lmaze-v5/v6");
  if (T < 1) return fail(LMZ_ERR_INVALID, "T must be >= 1 (got %d)", T);
  if (!global_rewards || !local_rewards || !global_dones || !local_dones)
    return fail(LMZ_ERR_INVALID, "reward / done buffers must not be NULL");
  if ((goals == nullptr) != (actions == nullptr))
    return fail(LMZ_ERR_INVALID, "goals and actions must both be given, or both NULL (device-side random goals and actions)");
  if (actions)
    if (int rc = check_action_dtype(dtype, "dtype")) return rc;
  DeviceGuard guard(h->cfg.device);
  lmz::KParams p = base_params(h);
  p.mode = lmz::MODE_STEP; p.actions = actions; p.goals = goals; p.action_dtype = dtype;
  p.reward = global_rewards; p.reward2 = local_rewards; p.done = global_dones; p.done2 = local_dones;
  p.obs = nullptr; p.obs2 = nullptr; p.loc_err = nullptr; p.T = T; p.t0 = h->rollout_t;
  const int rc = launch_fov_rollout<lmz::V5>(h, p, static_cast<cudaStream_t>(stream));
  if (rc == LMZ_OK) h->rollout_t += (uint64_t)T;
  return rc;
}

int lmz_hier_rollout_dl(lmz_env *h, int32_t T, DLManagedTensor *goals, DLManagedTensor *actions, DLManagedTensor *global_rewards,
                        DLManagedTensor *local_rewards, DLManagedTensor *global_dones, DLManagedTensor *local_dones,
                        void *stream) {
  if (int rc = check_handle(h)) return rc;
  void *pg = nullptr, *pa = nullptr, *pr = nullptr, *pr2 = nullptr, *pd = nullptr, *pd2 = nullptr;
  int ad = 0, gd = 0;
  if (actions)
    if (int rc = check_dl(h, actions, per_step(h, "actions", T, ANY_INT), &pa, &ad)) return rc;
  if (goals) {
    if (int rc = check_dl(h, goals, per_step(h, "goals", T, ANY_INT), &pg, &gd)) return rc;
    if (actions && gd != ad) return fail(LMZ_ERR_INVALID, "goals and actions must have the same dtype");
  }
  if (int rc = check_dl(h, global_rewards, per_step(h, "global_rewards", T, kDLFloat, 32), &pr)) return rc;
  if (int rc = check_dl(h, local_rewards, per_step(h, "local_rewards", T, kDLFloat, 32), &pr2)) return rc;
  if (int rc = check_dl(h, global_dones, per_step(h, "global_dones", T, kDLUInt, 8), &pd)) return rc;
  if (int rc = check_dl(h, local_dones, per_step(h, "local_dones", T, kDLUInt, 8), &pd2)) return rc;
  return lmz_hier_rollout(h, T, pg, pa, ad, static_cast<float *>(pr), static_cast<float *>(pr2), static_cast<uint8_t *>(pd),
                          static_cast<uint8_t *>(pd2), stream);
}

int lmz_planner_step_dl(lmz_env *h, DLManagedTensor *goals, DLManagedTensor *mask, void *stream) {
  if (int rc = check_handle(h)) return rc;
  void *pg = nullptr, *pm = nullptr;
  int ad = 0;
  if (int rc = check_dl(h, goals, per_env(h, "goals", ANY_INT), &pg, &ad)) return rc;
  if (mask)
    if (int rc = check_dl(h, mask, per_env(h, "mask", kDLUInt, 8), &pm)) return rc;
  return lmz_planner_step(h, pg, ad, static_cast<const uint8_t *>(pm), stream);
}

int lmz_safe_goal(lmz_env *h, const int64_t *draws, int32_t n_draws, uint8_t *goals_out, int32_t *used_out, void *stream) {
  if (int rc = check_handle(h)) return rc;
  if (!h->var->hier) return fail(LMZ_ERR_UNSUPPORTED, "lmz_safe_goal: only lmaze-v6 (variant 5) has safeFovealGoal");
  if (!goals_out) return fail(LMZ_ERR_INVALID, "goals_out is NULL");
  if (draws && n_draws < 1) return fail(LMZ_ERR_INVALID, "n_draws must be >= 1 when draws are given");
  DeviceGuard guard(h->cfg.device);
  const int64_t n = h->cfg.num_envs;
  return launch(h, lmz::lmz_safe_goal_kernel<lmz::V5>, ceil_div(n, 256), 256, 0, static_cast<cudaStream_t>(stream), n,
                h->state, h->aux2, h->episode, h->blob, reinterpret_cast<const long long *>(draws), n_draws, goals_out,
                used_out, h->cfg.seed, (uint64_t)h->cfg.env_id0);
}

int lmz_safe_goal_dl(lmz_env *h, DLManagedTensor *draws, DLManagedTensor *goals_out, DLManagedTensor *used_out,
                     void *stream) {
  if (int rc = check_handle(h)) return rc;
  const int64_t n = h->cfg.num_envs;
  void *pd = nullptr, *pg = nullptr, *pu = nullptr;
  int32_t nd = 0;
  if (draws) {
    if (draws->dl_tensor.ndim != 2) return fail(LMZ_ERR_INVALID, "draws: ndim %d, want 2", draws->dl_tensor.ndim);
    nd = (int32_t)draws->dl_tensor.shape[1];
    const Want w{"draws", kDLInt, 64, 2, {n, nd, 0, 0}, 8};
    if (int rc = check_dl(h, draws, w, &pd)) return rc;
  }
  if (int rc = check_dl(h, goals_out, per_env(h, "goals_out", kDLUInt, 8), &pg)) return rc;
  if (used_out)
    if (int rc = check_dl(h, used_out, per_env(h, "used_out", kDLInt, 32), &pu)) return rc;
  return lmz_safe_goal(h, static_cast<const int64_t *>(pd), nd, static_cast<uint8_t *>(pg), static_cast<int32_t *>(pu), stream);
}

int lmz_stats(lmz_env *h, int64_t *out_host, int64_t *errors_host, void *stream) {
  if (int rc = check_handle(h)) return rc;
  if (!out_host) return fail(LMZ_ERR_INVALID, "out_host is NULL");
  DeviceGuard guard(h->cfg.device);
  unsigned long long tmp[lmz::NUM_STATS + 1];
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  LMZ_CUDA(cudaMemcpyAsync(tmp, h->stats, sizeof(tmp), cudaMemcpyDeviceToHost, s));
  LMZ_CUDA(cudaStreamSynchronize(s));
  for (int i = 0; i < lmz::NUM_STATS; ++i) out_host[i] = (int64_t)tmp[i];
  if (errors_host) *errors_host = (int64_t)(tmp[lmz::NUM_STATS] & 0xffffffffull);
  return LMZ_OK;
}

int lmz_stats_reset(lmz_env *h, void *stream) {
  if (int rc = check_handle(h)) return rc;
  DeviceGuard guard(h->cfg.device);
  LMZ_CUDA(cudaMemsetAsync(h->stats, 0, (lmz::NUM_STATS + 1) * sizeof(unsigned long long),
                           static_cast<cudaStream_t>(stream)));
  return LMZ_OK;
}

int64_t lmz_launch_count(const lmz_env *h) { return h ? h->launches : 0; }

}  // extern "C"
