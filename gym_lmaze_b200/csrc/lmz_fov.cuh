// lmz_fov.cuh -- the fused reset / step / render kernel of the FOVEAL variants: lmaze-v2, lmaze-v4
// (lmz_v2.cuh) and the planner / actor env lmaze-v5 / v6 (lmz_v5.cuh, which adds plannerStep and a second,
// "local" observation tensor).
//
// An observation here is C planes of 5x5 values, each upsampled x7 to 35x35 floats
// (lmaze_env_v2.py:197-203, lmaze_env_v4.py:241-247, lmaze_env_v5.py:337-343,372-378): 6,125 / 8,575
// floats per env, NOT a multiple of 4, so an env row is not 16-byte aligned -- but four consecutive rows
// are.  The render therefore works on GROUPS of 4 envs: a group's image is OBS_FLOATS float4s, and because
// every cell value repeats 7 times along a row, the four floats of one float4 take at most TWO different
// cell values (a prefix of k floats from cell A, the rest from cell B).  One host-built table entry per
// float4 -- A:11 | B:11 | k:3, A and B indexing the group's [4][NSLOT][25] value planes -- turns the whole
// render into: 1 table load, 2 value loads, 3 selects, 1 streaming 128-bit store.  (The first version looked
// every FLOAT up through a byte table and was issue-bound at 91 % issue-slot utilisation, 5.8 TB/s on v4.)
//
// CTA organisation: ONE small persistent CTA per SM; tiles of 32 envs are handed out by the global work counter.
// Warp 0 is a dedicated producer: it runs the tile's 32 transitions (one env per lane, state in registers) and
// expands each env's 25-bit planes into float planes in shared memory, one tile ahead of the rendering warps and
// one tile ahead of its OWN loads (next tile's index, state words, actions).  For the variants with a float visit
// layer (v4, v5) the same producer warp keeps the layer: as its HISTORY (lmz_v2.cuh, "visit layer") -- 64 bytes of
// window centres per env, loaded with the state words; an averaging appends a byte, and the two 5x5 visit crops an
// observation shows are folded from the history in registers (bit-identical to the reference's float expression) and
// go into the same value planes.  No layer is read or written.  Everything is double buffered; one __syncthreads per
// tile.  FEWER rendering warps reach a HIGHER write bandwidth (tools/fov_sweep2.py): 1 producer + 3 rendering warps per SM.
#pragma once
#include "lmz_v2.cuh"
#include "lmz_v5.cuh"

#ifndef LMZ_VISIT_PROD
#define LMZ_VISIT_PROD 32     // v4 / v5: producer threads (round 1 used 128 for a full-layer pass; the visit history needs one warp)
#endif
#ifndef LMZ_V2_PROD
#define LMZ_V2_PROD 32    // v2: one dedicated producer warp (0: warp 0 produces, then renders with the others)
#endif

namespace lmz {

// state[2] = (state[2] + visitMap) / 2, which the reference evaluates in float64 and stores as float32
// (lmaze_env_v4.py:116-119,211-214; lmaze_env_v5.py:308-312).  For 0 <= v <= 1 the float32 expression below is
// bit-identical to float32((float64(v) + m) * 0.5): v/2 is a single correctly rounded operation either way, and
// v + 1 is either exact in float64 (v >= 2^-29) -- then both paths round the same exact value at the same bit --
// or so close to 1 that both give exactly 1.0 before the halving.  (Checked bit for bit by the v4 / v5 parity
// tests over the whole layer.)  It keeps FP64 and the f32<->f64 conversions off the producers' path.
__device__ __forceinline__ float visit_average(float v, bool in_window) {
  return in_window ? __fmul_rn(__fadd_rn(v, 1.0f), 0.5f) : __fmul_rn(v, 0.5f);
}

// ---- the visit layer of one 32-env tile, one env per lane (whole warp must call) --------------------------------
// The layer is kept as its HISTORY (lmz_v2.cuh, "visit layer"): hw = the lane's 64 history bytes (loaded with the
// state words a tile ahead), entry k = the window centre of averaging k.  info / vinfo: the lane's FovLane words;
// plane_cur / plane_prev: the lane's two 25-float visit planes in shared memory (crop at the ball / crop at the
// previous window, both showing the layer AFTER this call's update -- the reference's retStatelast is a view of the
// live state, lmaze_env_v4.py:122,258-259), written when want_planes.
struct VisitHist {
  uint32_t w[16];
};
__device__ __forceinline__ VisitHist visit_hist_of(const FovPre &pre) {
  VisitHist h;
#pragma unroll
  for (int k = 0; k < 4; ++k) { h.w[4 * k] = pre.h[k].x; h.w[4 * k + 1] = pre.h[k].y; h.w[4 * k + 2] = pre.h[k].z; h.w[4 * k + 3] = pre.h[k].w; }
  return h;
}
__device__ __forceinline__ uint32_t visit_entry(int x, int y) { return (uint32_t)(((x - 2) << 4) | (y - 2)); }
// bits i = 0..4 with |o + i - h| <= 2: the rows (columns) of the 5-window at origin o that entry centre h covers
__device__ __forceinline__ uint32_t visit_cover(int h, int o) {
  const int d = h - 2 - o;                                   // covered indices: [d, d + 4] cut to [0, 4]
  const int lo = d < 0 ? 0 : d, hi = d + 4 > 4 ? 4 : d + 4;
  return hi >= lo ? ((2u << hi) - (1u << lo)) : 0u;
}

// Packed float32 pairs (Blackwell FFMA2, PTX fma.rn.f32x2): two independent correctly rounded f32 fmas in one issue
// slot -- tools/ffma2_bench.cu: 1.46x the lane-fma rate of FFMA on a B200.  Each half is an ordinary IEEE fma.rn.f32.
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}

// The layer's values on TWO 5x5 windows (origins (ax, ay) and (bx, by) = centre - 2) after the first `T` averagings
// of the history.  The reference's fold  v <- RN((v + m_k) / 2), k = 0 .. T-1  is evaluated as the WEIGHTED SUM
//     u <- RN(u + m_k * 2^(k-T)),   u = v * 2^-(T-1-k) after entry k,
// which is the same float32 sequence scaled by a power of two (scaling by 2^n commutes with rounding: T <= 64, so
// nothing leaves the normal range; the product m_k * 2^(k-T) is exact) -- u after the last entry IS v, bit for bit
// (tests: every v4 / v5 parity run compares the whole layer; DESIGN.md 3.5).  In this form an entry is ONE fma per
// cell, fma(r_i, c_j, u): r_i = 1.0 / 0.0 (entry covers row i of the window, and k < this lane's T), c_j = 2^(k-T) /
// 0.0 (covers column j) -- 10 + 10 selects per entry instead of one per cell, and the 50 fmas go two per instruction
// (f2_fma; accumulator pairs: row i of a window = (0,1), (2,3), and column 4 of window A pairs with column 4 of
// window B).  `tmax` >= T is warp-uniform (the loop bound); no branch depends on a lane's own T.
// The loop over the history words is ROLLED on purpose (one word = 4 entries per trip): fully unrolled, the fold was
// 64 x ~150 instructions = 150 KB of straight-line code that every warp streams through once per tile -- far beyond
// the instruction caches; the compact kernel then waited for instruction FETCH instead of issuing (steady state,
// v4 compact: 0.85 G env-steps/s unrolled, 4.1 G rolled).  Registers cannot be indexed by the trip count, so the
// words are ROTATED through h.w[0] instead (15 moves per trip); `h` is consumed.
// `Told` of the T entries come from the history words `h`; entry T-1 is `last` when T > Told (the entry this very
// step appends: it is folded from registers, so the words never have to be modified -- a store into h.w[runtime index]
// sends the whole array to local memory).
__device__ __forceinline__ void visit_fold2(VisitHist &h, int Told, int T, uint32_t last, int tmax, int ax, int ay,
                                            int bx, int by, float *va, float *vb) {
  uint64_t acc[25];
#pragma unroll
  for (int c = 0; c < 25; ++c) acc[c] = 0ull;                // (+0.0f, +0.0f)
  const int kend = (tmax + 3) & ~3;                          // (warp-uniform)
#pragma unroll 1
  for (int k0 = 0; k0 <= kend; k0 += 4) {                    // the trip k0 == kend folds `last`
    const bool tail = k0 == kend;
    const uint32_t w = tail ? last : h.w[0];
#pragma unroll
    for (int g = 0; g < 15; ++g) h.w[g] = h.w[g + 1];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      if (tail && b > 0) break;                              // (uniform)
      const int k = tail ? T - 1 : k0 + b;
      const bool live = tail ? T > Told : k < Told;
      const float wk = __uint_as_float(live ? (uint32_t)(k - T + 127) << 23 : 0u);   // 2^(k-T); 0 for a dead entry
      const uint32_t e = (w >> (8 * b)) & 255u;
      const int hx = (int)(e >> 4), hy = (int)(e & 15u);      // centre - 2 = the entry's window origin
      // row i of window A (absolute row ax + i) is covered by the entry iff 0 <= ax + i - hx < 5
      const int rxa = ax - hx, rya = ay - hy, rxb = bx - hx, ryb = by - hy;
      float ca[5], cb[5], ra[5], rb[5];
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        ca[j] = ((unsigned)(rya + j) < 5u) ? wk : 0.0f;
        cb[j] = ((unsigned)(ryb + j) < 5u) ? wk : 0.0f;
        ra[j] = ((unsigned)(rxa + j) < 5u) ? 1.0f : 0.0f;
        rb[j] = ((unsigned)(rxb + j) < 5u) ? 1.0f : 0.0f;
      }
      const uint64_t ca01 = f2_pack(ca[0], ca[1]), ca23 = f2_pack(ca[2], ca[3]);
      const uint64_t cb01 = f2_pack(cb[0], cb[1]), cb23 = f2_pack(cb[2], cb[3]);
      const uint64_t c44 = f2_pack(ca[4], cb[4]);
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        const uint64_t ra2 = f2_pack(ra[i], ra[i]), rb2 = f2_pack(rb[i], rb[i]), rab = f2_pack(ra[i], rb[i]);
        acc[2 * i] = f2_fma(ra2, ca01, acc[2 * i]);
        acc[2 * i + 1] = f2_fma(ra2, ca23, acc[2 * i + 1]);
        acc[10 + 2 * i] = f2_fma(rb2, cb01, acc[10 + 2 * i]);
        acc[11 + 2 * i] = f2_fma(rb2, cb23, acc[11 + 2 * i]);
        acc[20 + i] = f2_fma(rab, c44, acc[20 + i]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    f2_unpack(acc[2 * i], va[i * 5], va[i * 5 + 1]);
    f2_unpack(acc[2 * i + 1], va[i * 5 + 2], va[i * 5 + 3]);
    f2_unpack(acc[10 + 2 * i], vb[i * 5], vb[i * 5 + 1]);
    f2_unpack(acc[11 + 2 * i], vb[i * 5 + 2], vb[i * 5 + 3]);
    f2_unpack(acc[20 + i], va[i * 5 + 4], vb[i * 5 + 4]);
  }
}

// one cell of the layer from the history of lane `src` (warp-cooperative materialisation: every lane a different cell)
__device__ __forceinline__ float visit_fold_cell(const VisitHist &h, int src, int T, int x, int y) {
  float v = 0.0f;
#pragma unroll
  for (int g = 0; g < 16; ++g) {
    const uint32_t w = __shfl_sync(0xffffffffu, h.w[g], src);
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const uint32_t e = (w >> (8 * b)) & 255u;
      const int hx = (int)(e >> 4) + 2, hy = (int)(e & 15u) + 2;
      const bool in = (unsigned)(x - hx + 2) < 5u && (unsigned)(y - hy + 2) < 5u;
      if (4 * g + b < T) v = visit_avg1(v, in);
    }
  }
  return v;
}

// The whole visit step of a tile.  Rare whole-layer work first, warp-cooperatively: an averaging in DIRECT mode is the
// literal full pass over the env's layer in memory, and the averaging that finds the history full materialises the
// layer from the history on the way.  Then every lane: append / reset its history (a one-byte store of the new entry)
// and fold the two windows (history mode), or read them from the layer (direct mode).
// Returns true when vc / vp hold the lane's two visit crops (the CALLER stores them into its value planes: the compact
// kernel first waits, after the fold, for the bulk copy that is still reading those planes).
template <class W>
__device__ __forceinline__ bool visit_step(const KParams &p, int64_t e0, int lane, bool valid, uint32_t info,
                                           uint32_t vinfo, bool want_planes, VisitHist &h, float *vc, float *vp) {
  constexpr int GG = W::G * W::G;
  const uint32_t op = valid ? (vinfo & 7u) : (uint32_t)VOP_READ;
  const int tpre = (vinfo >> 3) & 127, tpost = (vinfo >> 10) & 127;
  const int bx = info & 31, by = (info >> 5) & 31, px = (info >> 10) & 31, py = (info >> 15) & 31;
  unsigned full = __ballot_sync(0xffffffffu, op == VOP_FULL);
  if (full) {
    while (full) {
      const int src = __ffs(full) - 1;
      full &= full - 1;
      const int st = __shfl_sync(0xffffffffu, tpre, src);
      const int sx = __shfl_sync(0xffffffffu, bx, src), sy = __shfl_sync(0xffffffffu, by, src);
      float *layer = p.visit + (e0 + src) * GG;
      for (int c0 = 0; c0 < GG; c0 += 32) {                 // (uniform trip count: the shuffles inside need the whole warp)
        const int c = c0 + lane, x = c / W::G, y = c - x * W::G;
        float v = (st == VT_DIRECT) ? 0.0f : visit_fold_cell(h, src, st, x, y);
        if (c < GG) {
          if (st == VT_DIRECT) v = __ldcg(layer + c);
          const bool in_cur = (unsigned)(x - sx + 2) < 5u && (unsigned)(y - sy + 2) < 5u;
          __stcg(layer + c, visit_average(v, in_cur));
        }
      }
    }
    __syncwarp();                                           // the cooperative stores are visible to the owning lane
  }
  const bool direct = valid && tpost == VT_DIRECT;
  const bool hmode = valid && !direct;                      // history mode
  // history mode: a reset empties the history (v4: its first averaging is the spawn cell), an averaging appends
  // ONE BYTE at position tpost - 1
  const bool app = hmode && (op == VOP_AVG || (op == VOP_RESET && W::VT_RESET == 1));
  const uint32_t last = visit_entry(bx, by);
  if (app) p.hist[(e0 + lane) * HIST_MAX + (tpost - 1)] = (uint8_t)last;
  const int need = (hmode && want_planes) ? tpost : 0;      // entries this lane folds ...
  const int told = need - ((app && need > 0) ? 1 : 0);      // ... of which these come from the loaded words
  const int tmax = __reduce_max_sync(0xffffffffu, told);
  const bool any = __any_sync(0xffffffffu, need > 0);
  if (any) visit_fold2(h, told, need, last, tmax, bx - 2, by - 2, px - 2, py - 2, vc, vp);   // (need == 0: all zeros)
  if (direct && want_planes) {                              // direct mode: the windows come from the layer in memory
    const float *vis = p.visit + (e0 + lane) * GG;
#pragma unroll
    for (int k = 0; k < 25; ++k) {
      vc[k] = __ldcg(vis + (bx - 2 + k / 5) * W::G + (by - 2 + k % 5));
      vp[k] = __ldcg(vis + (px - 2 + k / 5) * W::G + (py - 2 + k % 5));
    }
  }
  if (!any && !direct) {
#pragma unroll
    for (int k = 0; k < 25; ++k) { vc[k] = 0.0f; vp[k] = 0.0f; }
  }
  return valid && want_planes;
}

// lmz_get_visit / lmz_set_visit: the layer crosses the ABI as values.  get: the fold of the env's history (or the layer
// in memory for an env in direct mode).  set: the values are stored as given and the env goes to direct mode until its
// next reset (arbitrary values have no history).
// tword: the state word that carries the env's T field (v4: aux word, bits 16-22; v5: w0, bits 25-31).
__global__ void lmz_visit_xfer_kernel(int64_t n, float *visit, const uint8_t *hist, uint32_t *tword, int shift, float *io, int set) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * 324) return;
  const int64_t e = idx / 324;
  const int cell = (int)(idx - e * 324);
  if (set) {
    visit[idx] = io[idx];
    if (cell == 0) tword[e] = (tword[e] & ~(127u << shift)) | ((uint32_t)VT_DIRECT << shift);
    return;
  }
  const int T = (int)((tword[e] >> shift) & 127u);
  if (T == VT_DIRECT) { io[idx] = visit[idx]; return; }
  const int x = cell / 18, y = cell - x * 18;
  const uint8_t *hp = hist + e * HIST_MAX;
  float v = 0.0f;
  for (int k = 0; k < T; ++k) {
    const int hx = (hp[k] >> 4) + 2, hy = (hp[k] & 15) + 2;
    v = visit_avg1(v, (unsigned)(x - hx + 2) < 5u && (unsigned)(y - hy + 2) < 5u);
  }
  io[idx] = v;
}

template <int ID, int C>
__device__ __forceinline__ FovLane<5> fov_lane(const Fov<ID, C> *, const KParams &p, int64_t e,
                                               const FovTables<Fov<ID, C>> &t, const unsigned char *, const FovPre &pre) {
  return v2_lane<Fov<ID, C>>(p, e, t, pre);
}
__device__ __forceinline__ V5Lane fov_lane(const V5 *, const KParams &p, int64_t e, const FovTables<V5> &t,
                                           const unsigned char *smem, const FovPre &pre) {
  return v5_lane<V5>(p, e, t, smem, pre);
}

template <class W, int THREADS>
__global__ void __launch_bounds__(THREADS) lmz_env_fov_kernel(const KParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t s_flags[2][2];         // [buf][0 obs, 1 local obs]: bit l = env l of the tile is written
  __shared__ long long s_tile[2];
  constexpr int PROD = (W::NVIS > 0) ? LMZ_VISIT_PROD : LMZ_V2_PROD;   // threads that never render
  constexpr int CTHREADS = THREADS - PROD;
  static_assert(CTHREADS >= 32, "need at least one rendering warp");
  static_assert((uint32_t)CTHREADS < W::OBS_FLOATS, "index stepping assumes fewer threads than entries");
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  stage_blob<W>(smem, &bar, p.blob);
  const FovTables<W> t(smem);
  float *vals = reinterpret_cast<float *>(smem + W::BLOB_BYTES);          // [2][32][NSLOT][25]
  const int64_t tiles = p.tile_end;
  const bool need_visit = W::NVIS > 0 && p.mode != MODE_PLANNER;
  WarpStats ws;

  // Warp 0 runs ONE TILE AHEAD of its own loads: when it turns to a tile, the tile's index was grabbed and its
  // state words / actions (and, for the visit variants, the envs' 64-byte visit histories: 2 KB of contiguous
  // memory per tile) were requested a whole tile time earlier, so no DRAM or atomic round trip -- several
  // microseconds each under a saturated write stream -- sits between two tiles of the producer.
  int64_t tl_next = 0;                       // warp 0: the tile produce() turns to next
  FovPre pre_next;                           // ... and its preloaded words (this lane's env)
  pre_next.w0 = pre_next.w1 = pre_next.w2 = 0u; pre_next.act = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) pre_next.h[k] = make_uint4(0u, 0u, 0u, 0u);
  // (Measured, tools/_gpu15.sh: making these loads unconditional and broadcasting the grabbed tile index late --
  // both of which help the compact kernel below -- costs THIS kernel 28 % on v2, 305 -> 221 M env-steps/s.)
  auto prefetch = [&](int64_t tl) {          // warp 0: start everything tile `tl` will need
    const int64_t e = tl * 32 + lane;
    if (tl < tiles && e < p.n) pre_next = fov_preload<W>(p, e);
    tl_next = tl;
  };
  auto grab = [&]() { return warp_grab(p, lane, 1); };
  auto produce = [&](int buf) {              // warp 0 only
    const int64_t tl = tl_next;
    const FovPre pre = pre_next;
    const int64_t tl_after = grab();         // in flight while this tile's transitions run
    const int64_t e = tl * 32 + lane;
    const bool valid = tl < tiles && e < p.n;
    FovLane<W::NBIT> v;
    v.o = LaneOut::blank(); v.info = 0; v.vinfo = 0; v.rfov = false; v.rloc = false;
    if (valid) v = fov_lane(static_cast<const W *>(nullptr), p, e, t, smem, pre);
    if (p.mode == MODE_STEP) ws.add(valid, v.o);
    float *mv = vals + (buf * 32 + lane) * W::VALS;
#ifndef LMZ_DEBUG_NO_VISIT                   // (tuning builds only: how fast is the kernel without the visit layer?)
    if (W::NVIS > 0 && need_visit) {         // append to / fold the visit history: the two 5x5 visit crops
      VisitHist vh = visit_hist_of(pre);
      float vc[25], vp[25];
      if (visit_step<W>(p, tl * 32, lane, valid, v.info, v.vinfo, valid && v.rfov, vh, vc, vp)) {
#pragma unroll
        for (int k = 0; k < 25; ++k) { mv[W::VIS_SLOT0 * 25 + k] = vc[k]; mv[W::VIS_SLOT1 * 25 + k] = vp[k]; }
      }
    }
#endif
    if (valid && (v.rfov || v.rloc)) {       // 25-bit planes -> float planes (lane stride VALS is odd: no bank conflicts)
#pragma unroll
      for (int b = 0; b < W::NBIT; ++b) expand_plane(v.mask[b], mv + W::bit_slot(b) * 25);
    }
    const unsigned ff = __ballot_sync(0xffffffffu, valid && v.rfov);
    const unsigned fl = __ballot_sync(0xffffffffu, valid && v.rloc);
    if (lane == 0) { s_flags[buf][0] = ff; s_flags[buf][1] = fl; s_tile[buf] = tl; }
    prefetch(tl_after);
  };
  auto pick = [](uint32_t en, const float *gv) -> uint4 { return f4_pick(en, gv); };

  if (warp == 0) { prefetch(grab()); produce(0); }
  for (int buf = 0;; buf ^= 1) {
    __syncthreads();                          // tile(buf) is complete; buffers buf^1 are free again
    const int64_t tile = s_tile[buf];
    if (tile >= tiles) break;
    if (PROD > 0 && tid < PROD) {
      if (warp == 0) produce(buf ^ 1);
      continue;
    }
    if (PROD == 0 && warp == 0) produce(buf ^ 1);
    const int ctid = tid - PROD;
    const float *tv = vals + buf * 32 * W::VALS;
    const int64_t row0 = tile * 32 - p.win_lo;                     // obs row of the tile's first env
    uint32_t flags = s_flags[buf][0];
    if (flags) {
      unsigned char *dst = reinterpret_cast<unsigned char *>(p.obs) + row0 * (int64_t)W::OBS_BYTES;
      constexpr uint32_t TOTAL = 8 * W::OBS_FLOATS;                // float4s of the tile = 8 groups x OBS_FLOATS entries
      uint32_t ent = ctid, grp = 0;
      if (flags == 0xffffffffu && (row0 & 3) == 0) {
        // fast path: the whole tile is rendered and 16-byte aligned
#pragma unroll 4
        for (uint32_t q = ctid; q < TOTAL; q += CTHREADS) {
          st_stream_v4(dst + ((size_t)q << 4), pick(t.lut[ent], tv + grp * 4 * W::VALS));
          ent += CTHREADS;
          if (ent >= W::OBS_FLOATS) { ent -= W::OBS_FLOATS; ++grp; }
        }
      } else {
        // partial tile (batch tail, reset mask, render-window edge): guarded 32-bit stores
        for (uint32_t q = ctid; q < TOTAL; q += CTHREADS) {
          const uint32_t en = t.lut[ent], a = en & 2047u, b = (en >> 11) & 2047u, k = en >> 22;
          const float *gv = tv + grp * 4 * W::VALS;
#pragma unroll
          for (uint32_t j = 0; j < 4; ++j) {
            const uint32_t code = j < k ? a : b, env = grp * 4 + code / W::VALS;
            if ((flags >> env) & 1u)
              __stcs(reinterpret_cast<unsigned int *>(dst) + ((size_t)q * 4 + j), __float_as_uint(gv[code]));
          }
          ent += CTHREADS;
          if (ent >= W::OBS_FLOATS) { ent -= W::OBS_FLOATS; ++grp; }
        }
      }
    }
    if (W::HAS_LOC) {
      // local observation (lmaze_env_v5.py:356-380): every env row is 16-byte aligned (19,600 = 16 x 1,225)
      flags = s_flags[buf][1];
      if (flags) {
        constexpr uint32_t PER = W::LOC_FLOATS / 4 > 0 ? W::LOC_FLOATS / 4 : 1;
        const uint32_t *loclut = reinterpret_cast<const uint32_t *>(smem + W::LOCLUT_OFF);
        unsigned char *dst = reinterpret_cast<unsigned char *>(p.obs2) + row0 * (int64_t)(W::LOC_FLOATS * 4);
        if (flags == 0xffffffffu) {
          uint32_t ent = ctid % PER, env = ctid / PER;
#pragma unroll 4
          for (uint32_t q = ctid; q < 32 * PER; q += CTHREADS) {
            // (an IndexError row is all zero: the producer zeroed the four local planes of that env)
            st_stream_v4(dst + ((size_t)q << 4), pick(loclut[ent], tv + env * W::VALS));
            ent += CTHREADS;
            while (ent >= PER) { ent -= PER; ++env; }
          }
        } else {
          while (flags) {                                          // a few envs of the tile (masked plannerStep)
            const uint32_t env = __ffs(flags) - 1;
            flags &= flags - 1;
            for (uint32_t q = ctid; q < PER; q += CTHREADS)
              st_stream_v4(dst + ((size_t)(env * PER + q) << 4), pick(loclut[q], tv + env * W::VALS));
          }
        }
      }
    }
  }
  if (warp == 0) {
    if (p.mode == MODE_STEP) ws.flush(p.stats, lane);
    if (lane == 0) finish_grabber(p.work, (unsigned long long)gridDim.x);
  }
}

// ---- compact observations / transition-only launches of the foveal variants -----------------------------------
// obs_mode = LMZ_OBS_COMPACT: the observation is written as f32 [C][5][5] -- the reference's `retState` BEFORE its
// x7 upsample (lmaze_env_v2.py:185-203, lmaze_env_v4.py:236-247, lmaze_env_v5.py:333-343,372-378) -- 500 / 700 /
// 700 + 400 bytes per env instead of 24,500 / 34,300 / 53,900; the reference image is exactly
// repeat_interleave(compact, 7) on both axes.  The same kernel serves launches with no observation bound.  The work
// per tile is small, so the organisation is warp-granular like lmz_env_compact_kernel: every warp grabs its own
// tiles (the next tile's index and state words requested one tile ahead), runs the 32 transitions, updates the
// visit history of each env itself (v4 / v5, visit_step), and ASSEMBLES the tile's 32 rows in shared
// memory exactly as they lie in the tensor (lane l expands env l's 25-bit planes into floats, the visit crops land
// in their planes directly).  The tile's rows are one contiguous, 16-byte aligned run of the tensor, so the copy
// out is ONE shared -> global bulk copy (cp.async.bulk) per tile: no per-float indexing and no store instruction.  (Round 1 looked every float up
// through (plane, cell) index arithmetic and was math-pipe bound at 74 % issue-slot use, 4.7 TB/s on v2.)
template <class W>
struct FovSmall {
  static constexpr uint32_t STAGE_OFF = W::ROWBITS_OFF;                 // the render tables are not needed here
  static constexpr uint32_t TAB_BYTES = (W::BLOB_BYTES - STAGE_OFF + 15u) & ~15u;
  static constexpr uint32_t PER = W::C * 25;                            // floats per env row (the obs channels are slots 0..C-1)
  static constexpr uint32_t PERL = 4 * 25;                              // v5 local obs row
  static constexpr uint32_t IN_HIST = W::NVIS > 0 ? 2048u : 0u;                // v4 / v5: a tile's visit histories
  static constexpr uint32_t IN_BYTES = W::NVIS > 0 ? IN_HIST + 3u * 128u : 0u;  // ... + 3 state-word arrays
  static constexpr uint32_t smem_bytes(int threads) { return TAB_BYTES + (threads / 32) * (32 * PER * 4 + IN_BYTES); }
};

template <class W, int THREADS>
__global__ void __launch_bounds__(THREADS) lmz_fov_small_kernel(const KParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar;
  using FS = FovSmall<W>;
  constexpr int WARPS = THREADS / 32;
  __shared__ __align__(8) uint64_t in_bar[WARPS];                // v4 / v5: one input barrier per warp
  constexpr uint32_t PER = FS::PER, PERL = FS::PERL;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    mbar_init(&bar, 1);
#pragma unroll
    for (int w = 0; w < WARPS; ++w) mbar_init(&in_bar[w], 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (tid == 0) {
    mbar_expect_tx(&bar, W::BLOB_BYTES - FS::STAGE_OFF);
    bulk_g2s(smem, p.blob + FS::STAGE_OFF, W::BLOB_BYTES - FS::STAGE_OFF, &bar);
  }
  mbar_wait(&bar, 0);
  const unsigned char *sb = smem - FS::STAGE_OFF;                // sb + X_OFF addresses staged table X
  const FovTables<W> t(sb);
  float *rows = reinterpret_cast<float *>(smem + FS::TAB_BYTES) + warp * (32 * PER);   // this warp's tile: [32][PER]
  const uint32_t rows_s = smem_addr(rows);
  const int64_t tiles = p.tile_end;
  const bool need_visit = W::NVIS > 0 && p.mode != MODE_PLANNER;
  WarpStats ws;
  auto grab = [&]() { return warp_grab(p, lane, 1); };
  // copy of the first `bytes` of the warp's smem tile to global (both 16-byte aligned): ONE shared -> global bulk
  // copy issued by lane 0 -- the TMA engine moves the tile's rows as one contiguous run, no LSU store is issued
  auto copy_out = [&](float *dst, uint32_t bytes) {
    fence_proxy_async();                                         // every lane's row writes -> async proxy
    __syncwarp();
    if (lane == 0) { bulk_s2g(dst, rows_s, bytes); bulk_commit(); }
  };
  auto rows_free = [&]() {                                       // the last bulk copy has finished READING the rows
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncwarp();
  };
  // the tile's observation rows: bit planes -> floats in the warp's rows (the visit crops are already there), copy out
  auto emit = [&](const FovLane<W::NBIT> &v, bool valid, int64_t tile, unsigned ff, unsigned fl) {
    float *mine = rows + lane * PER;
    const int64_t row0 = tile * 32 - p.win_lo;                   // obs row of the tile's first env
    if (ff) {
      if (valid && v.rfov) {                                     // 25-bit planes -> float planes (stride PER is odd: no bank conflicts)
#pragma unroll
        for (int b = 0; b < W::NBIT; ++b) {
          if (W::bit_slot(b) < W::C) expand_plane(v.mask[b], mine + W::bit_slot(b) * 25);   // (v5: local planes below)
        }
      }
      float *dst = reinterpret_cast<float *>(p.obs) + row0 * (int64_t)PER;
      if (ff == 0xffffffffu && (row0 & 3) == 0) copy_out(dst, 32 * PER * 4);
      else {                                                     // batch tail, masked reset, window edge
        __syncwarp();
        for (unsigned m = ff; m; m &= m - 1) {
          const uint32_t env = __ffs(m) - 1;
          for (uint32_t pos = lane; pos < PER; pos += 32) __stcs(dst + env * PER + pos, rows[env * PER + pos]);
        }
      }
    }
    if (W::HAS_LOC && fl) {
      // local obs (lmaze_env_v5.py:360-368): free crop, ball and previous ball relative to the planner-time fovea,
      // fovealGoal = bit planes 7, 5, 6, 8 (all-zero on an IndexError row); 400 bytes per env, always 16-byte aligned
      rows_free();                                               // the foveal rows have been copied out
      float *minel = rows + lane * PERL;
      if (valid && v.rloc) {
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4)
          expand_plane(v.mask[W::NBIT > 8 ? (c4 == 0 ? 7 : c4 == 1 ? 5 : c4 == 2 ? 6 : 8) : 0], minel + c4 * 25);
      }
      float *dst = reinterpret_cast<float *>(p.obs2) + row0 * (int64_t)PERL;
      if (fl == 0xffffffffu) copy_out(dst, 32 * PERL * 4);
      else {
        // some envs of the tile (plannerStep: the envs waiting for their planner, about half of them in steady state):
        // every local row is 400 bytes and 16-byte aligned, so each RUN of flagged envs leaves as one bulk copy
        // (per-env 32-bit stores made the compact plannerStep launch as long as the step launch itself)
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          unsigned m = fl;
          while (m) {
            const uint32_t lo = __ffs(m) - 1;
            const unsigned gap = ~(m >> lo);                     // first zero above lo ends the run
            const uint32_t len = gap ? (uint32_t)(__ffs(gap) - 1) : 32u - lo;
            bulk_s2g(dst + lo * PERL, rows_s + lo * PERL * 4, len * PERL * 4);
            m = (lo + len >= 32u) ? 0u : (m >> (lo + len)) << (lo + len);
          }
          bulk_commit();
        }
      }
    }
  };
  auto blank_lane = [](FovLane<W::NBIT> &v) {
    v.o.st = 0; v.o.st_old = 0; v.o.render = false; v.o.done = false; v.o.cls = -1; v.o.eplen = 0; v.info = 0;
    v.vinfo = 0; v.rfov = false; v.rloc = false;
#pragma unroll
    for (int b = 0; b < W::NBIT; ++b) v.mask[b] = 0;
  };

  if constexpr (W::NVIS > 0) {
    // ---- the visit variants (v4, v5): the tile's INPUTS come through the TMA engine too ------------------------
    // (v2 keeps the register pipeline below: with its two state words per env the TMA form is SLOWER, 10.9 vs 11.5 G
    // env-steps/s, profiles/r2_ab18.txt)
    // A tile's state words and visit histories are contiguous runs (128 bytes per word array, 2 KB of history), so
    // lane 0 requests them as bulk copies into the warp's input buffer one whole tile ahead and the warp picks them up
    // behind an mbarrier.  Loading them into registers a tile ahead does NOT work: the compiler moves a loaded
    // register to its loop-carried home right behind the load, and that move waits for the load (ncu: 22 % of the
    // warp's cycles in long_scoreboard at those moves and at the shuffle behind the work-counter atomic).  The
    // atomic is issued WITHOUT the compiler's warp aggregation (grab_tile_async) two tiles ahead and its result is
    // first touched a tile later.  The handle's state arrays are padded to whole tiles (lmz_abi.cu).
    constexpr uint32_t IN_HIST = 0, IN_W0 = FS::IN_HIST, IN_W1 = IN_W0 + 128, IN_W2 = IN_W0 + 256;
    unsigned char *inb = smem + FS::TAB_BYTES + WARPS * (32 * PER * 4) + warp * FS::IN_BYTES;
    uint64_t *ibar = &in_bar[warp];
    const bool need_hist = W::NVIS > 0 && p.mode != MODE_PLANNER;
    const bool need_act = p.mode == MODE_STEP || p.mode == MODE_PLANNER;
    auto issue_inputs = [&](int64_t tl) {                        // lane 0
      const int64_t e0 = tl * 32;
      mbar_expect_tx(ibar, (need_hist ? 2048u : 0u) + (W::HAS_LOC ? 384u : 256u));
      if (need_hist) bulk_g2s(inb + IN_HIST, p.hist + e0 * HIST_MAX, 2048u, ibar);
      bulk_g2s(inb + IN_W0, p.state + e0, 128u, ibar);
      bulk_g2s(inb + IN_W1, p.goal_count + e0, 128u, ibar);
      if (W::HAS_LOC) bulk_g2s(inb + IN_W2, p.aux2 + e0, 128u, ibar);
    };
    auto load_act = [&](int64_t tl) -> long long {               // (unconditional: lanes past the end re-read the last action)
      const int64_t e = tl * 32 + lane;
      return need_act ? load_action(p.actions, p.action_dtype, e < p.n ? e : p.n - 1) : 0ll;
    };
    int64_t cur_t = grab(), nxt_t = grab();
    int64_t raw = 0;                                             // lane 0: the tile after those, still in flight
    if (lane == 0) raw = p.tile_begin + grab_tile_async(p.work);
    long long act_next = 0;
    if (cur_t < tiles) {
      if (lane == 0) issue_inputs(cur_t);
      act_next = load_act(cur_t);
    }
    uint32_t phase = 0;
    while (cur_t < tiles) {
      const int64_t tile = cur_t;
      mbar_wait(ibar, phase);
      phase ^= 1u;
      FovPre pre;
      pre.w0 = reinterpret_cast<const uint32_t *>(inb + IN_W0)[lane];
      pre.w1 = reinterpret_cast<const uint32_t *>(inb + IN_W1)[lane];
      pre.w2 = W::HAS_LOC ? reinterpret_cast<const uint32_t *>(inb + IN_W2)[lane] : 0u;
      pre.act = act_next;
#pragma unroll
      for (int k = 0; k < 4; ++k)
        pre.h[k] = need_hist ? reinterpret_cast<const uint4 *>(inb + IN_HIST)[lane * 4 + k] : make_uint4(0u, 0u, 0u, 0u);
      __syncwarp();                                              // every lane has read the buffer: it can be refilled
      const int64_t after = __shfl_sync(0xffffffffu, raw, 0);    // grabbed a tile ago
      if (lane == 0) raw = p.tile_begin + grab_tile_async(p.work);
      if (nxt_t < tiles) {
        if (lane == 0) { fence_proxy_async(); issue_inputs(nxt_t); }
        act_next = load_act(nxt_t);
      }
      const int64_t e = tile * 32 + lane;
      const bool valid = e < p.n;
      FovLane<W::NBIT> v;
      blank_lane(v);
      if (valid) v = fov_lane(static_cast<const W *>(nullptr), p, e, t, sb, pre);
      if (p.mode == MODE_STEP) ws.add(valid, v.o);
      const unsigned ff = __ballot_sync(0xffffffffu, valid && v.rfov);
      const unsigned fl = __ballot_sync(0xffffffffu, valid && v.rloc);
      if (W::NVIS > 0 && need_hist) {                            // append to / fold the visit history: the two crops ...
        VisitHist h = visit_hist_of(pre);
        float vc[25], vp[25];
        const bool have = visit_step<W>(p, tile * 32, lane, valid, v.info, v.vinfo, valid && v.rfov, h, vc, vp);
        rows_free();                                             // ... while the previous tile's copy out still reads the rows
        if (have) {
          float *mine = rows + lane * PER;
#pragma unroll
          for (int k = 0; k < 25; ++k) { mine[W::VIS_SLOT0 * 25 + k] = vc[k]; mine[W::VIS_SLOT1 * 25 + k] = vp[k]; }
        }
      } else {
        rows_free();
      }
      emit(v, valid, tile, ff, fl);
      cur_t = nxt_t; nxt_t = after;
    }
  } else {
    // ---- v2: software pipeline over the warp's tiles: the transitions of tile t+1 run while the TMA engine drains
    // tile t's rows (state words in registers, requested one tile ahead)
    auto preload = [&](int64_t tl, FovPre &q) {
      const int64_t e = tl * 32 + lane;
      q.w0 = q.w1 = q.w2 = 0u; q.act = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) q.h[k] = make_uint4(0u, 0u, 0u, 0u);
      if (tl < tiles && e < p.n) q = fov_preload<W>(p, e);
    };
    struct Slot {
      FovLane<W::NBIT> v;
      int64_t tile;
      bool valid;
    };
    int64_t ntile = grab(), nntile = grab();
    FovPre pre;
    preload(ntile, pre);
    auto stage_a = [&](Slot &sl) {                               // transitions of the next tile
      sl.tile = ntile;
      const int64_t after = grab();                              // needed two tiles from now
      const int64_t e = sl.tile * 32 + lane;
      sl.valid = sl.tile < tiles && e < p.n;
      blank_lane(sl.v);
      const FovPre pre_used = pre;
      if (sl.valid) sl.v = fov_lane(static_cast<const W *>(nullptr), p, e, t, sb, pre_used);
      if (p.mode == MODE_STEP) ws.add(sl.valid, sl.v.o);
      ntile = nntile; nntile = after;
      preload(ntile, pre);                                       // the tile after's words fly meanwhile
    };
    Slot cur, nxt;
    stage_a(cur);
    while (cur.tile < tiles) {
      const FovLane<W::NBIT> v = cur.v;
      const bool valid = cur.valid;
      const int64_t tile = cur.tile;
      const unsigned ff = __ballot_sync(0xffffffffu, valid && v.rfov);
      const unsigned fl = __ballot_sync(0xffffffffu, valid && v.rloc);
      stage_a(nxt);                                              // the next tile's transitions overlap the draining copy
      rows_free();                                               // the previous tile's copy out has read the buffer
      emit(v, valid, tile, ff, fl);
      cur = nxt;
    }
  }
  if (lane == 0) bulk_wait_all();                                // the last tile's rows have left shared memory
  if (p.mode == MODE_STEP) ws.flush(p.stats, lane);
  if (lane == 0) finish_grabber(p.work, (unsigned long long)gridDim.x * WARPS);
}

}  // namespace lmz
