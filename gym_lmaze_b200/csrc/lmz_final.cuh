// lmz_final.cuh -- terminal observations under auto-reset (lmz_bind_final).
//
// With autoreset an env that finishes is re-spawned inside the step kernel, and the obs row it returns already shows
// the next episode.  A learner bootstrapping a truncated episode needs the observation the episode ENDED in -- the row
// the step would have returned with autoreset off.  These kernels write it: when a final buffer is bound, lmz_step
// enqueues one of them BEFORE the unchanged step kernel.  The transition is deterministic, so the pre-pass re-runs it
// on the same state words and actions, in registers, and writes the un-expanded row (compact, or bit-packed) of every
// env whose done flag rises; nothing else is written (no state, no history, no statistics).  So it covers every render
// and obs mode of the step and leaves the step kernels as they are.
//
// Organisation: one warp per 32-env tile (FINAL_TILES tiles per warp, their loads issued together), one lane per env
// for the transition; a ballot finds the finishing envs, and the warp then writes each such row with coalesced 32-bit
// stores (right after a batch reset the episodes are synchronised and one step finishes nearly every env).  A plain
// grid: no work counter is touched, so the step kernel that follows re-arms nothing it did not arm itself.
#pragma once
#include "lmz_kernels.cuh"
#include "lmz_fov.cuh"

namespace lmz {

struct FinalParams {
  int64_t n;                    // envs in the handle
  const uint32_t *state;        // packed state word per env
  const uint32_t *aux;          // v2 / v4: the second state word (the handle's goal_count array)
  const uint8_t *hist;          // v4: visit history u8 [n][64]
  const float *visit;           // v4: the layer of envs in direct mode, f32 [n][324]
  const void *actions;          // [n]
  int action_dtype;
  void *out;                    // final rows: u8 [n][C][G][G], u8 [n][R] (bits) or f32 [n][C][5][5] (foveal)
  int bits;                     // v0 / v3: the rows are bit-packed (OBS_BITS)
  const uint8_t *blob;          // template blob in global memory
  unsigned int *scratch;        // v2_step_core counts out-of-range actions here: the step kernel counts them once
};

constexpr int FINAL_TILES = 4;  // tiles per warp
constexpr int FINAL_COOP_MAX = 2;   // v4: tiles with at most this many finishing envs fold them one at a time

// the foveal pre-pass stages the row bits and cell classes of the blob (dynamic shared memory of this size)
template <class W>
__host__ __device__ constexpr uint32_t final_fov_smem() { return W::GCAND_OFF - W::ROWBITS_OFF; }

// ---- v0 / v3 ------------------------------------------------------------------------------------------------------
template <class V, int THREADS>
__global__ void __launch_bounds__(THREADS) lmz_final_kernel(const FinalParams p) {
  __shared__ __align__(16) unsigned char tab[V::TABLES_BYTES];
  constexpr int WARPS = THREADS / 32;
  constexpr uint32_t W = V::COMPACT_BYTES / 4;           // 32-bit words of a compact row (v0 144, v3 243)
  constexpr int K = (W + 31) / 32;
  constexpr uint32_t BW = V::BITS_WORDS;                 // 32-bit words of a bit-packed row (v0 18, v3 31)
  const int lane = threadIdx.x & 31;
  for (uint32_t i = threadIdx.x; i < V::TABLES_BYTES / 4; i += THREADS)
    reinterpret_cast<uint32_t *>(tab)[i] = reinterpret_cast<const uint32_t *>(p.blob + V::TABLES_OFF)[i];
  __syncthreads();
  const uint8_t *cls = tab;
  const uint32_t *tmpl = reinterpret_cast<const uint32_t *>(tab + (V::COMPACT_OFF - V::TABLES_OFF));
  const uint32_t *btmpl = reinterpret_cast<const uint32_t *>(tab + (V::BITS_OFF - V::TABLES_OFF));
  const int64_t tile0 = ((int64_t)blockIdx.x * WARPS + (threadIdx.x >> 5)) * FINAL_TILES;
  uint32_t st[FINAL_TILES];
  long long act[FINAL_TILES];
#pragma unroll
  for (int k = 0; k < FINAL_TILES; ++k) {                // every load of the warp's tiles in flight at once
    const int64_t e = (tile0 + k) * 32 + lane;
    st[k] = 0; act[k] = 0;
    if (e < p.n) { st[k] = p.state[e]; act[k] = load_action(p.actions, p.action_dtype, e); }
  }
#pragma unroll
  for (int k = 0; k < FINAL_TILES; ++k) {
    const int64_t e0 = (tile0 + k) * 32;
    bool done = false;
    uint32_t hot[V::NHOT];
    EnvRegs r = V::unpack(st[k]);
    if (e0 + lane < p.n) {
      uint32_t hits = 0;
      done = transition<V>(r, act[k], cls, hits).done;   // the step kernels' transition: the terminal state
    }
    V::hot_bytes(r, hot);
    const unsigned m = __ballot_sync(0xffffffffu, done);
    if (!m) continue;
    if (p.bits) {
      // the tile's rows are one flat run of 32 * BW words: lane l stores words l, l+32, ... of the run
      uint32_t *dst = reinterpret_cast<uint32_t *>(p.out) + e0 * (int64_t)BW;
#pragma unroll
      for (uint32_t j = 0; j < BW; ++j) {
        const uint32_t w = lane + 32 * j, env = w / BW, kk = w - env * BW;
        uint32_t v = btmpl[kk];
#pragma unroll
        for (int q = 0; q < V::NHOT; ++q) {
          const uint32_t h = __shfl_sync(0xffffffffu, hot[q], env);
          v |= ((h >> 5) == kk) ? (1u << (h & 31)) : 0u;
        }
        if ((m >> env) & 1u) __stcs(dst + w, v);
      }
      continue;
    }
    uint32_t base[K];
#pragma unroll
    for (int kk = 0; kk < K; ++kk) base[kk] = (lane + 32 * kk < (int)W) ? tmpl[lane + 32 * kk] : 0u;
    uint32_t *dst = reinterpret_cast<uint32_t *>(p.out) + e0 * (int64_t)W;
    for (unsigned mm = m; mm; mm &= mm - 1) {
      const int env = __ffs(mm) - 1;
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
}

// ---- v2 / v4 ------------------------------------------------------------------------------------------------------
// The row is the compact observation f32 [C][5][5] of the post-step registers: the five bit planes v2_lane builds
// (free and goal crop at the ball, the action one-hot, the previous crops) and, for v4, the two visit crops AFTER the
// step's averaging, computed as visit_step computes them: the env's history with the step's new entry appended (the
// window at the new ball); an env in direct mode (lmz_set_visit) or with a full history takes the full-pass form
// (visit_average) of its layer.  Two organisations, chosen per tile by how many of its envs finish (profiles/
// r3_final_obs_bench.json, v4 compact 2^23 on a B200): up to FINAL_COOP_MAX, one lane per cell of the env's two windows
// (visit_fold_cell) -- the steady state, about one finishing env per tile; more, ONE warp-wide visit_fold2 in which
// every finishing lane folds its own env -- right after a batch reset the whole tile finishes in the same step, and the
// per-env form made that step 15x as long as the step itself.  Nothing is written back to the layer or the history.
template <class W, int THREADS>
__global__ void __launch_bounds__(THREADS) lmz_final_fov_kernel(const FinalParams p) {
  constexpr uint32_t TAB_OFF = W::ROWBITS_OFF, TAB_BYTES = final_fov_smem<W>();
  extern __shared__ __align__(16) unsigned char tab[];
  constexpr int WARPS = THREADS / 32;
  constexpr int VSTRIDE = 51;                            // (odd: the lanes' rows fall in different banks)
  __shared__ float s_vis[W::NVIS > 0 ? WARPS * 32 * VSTRIDE : 1];   // v4: each lane's two visit crops
  constexpr uint32_t PER = W::C * 25;                    // floats per row
  constexpr int GG = W::G * W::G;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (uint32_t i = threadIdx.x; i < TAB_BYTES / 4; i += THREADS)
    reinterpret_cast<uint32_t *>(tab)[i] = reinterpret_cast<const uint32_t *>(p.blob + TAB_OFF)[i];
  __syncthreads();
  const FovTables<W> t(tab - TAB_OFF);                   // only rowbits and cls are used (and staged)
  float *vis = s_vis + (W::NVIS > 0 ? warp * 32 * VSTRIDE : 0);
  const int64_t tile0 = ((int64_t)blockIdx.x * WARPS + warp) * FINAL_TILES;
  uint32_t w0[FINAL_TILES], w1[FINAL_TILES];
  long long act[FINAL_TILES];
#pragma unroll
  for (int k = 0; k < FINAL_TILES; ++k) {
    const int64_t e = (tile0 + k) * 32 + lane;
    w0[k] = 0; w1[k] = 0; act[k] = 0;
    if (e < p.n) { w0[k] = p.state[e]; w1[k] = p.aux[e]; act[k] = load_action(p.actions, p.action_dtype, e); }
  }
#pragma unroll 1
  for (int k = 0; k < FINAL_TILES; ++k) {                // rolled (the v4 body is large): tile k's words are in [0]
    const int64_t e0 = (tile0 + k) * 32, e = e0 + lane;
    bool done = false;
    V2Regs r = v2_unpack(w0[0], w1[0]);
    const long long a = act[0];
#pragma unroll
    for (int j = 0; j + 1 < FINAL_TILES; ++j) { w0[j] = w0[j + 1]; w1[j] = w1[j + 1]; act[j] = act[j + 1]; }
    const int tpre = r.vt;                               // v4: history entries before the step (or VT_DIRECT)
    if (e < p.n) {
      int rcode, cls;
      done = v2_step_core<W>(r, a, t, p.scratch, rcode, cls);
    }
    const unsigned m = __ballot_sync(0xffffffffu, done);
    if (!m) continue;
    uint32_t mask[5] = {0u, 0u, 0u, 0u, 0u};
    if (done) {                                          // (a lane past the end holds no maze position)
      mask[0] = v2_free_crop<W>(t, r.L, r.x, r.y);
      mask[1] = v2_goal_crop(r.x, r.y, r.gx, r.gy);
      mask[2] = r.a >= 0 ? (1u << r.a) : 0u;
      mask[3] = v2_free_crop<W>(t, r.L, r.px, r.py);
      mask[4] = v2_goal_crop(r.px, r.py, r.gx, r.gy);
    }
    if (W::NVIS > 0) {
      const bool hmode = done && tpre != VT_DIRECT;      // history mode (the history of a finishing env only is read)
      VisitHist h;
#pragma unroll
      for (int g = 0; g < 16; ++g) h.w[g] = 0u;
      if (hmode) {
        const uint4 *hp = reinterpret_cast<const uint4 *>(p.hist + e * HIST_MAX);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint4 v = __ldcg(hp + q);
          h.w[4 * q] = v.x; h.w[4 * q + 1] = v.y; h.w[4 * q + 2] = v.z; h.w[4 * q + 3] = v.w;
        }
      }
      __syncwarp();                                      // the previous tile's rows have been read
      if (__popc(m) <= FINAL_COOP_MAX) {
        for (unsigned mm = m; mm; mm &= mm - 1) {
          const int env = __ffs(mm) - 1;
          const int st = __shfl_sync(0xffffffffu, tpre, env);
          const int bx = __shfl_sync(0xffffffffu, r.x, env), by = __shfl_sync(0xffffffffu, r.y, env);
          const int px = __shfl_sync(0xffffffffu, r.px, env), py = __shfl_sync(0xffffffffu, r.py, env);
#pragma unroll 1
          for (int q0 = 0; q0 < 50; q0 += 32) {          // cell q: q < 25 the window at the ball, else the previous one
            const int q = q0 + lane, c = q < 25 ? q : q - 25;
            const int x = (q < 25 ? bx : px) - 2 + c / 5, y = (q < 25 ? by : py) - 2 + c % 5;
            const bool in_cur = (unsigned)(x - bx + 2) < 5u && (unsigned)(y - by + 2) < 5u;
            float v = visit_fold_cell(h, env, st < HIST_MAX ? st : HIST_MAX, x, y);   // (all lanes: shuffles)
            if (st < HIST_MAX) v = visit_avg1(v, in_cur);
            else {
              if (st == VT_DIRECT && q < 50) v = __ldcg(p.visit + (e0 + env) * GG + x * W::G + y);
              v = visit_average(v, in_cur);
            }
            if (q < 50) vis[env * VSTRIDE + q] = v;
          }
        }
        __syncwarp();
      } else {
        // history mode: the T entries and the one this step appends (the window at the new ball); a full history: its
        // 64 entries, then the full pass below
        const int told = hmode ? (tpre < HIST_MAX ? tpre : HIST_MAX) : 0;
        const int tnew = hmode ? (tpre < HIST_MAX ? tpre + 1 : HIST_MAX) : 0;
        const int tmax = __reduce_max_sync(0xffffffffu, told);
        float vc[25], vp[25];
        visit_fold2(h, told, tnew, visit_entry(r.x, r.y), tmax, r.x - 2, r.y - 2, r.px - 2, r.py - 2, vc, vp);
        if (done && tpre >= HIST_MAX) {                    // direct mode / full history: one literal averaging
#pragma unroll
          for (int c = 0; c < 25; ++c) {
            const int cx = r.x - 2 + c / 5, cy = r.y - 2 + c % 5, qx = r.px - 2 + c / 5, qy = r.py - 2 + c % 5;
            if (tpre == VT_DIRECT) {
              vc[c] = __ldcg(p.visit + e * GG + cx * W::G + cy);
              vp[c] = __ldcg(p.visit + e * GG + qx * W::G + qy);
            }
            vc[c] = visit_average(vc[c], true);            // the crop at the ball IS the new window
            vp[c] = visit_average(vp[c], (unsigned)(qx - r.x + 2) < 5u && (unsigned)(qy - r.y + 2) < 5u);
          }
        }
        if (done) {
#pragma unroll
          for (int c = 0; c < 25; ++c) { vis[lane * VSTRIDE + c] = vc[c]; vis[lane * VSTRIDE + 25 + c] = vp[c]; }
        }
        __syncwarp();
      }
    }
    float *dst = reinterpret_cast<float *>(p.out) + e0 * (int64_t)PER;
    for (unsigned mm = m; mm; mm &= mm - 1) {
      const int env = __ffs(mm) - 1;
      uint32_t pm[5];
#pragma unroll
      for (int b = 0; b < 5; ++b) pm[b] = __shfl_sync(0xffffffffu, mask[b], env);
      float *row = dst + (size_t)env * PER;
#pragma unroll
      for (uint32_t k2 = 0; k2 < (PER + 31) / 32; ++k2) {
        const uint32_t pos = lane + 32 * k2;
        if (pos < PER) {
          const int slot = (int)(pos / 25), c = (int)(pos - 25 * (pos / 25));
          float v;
          if (W::NVIS > 0 && slot == W::VIS_SLOT0) v = vis[env * VSTRIDE + c];
          else if (W::NVIS > 0 && slot == W::VIS_SLOT1) v = vis[env * VSTRIDE + 25 + c];
          else {
            const int b = W::NVIS > 0 ? (slot < 2 ? slot : slot - 1) : slot;      // inverse of W::bit_slot
            const uint32_t bm = b == 0 ? pm[0] : b == 1 ? pm[1] : b == 2 ? pm[2] : b == 3 ? pm[3] : pm[4];
            v = ((bm >> c) & 1u) ? 1.0f : 0.0f;
          }
          __stcs(row + pos, v);
        }
      }
    }
  }
}

}  // namespace lmz
