// snk_kernels.cu -- sm_100a kernels of the batched Snake-v1 step path.
//
// A TILE is up to 32/G consecutive environments, G = num_snakes rounded up to a power of two, so that in the rule
// phase lane = (environment in tile, snake).  The tile's records are contiguous in HBM; one elected thread stages them
// into shared memory with a 1-D bulk copy (cp.async.bulk + mbarrier), the tile is stepped there and written back the
// same way.  Two tile modes: warp-private (every warp owns a tile, no block barrier after the table copy: one warp's
// rule phase overlaps the other warps' observation stores) and CTA-cooperative (one tile per CTA, warp 0 runs the
// rules, then all warps share the tile's viewers).  Two record layouts: the whole working record in HBM, or the
// compact one without the grid, which is then rebuilt in shared memory (expand_tile) from the handle's wall layout,
// the record's fruit slots and the bodies spelled out by the direction plane.
//
//   rules    lanes = snakes: turn, head advance, __match_any_sync on target cells (head-on and arrival
//            order), ballots for deaths / fruit cells / alive set, shared-memory scatter for kill credit, one more
//            match for the tail-growth rule, float64 reward, clear-then-write grid update      (step_group)
//   rare     whole warp per environment: fruit respawn = k-th empty cell by word-wise rank-select;
//            auto-reset = spawn picks + paint-and-vote overlap test + fruit seeding
//   encode   whole warp per (environment, viewer), or per pair of viewers on 16-byte aligned blocks: two crop cells
//            per lane -> LUT -> one 128-bit streaming store (frame_stack 1; register / direct / padded-plane / table
//            flavours); channel-bit frames
//            staged in output order and expanded with flat 128-bit stores (frame_stack > 1); optionally the channel
//            bits themselves instead of / beside the NHWC bytes
//
// Reference: SnakeEnv.step / reset / _encode (envs/snake_env.py:301-414, 131-159, 474-519) and the
// vector worker's auto-reset (wrappers.py:138-146).
#include <cuda_runtime.h>
#include <stdint.h>

#include "snk_core.cuh"
#include <atomic>

#include "snk_kernels.h"

namespace snk {

enum : uint8_t { F_RESET = 1, F_INIT = 2, F_SKIP = 4 };

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

// ---- debug build (-DSNK_DEBUG_CHECKS -> libsnk_dbg.so): compute-sanitizer is not available on the GPU pool, so
// this build checks every observation / history store against the caller's buffers and every grid index against
// the record, and raises the sticky ERR_INTERNAL bit.  The test suite runs against it via SNK_LIB_PATH.
#ifdef SNK_DEBUG_CHECKS
__device__ const uint8_t* dbg_obs_lo; __device__ const uint8_t* dbg_obs_hi;
__device__ const uint8_t* dbg_hist_lo; __device__ const uint8_t* dbg_hist_hi;
__device__ const uint8_t* dbg_bits_lo; __device__ const uint8_t* dbg_bits_hi;
__device__ uint32_t* dbg_err;
__device__ __forceinline__ void dbg_arm(const KParams& p) {        // every thread writes the same values
  const size_t blocks = (p.T > 1 && p.obs_every_step) ? (size_t)p.T : 1;      // snk_step_many: one block per step
  dbg_obs_lo = p.obs; dbg_obs_hi = p.obs ? p.obs + blocks * p.d.N * p.d.obs_env_bytes : nullptr;
  dbg_hist_lo = p.hist; dbg_hist_hi = p.hist ? p.hist + (size_t)p.d.N * p.d.hist_env_bytes : nullptr;
  dbg_bits_lo = p.bits; dbg_bits_hi = p.bits ? p.bits + blocks * p.d.N * p.d.stage_env_bytes : nullptr;
  dbg_err = p.err;
}
__device__ __forceinline__ void dbg_store(const void* q, size_t n, const uint8_t* lo, const uint8_t* hi) {
  const uint8_t* a = reinterpret_cast<const uint8_t*>(q);
  if (a < lo || a + n > hi || (reinterpret_cast<uintptr_t>(a) & (n - 1))) atomicOr(dbg_err, ERR_INTERNAL);
}
#define SNK_CHECK_OBS(q, n) dbg_store((q), (n), dbg_obs_lo, dbg_obs_hi)
#define SNK_CHECK_BITS(q, n) dbg_store((q), (n), dbg_bits_lo, dbg_bits_hi)
#define SNK_CHECK_HIST(q, n) dbg_store((q), (n), dbg_hist_lo, dbg_hist_hi)
#define SNK_ASSERT(p, cond) do { if (!(cond)) atomicOr((p).err, ERR_INTERNAL); } while (0)
#else
#define SNK_CHECK_OBS(q, n) ((void)0)
#define SNK_CHECK_BITS(q, n) ((void)0)
#define SNK_CHECK_HIST(q, n) ((void)0)
#define SNK_ASSERT(p, cond) ((void)0)
#endif


// ---- profiling build (-DSNK_PHASE_TIMING -> libsnk_prof.so): per-phase SM cycle counts of the tile kernel,
// accumulated per warp role into snk_phase_cycles[] (read back with snk_prof_phases).  Never in libsnk.so.
#ifdef SNK_PHASE_TIMING
// trace[(cta * 8 + warp) * 8 + k]: %globaltimer (ns) at phase boundary k of warps 0..7 of every CTA of the last launch
__device__ unsigned long long* snk_trace_buf;
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define SNK_T(var) const unsigned long long var = gtime()
// reset timeline of the last reset of a CTA: trace2[cta * 8 + k], k = entry, walls, spawn, snakes, fruits, attempts
__device__ unsigned long long* snk_trace2_buf;
#define SNK_R(k) do { if (lane_id() == 0 && snk_trace2_buf) snk_trace2_buf[(size_t)blockIdx.x * 8 + (k)] = gtime(); } while (0)
#define SNK_RV(k, v) do { if (lane_id() == 0 && snk_trace2_buf) snk_trace2_buf[(size_t)blockIdx.x * 8 + (k)] = (v); } while (0)
#else
#define SNK_R(k) ((void)0)
#define SNK_RV(k, v) ((void)0)
#define SNK_T(var) ((void)0)
#endif

// ---- phase R helpers (warp-cooperative) -----------------------------------------------------------

// 0x80 in every byte of x that is zero (exact, no carries between bytes).
__device__ __forceinline__ uint32_t zero_bytes(uint32_t x) {
  const uint32_t t = (x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu;
  return ~(t | x | 0x7F7F7F7Fu);
}
__device__ __forceinline__ uint32_t warp_inclusive_sum(uint32_t v, uint32_t lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, v, o);
    if ((int)lane >= o) v += t;
  }
  return v;
}

// Compact records: the new fruit cells of a placement also go into the record's slot list (duplicate draws collapse to
// one cell, one slot): the a-th distinct new cell takes the a-th free slot.  Out of line on purpose -- inlined into
// place_fruits_warp its live values raised the register count of every kernel instance.
__device__ __noinline__ void fruit_slots_add(uint16_t* fruit, int fcap, int mycell, uint32_t* err) {
  const uint32_t FULL = 0xffffffffu;
  const uint32_t lane = lane_id();
  const uint32_t dup = __match_any_sync(FULL, mycell);
  const bool adds = mycell >= 0 && (__ffs(dup) - 1) == (int)lane;
  const uint32_t adders = __ballot_sync(FULL, adds);
  const uint32_t free_lo = __ballot_sync(FULL, (int)lane < fcap && fruit[lane] == 0);              // slots 0..31
  const uint32_t free_hi = __ballot_sync(FULL, (int)lane + 32 < fcap && fruit[lane + 32] == 0);    // slots 32..63
  if (adds) {
    const int a = __popc(adders & ((1u << lane) - 1u)), nlo = __popc(free_lo);
    uint32_t slot = a < nlo ? __fns(free_lo, 0, a + 1) : __fns(free_hi, 0, a - nlo + 1);     // 0xffffffff: none left
    if (a >= nlo && slot < 32u) slot += 32u;
    if (slot < (uint32_t)fcap) fruit[slot] = (uint16_t)(mycell + 1);
    else atomicOr(err, ERR_STATE);
  }
}

// Place k fruits on the k drawn ranks of the row-major empty-cell list (all ranks refer to the
// grid as it is before any of them is placed; duplicates collapse)    core/grid_util.py:126-133
// The grid is scanned as 32-bit words (four cells): lane l owns the contiguous word range
// [l*cw, (l+1)*cw), so lane order is row-major order; one pass counts the empty cells per lane, a warp
// prefix sum locates the lane range holding a drawn rank, and the warp then scans only that range.
// (The record is passed as its base address, not as a Rec&: a Rec whose address escapes lives in local
// memory, and every byte store into the grid would force its pointer fields to be reloaded from there.)
// (Likewise every configuration value is copied into a local first: `p` arrives as a generic reference here, and
// a field read after a shared-memory store would be reloaded through a generic load -- 1 to 2 us per reset.)
// g: the environment's grid, vb: its virtual record base (c-part address minus off_c0; == g for a contiguous record).
__device__ __noinline__ void place_fruits_warp(const KParams& p, uint8_t* g, uint8_t* vb, uint32_t env_local, int k, int purpose) {
  const Dims& d = p.d;
  const Rec r = rec_view2(g, vb + d.off_c0, d);
  const uint32_t FULL = 0xffffffffu;
  const uint32_t lane = lane_id();
  const int HW = d.HW, rng_mode = d.rng_mode;
  const int nwords = (HW + 3) >> 2, cw = (nwords + 31) >> 5;
  const uint32_t* gw = reinterpret_cast<const uint32_t*>(r.grid);        // record start is 16-byte aligned
  auto load_zeros = [&](int w) -> uint32_t {                              // 0x80 per EMPTY cell of word w
    if (w >= nwords) return 0u;
    uint32_t x = gw[w];
    if (4 * w + 4 > HW) x |= 0xFFFFFFFFu << (8 * (HW - 4 * w));           // bytes past the grid are not cells
    return zero_bytes(x);
  };
  // (A four-words-per-load variant of this scan and of the walk below cut the fruit seeding of a cfg4 reset from 7.0
  //  to 4.6 us, but its live values raised the register count of every kernel instance -- cfg2 48 -> 62, cfg4 64 -> 78,
  //  cfg5 88 -> 94 -- and the step times did not improve: removed again, profiles/README.md.)
  uint32_t cnt = 0;
  const int rot = (int)lane % cw;                                        // rotate: lanes start in different banks
  for (int j = 0; j < cw; ++j) {
    int jj = j + rot;
    jj -= (jj >= cw) ? cw : 0;
    cnt += (uint32_t)__popc(load_zeros((int)lane * cw + jj));
  }
  const uint32_t incl = warp_inclusive_sum(cnt, lane);
  const int n_empty = (int)__shfl_sync(FULL, incl, 31);
  if (n_empty == 0 || k <= 0) return;              // reference draws nothing when no cell is empty
  int rank = -1;
  if ((int)lane < k) {
    if (rng_mode == RNG_PHILOX) {
      rank = (int)draw_below(d, env_local, r.hdr->event, purpose, lane, (uint32_t)n_empty);
    } else {
      const int64_t lo = p.replay_off[env_local], hi = p.replay_off[env_local + 1];
      const int64_t at = lo + r.hdr->cursor + lane;
      if (at >= hi) { atomicOr(p.err, ERR_REPLAY_UNDERRUN); rank = 0; }
      else {
        rank = p.replay[at];
        if (rank < 0 || rank >= n_empty) { atomicOr(p.err, ERR_REPLAY_RANGE); rank = 0; }
      }
    }
  }
  __syncwarp();
  if (lane == 0 && rng_mode == RNG_REPLAY) r.hdr->cursor += (uint32_t)k;
  int mycell = -1;
  if (cw <= 64) {
    // Every drawing lane resolves its own rank, all draws in parallel: a binary search over the lanes' prefix sums
    // (five shuffles, executed by the whole warp) finds the lane range holding the rank, then the lane walks that
    // range's words itself and picks the byte from the word's zero-byte flags.
    int lo = 0, hi = 31;
    const uint32_t key = rank >= 0 ? (uint32_t)rank : 0u;
#pragma unroll
    for (int it = 0; it < 5; ++it) {
      const int mid = (lo + hi) >> 1;
      const uint32_t v = __shfl_sync(FULL, incl, mid);
      if (v > key) hi = mid; else lo = mid + 1;
    }
    const int owner = lo;                                                 // first lane whose prefix exceeds the rank
    uint32_t rr = key - __shfl_sync(FULL, incl - cnt, owner);             // rank inside the owner's word range
    if (rank >= 0) {
#pragma unroll 1
      for (int t = 0; t < cw; ++t) {
        const uint32_t z = load_zeros(owner * cw + t);
        const uint32_t c = (uint32_t)__popc(z);
        if (rr < c) {
          const uint32_t c0 = (z >> 7) & 1u, c1 = c0 + ((z >> 15) & 1u), c2 = c1 + ((z >> 23) & 1u);
          mycell = 4 * (owner * cw + t) + (int)((c0 <= rr) + (c1 <= rr) + (c2 <= rr));
          break;
        }
        rr -= c;
      }
    }
  } else
#pragma unroll 1
  for (int j = 0; j < k; ++j) {
    uint32_t rr = (uint32_t)__shfl_sync(FULL, rank, j);
    const int owner = __popc(__ballot_sync(FULL, incl <= rr));            // first lane whose prefix exceeds the rank
    rr -= __shfl_sync(FULL, incl - cnt, owner);                           // rank inside the owner's word range
    int cell = -1;
#pragma unroll 1
    for (int t0 = 0; t0 < cw; t0 += 32) {
      const int t = t0 + (int)lane;
      const uint32_t z = t < cw ? load_zeros(owner * cw + t) : 0u;
      const uint32_t c = (uint32_t)__popc(z);
      const uint32_t in2 = warp_inclusive_sum(c, lane);
      const uint32_t total = __shfl_sync(FULL, in2, 31);
      if (rr < total) {
        const int wl = __popc(__ballot_sync(FULL, in2 <= rr));
        const uint32_t zsel = __shfl_sync(FULL, z, wl);
        const uint32_t rin = rr - __shfl_sync(FULL, in2 - c, wl);
        cell = 4 * (owner * cw + t0 + wl) + (int)(__fns(zsel, 0, (int)rin + 1) >> 3);
        break;
      }
      rr -= total;
    }
    if ((int)lane == j) mycell = cell;
  }
  __syncwarp();
  SNK_ASSERT(p, mycell < HW);
  if (mycell >= 0) r.grid[mycell] = (uint8_t)FRUIT;
  if (d.compact) fruit_slots_add(r.fruit, d.fcap, mycell, p.err);
  __syncwarp();
}

// Several lanes of one environment may update plane bytes that share a word: atomic read-modify-write.
__device__ __forceinline__ void dirp_set_atomic(uint8_t* dirp, int c, int v) {
  uint32_t* w = reinterpret_cast<uint32_t*>(dirp) + (c >> 4);
  const int sh = (c & 15) * 2;
  atomicAnd(w, ~(3u << sh));
  atomicOr(w, (uint32_t)v << sh);
}

// Wall-map pool: the map id `m` read from a caller-written array, checked.  An id that is not a map raises the sticky
// ERR_MAP_RANGE bit and reads as map 0, so a bad id never leads to a read outside the pool.
__device__ __forceinline__ uint32_t checked_map(uint32_t m, int num_maps, uint32_t* err) {
  if (m >= (uint32_t)num_maps) { atomicOr(err, ERR_MAP_RANGE); m = 0u; }
  return m;
}

// SnakeEnv.reset for one environment record in shared memory      envs/snake_env.py:131-159, 576-596
// kPool: the handle has a wall-map pool; the environment's next_map picks the layout and the spawn table, and becomes
// its cur_map.
template <bool kPool>
__device__ __noinline__ void reset_env_warp(const KParams& p, uint8_t* g, uint8_t* vb, uint32_t env_local) {
  const Dims& d = p.d;
  const Rec r = rec_view2(g, vb + d.off_c0, d);
  const uint32_t lane = lane_id();
  // values read inside loops live in registers (see place_fruits_warp); what a rare branch reads once stays in `p`
  const int ns = d.ns, K = d.K, W = d.W, H = d.H, rng_mode = d.rng_mode;
  uint32_t m = 0;
  if constexpr (kPool) {
    if (lane == 0) {
      m = checked_map(p.next_map[env_local], p.num_maps, p.err);
      p.cur_map[env_local] = (uint8_t)m;
    }
    m = __shfl_sync(0xffffffffu, m, 0);
  }
  const uint32_t n_cand = kPool ? p.map_tab[m].y : d.n_cand, inv_row_words = p.inv_row_words;
  const uint64_t* const spawn = kPool ? p.spawn + p.map_tab[m].x : p.spawn;
  SNK_R(0);
  if (d.compact) for (int j = (int)lane; j < d.fcap; j += 32) r.fruit[j] = 0;
  // make_grid: walled empty box (core/grid_util.py:14-20), one grid row at a time so no division is needed --
  // or the handle's custom wall layout (snk_create_map, or the pool's map), copied word by word from its L2-resident plane
  if (kPool || p.wall_map) {
    const uint32_t* const wm = kPool ? reinterpret_cast<const uint32_t*>(p.pool + (size_t)m * d.off_c0) : p.wall_map;
    const int HW = d.HW, nfull = HW >> 2;
    uint32_t* gw = reinterpret_cast<uint32_t*>(r.grid);
    for (int j = (int)lane; j < nfull; j += 32) gw[j] = __ldg(wm + j);
    if ((int)lane < (HW & 3)) r.grid[4 * nfull + lane] = reinterpret_cast<const uint8_t*>(wm)[4 * nfull + lane];
  } else if ((W & 3) == 0 && W >= 8) {          // flat over the grid's 32-bit words; row = word / (W/4) by a multiply-high
    uint32_t* gw = reinterpret_cast<uint32_t*>(r.grid);
    const int wpr = W >> 2, nw = H * wpr;
    for (int j = (int)lane; j < nw; j += 32) {
      const int rr = (int)__umulhi((uint32_t)j, inv_row_words), x = j - rr * wpr;
      const bool edge = rr == 0 || rr == H - 1;
      gw[j] = edge ? 0x01010101u : (x == 0 ? 0x00000001u : 0u) | (x == wpr - 1 ? 0x01000000u : 0u);
    }
  } else {
    for (int rr = 0; rr < H; ++rr) {
      const bool edge = rr == 0 || rr == H - 1;
      for (int c = (int)lane; c < W; c += 32) r.grid[rr * W + c] = (uint8_t)((edge || c == 0 || c == W - 1) ? WALL : EMPTY);
    }
  }
  __syncwarp();

  SNK_R(1);
  uint64_t entry = 0;
  const bool me = (int)lane < ns;
  if (rng_mode == RNG_REPLAY) {
    if (me) {
      const int64_t lo = p.replay_off[env_local], hi = p.replay_off[env_local + 1];
      const int64_t at = lo + r.hdr->cursor + lane;
      int pick = 0;
      if (at >= hi) atomicOr(p.err, ERR_REPLAY_UNDERRUN);
      else {
        pick = p.replay[at];
        if (pick < 0 || (uint32_t)pick >= n_cand) { atomicOr(p.err, ERR_REPLAY_RANGE); pick = 0; }
      }
      entry = spawn[pick];
    }
    __syncwarp();
    if (lane == 0) r.hdr->cursor += (uint32_t)ns;
  }
  // sample poses until no two snakes share a cell (np.random.permutation(n)[:ns] retry loop, :579-586;
  // ns independent uniform picks conditioned on "no shared cell" have the same law)
  for (uint32_t attempt = 0;; ++attempt) {
    if (rng_mode == RNG_PHILOX && me)
      entry = spawn[draw_below(d, env_local, r.hdr->event, DRAW_SPAWN, attempt * (uint32_t)ns + lane, n_cand)];
    if (me) {
      int c = spawn_head(entry);
      r.grid[c] = (uint8_t)(BODY + 10 * lane);
      for (int j = 1; j < K; ++j) { c += dir_delta(spawn_link(entry, j), W); r.grid[c] = (uint8_t)(BODY + 10 * lane); }
    }
    __syncwarp();
    bool clash = false;
    if (me) {
      int c = spawn_head(entry);
      clash = r.grid[c] != BODY + 10 * lane;
      for (int j = 1; j < K; ++j) { c += dir_delta(spawn_link(entry, j), W); clash |= r.grid[c] != BODY + 10 * lane; }
    }
    const uint32_t any_clash = __ballot_sync(0xffffffffu, clash);
    SNK_RV(5, (unsigned long long)attempt + 1);
    if (!any_clash) break;
    if (rng_mode == RNG_REPLAY) { if (lane == 0) atomicOr(p.err, ERR_REPLAY_RANGE); break; }
    if (attempt + 1 >= SPAWN_ATTEMPT_CAP) { if (lane == 0) atomicOr(p.err, ERR_SPAWN_GIVEUP); break; }
    __syncwarp();
    if (me) {
      int c = spawn_head(entry);
      r.grid[c] = (uint8_t)EMPTY;
      for (int j = 1; j < K; ++j) { c += dir_delta(spawn_link(entry, j), W); r.grid[c] = (uint8_t)EMPTY; }
    }
    __syncwarp();
  }
  __syncwarp();
  // snake table + body directions (toward the head), all snakes at once: with directions in the grid bytes (dig) a
  // snake only touches its own cells, with a direction plane the shared words are updated atomically
  SNK_R(2);
  auto write_snake = [&](int s) {
    int c = spawn_head(entry);
    r.head[s] = (uint16_t)c;
    r.grid[c] = (uint8_t)(HEAD + 10 * s);
    for (int j = 1; j < K; ++j) {
      const int l = spawn_link(entry, j);
      c += dir_delta(l, W);
      r.grid[c] = (uint8_t)((j == K - 1 ? TAIL : BODY) + 10 * s);
      if (d.dig) r.grid[c] = (uint8_t)((r.grid[c] & 63) | (((l + 2) & 3) << 6));   // toward the head
      else dirp_set_atomic(r.dirp, c, (l + 2) & 3);    // plane words are shared between snakes
    }
    r.tail[s] = (uint16_t)c;
    r.len[s] = (uint16_t)K;
    r.dir[s] = (uint8_t)((spawn_link(entry, 1) + 2) & 3);   // coords[0] - coords[1]  core/snake.py:58-61
    r.alive[s] = 1;
    stats_zero(d, r, s);
  };
  if (me) write_snake((int)lane);
  __syncwarp();
  SNK_R(3);
  place_fruits_warp(p, g, vb, env_local, d.nfruits, DRAW_RESET_FRUIT);
  if (lane == 0) { r.hdr->alive_counter = (int16_t)ns; r.hdr->episode_length = 0; }
  __syncwarp();
  SNK_R(4);
}

// ---- the fused step / reset / encode kernel -------------------------------------------------------
//
// Template parameters are compile-time copies of configuration values (0 = read the runtime value):
// the BASELINE shapes get specialised instances so index arithmetic folds to shifts and multiplies.
template <int kNS, int kW, int kOH, int kOW, int kFS>
struct Shape {
  const Dims& d;
  __device__ __forceinline__ explicit Shape(const Dims& dd) : d(dd) {}
  __device__ __forceinline__ int ns() const { return kNS ? kNS : d.ns; }
  __device__ __forceinline__ int W() const { return kW ? kW : d.W; }
  __device__ __forceinline__ int oh() const { return kOH ? kOH : d.oh; }
  __device__ __forceinline__ int ow() const { return kOW ? kOW : d.ow; }
  __device__ __forceinline__ int ohw() const { return oh() * ow(); }
  __device__ __forceinline__ int fs() const { return kFS ? kFS : d.fs; }
  __device__ __forceinline__ int lut_stride() const { return 10 * ns() + 6; }   // cell codes 0 .. 10*(ns-1)+5
  // ENC_PAD plane geometry (mirrors finalize_layout; egocentric windows only, so V = (oh - 1) / 2)
  static constexpr int kV = (kOH - 1) / 2, kPadLeft = (kV + 3) / 4 * 4, kPitch0 = (kPadLeft + kW + kV + 3) / 4 * 4;
  static constexpr int kPitch = ((kPitch0 >> 2) & 1) ? kPitch0 : kPitch0 + 4;
  // ENC_REG packing (see make_viewer_word): width of the row / column one-hot field, and the bias that makes a crop
  // origin non-negative
  __device__ __forceinline__ int view_bits() const { return oh() + ow(); }
  __device__ __forceinline__ int view_bias() const { return (kW && kOH) ? kV * kW + kV : d.V * d.W + d.V; }
  __device__ __forceinline__ int pad_pitch() const { return (kW && kOH) ? kPitch : d.pad_pitch; }
  __device__ __forceinline__ int pad_left() const { return (kW && kOH) ? kPadLeft : d.pad_left; }
  static constexpr int kUnits = (kOH * kOW != 0 && kOH * kOW <= 127) ? 2 : 4;   // 16-byte units a lane owns per viewer
  // the {as-other, as-own} LUT pair is only ever used when one LUT per viewer would exceed 8 KB
  static constexpr bool kMayDual = kNS == 0 || kNS * (10 * kNS + 6) * 8 > 8 * 1024;
  static constexpr int kNSc = kNS;                                              // 0 = runtime
  __device__ __forceinline__ int group() const {                                // lanes per environment
    const int n = ns();
    return n <= 1 ? 1 : n <= 2 ? 2 : n <= 4 ? 4 : n <= 8 ? 8 : n <= 16 ? 16 : 32;
  }
};

__device__ __forceinline__ void st_cs_128(void* p, uint2 a, uint2 b) {
  SNK_CHECK_OBS(p, 16);
  __stcs(reinterpret_cast<uint4*>(p), make_uint4(a.x, a.y, b.x, b.y));
}
__device__ __forceinline__ void st_cs_64(void* p, uint2 a) {
  SNK_CHECK_OBS(p, 8);
  __stcs(reinterpret_cast<uint2*>(p), a);
}
// One 16-byte unit of a viewer block at dst: window cells a and b, 8 bytes each.  A block of an odd cell count is only
// 8-byte aligned, so the unit at either end of it may hold one cell; has_a / has_b say which cells lie in the block.
// A lane's second unit never starts before the block, so its callers pass has_a = true rather than a test the
// compiler cannot fold.
__device__ __forceinline__ void st_cs_unit(uint8_t* dst, bool has_a, bool has_b, uint2 a, uint2 b) {
  if (has_a && has_b) st_cs_128(dst, a, b);
  else if (has_a) st_cs_64(dst, a);
  else st_cs_64(dst + 8, b);
}

// Channel-bit output (snk_step_bits): one byte per window cell, bit c = channel c.  The byte LUT mirrors the 8-byte
// LUT entry for entry, so the entry address `e8` of a cell (lut32 + 8 * index) names its byte at lutb32 + index.
__device__ __forceinline__ void st_bits(uint8_t* q, uint32_t v) {
  SNK_CHECK_BITS(q, 1);
  *q = (uint8_t)v;
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t a);
__device__ __forceinline__ void emit_bits(uint8_t* bitsv, int ca, int ohw, uint32_t lut32, uint32_t lutb32, uint32_t e8a, uint32_t e8b) {
  if (ca >= 0 && ca < ohw) st_bits(bitsv + ca, lds_u8(lutb32 + ((e8a - lut32) >> 3)));
  if (ca + 1 >= 0 && ca + 1 < ohw) st_bits(bitsv + ca + 1, lds_u8(lutb32 + ((e8b - lut32) >> 3)));
}

__device__ __forceinline__ uint32_t lds_u8(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint2 lds_v2(uint32_t a) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
  return v;
}

// ---- 1-D bulk asynchronous copies (TMA engine): cp.async.bulk + mbarrier --------------------------
// The record tile is one contiguous, 16-byte aligned range, so one elected thread moves it with a single
// instruction each way; no registers or LSU wavefronts are spent on it.
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// One arrival that also announces `bytes` of bulk-copy traffic; the phase completes when they have landed.
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}
// Waits for the phase; gives up after two seconds of wall time (%globaltimer, not a poll count: a debugger, a
// profiler replay or a time-sliced GPU may stall a correct run for long) and returns false -- the caller raises the
// sticky ERR_TMA_TIMEOUT bit and skips the tile instead of trapping the whole context.
__device__ __forceinline__ bool mbar_wait(uint32_t mbar, uint32_t parity) {
  uint32_t done = 0;
  unsigned long long t0 = 0;
  for (uint32_t spins = 1; ; ++spins) {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(done) : "r"(mbar), "r"(parity) : "memory");
    if (done) return true;
    if ((spins & 1023u) == 0u) {
      unsigned long long now;
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 2000000000ull) return false;
    }
  }
}
// L2 eviction priority for the record tiles (SNK_L2_KEEP): the records are re-read every step while the observation
// block streams through once, so the record lines are asked to stay (evict_last) under the evict-first observation stores.
// Measured (profiles/r02_ab_l2keep*.txt): cfg3 0.2028 -> 0.1960 ms (its 16 MB of records then never leave the L2), cfg5
// unchanged (252 MB of records against 126 MB of L2), cfg4 and the cfg5 shard 1.5-2 % slower; on by default with a
// frame stack only.  The same hint on the frame-history load did not pay (0.1987 ms).
__device__ __forceinline__ uint64_t l2_policy_evict_last(float fraction) {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, %1;" : "=l"(pol) : "f"(fraction));
  return pol;
}
__device__ __forceinline__ void bulk_load_hint(uint32_t dst, const void* src, uint32_t bytes, uint32_t mbar, uint64_t pol) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar), "l"(pol) : "memory");
}
__device__ __forceinline__ void bulk_store_hint(void* dst, uint32_t src, uint32_t bytes, uint64_t pol) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst), "r"(src), "r"(bytes), "l"(pol) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_store(void* dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// The record tile's bulk copies between HBM (the ne records from e0 on) and shared memory (shared address s32), hinted
// evict_last when the handle asks for it (KParams::l2_keep).  The address is spelled out in each branch on purpose:
// computed once ahead of the branch, it changes the register allocation of every kernel instance.
__device__ __forceinline__ void load_records(const KParams& p, int e0, uint32_t s32, uint32_t bytes, uint32_t mbar) {
  if (p.l2_keep) bulk_load_hint(s32, p.recs + (size_t)e0 * p.d.hbm_rec_bytes, bytes, mbar, l2_policy_evict_last(p.l2_keep_frac));
  else bulk_load(s32, p.recs + (size_t)e0 * p.d.hbm_rec_bytes, bytes, mbar);
}
// Write the tile's records back, shared -> HBM: the elected thread's bulk store, or without TMA 16-byte copies by the
// tile's threads (first, step).  `wait`: the issuer waits for the store's shared-memory reads here; otherwise the
// caller does before the shared memory is reused or the CTA exits.  `s` is the tile's first byte as it lies in HBM,
// s32 its shared address.
__device__ __forceinline__ void store_records(const KParams& p, int e0, int ne, const uint8_t* s, uint32_t s32,
                                              uint32_t bytes, bool elected, bool wait, int first, int step) {
  if (p.use_tma) {
    if (elected) {
      if (p.l2_keep) bulk_store_hint(p.recs + (size_t)e0 * p.d.hbm_rec_bytes, s32, bytes, l2_policy_evict_last(p.l2_keep_frac));
      else bulk_store(p.recs + (size_t)e0 * p.d.hbm_rec_bytes, s32, bytes);
      if (wait) bulk_store_wait_read();
    }
  } else {
    uint4* dst = reinterpret_cast<uint4*>(p.recs + (size_t)e0 * p.d.hbm_rec_bytes);
    const uint4* src = reinterpret_cast<const uint4*>(s);
    const int n16 = ne * (p.d.hbm_rec_bytes >> 4);
    for (int k = first; k < n16; k += step) dst[k] = src[k];
  }
}

struct GroupOut {
  int fruit_taken;     // fruit draws owed by this lane's environment (same on all its lanes)
  bool finished;       // episode ended this step (same on all lanes of the environment)
  bool newly_dead;     // this lane's snake died this step
};

// The step rules with lanes = snakes.  Restates env_step_logic (snk_core.cuh, the sequential form the
// host simulation runs) for a group of G lanes per environment; tests compare the two on the GPU.
// `active`: this lane holds a real snake of a real environment.  All 32 lanes must call.
template <class SH>
__device__ __forceinline__ GroupOut step_group(const KParams& p, const SH& sh, Rec& r, bool active, int i,
                                               uint32_t gmask, int gbase, size_t io, uint32_t action,
                                               uint32_t* kl_scratch) {
  const Dims& d = p.d;
  const uint32_t FULL = 0xffffffffu;
  const uint32_t lane = lane_id();
  const int ns = sh.ns(), W = sh.W(), G = sh.group();

  // 1. relative turn + head advance for live snakes                     snake_env.py:320-330, 598-608
  const bool was_alive = active && r.alive[i] != 0;
  int dirv = 0;
  uint32_t tgt = 0x10000u + lane;                       // unique dummy: never matches a real cell
  if (was_alive) {
    uint32_t a = action;                                  // fetched while the record tile was in flight
    if (a > 2u && !d.observer) { atomicOr(p.err, ERR_BAD_ACTION); a = 0; }
    dirv = d.observer ? turn_absolute(r.dir[i], a) : turn_relative(r.dir[i], a);            // :598-632
    tgt = (uint32_t)(r.head[i] + dir_delta(dirv, W));
    SNK_ASSERT(p, tgt < (uint32_t)d.HW && r.head[i] < d.HW && r.tail[i] < d.HW);
  }
  // 2. one verdict per distinct target cell, on the pre-move grid                      :521-544
  const uint32_t same = __match_any_sync(FULL, tgt) & gmask;     // snakes of my env entering my cell
  const int n = __popc(same);
  const bool first = (__ffs(same) - 1) == (int)lane;             // lowest-index arrival speaks for the cell
  const uint32_t code = was_alive ? cell_code(d, r.grid[tgt]) : 0u;
  const uint32_t owner = (code * 205u) >> 11;
  const uint32_t kind = code - owner * 10u;
  const bool lethal = (kind == WALL) | (kind == BODY) | (kind == HEAD);
  bool died = was_alive && (n > 1 || lethal);
  const bool credit = died && first && (kind == BODY || kind == HEAD);     // owner paid once per cell (C2)
  const bool eater = was_alive && !died && kind == FRUIT;
  if (d.compact && eater) {                           // the eaten fruit leaves the record's slot list
    const int fcap = d.fcap;
#pragma unroll 1
    for (int j = 0; j < fcap; ++j)
      if (r.fruit[j] == (uint16_t)(tgt + 1u)) { r.fruit[j] = 0; break; }
  }
  const int fruit_taken = __popc(__ballot_sync(FULL, was_alive && first && kind == FRUIT) & gmask);   // (C3)
  int counter = r.hdr->alive_counter - __popc(__ballot_sync(FULL, died) & gmask);        // :334

  // 3. kill attribution, tail-growth rule                                              :338-346
  //    No loop over the group: kill credit is a shared-memory scatter (one word per lane), the tail-growth
  //    rule one more match on {eater: own tail, others: target cell}.
  kl_scratch[lane] = 0u;
  __syncwarp();
  if (credit && owner < (uint32_t)G) atomicAdd(&kl_scratch[gbase + (int)owner], 1u);   // once per cell (C2)
  const uint32_t my_tail = active ? (uint32_t)r.tail[i] : 0u;
  // An eater's tail stays this step (:338-346): every snake entering it dies and is counted again even if
  // it already died (C4); each such snake is one kill for the eater.  A target cell is FRUIT for an eater
  // and TAIL for its victims, so an eater never matches as a victim, and tails of two snakes never coincide.
  const uint32_t meet = __match_any_sync(FULL, eater ? my_tail : tgt) & gmask;
  const uint32_t eaters = __ballot_sync(FULL, eater);
  const bool victim = was_alive && !eater && (meet & eaters) != 0u;
  counter -= __popc(__ballot_sync(FULL, victim) & gmask);
  __syncwarp();
  int kl = (int)kl_scratch[lane] + (eater ? __popc(meet) - 1 : 0);
  died |= victim;
  const bool alive_now = was_alive && !died;
  const uint32_t alive_m = __ballot_sync(FULL, alive_now) & gmask;
  const bool won = counter == 1 && ns > 1 && alive_now && (__ffs(alive_m) - 1) == (int)lane;   // :347-352

  // 4. reward: float64, the reference's order, no FMA                                  :365-369
  double rw = 0.0;
  if (was_alive) {
    rw = __dmul_rn(d.r_time, alive_now ? 1.0 : 0.0);
    rw = __dadd_rn(rw, __dmul_rn(d.r_fruit, eater ? 1.0 : 0.0));
    rw = __dadd_rn(rw, __dmul_rn(d.r_lose, died ? 1.0 : 0.0));
    rw = __dadd_rn(rw, __dmul_rn(d.r_kill, (double)kl));
    rw = __dadd_rn(rw, __dmul_rn(d.r_win, won ? 1.0 : 0.0));
  }

  // 5. grid update.  The reference walks snakes in index order (:358-373, :546-566); the final grid is
  //    the same when every clear (vacated tails, bodies of the dead) happens before every write.
  const int tag = 10 * i;
  int new_tail = 0;
  if (was_alive) {
    if (!alive_now) {
      int c = r.tail[i];
      const int hd = r.head[i];
#pragma unroll 1
      for (int guard = 0; guard < d.HW; ++guard) {
        SNK_ASSERT(p, (unsigned)c < (unsigned)d.HW);
        const int nxt = c + dir_delta(body_dir(d, r, c), W);
        r.grid[c] = (uint8_t)EMPTY;
        if (c == hd) break;
        c = nxt;
      }
    } else if (!eater) {
      const int ot = r.tail[i];
      new_tail = ot + dir_delta(body_dir(d, r, ot), W);
      SNK_ASSERT(p, (unsigned)new_tail < (unsigned)d.HW);
      r.grid[ot] = (uint8_t)EMPTY;
    } else {
      new_tail = r.tail[i];
    }
  }
  __syncwarp();
  if (active) {
    if (alive_now) {
      const int oh = r.head[i];
      r.grid[oh] = (uint8_t)((BODY + tag) | (d.dig ? dirv << 6 : 0));
      if (!d.dig) dirp_set_atomic(r.dirp, oh, dirv);
      r.dir[i] = (uint8_t)dirv;
      r.tail[i] = (uint16_t)new_tail;
      if (eater) r.len[i] = (uint16_t)(r.len[i] + 1);
      // length 2: overwrites the BODY just written; the cell keeps its direction bits
      r.grid[new_tail] = (uint8_t)((TAIL + tag) | (d.dig ? (r.grid[new_tail] & 0xC0) : 0));
      r.head[i] = (uint16_t)tgt;
      r.grid[tgt] = (uint8_t)(HEAD + tag);
      r.score[i] = __dadd_rn(r.score[i], rw);          // statistics gate on this step's dones  :385-389
      cnt_step(d, r, i, eater ? 1u : 0u, (uint32_t)kl);
    } else if (was_alive) {
      r.alive[i] = 0; r.len[i] = 0; r.dir[i] = (uint8_t)dirv;
    }
  }
  __syncwarp();

  // 6. outputs, step cap, episode end                                                  :374, :391-412
  const int n_done = __popc(__ballot_sync(FULL, active && !alive_now) & gmask);
  uint32_t ep_len = r.hdr->episode_length + 1u;
  const bool capped = (double)ep_len >= d.max_steps;
  const bool fin = d.done_mode == 0 ? (capped || n_done == ns) : (capped || n_done > 0);
  __syncwarp();
  if (active) {
    if (i == 0) { r.hdr->episode_length = ep_len; r.hdr->alive_counter = (int16_t)counter; }
    p.rew[io] = rw;
    p.done[io] = (capped || !alive_now || (fin && d.done_mode == 1)) ? 1 : 0;
  }
  GroupOut out;
  out.fruit_taken = fruit_taken;
  out.finished = fin;
  out.newly_dead = was_alive && !alive_now;
  return out;
}

// Where a tile's environments live in shared memory: grid of environment q at g + q * gs, its virtual record base
// (c-part address minus off_c0) at vb + q * cs.  Contiguous working records: g == vb, gs == cs == rec_bytes.
// Compact handle: the grids (rebuilt, never stored) in one block, the c-parts (the HBM records) behind it.
struct TilePtr {
  uint8_t* g; uint8_t* vb; int gs, cs;
  __device__ __forceinline__ uint8_t* G(int q) const { return g + (size_t)q * gs; }
  __device__ __forceinline__ uint8_t* VB(int q) const { return vb + (size_t)q * cs; }
};

// Compact records: the grids of the tile arrived as copies of the handle's wall layout; put the fruit cells and the
// live snakes' bodies on them.  Lanes = (environment, snake) as in the rule phase.  A body is walked from its tail
// along the direction plane (each cell's entry points toward the head)      inverse of core/snake.py:86-94
template <class SH>
__device__ __forceinline__ void expand_tile(const KParams& p, const SH& sh, const TilePtr& tp, int ne) {
  const Dims& d = p.d;
  const int lane = (int)lane_id();
  const int ns = sh.ns(), G = sh.group(), W = sh.W();
  const int g = lane / G, i = lane - g * G;
  if (g < ne) {
    const Rec r = rec_view2(tp.G(g), tp.VB(g) + d.off_c0, d);
    const int fcap = d.fcap;
    for (int j = i; j < fcap; j += G) {
      const uint32_t s = r.fruit[j];
      if (s) { SNK_ASSERT(p, s <= (uint32_t)d.HW); r.grid[s - 1u] = (uint8_t)FRUIT; }
    }
  }
  __syncwarp();          // a snake never lies on a fruit cell, but keep the two passes ordered anyway
  if (g < ne && i < ns) {
    const Rec r = rec_view2(tp.G(g), tp.VB(g) + d.off_c0, d);
    if (r.alive[i]) {
      const int hd = r.head[i], tag = 10 * i;
      int c = r.tail[i];
      uint8_t code = (uint8_t)(TAIL + tag);
#pragma unroll 1
      for (int guard = 0; guard < d.HW && c != hd; ++guard) {
        SNK_ASSERT(p, (unsigned)c < (unsigned)d.HW);
        r.grid[c] = code;
        code = (uint8_t)(BODY + tag);
        c += dir_delta(dirp_get(r.dirp, c), W);
      }
      r.grid[hd] = (uint8_t)(HEAD + tag);
    }
  }
  __syncwarp();
}

// ---- one warp: rules + terminal info + rollout statistics + rare events for a tile ----------------
// Leaves per-environment flags in s_flag[] (F_RESET / F_INIT / F_SKIP).
template <bool kPool, class SH>
__device__ __forceinline__ void tile_rules(const KParams& p, const SH& sh, const TilePtr& tp, int e0, int ne,
                                           uint8_t* s_flag, uint32_t action, int t) {
  const Dims& d = p.d;
  const uint32_t FULL = 0xffffffffu;
  const uint32_t lane = lane_id();
  const int ns = sh.ns(), G = sh.group();
  // lane = (environment g of the tile, snake i)
  const int g = (int)lane / G, i = (int)lane - g * G;
  const int gbase = g * G;
  const uint32_t gmask = (G == 32 ? FULL : ((1u << G) - 1u)) << gbase;
  const bool env_ok = g < ne;
  const bool active = env_ok && i < ns;
  const int e = e0 + g;
  Rec r = rec_view2(tp.G(env_ok ? g : 0), tp.VB(env_ok ? g : 0) + d.off_c0, d);
  // outputs of step t of a multi-step launch (snk_step_many) land t * [N, ns] (t * [N] for `finished`) further on
  const size_t io = (size_t)t * d.N * ns + (size_t)e * ns + i;
  const size_t ie = (size_t)t * d.N + e;

  uint8_t flag = 0;            // per environment (identical on its lanes)
  int fruit = 0;
  if (p.mode == MODE_STEP) {
    if (e0 == 0 && lane == 0) atomicAdd(p.stats + STAT_ENV_STEPS, (double)d.N);   // once per launch: env steps executed
    if (active && i == 0) r.hdr->event += 1;
    __syncwarp();
    // kill-credit scratch: the tile's 32 viewer words, which are only filled after the rules
    const GroupOut res = step_group(p, sh, r, active, i, gmask, gbase, io, action,
                                    reinterpret_cast<uint32_t*>(s_flag + 48));
    fruit = res.fruit_taken;
    // terminal info, rollout statistics, statistics reset                          :396-412
    const bool fin = env_ok && res.finished;
    if (active && i == 0 && p.fin) p.fin[ie] = fin ? 1 : 0;
    const uint32_t fin_m = __ballot_sync(FULL, fin && i == 0);
    const uint32_t dead_m = __ballot_sync(FULL, res.newly_dead);
    if (lane == 0 && dead_m) atomicAdd(p.stats + STAT_DEATHS, (double)__popc(dead_m));
    if (fin_m) {                                                  // some environment of the tile ended
      const double my_score = active ? r.score[i] : 0.0;
      int rk = 1;
      for (int j = 0; j < G; ++j) {
        const double sj = __shfl_sync(FULL, my_score, gbase + j);
        rk += (j < ns && sj > my_score) ? 1 : 0;                  // competition rank          :397-404
      }
      double ret = 0.0; uint32_t fr = 0, kl = 0, ln = 0;
      if (fin && active) {
        if (p.rank) p.rank[io] = rk;
        if (p.ep_scores) p.ep_scores[io] = my_score;
        fr = cnt_get(d, r, CNT_FRUITS, i); kl = cnt_get(d, r, CNT_KILLS, i);
        if (p.ep_steps) p.ep_steps[io] = (int32_t)cnt_get(d, r, CNT_STEPS, i);
        if (p.ep_fruits) p.ep_fruits[io] = (int32_t)fr;
        if (p.ep_kills) p.ep_kills[io] = (int32_t)kl;
        ret = my_score;
        if (i == 0) ln = r.hdr->episode_length;
        stats_zero(d, r, i);
      }
      for (int o = 16; o; o >>= 1) ret += __shfl_xor_sync(FULL, ret, o);
      fr = __reduce_add_sync(FULL, fr); kl = __reduce_add_sync(FULL, kl); ln = __reduce_add_sync(FULL, ln);
      if (lane == 0) {
        atomicAdd(p.stats + STAT_EPISODES, (double)__popc(fin_m));
        atomicAdd(p.stats + STAT_RETURN, ret);
        atomicAdd(p.stats + STAT_EP_STEPS, (double)ln);
        atomicAdd(p.stats + STAT_FRUITS, (double)fr);
        atomicAdd(p.stats + STAT_KILLS, (double)kl);
      }
      if (fin && d.auto_reset) flag |= F_RESET;                   // wrappers.py:141-143
    }
  } else {
    const bool sel = env_ok && (p.mask == nullptr || p.mask[e] != 0);
    if (!sel) flag = F_SKIP;
    else if (p.mode == MODE_RESET) { if (i == 0) r.hdr->event += 1; flag = F_RESET; }
    else flag = F_INIT;
  }
  if (!env_ok) flag = F_SKIP;
  __syncwarp();

  // ---- rare events, whole warp per environment: only environments that owe a fruit draw or a reset
  if (env_ok && i == 0) s_flag[g] = flag;
  uint32_t ev = __ballot_sync(FULL, env_ok && i == 0 && (fruit != 0 || (flag & F_RESET)));
#pragma unroll 1
  while (ev) {
    const int src = __ffs(ev) - 1;                 // first lane of the environment's lane group
    ev &= ev - 1;
    const int q = src / G;
    const int qf = __shfl_sync(FULL, fruit, src);
    const int qflag = __shfl_sync(FULL, (int)flag, src);
    if (qf) place_fruits_warp(p, tp.G(q), tp.VB(q), (uint32_t)(e0 + q), qf, DRAW_STEP_FRUIT);
    if (qflag & F_RESET) reset_env_warp<kPool>(p, tp.G(q), tp.VB(q), (uint32_t)(e0 + q));
  }
  __syncwarp();
}

// Crop origin of viewer v: own head, or cell (0,0) when it has no head in the grid       :500-502
__device__ __forceinline__ void viewer_origin(const Dims& d, const uint8_t* base, int ns, int W, int V, int v,
                                              int& r0, int& c0) {
  const uint8_t alive = base[d.off_snk + 7 * ns + v];
  const int hc = alive ? (int)((const uint16_t*)(base + d.off_snk))[v] : 0;
  r0 = 0; c0 = 0;
  if (V > 0) { const int hr = hc / W; r0 = hr - V; c0 = hc - hr * W - V; }
}

// Window rows / columns of a viewer that fall inside the grid, as bit masks: rows in bits 0..oh-1, columns from bit
// `col_shift` on.
__device__ __forceinline__ uint32_t window_valid(int oh, int ow, int H, int W, int r0, int c0, int col_shift) {
  const int rlo = max(0, -r0), rhi = min(oh, H - r0), clo = max(0, -c0), chi = min(ow, W - c0);
  return (((1u << rhi) - 1u) & ~((1u << rlo) - 1u)) | ((((1u << chi) - 1u) & ~((1u << clo) - 1u)) << col_shift);
}
// The same for the encode table's entries (rows in bits 0..15, columns in 16..31).
__device__ __forceinline__ uint32_t window_mask(int V, int oh, int ow, int H, int W, int r0, int c0) {
  if (V <= 0) return 0u;
  return window_valid(oh, ow, H, W, r0, c0, 16);
}

// frame_stack 1: one warp encodes one viewer straight to global memory.  snake_env.py:474-519.
// Each lane produces 16 output bytes (two window cells x 8 channels) per unit: window-table entry ->
// AND/compare against the viewer's valid row/column masks (the zero padding of :506-515) -> grid byte
// -> LUT row -> one 128-bit streaming store.  A viewer block of ohw*8 bytes is only 8-byte aligned
// when ohw is odd, so units are laid out from the address parity and the end units may be half units.
template <class SH>
__device__ __forceinline__ void encode_viewer_fs1(const KParams& p, const SH& sh, const uint8_t* base, const uint8_t* vb,
                                                  uint32_t grid32, int v, uint8_t* outv, uint32_t lut32,
                                                  uint8_t* bitsv, uint32_t lutb32) {
  const Dims& d = p.d;
  const uint32_t lane = lane_id();
  const int ns = sh.ns(), W = sh.W(), ohw = sh.ohw(), ow = sh.ow(), oh = sh.oh(), LS = sh.lut_stride();
  const int H = d.H, V = d.V;
  const uint8_t* grid = base;
  int r0, c0;
  viewer_origin(d, vb, ns, W, V, v, r0, c0);
  const int shift = (int)((reinterpret_cast<uintptr_t>(outv) >> 3) & 1);
  const int units = (ohw + shift + 1) >> 1;
  if (p.use_tab) {
    const uint32_t tab32 = lut32 + (uint32_t)p.enc_tab_off + 8u;       // entry of window cell 0
    const uint32_t maskpk = window_mask(V, oh, ow, H, W, r0, c0);
    // per-viewer LUT (small ns) or the {as-other, as-own} pair selected per cell by owner == v
    const bool dual = SH::kMayDual && p.lut_dual != 0;
    const uint32_t lutv32 = dual ? lut32 : lut32 + (uint32_t)(v * LS) * 8u;   // entry 0 is all zero
    const uint32_t lutown = lut32 + (uint32_t)LS * 8u;
    const uint32_t gorg = grid32 + (uint32_t)(r0 * W + c0);
    // two units per lane per trip: all table loads, then all grid bytes, then all LUT rows, so the
    // three dependent shared-memory round trips of both units overlap
    for (int u0 = (int)lane; u0 < units; u0 += 64) {
      const int u1 = u0 + 32;
      const bool has1 = u1 < units;
      const int ca0 = 2 * u0 - shift, ca1 = 2 * (has1 ? u1 : u0) - shift;
      const uint2 ea0 = lds_v2(tab32 + (uint32_t)(ca0 * 8));
      const uint2 eb0 = lds_v2(tab32 + (uint32_t)(ca0 * 8 + 8));
      const uint2 ea1 = lds_v2(tab32 + (uint32_t)(ca1 * 8));
      const uint2 eb1 = lds_v2(tab32 + (uint32_t)(ca1 * 8 + 8));
      const uint32_t aa0 = ((ea0.x & maskpk) == ea0.x) ? gorg + ea0.y : lutv32;
      const uint32_t ab0 = ((eb0.x & maskpk) == eb0.x) ? gorg + eb0.y : lutv32;
      const uint32_t aa1 = ((ea1.x & maskpk) == ea1.x) ? gorg + ea1.y : lutv32;
      const uint32_t ab1 = ((eb1.x & maskpk) == eb1.x) ? gorg + eb1.y : lutv32;
      const uint32_t cm = (uint32_t)d.code_mask;
      const uint32_t ka0 = lds_u8(aa0) & cm, kb0 = lds_u8(ab0) & cm, ka1 = lds_u8(aa1) & cm, kb1 = lds_u8(ab1) & cm;
      uint32_t la0 = lutv32, lb0 = lutv32, la1 = lutv32, lb1 = lutv32;
      if (dual) {
        la0 = (((ka0 * 205u) >> 11) == (uint32_t)v) ? lutown : lut32;
        lb0 = (((kb0 * 205u) >> 11) == (uint32_t)v) ? lutown : lut32;
        la1 = (((ka1 * 205u) >> 11) == (uint32_t)v) ? lutown : lut32;
        lb1 = (((kb1 * 205u) >> 11) == (uint32_t)v) ? lutown : lut32;
      }
      if (outv) {
        const uint2 qa0 = lds_v2(la0 + ka0 * 8u), qb0 = lds_v2(lb0 + kb0 * 8u);
        const uint2 qa1 = lds_v2(la1 + ka1 * 8u), qb1 = lds_v2(lb1 + kb1 * 8u);
        st_cs_unit(outv + (ptrdiff_t)ca0 * 8, ca0 >= 0, ca0 + 1 < ohw, qa0, qb0);
        if (has1) st_cs_unit(outv + (ptrdiff_t)ca1 * 8, true, ca1 + 1 < ohw, qa1, qb1);
      }
      if (bitsv) {
        emit_bits(bitsv, ca0, ohw, lut32, lutb32, la0 + ka0 * 8u, lb0 + kb0 * 8u);
        if (has1) emit_bits(bitsv, ca1, ohw, lut32, lutb32, la1 + ka1 * 8u, lb1 + kb1 * 8u);
      }
    }
  } else {                       // windows wider than 16 cells: plain index arithmetic, per-viewer LUT
    const uint2* lut = reinterpret_cast<const uint2*>(__cvta_shared_to_generic(lut32)) + v * LS;
    for (int u = (int)lane; u < units; u += 32) {
      const int ca = 2 * u - shift, cb = ca + 1;
      const bool va = ca >= 0, vb = cb < ohw;
      uint2 qa, qb;
      uint32_t codea = 0, codeb = 0;
      {
        const int c = va ? ca : 0;
        const int ci = c / ow, cj = c - ci * ow;
        const int rr = r0 + ci, cc = c0 + cj;
        if ((unsigned)rr < (unsigned)H && (unsigned)cc < (unsigned)W) codea = cell_code(d, grid[rr * W + cc]);
        qa = lut[codea];
      }
      {
        const int c = vb ? cb : 0;
        const int ci = c / ow, cj = c - ci * ow;
        const int rr = r0 + ci, cc = c0 + cj;
        if ((unsigned)rr < (unsigned)H && (unsigned)cc < (unsigned)W) codeb = cell_code(d, grid[rr * W + cc]);
        qb = lut[codeb];
      }
      if (outv) {               // st_cs_unit, written out: through the helper this loop is scheduled differently
        uint8_t* dst = outv + (ptrdiff_t)ca * 8;
        if (va && vb) st_cs_128(dst, qa, qb);
        else if (va) st_cs_64(dst, qa);
        else st_cs_64(dst + 8, qb);
      }
      if (bitsv) {
        const uint32_t lv = lut32 + (uint32_t)(v * LS) * 8u;
        emit_bits(bitsv, ca, ohw, lut32, lutb32, lv + codea * 8u, lv + codeb * 8u);
      }
    }
  }
}

// ---- ENC_REG / ENC_DIRECT ------------------------------------------------------------------------
// Packed words (B = view_bits = oh + ow):
//   cell word    bits [0,oh) one-hot window row | bits [oh,B) one-hot window column | grid offset << B;
//                bit 31 set for a cell outside the viewer block (half units at the block ends)
//   viewer word  bits [0,B) rows / columns of the window that fall OUTSIDE the grid | (origin + bias) << B
// A window cell reads the grid iff (cell & (viewer | 1<<31)) has no bit in [0,B) or bit 31; otherwise it
// reads LUT entry 0 (all zero), the reference's zero padding (snake_env.py:506-515).
struct CellWords { uint32_t w[2][4]; };     // [address parity of the viewer block][unit 0 cell a, b, unit 1 cell a, b]

// Cell word of window cell c (inside the viewer block).
template <class SH>
__device__ __forceinline__ uint32_t cell_word(const SH& sh, int c, int B) {
  const int ow = sh.ow(), ci = c / ow, cj = c - ci * ow;
  return (1u << ci) | (1u << (sh.oh() + cj)) | ((uint32_t)(ci * sh.W() + cj) << B);
}

template <class SH>
__device__ __forceinline__ CellWords make_cell_words(const SH& sh, int B) {
  const int lane = (int)lane_id(), ohw = sh.ohw();
  CellWords cw;
#pragma unroll
  for (int s = 0; s < 2; ++s)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int c = 2 * (lane + 32 * (k >> 1)) - s + (k & 1);
      cw.w[s][k] = (c >= 0 && c < ohw) ? cell_word(sh, c, B) : 0x80000000u;
    }
  return cw;
}

// Viewer word of snake v of the record at `base` (rule warp, after rules and resets).
template <class SH>
__device__ __forceinline__ uint32_t make_viewer_word(const KParams& p, const SH& sh, const uint8_t* base, int v) {
  const Dims& d = p.d;
  const int W = sh.W(), oh = sh.oh(), ow = sh.ow(), B = sh.view_bits();
  int r0, c0;
  viewer_origin(d, base, sh.ns(), W, d.V, v, r0, c0);
  const uint32_t valid = window_valid(oh, ow, d.H, W, r0, c0, oh);
  return (~valid & ((1u << B) - 1u)) | ((uint32_t)(r0 * W + c0 + sh.view_bias()) << B);
}

// ---- ENC_REG, viewer pairs (warp-private tiles, frame_stack 1, NHWC only) ---------------------------
// With an odd window (ohw cells) a viewer block of 8 * ohw bytes is only 8-byte aligned, but two consecutive viewers
// (v, v+1) make 2 * ohw cells = ohw whole 16-byte units, and with an even number of viewers per environment every such
// pair block starts 16-byte aligned whenever the environment blocks do (p.vec16).  Unit S = ohw / 2 holds the last cell
// of v and the first of v+1.  Lane l owns four units, at the same place in every pair block:
//   slot 0: unit l,  slot 1: unit 32 + l      (viewer v, while <= S; cell b of unit S is cell 0 of v+1)
//   slot 2: unit S+1 + l,  slot 3: unit S+33 + l  (viewer v+1, while < ohw)
// so which viewer a cell belongs to is fixed per lane: only the one lane holding unit S switches viewers for cell b.
// The cell words (same packing as make_cell_words, idle cells flagged in bit 31) live in a CellWords:
// w[0][k] = cell a, w[1][k] = cell b of slot k.
__device__ __forceinline__ int pair_unit(int k, int lane, int S) { return k < 2 ? 32 * k + lane : S + 1 + 32 * (k - 2) + lane; }

template <class SH>
__device__ __forceinline__ bool pair_unit_used(const SH& sh, int k, int lane) {
  const int S = sh.ohw() >> 1, u = pair_unit(k, lane, S);
  return k < 2 ? u <= S : u < sh.ohw();
}

template <class SH>
__device__ __forceinline__ CellWords make_pair_cell_words(const SH& sh) {
  const int lane = (int)lane_id(), ohw = sh.ohw(), B = sh.view_bits();
  CellWords cw;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int u = pair_unit(k, lane, ohw >> 1);
    const bool used = pair_unit_used(sh, k, lane);
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      int c = 2 * u + s;
      if (c >= ohw) c -= ohw;                                  // window cell inside its own viewer
      cw.w[s][k] = used ? cell_word(sh, c, B) : 0x80000000u;
    }
  }
  return cw;
}

// All viewer pairs of one environment.  view32: shared address of the environment's viewer words (s_view), outl: its
// observation block plus 16 * lane.  kMask: grid bytes carry direction bits (code_mask 63).
template <class SH, bool kMask>
__device__ __forceinline__ void encode_env_pairs(const KParams& p, const SH& sh, uint32_t grid32, uint32_t view32,
                                                 const CellWords& cw, uint8_t* outl, uint32_t lut32) {
  const int lane = (int)lane_id();
  const int ns = sh.ns(), ohw = sh.ohw(), S = ohw >> 1, B = sh.view_bits(), LS = sh.lut_stride();
  const uint32_t field = (1u << B) - 1u;
  const uint32_t gbase = grid32 - (uint32_t)sh.view_bias();
  const uint32_t zero = lut32;                                   // LUT entry 0 of viewer 0: a zero byte (code EMPTY)
  const uint32_t cm = (uint32_t)p.d.code_mask;
  // the lane holding unit S, in slot 0 or 1
  const bool split0 = S < 32 && lane == S, split1 = S >= 32 && lane == S - 32;
  const bool st0 = pair_unit_used(sh, 0, lane), st1 = pair_unit_used(sh, 1, lane);
  const bool st2 = pair_unit_used(sh, 2, lane), st3 = pair_unit_used(sh, 3, lane);
  const int o2 = 16 * (S + 1), o3 = 16 * (S + 33);              // byte offsets of slots 2 and 3 (lane part in outl)
  auto cell = [&](uint32_t e, uint32_t bad, uint32_t org, uint32_t lut) -> uint2 {
    const uint32_t a = (e & bad) ? zero : org + (e >> B);
    SNK_ASSERT(p, a == zero || a - grid32 < (uint32_t)p.d.HW);
    const uint32_t k = kMask ? lds_u8(a) & cm : lds_u8(a);      // (an AND with 0xff would not be folded: lds_u8 is asm)
    SNK_ASSERT(p, k < (uint32_t)LS);
    return lds_v2(lut + k * 8u);
  };
#pragma unroll 1
  for (int v = 0; v < ns; v += 2) {
    const uint2 vw = lds_v2(view32 + 4u * (uint32_t)v);
    const uint32_t bad0 = (vw.x & field) | 0x80000000u, bad1 = (vw.y & field) | 0x80000000u;
    const uint32_t org0 = gbase + (vw.x >> B), org1 = gbase + (vw.y >> B);
    const uint32_t lut0 = lut32 + (uint32_t)(v * LS) * 8u, lut1 = lut0 + (uint32_t)LS * 8u;
    const uint2 q0a = cell(cw.w[0][0], bad0, org0, lut0);
    const uint2 q0b = cell(cw.w[1][0], split0 ? bad1 : bad0, split0 ? org1 : org0, split0 ? lut1 : lut0);
    const uint2 q1a = cell(cw.w[0][1], bad0, org0, lut0);
    const uint2 q1b = cell(cw.w[1][1], split1 ? bad1 : bad0, split1 ? org1 : org0, split1 ? lut1 : lut0);
    const uint2 q2a = cell(cw.w[0][2], bad1, org1, lut1), q2b = cell(cw.w[1][2], bad1, org1, lut1);
    const uint2 q3a = cell(cw.w[0][3], bad1, org1, lut1), q3b = cell(cw.w[1][3], bad1, org1, lut1);
    uint8_t* const o = outl + (size_t)v * ohw * 8;
    if (st0) st_cs_128(o, q0a, q0b);
    if (st1) st_cs_128(o + 512, q1a, q1b);
    if (st2) st_cs_128(o + o2, q2a, q2b);
    if (st3) st_cs_128(o + o3, q3a, q3b);
  }
}

template <class SH>
__device__ __forceinline__ void encode_viewer_reg(const KParams& p, const SH& sh, uint32_t grid32, uint32_t vw,
                                                  const CellWords& cw, int v, uint8_t* outv, uint32_t lut32,
                                                  uint8_t* bitsv, uint32_t lutb32) {
  const int lane = (int)lane_id();
  const int ohw = sh.ohw(), B = sh.view_bits();
  const uint32_t lutv32 = lut32 + (uint32_t)(v * sh.lut_stride()) * 8u;          // entry 0 is all zero
  const uint32_t bad = (vw & ((1u << B) - 1u)) | 0x80000000u;
  const uint32_t gorg = grid32 + (vw >> B) - (uint32_t)sh.view_bias();
  const int shift = (int)((reinterpret_cast<uintptr_t>(outv) >> 3) & 1);
  const int units = (ohw + shift + 1) >> 1;                                       // <= 64
  const uint32_t e0 = shift ? cw.w[1][0] : cw.w[0][0], e1 = shift ? cw.w[1][1] : cw.w[0][1];
  const uint32_t e2 = shift ? cw.w[1][2] : cw.w[0][2], e3 = shift ? cw.w[1][3] : cw.w[0][3];
  const uint32_t a0 = (e0 & bad) ? lutv32 : gorg + ((e0 & 0x7fffffffu) >> B);
  const uint32_t a1 = (e1 & bad) ? lutv32 : gorg + ((e1 & 0x7fffffffu) >> B);
  const uint32_t a2 = (e2 & bad) ? lutv32 : gorg + ((e2 & 0x7fffffffu) >> B);
  const uint32_t a3 = (e3 & bad) ? lutv32 : gorg + ((e3 & 0x7fffffffu) >> B);
  SNK_ASSERT(p, (a0 == lutv32 || a0 - grid32 < (uint32_t)p.d.HW) && (a1 == lutv32 || a1 - grid32 < (uint32_t)p.d.HW) &&
                (a2 == lutv32 || a2 - grid32 < (uint32_t)p.d.HW) && (a3 == lutv32 || a3 - grid32 < (uint32_t)p.d.HW));
  const uint32_t cm = (uint32_t)p.d.code_mask;
  const uint32_t k0 = lds_u8(a0) & cm, k1 = lds_u8(a1) & cm, k2 = lds_u8(a2) & cm, k3 = lds_u8(a3) & cm;
  SNK_ASSERT(p, k0 < (uint32_t)sh.lut_stride() && k1 < (uint32_t)sh.lut_stride() && k2 < (uint32_t)sh.lut_stride() &&
                k3 < (uint32_t)sh.lut_stride());
  const int ca0 = 2 * lane - shift, ca1 = ca0 + 64;
  if (outv) {
    const uint2 q0 = lds_v2(lutv32 + k0 * 8u), q1 = lds_v2(lutv32 + k1 * 8u);
    const uint2 q2 = lds_v2(lutv32 + k2 * 8u), q3 = lds_v2(lutv32 + k3 * 8u);
    if (lane < units) st_cs_unit(outv + (ptrdiff_t)ca0 * 8, ca0 >= 0, ca0 + 1 < ohw, q0, q1);
    if (lane + 32 < units) st_cs_unit(outv + (ptrdiff_t)ca1 * 8, true, ca1 + 1 < ohw, q2, q3);
  }
  if (bitsv) {
    emit_bits(bitsv, ca0, ohw, lut32, lutb32, lutv32 + k0 * 8u, lutv32 + k1 * 8u);
    emit_bits(bitsv, ca1, ohw, lut32, lutb32, lutv32 + k2 * 8u, lutv32 + k3 * 8u);
  }
}

// ---- ENC_PAD ---------------------------------------------------------------------------------------
// The tile's grids have been copied into zero-bordered planes (cell codes, direction bits masked off), so the
// window of a viewer is a plain rectangle of the plane: cell (ci, cj) is byte origin + ci * pitch + cj, and
// cells outside the grid read the zero border -- the reference's zero padding (snake_env.py:506-515).
template <int kU> struct PadCells { uint32_t off[2 * kU]; };

// Plane offsets of the window cells a lane owns, for viewer blocks of address parity `shift`: unit k of a
// lane holds window cells 2 * (lane + 32 k) - shift and the next one (one 16-byte store).
template <class SH, int kU>
__device__ __forceinline__ PadCells<kU> make_pad_cells(const SH& sh, int shift) {
  const int lane = (int)lane_id(), ohw = sh.ohw(), ow = sh.ow(), P = sh.pad_pitch();
  PadCells<kU> pc;
#pragma unroll
  for (int k = 0; k < 2 * kU; ++k) {
    const int c = 2 * (lane + 32 * (k >> 1)) - shift + (k & 1);
    uint32_t o = 0u;                       // outside the viewer block: reads the window's first cell, never stored
    if (c >= 0 && c < ohw) { const int ci = c / ow; o = (uint32_t)(ci * P + (c - ci * ow)); }
    pc.off[k] = o;
  }
  return pc;
}

template <class SH, int kU>
__device__ __forceinline__ void encode_viewer_pad(const KParams& p, const SH& sh, uint32_t org32, const PadCells<kU>& pc,
                                                  int shift, int v, uint8_t* outv, uint32_t lut32,
                                                  uint8_t* bitsv, uint32_t lutb32) {
  const int lane = (int)lane_id(), ohw = sh.ohw(), LS = sh.lut_stride();
  const bool dual = SH::kMayDual && p.lut_dual != 0;        // {as-other, as-own} pair instead of one LUT per viewer
  const uint32_t lutv32 = dual ? lut32 : lut32 + (uint32_t)(v * LS) * 8u;
  const uint32_t own_lo = 10u * (uint32_t)v + 3u, own_delta = (uint32_t)LS * 8u;
  const int units = (ohw + shift + 1) >> 1;
#pragma unroll
  for (int k2 = 0; k2 < kU; k2 += 2) {                       // two units (four cells) in flight
    const uint32_t c0 = lds_u8(org32 + pc.off[2 * k2]), c1 = lds_u8(org32 + pc.off[2 * k2 + 1]);
    const uint32_t c2 = lds_u8(org32 + pc.off[2 * k2 + 2]), c3 = lds_u8(org32 + pc.off[2 * k2 + 3]);
    SNK_ASSERT(p, c0 < (uint32_t)LS && c1 < (uint32_t)LS && c2 < (uint32_t)LS && c3 < (uint32_t)LS);
    uint32_t a0 = lutv32 + c0 * 8u, a1 = lutv32 + c1 * 8u, a2 = lutv32 + c2 * 8u, a3 = lutv32 + c3 * 8u;
    if (dual) {                                              // own HEAD / BODY / TAIL: codes 10v+3 .. 10v+5
      a0 += (c0 - own_lo < 3u) ? own_delta : 0u; a1 += (c1 - own_lo < 3u) ? own_delta : 0u;
      a2 += (c2 - own_lo < 3u) ? own_delta : 0u; a3 += (c3 - own_lo < 3u) ? own_delta : 0u;
    }
    const int u0 = lane + 32 * k2, u1 = u0 + 32;
    const int ca0 = 2 * u0 - shift, ca1 = 2 * u1 - shift;
    if (outv) {
      const uint2 q0 = lds_v2(a0), q1 = lds_v2(a1), q2 = lds_v2(a2), q3 = lds_v2(a3);
      if (u0 < units) st_cs_unit(outv + (ptrdiff_t)ca0 * 8, ca0 >= 0, ca0 + 1 < ohw, q0, q1);
      if (u1 < units) st_cs_unit(outv + (ptrdiff_t)ca1 * 8, true, ca1 + 1 < ohw, q2, q3);
    }
    if (bitsv) {
      emit_bits(bitsv, ca0, ohw, lut32, lutb32, a0, a1);
      emit_bits(bitsv, ca1, ohw, lut32, lutb32, a2, a3);
    }
  }
}

// Full-grid observation: the window IS the grid, so window cell c reads grid byte c.
template <class SH>
__device__ __forceinline__ void encode_viewer_direct(const SH& sh, uint32_t grid32, int v, uint8_t* outv, uint32_t lut32,
                                                     uint32_t cm, uint8_t* bitsv, uint32_t lutb32) {
  const int lane = (int)lane_id();
  const int ohw = sh.ohw();
  const uint32_t lutv32 = lut32 + (uint32_t)(v * sh.lut_stride()) * 8u;
  const int shift = (int)((reinterpret_cast<uintptr_t>(outv) >> 3) & 1);
  const int units = (ohw + shift + 1) >> 1;
  for (int u0 = lane; u0 < units; u0 += 64) {
    const int u1 = u0 + 32;
    const bool has1 = u1 < units;
    const int ca0 = 2 * u0 - shift, ca1 = 2 * (has1 ? u1 : u0) - shift;
    const uint32_t k0 = lds_u8(ca0 >= 0 ? grid32 + (uint32_t)ca0 : lutv32) & cm;     // cm: grid byte -> cell code
    const uint32_t k1 = lds_u8(ca0 + 1 < ohw ? grid32 + (uint32_t)(ca0 + 1) : lutv32) & cm;
    const uint32_t k2 = lds_u8(ca1 >= 0 ? grid32 + (uint32_t)ca1 : lutv32) & cm;
    const uint32_t k3 = lds_u8(ca1 + 1 < ohw ? grid32 + (uint32_t)(ca1 + 1) : lutv32) & cm;
    if (outv) {
      const uint2 q0 = lds_v2(lutv32 + k0 * 8u), q1 = lds_v2(lutv32 + k1 * 8u);
      const uint2 q2 = lds_v2(lutv32 + k2 * 8u), q3 = lds_v2(lutv32 + k3 * 8u);
      st_cs_unit(outv + (ptrdiff_t)ca0 * 8, ca0 >= 0, ca0 + 1 < ohw, q0, q1);
      if (has1) st_cs_unit(outv + (ptrdiff_t)ca1 * 8, true, ca1 + 1 < ohw, q2, q3);
    }
    if (bitsv) {
      emit_bits(bitsv, ca0, ohw, lut32, lutb32, lutv32 + k0 * 8u, lutv32 + k1 * 8u);
      if (has1) emit_bits(bitsv, ca1, ohw, lut32, lutb32, lutv32 + k2 * 8u, lutv32 + k3 * 8u);
    }
  }
}

// frame_stack 1, one viewer in the flavour kEnc (not the viewer pairs): grid `base` of the environment at shared address
// grid32, its virtual record base vb, the viewer's packed word vw (ENC_REG).
template <int kEnc, class SH>
__device__ __forceinline__ void encode_viewer(const KParams& p, const SH& sh, const uint8_t* base, const uint8_t* vb,
                                              uint32_t grid32, uint32_t vw, const CellWords& cw, int v, uint8_t* outv,
                                              uint32_t lut32, uint8_t* bitsv, uint32_t lutb32) {
  if (kEnc == ENC_REG) encode_viewer_reg(p, sh, grid32, vw, cw, v, outv, lut32, bitsv, lutb32);
  else if (kEnc == ENC_DIRECT) encode_viewer_direct(sh, grid32, v, outv, lut32, (uint32_t)p.d.code_mask, bitsv, lutb32);
  else encode_viewer_fs1(p, sh, base, vb, grid32, v, outv, lut32, bitsv, lutb32);
}

// frame_stack > 1: one warp encodes one environment.  Channel-bit bytes of all fs frames are staged in
// output order ([viewer][cell][frame], oldest first) in the warp's staging area, then expanded to NHWC
// with flat 128-bit stores.  The frame history lives in HBM as one byte per window cell per stored frame,
// rows of a ring (hist layout); each step reads fs-1 rows and writes one.
template <class SH, int kFS, bool kBits>
__device__ __forceinline__ void encode_env_stacked(const KParams& p, const SH& sh, const uint8_t* base, const uint8_t* vb, int e,
                                                   int qflag, uint8_t* s_stage, uint32_t lut32, const uint8_t* s_lut,
                                                   const uint8_t* s_hist) {
  const Dims& d = p.d;
  const uint32_t lane = lane_id();
  const int ns = sh.ns(), W = sh.W(), ohw = sh.ohw(), ow = sh.ow(), oh = sh.oh(), LS = sh.lut_stride(), fs = sh.fs();
  const int H = d.H, V = d.V;
  uint8_t* const bits_out = kBits ? p.bits : nullptr;
  const bool want_nhwc = p.obs != nullptr;
  const bool want_obs = want_nhwc || bits_out != nullptr;      // staging is needed for either output
  const bool vec16 = want_nhwc && p.vec16 != 0;
  const uint32_t tab32 = lut32 + (uint32_t)p.enc_tab_off + 8u;
  const uint8_t* grid = base;
  const uint32_t grid32 = (uint32_t)__cvta_generic_to_shared(grid);
  const bool init = (qflag & (F_RESET | F_INIT)) != 0;
  const int hpos = (int)((const EnvHdr*)(vb + d.off_hdr))->hpos;
  // The environment's whole history block (ns x fs rows) was staged into shared memory by the same bulk copy
  // barrier as its record, so the kept frames cost no HBM round trip here; only the new row goes out.
#pragma unroll 1
  for (int v = 0; v < ns; ++v) {
    int r0, c0;
    viewer_origin(d, vb, ns, W, V, v, r0, c0);
    uint8_t* stg = s_stage + (size_t)v * ohw * fs;
    uint8_t* hrow = p.hist + (size_t)e * d.hist_env_bytes + (size_t)(v * fs) * d.ohw_p;
    const uint8_t* srow = s_hist + (size_t)(v * fs) * d.ohw_p;                  // the same rows, staged
    if (kFS == 4 && p.use_tab) {
      // four consecutive window cells per lane: the new frame's bits as one word, the three kept history
      // rows as one word each, 4x4 byte transpose to per-cell words of four frames
      const uint32_t maskpk = window_mask(V, oh, ow, H, W, r0, c0);
      const uint32_t lutv32 = lut32 + (uint32_t)(v * LS);               // entry 0 is zero
      const uint32_t gorg = grid32 + (uint32_t)(r0 * W + c0);
      for (int c4 = (int)lane * 4; c4 < ohw; c4 += 128) {
        uint32_t nw = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int c = min(c4 + k, ohw);                                 // c == ohw: sentinel entry
          const uint2 en = lds_v2(tab32 + (uint32_t)(c * 8));
          const uint32_t a = ((en.x & maskpk) == en.x) ? gorg + en.y : lutv32;
          nw |= lds_u8(lutv32 + (lds_u8(a) & (uint32_t)d.code_mask)) << (8 * k);
        }
        uint32_t f0, f1, f2;
        if (!init) {
          f0 = *reinterpret_cast<const uint32_t*>(srow + (size_t)((hpos + 1) & 3) * d.ohw_p + c4);
          f1 = *reinterpret_cast<const uint32_t*>(srow + (size_t)((hpos + 2) & 3) * d.ohw_p + c4);
          f2 = *reinterpret_cast<const uint32_t*>(srow + (size_t)((hpos + 3) & 3) * d.ohw_p + c4);
          SNK_CHECK_HIST(hrow + (size_t)hpos * d.ohw_p + c4, 4);
          *reinterpret_cast<uint32_t*>(hrow + (size_t)hpos * d.ohw_p + c4) = nw;
        } else {                                   // reset: every slot holds the first frame (:452-457)
          f0 = f1 = f2 = nw;
#pragma unroll
          for (int f = 0; f < 4; ++f) {
            SNK_CHECK_HIST(hrow + (size_t)f * d.ohw_p + c4, 4);
            *reinterpret_cast<uint32_t*>(hrow + (size_t)f * d.ohw_p + c4) = nw;
          }
        }
        if (want_obs) {
          const uint32_t t0 = __byte_perm(f0, f1, 0x5140), t1 = __byte_perm(f2, nw, 0x5140);
          const uint32_t t2 = __byte_perm(f0, f1, 0x7362), t3 = __byte_perm(f2, nw, 0x7362);
          uint32_t* dst = reinterpret_cast<uint32_t*>(stg) + c4;
          dst[0] = __byte_perm(t0, t1, 0x5410);
          if (c4 + 1 < ohw) dst[1] = __byte_perm(t0, t1, 0x7632);
          if (c4 + 2 < ohw) dst[2] = __byte_perm(t2, t3, 0x5410);
          if (c4 + 3 < ohw) dst[3] = __byte_perm(t2, t3, 0x7632);
        }
      }
    } else {
      if (want_obs && !init) {
#pragma unroll 1
        for (int slot = 0; slot < fs; ++slot) {
          if (slot == hpos) continue;                // about to be overwritten by the new frame
          int f = slot - hpos - 1; if (f < 0) f += fs;
          const uint8_t* src = srow + (size_t)slot * d.ohw_p;
          for (int c4 = (int)lane * 4; c4 < ohw; c4 += 128) {
            const uint32_t w = *reinterpret_cast<const uint32_t*>(src + c4);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (c4 + k < ohw) stg[(size_t)(c4 + k) * fs + f] = (uint8_t)(w >> (8 * k));
          }
        }
      }
      const uint8_t* lut = s_lut + v * LS;
      for (int cell = (int)lane; cell < ohw; cell += 32) {
        const int ci = cell / ow, cj = cell - ci * ow;
        const int rr = r0 + ci, cc = c0 + cj;
        uint32_t code = 0;
        if ((unsigned)rr < (unsigned)H && (unsigned)cc < (unsigned)W) code = cell_code(d, grid[rr * W + cc]);
        const uint8_t bits = lut[code];
        if (!init) {
          if (want_obs) stg[(size_t)cell * fs + (fs - 1)] = bits;
          SNK_CHECK_HIST(hrow + (size_t)hpos * d.ohw_p + cell, 1);
          hrow[(size_t)hpos * d.ohw_p + cell] = bits;
        } else {
          for (int f = 0; f < fs; ++f) {
            if (want_obs) stg[(size_t)cell * fs + f] = bits;
            SNK_CHECK_HIST(hrow + (size_t)f * d.ohw_p + cell, 1);
            hrow[(size_t)f * d.ohw_p + cell] = bits;
          }
        }
      }
    }
  }
  __syncwarp();
  // ---- channel bits as they are (snk_step_bits): the staging area IS the [viewer][cell][frame] block
  if (bits_out) {
    uint8_t* outb = bits_out + (size_t)e * d.stage_env_bytes;
    const int total = d.stage_env_bytes;
    if (((reinterpret_cast<uintptr_t>(outb) | (uintptr_t)total) & 3) == 0) {
      const uint32_t* s4 = reinterpret_cast<const uint32_t*>(s_stage);
      for (int u = (int)lane; u < (total >> 2); u += 32) { SNK_CHECK_BITS(outb + 4 * u, 4); reinterpret_cast<uint32_t*>(outb)[u] = s4[u]; }
    } else {
      for (int u = (int)lane; u < total; u += 32) st_bits(outb + u, s_stage[u]);
    }
  }
  // ---- channel bits -> NHWC uint8, coalesced
  if (want_nhwc) {
    uint8_t* out = p.obs + (size_t)e * d.obs_env_bytes;
    const int total = d.stage_env_bytes;                 // staging bytes == 8-byte output units
    if (vec16) {
      const uint16_t* s2 = reinterpret_cast<const uint16_t*>(s_stage);
      uint4* o4 = reinterpret_cast<uint4*>(out);
#pragma unroll 2
      for (int u = (int)lane; u < (total >> 1); u += 32) {
        const uint32_t two = s2[u];
        uint4 qv;
        qv.x = spread4(two & 15u); qv.y = spread4((two >> 4) & 15u);
        qv.z = spread4((two >> 8) & 15u); qv.w = spread4(two >> 12);
        SNK_CHECK_OBS(o4 + u, 16);
        __stcs(o4 + u, qv);
      }
    } else {
      uint2* o2 = reinterpret_cast<uint2*>(out);
      for (int u = (int)lane; u < total; u += 32) {
        const uint32_t b = s_stage[u];
        SNK_CHECK_OBS(o2 + u, 8);
        __stcs(o2 + u, make_uint2(spread4(b & 15u), spread4(b >> 4)));
      }
    }
  }
  __syncwarp();
}

// ---- global state output (KParams::grid_out): the tile's final grids -> rows e0 .. e0+ne-1 of [N, H*W] -------------
// bulk: compact records with H*W a multiple of 16 (off_c0 == H*W, so the tile's grids are ONE contiguous block, and
// they carry no direction bits) and a 16-byte aligned output: one bulk copy by the tile's elected thread, after the
// rule warp's fence.proxy.async; the issuer waits for its shared-memory reads before the CTA exits or the next step's
// rules run.  Otherwise plain stores of cell codes by the tile's threads (first, step) (full records: stride rec_bytes,
// direction bits masked off).
__device__ __forceinline__ void store_grid_rows(const KParams& p, const TilePtr& tp, int e0, int ne, uint8_t* out,
                                                bool bulk, bool elected, int first, int step) {
  const Dims& d = p.d;
  uint8_t* const rows = out + (size_t)e0 * d.HW;
  if (bulk) {
    if (elected) bulk_store(rows, (uint32_t)__cvta_generic_to_shared(tp.g), (uint32_t)(ne * d.HW));
    return;
  }
  if (((d.HW | (int)reinterpret_cast<uintptr_t>(rows)) & 15) == 0) {
    const uint32_t cm4 = (uint32_t)d.code_mask * 0x01010101u;
    const int n16 = d.HW >> 4;
    for (int k = first; k < ne * n16; k += step) {
      const int q = k / n16;
      uint4 v = reinterpret_cast<const uint4*>(tp.G(q))[k - q * n16];
      v.x &= cm4; v.y &= cm4; v.z &= cm4; v.w &= cm4;
      reinterpret_cast<uint4*>(rows)[k] = v;
    }
  } else {
    for (int k = first; k < ne * d.HW; k += step) {
      const int q = k / d.HW;
      rows[k] = (uint8_t)cell_code(d, tp.G(q)[k - q * d.HW]);
    }
  }
}

// ---- the fused step / reset / encode kernel -------------------------------------------------------
// kCoop = false: every warp owns its own tile (records in a private shared-memory slice), no block
//                barrier after the table copy -- the mode for large batches.
// kCoop = true:  the CTA owns ONE tile; all threads move the records, warp 0 runs the rules, then the
//                warps share the tile's viewers -- for small batches and large records, where one warp per
//                tile leaves the GPU short of parallel work.
// kVar: 0 the plain step (NHWC observation, one step per launch) -- the lean instance every benchmark line runs;
//       1 channel-bit output as well / instead (snk_step_bits); 2 several steps per launch (snk_step_many), any output.
//       The variants only differ in code that is compiled out of variant 0, which keeps its register count.
//       3 the plain step again, compiled without a register cap (88 registers instead of 64): fewer resident warps, more
//         loads in flight per warp -- 2 % faster once the batch is many waves deep (cfg5: 0.756 against 0.772 ms), 3.5 %
//         slower on a 131 072-env shard (profiles/r02_ab_tiles3.txt); the launch picks by batch size (KParams::bigreg).
//         Only while the observation writes are bound by DRAM: into a compressible block (snk_alloc_obs) the capped
//         instance is 11 % faster at cfg5 (0.671 against 0.758 ms, profiles/r03_retune.txt), and the step picks it.
//       4, 5, 6 variants 0, 1, 2 of a handle with a wall-map pool (snk_create_maps, KParams::pool): compact tiles paint
//         each environment's grid from its own map, resets pick the map from next_map.  Handles without a pool run
//         variants 0..3, which hold none of that code.
//       8, 10 (12, 14 with a pool) variants 0 and 2 that also write the global state (KParams::grid_out): 8 / 12 the
//         plain step with or without its NHWC observation, 10 / 14 everything else (channel bits, several steps).  Calls
//         without grid_out run the variants above, which hold none of that code.
//       Specialised shapes (launch_tile_kernel) are built only in the tile modes their defaults select, and those with
//       frame_stack > 1 without variants 2 and 6 (snk_step_many runs one launch per step there); the generic instances
//       have every variant, and serve the calls a forced mode sends past a specialisation.
// Warp-private instances of variants 0, 1, 4, 5, 8 and 12 are capped at 64 registers (eight 128-thread CTAs per SM).
template <int kNS, int kW, int kOH, int kOW, int kFS, bool kCoop, int kEnc, int kVar>
__global__ void __launch_bounds__(kCoop ? SNK_MAX_THREADS_COOP : SNK_MAX_THREADS, (!kCoop && (kVar & 3) <= 1) ? 8 : (!kCoop && kVar == 3) ? 1 : 0)
snk_tile_kernel(const __grid_constant__ KParams p) {
  constexpr bool kPool = (kVar & 4) != 0, kGrid = (kVar & 8) != 0;
  constexpr int kV = kVar & 3;                            // the variant apart from the pool and the global state
  constexpr bool kBits = kV == 1 || kV == 2, kMulti = kV == 2;
  uint8_t* const bits_out = kBits ? p.bits : nullptr;
  extern __shared__ __align__(16) uint8_t smem[];
  const Dims& d = p.d;
  const Shape<kNS, kW, kOH, kOW, kFS> sh(d);
  // Programmatic dependent launch: nothing above touches global memory.  Wait for the grid this one depends on (the
  // previous step; a no-op for an ordinary launch), then let the next step's CTAs be scheduled behind this grid's.
  asm volatile("griddepcontrol.wait;" ::: "memory");
#ifdef SNK_DEBUG_CHECKS
  dbg_arm(p);       // after the wait: the bounds are device globals, and the previous step (maybe of another handle) still runs before it
#endif
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  SNK_T(t_start);
  const int tid = threadIdx.x, nt = blockDim.x;
  const int warp = tid >> 5, nwarps = nt >> 5;
  const uint32_t lane = lane_id();
  const int ns = sh.ns(), G = sh.group(), EPW = p.E;             // environments per tile (<= 32 / G)
  const int fs = sh.fs(), ohw = sh.ohw();
  const int tile = kCoop ? (int)blockIdx.x : (int)blockIdx.x * nwarps + warp;
  const int e0 = tile * EPW;
  const int ne = max(0, min(EPW, d.N - e0));

  // shared memory (mirrored by tile_smem_bytes): tiles' records, per-warp staging (fs > 1), per-tile
  // flags, then the CTA-wide encode tables
  const int rec_tile_bytes = EPW * d.rec_bytes;
  const int tile_bytes = rec_tile_bytes + EPW * d.hist_env_bytes;      // records, then (fs > 1) the frame histories
  const int stage_bytes = fs == 1 ? 0 : round_up(d.stage_env_bytes, 16);
  const int ntiles = kCoop ? 1 : nwarps;
  uint8_t* s_rec = smem + (size_t)(kCoop ? 0 : warp) * tile_bytes;
  uint8_t* s_hist = s_rec + rec_tile_bytes;
  uint8_t* s_stage = smem + (size_t)ntiles * tile_bytes + (size_t)warp * stage_bytes;
  uint8_t* s_flag = smem + (size_t)ntiles * tile_bytes + (size_t)nwarps * stage_bytes + (size_t)(kCoop ? 0 : warp) * TILE_AUX_BYTES;
  uint32_t* s_view = reinterpret_cast<uint32_t*>(s_flag + 48);         // one packed word per (environment, viewer) lane
  uint8_t* s_lut = smem + (size_t)ntiles * tile_bytes + (size_t)nwarps * stage_bytes + (size_t)ntiles * TILE_AUX_BYTES;
  uint8_t* s_pad = s_lut + p.enc_blob_bytes + 16;                       // ENC_PAD: zero-bordered planes of the tile's grids
  // compact handle: [EPW grids (wall layout copies, then rebuilt)][EPW c-parts = the HBM records]; otherwise EPW
  // contiguous working records
  TilePtr tp;
  tp.g = s_rec;
  if (d.compact) { tp.gs = d.off_c0; tp.cs = d.hbm_rec_bytes; tp.vb = s_rec + (size_t)EPW * d.off_c0 - d.off_c0; }
  else { tp.gs = tp.cs = d.rec_bytes; tp.vb = s_rec; }
  uint8_t* const s_c = tp.vb + d.off_c0 - d.hbm_c0;                     // first byte of the tile as it lies in HBM

  // ---- stage the tile's records: HBM -> shared.  One bulk asynchronous copy (TMA) issued by the tile's
  //      elected thread and awaited on an mbarrier, or 128-bit coalesced loads (p.use_tma == 0).
  const bool elected = kCoop ? tid == 0 : lane == 0;
  const int first = kCoop ? tid : (int)lane, step = kCoop ? nt : 32;    // the tile's threads, for strided copies
  const uint32_t rec32 = (uint32_t)__cvta_generic_to_shared(s_c);
  const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(s_flag) + 32u;     // flags: 32 B, mbarrier: 8 B
  const uint32_t tile_load_bytes = (uint32_t)ne * (uint32_t)d.hbm_rec_bytes;
  const uint32_t grid_load_bytes = d.compact ? (uint32_t)ne * (uint32_t)d.off_c0 : 0u;   // wall-layout copies (L2-resident)
  const uint32_t hist_load_bytes = (fs > 1 && p.mode == MODE_STEP) ? (uint32_t)ne * (uint32_t)d.hist_env_bytes : 0u;
  // The encode tables ride on the same barrier when the tile's elected thread can speak for every reader
  // of s_lut (coop CTA, or a single-warp CTA); otherwise the CTA copies them with 128-bit loads below.
  const bool blob_by_tma = p.use_tma && (kCoop || nwarps == 1);
  if (p.use_tma) {
    if (elected) {
      mbar_init(mbar, 1);
      if (ne > 0) {
        mbar_expect_tx(mbar, tile_load_bytes + grid_load_bytes + hist_load_bytes + (blob_by_tma ? (uint32_t)p.enc_copy_bytes : 0u));
        load_records(p, e0, rec32, tile_load_bytes, mbar);
        if (!kPool && grid_load_bytes) bulk_load((uint32_t)__cvta_generic_to_shared(s_rec), p.base_grid, grid_load_bytes, mbar);
        if (hist_load_bytes) bulk_load((uint32_t)__cvta_generic_to_shared(s_hist), p.hist + (size_t)e0 * d.hist_env_bytes, hist_load_bytes, mbar);
        if (blob_by_tma) bulk_load((uint32_t)__cvta_generic_to_shared(s_lut), p.enc_blob, (uint32_t)p.enc_copy_bytes, mbar);
      }
    }
    if constexpr (kPool) {
      // one bulk copy per environment from its own map, issued by the environment's lane of the electing warp once
      // the barrier is armed (the same expect_tx total as the single-layout copy)
      if (grid_load_bytes && (!kCoop || warp == 0)) {
        __syncwarp();
        if ((int)lane < ne) {
          const uint32_t m = checked_map(p.cur_map[e0 + (int)lane], p.num_maps, p.err);
          bulk_load((uint32_t)__cvta_generic_to_shared(s_rec) + lane * (uint32_t)d.off_c0, p.pool + (size_t)m * d.off_c0,
                    (uint32_t)d.off_c0, mbar);
        }
      }
    }
  } else {
    const uint4* src = reinterpret_cast<const uint4*>(p.recs + (size_t)e0 * d.hbm_rec_bytes);
    uint4* dst = reinterpret_cast<uint4*>(s_c);
    const int n16 = ne * (d.hbm_rec_bytes >> 4);
    for (int k = first; k < n16; k += step) dst[k] = __ldcs(src + k);
    const uint4* gsrc = reinterpret_cast<const uint4*>(p.base_grid);
    uint4* gdst = reinterpret_cast<uint4*>(s_rec);
    const int g16 = (int)(grid_load_bytes >> 4);
    if constexpr (kPool) {       // unit k of the tile's grids is unit k % (off_c0 / 16) of environment k / (off_c0 / 16)'s map
      const int u16 = d.off_c0 >> 4;
      for (int k = first; k < g16; k += step) {
        const int q = k / u16;
        const uint32_t m = checked_map(p.cur_map[e0 + q], p.num_maps, p.err);
        gdst[k] = __ldg(reinterpret_cast<const uint4*>(p.pool + (size_t)m * d.off_c0) + (k - q * u16));
      }
    } else {
      for (int k = first; k < g16; k += step) gdst[k] = __ldg(gsrc + k);
    }
    const uint4* hsrc = reinterpret_cast<const uint4*>(p.hist + (size_t)e0 * d.hist_env_bytes);
    uint4* hdst = reinterpret_cast<uint4*>(s_hist);
    const int h16 = (int)(hist_load_bytes >> 4);
    for (int k = first; k < h16; k += step) hdst[k] = __ldcs(hsrc + k);
  }
  // ---- encode tables: host-built blob, L2-resident, copied with 128-bit loads.  fs == 1: {cell code ->
  //      8 output bytes, window-cell table}; fs > 1: {cell code -> channel-bit byte, table}.
  if (!blob_by_tma) {
    const uint4* src = reinterpret_cast<const uint4*>(p.enc_blob);
    uint4* dst = reinterpret_cast<uint4*>(s_lut);
    for (int k = tid; k < (p.enc_copy_bytes >> 4); k += nt) dst[k] = __ldg(src + k);
  }
  // this lane's action (lane = environment lane/G of the tile, snake lane%G), fetched before the waits
  uint32_t action = 0;
  if (p.mode == MODE_STEP && (!kCoop || warp == 0)) {
    const int g = (int)lane / G, i = (int)lane - g * G;
    if (g < ne && i < ns) action = __ldg(p.actions + (size_t)(e0 + g) * ns + i);
  }
  __syncthreads();
  SNK_T(t_issued);
  if (!kCoop && ne == 0) return;
  const bool want_obs = p.obs != nullptr || bits_out != nullptr;          // NHWC bytes, channel bits, or both
  constexpr int kU = Shape<kNS, kW, kOH, kOW, kFS>::kUnits;
  PadCells<kU> pc;
  int pc_shift = -1;
  if (kEnc == ENC_PAD && kCoop && want_obs && ne > 0) {
    // While the records are in flight and warp 0 runs the rules, the other warps clear the padded planes and
    // prepare the window-cell offsets of their first viewer (a single-warp CTA does it all itself).
    const int zw = nwarps > 1 ? 1 : 0;
    if (warp >= zw) {
      uint4* z = reinterpret_cast<uint4*>(s_pad);
      const int n16 = (ne * d.pad_env_bytes) >> 4;
      for (int k = tid - 32 * zw; k < n16; k += nt - 32 * zw) z[k] = make_uint4(0u, 0u, 0u, 0u);
    }
    if (warp != 0 && warp < ne * ns) {
      pc_shift = p.obs ? (int)((reinterpret_cast<uintptr_t>(p.obs + ((size_t)e0 * ns + warp) * (size_t)ohw * 8) >> 3) & 1) : 0;
      pc = make_pad_cells<Shape<kNS, kW, kOH, kOW, kFS>, kU>(sh, pc_shift);
    }
  }
  if (p.use_tma && ne > 0 && !mbar_wait(mbar, 0)) {      // lost transaction: flag it, leave the tile untouched
    if (lane == 0) atomicOr(p.err, ERR_TMA_TIMEOUT);
    return;
  }
  SNK_T(t_loaded);

  const uint32_t lut32 = (uint32_t)__cvta_generic_to_shared(s_lut);
  const uint32_t lutb32 = lut32 + (uint32_t)p.enc_lutb_off;            // fs == 1: byte LUT (channel bits) behind the 8-byte LUT
  const int wfirst = kCoop ? warp : 0, wstep = kCoop ? nwarps : 1;
  // snk_step_many: T > 1 steps of this tile back to back with the records resident in shared memory (frame_stack 1
  // only; T == 1 is the ordinary step).  Step t reads actions[t], writes rewards[t] / dones[t] and, when asked for
  // every step, obs[t]; otherwise only the last step renders.
  const int T = (kMulti && fs == 1 && p.mode == MODE_STEP) ? p.T : 1;
  CellWords cw;
  bool cw_ready = false;
  const bool grid_bulk = kGrid && p.use_tma && d.compact && (d.HW & 15) == 0 && (reinterpret_cast<uintptr_t>(p.grid_out) & 15) == 0;
#pragma unroll 1
  for (int t = 0; t < T; ++t) {
  const bool last = t == T - 1;
  // this step's global state rows (every step of a multi-step launch, or only the last one, as the observation)
  uint8_t* const grid_t = (kGrid && p.grid_out && (last || (kMulti && p.obs_every_step)))
                              ? p.grid_out + ((kMulti && p.obs_every_step) ? (size_t)t * d.N * d.HW : 0) : nullptr;
  if (!kCoop || warp == 0) {
    if (t > 0) {
      const int g = (int)lane / G, i = (int)lane - g * G;
      action = (g < ne && i < ns) ? __ldg(p.actions + ((size_t)t * d.N + e0 + g) * ns + i) : 0u;
    }
    if (d.compact && t == 0 && ne > 0) expand_tile(p, sh, tp, ne);
    if (ne > 0) tile_rules<kPool>(p, sh, tp, e0, ne, s_flag, action, t);
    if (kEnc == ENC_REG && ne > 0) {           // crop origin + out-of-grid rows / columns of every viewer of the tile
      const int g = (int)lane / G, i = (int)lane - g * G;
      if (g < ne && i < ns) s_view[lane] = make_viewer_word(p, sh, tp.VB(g), i);
    }
    if (kEnc == ENC_PAD && ne > 0) {           // crop origin of every viewer inside its padded plane
      const int g = (int)lane / G, i = (int)lane - g * G;
      if (g < ne && i < ns) {
        int r0, c0;
        viewer_origin(d, tp.VB(g), ns, sh.W(), d.V, i, r0, c0);
        s_view[lane] = (uint32_t)((r0 + d.V) * sh.pad_pitch() + c0 + sh.pad_left());
      }
    }
    if (p.use_tma && (last || (kGrid && grid_t))) fence_proxy_async();   // the rules' shared-memory writes -> visible to the bulk stores
    __syncwarp();
  }
  SNK_T(t_ruled);
  if (kCoop) __syncthreads();
  SNK_T(t_synced);
  if (ne == 0) return;
  if constexpr (kGrid) {
    if (grid_t) store_grid_rows(p, tp, e0, ne, grid_t, grid_bulk, elected, first, step);
  }

  if (fs == 1) {
    // ---- write the records back: shared -> HBM (nothing below modifies them).  The bulk store runs
    //      asynchronously under the encode; its issuer waits for the shared-memory reads before exiting.
    if (last) store_records(p, e0, ne, s_c, rec32, tile_load_bytes, elected, false, first, step);
    // this step's observation block (every step of a multi-step launch, or only the last one)
    const bool render = want_obs && (last || (kMulti && p.obs_every_step));
    uint8_t* const obs_t = (p.obs && render) ? p.obs + ((kMulti && p.obs_every_step) ? (size_t)t * d.N * d.obs_env_bytes : 0) : nullptr;
    uint8_t* const bits_t = (kBits && bits_out && render) ? bits_out + (p.obs_every_step ? (size_t)t * d.N * d.stage_env_bytes : 0) : nullptr;
    if (kEnc == ENC_PAD) {
      if (kCoop && render) {
        // ---- grid interiors -> padded planes (whole CTA, flat over the tile's grid words), then the viewers
        const int W = sh.W(), wpr = W >> 2, nw = d.H * wpr, P4 = sh.pad_pitch() >> 2;
        const uint32_t cm4 = (uint32_t)d.code_mask * 0x01010101u;
        const bool may_skip = p.mode != MODE_STEP;
        for (int idx = tid; idx < ne * nw; idx += nt) {
          const int q = (int)__umulhi((uint32_t)idx, (uint32_t)p.inv_grid_words);
          const int j = idx - q * nw;
          const int rr = kW ? j / wpr : (int)__umulhi((uint32_t)j, (uint32_t)p.inv_row_words);
          const uint32_t w = reinterpret_cast<const uint32_t*>(tp.G(q))[j];
          uint32_t* dst = reinterpret_cast<uint32_t*>(s_pad + (size_t)q * d.pad_env_bytes + d.V * sh.pad_pitch() + sh.pad_left());
          dst[rr * P4 + (j - rr * wpr)] = w & cm4;
        }
        __syncthreads();
        const int nv = ne * ns;
        const size_t vbytes = (size_t)ohw * 8;
        uint8_t* out_tile = obs_t ? obs_t + (size_t)e0 * ns * vbytes : nullptr;
        uint8_t* bits_tile = bits_t ? bits_t + (size_t)e0 * ns * ohw : nullptr;
        const uint32_t pad32 = (uint32_t)__cvta_generic_to_shared(s_pad);
        int q = wfirst / ns, v = wfirst - q * ns;
#pragma unroll 1
        for (int pv = wfirst; pv < nv; pv += wstep) {
          if (!(may_skip && (s_flag[q] & F_SKIP))) {
            uint8_t* outv = out_tile ? out_tile + (size_t)pv * vbytes : nullptr;
            const int shift = (int)((reinterpret_cast<uintptr_t>(outv) >> 3) & 1);
            if (shift != pc_shift) { pc = make_pad_cells<Shape<kNS, kW, kOH, kOW, kFS>, kU>(sh, shift); pc_shift = shift; }
            encode_viewer_pad<Shape<kNS, kW, kOH, kOW, kFS>, kU>(p, sh, pad32 + (uint32_t)(q * d.pad_env_bytes) + s_view[q * G + v],
                                                                 pc, shift, v, outv, lut32,
                                                                 bits_tile ? bits_tile + (size_t)pv * ohw : nullptr, lutb32);
          }
          v += wstep;
          while (v >= ns) { v -= ns; ++q; }
        }
      }
    } else if (render) {
      // viewer pairs (encode_env_pairs): warp-private ENC_REG tiles writing NHWC bytes only, odd window, even
      // viewer count, 16-byte aligned environment blocks
      constexpr bool kPairable = kEnc == ENC_REG && !kCoop && !(kV == 1) && (kOH * kOW == 0 || ((kOH * kOW) & 1)) &&
                                 (kNS == 0 || (kNS & 1) == 0);
      const bool pairs = kPairable && obs_t && !bits_t && p.vec16 && (ohw & 1) && (ns & 1) == 0;
      if (kEnc == ENC_REG && !cw_ready) { cw = pairs ? make_pair_cell_words(sh) : make_cell_words(sh, sh.view_bits()); cw_ready = true; }
      if (kPairable && pairs) {
        const uint32_t view32 = (uint32_t)__cvta_generic_to_shared(s_view);
        uint8_t* const outl = obs_t + (size_t)e0 * d.obs_env_bytes + 16 * lane;
        if (d.code_mask == 0xff) {
#pragma unroll 1
          for (int q = 0; q < ne; ++q) {
            if (s_flag[q] & F_SKIP) continue;
            encode_env_pairs<Shape<kNS, kW, kOH, kOW, kFS>, false>(p, sh, (uint32_t)__cvta_generic_to_shared(tp.G(q)),
                                                                   view32 + 4u * (uint32_t)(q * G), cw,
                                                                   outl + (size_t)q * d.obs_env_bytes, lut32);
          }
        } else {
#pragma unroll 1
          for (int q = 0; q < ne; ++q) {
            if (s_flag[q] & F_SKIP) continue;
            encode_env_pairs<Shape<kNS, kW, kOH, kOW, kFS>, true>(p, sh, (uint32_t)__cvta_generic_to_shared(tp.G(q)),
                                                                  view32 + 4u * (uint32_t)(q * G), cw,
                                                                  outl + (size_t)q * d.obs_env_bytes, lut32);
          }
        }
      } else if (kCoop) {
#pragma unroll 1
        for (int pv = wfirst; pv < ne * ns; pv += wstep) {
          const int q = pv / ns, v = pv - q * ns;
          if (s_flag[q] & F_SKIP) continue;
          const uint8_t* base = tp.G(q);
          const uint32_t grid32 = (uint32_t)__cvta_generic_to_shared(base);
          uint8_t* outv = obs_t ? obs_t + ((size_t)(e0 + q) * ns + v) * (size_t)ohw * 8 : nullptr;
          uint8_t* bitsv = bits_t ? bits_t + ((size_t)(e0 + q) * ns + v) * (size_t)ohw : nullptr;
          encode_viewer<kEnc>(p, sh, base, tp.VB(q), grid32, s_view[q * G + v], cw, v, outv, lut32, bitsv, lutb32);
        }
      } else {
#pragma unroll 1
        for (int q = 0; q < ne; ++q) {
          if (s_flag[q] & F_SKIP) continue;
          const uint8_t* base = tp.G(q);
          const uint32_t grid32 = (uint32_t)__cvta_generic_to_shared(base);
          uint8_t* outq = obs_t ? obs_t + (size_t)(e0 + q) * ns * (size_t)ohw * 8 : nullptr;
          uint8_t* bitsq = bits_t ? bits_t + (size_t)(e0 + q) * ns * (size_t)ohw : nullptr;
#pragma unroll 1
          for (int v = 0; v < ns; ++v) {
            uint8_t* outv = outq ? outq + (size_t)v * ohw * 8 : nullptr;
            uint8_t* bitsv = bitsq ? bitsq + (size_t)v * ohw : nullptr;
            encode_viewer<kEnc>(p, sh, base, tp.VB(q), grid32, s_view[q * G + v], cw, v, outv, lut32, bitsv, lutb32);
          }
        }
      }
    }
    if (!last) {                                // the next step's rules rewrite the records and viewer words
      if constexpr (kGrid) {                    // ... and the grids: this step's bulk store must have read them
        if (grid_bulk && grid_t && elected) bulk_store_wait_read();
      }
      if (kCoop) __syncthreads(); else __syncwarp();
      continue;
    }
    SNK_T(t_encoded);
    if (p.use_tma && elected) bulk_store_wait_read();
    SNK_T(t_end);
#ifdef SNK_PHASE_TIMING
    if (lane == 0 && warp < 8 && snk_trace_buf) {
      unsigned long long* tr = snk_trace_buf + ((size_t)blockIdx.x * 8 + warp) * 8;
      unsigned smid; asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
      tr[0] = t_start; tr[1] = t_issued; tr[2] = t_loaded; tr[3] = t_ruled; tr[4] = t_synced; tr[5] = t_encoded; tr[6] = t_end; tr[7] = smid;
    }
#endif
    return;
  }
  }   // step loop (frame_stack > 1 runs it once and continues below)

  // ---- frame_stack > 1
#pragma unroll 1
  for (int q = wfirst; q < ne; q += wstep) {
    const int qflag = s_flag[q];
    if (qflag & F_SKIP) continue;
    encode_env_stacked<Shape<kNS, kW, kOH, kOW, kFS>, kFS, kBits>(p, sh, tp.G(q), tp.VB(q), e0 + q, qflag,
                                                           s_stage, lut32, s_lut, s_hist + (size_t)q * d.hist_env_bytes);
  }
  if (kCoop) __syncthreads(); else __syncwarp();
  if (!kCoop || warp == 0) {
    if ((int)lane < ne && !(s_flag[lane] & F_SKIP)) {
      EnvHdr* h = (EnvHdr*)(tp.VB((int)lane) + d.off_hdr);
      h->hpos = (uint8_t)((s_flag[lane] & (F_RESET | F_INIT)) ? 0u : ((uint32_t)h->hpos + 1u) % (uint32_t)fs);
    }
  }
  if (p.use_tma && (!kCoop || warp == 0)) fence_proxy_async();        // hpos updates -> async proxy
  if (kCoop) __syncthreads(); else __syncwarp();
  // ---- write the records back: shared -> HBM
  store_records(p, e0, ne, s_c, rec32, tile_load_bytes, elected, true, first, step);
}

// ---- state export / import (parity + checkpoint interface; thread per environment) ----------------
// Compact handles keep no grid in HBM: `base_grid` (or, with a wall-map pool, the pool slot of the environment's cur_map)
// is the wall layout, the caller's array receives the rebuilt grid (walls + fruit slots + live bodies walked from the
// tail).  r.grid is never dereferenced for them.
__device__ __forceinline__ const uint8_t* env_walls(const Dims& d, const uint8_t* base_grid, const MapView& mv, int e,
                                                    uint32_t* err) {
  if (!mv.pool) return base_grid;
  const uint32_t m = checked_map(mv.map_ids[e], mv.num_maps, err);
  if (mv.cur_out) mv.cur_out[e] = (uint8_t)m;
  return mv.pool + (size_t)m * d.off_c0;
}

__global__ void snk_get_state_kernel(const Dims d, const uint8_t* __restrict__ recs, const uint8_t* __restrict__ base_grid,
                                     const MapView mv, uint32_t* err, StateView sv) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= d.N) return;
  base_grid = env_walls(d, base_grid, mv, e, err);
  uint8_t* hb = const_cast<uint8_t*>(recs) + (size_t)e * d.hbm_rec_bytes;
  Rec r = rec_view2(hb, hb + d.hbm_c0, d);
  if (sv.grid && !d.compact) for (int c = 0; c < d.HW; ++c) sv.grid[(size_t)e * d.HW + c] = (uint8_t)cell_code(d, r.grid[c]);
  if (sv.grid && d.compact) {
    uint8_t* out = sv.grid + (size_t)e * d.HW;
    for (int c = 0; c < d.HW; ++c) out[c] = base_grid[c];
    for (int j = 0; j < d.fcap; ++j) if (r.fruit[j]) out[r.fruit[j] - 1] = (uint8_t)FRUIT;
    for (int i = 0; i < d.ns; ++i) {
      if (!r.alive[i]) continue;
      int c = r.tail[i];
      uint8_t code = (uint8_t)(TAIL + 10 * i);
      for (int guard = 0; guard < d.HW && c != r.head[i]; ++guard) {
        out[c] = code; code = (uint8_t)(BODY + 10 * i);
        c += dir_delta(dirp_get(r.dirp, c), d.W);
      }
      out[r.head[i]] = (uint8_t)(HEAD + 10 * i);
    }
  }
  if (sv.alive_counter) sv.alive_counter[e] = r.hdr->alive_counter;
  if (sv.episode_length) sv.episode_length[e] = (int32_t)r.hdr->episode_length;
  for (int i = 0; i < d.ns; ++i) {
    const size_t o = (size_t)e * d.ns + i;
    const bool al = r.alive[i] != 0;
    if (sv.head) sv.head[o] = al ? r.head[i] : -1;
    if (sv.tail) sv.tail[o] = al ? r.tail[i] : -1;
    if (sv.length) sv.length[o] = al ? r.len[i] : 0;
    if (sv.dir) sv.dir[o] = r.dir[i];
    if (sv.alive) sv.alive[o] = r.alive[i];
    if (sv.cells) {
      int32_t* cl = sv.cells + o * sv.max_cells;
      for (int k = 0; k < sv.max_cells; ++k) cl[k] = -1;
      if (al) {
        int c = r.tail[i];
        for (int k = (int)r.len[i] - 1; k >= 0; --k) {
          if (k < sv.max_cells) cl[k] = c;
          c += dir_delta(body_dir(d, r, c), d.W);
        }
      }
    }
  }
}

__global__ void snk_set_state_kernel(const Dims d, uint8_t* __restrict__ recs, const uint8_t* __restrict__ base_grid,
                                     const MapView mv, uint32_t* __restrict__ err, StateView sv) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= d.N) return;
  base_grid = env_walls(d, base_grid, mv, e, err);      // set_state starts an episode on next_map, as a reset does
  uint8_t* hb = recs + (size_t)e * d.hbm_rec_bytes;
  Rec r = rec_view2(hb, hb + d.hbm_c0, d);
  if (!d.compact) for (int c = 0; c < d.HW; ++c) r.grid[c] = sv.grid[(size_t)e * d.HW + c];
  if (!d.compact && mv.pool) {
    // a wall-map pool names the layout of every episode (cur_map): the grid's walls must be exactly that map's
    bool bad = false;
    for (int c = 0; c < d.HW; ++c) bad |= (sv.grid[(size_t)e * d.HW + c] == (uint8_t)WALL) != (base_grid[c] == (uint8_t)WALL);
    if (bad) atomicOr(err, ERR_STATE);
  }
  if (d.compact) {
    // the record stores the fruit cells and the bodies; whatever else the caller's grid holds must be what they imply
    const uint8_t* in = sv.grid + (size_t)e * d.HW;
    int nf = 0;
    bool bad = false;
    for (int j = 0; j < d.fcap; ++j) r.fruit[j] = 0;
    for (int c = 0; c < d.HW; ++c) {
      const uint32_t code = in[c], kind = code % 10u;
      if (code == (uint32_t)FRUIT) { if (nf < d.fcap) r.fruit[nf] = (uint16_t)(c + 1); ++nf; }
      else if (kind < (uint32_t)HEAD) bad |= code != base_grid[c];                 // EMPTY / WALL: the handle's layout
    }
    bad |= nf > d.fcap;
    for (int i = 0; i < d.ns && !bad; ++i) {                                      // every live body cell carries its code
      const size_t o = (size_t)e * d.ns + i;
      const int len = sv.alive[o] ? sv.length[o] : 0;
      for (int k = 0; k < len; ++k) {
        const int c = sv.cells[o * sv.max_cells + k];
        bad |= (unsigned)c >= (unsigned)d.HW || in[c] != (k == 0 ? HEAD : k == len - 1 ? TAIL : BODY) + 10 * i;
      }
    }
    int body = 0, want = 0;
    for (int c = 0; c < d.HW; ++c) body += (in[c] % 10u) >= (uint32_t)HEAD;
    for (int i = 0; i < d.ns; ++i) want += sv.alive[(size_t)e * d.ns + i] ? sv.length[(size_t)e * d.ns + i] : 0;
    bad |= body != want;                                                          // no stray body cells either
    if (bad) atomicOr(err, ERR_STATE);
  }
  for (int i = 0; i < d.ns; ++i) {
    const size_t o = (size_t)e * d.ns + i;
    const int32_t* cl = sv.cells + o * sv.max_cells;
    const int len = sv.length[o];
    r.alive[i] = sv.alive[o];
    r.dir[i] = sv.dir[o];
    r.len[i] = (uint16_t)(sv.alive[o] ? len : 0);
    r.head[i] = 0; r.tail[i] = 0;
    if (sv.alive[o] && len > 0) {
      r.head[i] = (uint16_t)cl[0];
      r.tail[i] = (uint16_t)cl[len - 1];
      for (int k = 1; k < len; ++k) {
        const int diff = cl[k - 1] - cl[k];
        const int dd = diff == -d.W ? 0 : diff == 1 ? 1 : diff == d.W ? 2 : 3;
        set_body_dir(d, r, cl[k], dd);
      }
    }
    stats_zero(d, r, i);
  }
  r.hdr->alive_counter = (int16_t)sv.alive_counter[e];
  r.hdr->episode_length = (uint32_t)sv.episode_length[e];
  r.hdr->hpos = 0;
}

// ---- observation bytes -> channel-bit bytes (packed host transport, device replay buffers) ----------
// Eight consecutive observation bytes are the 0/1 channels of one (cell, frame); a 32-bit multiply gathers
// four of them into a nibble (bit c = byte c, no cross-term collisions for 0/1 bytes).
__device__ __forceinline__ uint32_t pack_unit(uint32_t lo, uint32_t hi) {
  return ((lo * 0x01020408u) >> 24) | (((hi * 0x01020408u) >> 24) << 4);
}
__global__ void __launch_bounds__(256) snk_pack_obs_kernel(const uint8_t* __restrict__ obs, uint8_t* __restrict__ bits,
                                                           size_t n_units) {
  const size_t n4 = n_units >> 2;                      // four units (32 input bytes) per thread
  const uint4* in = reinterpret_cast<const uint4*>(obs);
  uint32_t* out = reinterpret_cast<uint32_t*>(bits);
  const size_t stride = (size_t)gridDim.x * blockDim.x, t0 = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  for (size_t i = t0; i < n4; i += stride) {
    const uint4 a = __ldcs(in + 2 * i), b = __ldcs(in + 2 * i + 1);
    out[i] = pack_unit(a.x, a.y) | (pack_unit(a.z, a.w) << 8) | (pack_unit(b.x, b.y) << 16) | (pack_unit(b.z, b.w) << 24);
  }
  for (size_t u = (n4 << 2) + t0; u < n_units; u += stride) {
    const uint2 a = *reinterpret_cast<const uint2*>(obs + 8 * u);
    bits[u] = (uint8_t)pack_unit(a.x, a.y);
  }
}

__global__ void snk_init_records_kernel(const Dims d, uint8_t* __restrict__ recs) {
  const size_t n = (size_t)d.N * d.hbm_rec_bytes / 16;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    reinterpret_cast<uint4*>(recs)[i] = make_uint4(0, 0, 0, 0);
}

// ---- snapshot / restore: slots of SnapHdr + record + history, moved as 16-byte units, one per thread ----------------
// Unit j of a slot: 0 the header, 1 .. ru the record, then the history.  I is the index type: 32-bit while every unit
// index of the launch fits it (the division by the slot's unit count is the costly part of the address arithmetic).
template <class I>
__global__ void __launch_bounds__(256) snk_snapshot_kernel(const Dims d, const uint8_t* __restrict__ recs,
                                                           const uint8_t* __restrict__ hist, const uint8_t* __restrict__ cur_map,
                                                           const int32_t* __restrict__ ids, int count, uint64_t digest,
                                                           uint8_t* __restrict__ snap, uint32_t* err) {
  const I ru = (I)(d.hbm_rec_bytes >> 4), hu = (I)(d.hist_env_bytes >> 4), su = 1 + ru + hu;
  const I n = (I)count * su;
  const uint4* rec4 = reinterpret_cast<const uint4*>(recs);
  const uint4* hist4 = reinterpret_cast<const uint4*>(hist);
  uint4* out = reinterpret_cast<uint4*>(snap);
  for (I k = (I)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (I)gridDim.x * blockDim.x) {
    const I i = k / su, j = k - i * su;
    const int e = ids ? __ldg(ids + i) : (int)i;
    const bool ok = (unsigned)e < (unsigned)d.N;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (j == 0) {
      if (ok) { v.x = (uint32_t)digest; v.y = (uint32_t)(digest >> 32); v.z = cur_map ? cur_map[e] : 0u; }
      else atomicOr(err, ERR_SNAPSHOT);                 // digest 0: the slot matches no handle
    } else if (ok) {
      v = j <= ru ? __ldg(rec4 + (I)e * ru + (j - 1)) : __ldg(hist4 + (I)e * hu + (j - 1 - ru));
    }
    __stcs(out + k, v);
  }
}

// Indexed by destination: env e takes slot src[e] (-1 keeps it), so no two slots race for one env and one slot may
// fan out to any number of envs.  mask[e] ends 1 where env e was restored, 0 otherwise.
template <class I>
__global__ void __launch_bounds__(256) snk_restore_kernel(const Dims d, uint8_t* __restrict__ recs, uint8_t* __restrict__ hist,
                                                          uint8_t* __restrict__ cur_map, const int32_t* __restrict__ src,
                                                          int num_slots, const uint8_t* __restrict__ snap, uint64_t digest,
                                                          uint8_t* __restrict__ mask, uint32_t* err) {
  const I ru = (I)(d.hbm_rec_bytes >> 4), hu = (I)(d.hist_env_bytes >> 4), su = 1 + ru + hu;
  const I n = (I)d.N * su;
  uint4* rec4 = reinterpret_cast<uint4*>(recs);
  uint4* hist4 = reinterpret_cast<uint4*>(hist);
  const uint4* in = reinterpret_cast<const uint4*>(snap);
  for (I k = (I)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (I)gridDim.x * blockDim.x) {
    const I e = k / su, j = k - e * su;
    const int s = __ldg(src + e);
    if (s == -1) {
      if (j == 0) mask[e] = 0;
      continue;
    }
    bool ok = s >= 0 && s < num_slots;
    const uint4* slot = in + (I)(ok ? s : 0) * su;
    uint4 h = make_uint4(0u, 0u, 0u, 0u);
    if (ok) {
      h = __ldg(slot);                                  // every unit's thread checks the header it shares (one line)
      ok = h.x == (uint32_t)digest && h.y == (uint32_t)(digest >> 32);
    }
    if (!ok) {
      if (j == 0) { mask[e] = 0; atomicOr(err, ERR_SNAPSHOT); }
      continue;
    }
    if (j == 0) {
      mask[e] = 1;
      if (cur_map) cur_map[e] = (uint8_t)h.z;
    } else if (j <= ru) {
      rec4[e * ru + (j - 1)] = __ldg(slot + j);
    } else {
      hist4[e * hu + (j - 1 - ru)] = __ldg(slot + j);
    }
  }
}

// frame_stack > 1 after a restore: one warp per env with mask[e] != 0.  The observation is the env's history ring
// widened in ring order (oldest frame at hpos, the newest -- the current frame -- last), i.e. the bytes the step that
// wrote the newest frame returned; the tile kernel's encode cannot serve here, as its F_INIT refills every frame.  The
// grid row is rebuilt as snk_get_state_kernel does (walls of cur_map, fruit slots, bodies from the tail).
__global__ void __launch_bounds__(256) snk_emit_stacked_kernel(const Dims d, const uint8_t* __restrict__ recs,
                                                               const uint8_t* __restrict__ hist,
                                                               const uint8_t* __restrict__ base_grid, const MapView mv,
                                                               const uint8_t* __restrict__ mask, uint8_t* __restrict__ obs,
                                                               uint8_t* __restrict__ bits, uint8_t* __restrict__ grid,
                                                               uint32_t* err) {
  const int e = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
  if (e >= d.N || !mask[e]) return;                     // the whole warp leaves together
  const int lane = (int)lane_id();
  uint8_t* hb = const_cast<uint8_t*>(recs) + (size_t)e * d.hbm_rec_bytes;
  const Rec r = rec_view2(hb, hb + d.hbm_c0, d);
  if (obs || bits) {
    const int fs = d.fs, hpos = r.hdr->hpos, per_v = d.ohw * fs;
    const uint8_t* he = hist + (size_t)e * d.hist_env_bytes;
    uint8_t* be = bits ? bits + (size_t)e * d.stage_env_bytes : nullptr;
    uint2* oe = obs ? reinterpret_cast<uint2*>(obs + (size_t)e * d.obs_env_bytes) : nullptr;
    for (int u = lane; u < d.stage_env_bytes; u += 32) {        // u = (viewer, cell, frame), the staging order
      const int v = u / per_v, rem = u - v * per_v, cell = rem / fs, f = rem - cell * fs;
      int slot = hpos + f;
      if (slot >= fs) slot -= fs;
      const uint32_t b = he[(size_t)(v * fs + slot) * d.ohw_p + cell];
      if (be) be[u] = (uint8_t)b;
      if (oe) __stcs(oe + u, make_uint2(spread4(b & 15u), spread4(b >> 4)));
    }
  }
  if (!grid) return;
  uint8_t* out = grid + (size_t)e * d.HW;
  if (!d.compact) {
    for (int c = lane; c < d.HW; c += 32) out[c] = (uint8_t)cell_code(d, r.grid[c]);
    return;
  }
  const uint8_t* walls = env_walls(d, base_grid, mv, e, err);
  for (int c = lane; c < d.HW; c += 32) out[c] = walls[c];
  __syncwarp();
  for (int j = lane; j < d.fcap; j += 32)
    if (r.fruit[j]) out[r.fruit[j] - 1] = (uint8_t)FRUIT;
  __syncwarp();
  if (lane < d.ns && r.alive[lane]) {
    const int i = lane;
    int c = r.tail[i];
    uint8_t code = (uint8_t)(TAIL + 10 * i);
    for (int guard = 0; guard < d.HW && c != r.head[i]; ++guard) {
      out[c] = code; code = (uint8_t)(BODY + 10 * i);
      c += dir_delta(dirp_get(r.dirp, c), d.W);
    }
    out[r.head[i]] = (uint8_t)(HEAD + 10 * i);
  }
}

// ---- launch wrappers -----------------------------------------------------------------------------
int tile_group(int ns) { return ns <= 1 ? 1 : ns <= 2 ? 2 : ns <= 4 ? 4 : ns <= 8 ? 8 : ns <= 16 ? 16 : 32; }

bool encode_uses_table(const Dims& d) {
  return (d.V == 0 || (d.oh <= 16 && d.ow <= 16)) && (size_t)(d.ohw + 2) * 8 <= 16 * 1024;
}
// fs == 1 with many snakes: one {as-other, as-own} LUT pair instead of one LUT per viewer
bool encode_lut_dual(const Dims& d) {
  return d.fs == 1 && encode_uses_table(d) && (size_t)d.ns * (10 * d.ns + 6) * 8 > 8 * 1024;
}

// Encode blob: LUT over cell codes, then (optionally) uint2 tab[-1 .. ohw] per window cell.
//   fs == 1: uint2 (8 output bytes) per code, per viewer -- or {as-other, as-own} when encode_lut_dual
//   fs  > 1: one channel-bit byte per code, per viewer
size_t encode_blob_bytes(const Dims& d, size_t* tab_off, size_t* lutb_off) {
  const int LS = 10 * d.ns + 6;
  const int nl = encode_lut_dual(d) ? 2 : d.ns;
  size_t lut = (size_t)round_up(d.fs == 1 ? nl * LS * 8 : d.ns * LS, 16);
  if (lutb_off) *lutb_off = d.fs == 1 ? lut : 0;
  if (d.fs == 1) lut += (size_t)round_up(nl * LS, 16);          // channel-bit byte per code, same indexing
  if (tab_off) *tab_off = lut;
  return (size_t)round_up((int)(lut + (encode_uses_table(d) ? (size_t)(d.ohw + 2) * 8 : 0)), 16);
}

void encode_blob_fill(const Dims& d, uint8_t* out) {
  const int LS = 10 * d.ns + 6;
  uint32_t* w = reinterpret_cast<uint32_t*>(out);
  size_t off, lutb;
  encode_blob_bytes(d, &off, &lutb);
  uint8_t* wb = out + lutb;                                       // fs == 1: the byte LUT
  auto put_fs1 = [&](int k, uint32_t bits) {                      // fs == 1 entry k: 8 output bytes and the bits byte
    w[2 * k] = spread4(bits & 15u);
    w[2 * k + 1] = spread4(bits >> 4);
    wb[k] = (uint8_t)bits;
  };
  if (encode_lut_dual(d)) {
    for (int own = 0; own < 2; ++own)
      for (int code = 0; code < LS; ++code) {
        // viewer = owner of the code for the as-own half, some other snake for the as-other half
        const uint32_t owner = (uint32_t)code / 10u;
        put_fs1(own * LS + code, cell_bits((uint32_t)code, own ? owner : owner + 1u));
      }
  } else {
    for (int v = 0; v < d.ns; ++v)
      for (int code = 0; code < LS; ++code) {
        const uint32_t bits = cell_bits((uint32_t)code, (uint32_t)v);
        if (d.fs == 1) put_fs1(v * LS + code, bits);
        else out[v * LS + code] = (uint8_t)bits;
      }
  }
  if (!encode_uses_table(d)) return;
  uint32_t* t = reinterpret_cast<uint32_t*>(out + off);
  for (int c = -1; c <= d.ohw; ++c) {
    uint32_t bits = 0xFFFFFFFFu, goff = 0;            // out-of-window sentinels never validate
    if (c >= 0 && c < d.ohw) {
      const int ci = c / d.ow, cj = c % d.ow;
      bits = d.V > 0 ? ((1u << ci) | (1u << (16 + cj))) : 0u;
      goff = (uint32_t)(ci * d.W + cj);
    }
    t[2 * (c + 1)] = bits;
    t[2 * (c + 1) + 1] = goff;
  }
}

// Which frame_stack-1 encode a configuration runs (see ENC_* in snk_kernels.h).
static int bits_for(int max_value) { int b = 0; while ((1 << b) <= max_value) ++b; return b; }
int encode_flavour(const Dims& d, bool coop) {
  if (d.fs != 1) return ENC_LEGACY;
  const bool dual = encode_lut_dual(d);
  if (d.V == 0) return dual ? ENC_LEGACY : ENC_DIRECT;
  const int B = d.oh + d.ow;
  if (!dual && d.ohw <= 127 && B + bits_for((d.oh - 1) * d.W + d.ow - 1) <= 31 && B + bits_for(d.HW - 1) <= 32) return ENC_REG;
  // windows of 128..255 cells or many snakes, cooperative tiles: the padded-plane encode (measured on cfg4: the
  // table-driven encode saturates the shared-memory pipe at 79 %, this one runs it at 59 % with 15 % fewer instructions)
  if (coop && d.ohw <= 255 && (d.W & 3) == 0 && d.W >= 8) return ENC_PAD;
  return ENC_LEGACY;
}

size_t pad_plane_bytes(const Dims& d, int tile_envs) { return (size_t)tile_envs * (size_t)d.pad_env_bytes; }

// Shared memory of one CTA of `warps` warps (must mirror the carve-up in snk_tile_kernel).
size_t tile_smem_bytes(const Dims& d, int warps, bool coop, int EPW) {
  const size_t ntiles = coop ? 1 : (size_t)warps;
  size_t b = ntiles * (size_t)EPW * ((size_t)d.rec_bytes + (size_t)d.hist_env_bytes);
  if (d.fs > 1) b += (size_t)warps * (size_t)round_up(d.stage_env_bytes, 16);
  b += ntiles * TILE_AUX_BYTES;
  b += encode_blob_bytes(d, nullptr, nullptr) + 16;
  if (encode_flavour(d, coop) == ENC_PAD) b += pad_plane_bytes(d, EPW);
  return b;
}

template <int kNS, int kW, int kOH, int kOW, int kFS, bool kCoop, int kEnc, int kVar>
static cudaError_t launch_variant(const KParams& p, int threads, size_t smem_bytes, cudaStream_t stream) {
  // dynamic shared memory opt-in, once per (instance, device) and size: function attributes belong to the device's
  // context.  (Process-wide on purpose: the attribute is a property of the kernel, not of a handle; concurrent first
  // launches from two threads set the same or a larger value, which is harmless; the table itself is atomic.)
  static std::atomic<size_t> configured[64];
  auto kern = snk_tile_kernel<kNS, kW, kOH, kOW, kFS, kCoop, kEnc, kVar>;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= 64 || smem_bytes > configured[dev].load(std::memory_order_acquire)) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) {          // keep the maximum: a concurrent first launch may have stored a larger size
      size_t seen = configured[dev].load(std::memory_order_relaxed);
      while (seen < smem_bytes && !configured[dev].compare_exchange_weak(seen, smem_bytes, std::memory_order_release)) {}
    }
  }
  const int envs_per_cta = (kCoop ? 1 : threads / 32) * p.E;
  const int grid = (p.d.N + envs_per_cta - 1) / envs_per_cta;
  // Programmatic dependent launch: when the previous kernel on the stream is another step of this library, this
  // launch's CTAs are scheduled while that grid drains and park at griddepcontrol.wait -- the launch latency between
  // two steps disappears from the step time (the grids' memory operations stay ordered by the wait).
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)threads);
  cfg.dynamicSmemBytes = smem_bytes; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = p.pdl ? 1u : 0u;
  return cudaLaunchKernelEx(&cfg, kern, p);
}

template <int kNS, int kW, int kOH, int kOW, int kFS, bool kCoop, int kEnc>
static cudaError_t launch_instance(const KParams& p, int threads, size_t smem_bytes, cudaStream_t stream) {
  if (p.grid_out) {             // global state: variants 8 / 10, with a pool 12 / 14 (no uncapped copy like variant 3)
    const bool general = p.T > 1 || p.bits;
    if (p.pool) return general ? launch_variant<kNS, kW, kOH, kOW, kFS, kCoop, kEnc, 14>(p, threads, smem_bytes, stream)
                               : launch_variant<kNS, kW, kOH, kOW, kFS, kCoop, kEnc, 12>(p, threads, smem_bytes, stream);
    return general ? launch_variant<kNS, kW, kOH, kOW, kFS, kCoop, kEnc, 10>(p, threads, smem_bytes, stream)
                   : launch_variant<kNS, kW, kOH, kOW, kFS, kCoop, kEnc, 8>(p, threads, smem_bytes, stream);
  }
  if (p.T > 1) {                // several steps per launch: variants 2 / 6
    if constexpr (kFS > 1) return cudaErrorInvalidValue;     // step_many_impl steps frame stacks one launch at a time
    else return p.pool ? launch_variant<kNS, kW, kOH, kOW, kFS, kCoop, kEnc, 6>(p, threads, smem_bytes, stream)
                       : launch_variant<kNS, kW, kOH, kOW, kFS, kCoop, kEnc, 2>(p, threads, smem_bytes, stream);
  }
  if (p.pool) {                 // wall-map pool: variants 4 / 5 (no uncapped pool instance is built)
    if (p.bits) return launch_variant<kNS, kW, kOH, kOW, kFS, kCoop, kEnc, 5>(p, threads, smem_bytes, stream);
    return launch_variant<kNS, kW, kOH, kOW, kFS, kCoop, kEnc, 4>(p, threads, smem_bytes, stream);
  }
  if (p.bits) return launch_variant<kNS, kW, kOH, kOW, kFS, kCoop, kEnc, 1>(p, threads, smem_bytes, stream);
  if constexpr (!kCoop) {
    if (p.bigreg) return launch_variant<kNS, kW, kOH, kOW, kFS, kCoop, kEnc, 3>(p, threads, smem_bytes, stream);
  }
  return launch_variant<kNS, kW, kOH, kOW, kFS, kCoop, kEnc, 0>(p, threads, smem_bytes, stream);
}

// The tile modes a set of instances is built for (bit 0 cooperative, bit 1 warp-private).
enum : int { TILES_COOP = 1, TILES_WARP = 2, TILES_BOTH = 3 };
static bool serves(int tiles, int coop) { return (tiles & (coop ? TILES_COOP : TILES_WARP)) != 0; }

template <int kNS, int kW, int kOH, int kOW, int kFS, int kEnc, int kTiles>
static cudaError_t launch_tiles(const KParams& p, int threads, size_t smem_bytes, cudaStream_t stream) {
  if constexpr ((kTiles & TILES_COOP) != 0) {
    if (p.coop) return launch_instance<kNS, kW, kOH, kOW, kFS, true, kEnc>(p, threads, smem_bytes, stream);
  }
  if constexpr ((kTiles & TILES_WARP) != 0) {
    if (!p.coop) return launch_instance<kNS, kW, kOH, kOW, kFS, false, kEnc>(p, threads, smem_bytes, stream);
  }
  return cudaErrorInvalidValue;             // the generic ENC_PAD set without coop: encode_flavour never gives that
}

// Specialised instances for the BASELINE shapes, in the tile modes create_impl's defaults give them; every other
// call, forced modes included, runs the generic instance of its flavour.
cudaError_t launch_tile_kernel(const KParams& p, int threads, size_t smem_bytes, cudaStream_t stream) {
  const Dims& d = p.d;
  const bool generic = p.force_generic != 0;
#define SNK_TRY(NS, W_, OH, OW, FS, ENC, TILES)                                                             \
  if (!generic && d.ns == NS && d.W == W_ && d.oh == OH && d.ow == OW && d.fs == FS && p.enc_flavour == ENC && \
      serves(TILES, p.coop))                                                                                 \
    return launch_tiles<NS, W_, OH, OW, FS, ENC, TILES>(p, threads, smem_bytes, stream);
  SNK_TRY(4, 20, 11, 11, 1, ENC_REG, TILES_BOTH)      // cfg1 / cfg5: 20x20, 4 snakes, vision 5
  SNK_TRY(4, 20, 20, 20, 1, ENC_DIRECT, TILES_BOTH)   // cfg2: full-grid observation
  SNK_TRY(4, 20, 11, 11, 4, ENC_LEGACY, TILES_COOP)   // cfg3: frame_stack 4 (create_impl: d.fs > 1 picks coop)
  SNK_TRY(16, 64, 15, 15, 1, ENC_PAD, TILES_COOP)     // cfg4: 64x64, 16 snakes, vision 7 (create_impl: ENC_PAD picks coop)
#undef SNK_TRY
  switch (p.enc_flavour) {
    case ENC_REG: return launch_tiles<0, 0, 0, 0, 0, ENC_REG, TILES_BOTH>(p, threads, smem_bytes, stream);
    case ENC_DIRECT: return launch_tiles<0, 0, 0, 0, 0, ENC_DIRECT, TILES_BOTH>(p, threads, smem_bytes, stream);
    case ENC_PAD: return launch_tiles<0, 0, 0, 0, 0, ENC_PAD, TILES_COOP>(p, threads, smem_bytes, stream);
    default: return launch_tiles<0, 0, 0, 0, 0, ENC_LEGACY, TILES_BOTH>(p, threads, smem_bytes, stream);
  }
}

cudaError_t launch_get_state(const Dims& d, const uint8_t* recs, const uint8_t* base_grid, const MapView& mv, uint32_t* err,
                             const StateView& sv, cudaStream_t s) {
  snk_get_state_kernel<<<(d.N + 127) / 128, 128, 0, s>>>(d, recs, base_grid, mv, err, sv);
  return cudaGetLastError();
}
cudaError_t launch_set_state(const Dims& d, uint8_t* recs, const uint8_t* base_grid, const MapView& mv, uint32_t* err,
                             const StateView& sv, cudaStream_t s) {
  snk_set_state_kernel<<<(d.N + 127) / 128, 128, 0, s>>>(d, recs, base_grid, mv, err, sv);
  return cudaGetLastError();
}
cudaError_t launch_pack_obs(const uint8_t* obs, uint8_t* bits, size_t n_units, cudaStream_t s) {
  if (n_units == 0) return cudaSuccess;
  const size_t want = ((n_units >> 2) + 255) / 256 + 1;
  const int grid = (int)(want < 148 * 16 ? want : 148 * 16);        // 16 CTAs of 256 threads per SM, grid-stride
  snk_pack_obs_kernel<<<grid, 256, 0, s>>>(obs, bits, n_units);
  return cudaGetLastError();
}
#ifdef SNK_PHASE_TIMING
// Profiling build only: point the kernels at a device trace buffer (n_ctas * 64 u64), or detach with nullptr.
extern "C" int snk_prof_set_trace(unsigned long long* dev_buf) {
  return (int)cudaMemcpyToSymbol(snk_trace_buf, &dev_buf, sizeof dev_buf);
}
extern "C" int snk_prof_set_trace2(unsigned long long* dev_buf) {
  return (int)cudaMemcpyToSymbol(snk_trace2_buf, &dev_buf, sizeof dev_buf);
}
#endif

cudaError_t launch_init_records(const Dims& d, uint8_t* recs, cudaStream_t s) {
  snk_init_records_kernel<<<592, 256, 0, s>>>(d, recs);
  return cudaGetLastError();
}

// One 16-byte unit per thread (a grid-stride loop only beyond 2^20 blocks), 32-bit unit indices where they fit.
static bool units_fit_u32(size_t n) { return n + ((size_t)256 << 20) <= 0xffffffffull; }
static int unit_blocks(size_t n) { const size_t b = (n + 255) / 256; return (int)(b < ((size_t)1 << 20) ? b : (size_t)1 << 20); }

cudaError_t launch_snapshot(const Dims& d, const uint8_t* recs, const uint8_t* hist, const uint8_t* cur_map, const int32_t* ids,
                            int count, uint64_t digest, uint8_t* snap, uint32_t* err, cudaStream_t s) {
  const size_t n = (size_t)count * (snapshot_slot_bytes(d) / 16);
  if (units_fit_u32(n) && units_fit_u32((size_t)d.N * (snapshot_slot_bytes(d) / 16)))
    snk_snapshot_kernel<uint32_t><<<unit_blocks(n), 256, 0, s>>>(d, recs, hist, cur_map, ids, count, digest, snap, err);
  else
    snk_snapshot_kernel<uint64_t><<<unit_blocks(n), 256, 0, s>>>(d, recs, hist, cur_map, ids, count, digest, snap, err);
  return cudaGetLastError();
}
cudaError_t launch_restore(const Dims& d, uint8_t* recs, uint8_t* hist, uint8_t* cur_map, const int32_t* src, int num_slots,
                           const uint8_t* snap, uint64_t digest, uint8_t* mask, uint32_t* err, cudaStream_t s) {
  const size_t n = (size_t)d.N * (snapshot_slot_bytes(d) / 16);
  if (units_fit_u32(n) && units_fit_u32((size_t)num_slots * (snapshot_slot_bytes(d) / 16)))
    snk_restore_kernel<uint32_t><<<unit_blocks(n), 256, 0, s>>>(d, recs, hist, cur_map, src, num_slots, snap, digest, mask, err);
  else
    snk_restore_kernel<uint64_t><<<unit_blocks(n), 256, 0, s>>>(d, recs, hist, cur_map, src, num_slots, snap, digest, mask, err);
  return cudaGetLastError();
}
cudaError_t launch_emit_stacked(const Dims& d, const uint8_t* recs, const uint8_t* hist, const uint8_t* base_grid,
                                const MapView& mv, const uint8_t* mask, uint8_t* obs, uint8_t* bits, uint8_t* grid,
                                uint32_t* err, cudaStream_t s) {
  snk_emit_stacked_kernel<<<(d.N + 7) / 8, 256, 0, s>>>(d, recs, hist, base_grid, mv, mask, obs, bits, grid, err);
  return cudaGetLastError();
}

}  // namespace snk
