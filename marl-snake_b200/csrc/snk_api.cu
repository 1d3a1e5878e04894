// snk_api.cu -- the C ABI declared in include/snk.h.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cmath>
#include <mutex>
#include <new>
#include <map>
#include <vector>

#include "../../include/snk.h"
#include "snk_hostxfer.h"
#include "snk_kernels.h"

using namespace snk;

enum { XFER_RAW = 0, XFER_PACKED = 1, XFER_MAX_CHUNKS = 64 };

static thread_local char g_err[512] = "";

static bool in_compressible_block(const void* p);

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
  return code;
}

// Entry points run on the handle's device and leave the calling thread's current device as they found it.
struct DeviceGuard {
  int prev = -1, want = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int dev) : want(dev) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
  }
  ~DeviceGuard() { if (prev >= 0 && prev != want) cudaSetDevice(prev); }
};
#define ON_DEVICE(h)                                                                                   \
  DeviceGuard _guard((h)->device);                                                                     \
  if (_guard.err != cudaSuccess) return fail(SNK_E_CUDA, "cudaSetDevice(%d): %s", (h)->device, cudaGetErrorString(_guard.err))

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t _e = (call);                                                                  \
    if (_e != cudaSuccess)                                                                    \
      return fail(SNK_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

// The terminal-info outputs of snk_step_extra, in its field order: element size, and [N, ns] (per snake) or [N].
constexpr int N_EXTRA = 6;
struct ExtraOut { size_t elem; bool per_snake; };
static const ExtraOut EXTRA_OUT[N_EXTRA] = {{1, false}, {sizeof(int32_t), true}, {sizeof(double), true},
                                            {sizeof(int32_t), true}, {sizeof(int32_t), true}, {sizeof(int32_t), true}};
static_assert(sizeof(snk_step_extra) == N_EXTRA * sizeof(void*), "EXTRA_OUT describes every field of snk_step_extra");
static size_t extra_bytes(const Dims& d, int i) { return EXTRA_OUT[i].elem * d.N * (EXTRA_OUT[i].per_snake ? d.ns : 1); }
// snk_step_extra as the array of its pointers (null x: all null), and back
struct ExtraPtrs { uint8_t* p[N_EXTRA]; };
static ExtraPtrs extra_ptrs(const snk_step_extra* x) {
  ExtraPtrs a = {};
  if (x) memcpy(a.p, x, sizeof *x);
  return a;
}
static snk_step_extra extra_struct(const ExtraPtrs& a) {
  snk_step_extra x;
  memcpy(&x, a.p, sizeof x);
  return x;
}

struct snk_env {
  // The launch template: the shape, the resident device buffers and every launch decision of create_impl.  A launch
  // copies it and fills in its own I/O.  (Its `pool` is the wall-map pool, not the widening pool below.)
  KParams kp = {};
  int device = 0;
  int threads = 0;
  size_t smem_bytes = 0;
  int many_tile_envs = 0, many_threads = 0;      // tile shape of multi-step launches (snk_step_many, cooperative tiles)
  size_t many_smem_bytes = 0;
  uint64_t pool_digest = 0;                      // layouts + spawn-table sizes: a checkpoint only loads into the same pool
  uint64_t snap_digest = 0;                      // what gives a snapshot slot's bytes their meaning (snapshot_digest)
  uint8_t* restore_mask = nullptr;               // [N] envs the last snk_restore restored: its encode's mask
  // ordering between the caller's streams (device-pointer calls) and own_stream (host-buffer calls)
  cudaStream_t last_user_stream = nullptr;
  bool user_work_pending = false;
  cudaEvent_t user_ev = nullptr;
  // device mirrors used by the *_host entry points; h_extra in EXTRA_OUT order
  uint8_t* h_actions = nullptr; uint8_t* h_obs = nullptr; double* h_rew = nullptr; uint8_t* h_done = nullptr;
  uint8_t* h_extra[N_EXTRA] = {};
  // few environments: every output of a host-buffer step lives in ONE device block mirrored by ONE pinned host
  // block, so the step costs one copy in, one launch, one copy out (the latency-bound drop-in mode)
  uint8_t* small_dev = nullptr; uint8_t* small_host = nullptr; uint8_t* small_map = nullptr;
  int small_zero_copy = 1;
  cudaStream_t own_stream = nullptr;
  // packed host transport (snk_hostxfer.cpp): device channel-bit mirror, pinned staging, widening pool
  int xfer_mode = XFER_RAW, xfer_threads = 0;
  uint8_t* d_bits = nullptr; uint8_t* p_bits = nullptr;
  WidenPool* pool = nullptr;
  cudaEvent_t chunk_ev[XFER_MAX_CHUNKS] = {};
  int n_chunk_ev = 0;
  bool was_reset = false;
};

extern "C" const char* snk_last_error(void) { return g_err; }
extern "C" int snk_abi_version(void) { return SNK_ABI_VERSION; }

static int env_int(const char* name, int dflt) {
  const char* s = getenv(name);
  return (s && *s) ? atoi(s) : dflt;
}

// cudaMalloc of `bytes` filled from host memory; dst may be a pointer to const (the template's read-only buffers)
template <typename T>
static cudaError_t upload(T*& dst, const void* src, size_t bytes) {
  void* p = nullptr;
  const cudaError_t e = cudaMalloc(&p, bytes);
  dst = static_cast<T*>(p);
  return e != cudaSuccess ? e : cudaMemcpy(p, src, bytes, cudaMemcpyHostToDevice);
}

// num_maps == 0: snk_create (walls_host null) or snk_create_map (one layout, no pool); num_maps >= 1: a wall-map pool of
// num_maps layouts of height * width bytes, back to back in walls_host
static int create_impl(const snk_config* c, int num_maps, const uint8_t* walls_host, const uint8_t* map_ids_host, snk_env** out);
extern "C" int snk_create(const snk_config* c, snk_env** out) { return create_impl(c, 0, nullptr, nullptr, out); }
extern "C" int snk_create_map(const snk_config* c, const uint8_t* walls_host, snk_env** out) {
  if (!walls_host) return fail(SNK_E_INVALID, "null wall map");
  return create_impl(c, 0, walls_host, nullptr, out);
}
extern "C" int snk_create_maps(const snk_config* c, int32_t num_maps, const uint8_t* walls_host, const uint8_t* map_ids_host,
                               snk_env** out) {
  if (num_maps < 1 || num_maps > SNK_MAX_MAPS) return fail(SNK_E_INVALID, "num_maps must be in 1..%d", SNK_MAX_MAPS);
  if (!walls_host) return fail(SNK_E_INVALID, "null wall maps");
  return create_impl(c, num_maps, walls_host, map_ids_host, out);
}

static uint64_t fnv1a(uint64_t h, const void* data, size_t n) {
  const uint8_t* b = (const uint8_t*)data;
  for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 0x100000001B3ull; }
  return h;
}

// Snapshot slots (snk_snapshot) hold raw records: they restore only into handles whose records mean the same bytes --
// shape, record layout, counter width, fruit slots and wall layout (pool digest or the single layout's).  Never 0.
static uint64_t snapshot_digest(const Dims& d, uint64_t walls) {
  struct { int32_t H, W, ns, V, fs, ohw_p, compact, dig, hbm_rec_bytes, hist_env_bytes, stat16, fcap; uint64_t walls; } k;
  memset(&k, 0, sizeof k);
  k.H = d.H; k.W = d.W; k.ns = d.ns; k.V = d.V; k.fs = d.fs; k.ohw_p = d.ohw_p; k.compact = d.compact; k.dig = d.dig;
  k.hbm_rec_bytes = d.hbm_rec_bytes; k.hist_env_bytes = d.hist_env_bytes; k.stat16 = d.stat16; k.fcap = d.fcap; k.walls = walls;
  const uint64_t h = fnv1a(0xCBF29CE484222325ull, &k, sizeof k);
  return h ? h : 1;
}

static int create_impl(const snk_config* c, int num_maps, const uint8_t* walls_host, const uint8_t* map_ids_host, snk_env** out) {
  if (!c || !out) return fail(SNK_E_INVALID, "null argument");
  if (c->abi_version != SNK_ABI_VERSION) return fail(SNK_E_INVALID, "abi_version %d != %d", c->abi_version, SNK_ABI_VERSION);
  if (c->num_envs < 1) return fail(SNK_E_INVALID, "num_envs must be >= 1");
  if (c->num_snakes < 1 || c->num_snakes > MAX_SNAKES) return fail(SNK_E_INVALID, "num_snakes must be in 1..%d", MAX_SNAKES);
  if (c->snake_length < 2 || c->snake_length > MAX_SNAKE_LENGTH) return fail(SNK_E_INVALID, "snake_length must be in 2..%d", MAX_SNAKE_LENGTH);
  if (c->height < 4 || c->width < 4 || (int64_t)c->height * c->width > 65535) return fail(SNK_E_INVALID, "grid must be at least 4x4 and at most 65535 cells");
  if (c->vision_range < 0 || c->frame_stack < 1 || c->frame_stack > 64) return fail(SNK_E_INVALID, "bad vision_range / frame_stack");
  if (c->rng_mode != SNK_RNG_PHILOX && c->rng_mode != SNK_RNG_REPLAY) return fail(SNK_E_INVALID, "bad rng_mode");
  if (c->observer != SNK_OBSERVER_SNAKE && c->observer != SNK_OBSERVER_HUMAN) return fail(SNK_E_INVALID, "bad observer");
  int nfruits = c->num_fruits < 0 ? (int)nearbyint(c->num_snakes * 0.8) : c->num_fruits;   // snake_env.py:87-88
  if (nfruits > MAX_FRUIT_DRAWS) return fail(SNK_E_INVALID, "num_fruits must be <= %d", MAX_FRUIT_DRAWS);

  snk_env* h = new (std::nothrow) snk_env();
  if (!h) return fail(SNK_E_NOMEM, "out of host memory");
  Dims& d = h->kp.d;
  memset(&d, 0, sizeof d);
  d.N = c->num_envs; d.H = c->height; d.W = c->width; d.ns = c->num_snakes; d.K = c->snake_length;
  d.V = c->vision_range; d.fs = c->frame_stack; d.nfruits = nfruits;
  d.auto_reset = c->auto_reset ? 1 : 0; d.done_mode = c->done_mode ? 1 : 0; d.rng_mode = c->rng_mode;
  d.observer = c->observer;
  d.dig = default_dig(d.ns);
  d.compact = 1;                      // decided with the tile mode below
  d.seed_lo = (uint32_t)c->seed; d.seed_hi = (uint32_t)(c->seed >> 32);
  d.env_off_lo = (uint32_t)c->env_id_offset; d.env_off_hi = (uint32_t)(c->env_id_offset >> 32);
  d.r_fruit = c->reward_fruit; d.r_kill = c->reward_kill; d.r_lose = c->reward_lose;
  d.r_win = c->reward_win; d.r_time = c->reward_time; d.max_steps = c->max_episode_steps;
  finalize_layout(d);
  h->device = c->device;

  // custom wall layout (make_grid_from_txt, core/grid_util.py:23-33): normalised to cell codes, one word-padded plane.
  // The outer ring must be wall -- it is what keeps a head inside the array (the reference would index out of it).
  // A wall-map pool keeps every map so, off_c0 bytes apart.
  const int nmaps = walls_host ? (num_maps ? num_maps : 1) : 0;
  const size_t plane = num_maps ? (size_t)d.off_c0 : ((size_t)d.HW + 3) / 4 * 4;
  std::vector<uint8_t> walls;
  if (walls_host) {
    walls.assign((size_t)nmaps * plane, 0);
    for (int m = 0; m < nmaps; ++m) {
      const uint8_t* src = walls_host + (size_t)m * d.HW;
      uint8_t* dst = walls.data() + (size_t)m * plane;
      for (int i = 0; i < d.HW; ++i) dst[i] = src[i] ? (uint8_t)WALL : (uint8_t)EMPTY;
      for (int i = 0; i < d.HW; ++i) {
        const int r = i / d.W, cc = i % d.W;
        if ((r == 0 || r == d.H - 1 || cc == 0 || cc == d.W - 1) && !dst[i]) {
          delete h;
          if (num_maps) return fail(SNK_E_INVALID, "wall map %d: border cell (%d, %d) is not a wall", m, r, cc);
          return fail(SNK_E_INVALID, "wall map: border cell (%d, %d) is not a wall", r, cc);
        }
      }
    }
  }
  const uint8_t* wm = walls_host ? walls.data() : nullptr;
  uint64_t layout_digest = 0;                    // of the single wall layout (walled box or custom map), no pool

  // spawn table (host) -- core/grid_util.py:73-115.  A pool concatenates one table per map.
  std::vector<uint64_t> table;
  std::vector<uint2> map_tab;
  for (int m = 0; m < (nmaps ? nmaps : 1); ++m) {
    const uint8_t* wmm = wm ? wm + (size_t)m * plane : nullptr;
    const int64_t n_cand = spawn_enumerate(d.H, d.W, d.K, nullptr, nullptr, 0, SPAWN_TABLE_LIMIT, wmm);
    if (n_cand < d.ns) {
      delete h;
      if (num_maps) return fail(SNK_E_INVALID, "wall map %d: only %lld spawn poses for %d snakes", m, (long long)n_cand, c->num_snakes);
      return fail(SNK_E_INVALID, "only %lld spawn poses for %d snakes", (long long)n_cand, c->num_snakes);
    }
    if (n_cand > SPAWN_TABLE_LIMIT) {
      delete h;
      if (num_maps) return fail(SNK_E_INVALID, "wall map %d: more than %lld spawn poses for snake_length %d", m,
                                (long long)SPAWN_TABLE_LIMIT, c->snake_length);
      return fail(SNK_E_INVALID, "more than %lld spawn poses for a %dx%d grid and snake_length %d (the reference enumerates "
                  "them on every reset; here the table would not fit)", (long long)SPAWN_TABLE_LIMIT, c->height, c->width, c->snake_length);
    }
    if ((int64_t)table.size() + n_cand > SPAWN_TABLE_LIMIT) {
      delete h;
      return fail(SNK_E_INVALID, "wall maps 0..%d: more than %lld spawn poses together (%lld MB of tables)", m,
                  (long long)SPAWN_TABLE_LIMIT, (long long)(SPAWN_TABLE_LIMIT * 8 >> 20));
    }
    map_tab.push_back(make_uint2((uint32_t)table.size(), (uint32_t)n_cand));
    table.resize(table.size() + (size_t)n_cand);
    spawn_enumerate(d.H, d.W, d.K, table.data() + map_tab.back().x, nullptr, n_cand, 0, wmm);
  }
  d.n_cand = map_tab[0].y;
  std::vector<uint8_t> ids;
  if (num_maps) {
    // next_map: the caller's assignment, or global env id modulo the number of maps (a sharded run equals one run)
    ids.resize((size_t)d.N);
    for (int e = 0; e < d.N; ++e) {
      if (map_ids_host && map_ids_host[e] >= num_maps) {
        delete h;
        return fail(SNK_E_INVALID, "map_ids[%d] = %d names no map (num_maps %d)", e, map_ids_host[e], num_maps);
      }
      ids[e] = map_ids_host ? map_ids_host[e] : (uint8_t)((c->env_id_offset + (uint64_t)e) % (uint64_t)num_maps);
    }
    h->kp.num_maps = num_maps;
    uint64_t dg = fnv1a(0xCBF29CE484222325ull, walls.data(), walls.size());
    h->pool_digest = fnv1a(dg, map_tab.data(), map_tab.size() * sizeof(uint2));
  }

  // tile shape: a tile is 32/G environments (G = num_snakes rounded up to a power of two).  Large
  // batches: every warp owns a tile, the CTA's warps share only the encode tables.  Small batches or
  // large records: the CTA owns one tile and its warps share the tile's viewers (coop).
  const int EPW_full = 32 / tile_group(d.ns);
  const int64_t tiles_full = ((int64_t)d.N + EPW_full - 1) / EPW_full;
  // Measured on the B200 (profiles/README.md, tools/sweep_tiles*.sh): warp-private tiles win once the batch
  // is several waves deep; below that, and for large records or frame stacks, the CTA-cooperative mode does.
  // With compact records (profiles/r02_ab_compact*.txt) warp-private tiles already win from ~6 000 tiles on:
  // 65 536 envs of the cfg5 shape 0.057 ms against 0.061 ms cooperative, 131 072 envs 0.097 against 0.114 ms.
  int coop = env_int("SNK_COOP", -1);
  // Windows of 128..255 cells have their fast encode (padded planes) only in cooperative tiles: a 32x32 / 8-snake /
  // vision-7 batch runs 0.101 ms cooperative against 0.119 ms warp-private at 32 768 envs, 0.70 against 0.78 ms at
  // 262 144 (profiles/r02_ab_shapes.txt).
  if (coop < 0) coop = (tiles_full < 148 * 40 || (size_t)EPW_full * d.rec_bytes > 8 * 1024 || d.fs > 1 ||
                        encode_flavour(d, true) == ENC_PAD) ? 1 : 0;
  // Compact records (the grid is rebuilt in shared memory from walls + fruit slots + bodies instead of being read
  // from and written to HBM) save 2 * H * W bytes per env-step and cost the rule warp a walk along every live body.
  // That pays wherever bytes bound the step: warp-private tiles (cfg5 0.855 -> 0.769 ms), frame stacks (cfg3 0.207 ->
  // 0.202 ms) and large grids (cfg4 0.124 -> 0.121 ms); a cooperative tile of a small grid is bound by the latency of
  // its single rule warp, and there the walk costs more than the bytes (131 072-env shard 0.114 -> 0.118 ms, cfg2
  // 0.0187 -> 0.0208 ms).  SNK_COMPACT=0/1 (or the older SNK_NO_COMPACT=1) forces the layout.
  {
    int compact = env_int("SNK_COMPACT", -1);
    if (compact < 0) compact = default_compact() ? ((!coop || d.fs > 1 || d.HW >= 1024) ? 1 : 0) : 0;
    if (!compact) { d.compact = 0; d.dig = default_dig(d.ns); finalize_layout(d); }
  }
  // A coop tile may hold fewer environments than the rule warp has lane groups: shorter per-CTA latency
  // (the rule phase of one warp, then the tile's encode) and more rule warps in flight.  Shrink until a
  // tile's observation block is <= 64 KB (32 KB with a frame stack, where a warp encodes a whole environment), and
  // further while the launch would not fill every SM 16 times.  (cfg4, 28.8 KB per environment: two environments per
  // tile -- a full rule warp -- 0.108 ms against 0.121 ms with one, profiles/r02_ab_tiles.txt.)
  int EPW = env_int("SNK_TILE_ENVS", 0);
  if (EPW <= 0) {
    EPW = EPW_full;
    if (coop) {
      while (EPW > 1 && (size_t)EPW * d.obs_env_bytes > (size_t)(d.fs > 1 ? 32 : 64) * 1024) EPW >>= 1;
      while (EPW > 1 && ((int64_t)d.N + EPW - 1) / EPW < 148 * 16) EPW >>= 1;
    }
  }
  if (EPW > EPW_full || (EPW & (EPW - 1))) {
    delete h;
    return fail(SNK_E_INVALID, "SNK_TILE_ENVS must be a power of two <= %d", EPW_full);
  }
  // frame_stack > 1 encodes one environment per warp, so more warps than environments would idle
  // (the padded-plane encode wants an even number of warps: with an odd window a warp then only ever sees viewer
  // blocks of one address parity and keeps one set of cell offsets in registers)
  // (warp-private tiles: four warps per CTA share the encode tables and the per-CTA shared-memory overhead -- half
  // a percent over single-warp CTAs at every batch size measured, profiles/r02_ab_tiles.txt)
  int threads = env_int("SNK_THREADS", !coop ? 128 : d.fs > 1 ? 32 * (EPW < 8 ? EPW : 8)
                                       : encode_flavour(d, true) == ENC_PAD ? 128 : 64);    // 64: cfg2 0.0177 ms against 0.0199 at 96 (r02_ab_coop_threads.txt)
  const int max_threads = coop ? SNK_MAX_THREADS_COOP : SNK_MAX_THREADS;
  if (threads < 32 || threads > max_threads || (threads & 31)) { delete h; return fail(SNK_E_INVALID, "SNK_THREADS must be a multiple of 32 in 32..%d", max_threads); }
  // large grids: fewer environments per tile until two CTAs fit an SM, then fewer warps if it still does not fit
  if (env_int("SNK_TILE_ENVS", 0) <= 0)
    while (EPW > 1 && tile_smem_bytes(d, coop ? threads / 32 : 1, coop != 0, EPW) > 100 * 1024) EPW >>= 1;
  while (threads > 32 && tile_smem_bytes(d, threads / 32, coop != 0, EPW) > 200 * 1024) threads -= 32;
  h->kp.E = EPW; h->threads = threads; h->kp.coop = coop;
  {
    // snk_step_many: every CTA lives for the whole launch, so the grid should be ONE resident wave -- as many
    // environments per cooperative tile as the rule warp has lane groups (fewer, longer-lived CTAs), more warps to
    // share the tile's viewers.  Warp-private tiles keep their shape.
    int me = coop ? env_int("SNK_MANY_TILE_ENVS", EPW_full) : EPW;
    int mt = coop ? env_int("SNK_MANY_THREADS", 128) : threads;
    if (me < 1 || me > EPW_full || (me & (me - 1)) || mt < 32 || mt > max_threads || (mt & 31)) { me = EPW; mt = threads; }
    while (me > 1 && tile_smem_bytes(d, coop ? mt / 32 : 1, coop != 0, me) > 100 * 1024) me >>= 1;
    h->many_tile_envs = me; h->many_threads = mt;
    h->many_smem_bytes = tile_smem_bytes(d, mt / 32, coop != 0, me);
  }
  h->kp.force_generic = env_int("SNK_FORCE_GENERIC", 0);
  h->kp.use_tma = env_int("SNK_TMA", 1);
  h->kp.pdl = env_int("SNK_PDL", 1);
  h->small_zero_copy = env_int("SNK_SMALL_ZEROCOPY", 1);
  h->kp.l2_keep = env_int("SNK_L2_KEEP", d.fs > 1 ? 1 : 0);
  h->kp.l2_keep_frac = (float)env_int("SNK_L2_KEEP_PCT", 100) / 100.0f;
  {
    // the uncapped-register instance of the warp-private kernel once the batch is many waves deep (a step that writes
    // its observation into a compressible block runs the capped one all the same: see step_impl).  Pool handles run
    // the capped instances: no uncapped pool instance is built.
    const int64_t tiles = ((int64_t)d.N + EPW - 1) / EPW;
    h->kp.bigreg = (!coop && !num_maps && tiles >= (int64_t)env_int("SNK_BIGREG_TILES", 24576)) ? 1 : 0;
  }
  {
    // ENC_PAD: ceil(2^32 / words) of a grid and of a row (at least two words a row)
    const uint64_t one = (uint64_t)1 << 32;
    const uint64_t wpr = (uint64_t)(d.W >> 2 > 1 ? d.W >> 2 : 2), nw = (uint64_t)d.H * wpr;
    h->kp.inv_grid_words = (uint32_t)((one + nw - 1) / nw);
    h->kp.inv_row_words = (uint32_t)((one + wpr - 1) / wpr);
  }
  h->kp.T = 1;
  h->smem_bytes = tile_smem_bytes(d, threads / 32, coop != 0, EPW);
  if (h->smem_bytes > 227 * 1024) {
    const size_t need = h->smem_bytes;
    delete h;
    return fail(SNK_E_INVALID, "configuration needs %zu bytes of shared memory per tile", need);
  }

  DeviceGuard guard(c->device);
  if (guard.err != cudaSuccess) { delete h; return fail(SNK_E_CUDA, "cudaSetDevice(%d): %s", c->device, cudaGetErrorString(guard.err)); }
#define CUH(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) { int rc = fail(SNK_E_CUDA, "%s failed: %s", #call, cudaGetErrorString(_e)); snk_destroy(h); return rc; } } while (0)
  CUH(cudaMalloc(&h->kp.recs, (size_t)d.N * d.hbm_rec_bytes));
  if (d.hist_env_bytes) CUH(cudaMalloc(&h->kp.hist, (size_t)d.N * d.hist_env_bytes));
  CUH(upload(h->kp.spawn, table.data(), table.size() * sizeof(uint64_t)));
  CUH(cudaMalloc(&h->kp.err, sizeof(uint32_t)));
  CUH(cudaMalloc(&h->kp.stats, STAT_COUNT * sizeof(double)));
  CUH(cudaMalloc((void**)&h->kp.replay_off, ((size_t)d.N + 1) * sizeof(int64_t)));
  if (num_maps) {
    // the pool serves the resets and (compact records) the tile loads, which paint each grid from its own map
    CUH(upload(h->kp.pool, walls.data(), walls.size()));
    CUH(upload(h->kp.map_tab, map_tab.data(), map_tab.size() * sizeof(uint2)));
    CUH(upload(h->kp.next_map, ids.data(), ids.size()));
    CUH(upload(h->kp.cur_map, ids.data(), ids.size()));
  } else if (wm) {
    CUH(upload(h->kp.wall_map, walls.data(), walls.size()));
  }
  if (!num_maps) {
    // the wall layout every reset starts from: make_grid's walled box (core/grid_util.py:14-20) or the custom map,
    // padded to 16 bytes.  Compact records: it is also what the grid every record implies starts from -- as many
    // copies as the widest tile has environments, so ONE bulk copy paints a tile's grids
    const int copies = !d.compact ? 1 : h->kp.E > h->many_tile_envs ? h->kp.E : h->many_tile_envs;
    std::vector<uint8_t> tpl((size_t)copies * d.off_c0, 0);
    for (int i = 0; i < d.HW; ++i) tpl[i] = wm ? wm[i] : wall_or_empty(i, d.H, d.W);
    layout_digest = fnv1a(0xCBF29CE484222325ull, tpl.data(), (size_t)d.HW);
    for (int k = 1; k < copies; ++k) memcpy(tpl.data() + (size_t)k * d.off_c0, tpl.data(), (size_t)d.off_c0);
    CUH(upload(h->kp.base_grid, tpl.data(), tpl.size()));
  }
  {
    size_t tab_off = 0, lutb_off = 0;
    const size_t nb = encode_blob_bytes(d, &tab_off, &lutb_off);
    std::vector<uint8_t> blob(nb, 0);
    encode_blob_fill(d, blob.data());
    CUH(upload(h->kp.enc_blob, blob.data(), nb));
    KParams& p = h->kp;
    p.enc_blob_bytes = (int)nb; p.enc_tab_off = (int)tab_off; p.enc_lutb_off = (int)lutb_off;
    p.lut_dual = encode_lut_dual(d) ? 1 : 0;
    p.use_tab = encode_uses_table(d) && (p.lut_dual || !env_int("SNK_NO_TABLE", 0)) ? 1 : 0;
    // SNK_ENC_LEGACY=1 / SNK_ENC_NOPAD=1: A/B switches (the cooperative ENC_PAD encode falls back to what warp-private
    // tiles of the same shape run)
    p.enc_flavour = env_int("SNK_ENC_LEGACY", 0) ? ENC_LEGACY : encode_flavour(d, coop != 0 && !env_int("SNK_ENC_NOPAD", 0));
    p.enc_copy_bytes = (p.enc_flavour == ENC_LEGACY) ? p.enc_blob_bytes : p.enc_tab_off;     // LUT only
  }
  CUH(cudaMemset(h->kp.err, 0, sizeof(uint32_t)));
  CUH(cudaMemset(h->kp.stats, 0, STAT_COUNT * sizeof(double)));
  CUH(cudaMemset((void*)h->kp.replay_off, 0, ((size_t)d.N + 1) * sizeof(int64_t)));
  if (d.hist_env_bytes) CUH(cudaMemset(h->kp.hist, 0, (size_t)d.N * d.hist_env_bytes));
  CUH(launch_init_records(d, h->kp.recs, nullptr));
  CUH(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  CUH(cudaEventCreateWithFlags(&h->user_ev, cudaEventDisableTiming));
  CUH(cudaMalloc(&h->restore_mask, (size_t)d.N));     // last: every buffer before it lies where it did without it
  CUH(cudaDeviceSynchronize());
#undef CUH
  h->snap_digest = snapshot_digest(d, num_maps ? h->pool_digest : layout_digest);
  {
    // host entry points: ship channel bits and widen on the host once the observation block is large
    // enough for the PCIe link to matter (SNK_HOST_TRANSPORT = raw | packed overrides)
    const char* t = getenv("SNK_HOST_TRANSPORT");
    const bool big = (size_t)d.N * d.obs_env_bytes >= ((size_t)4 << 20);
    h->xfer_mode = (t && !strcmp(t, "raw")) ? XFER_RAW : (t && !strcmp(t, "packed")) ? XFER_PACKED
                   : big ? XFER_PACKED : XFER_RAW;
    h->xfer_threads = env_int("SNK_HOST_THREADS", 0);
  }
  *out = h;
  return SNK_OK;
}

extern "C" int snk_destroy(snk_env* h) {
  if (!h) return SNK_OK;
  DeviceGuard guard(h->device);
  const KParams& p = h->kp;
  const void* bufs[] = {p.recs, p.hist, p.spawn, p.replay, p.replay_off, p.err, p.stats, p.enc_blob, p.wall_map, p.base_grid,
                        p.pool, p.map_tab, p.next_map, p.cur_map};
  for (const void* b : bufs) cudaFree(const_cast<void*>(b));
  cudaFree(h->h_actions); cudaFree(h->h_obs); cudaFree(h->h_rew); cudaFree(h->h_done);
  for (uint8_t* b : h->h_extra) cudaFree(b);
  cudaFree(h->small_dev);
  cudaFree(h->restore_mask);
  if (h->small_host) cudaFreeHost(h->small_host);
  cudaFree(h->d_bits);
  if (h->p_bits) cudaFreeHost(h->p_bits);
  delete h->pool;
  for (int i = 0; i < h->n_chunk_ev; ++i) cudaEventDestroy(h->chunk_ev[i]);
  if (h->user_ev) cudaEventDestroy(h->user_ev);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
  return SNK_OK;
}

extern "C" int snk_obs_shape(const snk_env* h, int32_t out[4]) {
  if (!h || !out) return fail(SNK_E_INVALID, "null argument");
  out[0] = h->kp.d.ns; out[1] = h->kp.d.oh; out[2] = h->kp.d.ow; out[3] = 8 * h->kp.d.fs;
  return SNK_OK;
}
extern "C" size_t snk_obs_bytes(const snk_env* h) { return h ? (size_t)h->kp.d.N * h->kp.d.obs_env_bytes : 0; }
extern "C" int snk_num_envs(const snk_env* h) { return h ? h->kp.d.N : 0; }
extern "C" int snk_num_maps(const snk_env* h) { return h ? h->kp.num_maps : 0; }

extern "C" int snk_map_ids_dev(snk_env* h, uint8_t** next_dev, uint8_t** cur_dev) {
  if (!h || !next_dev || !cur_dev) return fail(SNK_E_INVALID, "null argument");
  if (!h->kp.num_maps) return fail(SNK_E_STATE, "handle has no wall-map pool (create it with snk_create_maps)");
  *next_dev = const_cast<uint8_t*>(h->kp.next_map); *cur_dev = h->kp.cur_map;
  return SNK_OK;
}

extern "C" size_t snk_algorithmic_bytes_per_env_step(const snk_env* h) {
  if (!h) return 0;
  const Dims& d = h->kp.d;
  // state record read + write, frame history (read fs-1 rows, write 1), observation write,
  // actions in, rewards (f64) and dones out.
  size_t b = 2 * (size_t)d.hbm_rec_bytes + (size_t)d.obs_env_bytes + (size_t)d.ns * (1 + 8 + 1);
  if (d.fs > 1) b += (size_t)d.ns * d.fs * d.ohw;
  return b;
}

// Device-pointer calls only enqueue work on the caller's stream.  The host-buffer calls run on the handle's own
// stream and synchronise before they return, so ordering is needed in one direction only: before a host-buffer
// call launches, own_stream waits for whatever the last device-pointer call left on the caller's stream.
static void note_user_stream(snk_env* h, cudaStream_t s) {
  if (s == h->own_stream) return;
  h->last_user_stream = s;
  h->user_work_pending = true;
}
static int own_stream_after_user_work(snk_env* h) {
  if (!h->user_work_pending) return SNK_OK;
  h->user_work_pending = false;
  // (a stream that is being captured cannot record an event for the outside world; such work is ordered by the
  // graph launch, which the caller issues on a stream of their own)
  if (cudaEventRecord(h->user_ev, h->last_user_stream) != cudaSuccess) { cudaGetLastError(); return SNK_OK; }
  CU(cudaStreamWaitEvent(h->own_stream, h->user_ev, 0));
  return SNK_OK;
}

extern "C" int snk_note_stream(snk_env* h, void* stream) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  note_user_stream(h, (cudaStream_t)stream);
  return SNK_OK;
}

// The parameters of one launch: the handle's template plus the call's I/O, once the pointers pass their checks.  A step
// needs actions, rewards and dones and a reset before it; a reset and the encode of set_state take none of the three.
// With T steps, actions / rewards / dones / extras are [T, ...], and obs / bits / grid too when `every`.
static int call_params(snk_env* h, KParams& p, int mode, const uint8_t* actions, uint8_t* obs, uint8_t* bits, uint8_t* grid,
                       double* rew, uint8_t* done, const snk_step_extra* x, int T = 1, int every = 0) {
  if (mode == MODE_STEP) {
    if (!actions || !rew || !done) return fail(SNK_E_INVALID, "actions, rewards and dones are required");
    if (!h->was_reset) return fail(SNK_E_STATE, "step before reset");
  }
  if (obs && ((uintptr_t)obs & 7)) return fail(SNK_E_INVALID, "obs must be 8-byte aligned");
  if ((uintptr_t)rew & 7) return fail(SNK_E_INVALID, "rewards must be 8-byte aligned");
  p = h->kp;
  p.mode = mode; p.T = T; p.obs_every_step = every ? 1 : 0;
  p.actions = actions; p.obs = obs; p.bits = bits; p.grid_out = grid; p.rew = rew; p.done = done;
  if (x) {
    p.fin = x->finished; p.rank = x->rank; p.ep_scores = x->episode_scores;
    p.ep_steps = x->episode_steps; p.ep_fruits = x->episode_fruits; p.ep_kills = x->episode_kills;
  }
  // every env block 16-byte aligned (the per-step blocks of `every` are whole env blocks apart)
  p.vec16 = (obs && ((uintptr_t)obs & 15) == 0 && h->kp.d.obs_env_bytes % 16 == 0) ? 1 : 0;
  return SNK_OK;
}

static int reset_impl(snk_env* h, const uint8_t* mask_dev, uint8_t* obs_dev, uint8_t* bits_dev, uint8_t* grid_dev,
                      cudaStream_t stream) {
  KParams p;
  const int rc = call_params(h, p, MODE_RESET, nullptr, obs_dev, bits_dev, grid_dev, nullptr, nullptr, nullptr);
  if (rc) return rc;
  p.mask = mask_dev;
  CU(launch_tile_kernel(p, h->threads, h->smem_bytes, stream));
  note_user_stream(h, stream);
  h->was_reset = true;
  return SNK_OK;
}

static int step_impl(snk_env* h, const uint8_t* actions_dev, uint8_t* obs_dev, uint8_t* bits_dev, uint8_t* grid_dev,
                     double* rewards_dev, uint8_t* dones_dev, const snk_step_extra* x, cudaStream_t stream) {
  KParams p;
  const int rc = call_params(h, p, MODE_STEP, actions_dev, obs_dev, bits_dev, grid_dev, rewards_dev, dones_dev, x);
  if (rc) return rc;
  // An observation block in compressible memory costs the step far less DRAM time, and the step is then bound by the
  // latency of its rule phase: the 64-register instance, with twice the resident warps, is the faster one there
  // (cfg5, 1 048 576 envs on a B200 at 1000 W: 0.671 ms against 0.758 ms uncapped; profiles/r03_retune.txt).
  // (A step that writes the global state runs a capped instance in any case: the grid variants have no uncapped one.)
  const uint8_t* out_dev = obs_dev ? obs_dev : grid_dev;
  if (p.bigreg && out_dev && in_compressible_block(out_dev)) p.bigreg = 0;
  CU(launch_tile_kernel(p, h->threads, h->smem_bytes, stream));
  note_user_stream(h, stream);
  return SNK_OK;
}

// T steps in one call.  frame_stack 1: ONE launch, every tile's records stay in shared memory for all T steps.
// frame_stack > 1 (the frame history is written per step): T ordinary launches -- same results, same arrays.
static int step_many_impl(snk_env* h, int T, const uint8_t* actions_dev, uint8_t* obs_dev, uint8_t* bits_dev, uint8_t* grid_dev,
                          int every, double* rewards_dev, uint8_t* dones_dev, const snk_step_extra* x, cudaStream_t stream) {
  if (!actions_dev || !rewards_dev || !dones_dev) return fail(SNK_E_INVALID, "actions, rewards and dones are required");
  if (T < 1 || T > 65536) return fail(SNK_E_INVALID, "num_steps must be in 1..65536");
  const Dims& d = h->kp.d;
  const size_t nn = (size_t)d.N * d.ns;
  if (d.fs == 1) {
    KParams p;
    const int rc = call_params(h, p, MODE_STEP, actions_dev, obs_dev, bits_dev, grid_dev, rewards_dev, dones_dev, x, T, every);
    if (rc) return rc;
    const bool many = T > 1;
    if (many) p.E = h->many_tile_envs;
    CU(launch_tile_kernel(p, many ? h->many_threads : h->threads, many ? h->many_smem_bytes : h->smem_bytes, stream));
    note_user_stream(h, stream);
    return SNK_OK;
  }
  for (int t = 0; t < T; ++t) {
    ExtraPtrs xp = extra_ptrs(x);
    for (int i = 0; i < N_EXTRA; ++i)
      if (xp.p[i]) xp.p[i] += t * extra_bytes(d, i);
    const snk_step_extra xt = extra_struct(xp);
    const bool render = every || t == T - 1;
    uint8_t* o = (obs_dev && render) ? obs_dev + (every ? (size_t)t * d.N * d.obs_env_bytes : 0) : nullptr;
    uint8_t* b = (bits_dev && render) ? bits_dev + (every ? (size_t)t * d.N * d.stage_env_bytes : 0) : nullptr;
    uint8_t* g = (grid_dev && render) ? grid_dev + (every ? (size_t)t * d.N * d.HW : 0) : nullptr;
    int rc = step_impl(h, actions_dev + t * nn, o, b, g, rewards_dev + t * nn, dones_dev + t * nn, x ? &xt : nullptr, stream);
    if (rc) return rc;
  }
  return SNK_OK;
}

extern "C" int snk_step_many(snk_env* h, int32_t num_steps, const uint8_t* actions_dev, uint8_t* obs_dev, uint8_t* bits_dev,
                             int32_t obs_every_step, double* rewards_dev, uint8_t* dones_dev, const snk_step_extra* x,
                             void* stream) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  ON_DEVICE(h);
  return step_many_impl(h, num_steps, actions_dev, obs_dev, bits_dev, nullptr, obs_every_step, rewards_dev, dones_dev, x,
                        (cudaStream_t)stream);
}

extern "C" int snk_step_many_grid(snk_env* h, int32_t num_steps, const uint8_t* actions_dev, uint8_t* obs_dev, uint8_t* bits_dev,
                                  uint8_t* grid_dev, int32_t obs_every_step, double* rewards_dev, uint8_t* dones_dev,
                                  const snk_step_extra* x, void* stream) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  ON_DEVICE(h);
  return step_many_impl(h, num_steps, actions_dev, obs_dev, bits_dev, grid_dev, obs_every_step, rewards_dev, dones_dev, x,
                        (cudaStream_t)stream);
}

extern "C" int snk_reset(snk_env* h, const uint8_t* mask_dev, uint8_t* obs_dev, void* stream) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  ON_DEVICE(h);
  return reset_impl(h, mask_dev, obs_dev, nullptr, nullptr, (cudaStream_t)stream);
}

extern "C" int snk_reset_bits(snk_env* h, const uint8_t* mask_dev, uint8_t* bits_dev, void* stream) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  ON_DEVICE(h);
  return reset_impl(h, mask_dev, nullptr, bits_dev, nullptr, (cudaStream_t)stream);
}

extern "C" int snk_reset_grid(snk_env* h, const uint8_t* mask_dev, uint8_t* obs_dev, uint8_t* bits_dev, uint8_t* grid_dev,
                              void* stream) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  ON_DEVICE(h);
  return reset_impl(h, mask_dev, obs_dev, bits_dev, grid_dev, (cudaStream_t)stream);
}

extern "C" int snk_step(snk_env* h, const uint8_t* actions_dev, uint8_t* obs_dev, double* rewards_dev,
                        uint8_t* dones_dev, const snk_step_extra* x, void* stream) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  ON_DEVICE(h);
  return step_impl(h, actions_dev, obs_dev, nullptr, nullptr, rewards_dev, dones_dev, x, (cudaStream_t)stream);
}

extern "C" int snk_step_bits(snk_env* h, const uint8_t* actions_dev, uint8_t* bits_dev, double* rewards_dev,
                             uint8_t* dones_dev, const snk_step_extra* x, void* stream) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  ON_DEVICE(h);
  return step_impl(h, actions_dev, nullptr, bits_dev, nullptr, rewards_dev, dones_dev, x, (cudaStream_t)stream);
}

extern "C" int snk_step_grid(snk_env* h, const uint8_t* actions_dev, uint8_t* obs_dev, uint8_t* bits_dev, uint8_t* grid_dev,
                             double* rewards_dev, uint8_t* dones_dev, const snk_step_extra* x, void* stream) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  ON_DEVICE(h);
  return step_impl(h, actions_dev, obs_dev, bits_dev, grid_dev, rewards_dev, dones_dev, x, (cudaStream_t)stream);
}

static bool packed(const snk_env* h) { return h->xfer_mode == XFER_PACKED; }

// Device mirrors of the host-buffer calls.  The NHWC mirror (N * obs bytes) exists only for the raw transport;
// the packed transport has the step kernel emit channel bits straight into d_bits (an eighth of the bytes).
static int ensure_mirrors(snk_env* h, bool want_obs, bool want_bits) {
  const Dims& d = h->kp.d;
  if (!h->h_actions) CU(cudaMalloc(&h->h_actions, (size_t)d.N * d.ns));
  if (want_obs && !h->h_obs) CU(cudaMalloc(&h->h_obs, (size_t)d.N * d.obs_env_bytes));
  if (want_bits && !h->d_bits) CU(cudaMalloc(&h->d_bits, (size_t)d.N * d.stage_env_bytes));
  if (!h->h_rew) CU(cudaMalloc(&h->h_rew, (size_t)d.N * d.ns * sizeof(double)));
  if (!h->h_done) CU(cudaMalloc(&h->h_done, (size_t)d.N * d.ns));
  return SNK_OK;
}

// Observation block of the device mirror -> obs_host on stream s.  Raw: one D2H of the NHWC bytes (h_obs).
// Packed: the kernel already wrote channel bits into d_bits; D2H in chunks, widen each chunk on the host pool as
// soon as its copy lands while the next chunks are still on the link.  Returns with the host buffer complete.
static int obs_to_host(snk_env* h, uint8_t* obs_host, cudaStream_t s) {
  const Dims& d = h->kp.d;
  const size_t total = (size_t)d.N * d.obs_env_bytes;
  if (!packed(h)) {
    CU(cudaMemcpyAsync(obs_host, h->h_obs, total, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    return SNK_OK;
  }
  const size_t units = total / 8;
  if (!h->p_bits) CU(cudaMallocHost(&h->p_bits, units));
  if (!h->pool) {
    h->pool = new (std::nothrow) WidenPool(h->xfer_threads > 0 ? h->xfer_threads : default_host_threads());
    if (!h->pool) return fail(SNK_E_NOMEM, "out of host memory");
  }
  size_t chunk = (size_t)8 << 20;
  if ((units + chunk - 1) / chunk > XFER_MAX_CHUNKS) chunk = ((units + XFER_MAX_CHUNKS - 1) / XFER_MAX_CHUNKS + 4095) / 4096 * 4096;
  const int nchunks = (int)((units + chunk - 1) / chunk);
  while (h->n_chunk_ev < nchunks) {
    CU(cudaEventCreateWithFlags(&h->chunk_ev[h->n_chunk_ev], cudaEventDisableTiming));
    ++h->n_chunk_ev;
  }
  for (int c = 0; c < nchunks; ++c) {
    const size_t off = (size_t)c * chunk, len = off + chunk < units ? chunk : units - off;
    CU(cudaMemcpyAsync(h->p_bits + off, h->d_bits + off, len, cudaMemcpyDeviceToHost, s));
    CU(cudaEventRecord(h->chunk_ev[c], s));
  }
  int rc = SNK_OK;
  for (int c = 0; c < nchunks; ++c) {
    const size_t off = (size_t)c * chunk, len = off + chunk < units ? chunk : units - off;
    cudaError_t e = cudaEventSynchronize(h->chunk_ev[c]);
    if (e != cudaSuccess) { rc = fail(SNK_E_CUDA, "cudaEventSynchronize failed: %s", cudaGetErrorString(e)); break; }
    h->pool->submit(h->p_bits + off, obs_host + 8 * off, len);
  }
  h->pool->wait();
  if (rc) return rc;
  CU(cudaStreamSynchronize(s));
  return SNK_OK;
}

// Layout of the single output block used for small batches (all offsets 16-byte aligned).
struct SmallLayout { size_t act, obs, rew, done, extra[N_EXTRA], total; };
static SmallLayout small_layout(const Dims& d) {
  auto up = [](size_t x) { return (x + 15) & ~(size_t)15; };
  const size_t nn = (size_t)d.N * d.ns;
  SmallLayout L;
  L.act = 0;
  L.obs = up(nn);
  L.rew = L.obs + up((size_t)d.N * d.obs_env_bytes);
  L.done = L.rew + up(nn * sizeof(double));
  L.total = L.done + up(nn);
  for (int i = 0; i < N_EXTRA; ++i) {
    L.extra[i] = L.total;
    L.total += up(extra_bytes(d, i));
  }
  return L;
}

static int step_host_small(snk_env* h, const SmallLayout& L, const uint8_t* actions_host, uint8_t* obs_host,
                           double* rewards_host, uint8_t* dones_host, const snk_step_extra* xh) {
  const Dims& d = h->kp.d;
  const size_t nn = (size_t)d.N * d.ns;
  cudaStream_t s = h->own_stream;
  // Zero-copy (default): the block is pinned host memory mapped into the device's address space; the kernel reads
  // the actions from it and writes every output to it over PCIe, so a step is one launch and one synchronise --
  // no copy commands at all (a few KB per step; SNK_SMALL_ZEROCOPY=0 restores copy in / launch / copy out).
  const bool zero_copy = h->small_zero_copy != 0;
  if (!h->small_host) {
    if (zero_copy) {
      CU(cudaHostAlloc((void**)&h->small_host, L.total, cudaHostAllocMapped));
      CU(cudaHostGetDevicePointer((void**)&h->small_map, h->small_host, 0));
    } else {
      CU(cudaMallocHost(&h->small_host, L.total));
    }
  }
  if (!zero_copy && !h->small_dev) CU(cudaMalloc(&h->small_dev, L.total));
  uint8_t* dv = zero_copy ? h->small_map : h->small_dev;
  uint8_t* hv = h->small_host;
  memcpy(hv + L.act, actions_host, nn);
  { int rc0 = own_stream_after_user_work(h); if (rc0) return rc0; }
  if (!zero_copy) CU(cudaMemcpyAsync(dv + L.act, hv + L.act, nn, cudaMemcpyHostToDevice, s));
  ExtraPtrs xdp;                                 // with terminal info, the kernel writes all of it into the block
  for (int i = 0; i < N_EXTRA; ++i) xdp.p[i] = dv + L.extra[i];
  const snk_step_extra xd = extra_struct(xdp);
  int rc = step_impl(h, dv + L.act, obs_host ? dv + L.obs : nullptr, nullptr, nullptr, (double*)(dv + L.rew), dv + L.done, xh ? &xd : nullptr, s);
  if (rc) return rc;
  const size_t lo = obs_host ? L.obs : L.rew, hi = xh ? L.total : L.extra[0];
  if (!zero_copy) CU(cudaMemcpyAsync(hv + lo, dv + lo, hi - lo, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (obs_host) memcpy(obs_host, hv + L.obs, (size_t)d.N * d.obs_env_bytes);
  memcpy(rewards_host, hv + L.rew, nn * sizeof(double));
  memcpy(dones_host, hv + L.done, nn);
  const ExtraPtrs out = extra_ptrs(xh);
  for (int i = 0; i < N_EXTRA; ++i)
    if (out.p[i]) memcpy(out.p[i], hv + L.extra[i], extra_bytes(d, i));
  return SNK_OK;
}

extern "C" int snk_step_host_info(snk_env* h, const uint8_t* actions_host, uint8_t* obs_host,
                                  double* rewards_host, uint8_t* dones_host, const snk_step_extra* xh) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  if (!actions_host || !rewards_host || !dones_host) return fail(SNK_E_INVALID, "actions, rewards and dones are required");
  ON_DEVICE(h);
  {
    const SmallLayout L = small_layout(h->kp.d);
    if (L.total <= 64 * 1024) return step_host_small(h, L, actions_host, obs_host, rewards_host, dones_host, xh);
  }
  const bool as_bits = obs_host && packed(h);  // packed transport: the kernel emits channel bits, no NHWC block at all
  int rc = ensure_mirrors(h, obs_host && !as_bits, as_bits);
  if (rc) return rc;
  rc = own_stream_after_user_work(h);
  if (rc) return rc;
  const Dims& d = h->kp.d;
  const size_t nn = (size_t)d.N * d.ns;
  cudaStream_t s = h->own_stream;
  const ExtraPtrs out = extra_ptrs(xh);
  ExtraPtrs dev = {};                          // device mirrors of the terminal-info outputs the caller asked for
  for (int i = 0; i < N_EXTRA; ++i) {
    if (!out.p[i]) continue;
    if (!h->h_extra[i]) CU(cudaMalloc(&h->h_extra[i], extra_bytes(d, i)));
    dev.p[i] = h->h_extra[i];
  }
  const snk_step_extra xd = extra_struct(dev);
  CU(cudaMemcpyAsync(h->h_actions, actions_host, nn, cudaMemcpyHostToDevice, s));
  rc = step_impl(h, h->h_actions, obs_host && !as_bits ? h->h_obs : nullptr, as_bits ? h->d_bits : nullptr, nullptr, h->h_rew, h->h_done,
                 xh ? &xd : nullptr, s);
  if (rc) return rc;
  CU(cudaMemcpyAsync(rewards_host, h->h_rew, nn * sizeof(double), cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(dones_host, h->h_done, nn, cudaMemcpyDeviceToHost, s));
  for (int i = 0; i < N_EXTRA; ++i)
    if (dev.p[i]) CU(cudaMemcpyAsync(out.p[i], dev.p[i], extra_bytes(d, i), cudaMemcpyDeviceToHost, s));
  if (obs_host) return obs_to_host(h, obs_host, s);
  CU(cudaStreamSynchronize(s));
  return SNK_OK;
}

extern "C" int snk_step_host_bits(snk_env* h, const uint8_t* actions_host, uint8_t* bits_host,
                                  double* rewards_host, uint8_t* dones_host) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  if (!actions_host || !bits_host || !rewards_host || !dones_host) return fail(SNK_E_INVALID, "null argument");
  ON_DEVICE(h);
  int rc = ensure_mirrors(h, false, true);
  if (rc) return rc;
  rc = own_stream_after_user_work(h);
  if (rc) return rc;
  const Dims& d = h->kp.d;
  const size_t nn = (size_t)d.N * d.ns, units = (size_t)d.N * d.stage_env_bytes;
  cudaStream_t s = h->own_stream;
  CU(cudaMemcpyAsync(h->h_actions, actions_host, nn, cudaMemcpyHostToDevice, s));
  rc = step_impl(h, h->h_actions, nullptr, h->d_bits, nullptr, h->h_rew, h->h_done, nullptr, s);   // channel bits straight from the encode
  if (rc) return rc;
  CU(cudaMemcpyAsync(rewards_host, h->h_rew, nn * sizeof(double), cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(dones_host, h->h_done, nn, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(bits_host, h->d_bits, units, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return SNK_OK;
}

extern "C" int snk_step_host(snk_env* h, const uint8_t* actions_host, uint8_t* obs_host,
                             double* rewards_host, uint8_t* dones_host) {
  return snk_step_host_info(h, actions_host, obs_host, rewards_host, dones_host, nullptr);
}

extern "C" int snk_reset_host(snk_env* h, uint8_t* obs_host) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  ON_DEVICE(h);
  const bool as_bits = obs_host && packed(h);
  int rc = ensure_mirrors(h, obs_host && !as_bits, as_bits);
  if (rc) return rc;
  rc = own_stream_after_user_work(h);
  if (rc) return rc;
  cudaStream_t s = h->own_stream;
  rc = reset_impl(h, nullptr, obs_host && !as_bits ? h->h_obs : nullptr, as_bits ? h->d_bits : nullptr, nullptr, s);
  if (rc) return rc;
  if (obs_host) return obs_to_host(h, obs_host, s);
  CU(cudaStreamSynchronize(s));
  return SNK_OK;
}

extern "C" int snk_set_host_transport(snk_env* h, int mode, int threads) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  if (mode != XFER_RAW && mode != XFER_PACKED) return fail(SNK_E_INVALID, "mode must be SNK_XFER_RAW or SNK_XFER_PACKED");
  if (threads < 0 || threads > 256) return fail(SNK_E_INVALID, "threads must be in 0..256");
  h->xfer_mode = mode;
  if (threads != h->xfer_threads) { delete h->pool; h->pool = nullptr; h->xfer_threads = threads; }
  return SNK_OK;
}

extern "C" int snk_get_host_transport(const snk_env* h, int* mode, int* threads) {
  if (!h) return fail(SNK_E_INVALID, "null handle");
  if (mode) *mode = h->xfer_mode;
  if (threads) *threads = h->xfer_threads > 0 ? h->xfer_threads : default_host_threads();
  return SNK_OK;
}

extern "C" int snk_pack_obs(snk_env* h, const uint8_t* obs_dev, uint8_t* bits_dev, size_t n_bytes, void* stream) {
  if (!h || !obs_dev || !bits_dev) return fail(SNK_E_INVALID, "null argument");
  if (((uintptr_t)obs_dev & 15) || ((uintptr_t)bits_dev & 3) || (n_bytes & 7))
    return fail(SNK_E_INVALID, "obs must be 16-byte aligned, bits 4-byte aligned, n_bytes a multiple of 8");
  ON_DEVICE(h);
  CU(launch_pack_obs(obs_dev, bits_dev, n_bytes / 8, (cudaStream_t)stream));
  return SNK_OK;
}

extern "C" int snk_widen_bits_host(const uint8_t* bits_host, uint8_t* obs_host, size_t n_units, int threads) {
  if ((!bits_host || !obs_host) && n_units) return fail(SNK_E_INVALID, "null argument");
  if (threads <= 1) { widen_bits(bits_host, obs_host, n_units); return SNK_OK; }
  WidenPool pool(threads);
  pool.submit(bits_host, obs_host, n_units);
  pool.wait();
  return SNK_OK;
}

// ---- observation blocks in compressible memory ---------------------------------------------------------------------
// The driver API is reached through the runtime's entry-point query, so libsnk.so does not link libcuda and still
// loads on a machine without a GPU driver.
struct DriverVmm {
  decltype(&::cuGetErrorString) error_string = nullptr;
  decltype(&::cuDeviceGetAttribute) device_attribute = nullptr;
  decltype(&::cuMemGetAllocationGranularity) granularity = nullptr;
  decltype(&::cuMemCreate) create = nullptr;
  decltype(&::cuMemGetAllocationPropertiesFromHandle) properties = nullptr;
  decltype(&::cuMemAddressReserve) reserve = nullptr;
  decltype(&::cuMemMap) map = nullptr;
  decltype(&::cuMemSetAccess) set_access = nullptr;
  decltype(&::cuMemUnmap) unmap = nullptr;
  decltype(&::cuMemAddressFree) address_free = nullptr;
  decltype(&::cuMemRelease) release = nullptr;
};
struct ObsAlloc {
  int device;
  size_t size;                                   // mapped bytes (granularity-rounded) of a compressible block
  CUmemGenericAllocationHandle handle;
  bool vmm;                                      // false: the block came from cudaMalloc
};
static std::mutex g_obs_mu;                      // guards everything below
static DriverVmm g_vmm;
static bool g_vmm_loaded = false;
static std::map<uintptr_t, ObsAlloc> g_obs_allocs;   // by base address

template <typename F>
static cudaError_t driver_fn(const char* name, F* fn) {
  cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
  void* p = nullptr;
  cudaError_t e = cudaGetDriverEntryPointByVersion(name, &p, 12000, cudaEnableDefault, &q);
  if (e == cudaSuccess && (q != cudaDriverEntryPointSuccess || !p)) e = cudaErrorSymbolNotFound;
  *fn = reinterpret_cast<F>(p);
  return e;
}

static int load_vmm() {                          // called with g_obs_mu held
  if (g_vmm_loaded) return SNK_OK;
  CU(driver_fn("cuGetErrorString", &g_vmm.error_string));
  CU(driver_fn("cuDeviceGetAttribute", &g_vmm.device_attribute));
  CU(driver_fn("cuMemGetAllocationGranularity", &g_vmm.granularity));
  CU(driver_fn("cuMemCreate", &g_vmm.create));
  CU(driver_fn("cuMemGetAllocationPropertiesFromHandle", &g_vmm.properties));
  CU(driver_fn("cuMemAddressReserve", &g_vmm.reserve));
  CU(driver_fn("cuMemMap", &g_vmm.map));
  CU(driver_fn("cuMemSetAccess", &g_vmm.set_access));
  CU(driver_fn("cuMemUnmap", &g_vmm.unmap));
  CU(driver_fn("cuMemAddressFree", &g_vmm.address_free));
  CU(driver_fn("cuMemRelease", &g_vmm.release));
  g_vmm_loaded = true;
  return SNK_OK;
}

static int drv_fail(CUresult r, const char* what) {
  const char* s = nullptr;
  if (g_vmm.error_string(r, &s) != CUDA_SUCCESS || !s) s = "unknown error";
  return fail(SNK_E_CUDA, "%s failed: %s (%d)", what, s, (int)r);
}
#define DRV(call)                                                                                                \
  do {                                                                                                           \
    CUresult _r = (call);                                                                                        \
    if (_r != CUDA_SUCCESS) return drv_fail(_r, #call);                                                          \
  } while (0)

// A compressible block of `bytes` on `device`: *ptr = nullptr when the driver did not grant compression.
static int alloc_compressible(int device, size_t bytes, void** ptr, ObsAlloc* rec) {
  *ptr = nullptr;
  int supported = 0;
  DRV(g_vmm.device_attribute(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, device));
  if (!supported) return SNK_OK;
  CUmemAllocationProp prop;
  memset(&prop, 0, sizeof prop);
  prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
  prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
  prop.location.id = device;
  prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
  size_t gran = 0;
  DRV(g_vmm.granularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED));
  const size_t size = (bytes + gran - 1) / gran * gran;
  CUmemGenericAllocationHandle handle;
  DRV(g_vmm.create(&handle, size, &prop, 0));
  CUmemAllocationProp got;
  memset(&got, 0, sizeof got);
  CUresult r = g_vmm.properties(&got, handle);
  if (r != CUDA_SUCCESS || got.allocFlags.compressionType != CU_MEM_ALLOCATION_COMP_GENERIC) {
    g_vmm.release(handle);
    if (r != CUDA_SUCCESS) return drv_fail(r, "cuMemGetAllocationPropertiesFromHandle");
    return SNK_OK;                               // not granted: the caller falls back to cudaMalloc
  }
  CUdeviceptr va = 0;
  r = g_vmm.reserve(&va, size, gran, 0, 0);
  if (r != CUDA_SUCCESS) { g_vmm.release(handle); return drv_fail(r, "cuMemAddressReserve"); }
  r = g_vmm.map(va, size, 0, handle, 0);
  if (r != CUDA_SUCCESS) { g_vmm.address_free(va, size); g_vmm.release(handle); return drv_fail(r, "cuMemMap"); }
  CUmemAccessDesc access;
  memset(&access, 0, sizeof access);
  access.location = prop.location;
  access.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
  r = g_vmm.set_access(va, size, &access, 1);
  if (r != CUDA_SUCCESS) {
    g_vmm.unmap(va, size); g_vmm.address_free(va, size); g_vmm.release(handle);
    return drv_fail(r, "cuMemSetAccess");
  }
  *ptr = reinterpret_cast<void*>(va);
  *rec = ObsAlloc{device, size, handle, true};
  return SNK_OK;
}

extern "C" int snk_alloc_obs(int device, size_t bytes, void** ptr_out, int* compressed_out) {
  if (!ptr_out || !compressed_out || !bytes) return fail(SNK_E_INVALID, "null argument or zero size");
  *ptr_out = nullptr;
  *compressed_out = 0;
  DeviceGuard guard(device);
  if (guard.err != cudaSuccess) return fail(SNK_E_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(guard.err));
  std::lock_guard<std::mutex> lock(g_obs_mu);
  int rc = load_vmm();
  if (rc) return rc;
  void* p = nullptr;
  ObsAlloc rec{device, bytes, 0, false};
  rc = alloc_compressible(device, bytes, &p, &rec);
  if (rc) return rc;
  if (!p) CU(cudaMalloc(&p, bytes));
  g_obs_allocs[(uintptr_t)p] = rec;
  *ptr_out = p;
  *compressed_out = rec.vmm ? 1 : 0;
  return SNK_OK;
}

// Whether `p` points into a live compressible block of snk_alloc_obs.
static bool in_compressible_block(const void* p) {
  std::lock_guard<std::mutex> lock(g_obs_mu);
  auto it = g_obs_allocs.upper_bound((uintptr_t)p);
  if (it == g_obs_allocs.begin()) return false;
  --it;
  return it->second.vmm && (uintptr_t)p < it->first + it->second.size;
}

extern "C" int snk_free_obs(void* ptr) {
  if (!ptr) return SNK_OK;
  std::lock_guard<std::mutex> lock(g_obs_mu);
  auto it = g_obs_allocs.find((uintptr_t)ptr);
  if (it == g_obs_allocs.end()) return fail(SNK_E_INVALID, "pointer was not returned by snk_alloc_obs");
  const ObsAlloc rec = it->second;
  g_obs_allocs.erase(it);
  DeviceGuard guard(rec.device);
  if (guard.err != cudaSuccess) return fail(SNK_E_CUDA, "cudaSetDevice(%d): %s", rec.device, cudaGetErrorString(guard.err));
  if (!rec.vmm) {
    CU(cudaFree(ptr));                           // synchronises the device itself
    return SNK_OK;
  }
  CU(cudaDeviceSynchronize());                   // no kernel or copy may still touch the mapping
  const CUdeviceptr va = reinterpret_cast<CUdeviceptr>(ptr);
  DRV(g_vmm.unmap(va, rec.size));
  DRV(g_vmm.address_free(va, rec.size));
  DRV(g_vmm.release(rec.handle));
  return SNK_OK;
}

static StateView to_view(const snk_state_view* v) {
  StateView s;
  s.grid = v->grid; s.head = v->head; s.tail = v->tail; s.length = v->length; s.dir = v->dir; s.alive = v->alive;
  s.alive_counter = v->alive_counter; s.episode_length = v->episode_length; s.cells = v->cells; s.max_cells = v->max_cells;
  return s;
}

extern "C" int snk_get_state(snk_env* h, const snk_state_view* out, void* stream) {
  if (!h || !out) return fail(SNK_E_INVALID, "null argument");
  if (out->cells && out->max_cells < 1) return fail(SNK_E_INVALID, "max_cells must be >= 1 when cells is given");
  ON_DEVICE(h);
  const MapView mv = {h->kp.pool, h->kp.cur_map, nullptr, h->kp.num_maps};
  CU(launch_get_state(h->kp.d, h->kp.recs, h->kp.base_grid, mv, h->kp.err, to_view(out), (cudaStream_t)stream));
  note_user_stream(h, (cudaStream_t)stream);
  return SNK_OK;
}

extern "C" int snk_set_state(snk_env* h, const snk_state_view* in, uint8_t* obs_dev, void* stream) {
  if (!h || !in) return fail(SNK_E_INVALID, "null argument");
  if (!in->grid || !in->alive || !in->dir || !in->cells || !in->length || !in->alive_counter || !in->episode_length || in->max_cells < 2)
    return fail(SNK_E_INVALID, "set_state needs grid, alive, dir, cells, length, alive_counter, episode_length");
  KParams p;
  const int rc = call_params(h, p, MODE_ENCODE, nullptr, obs_dev, nullptr, nullptr, nullptr, nullptr, nullptr);
  if (rc) return rc;
  ON_DEVICE(h);
  const MapView mv = {h->kp.pool, h->kp.next_map, h->kp.cur_map, h->kp.num_maps};
  CU(launch_set_state(h->kp.d, h->kp.recs, h->kp.base_grid, mv, h->kp.err, to_view(in), (cudaStream_t)stream));
  CU(launch_tile_kernel(p, h->threads, h->smem_bytes, (cudaStream_t)stream));
  note_user_stream(h, (cudaStream_t)stream);
  h->was_reset = true;
  return SNK_OK;
}

// ---- per-env snapshot / restore on the device: slots of SnapHdr + raw record + frame history (snapshot_slot_bytes)
extern "C" size_t snk_snapshot_bytes(const snk_env* h) { return h ? snapshot_slot_bytes(h->kp.d) : 0; }

extern "C" int snk_snapshot(snk_env* h, const int32_t* env_ids_dev, int32_t count, void* snap_dev, void* stream) {
  if (!h || !snap_dev) return fail(SNK_E_INVALID, "null argument");
  if (!h->was_reset) return fail(SNK_E_STATE, "snapshot before reset");
  if ((uintptr_t)snap_dev & 15) return fail(SNK_E_INVALID, "snap must be 16-byte aligned");
  if (count < 1 || count > h->kp.d.N) return fail(SNK_E_INVALID, "count must be in 1..%d", h->kp.d.N);
  ON_DEVICE(h);
  const KParams& p = h->kp;
  CU(launch_snapshot(p.d, p.recs, p.hist, p.cur_map, env_ids_dev, count, h->snap_digest, (uint8_t*)snap_dev, p.err,
                     (cudaStream_t)stream));
  note_user_stream(h, (cudaStream_t)stream);
  return SNK_OK;
}

extern "C" int snk_restore(snk_env* h, const int32_t* src_dev, int32_t num_slots, const void* snap_dev, uint8_t* obs_dev,
                           uint8_t* bits_dev, uint8_t* grid_dev, void* stream) {
  if (!h || !src_dev || !snap_dev) return fail(SNK_E_INVALID, "null argument");
  if (!h->was_reset) return fail(SNK_E_STATE, "restore before reset");
  if ((uintptr_t)snap_dev & 15) return fail(SNK_E_INVALID, "snap must be 16-byte aligned");
  if (num_slots < 1) return fail(SNK_E_INVALID, "num_slots must be >= 1");
  ON_DEVICE(h);
  const Dims& d = h->kp.d;
  const bool out = obs_dev || bits_dev || grid_dev;
  KParams p;                                     // the observation's launch: the encode of the restored envs only
  if (out && d.fs == 1) {
    const int rc = call_params(h, p, MODE_ENCODE, nullptr, obs_dev, bits_dev, grid_dev, nullptr, nullptr, nullptr);
    if (rc) return rc;
    p.mask = h->restore_mask;
  } else if (obs_dev && ((uintptr_t)obs_dev & 7)) {
    return fail(SNK_E_INVALID, "obs must be 8-byte aligned");
  }
  cudaStream_t s = (cudaStream_t)stream;
  CU(launch_restore(d, h->kp.recs, h->kp.hist, h->kp.cur_map, src_dev, num_slots, (const uint8_t*)snap_dev, h->snap_digest,
                    h->restore_mask, h->kp.err, s));
  // frame_stack 1: MODE_ENCODE rebuilds each restored env's grid from its record (and cur_map) and encodes it; it skips
  // the other envs and writes no record byte that differs.  frame_stack > 1: its F_INIT would refill the history, so
  // the restored ring is widened as it stands.
  if (out && d.fs == 1) CU(launch_tile_kernel(p, h->threads, h->smem_bytes, s));
  if (out && d.fs > 1) {
    const MapView mv = {h->kp.pool, h->kp.cur_map, nullptr, h->kp.num_maps};
    CU(launch_emit_stacked(d, h->kp.recs, h->kp.hist, h->kp.base_grid, mv, h->restore_mask, obs_dev, bits_dev, grid_dev,
                           h->kp.err, s));
  }
  note_user_stream(h, s);
  return SNK_OK;
}

// ---- exact checkpoint: the raw records (grid, snakes, counters, Philox event, replay cursor, statistics),
// the frame histories and the rollout statistics vector, byte for byte
static const uint64_t CKPT_MAGIC = 0x0031544B434B4E53ull;     // "SNKCKT1"
// A handle with a wall-map pool writes its own magic and appends the pool's digest, next_map and cur_map, so its blob
// and that of a handle without a pool never load into each other.
static const uint64_t CKPT_MAGIC_POOL = 0x0031504B434B4E53ull;  // "SNKCKP1"
struct CkptHeader { uint64_t magic; int32_t N, H, W, ns, K, V, fs, dig, rec_bytes, hist_env_bytes; double env_steps; };   // rec_bytes: per env in HBM

static size_t ckpt_pool_bytes(const snk_env* h) { return h->kp.num_maps ? sizeof(uint64_t) + 2 * (size_t)h->kp.d.N : 0; }

extern "C" size_t snk_checkpoint_bytes(const snk_env* h) {
  if (!h) return 0;
  return sizeof(CkptHeader) + (size_t)h->kp.d.N * ((size_t)h->kp.d.hbm_rec_bytes + (size_t)h->kp.d.hist_env_bytes) + STAT_COUNT * sizeof(double) +
         ckpt_pool_bytes(h);
}

extern "C" int snk_checkpoint_save(snk_env* h, void* blob_host, size_t bytes) {
  if (!h || !blob_host) return fail(SNK_E_INVALID, "null argument");
  if (bytes < snk_checkpoint_bytes(h)) return fail(SNK_E_INVALID, "checkpoint buffer too small: %zu < %zu", bytes, snk_checkpoint_bytes(h));
  ON_DEVICE(h);
  CU(cudaDeviceSynchronize());
  const Dims& d = h->kp.d;
  uint8_t* out = (uint8_t*)blob_host;
  CkptHeader hd = {h->kp.num_maps ? CKPT_MAGIC_POOL : CKPT_MAGIC, d.N, d.H, d.W, d.ns, d.K, d.V, d.fs, d.dig | (d.compact << 1),
                   d.hbm_rec_bytes, d.hist_env_bytes, 0.0};
  memcpy(out, &hd, sizeof hd); out += sizeof hd;
  CU(cudaMemcpy(out, h->kp.recs, (size_t)d.N * d.hbm_rec_bytes, cudaMemcpyDeviceToHost)); out += (size_t)d.N * d.hbm_rec_bytes;
  if (d.hist_env_bytes) { CU(cudaMemcpy(out, h->kp.hist, (size_t)d.N * d.hist_env_bytes, cudaMemcpyDeviceToHost)); out += (size_t)d.N * d.hist_env_bytes; }
  CU(cudaMemcpy(out, h->kp.stats, STAT_COUNT * sizeof(double), cudaMemcpyDeviceToHost));
  if (h->kp.num_maps) {
    out += STAT_COUNT * sizeof(double);
    memcpy(out, &h->pool_digest, sizeof(uint64_t)); out += sizeof(uint64_t);
    CU(cudaMemcpy(out, h->kp.next_map, (size_t)d.N, cudaMemcpyDeviceToHost)); out += d.N;
    CU(cudaMemcpy(out, h->kp.cur_map, (size_t)d.N, cudaMemcpyDeviceToHost));
  }
  return SNK_OK;
}

extern "C" int snk_checkpoint_load(snk_env* h, const void* blob_host, size_t bytes) {
  if (!h || !blob_host) return fail(SNK_E_INVALID, "null argument");
  if (bytes < snk_checkpoint_bytes(h)) return fail(SNK_E_INVALID, "checkpoint too small for this handle");
  const Dims& d = h->kp.d;
  const uint8_t* in = (const uint8_t*)blob_host;
  CkptHeader hd;
  memcpy(&hd, in, sizeof hd); in += sizeof hd;
  if (hd.magic != (h->kp.num_maps ? CKPT_MAGIC_POOL : CKPT_MAGIC) && (hd.magic == CKPT_MAGIC || hd.magic == CKPT_MAGIC_POOL))
    return fail(SNK_E_INVALID, h->kp.num_maps ? "checkpoint was written by a handle without a wall-map pool"
                                           : "checkpoint was written by a handle with a wall-map pool");
  if (hd.magic != (h->kp.num_maps ? CKPT_MAGIC_POOL : CKPT_MAGIC) || hd.N != d.N || hd.H != d.H || hd.W != d.W || hd.ns != d.ns || hd.K != d.K || hd.V != d.V ||
      hd.fs != d.fs || hd.dig != (d.dig | (d.compact << 1)) || hd.rec_bytes != d.hbm_rec_bytes || hd.hist_env_bytes != d.hist_env_bytes)
    return fail(SNK_E_INVALID, "checkpoint was written by a handle of a different shape");
  const uint8_t* pool_part = in + (size_t)d.N * ((size_t)d.hbm_rec_bytes + (size_t)d.hist_env_bytes) + STAT_COUNT * sizeof(double);
  if (h->kp.num_maps) {
    uint64_t digest;
    memcpy(&digest, pool_part, sizeof digest);
    if (digest != h->pool_digest) return fail(SNK_E_INVALID, "checkpoint was written by a handle with a different wall-map pool");
    const uint8_t* cur = pool_part + sizeof(uint64_t) + d.N;
    for (int e = 0; e < d.N; ++e)
      if (cur[e] >= h->kp.num_maps) return fail(SNK_E_INVALID, "checkpoint: cur_map[%d] = %d names no map", e, cur[e]);
  }
  ON_DEVICE(h);
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(h->kp.recs, in, (size_t)d.N * d.hbm_rec_bytes, cudaMemcpyHostToDevice)); in += (size_t)d.N * d.hbm_rec_bytes;
  if (d.hist_env_bytes) { CU(cudaMemcpy(h->kp.hist, in, (size_t)d.N * d.hist_env_bytes, cudaMemcpyHostToDevice)); in += (size_t)d.N * d.hist_env_bytes; }
  CU(cudaMemcpy(h->kp.stats, in, STAT_COUNT * sizeof(double), cudaMemcpyHostToDevice));
  if (h->kp.num_maps) {
    CU(cudaMemcpy(const_cast<uint8_t*>(h->kp.next_map), pool_part + sizeof(uint64_t), (size_t)d.N, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(h->kp.cur_map, pool_part + sizeof(uint64_t) + d.N, (size_t)d.N, cudaMemcpyHostToDevice));
  }
  h->was_reset = true;
  return SNK_OK;
}

extern "C" int snk_set_replay(snk_env* h, const int32_t* draws_host, const int64_t* offsets_host) {
  if (!h || !offsets_host) return fail(SNK_E_INVALID, "null argument");
  if (h->kp.d.rng_mode != RNG_REPLAY) return fail(SNK_E_STATE, "handle was not created with SNK_RNG_REPLAY");
  ON_DEVICE(h);
  const int N = h->kp.d.N;
  const int64_t total = offsets_host[N];
  if (offsets_host[0] != 0 || total < 0) return fail(SNK_E_INVALID, "offsets must start at 0 and be non-decreasing");
  for (int e = 0; e < N; ++e) if (offsets_host[e + 1] < offsets_host[e]) return fail(SNK_E_INVALID, "offsets must be non-decreasing");
  CU(cudaDeviceSynchronize());
  cudaFree(const_cast<int32_t*>(h->kp.replay)); h->kp.replay = nullptr;
  int32_t* replay = nullptr;
  CU(cudaMalloc(&replay, (size_t)(total > 0 ? total : 1) * sizeof(int32_t)));
  h->kp.replay = replay;                         // every later launch copies the template, so it reads the new stream
  if (total > 0) {
    if (!draws_host) return fail(SNK_E_INVALID, "null draws");
    CU(cudaMemcpy(replay, draws_host, (size_t)total * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  CU(cudaMemcpy(const_cast<int64_t*>(h->kp.replay_off), offsets_host, ((size_t)N + 1) * sizeof(int64_t), cudaMemcpyHostToDevice));
  // cursors live in the records: zero them
  CU(cudaMemset2D(h->kp.recs + h->kp.d.hbm_c0 + (h->kp.d.off_hdr - h->kp.d.off_c0) + offsetof(EnvHdr, cursor), (size_t)h->kp.d.hbm_rec_bytes, 0,
                  sizeof(uint32_t), (size_t)N));
  return SNK_OK;
}

extern "C" int snk_replay_cursors(snk_env* h, int32_t* cursors_host) {
  if (!h || !cursors_host) return fail(SNK_E_INVALID, "null argument");
  ON_DEVICE(h);
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy2D(cursors_host, sizeof(int32_t), h->kp.recs + h->kp.d.hbm_c0 + (h->kp.d.off_hdr - h->kp.d.off_c0) + offsetof(EnvHdr, cursor),
                  (size_t)h->kp.d.hbm_rec_bytes,
                  sizeof(int32_t), (size_t)h->kp.d.N, cudaMemcpyDeviceToHost));
  return SNK_OK;
}

extern "C" int snk_device_errors(snk_env* h, uint32_t* bits, int clear) {
  if (!h || !bits) return fail(SNK_E_INVALID, "null argument");
  ON_DEVICE(h);
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(bits, h->kp.err, sizeof(uint32_t), cudaMemcpyDeviceToHost));
  if (clear) CU(cudaMemset(h->kp.err, 0, sizeof(uint32_t)));
  return SNK_OK;
}

extern "C" int snk_stats_dev(snk_env* h, double** stats_dev) {
  if (!h || !stats_dev) return fail(SNK_E_INVALID, "null argument");
  *stats_dev = h->kp.stats;
  return SNK_OK;
}

extern "C" int snk_stats(snk_env* h, double* out_host, int clear) {
  if (!h || !out_host) return fail(SNK_E_INVALID, "null argument");
  ON_DEVICE(h);
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(out_host, h->kp.stats, STAT_COUNT * sizeof(double), cudaMemcpyDeviceToHost));
  if (clear) CU(cudaMemset(h->kp.stats, 0, STAT_COUNT * sizeof(double)));
  return SNK_OK;
}

extern "C" int64_t snk_spawn_count(int32_t H, int32_t W, int32_t K) {
  if (H < 3 || W < 3 || K < 1 || K > MAX_SNAKE_LENGTH) { fail(SNK_E_INVALID, "bad spawn table shape"); return -1; }
  const int64_t n = spawn_enumerate(H, W, K, nullptr, nullptr, 0, SPAWN_TABLE_LIMIT);
  if (n > SPAWN_TABLE_LIMIT) { fail(SNK_E_INVALID, "more than %lld spawn poses", (long long)SPAWN_TABLE_LIMIT); return -1; }
  return n;
}

extern "C" int snk_spawn_cells(int32_t H, int32_t W, int32_t K, int32_t* out, int64_t count) {
  if (!out || H < 3 || W < 3 || K < 1 || K > MAX_SNAKE_LENGTH) return fail(SNK_E_INVALID, "bad argument");
  spawn_enumerate(H, W, K, nullptr, out, count);
  return SNK_OK;
}

extern "C" int64_t snk_spawn_count_map(int32_t H, int32_t W, int32_t K, const uint8_t* walls_host) {
  if (!walls_host || H < 3 || W < 3 || K < 1 || K > MAX_SNAKE_LENGTH) { fail(SNK_E_INVALID, "bad spawn table shape"); return -1; }
  const int64_t n = spawn_enumerate(H, W, K, nullptr, nullptr, 0, SPAWN_TABLE_LIMIT, walls_host);
  if (n > SPAWN_TABLE_LIMIT) { fail(SNK_E_INVALID, "more than %lld spawn poses", (long long)SPAWN_TABLE_LIMIT); return -1; }
  return n;
}

extern "C" int snk_spawn_cells_map(int32_t H, int32_t W, int32_t K, const uint8_t* walls_host, int32_t* out, int64_t count) {
  if (!out || !walls_host || H < 3 || W < 3 || K < 1 || K > MAX_SNAKE_LENGTH) return fail(SNK_E_INVALID, "bad argument");
  spawn_enumerate(H, W, K, nullptr, out, count, 0, walls_host);
  return SNK_OK;
}
