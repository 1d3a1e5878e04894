// snk_core.cuh -- record layout, Philox stream and the per-environment Snake-v1 step logic.
//
// Everything here is SNK_HD (host + device): the CUDA kernels in snk_kernels.cu call these
// functions on environment records staged in shared memory; tests/hostsim compiles the very same
// source with g++ so the rule implementation can be checked against the golden vectors on a box
// without a GPU.  (That host build is test infrastructure; libsnk.so never runs env logic on
// the CPU.)
//
// Reference lines (relative to /root/reference/marlenv/marlenv/) are cited at each rule.
#pragma once
#include <stdint.h>
#include <stdlib.h>

#if defined(__CUDACC__)
#define SNK_HD __host__ __device__ __forceinline__
#else
#define SNK_HD inline
#endif

namespace snk {

// cell codes: type + 10*owner                                        core/snake.py:5-11
enum : int { EMPTY = 0, WALL = 1, FRUIT = 2, HEAD = 3, BODY = 4, TAIL = 5 };
// direction codes 0 UP(-1,0) 1 RIGHT(0,1) 2 DOWN(1,0) 3 LEFT(0,-1)    core/snake.py:33-37
enum : int { RNG_PHILOX = 0, RNG_REPLAY = 1 };
enum : uint32_t { ERR_BAD_ACTION = 1, ERR_REPLAY_UNDERRUN = 2, ERR_REPLAY_RANGE = 4, ERR_SPAWN_GIVEUP = 8,
                  ERR_INTERNAL = 16,       // a bounds / alignment check of the debug build (-DSNK_DEBUG_CHECKS) failed
                  ERR_TMA_TIMEOUT = 32,    // a record tile's bulk copy did not land within two seconds; tile skipped
                  ERR_STATE = 64,          // compact records: set_state grid is not walls + fruits + live snakes, or more
                                           // fruit cells than the record has slots for
                  ERR_MAP_RANGE = 128,     // wall-map pool: a map id was not below the number of maps; map 0 was used
                  ERR_SNAPSHOT = 256 };    // snapshot of an env id outside [0, N), or restore from a slot index out of
                                           // range or a slot of another configuration; that env was left unchanged
enum : int { DRAW_STEP_FRUIT = 0, DRAW_SPAWN = 1, DRAW_RESET_FRUIT = 2 };
enum : int { STAT_EPISODES = 0, STAT_RETURN, STAT_EP_STEPS, STAT_FRUITS, STAT_KILLS, STAT_DEATHS,
             STAT_ENV_STEPS, STAT_COUNT = 8 };

constexpr int MAX_SNAKES = 25;        // 10*24+5 = 245 fits a uint8 cell
constexpr int MAX_SNAKE_LENGTH = 25;  // 16-bit head + 24 two-bit links in one 64-bit table entry
constexpr int MAX_FRUIT_DRAWS = 32;   // one warp lane per draw
constexpr uint32_t SPAWN_ATTEMPT_CAP = 1u << 16;

// Per-step flag bits kept in the scratch area while a step is resolved.
enum : uint8_t { ST_WAS_ALIVE = 1, ST_DIED = 2, ST_ATE = 4, ST_WON = 8, ST_EATER = 16 };

struct EnvHdr {            // per-environment scalars inside the record (16 bytes)
  int16_t alive_counter;   // SnakeEnv.alive_snakes: signed, drifts below the true count (:334-345).  A snake dies once
                           // per episode and is counted at most twice, so the value stays within [-ns, ns]
  uint8_t hpos;            // frame-stack ring: slot that holds the oldest frame / gets the next one (< fs <= 64)
  uint8_t pad;
  uint32_t episode_length; // SnakeEnv.episode_length (:392)
  uint32_t event;          // Philox event counter: +1 per step and per explicit reset
  uint32_t cursor;         // replay-stream cursor
};
static_assert(sizeof(EnvHdr) == 16, "EnvHdr is part of the record layout");

// Everything a kernel needs to know about the configuration; passed by value.
struct Dims {
  int32_t N, H, W, HW, ns, K, V, fs, nfruits;
  int32_t oh, ow, ohw;            // observation window
  int32_t ohw_p;                  // history row stride (ohw rounded up to 16)
  int32_t auto_reset, done_mode, rng_mode;
  int32_t observer;               // 0 'snake': three relative actions; 1 'human': five absolute actions
  int32_t dig;                    // 1: body directions live in bits 6..7 of the grid byte (cell codes < 64, i.e.
                                  //    at most 6 snakes) and the record has no direction plane
  int32_t code_mask;              // 63 when dig, else 255: grid byte -> cell code
  int32_t stat16;                 // 1: the per-snake episode counters (steps, fruits, kills) are uint16 -- they are
                                  //    bounded by the step cap, which then is <= 65535 (the default is 1e4) -- else uint32
  int32_t compact;                // 1: the record kept in HBM is the working record WITHOUT its grid: the grid is a function
                                  //    of the rest (wall layout + fruit cells + the live snakes' bodies, which the direction
                                  //    plane spells out from tail to head) and is rebuilt in shared memory when a tile is
                                  //    loaded.  Implies the direction plane (dig == 0) and a fruit slot list in the record.
  int32_t fcap;                   // compact: fruit slots per environment (uint16 cell + 1, 0 = free)
  // working-record layout (bytes from the record start; grid is at 0).  rec_bytes is the working record; the part from
  // off_c0 on ("c-part": plane, snake table, header, statistics, fruit slots) is what a compact handle keeps in HBM
  int32_t off_dirp, off_snk, off_hdr, off_stats, off_fruit, rec_bytes;
  int32_t off_c0;                 // start of the c-part inside the working record (= round_up(HW, 16))
  int32_t hbm_rec_bytes;          // bytes per environment in HBM: rec_bytes, or rec_bytes - off_c0 when compact
  int32_t hbm_c0;                 // offset of the c-part inside the HBM record: off_c0, or 0 when compact
  int32_t hist_env_bytes;         // ns*fs*ohw_p, 0 when fs == 1
  int32_t stage_env_bytes;        // ns*ohw*fs  (staging area per env, output order)
  int32_t obs_env_bytes;          // ns*ohw*fs*8
  int32_t scr_bytes;              // per-env scratch: tgt u16[ns], st u8[ns], kl u8[ns], tdir u8[ns], padded to 8
  // zero-bordered copy of a grid for the ENC_PAD encode: (H + 2V) rows of pad_pitch bytes, grid column c at
  // byte pad_left + c; pad_left >= V is a multiple of 4 and pad_pitch / 4 is odd (rows rotate through the banks)
  int32_t pad_pitch, pad_left, pad_env_bytes;
  uint32_t n_cand;
  uint32_t seed_lo, seed_hi, env_off_lo, env_off_hi;
  double r_fruit, r_kill, r_lose, r_win, r_time, max_steps;
};

SNK_HD int round_up(int x, int m) { return (x + m - 1) / m * m; }

inline void finalize_layout(Dims& d) {
  d.HW = d.H * d.W;
  if (d.V > 0) { d.oh = d.ow = 2 * d.V + 1; } else { d.oh = d.H; d.ow = d.W; }
  d.ohw = d.oh * d.ow;
  d.ohw_p = round_up(d.ohw, 16);
  if (d.compact) d.dig = 0;
  d.code_mask = d.dig ? 63 : 255;
  d.off_dirp = round_up(d.HW, 16);
  d.off_c0 = d.off_dirp;
  d.off_snk = d.off_dirp + (d.dig ? 0 : round_up((d.HW + 3) / 4, 16));
  d.off_hdr = d.off_snk + round_up(8 * d.ns, 16);
  d.off_stats = d.off_hdr + (int)sizeof(EnvHdr);
  d.stat16 = d.max_steps <= 65535.0 ? 1 : 0;
  d.off_fruit = d.off_stats + round_up((8 + (d.stat16 ? 6 : 12)) * d.ns, 16);
  // A step can add a fruit without removing one (two heads meeting on a fruit: both die, the fruit stays and one more
  // is drawn, C3) -- at most once per two deaths, so nfruits + ns / 2 cells bound an episode; ns more for set_state
  d.fcap = d.compact ? round_up(d.nfruits + d.ns, 8) : 0;      // <= 32 + 25 -> at most 64: two slots per warp lane
  d.rec_bytes = d.off_fruit + round_up(2 * d.fcap, 16);
  d.hbm_rec_bytes = d.compact ? d.rec_bytes - d.off_c0 : d.rec_bytes;
  d.hbm_c0 = d.compact ? 0 : d.off_c0;
  d.hist_env_bytes = d.fs > 1 ? d.ns * d.fs * d.ohw_p : 0;
  d.stage_env_bytes = d.ns * d.ohw * d.fs;
  d.obs_env_bytes = d.stage_env_bytes * 8;
  d.scr_bytes = round_up(5 * d.ns, 8);
  d.pad_left = round_up(d.V, 4);
  d.pad_pitch = round_up(d.pad_left + d.W + d.V, 4);
  if (((d.pad_pitch >> 2) & 1) == 0) d.pad_pitch += 4;
  d.pad_env_bytes = round_up((d.H + 2 * d.V) * d.pad_pitch, 16);
}

// ---- record field accessors ---------------------------------------------------------------------
struct Rec {
  uint8_t* grid;
  uint8_t* dirp;
  uint16_t* head;
  uint16_t* tail;
  uint16_t* len;
  uint8_t* dir;
  uint8_t* alive;
  EnvHdr* hdr;
  double* score;
  uint8_t* cnt;              // episode counters [3][ns] (steps, fruits, kills), uint16 or uint32 (Dims::stat16)
  uint16_t* fruit;           // compact: fcap fruit slots, cell + 1 or 0
};
enum : int { CNT_STEPS = 0, CNT_FRUITS = 1, CNT_KILLS = 2 };

// g: the grid, c: the c-part (working-record offsets minus off_c0).  A contiguous working record has c == g + off_c0;
// a compact handle keeps the two in separate shared-memory areas (and only the c-part in HBM).
SNK_HD Rec rec_view2(uint8_t* g, uint8_t* c, const Dims& d) {
  Rec r;
  uint8_t* base = c - d.off_c0;
  r.grid = g;
  r.dirp = base + d.off_dirp;
  r.head = (uint16_t*)(base + d.off_snk);
  r.tail = r.head + d.ns;
  r.len = r.tail + d.ns;
  r.dir = (uint8_t*)(r.len + d.ns);
  r.alive = r.dir + d.ns;
  r.hdr = (EnvHdr*)(base + d.off_hdr);
  r.score = (double*)(base + d.off_stats);
  r.cnt = (uint8_t*)(r.score + d.ns);
  r.fruit = (uint16_t*)(base + d.off_fruit);
  return r;
}
SNK_HD Rec rec_view(uint8_t* base, const Dims& d) { return rec_view2(base, base + d.off_c0, d); }
SNK_HD uint32_t cnt_get(const Dims& d, const Rec& r, int field, int i) {
  const int k = field * d.ns + i;
  return d.stat16 ? (uint32_t)((const uint16_t*)r.cnt)[k] : ((const uint32_t*)r.cnt)[k];
}
SNK_HD void cnt_set(const Dims& d, const Rec& r, int field, int i, uint32_t v) {
  const int k = field * d.ns + i;
  if (d.stat16) ((uint16_t*)r.cnt)[k] = (uint16_t)v; else ((uint32_t*)r.cnt)[k] = v;
}
// one snake's step: +1 step, +ate fruits, +kl kills
SNK_HD void cnt_step(const Dims& d, const Rec& r, int i, uint32_t ate, uint32_t kl) {
  cnt_set(d, r, CNT_STEPS, i, cnt_get(d, r, CNT_STEPS, i) + 1u);
  if (ate) cnt_set(d, r, CNT_FRUITS, i, cnt_get(d, r, CNT_FRUITS, i) + ate);
  if (kl) cnt_set(d, r, CNT_KILLS, i, cnt_get(d, r, CNT_KILLS, i) + kl);
}
SNK_HD void stats_zero(const Dims& d, const Rec& r, int i) {
  r.score[i] = 0.0;
  cnt_set(d, r, CNT_STEPS, i, 0u); cnt_set(d, r, CNT_FRUITS, i, 0u); cnt_set(d, r, CNT_KILLS, i, 0u);
}

// body-direction plane: 2 bits per cell = the direction the owning snake left the cell in
// (i.e. toward its head).  Equivalent to Snake.directions (core/snake.py:71, 96-107).
SNK_HD int dirp_get(const uint8_t* dirp, int c) { return (dirp[c >> 2] >> ((c & 3) * 2)) & 3; }
SNK_HD void dirp_set(uint8_t* dirp, int c, int v) {
  const int sh = (c & 3) * 2;
  dirp[c >> 2] = (uint8_t)((dirp[c >> 2] & ~(3 << sh)) | (v << sh));
}
SNK_HD int dir_delta(int dir, int W) { return dir == 0 ? -W : dir == 1 ? 1 : dir == 2 ? W : -1; }

// With at most 6 snakes every cell code (type + 10*owner <= 55) fits 6 bits, so the 2-bit direction of a
// BODY / TAIL cell rides in bits 6..7 of its grid byte and the plane is dropped from the record ("dig").
// EMPTY / WALL / FRUIT / HEAD bytes carry no direction bits, so an empty cell is still exactly 0.
// SNK_NO_COMPACT=1 keeps the whole working record (grid included) in HBM -- the round-1 layout, kept for A/B runs.
inline int default_compact() {
  const char* off = getenv("SNK_NO_COMPACT");
  return (off && *off == '1') ? 0 : 1;
}
inline int default_dig(int ns) {
  const char* off = getenv("SNK_NO_DIG");
  return (10 * (ns - 1) + 5 < 64 && !(off && *off == '1')) ? 1 : 0;
}
SNK_HD uint32_t cell_code(const Dims& d, uint32_t grid_byte) { return grid_byte & (uint32_t)d.code_mask; }
SNK_HD int body_dir(const Dims& d, const Rec& r, int c) { return d.dig ? (r.grid[c] >> 6) : dirp_get(r.dirp, c); }
// single-writer contexts only (host simulation, thread-per-environment kernels)
SNK_HD void set_body_dir(const Dims& d, const Rec& r, int c, int v) {
  if (d.dig) r.grid[c] = (uint8_t)((r.grid[c] & 63) | (v << 6));
  else dirp_set(r.dirp, c, v);
}

// observer='snake': 0 keep, 1 turn left, 2 turn right (the exact table of the reference's trigonometric
// _next_direction, snake_env.py:598-608; a > 2 is the reference's KeyError, reported by the caller).
SNK_HD int turn_relative(int dir, uint32_t a) { return (dir + (a == 1u ? 3 : a == 2u ? 1 : 0)) & 3; }
// observer='human': 0 noop, 1 left, 2 right, 3 down, 4 up; a horizontal mover may only turn down/up, a
// vertical one only left/right, anything else keeps the direction      snake_env.py:610-632
SNK_HD int turn_absolute(int dir, uint32_t a) {
  if (dir & 1) return a == 3u ? 2 : a == 4u ? 0 : dir;     // RIGHT / LEFT
  return a == 1u ? 3 : a == 2u ? 1 : dir;                  // UP / DOWN
}

// ---- Philox4x32-10 counter-based stream ----------------------------------------------------------
// word(seed; env, event, purpose, idx): counter = {env_lo, env_hi ^ 'SNK1', event, purpose<<24 | idx/4},
// key = seed; the idx%4-th output word.  Bounded draw: mulhi(word, n).
SNK_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

SNK_HD void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = mulhi32(M0, c[0]), lo0 = M0 * c[0];
    const uint32_t hi1 = mulhi32(M1, c[2]), lo1 = M1 * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += W0; k1 += W1;
  }
}

// The stream parameters by value: functions that receive the configuration by reference (out-of-line device
// functions read it through generic loads) copy them once instead of reloading them around every store.
struct StreamKey { uint32_t seed_lo, seed_hi, env_off_lo, env_off_hi; };
SNK_HD StreamKey stream_key(const Dims& d) { StreamKey k = {d.seed_lo, d.seed_hi, d.env_off_lo, d.env_off_hi}; return k; }

SNK_HD uint32_t draw_word(const StreamKey& sk, uint32_t env_local, uint32_t event, int purpose, uint32_t idx) {
  const uint64_t gid = ((uint64_t)sk.env_off_hi << 32 | sk.env_off_lo) + env_local;
  uint32_t c[4] = {(uint32_t)gid, (uint32_t)(gid >> 32) ^ 0x534E4B31u, event,
                   ((uint32_t)purpose << 24) | (idx >> 2)};
  philox4x32_10(c, sk.seed_lo, sk.seed_hi);
  const uint32_t k = idx & 3u;                 // select chain: a dynamic index would put c[] in local memory
  return k == 0u ? c[0] : k == 1u ? c[1] : k == 2u ? c[2] : c[3];
}
SNK_HD uint32_t draw_word(const Dims& d, uint32_t env_local, uint32_t event, int purpose, uint32_t idx) {
  return draw_word(stream_key(d), env_local, event, purpose, idx);
}

SNK_HD uint32_t draw_below(const StreamKey& sk, uint32_t env_local, uint32_t event, int purpose, uint32_t idx, uint32_t n) {
  return mulhi32(draw_word(sk, env_local, event, purpose, idx), n);
}
SNK_HD uint32_t draw_below(const Dims& d, uint32_t env_local, uint32_t event, int purpose, uint32_t idx,
                           uint32_t n) {
  return mulhi32(draw_word(d, env_local, event, purpose, idx), n);
}

// ---- spawn table entry: bits 0..15 head cell, then (K-1) two-bit links head->tail ----------------
// link j (j = 1..K-1) = direction from body cell j-1 to body cell j.
SNK_HD int spawn_head(uint64_t e) { return (int)(e & 0xFFFF); }
SNK_HD int spawn_link(uint64_t e, int j) { return (int)((e >> (16 + 2 * (j - 1))) & 3); }

// ---- observation encoding ------------------------------------------------------------------------
// One cell as seen by viewer v -> 8 channel bits: 0 WALL, 1 FRUIT, 2/3/4 other HEAD/BODY/TAIL,
// 5/6/7 own HEAD/BODY/TAIL                                            envs/snake_env.py:474-496
SNK_HD uint32_t cell_bits(uint32_t code, uint32_t v) {
  const uint32_t owner = (code * 205u) >> 11;        // code / 10 for code < 1029
  const uint32_t kind = code - owner * 10u;
  if (kind == 0) return 0u;
  uint32_t ch = kind - 1u;
  if (kind >= 3u && owner == v) ch += 3u;
  return 1u << ch;
}

// 4 bits -> 4 bytes of 0/1 (bit i -> byte i)
SNK_HD uint32_t spread4(uint32_t nib) { return (nib * 0x00204081u) & 0x01010101u; }

// ---- the step rules for ONE environment ----------------------------------------------------------
struct StepResult {
  uint8_t fruit_taken;   // fruit draws owed after the moves (:377)
  uint8_t finished;      // episode ended this step (:396)
  uint8_t deaths;
};

// scr: tgt u16[ns] | st u8[ns] | kl u8[ns] | tdir u8[ns]
// act: ns actions; rew/done: ns outputs.
SNK_HD StepResult env_step_logic(const Dims& d, uint8_t* rec_base, uint8_t* scr, const uint8_t* act,
                                 double* rew, uint8_t* done, uint32_t* err_bits) {
  Rec r = rec_view(rec_base, d);
  const int ns = d.ns, W = d.W;
  uint16_t* tgt = (uint16_t*)scr;
  uint8_t* st = scr + 2 * ns;
  uint8_t* kl = st + ns;
  uint8_t* tdir = kl + ns;
  StepResult out;
  out.fruit_taken = 0; out.finished = 0; out.deaths = 0;

  // 1. relative turn + head advance for live snakes                     snake_env.py:320-330, 598-608
  for (int i = 0; i < ns; ++i) {
    st[i] = 0; kl[i] = 0; tgt[i] = 0xFFFF;
    if (r.alive[i]) {
      uint32_t a = act[i];
      if (a > 2u && !d.observer) { *err_bits |= ERR_BAD_ACTION; a = 0; }
      const int nd = d.observer ? turn_absolute(r.dir[i], a) : turn_relative(r.dir[i], a);
      r.dir[i] = (uint8_t)nd;
      tgt[i] = (uint16_t)(r.head[i] + dir_delta(nd, W));
      st[i] = ST_WAS_ALIVE;
    }
  }

  // 2. collisions against the pre-move grid, one verdict per distinct target cell    :521-544
  int counter = r.hdr->alive_counter;
  int fruit_taken = 0, ndead = 0;
  for (int i = 0; i < ns; ++i) {
    if (!(st[i] & ST_WAS_ALIVE)) continue;
    const uint32_t code = cell_code(d, r.grid[tgt[i]]);
    const uint32_t owner = (code * 205u) >> 11;
    const uint32_t kind = code - owner * 10u;
    int n = 0; bool first = true;
    for (int j = 0; j < ns; ++j)
      if ((st[j] & ST_WAS_ALIVE) && tgt[j] == tgt[i]) { ++n; if (j < i) first = false; }
    const bool lethal = (kind == WALL) | (kind == BODY) | (kind == HEAD);
    if (n > 1 || lethal) {
      st[i] |= ST_DIED; ++ndead;
      if (first) {
        if (kind == FRUIT) ++fruit_taken;                  // fruit stays, a draw is still owed (C3)
        if ((kind == BODY || kind == HEAD) && owner < (uint32_t)ns) ++kl[owner];   // once per cell (C2)
      }
    } else if (kind == FRUIT) {
      st[i] |= ST_EATER; ++fruit_taken;
    }
  }

  // 3. death bookkeeping, tail-growth rule, win rule                                  :334-352
  counter -= ndead;
  for (int i = 0; i < ns; ++i) if (st[i] & ST_DIED) r.alive[i] = 0;
  for (int e = 0; e < ns; ++e) {
    if (!(st[e] & ST_EATER)) continue;
    const uint16_t t = r.tail[e];
    for (int j = 0; j < ns; ++j)
      if ((st[j] & ST_WAS_ALIVE) && tgt[j] == t) {         // may already be dead: counted again (C4)
        st[j] |= ST_DIED; r.alive[j] = 0; --counter; ++kl[e];
      }
    st[e] |= ST_ATE;
  }
  if (counter == 1 && ns > 1)
    for (int i = 0; i < ns; ++i) if (r.alive[i]) { st[i] |= ST_WON; break; }
  r.hdr->alive_counter = counter;

  // The direction stored with a tail cell is read before any snake moves: in this sequential walk an
  // earlier snake's head may already sit in a later snake's vacated tail cell (:555) and, when directions
  // ride in the grid byte, would have overwritten it.
  for (int i = 0; i < ns; ++i) tdir[i] = (st[i] & ST_WAS_ALIVE) ? (uint8_t)body_dir(d, r, r.tail[i]) : 0;

  // 4. rewards (float64, fixed order, no FMA) and sequential grid update              :358-374, :546-566
  int n_alive = 0, n_done = 0;
  for (int i = 0; i < ns; ++i) {
    double rw = 0.0;
    if (st[i] & ST_WAS_ALIVE) {
      const bool alive = r.alive[i] != 0;
      const bool ate = (st[i] & ST_ATE) != 0, died = (st[i] & ST_DIED) != 0, won = (st[i] & ST_WON) != 0;
#if defined(__CUDA_ARCH__)
      rw = __dmul_rn(d.r_time, alive ? 1.0 : 0.0);
      rw = __dadd_rn(rw, __dmul_rn(d.r_fruit, ate ? 1.0 : 0.0));
      rw = __dadd_rn(rw, __dmul_rn(d.r_lose, died ? 1.0 : 0.0));
      rw = __dadd_rn(rw, __dmul_rn(d.r_kill, (double)kl[i]));
      rw = __dadd_rn(rw, __dmul_rn(d.r_win, won ? 1.0 : 0.0));
#else
      volatile double acc = d.r_time * (alive ? 1.0 : 0.0);
      volatile double term = d.r_fruit * (ate ? 1.0 : 0.0); acc = acc + term;
      term = d.r_lose * (died ? 1.0 : 0.0); acc = acc + term;
      term = d.r_kill * (double)kl[i]; acc = acc + term;
      term = d.r_win * (won ? 1.0 : 0.0); acc = acc + term;
      rw = acc;
#endif
      const int tag = 10 * i;
      if (alive) {                                         // _update_grid, live branch      :548-559
        const int oh = r.head[i];
        r.grid[oh] = (uint8_t)(BODY + tag);
        set_body_dir(d, r, oh, r.dir[i]);
        if (!ate) {
          const int ot = r.tail[i];
          const int nt = ot + dir_delta(tdir[i], W);
          if (cell_code(d, r.grid[ot]) == (uint32_t)(TAIL + tag)) r.grid[ot] = EMPTY;   // may already hold another head (:555)
          r.tail[i] = (uint16_t)nt;
        } else {
          r.len[i] = (uint16_t)(r.len[i] + 1);
        }
        r.head[i] = tgt[i];
        r.grid[tgt[i]] = (uint8_t)(HEAD + tag);
        r.grid[r.tail[i]] = (uint8_t)((TAIL + tag) | (d.dig ? (r.grid[r.tail[i]] & 0xC0) : 0));   // keeps the cell's direction
        // episode statistics gate on this step's done flags                                 :385-389
#if defined(__CUDA_ARCH__)
        r.score[i] = __dadd_rn(r.score[i], rw);
#else
        { volatile double s = r.score[i] + rw; r.score[i] = s; }
#endif
        cnt_step(d, r, i, ate ? 1u : 0u, (uint32_t)kl[i]);
        ++n_alive;
      } else {                                             // died this step: erase own cells :560-566
        int c = r.tail[i];
        const int hd = r.head[i];
        bool is_tail = true;
        for (int guard = 0; guard < d.HW; ++guard) {
          const int nxt = c + dir_delta(is_tail ? (int)tdir[i] : body_dir(d, r, c), W);
          if (!(is_tail && (int)((cell_code(d, r.grid[c]) * 205u) >> 11) != i)) r.grid[c] = EMPTY;
          if (c == hd) break;
          c = nxt; is_tail = false;
        }
        r.len[i] = 0;
        ++out.deaths;
      }
    }
    rew[i] = rw;
    const uint8_t dn = r.alive[i] ? 0 : 1;
    done[i] = dn;
    n_done += dn;
  }
  (void)n_alive;

  // 5. step cap and episode end                                                        :391-412
  r.hdr->episode_length += 1;
  const bool capped = (double)r.hdr->episode_length >= d.max_steps;
  if (capped) { for (int i = 0; i < ns; ++i) done[i] = 1; n_done = ns; }
  const bool fin = d.done_mode == 0 ? (n_done == ns) : (n_done > 0);
  if (fin && d.done_mode == 1) for (int i = 0; i < ns; ++i) done[i] = 1;   // coop_snake_env.py:16-20
  out.fruit_taken = (uint8_t)fruit_taken;
  out.finished = fin ? 1 : 0;
  return out;
}

// Sequential k-th-empty-cell lookup (host simulation and single-thread fallbacks).  Row-major rank
// over grid == 0, as np.where(grid == 0) enumerates it                      core/grid_util.py:126-133
SNK_HD int nth_empty_seq(const uint8_t* grid, int HW, int rank) {
  for (int c = 0; c < HW; ++c)
    if (grid[c] == EMPTY) { if (rank == 0) return c; --rank; }
  return -1;
}
SNK_HD int count_empty_seq(const uint8_t* grid, int HW) {
  int n = 0;
  for (int c = 0; c < HW; ++c) n += grid[c] == EMPTY;
  return n;
}

// Paint the walled empty box                                              core/grid_util.py:14-20
SNK_HD uint8_t wall_or_empty(int c, int H, int W) {
  const int rr = c / W, cc = c - rr * W;
  return (rr == 0 || rr == H - 1 || cc == 0 || cc == W - 1) ? (uint8_t)WALL : (uint8_t)EMPTY;
}

// Standard competition rank on descending score: 1 + #(scores strictly greater)   snake_env.py:397-404
SNK_HD int competition_rank(const double* score, int ns, int i) {
  int rk = 1;
  for (int j = 0; j < ns; ++j) rk += score[j] > score[i];
  return rk;
}

}  // namespace snk
