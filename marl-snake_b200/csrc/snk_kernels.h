// snk_kernels.h -- internal interface between the C-ABI layer (snk_api.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "snk_core.cuh"

// Launch bounds: tight bounds let ptxas keep the encode loop free of spills (48 registers at 128).
#define SNK_MAX_THREADS 128
#define SNK_MAX_THREADS_COOP 256

namespace snk {

enum : int { MODE_STEP = 0, MODE_RESET = 1, MODE_ENCODE = 2 };
// frame_stack 1 encode flavours (chosen per handle by encode_flavour):
//   ENC_LEGACY  window-cell table in shared memory, or plain index arithmetic for windows wider than 16
//   ENC_REG     egocentric window of at most 127 cells: the four window cells a lane owns live in registers
//               as packed words, one packed word per viewer (crop origin + invalid rows/columns) is
//               prepared by the rule warp -- no table loads, no per-viewer origin arithmetic
//   ENC_DIRECT  full-grid observation: window cell == grid cell
//   ENC_PAD     cooperative tiles, egocentric window of at most 255 cells, grid width a multiple of 4: the CTA
//               copies each grid into a zero-bordered plane with a bank-conflict-free pitch (Dims::pad_*), so a
//               window cell is origin + constant offset -- no validity masks, no window table, one byte load
//               and one LUT row per cell; the offsets of the cells a lane owns live in registers
enum : int { ENC_LEGACY = 0, ENC_REG = 1, ENC_DIRECT = 2, ENC_PAD = 3 };
constexpr int TILE_AUX_BYTES = 48 + 128;   // per tile: flags (32 B), mbarrier (8 B), pad, viewer words (32 x 4 B)

struct KParams {
  Dims d;
  // resident state
  uint8_t* recs;               // [N] records, rec_bytes each
  uint8_t* hist;               // [N, ns, fs, ohw_p] channel-bit frames (fs > 1 only)
  const uint64_t* spawn;       // [n_cand] packed spawn poses
  const uint32_t* wall_map;    // custom wall layout: the H*W cell codes (EMPTY / WALL) a reset starts from, as words; null = walled box
  const uint8_t* base_grid;    // compact handles: the wall layout (walled box or custom map), off_c0 bytes per copy, as many
                               //   copies back to back as a tile has environments -- one bulk copy paints a tile's grids
  const int32_t* replay;       // replay draws, all envs back to back
  const int64_t* replay_off;   // [N+1]
  uint32_t* err;               // sticky error bits
  double* stats;               // [STAT_COUNT]
  // per-call I/O
  const uint8_t* actions;
  uint8_t* obs;                // uint8 NHWC observation block, or null
  uint8_t* bits;               // channel-bit observation block [N, ns, oh, ow, fs] (one byte per cell and frame), or null
  double* rew;
  uint8_t* done;
  uint8_t* fin;
  int32_t* rank;
  double* ep_scores;
  int32_t* ep_steps;
  int32_t* ep_fruits;
  int32_t* ep_kills;
  const uint8_t* mask;
  int32_t mode;
  int32_t E;                   // environments per tile: 32 / group size, or fewer (a power of two) in coop mode
  int32_t vec16;               // every environment's observation block is 16-byte aligned (fs > 1 path, ENC_REG viewer pairs)
  int32_t force_generic;       // run the unspecialised kernel instance (tests)
  const uint8_t* enc_blob;     // fs == 1: host-built encode tables (see encode_blob_fill)
  int32_t enc_blob_bytes;
  int32_t enc_tab_off;         // byte offset of the window-cell table inside the blob
  int32_t enc_lutb_off;        // fs == 1: byte offset of the channel-bit byte LUT inside the blob
  int32_t use_tab;
  int32_t lut_dual;            // fs == 1: {as-other, as-own} LUT pair instead of one LUT per viewer
  int32_t coop;                // CTA-cooperative tile (small batches / large records)
  int32_t use_tma;             // move the record tile with cp.async.bulk (TMA) instead of LDG/STG
  int32_t enc_flavour;         // ENC_* (fs == 1)
  int32_t enc_copy_bytes;      // bytes of the blob the kernel stages (the table is skipped when unused)
  uint32_t inv_grid_words;     // ENC_PAD: ceil(2^32 / (H*W/4)) and ceil(2^32 / (W/4)): exact division of word indices
  uint32_t inv_row_words;      //          below 2^16 by a multiply-high
  int32_t pdl;                 // launch with programmatic stream serialization (SNK_PDL=0 switches it off)
  int32_t l2_keep;             // record tiles are loaded and stored with an L2 evict_last hint (SNK_L2_KEEP)
  float l2_keep_frac;          //   fraction of those lines the policy applies to
  int32_t bigreg;              // warp-private tiles, batch many waves deep: run the instance compiled without a register cap
  int32_t T;                   // steps per launch (snk_step_many; frame_stack 1).  actions / rewards / dones / extras are
  int32_t obs_every_step;      //   [T, ...]; obs / bits are [T, ...] when obs_every_step, else the last step's block only
  // wall-map pool (snk_create_maps); pool == null for every other handle, which then runs the instances without it
  const uint8_t* pool;         // [num_maps][off_c0] wall layouts (cell codes EMPTY / WALL, zero padded)
  const uint2* map_tab;        // [num_maps] {first pose in `spawn`, number of poses} of each map's spawn table
  const uint8_t* next_map;     // [N] map a reset of env e starts from (written by the caller)
  uint8_t* cur_map;            // [N] map of env e's current episode (written by every reset)
  int32_t num_maps;
  // global state (snk_*_grid): [N, H*W] cell codes of every environment's grid as the observation was encoded from it
  // ([T, N, H*W] when obs_every_step), or null -- and then the instances without it run
  uint8_t* grid_out;
};

struct StateView {
  uint8_t* grid; int32_t* head; int32_t* tail; int32_t* length; uint8_t* dir; uint8_t* alive;
  int32_t* alive_counter; int32_t* episode_length; int32_t* cells; int32_t max_cells;
};

int tile_group(int ns);
size_t tile_smem_bytes(const Dims& d, int warps, bool coop, int tile_envs);
bool encode_lut_dual(const Dims& d);
bool encode_uses_table(const Dims& d);
int encode_flavour(const Dims& d, bool coop);
size_t pad_plane_bytes(const Dims& d, int tile_envs);     // ENC_PAD: padded planes of one tile
size_t encode_blob_bytes(const Dims& d, size_t* tab_off, size_t* lutb_off);
void encode_blob_fill(const Dims& d, uint8_t* out);
cudaError_t launch_tile_kernel(const KParams& p, int threads, size_t smem_bytes, cudaStream_t stream);
// Wall layout of each environment: base_grid for every environment, or -- wall-map pool -- pool slot map_ids[e]
// (cur_map for get_state, next_map for set_state, which also copies it to cur_map)
struct MapView { const uint8_t* pool; const uint8_t* map_ids; uint8_t* cur_out; int32_t num_maps; };
cudaError_t launch_get_state(const Dims& d, const uint8_t* recs, const uint8_t* base_grid, const MapView& mv, uint32_t* err,
                             const StateView& sv, cudaStream_t s);
cudaError_t launch_set_state(const Dims& d, uint8_t* recs, const uint8_t* base_grid, const MapView& mv, uint32_t* err,
                             const StateView& sv, cudaStream_t s);
cudaError_t launch_init_records(const Dims& d, uint8_t* recs, cudaStream_t s);

// Snapshot slot (snk_snapshot / snk_restore): this header, the env's HBM record (hbm_rec_bytes), then its frame history
// (hist_env_bytes, frame_stack > 1).  Every part is a multiple of 16 bytes.  digest 0 marks a slot that matches no handle.
struct SnapHdr { uint64_t digest; uint8_t cur_map; uint8_t pad[7]; };
static_assert(sizeof(SnapHdr) == 16, "a snapshot slot is moved in 16-byte units");
inline size_t snapshot_slot_bytes(const Dims& d) { return sizeof(SnapHdr) + (size_t)d.hbm_rec_bytes + (size_t)d.hist_env_bytes; }
// slot i := env ids[i] (ids null: env i), i < count.  cur_map null: a handle without a wall-map pool
cudaError_t launch_snapshot(const Dims& d, const uint8_t* recs, const uint8_t* hist, const uint8_t* cur_map, const int32_t* ids,
                            int count, uint64_t digest, uint8_t* snap, uint32_t* err, cudaStream_t s);
// env e := slot src[e] where src[e] >= 0; mask[e] := 1 where it was restored, else 0
cudaError_t launch_restore(const Dims& d, uint8_t* recs, uint8_t* hist, uint8_t* cur_map, const int32_t* src, int num_slots,
                           const uint8_t* snap, uint64_t digest, uint8_t* mask, uint32_t* err, cudaStream_t s);
// frame_stack > 1: observation (obs NHWC and / or channel bits) of every env with mask[e] != 0, widened from its history
// ring as the step that wrote it returned it, and its grid row (grid null: none)
cudaError_t launch_emit_stacked(const Dims& d, const uint8_t* recs, const uint8_t* hist, const uint8_t* base_grid,
                                const MapView& mv, const uint8_t* mask, uint8_t* obs, uint8_t* bits, uint8_t* grid,
                                uint32_t* err, cudaStream_t s);
// obs: n_units * 8 bytes of 0/1 (16-byte aligned) -> bits: n_units bytes, bit c = byte c of the unit
cudaError_t launch_pack_obs(const uint8_t* obs, uint8_t* bits, size_t n_units, cudaStream_t s);

// host-side spawn table (snk_spawn.cpp)
// walls: [H*W] bytes, nonzero = wall, or null for make_grid's walled box
int64_t spawn_enumerate(int H, int W, int K, uint64_t* packed_out, int32_t* cells_out, int64_t cap, int64_t limit = 0,
                        const uint8_t* walls = nullptr);
constexpr int64_t SPAWN_TABLE_LIMIT = (int64_t)64 << 20;     // poses (512 MB of table); more is refused

}  // namespace snk
