/* snk.h -- C ABI of the B200-native batched Snake-v1 step path (libsnk.so).
 *
 * The reference (tranthai189765/MARL-Snake, a fork of kc-ml2/marlenv) is pure
 * Python and has no FFI for this path: its boundary is the gym.Env protocol of
 * `SnakeEnv` reached through `make_snake` / `gym.make('Snake-v1')`.  Every entry
 * point below states the reference interface it stands in for (paths relative to
 * /root/reference/marlenv/marlenv/).  INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add.
 *
 * Conventions: plain pointers and sizes only, no torch types.  Every call
 * returns 0 on success or a negative SNK_E_* code; snk_last_error() gives the
 * message for the calling thread.  Pointers named *_dev are CUDA device pointers
 * on the handle's device, *_host are host pointers.  `stream` is a cudaStream_t
 * passed as void* (NULL = legacy default stream); device-pointer calls only
 * enqueue work on it and never synchronise.  The *_host calls run on a stream
 * owned by the handle, first wait (on the device) for whatever the most recent
 * device-pointer call of this handle left on its stream, and synchronise before
 * they return -- so device-pointer and host-buffer calls may be mixed freely as
 * long as consecutive device-pointer calls use one stream (or are ordered by the
 * caller).  Every call leaves the calling thread's current CUDA device unchanged.
 * A handle is not thread-safe.
 *
 * Batched layouts (N = num_envs, ns = num_snakes, oh x ow = observation window):
 *   actions  uint8  [N, ns]             0 keep, 1 turn left, 2 turn right (observer 'snake');
 *                                       0 noop, 1 left, 2 right, 3 down, 4 up (observer 'human')
 *   obs      uint8  [N, ns, oh, ow, 8*frame_stack]   NHWC, values 0/1, frames oldest->newest
 *   rewards  double [N, ns]
 *   dones    uint8  [N, ns]
 */
#ifndef SNK_H_
#define SNK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNK_ABI_VERSION 1

enum {
  SNK_OK = 0,
  SNK_E_INVALID = -1,   /* bad argument / unsupported configuration            */
  SNK_E_CUDA = -2,      /* a CUDA runtime call failed                          */
  SNK_E_NOMEM = -3,
  SNK_E_STATE = -4      /* call not valid in the handle's current mode         */
};

/* sticky per-handle device error bits, read with snk_device_errors() */
enum {
  SNK_DEV_BAD_ACTION = 1,        /* observer 'snake': action outside {0,1,2} (reference: KeyError,
                                    snake_env.py:606); 'human' ignores unknown actions as the reference does */
  SNK_DEV_REPLAY_UNDERRUN = 2,   /* replay stream exhausted                                         */
  SNK_DEV_REPLAY_RANGE = 4,      /* replayed draw out of range / replayed spawn overlaps            */
  SNK_DEV_SPAWN_GIVEUP = 8,      /* no overlap-free spawn found within the attempt cap               */
  SNK_DEV_INTERNAL = 16,         /* a bounds / alignment check failed (debug build, -DSNK_DEBUG_CHECKS) */
  SNK_DEV_TMA_TIMEOUT = 32,      /* a record tile's bulk copy did not complete within 2 s; that tile was not stepped */
  SNK_DEV_STATE = 64,            /* snk_set_state: the grid is not the handle's walls + fruit cells + the live snakes'
                                    bodies (the resident record stores only those), or it holds more fruit cells than
                                    the record has slots (num_fruits + num_snakes, rounded up to 8); with a
                                    wall-map pool, in either record layout: its walls are not those of next_map */
  SNK_DEV_MAP_RANGE = 128,       /* wall-map pool: a map id (next_map, or cur_map rewritten by the caller) was not below
                                    the number of maps; map 0 was used instead                          */
  SNK_DEV_SNAPSHOT = 256         /* snk_snapshot: an env id outside [0, N) (its slot matches no handle); snk_restore: a slot
                                    index neither -1 nor below num_slots, or a slot of a handle whose digest differs --
                                    that env was left unchanged and its observation not written          */
};

enum { SNK_RNG_PHILOX = 0, SNK_RNG_REPLAY = 1 };
enum { SNK_OBSERVER_SNAKE = 0, SNK_OBSERVER_HUMAN = 1 };

/* Constructor arguments of SnakeEnv.__init__ (envs/snake_env.py:58-88) plus batching. */
typedef struct snk_config {
  int32_t abi_version;        /* must be SNK_ABI_VERSION                                   */
  int32_t device;             /* CUDA device ordinal                                        */
  int32_t num_envs;           /* N: environments resident on this device                   */
  int32_t height, width;      /* grid_shape, walls included (snake_env.py:60-61)           */
  int32_t num_snakes;         /* 1..25 (cell code 10*idx+type must fit uint8)               */
  int32_t snake_length;       /* initial length, 2..25 (snake_env.py:63)                    */
  int32_t vision_range;       /* 0 = full-grid observation (None / 0 in the reference)     */
  int32_t frame_stack;        /* >= 1 (snake_env.py:65)                                     */
  int32_t num_fruits;         /* <0: int(round(0.8*num_snakes)) (snake_env.py:87-88); <=32 */
  int32_t auto_reset;         /* 1: reset an env inside the step that ends it and return
                                 the reset observation (wrappers.py:138-146)                */
  int32_t done_mode;          /* 0: all(dones) ends the episode (snake_env.py:416);
                                 1: any(dones) (coop_snake_env.py:14-22)                    */
  int32_t rng_mode;           /* SNK_RNG_PHILOX or SNK_RNG_REPLAY                           */
  int32_t observer;           /* SNK_OBSERVER_SNAKE: actions 0 keep, 1 left, 2 right relative to the heading
                                 (_next_direction, snake_env.py:598-608); SNK_OBSERVER_HUMAN: 0 noop, 1 left,
                                 2 right, 3 down, 4 up in grid terms (_next_direction_global, :610-632)   */
  uint64_t seed;              /* Philox key                                                 */
  uint64_t env_id_offset;     /* global id of env 0: streams are keyed by global env id so a
                                 sharded run equals the single-device run                   */
  double max_episode_steps;   /* episode_length >= this forces all dones (snake_env.py:393)*/
  double reward_fruit, reward_kill, reward_lose, reward_win, reward_time;   /* :46-52      */
} snk_config;

typedef struct snk_env snk_env;   /* opaque handle: one shard of environments on one GPU */

/* Optional per-step outputs; any pointer may be NULL.  Device pointers. */
typedef struct snk_step_extra {
  uint8_t* finished;          /* [N]     1 where the episode ended this step (info emitted, :396) */
  int32_t* rank;              /* [N, ns] info['rank'] of envs with finished=1 (:397-404)          */
  double*  episode_scores;    /* [N, ns] info['episode_scores'] (:407)                            */
  int32_t* episode_steps;     /* [N, ns] info['episode_steps']  (integral in the reference)       */
  int32_t* episode_fruits;    /* [N, ns] info['episode_fruits']                                   */
  int32_t* episode_kills;     /* [N, ns] info['episode_kills']                                    */
} snk_step_extra;

/* Full environment state, the parity interface (reference: SnakeEnv.grid, .snakes[i].coords /
 * .direction / .alive, .alive_snakes, .episode_length).  Device pointers, any may be NULL.  */
typedef struct snk_state_view {
  uint8_t* grid;              /* [N, H*W]  cell codes type + 10*owner (core/snake.py:5-11)   */
  int32_t* head;              /* [N, ns]   flat cell index r*W+c, -1 for dead snakes          */
  int32_t* tail;              /* [N, ns]                                                      */
  int32_t* length;            /* [N, ns]   0 for dead snakes                                  */
  uint8_t* dir;               /* [N, ns]   0 UP 1 RIGHT 2 DOWN 3 LEFT (core/snake.py:33-37)   */
  uint8_t* alive;             /* [N, ns]                                                      */
  int32_t* alive_counter;     /* [N]       SnakeEnv.alive_snakes (signed, drifts: :334-345)   */
  int32_t* episode_length;    /* [N]                                                          */
  int32_t* cells;             /* [N, ns, max_cells] head-first body cells, -1 padded          */
  int32_t  max_cells;
} snk_state_view;

/* ---- lifecycle ------------------------------------------------------------------------------ */

/* SnakeEnv.__init__ for N environments (snake_env.py:58-129) + make_snake batching (wrappers.py:203-223).
 * Builds the spawn-candidate table (core/grid_util.py:73-115) and allocates all device state. */
int snk_create(const snk_config* cfg, snk_env** out);
/* The same with a custom wall layout instead of make_grid's walled box: walls_host is uint8 [height * width], row-major,
 * nonzero = WALL -- the array make_grid_from_txt(map_path, {'#': 1, '.': 0}) returns (core/grid_util.py:23-33; maps
 * under assets/).  Every reset starts from this layout, the spawn poses are enumerated on it (dfs_sweep_empty takes
 * any grid, :73-99) and fruits land on its empty cells.  The outer ring must be wall (SNK_E_INVALID otherwise): the
 * reference would let a snake walk out of the array there.  The map is copied; walls_host may be freed after the call. */
int snk_create_map(const snk_config* cfg, const uint8_t* walls_host, snk_env** out);
/* A POOL of num_maps wall layouts (1..SNK_MAX_MAPS), all height x width: walls_host is uint8 [num_maps, height, width],
 * each map following the rules of snk_create_map (nonzero = WALL, outer ring all wall, at least num_snakes spawn poses;
 * SNK_E_INVALID names the first map that breaks one).  Every environment has two map ids (uint8 [N] device arrays,
 * snk_map_ids_dev):
 *   next_map[e]  the map env e's next reset starts from -- every reset until it is rewritten.  The caller may rewrite it
 *                on the device between any two calls (e.g. fill it with random ids after every step to draw a fresh map
 *                for each auto-reset);
 *   cur_map[e]   the map of env e's current episode.  Every reset -- snk_reset / _bits (masked or not), the auto-reset of
 *                a step, snk_reset_host, snk_set_state -- sets it to next_map[e]; nothing else changes it.
 * map_ids_host: the initial next_map (uint8 [N], every id < num_maps), or NULL for (env_id_offset + e) % num_maps, so a
 * sharded run equals the single-device run.  A reset on map m draws its spawn pose from map m's table with the same
 * Philox counters as snk_create_map (a pool of identical maps gives that handle's trajectories); replayed spawn indices
 * index map m's table.  An id >= num_maps found at a reset reads as map 0 and raises SNK_DEV_MAP_RANGE. */
#define SNK_MAX_MAPS 256
int snk_create_maps(const snk_config* cfg, int32_t num_maps, const uint8_t* walls_host, const uint8_t* map_ids_host,
                    snk_env** out);
/* Device pointers of next_map and cur_map (uint8 [N] each) of a pool handle; SNK_E_STATE for a handle without a pool. */
int snk_map_ids_dev(snk_env* env, uint8_t** next_dev, uint8_t** cur_dev);
/* Number of maps in the handle's pool, 0 for a handle without one. */
int snk_num_maps(const snk_env* env);
/* SnakeEnv.close (snake_env.py:298) */
int snk_destroy(snk_env* env);
const char* snk_last_error(void);
int snk_abi_version(void);

/* observation_space.shape (snake_env.py:115-129): out[4] = {ns, oh, ow, 8*frame_stack} */
int snk_obs_shape(const snk_env* env, int32_t out[4]);
size_t snk_obs_bytes(const snk_env* env);       /* N * prod(shape) */
int snk_num_envs(const snk_env* env);
/* bytes the step kernel must move per env-step (state read+write, history, obs, I/O): the
 * algorithmic-traffic figure bench.py uses for the roofline (DESIGN.md section 4). */
size_t snk_algorithmic_bytes_per_env_step(const snk_env* env);

/* ---- the hot path --------------------------------------------------------------------------- */

/* SnakeEnv.reset (snake_env.py:131-159) for every env, or for envs with mask_dev[e] != 0.
 * Writes the initial stacked observation of the reset envs into obs_dev (NULL = skip). */
int snk_reset(snk_env* env, const uint8_t* mask_dev, uint8_t* obs_dev, void* stream);

/* SnakeEnv.step (snake_env.py:301-414) for all N envs, with the vector worker's auto-reset
 * (wrappers.py:138-146) when cfg.auto_reset.  One kernel launch on `stream`. */
int snk_step(snk_env* env, const uint8_t* actions_dev, uint8_t* obs_dev, double* rewards_dev,
             uint8_t* dones_dev, const snk_step_extra* extra, void* stream);

/* The same two calls delivering the observation as CHANNEL BITS: bits_dev is uint8 [N, ns, oh, ow, frame_stack],
 * one byte per window cell and frame, bit c = channel c of _encode (snake_env.py:484-492) -- i.e.
 * np.packbits(obs.reshape(..., frame_stack, 8), axis=-1, bitorder='little').  The encode writes them directly (no
 * NHWC block, an eighth of the observation traffic): the format for device-side replay buffers and for shipping
 * observations over PCIe.  snk_pack_obs gives the same bytes from an NHWC block. */
int snk_reset_bits(snk_env* env, const uint8_t* mask_dev, uint8_t* bits_dev, void* stream);
int snk_step_bits(snk_env* env, const uint8_t* actions_dev, uint8_t* bits_dev, double* rewards_dev,
                  uint8_t* dones_dev, const snk_step_extra* extra, void* stream);

/* num_steps consecutive snk_step calls as ONE call, for callers whose actions do not depend on the intermediate
 * observations (random or scripted rollouts, replaying recorded action streams, open-loop evaluation):
 *   actions_dev [T, N, ns], rewards_dev [T, N, ns], dones_dev [T, N, ns]; every non-NULL pointer of `extra` is
 *   [T, ...] likewise (finished [T, N], rank [T, N, ns], ...);
 *   obs_dev / bits_dev (either or both may be NULL): [T, N, ...] when obs_every_step != 0, else only the last
 *   step's block [N, ...] is written.
 * Bit-identical to T single steps.  frame_stack 1: one kernel launch -- a tile's records are loaded into shared memory
 * once, stepped T times there and written back once, so a small batch (BASELINE cfg2: 4 096 envs) is no longer bound
 * by T launch latencies and 2 x T record transfers.  frame_stack > 1: T launches (the frame history is per step). */
int snk_step_many(snk_env* env, int32_t num_steps, const uint8_t* actions_dev, uint8_t* obs_dev, uint8_t* bits_dev,
                  int32_t obs_every_step, double* rewards_dev, uint8_t* dones_dev, const snk_step_extra* extra,
                  void* stream);

/* GLOBAL STATE for centralized critics and mixers (MAPPO, QMIX, ...): the three calls above, plus grid_dev, uint8
 * [N, H*W] row-major -- the format of snk_state_view.grid, i.e. the reference's SnakeEnv.grid (cell codes
 * type + 10 * owner, no direction bits).  Row e is env e's grid as the returned observation was encoded from it: for
 * an env that auto-reset in this step, the grid of the new episode; after a masked reset, every env's row (the
 * others' unchanged grids); with a wall-map pool, on the walls of the env's cur_map.  The step kernel stores the rows
 * from shared memory as it stores the records, so no second launch reads the records again.  obs_dev, bits_dev and
 * grid_dev may each be NULL, in any combination; grid_dev may have any alignment (16-byte aligned is fastest).
 * snk_step_many_grid: grid_dev is [T, N, H*W] when obs_every_step != 0, else the last step's [N, H*W].  With grid_dev
 * NULL each call equals its counterpart. */
int snk_reset_grid(snk_env* env, const uint8_t* mask_dev, uint8_t* obs_dev, uint8_t* bits_dev, uint8_t* grid_dev,
                   void* stream);
int snk_step_grid(snk_env* env, const uint8_t* actions_dev, uint8_t* obs_dev, uint8_t* bits_dev, uint8_t* grid_dev,
                  double* rewards_dev, uint8_t* dones_dev, const snk_step_extra* extra, void* stream);
int snk_step_many_grid(snk_env* env, int32_t num_steps, const uint8_t* actions_dev, uint8_t* obs_dev, uint8_t* bits_dev,
                       uint8_t* grid_dev, int32_t obs_every_step, double* rewards_dev, uint8_t* dones_dev,
                       const snk_step_extra* extra, void* stream);

/* Same call with HOST buffers (the reference's step() takes and returns host objects,
 * snake_env.py:414): copies actions in, steps, copies obs / rewards / dones out and synchronises.
 * Pinned buffers make the copies asynchronous to the host until the final synchronise.  obs_host may
 * be NULL.  The observation block crosses the PCIe link in one of two ways (same bytes land in
 * obs_host either way):
 *   SNK_XFER_RAW     one device-to-host copy of the uint8 NHWC block;
 *   SNK_XFER_PACKED  the step kernel emits channel bits (as snk_step_bits: no NHWC block is written on the
 *                    device at all), the block crosses the link 8x smaller in chunks, and a pool of host
 *                    threads widens each chunk back to 0/1 bytes while the next ones are in flight.
 * Default: packed when the block is >= 4 MiB, raw below (environment SNK_HOST_TRANSPORT=raw|packed and
 * SNK_HOST_THREADS override at create time). */
int snk_step_host(snk_env* env, const uint8_t* actions_host, uint8_t* obs_host,
                  double* rewards_host, uint8_t* dones_host);
/* snk_step_host plus the terminal info dict (snake_env.py:396-410): extra_host holds HOST pointers here
 * (any may be NULL); entries of environments with finished[e] == 0 are unspecified. */
int snk_step_host_info(snk_env* env, const uint8_t* actions_host, uint8_t* obs_host, double* rewards_host,
                       uint8_t* dones_host, const snk_step_extra* extra_host);
int snk_reset_host(snk_env* env, uint8_t* obs_host);
/* For host callers that can consume channel bits directly: as snk_step_host, but delivers the observation as
 * one byte per (cell, frame) -- bits_host[u] bit c = channel c, N * prod(obs shape) / 8 bytes, the layout of
 * snk_pack_obs -- so nothing is widened on the host and an eighth of the bytes crosses the PCIe link. */
int snk_step_host_bits(snk_env* env, const uint8_t* actions_host, uint8_t* bits_host,
                       double* rewards_host, uint8_t* dones_host);

/* Work on this handle's buffers that the caller issued on `stream` outside the library -- a CUDA graph replay of
 * captured device-pointer calls, for instance -- must be reported here before the next *_host call, which then
 * waits for it on the device as it does for the library's own device-pointer calls.  Enqueues nothing. */
int snk_note_stream(snk_env* env, void* stream);

enum { SNK_XFER_RAW = 0, SNK_XFER_PACKED = 1 };
/* threads: widening threads of the packed transport, 0 = one per core this process may run on (<= 32) */
int snk_set_host_transport(snk_env* env, int mode, int threads);
int snk_get_host_transport(const snk_env* env, int* mode, int* threads);

/* Channel-bit form of an observation block for callers that keep observations on the device (replay
 * buffers, 8x smaller): bits_dev[u] bit c = obs_dev[8*u + c], u < n_bytes/8.  obs_dev 16-byte aligned,
 * bits_dev 4-byte aligned, n_bytes a multiple of 8.  One kernel launch on `stream`. */
int snk_pack_obs(snk_env* env, const uint8_t* obs_dev, uint8_t* bits_dev, size_t n_bytes, void* stream);
/* Host inverse (no GPU needed): obs_host[8*u + c] = (bits_host[u] >> c) & 1 -- the 0/1 channel bytes of
 * _encode (snake_env.py:484-492).  threads <= 1: on the calling thread. */
int snk_widen_bits_host(const uint8_t* bits_host, uint8_t* obs_host, size_t n_units, int threads);

/* Device memory for an observation block: `bytes` on `device`, mapped for that device only.  Where the device
 * supports generic memory compression and grants it, the block is a compressible allocation (cuMemCreate with
 * CU_MEM_ALLOCATION_COMP_GENERIC): the 0/1 observation bytes are mostly zero, and compressed lines cost less DRAM
 * traffic between L2 and HBM.  Kernels, copies and torch see ordinary device memory either way.  Otherwise the
 * block comes from cudaMalloc.  *compressed_out = 1 when compression was granted, else 0.  Free with
 * snk_free_obs, which synchronises the device first. */
int snk_alloc_obs(int device, size_t bytes, void** ptr_out, int* compressed_out);
int snk_free_obs(void* ptr);

/* ---- parity / checkpoint interface ---------------------------------------------------------- */

/* The reference's env.grid / env.snakes[i] of every environment.  A handle with compact records (the default for
 * warp-private tiles, frame stacks and large grids; INTEGRATION.md section 6) keeps no grid in device memory: the grid
 * returned here is rebuilt from the handle's wall layout, the record's fruit cells and the bodies -- which is exactly
 * what the reference's grid holds after every step (snake_env.py:546-566 never leaves anything else behind). */
int snk_get_state(snk_env* env, const snk_state_view* out, void* stream);
/* Needs grid, alive, dir, cells(+max_cells), length, alive_counter, episode_length. Rebuilds the
 * body-direction plane, zeroes episode statistics, fills every frame-stack slot with the encoding
 * of the given grid.  obs_dev (may be NULL) receives that stacked observation.  Compact records take the fruit cells
 * from `grid` and check the rest of it against the wall layout and the given bodies (SNK_DEV_STATE otherwise). */
int snk_set_state(snk_env* env, const snk_state_view* in, uint8_t* obs_dev, void* stream);

/* Exact checkpoint / resume of a shard (the reference never saves env state; its trainers checkpoint only
 * their networks, train_dqn.py:356-383): the raw records, frame histories and rollout statistics as one host
 * blob -- with a wall-map pool also next_map, cur_map and a digest of the pool, which must match on load.  A handle created with the same configuration (same seed and env_id_offset for the same Philox
 * stream; replay streams are set separately) continues bit for bit after snk_checkpoint_load. */
size_t snk_checkpoint_bytes(const snk_env* env);
int snk_checkpoint_save(snk_env* env, void* blob_host, size_t bytes);
int snk_checkpoint_load(snk_env* env, const void* blob_host, size_t bytes);

/* Per-env SNAPSHOT / RESTORE on the device, for search and lookahead (save a root, clone it into many envs, expand each
 * with other actions, rewind), restarts from an archive of states, fair population evaluation and A/B checks.
 *
 * A slot is a small header (a 64-bit configuration digest and the env's cur_map), then the env's raw record as it lies in
 * device memory, then its frame history (frame_stack > 1).  The digest covers what gives those bytes their meaning:
 * height, width, num_snakes, vision_range, frame_stack, the record layout (compact / full, body directions in the grid
 * byte or in a plane) and its sizes, the episode counters' width (16 bits unless max_episode_steps > 65535), the fruit
 * slots, and the wall layout (the pool's digest with a wall-map pool, else the single layout's).  Slots restore into any
 * handle with the same digest -- which may differ in num_envs, seed, env_id_offset, rewards and auto_reset -- and are
 * refused (SNK_DEV_SNAPSHOT) by every other.
 *
 * Restore copies the record byte for byte, so the whole episode carries over: bodies, fruit slots, directions,
 * alive_counter, episode_length, the per-snake episode statistics (the terminal info of a restored episode is the
 * original's), the frame ring and its position, the Philox event counter and the replay cursor.  Draws stay keyed by the
 * DESTINATION's global env id: a slot restored into the env it was taken from continues exactly as that env did after the
 * snapshot; restored into another env it continues that env's own stream from the source's event count -- a different,
 * deterministic future (a chance node).  In replay mode the cursor likewise indexes the destination's stream.  cur_map
 * comes from the slot; next_map is left alone.  No step is executed: snk_stats (SNK_STAT_ENV_STEPS included) does not
 * change.  Both calls only enqueue work on `stream` (stream rules as for the other device-pointer calls), never
 * synchronise and allocate nothing, so they can be captured in a CUDA graph.  Either call before the handle's first
 * reset returns SNK_E_STATE. */
/* Bytes of one snapshot slot (a 16-byte multiple).  Depends on the configuration, not on num_envs; 0 for NULL. */
size_t snk_snapshot_bytes(const snk_env* env);
/* Slot i of snap_dev := the state of env env_ids_dev[i], for i < count (env_ids_dev NULL: envs 0..count-1).  snap_dev is
 * count * snk_snapshot_bytes, 16-byte aligned (SNK_E_INVALID otherwise, and for count outside [1, N]).  Duplicated ids
 * are fine.  An id outside [0, N) raises SNK_DEV_SNAPSHOT and writes a slot that no handle accepts. */
int snk_snapshot(snk_env* env, const int32_t* env_ids_dev, int32_t count, void* snap_dev, void* stream);
/* For every env e with src_dev[e] >= 0 (int32 [N]), env e := slot src_dev[e] of snap_dev (num_slots >= 1 slots, 16-byte
 * aligned); src_dev[e] == -1 keeps env e.  Indexed by destination, so one slot may fan out to any number of envs.  Then
 * writes the observation of the restored envs into obs_dev / bits_dev and their grid rows into grid_dev (the formats of
 * snk_reset_grid; any of the three may be NULL, in any combination): the bytes the step that reached the restored state
 * returned.  Rows of other envs keep their bytes; grid rows of other envs may be rewritten with their unchanged grid.  A
 * slot index neither -1 nor below num_slots, or a slot whose digest differs, raises SNK_DEV_SNAPSHOT and leaves that env
 * and its rows unchanged. */
int snk_restore(snk_env* env, const int32_t* src_dev, int32_t num_slots, const void* snap_dev, uint8_t* obs_dev,
                uint8_t* bits_dev, uint8_t* grid_dev, void* stream);

/* Replay mode: per-env streams of recorded draw OUTPUTS in consumption order -- per reset the ns
 * accepted spawn-candidate indices (np.random.permutation, snake_env.py:581) then the fruit ranks
 * (np.random.randint, grid_util.py:130); per step its fruit ranks.  draws_host holds all streams
 * back to back, offsets_host[e]..offsets_host[e+1] delimits env e (N+1 entries).  Resets cursors. */
int snk_set_replay(snk_env* env, const int32_t* draws_host, const int64_t* offsets_host);
int snk_replay_cursors(snk_env* env, int32_t* cursors_host /* [N] */);

/* Sticky device error bits (SNK_DEV_*); synchronises the device. `clear` != 0 resets them. */
int snk_device_errors(snk_env* env, uint32_t* bits, int clear);

/* ---- rollout statistics (end-of-rollout allreduce payload) ----------------------------------- */
enum {
  SNK_STAT_EPISODES = 0,   /* episodes ended                                  */
  SNK_STAT_RETURN,         /* sum over ended episodes and snakes of episode_scores */
  SNK_STAT_EP_STEPS,       /* sum of episode lengths (env steps)              */
  SNK_STAT_FRUITS,         /* sum of episode_fruits                           */
  SNK_STAT_KILLS,          /* sum of episode_kills                            */
  SNK_STAT_DEATHS,         /* snakes that died                                */
  SNK_STAT_ENV_STEPS,      /* env steps executed (counted on the device, so CUDA-graph replays count too) */
  SNK_STAT_COUNT = 8
};
/* Device pointer to SNK_STAT_COUNT doubles accumulated on device (for an in-place NCCL allreduce). */
int snk_stats_dev(snk_env* env, double** stats_dev);
int snk_stats(snk_env* env, double* out_host /* [SNK_STAT_COUNT] */, int clear);

/* ---- spawn table (host only, no GPU needed) -------------------------------------------------- */

/* Number of spawn poses dfs_sweep_empty enumerates on the empty walled grid (grid_util.py:73-99). */
int64_t snk_spawn_count(int32_t height, int32_t width, int32_t snake_length);
/* Writes them, in the reference's order, as flat cell indices [count, snake_length], head first. */
int snk_spawn_cells(int32_t height, int32_t width, int32_t snake_length, int32_t* out, int64_t count);
/* The same two on a custom wall layout (walls_host as for snk_create_map; the border is not checked here). */
int64_t snk_spawn_count_map(int32_t height, int32_t width, int32_t snake_length, const uint8_t* walls_host);
int snk_spawn_cells_map(int32_t height, int32_t width, int32_t snake_length, const uint8_t* walls_host, int32_t* out,
                        int64_t count);

#ifdef __cplusplus
}
#endif
#endif /* SNK_H_ */
