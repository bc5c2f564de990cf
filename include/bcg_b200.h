/*
 * bcg_b200.h -- C-ABI of the B200-native batched PlanEnv.step path.
 *
 * The upstream reference (braincorp/bc-gym-planning-env, pure Python) has no FFI of its own; the
 * seams this library plugs into are (paths relative to bc_gym_planning_env/ in the reference):
 *   (i)  the env API            envs/base/env.py:278-361 (get_state/set_state/reset/step)
 *   (ii) the native-hook seam   `brain.shining_utils.*` imports at utilities/path_tools.py:101-103,
 *        utilities/coordinate_transformations.py:17-20,39-41,169-171, utilities/costmap_utils.py:106-107
 * Each entry point below names the reference function(s) it replaces for a *batch* of N environments.
 *
 * Conventions
 *   - plain C types only; every pointer marked "device" is a CUDA device pointer owned by the caller
 *     (the Python host allocates them as torch tensors); the library never allocates or frees them.
 *   - every function returns 0 on success, <0 on error; bcg_last_error() gives the message of the
 *     last failure on the calling thread.  No C++ exception crosses the boundary.
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it.
 *   - per-env dynamic state is structure-of-arrays: state_f[row * n_envs + env] (fp64 rows) and
 *     state_i[row * n_envs + env] (int32 rows); row numbers come from bcg_state_layout().
 *   - kernels never trap: out-of-map pixels are skipped exactly like envs/base/env.py:483-484 and
 *     anomalies are counted in the device `status` words (BCG_STATUS_*), which the host polls.
 */
#ifndef BCG_B200_H_
#define BCG_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BCG_ABI_VERSION 14

/* error codes */
#define BCG_OK 0
#define BCG_ERR_INVALID (-1) /* bad argument                     */
#define BCG_ERR_CUDA (-2)    /* a CUDA runtime call failed       */
#define BCG_ERR_NO_DEVICE (-3)

/* robot kinds (robot_models/robot_drive_types.py) */
/* reward providers (envs/base/reward_provider_examples.py) */
#define BCG_REWARD_CONTINUOUS 0
#define BCG_REWARD_PURE_PURSUIT 1

#define BCG_ROBOT_TRICYCLE 0
#define BCG_ROBOT_DIFFDRIVE 1

/* fixed fp64 state rows; ring rows follow (see BcgStateLayout) */
#define BCG_F_ROBOT 0    /* 7 rows: true robot x,y,th,v,w,steer_cmd,wheel   (tricycle_model.py:234-244) */
#define BCG_F_DROBOT 7   /* 7 rows: delayed robot state = State.robot_state (env.py:386-396)            */
#define BCG_F_DPOSE 14   /* 3 rows: delayed pose       = State.pose         (env.py:377-394)            */
#define BCG_F_TIME 17    /* State.current_time                                                         */
#define BCG_F_MIN_DIST 18 /* ContinuousRewardProviderState.min_spat_dist_so_far (reward.py:15)          */
#define BCG_F_EP_RETURN 19 /* sum of rewards since the last reset (statistics only)                     */
#define BCG_F_FIXED 20
/* int32 state rows */
#define BCG_I_ITER 0     /* State.current_iter                                 */
#define BCG_I_TARGET 1   /* ContinuousRewardProviderState.target_idx            */
#define BCG_I_COLLIDED 2 /* State.robot_collided (sticky, env.py:393)           */
#define BCG_I_QC 3       /* control queue: head | len << 16                     */
#define BCG_I_QP 4       /* pose queue                                          */
#define BCG_I_QS 5       /* robot-state queue                                   */
#define BCG_I_FIXED 6

/* device status words (uint32 counters, length BCG_STATUS_WORDS) */
#define BCG_STATUS_LUT_MISS 0     /* footprint tuple not found in the angle-bin table */
#define BCG_STATUS_PATH_EXHAUSTED 1 /* init: "Goal pose too close to initial pose" (reward.py:275-277) */
#define BCG_STATUS_SLOT_OVERFLOW 2  /* bcg_generate_aisles: a drawn map / path did not fit its slot; env left as it was */
#define BCG_STATUS_SAMPLER_EMPTY 3  /* bcg_generate_minis: "the sampling space looks empty" (mini_env.py:138,361)      */
#define BCG_STATUS_WORDS 8

/* episode statistics accumulated on device at episode end (fp64, length BCG_STATS_WORDS) */
#define BCG_STAT_EPISODES 0
#define BCG_STAT_RETURN 1
#define BCG_STAT_LENGTH 2
#define BCG_STAT_COLLIDED 3
#define BCG_STAT_GOAL 4
#define BCG_STAT_TIMEOUT 5
#define BCG_STATS_WORDS 8

/* Environment constants shared by the batch: EnvParams (envs/base/params.py:15-43), RewardParams
 * (envs/base/reward.py:162-171), robot dimension table (robot_models/robot_dimensions_examples.py). */
typedef struct BcgParams {
  double dt;
  double resolution;
  double inv_resolution;      /* 1./resolution, as coordinate_transformations.py:204 computes it */
  double spatial_precision;   /* sp */
  double angular_precision;   /* ap */
  double progress_multiplier; /* RewardParams.spatial_progress_multiplier */
  double wheel_base;          /* front_wheel_from_axis */
  double max_wheel_angle;
  double max_wheel_delta;     /* max_front_wheel_speed * dt (tricycle_model.py:143) */
  double p_gain;
  double max_lin_acc;
  double max_ang_acc;
  double alpha[6];            /* odometry noise; used when noise_on */
  double ego_x0, ego_y0;      /* egocentric crop origin in the robot frame (egocentric.py:113-114) */
  double ego_world_w, ego_world_h; /* CostMap2D.world_size() of the crop (costmap_2d.py:115-121) */
  uint64_t seed;              /* Philox key */
  uint64_t env_id_base;       /* global id of env 0 of this shard (distinct noise streams per GPU) */
  int32_t robot_kind;
  int32_t noise_on;
  int32_t delay_control, delay_pose, delay_state;
  int32_t iteration_timeout;
  int32_t ego_w, ego_h;       /* crop size in pixels */
  int32_t reward_kind;        /* 0 ContinuousRewardProvider (reward.py:173-288), 1 ContinuousRewardPurePursuitProvider
                                 (reward.py:291-371) */
  int32_t reserved;
  int32_t auto_reset;         /* envs that report done start their next episode inside the step: 0 no, 1 in the same world
                                 (the initial state the env has), BCG_AUTO_RESET_NEW_WORLD in a newly drawn world
                                 (needs BcgBatch.world_gen) */
  int32_t ego_variant;        /* 0: EgocentricCostmap wrapper (egocentric.py:125-160): crop about the delayed pose,
                                 9-vector goal_n_state.  1: ColoredEgoCostmapRandomAisleTurnEnv
                                 (synth_turn_env.py:396-420): crop about the TRUE robot pose, goal = unit vector
                                 towards the last path point, 5 values [gx, gy, v, w, wheel] (slots 5..8 zero) */
} BcgParams;

/* one costmap of the arena: CostMap2D (utilities/costmap_2d.py:13-37) + its derived planes: the lethal
 * bit-plane (collision) and the cell tiles (the same uint8 cells re-laid out as 128-byte tiles of 16 px x 8
 * rows, tile (ty, tx) at cell_tile_off + (ty * ctiles_x + tx) * 128, row r of a tile at + r * 16, zero
 * beyond the map; the egocentric kernel fetches whole HBM lines of a rotated window from it) */
#define BCG_MAP_ONLY_LETHAL 1
#define BCG_MAP_CELL_INDEX 4  /* the map's cell index (see BCG_BATCH_CELL_INDEX) is exact; set by bcg_build_lethal_tiles,
                                 callers leave it clear */
typedef struct BcgMapDesc {
  int64_t data_off;  /* byte offset of uint8 [H][pitch] in the map arena                      */
  int64_t tile_off;  /* uint32 offset of the lethal tile plane in the tile arena               */
  double origin_x, origin_y;
  int32_t height, width, pitch;
  int32_t tiles_x, tiles_y; /* 32 px x 16 rows per 64-byte tile                                */
  int32_t flags;            /* BCG_MAP_ONLY_LETHAL: every non-zero cell is 254 (set by the host before
                               bcg_build_lethal_tiles, cleared there when another value is met)       */
  int64_t cell_tile_off;    /* byte offset of the map's cell tiles in the cell-tile arena (multiple of 128) */
  int32_t ctiles_x, ctiles_y; /* 16 px x 8 rows per 128-byte cell tile: pitch / 16, ceil(height / 8)     */
  int32_t occupied;         /* cells != 0, counted by bcg_build_lethal_tiles: maps with more than 1 cell in 20
                               occupied skip the sparse egocentric kernel (their windows overflow its list) */
  int32_t sum_off;          /* uint32 offset of the map's tile summary in BcgBatch.occ_sum_arena: [tiles_y][(tiles_x + 31) / 32]
                               words, bit tx & 31 of word [ty][tx >> 5] set when tile (tx, ty) of the occupancy plane
                               holds a cell (a clear bit promises an empty tile; set by the host, kept by the
                               generators)                                                                          */
} BcgMapDesc;

/* one refined path: fp64 SoA rows x,y,th,cos(th),sin(th), each `pitch` long, then chunk bounds */
typedef struct BcgPathDesc {
  int64_t off;       /* fp64 offset of the 5 point rows in the path arena                       */
  int64_t chunk_off; /* fp64 offset of the 3 chunk rows (cx, cy, radius), each `chunk_pitch`     */
  int32_t n;         /* number of points                                                       */
  int32_t pitch;
  int32_t n_chunks;  /* ceil(n / 32)                                                           */
  int32_t chunk_pitch;
} BcgPathDesc;

/* angle-binned footprint table replacing get_pixel_footprint (utilities/path_tools.py:122-162) */
typedef struct BcgFootprintLut {
  const double* edges;    /* device [n_bins + 1] ascending, edges[0] = -pi, edges[n_bins] = +pi    */
  const int16_t* verts;   /* device [n_bins][2 * n_verts]  rounded vertices (x0,y0,x1,y1,...)       */
  const int16_t* header;  /* device [n_bins][4] = xmin, ymin, n_rows, width (mask bounding box)     */
  const uint64_t* rows;   /* device [n_bins][max_rows][wpr] bit i of word j <-> column xmin+64j+i   */
  const double* fp_pix;   /* device [2 * n_verts] footprint / resolution (fx0,fy0,...)             */
  const int32_t* bucket_first; /* device [n_buckets]: bin containing the left end of uniform bucket k  */
  double bucket_scale;    /* n_buckets / (2 pi)                                                     */
  int32_t n_bins, n_verts, max_rows, wpr;
  int32_t n_buckets;
  int32_t bin_stride;     /* int16 elements per row of `bins` (multiple of 8), 0 when bins is NULL         */
  const int16_t* bins;    /* optional, device [n_bins][bin_stride]: a bin's vertex tuple followed by its header
                             (xmin, ymin, n_rows, width), 16-byte aligned rows -- lets the lookup fetch two
                             candidate bins, tuple and header, in one memory round trip                     */
} BcgFootprintLut;

/* BcgBatch.flags */
#define BCG_BATCH_SPARSE_EGO_ONLY 1 /* no map of the batch is dense (BcgMapDesc.occupied below 1 cell in 20, read back by the
                                       host after bcg_build_lethal_tiles; always true for device-generated worlds): the
                                       sparse egocentric kernel renders the rare window that overflows its cell list
                                       itself and the dense kernel is not launched behind it */
#define BCG_BATCH_CELL_INDEX 2      /* the host reserved a cell-index trailer after the tile summary of every map that is
                                       not dense (occupied * 20 <= width * height): at uint32 offset
                                       sum_off + tiles_y * ((tiles_x + 31) / 32) of occ_sum_arena,
                                         [0] capacity (cells; written by the host), [1] total (cells),
                                         [2 .. 2 + tiles_y * tiles_x] prefix: exclusive counts of occupied cells per 32 x 16
                                             tile of the occupancy plane in row-major tile order (tiles_y * tiles_x + 1 words),
                                         then `capacity` words of cells: every occupied cell as x | y << 16 in map pixels,
                                             grouped by tile in that order, row-major inside a tile.
                                       bcg_build_lethal_tiles fills them and sets BCG_MAP_CELL_INDEX on the maps whose cells
                                       fit; the sparse egocentric kernel then reads a window's cells from there instead of
                                       listing them from the occupancy plane.  Without this bit no trailer is read or
                                       written (tile summaries may be packed tightly). */

/* everything a step touches; all pointers are device pointers */
typedef struct BcgBatch {
  int32_t n_envs;
  int32_t n_frows, n_irows; /* must equal bcg_state_layout() for the params in use */
  int32_t n_maps, n_paths;
  int32_t flags;            /* BCG_BATCH_* */
  double* state_f;
  int32_t* state_i;
  double* init_f;  /* the state reset() restores (env.py:247,302) */
  int32_t* init_i;
  double* cand;    /* scratch [3][n_envs]: the pose the last step proposed (before the collision verdict), written by
                      move_kernel                                                                           */
  int32_t* cand_i; /* scratch [2][n_envs] (reserved; must be allocated)                                      */
  void* ego_work;  /* scratch [n_envs][128 bytes]: per-env affine map + source window of the egocentric crop,
                      written by move_kernel / reward_kernel (or bcg_observe_ego) for the egocentric kernel; may
                      be NULL when no egocentric image is ever requested                                    */
  void* work;      /* scratch [n_envs][192 bytes]: the per-env record move_kernel leaves for reward_kernel, and the
                      work records (map / path / footprint references) of the stand-alone collision entry points */
  const int32_t* map_id;  /* [n_envs] index into maps  */
  const int32_t* path_id; /* [n_envs] index into paths */
  const BcgMapDesc* maps;
  const BcgPathDesc* paths;
  const uint8_t* map_arena;
  const uint32_t* tile_arena;
  const double* path_arena;
  BcgFootprintLut lut;
  const uint8_t* cell_tile_arena; /* cell tiles of every map (bcg_build_cell_tiles); needed for the egocentric image
                            (and by the world generators): the egocentric kernels stage only the 128-byte tiles
                            the rotated source window touches (zero fill outside the map); may be NULL when no
                            egocentric image is ever requested                                                */
  const uint32_t* occ_tile_arena; /* required: the occupancy plane (1 bit per cell, value != 0), laid out exactly
                            like the lethal tile plane (same tile_off); filled by bcg_build_lethal_tiles and kept
                            by the generators.  With cell_tile_arena and ego_list the egocentric observation takes
                            the sparse path: zero the crop, then scatter only the occupied source cells of its
                            window                                                                          */
  int32_t* ego_list;      /* optional scratch [n_envs + 4]: envs whose window holds too many occupied cells
                            for the sparse path, handed to the dense cell-tile kernel (count at [n_envs]; [n_envs + 1] is
                            the sparse kernel's env counter)                                                 */
  const uint32_t* occ_sum_arena; /* required: one bit per tile of the occupancy plane (BcgMapDesc.sum_off), filled by
                            bcg_build_lethal_tiles and kept by the generators; must start out zero (but for the capacity
                            words of BCG_BATCH_CELL_INDEX trailers).  The collision check loads only the non-empty tiles
                            under a footprint, and the sparse egocentric kernel only those of a window, or with a cell
                            index only the window's cells                                                           */
  uint32_t* status; /* [BCG_STATUS_WORDS] */
  double* stats;    /* [BCG_STATS_WORDS]  */
  uint64_t* step_counter; /* optional device [2], zero at start: when set, bcg_step ignores its step_index argument,
                            takes the step index from word 0 and increments it on the device when the step is done
                            (word 1 is its scratch) -- so that a captured CUDA graph of a step can be replayed
                            without changing a kernel argument                                                    */
  const struct BcgWorldGen* world_gen; /* device pointer, needed when BcgParams.auto_reset == BCG_AUTO_RESET_NEW_WORLD
                            (NULL otherwise): how the step draws a new world for an env whose episode ends */
} BcgBatch;

/* TurnParams (envs/synth_turn_env.py:18-31): geometry of one aisle turn */
typedef struct BcgTurnParams {
  double main_corridor_length, turn_corridor_length, turn_corridor_angle;
  double main_corridor_width, turn_corridor_width, margin, rot_theta;
  int32_t flip_arnd_oy, flip_arnd_ox;
} BcgTurnParams;

/* Fixed-size per-env slots for environments that are (re)generated on the device (bcg_generate_aisles).
 * Env e owns maps[e] and paths[e] (n_maps == n_paths == n_envs, map_id[e] == path_id[e] == e); the offsets in
 * its descriptors are set once by the host (e * slot size) and never change, the generator rewrites the
 * geometry fields (height, width, pitch, origin, tile counts, path length).  The map, cell-tile and lethal-tile
 * slots must be zero when an env is generated for the first time. */
typedef struct BcgAisleSlots {
  int64_t map_slot_bytes;    /* capacity of one env's uint8 rows, and of its cell tiles           */
  int64_t tile_slot_words;   /* capacity of one env's lethal tile plane (uint32 words)            */
  int32_t path_pitch;        /* row pitch of one env's 5 path rows (points); multiple of 4        */
  int32_t chunk_pitch;       /* row pitch of its 3 chunk rows; >= ceil(path_pitch / 32)           */
  void* gen_state;           /* device scratch [n_envs][128 bytes], zero before the first call:
                                the walls currently drawn in each slot (to erase them cheaply)     */
  BcgTurnParams* params_out; /* optional device [n_envs]: the turn each regenerated env now has   */
} BcgAisleSlots;

/* RandomMiniEnvParams (envs/mini_env.py:30-46) + the two goal tolerances of its EnvParams the sampler's final check
 * uses (:349-353) */
typedef struct BcgMiniGenParams {
  double inner_h, inner_w, mid_margin, out_margin;
  double min_obstacle_angle, max_obstacle_angle;
  double lim_euc_dist, lim_ang_dist, angular_pose_noise_scale;
  double goal_spat_dist, goal_ang_dist;
} BcgMiniGenParams;

/* MiniEnvParams (envs/mini_env.py:80-92): world size, start / end poses, the corner obstacle (two walls o-a, o-b) */
typedef struct BcgMiniParams {
  double h, w;
  double start[3], end[3];
  double a[2], o[2], b[2];
} BcgMiniParams;

/* BcgParams.auto_reset */
#define BCG_AUTO_RESET_NEW_WORLD 2
/* BcgWorldGen.kind */
#define BCG_WORLD_AISLE 0 /* bcg_generate_aisles' worlds */
#define BCG_WORLD_MINI 1  /* bcg_generate_minis' worlds   */

/* Auto-reset into a newly drawn world (BcgParams.auto_reset == BCG_AUTO_RESET_NEW_WORLD), in device memory, reached through
 * BcgBatch.world_gen.  The batch must be made of the generators' per-env slots (n_maps == n_paths == n_envs, cell tiles).
 * At a step, reward_kernel appends every env that is done to `list` (count[0] of them) instead of restoring its initial
 * state; a regeneration kernel behind it then gives each listed env what bcg_generate_aisles / bcg_generate_minis give a
 * masked env -- a drawn world in its slot, its path and initial state -- and writes its initial observation (obs_vec,
 * goal_n_state, egocentric record), so that the step's egocentric kernels render the new world.  With BcgEpisodeEnds and the
 * egocentric image, the final crop of an env with a slot is rendered from the old world before it is erased.  Draws are
 * keyed (p->seed; p->env_id_base + e, BCG_NEW_WORLD_DRAW | step index), a domain the host's draw indices never reach (see
 * bcg_generate_aisles).  A world that does not fit its slot (BCG_STATUS_SLOT_OVERFLOW) or a sampler that runs out of tries
 * (BCG_STATUS_SAMPLER_EMPTY) restarts the env in its current world, as auto_reset 1 does; the status word counts it. */
#define BCG_NEW_WORLD_DRAW 0x8000000000000000ull
typedef struct BcgWorldGen {
  int32_t kind;              /* BCG_WORLD_AISLE or BCG_WORLD_MINI                                                     */
  int32_t reserved;
  BcgAisleSlots slots;       /* the slots, as passed to the generator; params_out (optional) points at BcgTurnParams [n]
                                for aisles, BcgMiniParams [n] for minis                                              */
  BcgMiniGenParams mini;     /* the sampling space (BCG_WORLD_MINI)                                                   */
  double path_delta;
  int32_t* list;             /* device [n_envs] scratch: the envs to regenerate at this step                          */
  int32_t* count;            /* device [4], zero before the first step: [0] listed envs, [1] item counter, [2] finished
                                CTAs of the regeneration kernel (whose last CTA zeroes the words for the next step)    */
} BcgWorldGen;

typedef struct BcgStateLayout {
  int32_t n_frows, n_irows;
  int32_t ring_control; /* first fp64 row of the control ring: delay_control slots x 2 rows */
  int32_t ring_pose;    /* delay_pose slots x 3 rows                                         */
  int32_t ring_state;   /* delay_state slots x 7 rows                                        */
} BcgStateLayout;

/* Per-env parameters of a batch whose envs do not all share one EnvParams / noise setting: structure of arrays like
 * state_f / state_i, f[row * n_envs + env] (fp64 rows BCG_EP_F_*) and i[row * n_envs + env] (int32 rows BCG_EP_I_*).
 * They override the same fields of BcgParams for env `env`; everything else stays batch-wide.  The delays in BcgParams
 * are then the ring capacities (the per-field maxima of the rows: bcg_state_layout sizes the rings from them), and env e
 * uses the first min(d_e, capacity) slots of each ring.  A NULL BcgEnvRows* means "every env uses BcgParams". */
#define BCG_EP_F_SP 0       /* RewardParams.spatial_precision                          */
#define BCG_EP_F_AP 1       /* RewardParams.angular_precision                          */
#define BCG_EP_F_PM 2       /* RewardParams.spatial_progress_multiplier                */
#define BCG_EP_F_ALPHA 3    /* 6 rows: odometry noise alpha1..alpha6 (used when noise_on) */
#define BCG_EP_F_ROWS 9
#define BCG_EP_I_DELAY_CONTROL 0
#define BCG_EP_I_DELAY_POSE 1
#define BCG_EP_I_DELAY_STATE 2
#define BCG_EP_I_TIMEOUT 3  /* EnvParams.iteration_timeout                             */
#define BCG_EP_I_NOISE_ON 4 /* 0: the env's robot moves without odometry noise          */
#define BCG_EP_I_ROWS 5
typedef struct BcgEnvRows {
  const double* f;   /* device [BCG_EP_F_ROWS][n_envs] */
  const int32_t* i;  /* device [BCG_EP_I_ROWS][n_envs] */
} BcgEnvRows;

/* Episode ends of an auto-reset batch (bcg_step / bcg_rollout): why each env is done, and the observation of
 * every episode that ends at this step as it was before the in-kernel reset overwrote it.
 *
 * reason[e] is written for every env at every step:
 *   BCG_END_GOAL | BCG_END_COLLIDED | BCG_END_TIMEOUT  the causes of `done` (env.py:407-419), set while the env is done
 *                                                      (without auto-reset they stay set, like done)
 *   BCG_END_NOW                                        the episode ended at this step (done now, not done before it:
 *                                                      the condition under which the episode statistics count it)
 * terminated = done && (GOAL | COLLIDED); truncated = done && TIMEOUT && !terminated (a timeout on the step of a goal or
 * a collision is a termination).
 * Every env with BCG_END_NOW gets its final record, with or without auto-reset: final_obs_vec (BcgStepOut.obs_vec's
 * fields, [11] the post-step target index), final_goal_n_state (needs BcgStepOut.goal_n_state), final_return (the
 * episode return including this step's reward) and final_length (iterations).  These rows are dense, indexed by env
 * and valid only where BCG_END_NOW is set.
 * Final crops (needs BcgStepOut.ego_image and the cell-tile planes) are kept in `capacity` slots: count[0] numbers the
 * ends of the step in no particular order; end k < capacity gets slot k, final_slot[e] = k (else -1), its egocentric
 * record is copied to final_ego_work[k] before the reset rewrites it, and the egocentric kernels render it into
 * final_ego_image[k] in the launches that render the step's crops.  count[0] keeps counting past the capacity:
 * count[0] > capacity means that count[0] - capacity ended envs (which ones is unspecified) have final_slot -1 and no
 * crop; nothing is written past the capacity.  move_kernel zeroes count[] at the start of every step, so a captured
 * CUDA graph of a step replays correctly and the counts describe the last step. */
#define BCG_END_GOAL 1
#define BCG_END_COLLIDED 2
#define BCG_END_TIMEOUT 4
#define BCG_END_NOW 8
typedef struct BcgEpisodeEnds {
  uint8_t* reason;            /* [n]                                                                          */
  int32_t* final_slot;        /* [n] crop slot of an env that ended at this step, -1 otherwise                */
  float* final_obs_vec;       /* [n][12]                                                                      */
  float* final_goal_n_state;  /* [n][9]   (needed with BcgStepOut.goal_n_state)                               */
  double* final_return;       /* [n]                                                                          */
  int32_t* final_length;      /* [n]                                                                          */
  void* final_ego_work;       /* [capacity][128 bytes]          (these three are needed with BcgStepOut.ego_image) */
  uint8_t* final_ego_image;   /* [capacity][ego_h][ego_w]                                                     */
  int32_t* final_list;        /* [capacity] scratch: slots the sparse egocentric kernel hands to the dense one */
  int32_t* count;             /* [2]: [0] episodes that ended at this step, [1] scratch (hand-over count)     */
  int32_t capacity;           /* >= 1                                                                         */
  int32_t reserved;
} BcgEpisodeEnds;

/* outputs of one step; any pointer may be NULL to skip that output */
typedef struct BcgStepOut {
  double* reward;      /* [n] reward of this step (reward.py:214-259)                          */
  uint8_t* done;       /* [n] env.py:407-419                                                   */
  uint8_t* hit;        /* [n] collision verdict of this step's pose_collides (env.py:455)       */
  uint8_t* ego_image;  /* [n][ego_h][ego_w] egocentric crop (egocentric.py:125-160 'env')        */
  float* goal_n_state; /* [n][9] egocentric.py:152-159                                          */
  float* obs_vec;      /* [n][12] fp32 copy of delayed pose(3), delayed robot state(7), time, target_idx */
  /* compact form of ego_image for consumers behind a narrow link (optional; needs ego_image and the sparse kernel): per
   * env the list of its non-zero crop pixels, entry = pixel offset (v * ego_w + u) | cost value << 16, in no particular
   * order.  ego_hit_count[e] = number of entries (only the first ego_hit_cap are stored: a larger count means "read
   * ego_image[e]"), or -1 when the env was rendered by the dense kernel.  A crop is ~1 % walls, so this is ~0.8 KB per
   * env instead of 15.6 KB. */
  uint32_t* ego_hits;      /* [n][ego_hit_cap] */
  int32_t* ego_hit_count;  /* [n]              */
  int32_t ego_hit_cap;
  int32_t reserved;
} BcgStepOut;

/* -- library ------------------------------------------------------------------------------------ */
int bcg_abi_version(void);
/* copies the calling thread's last error message (NUL terminated) and returns its length */
size_t bcg_last_error(char* buf, size_t cap);
/* sizeof() of the ABI structs, in declaration order: 0 BcgParams, 1 BcgMapDesc, 2 BcgPathDesc,
 * 3 BcgFootprintLut, 4 BcgBatch, 5 BcgStateLayout, 6 BcgStepOut, 7 BcgTurnParams, 8 BcgAisleSlots, 9 BcgMiniGenParams,
 * 10 BcgMiniParams, 11 BcgEnvRows, 12 BcgEpisodeEnds, 13 BcgWorldGen; -1 for anything else.  Lets a
 * binding (ctypes, cffi, ...) verify its struct mirrors before the first call. */
int64_t bcg_sizeof(int32_t which);
/* number of CUDA devices visible, <0 on error; makes a missing GPU a loud failure for callers */
int bcg_device_count(void);
/* state row map for the delays in `p` (mirrors the three queues of env.py:64-66) */
int bcg_state_layout(const BcgParams* p, BcgStateLayout* out);

/* -- setup (at reset time, not per step) ------------------------------------------------------------ */
/* derive the lethal bit-plane (cell == 254, costmap_2d.py:21), the occupancy plane and its tile summary (both required:
 * BcgBatch.occ_tile_arena, occ_sum_arena) of maps [first, first+count) */
int bcg_build_lethal_tiles(const BcgBatch* b, int32_t first, int32_t count, void* stream);
/* derive the cell tiles (see BcgMapDesc) of maps [first, first+count) from the uint8 rows (CostMap2D.get_data,
 * costmap_2d.py:91-96: the bytes extract_egocentric_costmap samples, costmap_utils.py:25-75) */
int bcg_build_cell_tiles(const BcgBatch* b, int32_t first, int32_t count, void* stream);
/* make_initial_state (env.py:179-214) + ContinuousRewardProvider.generate_initial_state
 * (reward.py:261-288) for every env: writes init_f/init_i and copies them into state_f/state_i.  With `rows` env e's
 * initial target index uses its own spatial / angular precision (NULL: those of p). */
int bcg_init_state(const BcgParams* p, const BcgBatch* b, const BcgEnvRows* rows, void* stream);
/* PlanEnv.reset (env.py:293-303) for envs with mask[e] != 0 (mask NULL = all) */
int bcg_reset_where(const BcgBatch* b, const uint8_t* mask, void* stream);

/* RandomAisleTurnEnv.reset with draw_new_turn_on_reset (envs/synth_turn_env.py:278-291) on the device, for
 * envs with mask[e] != 0 (mask NULL = all): draw a turn (:317-332; Philox keyed (p->seed; env id, draw_index)
 * unless `turn_params`, device [n_envs], supplies them), build its walls like cv2.line and its way points
 * (path_and_costmap_from_config :110-192), refine the path (utilities/path_tools.py:178-240, spacing
 * `path_delta`), derive both tile planes, and make the initial state (env.py:179-214, reward.py:261-288).
 * The previous walls of the slot are erased pixel by pixel, so a reset costs O(wall pixels), not O(map).
 * With `rows` the initial states use each env's own goal tolerances (NULL: those of p); rows changed before the call (a
 * new parameter set at a reset) are what the new worlds' initial states see.  Needs BcgBatch.cell_tile_arena.
 * Draw keys: the host's calls use draw indices below BCG_NEW_WORLD_DRAW (2^63).  A step with auto_reset ==
 * BCG_AUTO_RESET_NEW_WORLD draws the new world of env e with (p->seed; p->env_id_base + e, BCG_NEW_WORLD_DRAW | s), s the
 * step index its odometry noise uses (bcg_step's step_index, or word 0 of BcgBatch.step_counter); an env ends at most
 * once per step, so every key is drawn once, a batch split over shards (env_id_base) draws the worlds one batch draws,
 * and a replay from the same step index draws the same worlds.  bcg_generate_minis keys its draws the same way. */
int bcg_generate_aisles(const BcgParams* p, const BcgBatch* b, const BcgEnvRows* rows, const BcgAisleSlots* slots,
                        const uint8_t* mask, const BcgTurnParams* turn_params, uint64_t draw_index, double path_delta,
                        void* stream);

/* RandomMiniEnv's env construction (envs/mini_env.py:323-389, what its reset repeats) on the device, for envs with
 * mask[e] != 0 (mask NULL = all), in the same per-env slots as bcg_generate_aisles: sample MiniEnvParams (:269-320,
 * Philox keyed (p->seed; env id, draw_index) in the reference's draw order) until neither end pose collides and the
 * two are not within the goal tolerances of each other (:336-358), rasterise the two walls like cv2.line incl. its
 * clipping of far end points (cv::clipLine), refine the path, make the initial state.  With `mini_params` (device
 * [n_envs]) the worlds are built from those parameters as they are, like MiniEnv(config) does.  `params_out`
 * (optional, device [n_envs]) receives the accepted parameters.  BCG_STATUS_SLOT_OVERFLOW counts worlds that do not
 * fit their slots, BCG_STATUS_SAMPLER_EMPTY envs whose sampling ran out of tries (both left as they were). */
int bcg_generate_minis(const BcgParams* p, const BcgBatch* b, const BcgAisleSlots* slots, const uint8_t* mask,
                       const BcgMiniGenParams* gen, const BcgMiniParams* mini_params, BcgMiniParams* params_out,
                       uint64_t draw_index, double path_delta, void* stream);

/* -- the hot path -------------------------------------------------------------------------------- */
/* PlanEnv.step (env.py:334-361) for all envs.  actions: device [n][2] (wheel_v, wheel_angle) or
 * (v, w) for diff-drive; action_is_f64 selects fp64 vs fp32 elements.  Launches move_kernel (one thread per env:
 * control delay env.py:371-373, robot model tricycle_model.py:478-538 / differential_drive.py:236-265, pose_collides
 * env.py:464-489, rollback :452-461, delay lines :377-389, compact observation, egocentric record), reward_kernel (a
 * group of lanes per env: reward.py:214-259, done env.py:400-419, statistics, goal vector egocentric.py:152-159,
 * auto-reset env.py:293-303) and -- only if out->ego_image is set -- the egocentric observation (egocentric.py:125-160):
 * with the occupancy plane and ego_list the sparse scatter kernel, followed by the dense cell-tile kernel for the
 * envs it hands over unless BCG_BATCH_SPARSE_EGO_ONLY, else one dense kernel.  Each kernel is launched as a programmatic
 * dependent of the one before it on `stream`.  step_index is the caller's global step counter (ignored when
 * BcgBatch.step_counter is set): odometry noise is Philox4x32-10 keyed by p->seed at counter (env id, step_index, draw),
 * replacing the reference's global np.random (differential_drive.py:50).
 *
 * rows (BcgEnvRows; NULL: every env uses p): per-env parameters.  move_kernel reads env e's delays, timeout, noise flag
 * and alphas from the rows with its other top-of-kernel loads and forwards its goal tolerances and progress multiplier
 * to reward_kernel in the env's work slot.  Ring capacities are p's delays; a row delay above its capacity is clamped to
 * it (memory safety does not depend on the row contents; the host validates them).
 *
 * ends (BcgEpisodeEnds; NULL: no episode ends are reported): the same launches also report episode ends.  move_kernel
 * zeroes the counters, reward_kernel writes the reasons and final records and copies the egocentric records of the
 * ended envs before it resets them, and the egocentric kernels render the final crops after the step's own.  Final
 * crops need the cell-tile planes (BcgBatch.cell_tile_arena).
 *
 * p->auto_reset == BCG_AUTO_RESET_NEW_WORLD (see BcgWorldGen): reward_kernel lists the done envs instead of resetting them
 * and regenerate_kernel, launched between reward_kernel and the egocentric kernels, gives them new worlds, initial states
 * and initial observations (and renders their final crops from the old worlds).
 *
 * events (NULL: none are recorded): per-kernel hooks, events[0..4] are caller-created cudaEvent_t handles recorded on
 * `stream`: [0], [1] before move_kernel, [2] between move_kernel and reward_kernel, [3] after reward_kernel, or after
 * regenerate_kernel when it runs (reward / done / compact observation are final: a host consumer's copies can start here
 * while the egocentric kernel runs), [4] after the egocentric kernels.  Any entry may be NULL (not recorded).  A kernel with an event recorded right before it
 * is not launched as a programmatic dependent of its predecessor. */
int bcg_step(const BcgParams* p, const BcgBatch* b, const BcgEnvRows* rows, const void* actions, int32_t action_is_f64,
             uint64_t step_index, const BcgStepOut* out, const BcgEpisodeEnds* ends, void* const* events, void* stream);

/* the pieces, individually addressable (used by tests, ncu and the hook seam) */
/* pose_collides (env.py:464-489) of poses [3][n] (rows x,y,th) against each env's map, using the
 * lethal tile plane; flags_out [n].  pixels_out (optional, [n]) = in-map footprint pixel count (warp-per-env
 * kernel; without it the thread-per-env kernel the step itself uses).  poses == NULL checks the poses the last
 * bcg_step proposed (b->cand).  Two launches: per-env work records (footprint
 * angle bin, mask box, map references) into b->work, then the collision kernel. */
int bcg_collision(const BcgParams* p, const BcgBatch* b, const double* poses, uint8_t* flags_out,
                  int32_t* pixels_out, void* stream);
/* same verdicts read straight from the uint8 costmap rows (no derived plane) */
int bcg_collision_u8(const BcgParams* p, const BcgBatch* b, const double* poses, uint8_t* flags_out,
                     void* stream);
/* only the collision kernel, on the work records the last bcg_collision / bcg_collision_u8 call left in b->work
 * (use_u8: the uint8-row kernel) -- the form the collision roofline is measured on */
int bcg_collision_recheck(const BcgParams* p, const BcgBatch* b, uint8_t* flags_out, int32_t use_u8, void* stream);
/* EgocentricCostmap.observation (egocentric.py:125-160) from the current state */
int bcg_observe_ego(const BcgParams* p, const BcgBatch* b, uint8_t* ego_image, float* goal_n_state,
                    void* stream);

/* -- snapshots: get_state / set_state (env.py:278-291) ------------------------------------------ */
/* gather columns idx[0..k) of state_f/state_i into out_f [n_frows][k], out_i [n_irows][k] */
int bcg_gather_state(const BcgBatch* b, const int64_t* idx, int32_t k, double* out_f,
                     int32_t* out_i, void* stream);
/* scatter columns back; load_delayed_robot != 0 applies env.py:284 (robot := delayed robot state) */
int bcg_scatter_state(const BcgBatch* b, const int64_t* idx, int32_t k, const double* in_f,
                      const int32_t* in_i, int32_t load_delayed_robot, void* stream);

/* -- compact observation ------------------------------------------------------------------------------ */
/* Packs the per-env hit lists a step left in BcgStepOut.ego_hits (fixed stride `cap`) into one contiguous array:
 * env e's min(count, cap) entries go to packed[offsets[e] ..], offsets = exclusive prefix sum of the counts with
 * dense / overflowed envs (count < 0 or > cap) counted as 0 -- what a host consumer copies over the link instead
 * of n crops of ego_w x ego_h bytes.  offsets_only == 0: packed is uint32 (pixel offset | value << 16);
 * offsets_only != 0: packed is uint16, the pixel offsets alone (for batches whose maps hold no cost value but 254,
 * BCG_MAP_ONLY_LETHAL: the value is implied). */
int bcg_pack_ego_hits(const uint32_t* hits, const int32_t* counts, int32_t cap, int32_t n, const int64_t* offsets,
                      void* packed, int32_t offsets_only, void* stream);

/* -- hook-seam helpers (batched forms of the brain.shining_utils.* scalars) --------------------- */
/* world_to_pixel (coordinate_transformations.py:185-205): xy [n][2] fp64 -> int32 [n][2] */
int bcg_world_to_pixel(const double* xy, int64_t n, double origin_x, double origin_y,
                       double resolution, int32_t* out, void* stream);
/* normalize_angle (coordinate_transformations.py:28-36) */
int bcg_normalize_angle(const double* in, int64_t n, double* out, void* stream);
/* is_footprint_colliding_impl (costmap_utils.py:106-136; contract test_costmap_utils.py:251-325): does any cell of the
 * blitted footprint equal `value`?  values, mask: device [n] (the image slice and the blit mask, flattened);
 * flag_out: device int32, 1 when any(values[mask != 0] == value) */
int bcg_masked_any_equal(const uint8_t* values, const uint8_t* mask, int64_t n, int32_t value, int32_t* flag_out, void* stream);
/* inverse_transform_2d_impl (coordinate_transformations.py:39-84): device [n][3] (x, y, angle) -> [n][3] */
int bcg_inverse_transform(const double* transforms, int64_t n, double* out, void* stream);
/* native_project_poses (coordinate_transformations.py:289-328): poses device [n][3] moved by the HOST transform
 * (x, y, angle): rotate, translate, wrap the angle */
int bcg_project_poses(const double* transform_host, const double* poses, int64_t n, double* out, void* stream);
/* Observation.path of every env (env.py:421-433: path[target_idx:]; pure pursuit: path[:target_idx + 1]) as a device
 * tensor in the robot frame (from_global_to_egocentric, coordinate_transformations.py:341-362, about the observed pose):
 * out device [n][max_points][3] zero padded, len_out (optional) device [n] = way points left (may exceed max_points) */
int bcg_observe_ego_path(const BcgParams* p, const BcgBatch* b, int32_t max_points, double* out, int32_t* len_out, void* stream);

/* H steps of a fixed action plan (Monte-Carlo fan-outs: the reference steps a copied env through a candidate plan,
 * README.md:45-61): bcg_step for plan[h], h = 0 .. horizon - 1, launched back to back from one call -- every kernel a
 * programmatic dependent of the one before, no host work in between.  plan: device float32 [horizon][n_envs][2];
 * step h uses the Philox step index step_index + h (or the device-side counter when BcgBatch.step_counter is set).
 * rows and ends as for bcg_step (either may be NULL); `ends` describes the last step. */
int bcg_rollout(const BcgParams* p, const BcgBatch* b, const BcgEnvRows* rows, const float* plan, int32_t horizon,
                uint64_t step_index, const BcgStepOut* out, const BcgEpisodeEnds* ends, void* stream);

/* -- image memory --------------------------------------------------------------------------------
 * Egocentric crops are mostly zeros.  A device allocation with compute-data compression (CUDA virtual memory
 * management, CU_MEM_ALLOCATION_COMP_GENERIC) makes the hardware write and read such lines at a fraction of their DRAM
 * cost; contents and addressing are unchanged for kernels and copies.  The one place where this library allocates: the
 * caller owns the block and returns it with bcg_free_image_memory.  (Nothing in the reference corresponds: its images
 * are NumPy arrays, egocentric.py:125-160.)
 * bytes: wanted size; *dptr: device address; *mapped_bytes: size actually mapped (granularity rounded), to be passed
 * back on free; *compressed: 1 when the allocation got compression, 0 when the device / driver gave a plain one. */
int bcg_alloc_image_memory(int64_t bytes, int32_t want_compression, void** dptr, int64_t* mapped_bytes, int32_t* compressed);
int bcg_free_image_memory(void* dptr, int64_t mapped_bytes);

#ifdef __cplusplus
}
#endif
#endif /* BCG_B200_H_ */
