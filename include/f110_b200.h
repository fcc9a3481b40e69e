/*
 * f110_b200.h — C ABI of the B200-native batched F1TENTH hot path (libf110_b200.so).
 *
 * The reference (f1tenth/f1tenth_gym) is pure Python + numba and has no FFI of its own; its
 * boundary for this path is the Python surface  F110Env -> Simulator -> @njit kernels.  Each entry
 * point below replaces one of those Python-level interfaces (cited file:line, paths relative to
 * gym/f110_gym/envs/ of the reference).  INTEGRATION.md shows the ctypes stub a maintainer of the
 * reference would add to bind them.
 *
 * Conventions
 *   - plain C types only; every pointer inside the structs is a DEVICE pointer owned by the caller
 *     (the Python host side allocates them as torch CUDA tensors), except in the *_host entry points.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - every function returns 0 on success or a negative f110_status; nothing is printed or thrown.
 *   - all arithmetic is IEEE fp64 without FMA contraction (the reference's numba path emits none);
 *     scans are written as fp32 (= fp32(reference fp64 value), <= 1.9e-6 m at 30 m).
 *   - agents are indexed a = env * num_agents + agent ("flat agent index"), SoA over a.
 */
#ifndef F110_B200_H
#define F110_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define F110_ABI_VERSION 2
#define F110_NPARAM 18     /* mu C_Sf C_Sr lf lr h m I s_min s_max sv_min sv_max v_switch a_max v_min v_max width length
                              (key order of the default dict, f110_env.py:130) */
#define F110_NSTATE 7      /* x y steer v yaw yaw_rate slip   (base_classes.py:97) */

typedef enum {
    F110_OK = 0,
    F110_ERR_INVALID = -1,      /* bad argument (NULL pointer, non-positive size, ...)            */
    F110_ERR_NO_MAP = -2,       /* scan before a map is set (laser_models.py:445-446 ValueError)  */
    F110_ERR_CUDA = -3,         /* a CUDA runtime call failed; see f110_last_cuda_error()          */
    F110_ERR_INTEGRATOR = -4,   /* integrator not RK4(1)/Euler(2) (base_classes.py:397-398)       */
    F110_ERR_POSE_COUNT = -5,   /* reset pose count mismatch (base_classes.py:625-626 ValueError) */
    F110_ERR_AGENT_INDEX = -6   /* update_params index out of range (base_classes.py:534)         */
} f110_status;

/* ScanSimulator2D state after set_map (laser_models.py:348-427). */
typedef struct {
    int32_t height, width;
    double resolution, orig_x, orig_y, orig_c, orig_s;
    double eps, max_range;          /* 1e-4, 30.0 (laser_models.py:360) */
    int32_t theta_dis;              /* 2000 */
    int32_t fast_path;              /* 1 iff resolution is a power of two and orig_c==1, orig_s==0:
                                       x/res == x*(1/res) exactly and the rotation is the identity */
    double dt_oob;                  /* dt[-1,-1]: what an off-map ray reads (laser_models.py:79-81) */
    const double *dt;               /* [height*width] fp64 distance transform, row 0 = image bottom */
    const double *dt_cells;         /* [height*width] dt / resolution (exact when fast_path), or NULL: enables
                                       the cell-unit march; ignored unless fast_path */
    const uint8_t *dt_codes;        /* [height*width] rank of dt_cells among the map's 255 smallest distinct values,
                                       255 = escape (read dt_cells); NULL disables the coded march */
    const double *dt_lut;           /* [256] code -> dt_cells value (bit-exact) */
    const double *sines, *cosines;  /* [theta_dis]  sin/cos(linspace(0, 2pi, theta_dis)) (:379-381) */
    const double *sincos;           /* [theta_dis][2] the same values interleaved (sin, cos), or NULL */
    const double *dt_cells_pad;     /* [(height+1)*(width+1)] dt_cells with one extra row and column that hold dt[-1,-1]/resolution
                                       (the off-map value): lets the lean march clamp instead of branch; NULL = round-1 kernels */
    const uint8_t *dt_codes_pad;    /* [(height+1)][codes_pitch] rank codes of dt_cells_pad (same code book as dt_lut; columns beyond
                                       width hold the off-map code too), or NULL */
    uint32_t codes_pitch;           /* row pitch of dt_codes_pad in bytes: >= width+1 and a multiple of 16 (TMA global stride) */
    const double *sincos2;          /* [2*theta_dis][2] the interleaved LUT stored twice back to back (index k and k + theta_dis
                                       hold the same pair), or NULL: lets the march index it without the wrap branch */
    double dt_min_positive;         /* smallest value > 0 in dt (= resolution for an exact EDT), or 0 if unknown.  When it
                                       exceeds eps, `d > eps` (laser_models.py:134) is the same predicate as `d != 0` and the
                                       lean march kernel (csrc/march_lean.cuh) may be used */
    int32_t num_layers;             /* 0/1: one map.  L > 1: dt and dt_cells hold L stacked [H][W] tables that share size,
                                       resolution and origin (multi-map batches); f110_sim.env_layer picks one per env */
} f110_map;

/* Beam tables RaceCar.__init__ builds once (base_classes.py:122-158) + ScanSimulator2D.__init__ (:360-368). */
typedef struct {
    int32_t num_beams;
    double fov, angle_increment, theta_index_increment;
    const double *scan_angles, *cosines, *side_distances;   /* [num_beams] */
    const double *cos_side;         /* [num_beams][2] (cosines[i], side_distances[i]) interleaved, or NULL */
    double side_max;                /* max(side_distances), or 0 if unknown: bound used by the per-agent iTTC pre-test */
} f110_beams;

/* Simulator / RaceCar / F110Env state for N envs x A agents, SoA, caller-owned device memory. */
typedef struct {
    int32_t num_envs, num_agents;
    int32_t integrator;             /* 1 = RK4, 2 = Euler (base_classes.py:40-42) */
    int32_t ego_idx;
    int32_t params_per_env;         /* 0: params is [A][18]; 1: params is [N*A][18] */
    double timestep, lidar_dist, ttc_thresh;   /* 0.01, 0.0, 0.005 (base_classes.py:115) */
    double sim_length, sim_width;   /* Simulator.params['length'/'width'] used by check_collision (:549) */
    const double *params;           /* [A][F110_NPARAM] per agent slot (update_params, base_classes.py:514-534), or
                                       [N*A][F110_NPARAM] per env and slot when params_per_env != 0 (dynamics randomisation) */
    double *state;                  /* [F110_NSTATE][N*A] */
    double *steer_buf;              /* [2][N*A]   steering delay FIFO, row 0 = newest (base_classes.py:270-278) */
    int32_t *steer_cnt;             /* [N*A] */
    double *scan_pose;              /* [N*A][4]   (scan_x, scan_y, first DT lookup in cells | yaw, theta_index0): dynamics -> march */
    double *agent_poses;            /* [N*A][5]   Simulator.agent_poses snapshot (base_classes.py:574): x, y, yaw, cos yaw, sin yaw */
    float *scans;                   /* [N*A][num_beams] */
    int32_t *wall_flag;             /* [N*A]      RaceCar.in_collision (iTTC) */
    double *collisions;             /* [N*A]      obs['collisions'] (0./1.) */
    int32_t *collision_idx;         /* [N*A]      Simulator.collision_idx (-1 = none) */
    /* F110Env level (f110_env.py:165-189); may be NULL if f110_env_post_step is never called */
    double *current_time;           /* [N] */
    double *lap_times, *lap_counts, *toggle_list;   /* [N*A] */
    int32_t *near_starts;           /* [N*A] */
    double *start_xs, *start_ys, *start_thetas;     /* [N*A] */
    double *start_rot;              /* [N][4] */
    uint8_t *done;                  /* [N] */
    uint8_t *checkpoint_done;       /* [N*A]  info['checkpoint_done'] */
    int32_t *env_arrivals;          /* reserved (ABI v1 used it as a per-env arrival counter of f110_tick); may be NULL */
    const int32_t *env_layer;       /* [N] map layer of each env for stacked maps (f110_map.num_layers > 1), or NULL */
    unsigned long long *lookup_counter;   /* optional [1]: total DT lookups (roofline denominator); NULL = off */
    unsigned long long *tick_counter;     /* optional [1]: incremented by every f110_step; keys the noise stream
                                             and the auto-reset draw so that CUDA-graph replays stay distinct */
    /* optional work queue of the persistent ray-march kernel (csrc/march.cuh): 32-beam items, last tick's
       heavy items first.  Results never depend on it.  All NULL/0 = off (one block per 64-beam tile instead).
       I = N*A*march_ipa items; march_ipa = ceil(num_beams/32) (32-beam items) or ceil(num_beams/64) (64-beam items), <= 256. */
    uint32_t *march_cost;           /* [N*A*256] indexed by (agent << 8 | item); initialised to 0xFFFFFFFF (= unknown) */
    uint32_t *march_order;          /* [3][I]  */
    uint32_t *march_count;          /* [4]     zero-initialised by the caller */
    int32_t march_ipa;
    double *march_rec;              /* [N*A][8] per-agent record k_dynamics hands to the lean march kernel (scan position in
                                       cell units, first lookup, fixed-point LUT index, iTTC threshold, map-layer offset;
                                       csrc/march_lean.cuh), or NULL: round-1 kernels */
    /* scan noise (laser_models.py:429,450-452): N(0, noise_std^2) per beam, added before iTTC; 0 = off */
    double noise_std;
    uint64_t noise_seed;
} f110_sim;

int f110_abi_version(void);
const char *f110_status_string(int status);
const char *f110_last_cuda_error(void);

/* ---- the per-tick hot path -------------------------------------------------------------------- */

/* Simulator.step (base_classes.py:553-612): pid + RK4/Euler dynamics -> 1080-beam ray-march (+fused
 * iTTC) -> GJK, wall-hit state zeroing, opponent ray-cast.  actions: device [N*A][2] = (steer, speed).
 * Launches 3 kernels on `stream`; no host synchronisation. */
int f110_step(const f110_sim *sim, const f110_map *map, const f110_beams *beams,
              const double *actions, void *stream);

/* f110_step with CUDA events recorded on `stream` around each of its three kernels; synchronises and
 * returns their durations in milliseconds: kernel_ms[0..2] = dynamics, ray-march, finalize (host array).
 * Measurement aid for bench.py's roofline figure; not for the hot loop. */
int f110_step_profile(const f110_sim *sim, const f110_map *map, const f110_beams *beams,
                      const double *actions, float *kernel_ms, void *stream);

/* Simulator.reset / RaceCar.reset (base_classes.py:183-204, 614-630) for the envs whose env_mask
 * byte is non-zero (env_mask == NULL: all).  poses: device [N*A][3].  No tick is executed. */
int f110_reset(const f110_sim *sim, const double *poses, const uint8_t *env_mask, void *stream);

/* The counters/start-frame part of F110Env.reset (f110_env.py:319-331) for masked envs. */
int f110_env_reset(const f110_sim *sim, const double *poses, const uint8_t *env_mask, void *stream);

/* F110Env.step tail: time, _check_done lap logic (f110_env.py:204-246, 294-302) -> done, lap arrays. */
int f110_env_post_step(const f110_sim *sim, void *stream);

/* Benchmark/RL convenience (no reference equivalent; SURVEY.md 8d policy): every env whose ego has
 * collisions != 0 is reset (Simulator.reset + env counters) to start_poses[k], k drawn from a
 * counter-based hash of (seed, tick, env); agent i takes start_poses[(k - pose_gap*i) mod K].
 * What the caller sees after a tick that ended an episode: done[env] = 1 and collisions / scans of the crash
 * (the finished episode's last observation), while state, steer FIFO, lap counters, toggles and current_time are
 * those of the NEW episode (a car at rest on its start pose, time 0); done is recomputed by the next tick.
 * At most 32 agents per env (F110_ERR_INVALID otherwise; stepping itself has no such limit). */
int f110_autoreset(const f110_sim *sim, const double *start_poses, int32_t num_start, int32_t pose_gap,
                   uint64_t seed, uint64_t tick, void *stream);

/* One whole tick in three launches: f110_step + (env_level != 0) f110_env_post_step + (start_poses != NULL)
 * f110_autoreset, with the finalize kernel of the step, the lap logic and the auto-reset fused into one kernel (a
 * block owns whole envs; with more than 32 agents per env they run as separate launches).  Same results as calling
 * the three entry points in that order.  This is what a training loop / CUDA graph should replay. */
int f110_tick(const f110_sim *sim, const f110_map *map, const f110_beams *beams, const double *actions,
              int32_t env_level, const double *start_poses, int32_t num_start, int32_t pose_gap, uint64_t seed,
              void *stream);

/* Same tick through HOST buffers: copies actions H2D, runs f110_step (+ f110_env_post_step when the
 * lap arrays are bound), copies the observation D2H and synchronises the stream.
 * Any output pointer may be NULL to skip that copy.  Host buffers should be pinned. */
typedef struct {
    float *scans;           /* [N*A][B] */
    double *state;          /* [7][N*A] */
    double *collisions;     /* [N*A] */
    uint8_t *done;          /* [N] */
    double *lap_times, *lap_counts;   /* [N*A] */
    uint8_t *scans_u24;     /* [N*A][B][3] optional narrow scan block for PCIe-bound host consumers (f110_step_host_async only,
                               used when `scans` is NULL): each range as 24-bit fixed point, little endian, value = q * 2^-19 m
                               (step 1.9e-6 m = the fp32 scan's own resolution at 30 m; |error| <= 9.6e-7 m; a noisy range
                               below 0 clamps to 0).  3 bytes per beam instead of 4: see f110_pack_scans_u24. */
} f110_host_obs;
int f110_step_host(const f110_sim *sim, const f110_map *map, const f110_beams *beams,
                   const double *actions_host, double *actions_dev_scratch, const f110_host_obs *out,
                   void *stream);

/* Pipelined variant for host-side consumers: the tick runs on `compute_stream`, its observation is
 * snapshotted into the DEVICE staging buffers `stage` (same layout as f110_host_obs), and the D2H copies
 * into `out` run on `copy_stream`, so that the copy of tick t overlaps the compute of tick t+1.  No host
 * synchronisation: the caller alternates between two (stage, out, event) sets and, before reusing a set or
 * reading its host buffers, waits for `ev_copy_done` (cudaEventSynchronize).  `ev_tick_done` and
 * `ev_copy_done` are cudaEvent_t created by the caller.  Before overwriting `stage` the compute stream
 * waits for the previous copy out of it (the event's last record). */
int f110_step_host_async(const f110_sim *sim, const f110_map *map, const f110_beams *beams,
                         const double *actions_host, double *actions_dev_scratch, const f110_host_obs *stage,
                         const f110_host_obs *out, void *compute_stream, void *copy_stream, void *ev_tick_done,
                         void *ev_copy_done);

/* scans [count] fp32 (device) -> out [count][3] bytes (device): q = round(range * 2^19) clamped to [0, 2^24-1], little endian.
 * No reference counterpart (the reference hands numpy arrays to a policy in the same process); batch extension for host-side
 * consumers behind PCIe.  Decode: (b0 | b1 << 8 | b2 << 16) * 2^-19. */
int f110_pack_scans_u24(const float *scans, int64_t count, uint8_t *out, void *stream);

/* ---- standalone kernels (unit-parity surface; device pointers) ------------------------------- */

/* ScanSimulator2D.scan without noise / get_scan (laser_models.py:148-186, 429-454): M poses -> [M][B]. */
int f110_scan(const f110_map *map, const f110_beams *beams, const double *poses /* [M][3] */, int32_t M,
              float *out_f32 /* [M][B] or NULL */, double *out_f64 /* [M][B] or NULL */,
              unsigned long long *lookup_counter /* [1] or NULL */, void *stream);
/* vehicle_dynamics_st (dynamic_models.py:123-176): x [M][7], u [M][2], params [18] -> f [M][7]. */
int f110_vehicle_dynamics_st(const double *x, const double *u, const double *params, int32_t M, double *f,
                             void *stream);
/* vehicle_dynamics_ks (dynamic_models.py:90-121): x [M][5] (x, y, steer, v, yaw), u [M][2], params [18] -> f [M][5]. */
int f110_vehicle_dynamics_ks(const double *x, const double *u, const double *params, int32_t M, double *f,
                             void *stream);
/* pid (dynamic_models.py:178-221): in [M][4] = (speed, steer, current_speed, current_steer) -> out [M][2] = (accl, sv). */
int f110_pid(const double *in, const double *params, int32_t M, double *out, void *stream);
/* get_vertices (collision_models.py:237-260): poses [M][3] -> [M][4][2] (rl, rr, fr, fl). */
int f110_get_vertices(const double *poses, double length, double width, int32_t M, double *out, void *stream);
/* collision (GJK, collision_models.py:113-182): va, vb [M][4][2] -> out [M] 0/1. */
int f110_collision(const double *va, const double *vb, int32_t M, int32_t *out, void *stream);
/* collision_multiple (collision_models.py:184-212): verts [M][n][4][2] -> collisions [M][n], collision_idx [M][n]. */
int f110_collision_multiple(const double *verts, int32_t M, int32_t n, double *collisions, double *collision_idx,
                            void *stream);
/* check_ttc_jit (laser_models.py:188-217): scans [M][B] fp64, vel [M] -> out [M] 0/1. */
int f110_check_ttc(const f110_beams *beams, const double *scans, const double *vel, double ttc_thresh, int32_t M,
                   int32_t *out, void *stream);
/* ray_cast (laser_models.py:318-346): pose [M][3], opponent vertices [M][4][2], scans [M][B] fp32 modified in
 * place; window [M][2] (min_ind, max_ind of get_blocked_view_indices :282-315) optional. */
int f110_ray_cast(const f110_beams *beams, const double *poses, const double *opp_vertices, int32_t M,
                  float *scans, int32_t *window, void *stream);
/* Seeded scan noise (laser_models.py:450-452; N(0, std^2) per beam).  Counter-based Philox-4x32 +
 * Box-Muller; statistical, not bit, parity with numpy's PCG64 stream. */
int f110_scan_noise(float *scans, int64_t count, double std_dev, uint64_t seed, uint64_t offset, void *stream);

/* Batched pure-pursuit policy (reference examples/waypoint_follow.py:15-217, PurePursuitPlanner.plan):
 * waypoint columns wx, wy, wv [num_waypoints] and poses pose_x/y/theta [M] (device) -> actions_out [M][2] =
 * (steering angle, speed), the layout f110_step consumes.  max_reacquire is 20.0 in the reference (:154). */
int f110_pure_pursuit(const double *wx, const double *wy, const double *wv, int32_t num_waypoints, const double *pose_x,
                      const double *pose_y, const double *pose_theta, int32_t M, double lookahead_distance, double vgain,
                      double wheelbase, double max_reacquire, double *actions_out, void *stream);

/* The same policy over several waypoint tables (one per track of a multi-map batch; batch extension, no reference
 * counterpart): the tables are concatenated in wx/wy/wv, table t occupies rows [table_start[t], table_start[t+1])
 * (table_start [num_tables+1] i32, device, every table >= 2 rows) and pose a follows table pose_table[a]
 * (i32 [M], device, values in [0, num_tables) -- not range-checked on the device). */
int f110_pure_pursuit_tables(const double *wx, const double *wy, const double *wv, const int32_t *table_start,
                             int32_t num_tables, const int32_t *pose_table, const double *pose_x, const double *pose_y,
                             const double *pose_theta, int32_t M, double lookahead_distance, double vgain, double wheelbase,
                             double max_reacquire, double *actions_out, void *stream);

/* Exact Euclidean distance transform on the device (load-time; reference laser_models.py:40-53 get_dt =
 * resolution * scipy.ndimage.distance_transform_edt(bitmap)): occupied [H][W] u8 (1 where the thresholded image
 * is 0), scratch [H][W] i32, dt_out [H][W] f64 = resolution * sqrt(k) with k the exact squared cell distance
 * (optionally written to k_out [H][W] i64).  Bit-identical to the scipy table. */
int f110_edt(const uint8_t *occupied, int32_t height, int32_t width, double resolution, int32_t *scratch, double *dt_out,
             int64_t *k_out, void *stream);

/* Walls of a generated track (reference unittest/random_trackgen.py:156-165 shapely buffer(+-WIDTH) of the closed
 * centerline, :167-178 the two offset curves drawn 3 pt wide): segments [num_segments][5] (device) = ax, ay, bx-ax,
 * by-ay, 1/|b-a|^2 of the closed centerline in PIXEL units (pixel (r, c) has its centre at (c+0.5, r+0.5), row 0 =
 * bottom of the map like the flipped image of laser_models.py:399); occupied [H][W] u8 = 1 where the pixel centre's
 * distance d to the centerline satisfies wall_inner <= d <= wall_outer (the input f110_edt takes); dist2_out
 * (optional) [H][W] f64 = d^2 in pixels^2 (d < wall_inner = on the track). */
int f110_rasterize_track(const double *segments, int32_t num_segments, double wall_inner, double wall_outer, int32_t height,
                          int32_t width, uint8_t *occupied, double *dist2_out, void *stream);

/* ---- headless renderer ------------------------------------------------------------------------ */

/* What a frame shows (reference rendering.py / F110Env.render, f110_env.py:387-418, drawn without a window).  Every pixel
 * gets a label: 0 free or off the map, 1 wall (the map cell under the pixel centre has dt == 0, found with the literal
 * xy_2_rc of laser_models.py:55-86; an env of a stacked map reads its own layer), 2 the viewer's car, 3 another car of the
 * viewer's env, 4 an endpoint of the viewer's last scan (draw_scan; ranges < max_range), 5 a waypoint; later layers win in
 * that order from 1 to 5, except that the viewer's car wins over other cars.  Row 0 is the top row; pixel (r, c) has its
 * centre at u = (c + 0.5 - 0.5 width) mpp, v = (0.5 height - r - 0.5) mpp camera metres, i.e. at world
 * x = cx + (u cr - v sr), y = cy + (u sr + v cr).  camera 0 is a fixed window, (cx, cy) = center, (cr, sr) = (1, 0);
 * camera 1 follows the viewer heading up, (cx, cy) = its (x, y) and (cr, sr) = (sin yaw, -cos yaw), from `state`.  A car
 * covers the pixels whose centre lies inside the rectangle of get_vertices (collision_models.py:237-260).  A point layer
 * lands on pixel c = floor(u / mpp + 0.5 width), r = floor(0.5 height - v / mpp) with (u, v) its camera coordinates, and
 * is dropped outside the frame.  Walls differ from the reference on purpose: it draws 1-pixel points at the corners of the
 * image pixels that are 0; here a frame fills the cells the simulator collides with (image pixels <= 128). */
typedef struct {
    int32_t width, height, channels, camera;   /* width % 4 == 0; channels 1 (label per pixel) | 3 (palette[label] RGB);
                                                  camera 0 (fixed window) | 1 (viewer, heading up) */
    double center_x, center_y, metres_per_pixel;   /* center: camera 0 only */
    int32_t draw_scan;                          /* != 0: label 4 layer (needs `beams`) */
    uint8_t palette[8][3];                      /* RGB of each label when channels == 3 */
    const double *wx, *wy; int32_t num_waypoints;          /* device [num_waypoints]; NULL / 0: no waypoint layer */
    const int32_t *table_start; int32_t num_tables; const int32_t *env_table;   /* optional planner layout
                                                  (f110_pure_pursuit_tables): env e draws rows [table_start[t], table_start[t+1])
                                                  of table t = env_table[e]; env_table holds num_envs entries (device i32);
                                                  NULL: every env draws every row */
} f110_view;

/* Render num_frames frames into out [num_frames][height][width][channels] u8 (device).  viewers [num_frames] (device i32)
 * holds the flat agent index each frame is drawn for, or is NULL: then num_frames == num_envs and frame e is env e seen from
 * its ego_idx.  An out-of-range viewer gives an all-0 frame (and camera (0, 0, 0, 0)).  camera_out (device [num_frames][4]
 * f64, optional) receives each frame's (cx, cy, cr, sr).  beams is read only with draw_scan.  Reads the simulation state,
 * writes nothing but out / camera_out; no host synchronisation and no allocation, so it can be captured in a CUDA graph
 * after f110_tick.  F110_ERR_NO_MAP when `map` has no table bound. */
int f110_render(const f110_sim *sim, const f110_map *map, const f110_beams *beams, const f110_view *view,
                const int32_t *viewers, int32_t num_frames, uint8_t *out, double *camera_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* F110_B200_H */
